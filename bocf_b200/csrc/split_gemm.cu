// split_gemm.cu -- the two candidate-side contractions of the GP posterior on the 5th-generation tensor cores.
//
//   V  = K* Linv^T   (posterior.py:312, the reference's dtrtrs route)      var  = k** - sum_k V^2
//   Wt = V  Linv     (= K* W^-1, gp.py:474)                                 dvar = gradients_X(-2 Wt, x*, X)
//
// Blackwell's tcgen05 has no fp64 kind, so the fp64 operands are split into signed 8-bit digits (balanced base-256
// expansion of round(x * 2^(8S-2-e)), e a per-row power-of-two scale; SA digits on the candidate side, SB on the
// factor side) and the product is assembled from exact integer GEMMs on `tcgen05.mma.kind::i8` (SASS UTCIMMA):
// int8 x int8 products accumulated EXACTLY in int32 tensor memory, one accumulator per digit weight 256^(ta+tb).
// A SCHEME (SA, SB, LMIN) keeps the digit pairs with ta + tb >= LMIN.  Which pairs are kept matters more than the
// number of digits: the low digits of an operand are full-size even where the operand is small, so a dropped pair
// costs the same absolute error everywhere, while the quantisation error is multiplied by the (usually small) other
// operand (tests/test_split_numerics.py; profiles/r2_pair_selection.md):
//     554  (15 pairs)  variance to ~3e-8 relative            -- first contraction of the default mode
//     442  (13 pairs)  variance ~3e-7, variance gradient ~4e-8 -- second contraction of the default mode
//     331  ( 8 pairs)  variance gradient ~1e-5               -- second contraction of the mixed mode
//     665  (21 pairs)  ill-conditioned factors
//
// Kernel structure (persistent, warp specialised, 1 CTA / SM):
//   warp 0   producer: one lane streams 64-byte-wide K chunks of the packed, pre-swizzled digit planes of A
//            (128 candidates) and B (NT factor rows) into a STAGES-deep shared-memory ring with bulk async copies
//            (TMA engine, cp.async.bulk + mbarrier complete_tx).
//   warp 1   MMA issuer: the WHOLE warp walks the tile / stage loop with warp-uniform control flow (the warp index
//            comes from a shuffle, so the compiler keeps descriptors and loop state on the uniform datapath) and one
//            elected lane issues, per 32-byte K step, one instruction per A digit plane
//                 D[128 x np NT] += A_ta * [B_tbmin .. B_{SB-1}]^T
//            whose B operand STACKS the kept digit planes along N, so every A plane is read from shared memory once
//            per step and each weight level lands in its own TMEM column block.  (Round 1 issued from one divergent
//            lane and rebuilt both descriptors per instruction: ~137 clocks per MMA against 24-120 clocks of tensor
//            work -- profiles/r2_mma_probe.log shows the same stream at 95 % of the tensor pipe when issued lean.)
//            Accumulators are double buffered so the epilogue of tile t overlaps the MMAs of tile t+1.
//   warps 2+ epilogue (EW / 4 warps per TMEM lane group, alternating 8-column groups): tcgen05.ld the int32 levels
//            of a row (lane = candidate), int32 -> fp64 by a magic-number add (no conversion-pipe instructions),
//            Horner them into one fp64 value, apply the column scale, and fuse the reductions of the reference:
//            VAR : sum_k V^2 per candidate (+ re-split V into S2 digit planes = the A operand of the second GEMM)
//            DVAR: T = Wt * G*,  sum_b T and sum_b T Xs_b  (finalize_kernel forms xs_i sum T - sum T Xs_b).
//            The sums live in registers across all column tiles of a work unit (see NP below).
// Triangular structure of Linv is exploited per column tile: K chunks (64) for the loads, K steps (32) for the MMAs.
#include <cmath>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "model.h"
#include "tc05.cuh"

namespace bocf {
namespace sg {

constexpr int KC = 64;        // bytes (= int8 elements) of K per shared-memory row: one SWIZZLE_64B span
constexpr int TM = 128;       // candidate rows per tile (= TMEM lanes)
constexpr int SMEM_MAX = 232448;

__host__ __device__ __forceinline__ uint32_t sw64(int r, int c) {   // byte offset of (row r, byte c) in a packed plane
  return (uint32_t)(r * 64 + ((((c >> 4) ^ ((r >> 1) & 3))) << 4) + (c & 15));
}
__host__ __device__ constexpr int pow2_cols(int c) { return c <= 32 ? 32 : c <= 64 ? 64 : c <= 128 ? 128 : c <= 256 ? 256 : 512; }

// A digit-pair scheme: SA digit planes of the candidate-side operand, SB of the factor side, pairs with
// ta + tb >= LMIN kept; NT = factor rows (output columns) per tile; EW = epilogue warps.
template <int SA_, int SB_, int LMIN_, int NT_, int EW_>
struct Scheme {
  static constexpr int SA = SA_, SB = SB_, LMIN = LMIN_, NT = NT_, EW = EW_;
  static constexpr int NL = SA + SB - 1 - LMIN;        // weight levels = TMEM accumulators per output column
  static constexpr int CODE = SA * 100 + SB * 10 + LMIN;
};
using P331 = Scheme<3, 3, 1, 64, 8>;
using P442 = Scheme<4, 4, 2, 48, 12>;
using P554 = Scheme<5, 5, 4, 48, 12>;
using P665 = Scheme<6, 6, 5, 32, 8>;

struct SchemeInfo {
  int code, SA, SB, LMIN, NT, EW, NL, pairs;
};
inline bool scheme_info(int code, SchemeInfo* o) {
  auto fill = [&](int SA, int SB, int LMIN, int NT, int EW) {
    int pairs = 0;
    for (int ta = 0; ta < SA; ++ta)
      for (int tb = 0; tb < SB; ++tb)
        if (ta + tb >= LMIN) ++pairs;
    *o = SchemeInfo{SA * 100 + SB * 10 + LMIN, SA, SB, LMIN, NT, EW, SA + SB - 1 - LMIN, pairs};
  };
  switch (code) {
    case 331: fill(3, 3, 1, 64, 8); return true;
    case 442: fill(4, 4, 2, 48, 12); return true;
    case 554: fill(5, 5, 4, 48, 12); return true;
    case 665: fill(6, 6, 5, 32, 8); return true;
  }
  return false;
}

template <class SCH, int DP = 0>
struct Cfg {
  static constexpr int SA = SCH::SA, SB = SCH::SB, LMIN = SCH::LMIN, NT = SCH::NT, NL = SCH::NL;
  static constexpr int EPI_WARPS = SCH::EW, EPI_THREADS = EPI_WARPS * 32, NTHREADS = 64 + EPI_THREADS;
  static constexpr int PART_SPLIT = EPI_WARPS / 4;       // partial sums per unit (one per warp of a lane group)
  static constexpr int A_PLANE = TM * KC, B_PLANE = NT * KC;
  static constexpr int A_STAGE = SA * A_PLANE, B_STAGE = SB * B_PLANE, STAGE = A_STAGE + B_STAGE;
  static constexpr int ACC_COLS = NL * NT;
  static constexpr int NBUF = (2 * ACC_COLS <= 512) ? 2 : 1;
  static constexpr int TMEM_COLS = pow2_cols(NBUF * ACC_COLS);
  static constexpr int XB_BYTES = NT * DP * 8;                       // DVAR: scaled training inputs of the column tile
  static constexpr int CS_OFF = 256, CS_BYTES = 2 * NT * 16;          // two buffers of {cs, cs * vq} pairs per column
  static constexpr int XB_OFF = CS_OFF + CS_BYTES;
  static constexpr int HEAD = XB_OFF + XB_BYTES;                      // barriers, tmem slot, column scales, xb tile
  static constexpr int STAGES_FIT = (SMEM_MAX - HEAD - 512) / STAGE;
  static constexpr int STAGES = STAGES_FIT > 8 ? 8 : STAGES_FIT;
  static constexpr int SMEM_BYTES = HEAD + 512 + STAGES * STAGE;
  // kept digit planes of B for A plane ta: tb = tbmin(ta) .. SB-1, landing on levels lev0(ta) .. lev0 + np - 1
  __host__ __device__ static constexpr int tbmin(int ta) { return LMIN - ta > 0 ? LMIN - ta : 0; }
  __host__ __device__ static constexpr int np(int ta) { return SB - tbmin(ta); }
  __host__ __device__ static constexpr int lev0(int ta) { return ta + tbmin(ta) - LMIN; }
  static_assert(SA >= 2 && SA <= 6 && SB >= 2 && SB <= 6 && NT % 16 == 0 && SB * NT <= 256,
                "stacked B operand must fit one MMA (N <= 256)");
  static_assert(LMIN <= SA - 1 + SB - 1 && LMIN >= 0 && LMIN <= SB - 1, "every A plane needs at least one partner");
  static_assert(STAGES >= 2, "need at least a double-buffered ring");
  static_assert(B_STAGE % 512 == 0 && A_STAGE % 512 == 0, "planes must keep the 512-byte swizzle period");
  static_assert((2 * STAGES + 2 * NBUF) * 8 + 16 <= CS_OFF && XB_OFF % 16 == 0, "head area too small");
  static_assert(EPI_WARPS % 4 == 0 && (NT / 8) % PART_SPLIT == 0, "column groups must divide evenly over the warps");
};

// EPI_DACQ: the second contraction with the fused acquisition-gradient epilogue -- instead of T = Wt G* it contracts
//   u_b = G*_b (WA_j alpha_b - 2 WB_j Wt_b)      (WA, WB: per-candidate weights from the MC pass, acq.cu)
// so that sum_j (xs_j sum_b u_b - sum_b u_b Xs_b) / l_j = sum_j WA_j dmu_j + WB_j dvar_j = grad acq  (uEI_noiseless.py:163-166).
enum { EPI_RAW = 0, EPI_VAR = 1, EPI_DVAR = 2, EPI_DACQ = 3 };
enum { TRI_FULL = 0, TRI_K_LE_N = 1, TRI_K_GE_N = 2 };

struct GemmParams {
  const uint8_t* A;        // [m][RT][KCH][SA][128][64]  packed digit planes of the candidate-side operand
  const uint8_t* B;        // [Hm][nct][KCH][SB][NT][64] packed digit planes of the factor-side operand
  const double* cs;        // [Hm][nct*NT]               column scale (power of two)
  int m, h, RT, nct, KCH, n, tri;
  int RTv;                 // candidate tiles that hold at least one valid candidate (<= RT): the others are skipped -- the
                           // ragged last chunk of a sweep and the tiny batches of the optimiser are mostly padding
  int64_t Nc, Nvalid;
  // RAW
  double* raw_out;         // [m*RT*128][ldo]
  const double* raw_rs;    // [m*RT*128] row scale
  int ldo;
  // VAR
  double* part_var;        // [m][np*PART_SPLIT][Nc]
  uint8_t* A2;             // [m][RT][KCH][S2][128][64]  digit planes of V (nullptr: not needed)
  const double* vq;        // [Hm] 2^(8 S2 - 2 - eV)
  // DVAR
  double* part_dvar;       // [m][np*PART_SPLIT][Nc][d]   sum_b T_b Xs_bq
  double* part_s0;         // [m][np*PART_SPLIT][Nc]      sum_b T_b
  const double* GsT;       // [m][n16][Nc]
  const double* Xc;        // [Nvalid][d]
  const double* Xs;        // [Hm][n_pad][d]
  const double* alpha;     // DACQ: [Hm][n_pad]
  const double* wa;        // DACQ: [m][Nc] weight of the mean gradient
  const double* wb;        // DACQ: [m][Nc] weight of the variance gradient
  const OutHyp* hyp;
  int d, n16, n_pad;
  int np;                  // parts per candidate tile
  // DACQ: the units (j, rt) to walk, as ids j * RTv + rt in ascending order, and their number (active_units_kernel,
  // posterior.cu).  nullptr: every unit.
  const int* unit_list;
  const int* unit_count;
};

// Work decomposition.  A UNIT is (output j, candidate tile rt, part p of NP): the column tiles ct = p, p+NP, ... of one
// 128-candidate tile.  A persistent CTA owns whole units and walks their column tiles back to back, so the epilogue
// keeps its per-candidate reductions in registers across the unit and writes ONE partial per (unit, epilogue warp)
// instead of one per column tile.  NP = 1 (a CTA owns the whole row of column tiles of its candidate tile) measured
// best on B200: 354 vs 371 (NP = 2) vs 390 ms (NP = 4) per 1M-candidate step at cfg 3 -- fewer partial sums, and the
// tile's digit planes are re-read by one SM back to back.  More parts only pay when there are fewer units than SMs.
// Two reasons to give a candidate tile to more than one CTA:
//  * small batches (the L-BFGS rounds of the acquisition optimiser: tens of candidates = one candidate tile per output)
//    have fewer units than SMs;
//  * LARGE n: a unit's A tile (SA planes x 128 candidates x n) is re-streamed once per column tile, and the tiles of all
//    resident units must stay in L2 for that to be cheap: 655 KB x 148 CTAs = 97 MB at n = 1000 (fits the 126 MB), 2.6 MB x
//    148 = 382 MB at n = 4000 -- there the re-streaming went to HBM and both contractions ran HBM-bound (cfg 5: 0.99 /
//    0.81 s per 200k candidates with one part, 0.59 / 0.54 s with four CTAs sharing each tile).
inline int parts_for(int units_at_np1, int sms, int64_t a_tile_bytes, int64_t l2_bytes) {
  int np = 1;
  if (units_at_np1 * 4 <= sms) np = 4;            // 8 parts measured no faster at 17 candidates: a small batch still
  else if (units_at_np1 * 2 <= sms) np = 2;       // streams every factor plane (148 MB at cfg 3), that is its floor
  const int64_t budget = l2_bytes * 4 / 5;
  while (np < 8 && (int64_t)(sms / np) * a_tile_bytes > budget) np *= 2;
  return np;
}

struct TileInfo {
  int j, rt, p, ct, kb, ke;
  int sb, se;                   // first / one-past-last 32-byte K STEP that touches the triangle (MMA issue range)
  bool valid, first, last;      // first / last column tile of the unit
};

// Walks the column tiles this CTA owns: units cta, cta + grid, ... and inside a unit the tiles ct = p, p + NP, ...
// The (output, candidate tile, part) decode costs integer divisions, so it is done once per unit; advancing inside a
// unit is additions only (every role of the kernel walks the same sequence, the epilogue one tile ahead as well).
// LIST (EPI_DACQ): the (output, candidate tile) pairs come from P.unit_list, each still split into the same NP parts,
// so a listed unit is computed exactly as in the dense walk; the grid stays what the host sized for the dense walk and
// CTAs left without a unit fall through.
template <int NT, bool LIST>
struct TileWalk {
  int u, units, j, rt, p, ct;
  __device__ __forceinline__ void start(const GemmParams& P) {
    units = (LIST && P.unit_list != nullptr) ? __ldg(P.unit_count) * P.np : P.m * P.RTv * P.np;
    u = (int)blockIdx.x - (int)gridDim.x;
    ct = P.nct;                                            // forces the first next() to open a unit
    j = rt = p = 0;
  }
  __device__ __forceinline__ bool next(const GemmParams& P, TileInfo& ti) {
    bool first = false;
    ct += P.np;
    while (ct >= P.nct) {                                  // open the next unit that has at least one column tile
      u += (int)gridDim.x;
      if (u >= units) return false;
      if (LIST && P.unit_list != nullptr) {
        const int e = u / P.np;
        p = u - e * P.np;
        const int id = __ldg(P.unit_list + e);
        j = id / P.RTv;
        rt = id - j * P.RTv;
      } else {
        j = u / (P.RTv * P.np);
        const int r = u - j * (P.RTv * P.np);
        rt = r / P.np;
        p = r - rt * P.np;
      }
      ct = p;
      first = true;
    }
    ti.j = j;
    ti.rt = rt;
    ti.p = p;
    ti.ct = ct;
    ti.valid = true;
    ti.first = first;
    ti.last = (ct + P.np >= P.nct);
    const int kch_used = (P.n + KC - 1) / KC;
    if (P.tri == TRI_K_LE_N) {                              // K index <= column index
      const int cend = min((ct + 1) * NT, P.n);
      ti.kb = 0;
      ti.ke = min(kch_used, (cend + KC - 1) / KC);
      ti.sb = 0;
      ti.se = min(ti.ke * (KC / 32), (cend + 31) / 32);
    } else if (P.tri == TRI_K_GE_N) {                       // K index >= column index
      ti.kb = (ct * NT) / KC;
      ti.ke = kch_used;
      ti.sb = (ct * NT) / 32;
      ti.se = ti.ke * (KC / 32);
    } else {
      ti.kb = 0;
      ti.ke = kch_used;
      ti.sb = 0;
      ti.se = ti.ke * (KC / 32);
    }
    return true;
  }
};

// digits of a 64-bit integer |Y| < 2^(8S-2): byte t of the result is the balanced base-256 digit of weight 256^t
template <int S>
__host__ __device__ constexpr unsigned long long digit_bias() {
  return (S == 6) ? 0x808080808080ull : (S == 5) ? 0x8080808080ull : (S == 4) ? 0x80808080ull : (S == 3) ? 0x808080ull : 0x8080ull;
}
template <int S>
__device__ __forceinline__ unsigned long long balanced_digits(long long Y) {
  constexpr unsigned long long BIAS = digit_bias<S>();
  return ((unsigned long long)Y + BIAS) ^ BIAS;
}

// int32 -> double without the (slow) I2F.F64 conversion pipe: (2^52 + 2^31 + c) is exactly representable, one DADD.
__device__ __forceinline__ double i32_to_f64(uint32_t c) {
  return __hiloint2double(0x43300000, (int)(c ^ 0x80000000u)) - 4503601774854144.0;
}
// int64 (|x| < 2^51) -> double the same way: 64-bit integer add of the 1.5 * 2^52 bit pattern, one DADD.
__device__ __forceinline__ double i64_to_f64(long long x) {
  return __longlong_as_double(x + 0x4338000000000000LL) - 6755399441055744.0;
}
// sum_lb 256^lb c[lb]: adjacent levels are merged in 64-bit integer arithmetic first (|c[lb]| < 2^29, so
// c[lb] * 256 + c[lb-1] < 2^38), so only ceil(NL/2) conversions and floor(NL/2) fused multiply-adds reach the fp64
// pipe instead of NL and NL-1.  The 1.5 * 2^52 bit pattern of the int64 -> fp64 trick rides in the addend of the
// widening multiply-add (one IMAD.WIDE per pair, no separate 64-bit add).
template <int NL, int W>
__device__ __forceinline__ double levels_to_f64(const uint32_t (&c)[NL][W], int e) {
  double v = 0.0;
#pragma unroll
  for (int lb = NL - 1; lb >= 0; lb -= 2) {
    if (lb >= 1) {
      const long long addend = (long long)(int)c[lb - 1][e] + 0x4338000000000000LL;
      const double t = __longlong_as_double((long long)(int)c[lb][e] * 256 + addend) - 6755399441055744.0;
      v = (lb == NL - 1) ? t : fma(v, 65536.0, t);
    } else {
      v = (lb == NL - 1) ? i32_to_f64(c[0][e]) : fma(v, 256.0, i32_to_f64(c[0][e]));
    }
  }
  return v;
}

// The same sum divided by 256, for the fused epilogues: level 0 is folded into level 1 first,
//   t = c[1] + round(c[0] / 256)   (|t| < 2^29 + 2^21),
// which drops at most half a unit of level 1 -- 2^7 in units of the full sum, against the ~2^10 those units already
// carry from the digit pairs below LMIN -- and saves one conversion and one fused multiply-add per element.  The
// factor 256 is folded into the (power-of-two) column scale by the caller.
template <int NL, int W>
__device__ __forceinline__ double levels_to_f64_merged(const uint32_t (&c)[NL][W], int e) {
  static_assert(NL >= 2, "needs at least two levels");
  const int t = (int)c[1][e] + (((int)c[0][e] + 128) >> 8);
  double v = 0.0;
#pragma unroll
  for (int lb = NL - 1; lb >= 1; lb -= 2) {
    if (lb >= 2) {
      const int lo = (lb - 1 == 1) ? t : (int)c[lb - 1][e];
      const long long addend = (long long)lo + 0x4338000000000000LL;
      const double x = __longlong_as_double((long long)(int)c[lb][e] * 256 + addend) - 6755399441055744.0;
      v = (lb == NL - 1) ? x : fma(v, 65536.0, x);
    } else {                                                 // lb == 1: t alone
      v = (lb == NL - 1) ? i32_to_f64((uint32_t)t) : fma(v, 256.0, i32_to_f64((uint32_t)t));
    }
  }
  return v;
}

// digits of rint(x) for |x| < 2^46 without F2I: adding 1.5 * 2^52 leaves rint(x) (two's complement) in the low mantissa bits
template <int S>
__device__ __forceinline__ unsigned long long balanced_digits_of(double x) {
  return balanced_digits<S>(__double_as_longlong(x + 6755399441055744.0));
}

// One 32-byte K step of the digit-pair scheme: one instruction per A plane, B planes stacked along N.  FIRST: the
// accumulators hold the previous tile -- every level is overwritten (accumulate = 0) by the first instruction that
// touches it; an instruction that reaches one level below the initialised range is split in two.
template <class C, bool FIRST>
__device__ __forceinline__ void issue_kstep(uint32_t a_lo, uint32_t b_lo, uint32_t d_tmem) {
  int init_lo = C::NL;                                   // levels >= init_lo are initialised (compile-time folded)
#pragma unroll
  for (int ta = C::SA - 1; ta >= 0; --ta) {
    const int tb0 = C::tbmin(ta), np = C::np(ta), l0 = C::lev0(ta);
    const uint64_t adesc = tc::desc_from_lo(a_lo + (uint32_t)(ta * (C::A_PLANE >> 4)));
    if (!FIRST || l0 >= init_lo) {
      tc::mma_i8(d_tmem + (uint32_t)(l0 * C::NT), adesc, tc::desc_from_lo(b_lo + (uint32_t)(tb0 * (C::B_PLANE >> 4))),
                 tc::idesc_i8(np * C::NT), 1u);
    } else {
      const int fresh = (init_lo - l0 < np) ? init_lo - l0 : np;      // levels l0 .. l0 + fresh - 1 are new
      tc::mma_i8(d_tmem + (uint32_t)(l0 * C::NT), adesc, tc::desc_from_lo(b_lo + (uint32_t)(tb0 * (C::B_PLANE >> 4))),
                 tc::idesc_i8(fresh * C::NT), 0u);
      if (fresh < np)
        tc::mma_i8(d_tmem + (uint32_t)((l0 + fresh) * C::NT), adesc,
                   tc::desc_from_lo(b_lo + (uint32_t)((tb0 + fresh) * (C::B_PLANE >> 4))),
                   tc::idesc_i8((np - fresh) * C::NT), 1u);
      init_lo = l0;
    }
  }
}

template <class SCH, int EPI, int DP, int S2>
__global__ void __launch_bounds__(Cfg<SCH, DP>::NTHREADS, 1) split_gemm_kernel(const GemmParams P) {
  using C = Cfg<SCH, DP>;
  constexpr int NT = C::NT, NL = C::NL, EPI_THREADS = C::EPI_THREADS, PART_SPLIT = C::PART_SPLIT;
  extern __shared__ uint8_t smem_raw[];
  // head: [0,256) barriers + tmem slot, then two buffers of per-column scale pairs, then the DVAR training-input
  // tile; stages start at the next 512-byte boundary
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
  uint64_t* full = bars;
  uint64_t* empty = bars + C::STAGES;
  uint64_t* tfull = bars + 2 * C::STAGES;
  uint64_t* tempty = tfull + C::NBUF;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + C::NBUF);
  double2* s_cs = reinterpret_cast<double2*>(smem_raw + C::CS_OFF);   // [2][NT] {256 cs, 256 cs vq}
  double* s_xb = reinterpret_cast<double*>(smem_raw + C::XB_OFF);     // [NT][DP]
  const uint32_t raw_addr = tc::smem_u32(smem_raw);
  const uint32_t stage_off = ((raw_addr + C::HEAD + 511u) & ~511u) - raw_addr;
  uint8_t* sA = smem_raw + stage_off;
  uint8_t* sB = sA + C::STAGES * C::A_STAGE;

  // warp index through a shuffle: provably warp-uniform, so the role branches below are uniform branches and the
  // MMA warp's loop state / descriptors stay on the uniform datapath
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < C::STAGES; ++s) {
      tc::mbar_init(&full[s], 1);
      tc::mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < C::NBUF; ++b) {
      tc::mbar_init(&tfull[b], 1);
      tc::mbar_init(&tempty[b], EPI_THREADS);
    }
    tc::fence_barrier_init();
  }
  if (warp == 1) tc::tmem_alloc<C::TMEM_COLS>(tmem_slot);
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================================ producer =================================================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      TileWalk<NT, EPI == EPI_DACQ> walk;
      walk.start(P);
      TileInfo ti;
      while (walk.next(P, ti)) {
        const uint8_t* gA = P.A + ((size_t)(ti.j * P.RT + ti.rt) * P.KCH) * C::A_STAGE;
        const uint8_t* gB = P.B + ((size_t)((P.h * P.m + ti.j) * P.nct + ti.ct) * P.KCH) * C::B_STAGE;
        if (EPI == EPI_DVAR || EPI == EPI_DACQ) {
          // the epilogue of this tile (one tile later in time) reads 128 G* values of each of its NT columns:
          // pull those 1 KB rows into L2 now so its loads do not pay HBM latency
          const double* g0 = P.GsT + (size_t)ti.j * P.n16 * P.Nc + (size_t)ti.rt * TM;
          const int bend = min(ti.ct * NT + NT, P.n);
          for (int b = ti.ct * NT; b < bend; ++b) tc::prefetch_l2(g0 + (size_t)b * P.Nc, TM * 8);
        }
        for (int kc = ti.kb; kc < ti.ke; ++kc) {
          tc::mbar_wait(&empty[stage], phase ^ 1u);
          tc::mbar_arrive_expect_tx(&full[stage], C::STAGE);
          tc::bulk_g2s(sA + stage * C::A_STAGE, gA + (size_t)kc * C::A_STAGE, C::A_STAGE, &full[stage]);
          tc::bulk_g2s(sB + stage * C::B_STAGE, gB + (size_t)kc * C::B_STAGE, C::B_STAGE, &full[stage]);
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer (whole warp, one elected lane issues) ==========
    const uint32_t a_lo0 = tc::desc_lo_sw64(tc::smem_u32(sA)), b_lo0 = tc::desc_lo_sw64(tc::smem_u32(sB));
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    TileWalk<NT, EPI == EPI_DACQ> walk;
    walk.start(P);
    TileInfo ti;
    while (walk.next(P, ti)) {
      const int buf = it % C::NBUF;
      const uint32_t use = (uint32_t)(it / C::NBUF);
      ++it;
      tc::mbar_wait(&tempty[buf], (use & 1u) ^ 1u);          // epilogue has drained this accumulator buffer
      tc::fence_after_sync();
      const uint32_t d_tmem = tmem_base + (uint32_t)(buf * C::ACC_COLS);
      bool first = true;
      for (int kc = ti.kb; kc < ti.ke; ++kc) {
        tc::mbar_wait(&full[stage], phase);
        tc::fence_after_sync();
        const uint32_t a_lo = a_lo0 + (uint32_t)(stage * (C::A_STAGE >> 4));
        const uint32_t b_lo = b_lo0 + (uint32_t)(stage * (C::B_STAGE >> 4));
#pragma unroll
        for (int ks = 0; ks < KC / 32; ++ks) {
          const int kstep = kc * (KC / 32) + ks;            // K steps wholly outside the triangle multiply zeros: skip
          if (kstep < ti.sb || kstep >= ti.se) continue;
          if (first) {
            if (tc::elect_one()) issue_kstep<C, true>(a_lo + ks * 2, b_lo + ks * 2, d_tmem);
          } else {
            if (tc::elect_one()) issue_kstep<C, false>(a_lo + ks * 2, b_lo + ks * 2, d_tmem);
          }
          first = false;
        }
        if (tc::elect_one()) tc::mma_commit(&empty[stage]);  // stage reusable once these MMAs have read it
        __syncwarp();
        if (++stage == C::STAGES) {
          stage = 0;
          phase ^= 1u;
        }
      }
      if (tc::elect_one()) tc::mma_commit(&tfull[buf]);      // accumulators of this tile complete
      __syncwarp();
    }
  } else {
    // ================================ epilogue (EPI_WARPS warps) ===============================
    const int et = threadIdx.x - 64;
    const int lg = warp & 3;                                    // TMEM lane group this warp may access
    const int hw = (warp - 2) >> 2;                             // which of the lane group's warps: owns column groups hw, hw+PART_SPLIT, ..
    const int row = lg * 32 + lane;
    int it = 0;
    // per-tile constants (column scales, scaled training inputs of the column tile) are fetched one tile AHEAD into
    // registers and parked in shared memory at the top of the tile, so their global-load latency is never exposed
    constexpr int DPA0 = DP > 0 ? DP : 1;
    constexpr bool GRADEPI = (EPI == EPI_DVAR || EPI == EPI_DACQ);
    constexpr int XPT = GRADEPI ? (NT * DPA0 + EPI_THREADS - 1) / EPI_THREADS : 1;
    double pre_cs = 0.0, pre_vq = 0.0, pre_xb[XPT];
    auto prefetch_tile_consts = [&](const TileInfo& tn) {
      const int hjn = P.h * P.m + tn.j;
      if (EPI == EPI_DACQ && et < NT) {
        // alpha_b / (256 cs2_b): the mean-gradient weight in the units of the merged, unscaled accumulator
        const int b = tn.ct * NT + et;
        pre_cs = (b < P.n) ? __ldg(P.alpha + (size_t)hjn * P.n_pad + b) / (256.0 * __ldg(P.cs + (size_t)hjn * P.nct * NT + b)) : 0.0;
      }
      if (!GRADEPI) {
        if (et < NT) pre_cs = __ldg(P.cs + (size_t)hjn * P.nct * NT + tn.ct * NT + et);
        if (EPI == EPI_VAR) pre_vq = __ldg(P.vq + hjn);
      } else {
        const double* Xb = P.Xs + (size_t)hjn * P.n_pad * P.d;
#pragma unroll
        for (int x = 0; x < XPT; ++x) {
          const int idx = et + x * EPI_THREADS;
          const int cc = idx / DPA0, q = idx - cc * DPA0;
          const int b = tn.ct * NT + cc;
          pre_xb[x] = (idx < NT * DPA0 && q < P.d && b < P.n) ? __ldg(Xb + (size_t)b * P.d + q) : 0.0;
        }
      }
    };
    TileWalk<NT, EPI == EPI_DACQ> walk;
    walk.start(P);
    TileInfo ti, tnext;
    bool have = walk.next(P, tnext);
    if (have) prefetch_tile_consts(tnext);
    // reductions over the column tiles of a unit live in registers
    constexpr int DPA = DP > 0 ? DP : 2;
    double sumsq = 0.0, s0 = 0.0, acc[DPA];
    double wa_i = 0.0, wb2_i = 0.0;                             // DACQ: this candidate's gradient weights for the unit's output
    while (have) {
      ti = tnext;
      have = walk.next(P, tnext);
      const int buf = it % C::NBUF;
      const uint32_t use = (uint32_t)(it / C::NBUF);
      const int col0 = ti.ct * NT;
      if (ti.first) {
        sumsq = 0.0;
        s0 = 0.0;
#pragma unroll
        for (int q = 0; q < DPA; ++q) acc[q] = 0.0;
      }
      // per-tile constants into shared memory.  VAR / RAW: {scale, scale * quantiser} pairs, double buffered (buffer
      // it & 1), so ONE barrier per tile suffices: a warp can be at most one tile ahead of the slowest one.
      // DVAR: the training-input tile is single buffered (it would cost a pipeline stage): two barriers.
      const double2* cs_t = s_cs + (it & 1) * NT;
      if (!GRADEPI) {
        if (et < NT) s_cs[(it & 1) * NT + et] = make_double2(pre_cs * (EPI == EPI_RAW ? 1.0 : 256.0), pre_cs * 256.0 * pre_vq);
      } else {
        if (EPI == EPI_DACQ && et < NT) s_cs[(it & 1) * NT + et] = make_double2(pre_cs, 0.0);    // double buffered
        tc::named_bar_sync(1, EPI_THREADS);                     // previous tile's readers of s_xb are done
#pragma unroll
        for (int x = 0; x < XPT; ++x) {
          const int idx = et + x * EPI_THREADS;
          if (idx < NT * DPA0) s_xb[idx] = pre_xb[x];
        }
      }
      tc::named_bar_sync(1, EPI_THREADS);
      ++it;
      if (have) prefetch_tile_consts(tnext);
      const int64_t i = (int64_t)ti.rt * TM + row;              // chunk-local candidate

      // per-tile thread state
      // columns per TMEM load group.  VAR: 16, so a thread's digits of one plane are ONE 16-byte piece of the swizzled
      // 64-byte row -- half as many L2 write requests as 8-byte stores (knock-out: the V-digit stores cost 22 of the
      // first contraction's 121 ms per 1M-candidate step as 8-byte pieces, profiles/r2_knockouts.md)
      constexpr int CGW = (EPI == EPI_VAR) ? 16 : (GRADEPI ? 4 : 8);
      static_assert(NT % (CGW * PART_SPLIT) == 0, "column groups must divide evenly over the warps");
      constexpr int NCG = NT / CGW;
      constexpr int NGW = NCG / PART_SPLIT;                     // column groups per warp
      double gv[CGW];
      // G* of this warp's column groups: rows b of GsT, one candidate per lane (coalesced).  Columns b >= n of the last
      // tile carry an exactly zero Wt (zero factor planes), so their G* is read from row n-1 instead of being masked.
      // (row index and stride are 32-bit: one widening multiply per address instead of a 64 x 64 one -- the address
      // arithmetic was 9 of the gradient epilogue's 48 instructions per element)
      const double* Gcol = nullptr;
      const uint32_t gstride = (uint32_t)P.Nc;                  // candidates per chunk: < 2^31
      const bool tile_full = (col0 + NT <= P.n);
      if (EPI == EPI_DACQ && ti.first) {                         // once per unit, not per column tile: the loads' latency
        wa_i = __ldg(P.wa + (size_t)ti.j * P.Nc + i);            // sat exposed at the top of every tile (13 % of the
        wb2_i = -2.0 * __ldg(P.wb + (size_t)ti.j * P.Nc + i);    // epilogue warps' samples in ncu)
      }
      if (GRADEPI) {
        Gcol = P.GsT + (size_t)ti.j * P.n16 * P.Nc + i;
#pragma unroll
        for (int e = 0; e < CGW; ++e) {                      // first column group: in flight while the MMAs finish
          const int b = col0 + hw * CGW + e;
          gv[e] = __ldg(Gcol + (uint64_t)(uint32_t)(tile_full ? b : min(b, P.n - 1)) * gstride);
        }
      }

      tc::mbar_wait(&tfull[buf], use & 1u);
      tc::fence_after_sync();
      const uint32_t taddr = tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(buf * C::ACC_COLS);

      // The levels of the NEXT column group are requested from tensor memory before the current group is processed (two
      // register buffers), so the TMEM round trip overlaps the fp64 work.  The gradient epilogues, whose 2 d + 2
      // accumulators leave fewer registers, do the same with 4-column groups (two buffers of NL x 4 words = the one
      // buffer of NL x 8 they had: the exposed TMEM latency was 12 % of their samples in ncu).
      uint32_t c[2][NL][CGW];
#pragma unroll
      for (int lb = 0; lb < NL; ++lb) tc::tmem_ldw<CGW>(taddr + (uint32_t)(lb * NT + hw * CGW), c[0][lb]);
#pragma unroll
      for (int gi = 0; gi < NGW; ++gi) {
        const int cg = hw + gi * PART_SPLIT;
        tc::tmem_ld_wait();
        if (gi + 1 < NGW) {
#pragma unroll
          for (int lb = 0; lb < NL; ++lb)
            tc::tmem_ldw<CGW>(taddr + (uint32_t)(lb * NT + (cg + PART_SPLIT) * CGW), c[(gi + 1) & 1][lb]);
        }
        const uint32_t (&cc)[NL][CGW] = c[gi & 1];
        uint32_t vec[S2][CGW / 4];
        unsigned long long dgv[CGW];
#pragma unroll
        for (int e = 0; e < CGW; ++e) {
          if (EPI == EPI_RAW) {
            const double v = levels_to_f64<NL, CGW>(cc, e) * cs_t[cg * CGW + e].x;
            const int col = col0 + cg * CGW + e;
            const size_t grow = (size_t)(ti.j * P.RT + ti.rt) * TM + row;
            if (col < P.ldo) P.raw_out[grow * P.ldo + col] = v * P.raw_rs[grow];
          } else if (EPI == EPI_VAR) {
            const double y = levels_to_f64_merged<NL, CGW>(cc, e);    // V / (256 cs)
            const double2 sc = cs_t[cg * CGW + e];
            const double v = y * sc.x;
            sumsq = fma(v, v, sumsq);
            // digits of rint(V vq): one fused multiply-add onto the 1.5 * 2^52 rounding constant
            // (the digit bias rides in the rounding constant -- exact, both are integers below 2^53 -- and the bias is
            // removed by one XOR per transposed word below: balanced_digits' 64-bit add + XOR per element are gone)
            dgv[e] = (unsigned long long)__double_as_longlong(fma(y, sc.y, 6755399441055744.0 + (double)digit_bias<S2>()));
          } else {
            // the column scale (and the factor 256 of the merged Horner) is folded into G* by the K* kernel
            const double y = levels_to_f64_merged<NL, CGW>(cc, e);
            const double w = (EPI == EPI_DACQ) ? fma(wb2_i, y, wa_i * cs_t[cg * CGW + e].x) * gv[e] : y * gv[e];
            if (gi + 1 < NGW) {                                // refill the slot with this warp's next column group's G*
              const int bn = col0 + (cg + PART_SPLIT) * CGW + e;
              gv[e] = __ldg(Gcol + (uint64_t)(uint32_t)(tile_full ? bn : min(bn, P.n - 1)) * gstride);
            }
            s0 += w;
            const double2* xb2 = reinterpret_cast<const double2*>(s_xb + (cg * CGW + e) * DPA);
#pragma unroll
            for (int q2 = 0; q2 < DPA / 2; ++q2) {
              const double2 x2 = xb2[q2];
              acc[2 * q2] = fma(w, x2.x, acc[2 * q2]);
              acc[2 * q2 + 1] = fma(w, x2.y, acc[2 * q2 + 1]);
            }
          }
        }
        if (EPI == EPI_VAR && P.A2 != nullptr) {
#pragma unroll
          for (int w = 0; w < CGW / 4; ++w) {                    // byte transpose: digit t of 4 columns -> one word
            const unsigned long long four[4] = {dgv[4 * w], dgv[4 * w + 1], dgv[4 * w + 2], dgv[4 * w + 3]};
            uint32_t o[S2];
            digits_transpose4<S2>(four, o);
#pragma unroll
            for (int tt = 0; tt < S2; ++tt) vec[tt][w] = o[tt] ^ 0x80808080u;
          }
          const int k = col0 + cg * CGW;
          if (k < P.KCH * KC) {
            const int kc = k >> 6;
            uint8_t* dst = P.A2 + (((size_t)(ti.j * P.RT + ti.rt) * P.KCH + kc) * S2) * C::A_PLANE + sw64(row, k & 63);
#pragma unroll
            for (int tt = 0; tt < S2; ++tt) {
              if (CGW == 16)
                *reinterpret_cast<uint4*>(dst + (size_t)tt * C::A_PLANE) = make_uint4(vec[tt][0], vec[tt][1], vec[tt][2], vec[tt][3]);
              else
                *reinterpret_cast<uint2*>(dst + (size_t)tt * C::A_PLANE) = make_uint2(vec[tt][0], vec[tt][1]);
            }
          }
        }
      }
      tc::fence_before_sync();
      tc::mbar_arrive(&tempty[buf]);                            // accumulator buffer may be overwritten

      // one partial per (unit part, warp of the lane group): summed in fixed order by finalize_kernel
      const size_t pidx = ((size_t)ti.j * P.np + ti.p) * PART_SPLIT + hw;
      if (EPI == EPI_VAR && ti.last) P.part_var[pidx * P.Nc + i] = sumsq;
      if (GRADEPI && ti.last) {
        // xs_iq * S0 - ACC_q is formed by finalize_kernel (one division per candidate instead of one per tile)
        P.part_s0[pidx * P.Nc + i] = s0;
        double* out = P.part_dvar + (pidx * P.Nc + i) * P.d;
#pragma unroll
        for (int q = 0; q < DPA; ++q)
          if (q < P.d) out[q] = acc[q];
      }
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc::fence_after_sync();
    tc::tmem_dealloc<C::TMEM_COLS>(tmem_base);
  }
}

// ---- digit-plane packing of a dense fp64 matrix ------------------------------------------------------------------
// element (r, k) of matrix `mat`: src[mat*mat_stride + r*sr + k*sk], zero outside r < R, k < K.
__global__ void row_exp_kernel(const double* __restrict__ src, int64_t mat_stride, int64_t sr, int64_t sk, int R, int K,
                               int Rpad, int* __restrict__ exps, double* __restrict__ cs,
                               const int* __restrict__ extra, int base) {
  const int mat = blockIdx.y;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= Rpad) return;
  double amax = 0.0;
  if (row < R)
    for (int k = lane; k < K; k += 32) amax = fmax(amax, fabs(src[mat * mat_stride + row * sr + k * sk]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) amax = fmax(amax, __shfl_xor_sync(0xffffffffu, amax, o));
  if (lane == 0) {
    int e = 0;
    if (amax > 0.0) frexp(amax * 1.02, &e);
    exps[(size_t)mat * Rpad + row] = e;
    if (cs) cs[(size_t)mat * Rpad + row] = ldexp(1.0, e + (extra ? extra[mat] : 0) + base);
  }
}

template <int S>
__global__ void pack_digits_kernel(const double* __restrict__ src, int64_t mat_stride, int64_t sr, int64_t sk, int R,
                                   int K, const int* __restrict__ exps, int Rpad, int TR, int ntile, int KCH,
                                   uint8_t* __restrict__ out) {
  const int kc = blockIdx.x, tile = blockIdx.y, mat = blockIdx.z;
  uint8_t* obase = out + (((size_t)(mat * ntile + tile) * KCH + kc) * S) * TR * KC;
  for (int idx = threadIdx.x; idx < TR * 4; idx += blockDim.x) {
    int r, piece;
    if (sk == 1) {
      r = idx >> 2;
      piece = idx & 3;
    } else {
      r = idx % TR;
      piece = idx / TR;
    }
    const int row = tile * TR + r;
    const int e = exps[(size_t)mat * Rpad + row];
    const double q = ldexp(1.0, 8 * S - 2 - e);
    uint32_t vec[S][4];
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      unsigned long long four[4];
#pragma unroll
      for (int e4 = 0; e4 < 4; ++e4) {
        const int k = kc * KC + piece * 16 + 4 * w + e4;
        const double x = (row < R && k < K) ? src[mat * mat_stride + row * sr + k * sk] : 0.0;
        four[e4] = balanced_digits_of<S>(x * q);
      }
      uint32_t o[S];
      digits_transpose4<S>(four, o);
#pragma unroll
      for (int tt = 0; tt < S; ++tt) vec[tt][w] = o[tt];
    }
#pragma unroll
    for (int tt = 0; tt < S; ++tt)
      *reinterpret_cast<uint4*>(obase + (size_t)tt * TR * KC + sw64(r, piece * 16)) =
          make_uint4(vec[tt][0], vec[tt][1], vec[tt][2], vec[tt][3]);
  }
}

__global__ void absmax_kernel(const double* __restrict__ src, size_t count, double* __restrict__ out) {
  double a = 0.0;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < count; idx += (size_t)gridDim.x * blockDim.x)
    a = fmax(a, fabs(src[idx]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a = fmax(a, __shfl_xor_sync(0xffffffffu, a, o));
  if ((threadIdx.x & 31) == 0 && a > 0.0)
    atomicMax(reinterpret_cast<unsigned long long*>(out), (unsigned long long)__double_as_longlong(a));
}

template <int S>
static int pack_t(const double* src, int64_t mat_stride, int64_t sr, int64_t sk, int R, int K, const int* exps, int Rpad,
                  int TR, int ntile, int KCH, int mats, uint8_t* out, cudaStream_t st) {
  dim3 grid((unsigned)KCH, (unsigned)ntile, (unsigned)mats);
  pack_digits_kernel<S><<<grid, 256, 0, st>>>(src, mat_stride, sr, sk, R, K, exps, Rpad, TR, ntile, KCH, out);
  BOCF_LAUNCH_OK("pack_digits_kernel");
  return 0;
}
static int pack_digits(int S, const double* src, int64_t mat_stride, int64_t sr, int64_t sk, int R, int K,
                       const int* exps, int Rpad, int TR, int ntile, int KCH, int mats, uint8_t* out, cudaStream_t st) {
  switch (S) {
    case 3: return pack_t<3>(src, mat_stride, sr, sk, R, K, exps, Rpad, TR, ntile, KCH, mats, out, st);
    case 4: return pack_t<4>(src, mat_stride, sr, sk, R, K, exps, Rpad, TR, ntile, KCH, mats, out, st);
    case 5: return pack_t<5>(src, mat_stride, sr, sk, R, K, exps, Rpad, TR, ntile, KCH, mats, out, st);
    case 6: return pack_t<6>(src, mat_stride, sr, sk, R, K, exps, Rpad, TR, ntile, KCH, mats, out, st);
  }
  set_error("split contraction supports 3..6 digit planes");
  return BOCF_ERR_INVALID;
}
static int row_exps(const double* src, int64_t mat_stride, int64_t sr, int64_t sk, int R, int K, int Rpad, int mats,
                    int* exps, double* cs, const int* extra, int base, cudaStream_t st) {
  dim3 grid((unsigned)ceil_div(Rpad, 8), (unsigned)mats);
  row_exp_kernel<<<grid, 256, 0, st>>>(src, mat_stride, sr, sk, R, K, Rpad, exps, cs, extra, base);
  BOCF_LAUNCH_OK("row_exp_kernel");
  return 0;
}

template <class SCH, int EPI, int DP, int S2>
static int launch_k(const GemmParams& P, cudaStream_t st) {
  using C = Cfg<SCH, DP>;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  static bool attr_done[64] = {false};          // per device: function attributes belong to the device's context
  if (dev >= 0 && dev < 64 && !attr_done[dev]) {
    BOCF_CUDA_OK(cudaFuncSetAttribute(split_gemm_kernel<SCH, EPI, DP, S2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      C::SMEM_BYTES));
    attr_done[dev] = true;
  }
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int units = P.m * P.RTv * P.np;           // scheduling entities
  const int grid = units < sms ? units : sms;
  split_gemm_kernel<SCH, EPI, DP, S2><<<grid, C::NTHREADS, C::SMEM_BYTES, st>>>(P);
  BOCF_LAUNCH_OK("split_gemm_kernel");
  return 0;
}

static int bad_scheme() {
  set_error("split contraction: unsupported digit-pair scheme (331, 442, 554, 665)");
  return BOCF_ERR_INVALID;
}
static int launch_raw(int sch, const GemmParams& P, cudaStream_t st) {
  switch (sch) {
    case 331: return launch_k<P331, EPI_RAW, 0, 3>(P, st);
    case 442: return launch_k<P442, EPI_RAW, 0, 4>(P, st);
    case 554: return launch_k<P554, EPI_RAW, 0, 5>(P, st);
    case 665: return launch_k<P665, EPI_RAW, 0, 6>(P, st);
  }
  return bad_scheme();
}
// first contraction with scheme `sch`, re-splitting V into the s2 digit planes the second contraction's scheme reads
static int launch_var(int sch, int s2, const GemmParams& P, cudaStream_t st) {
  switch (sch * 10 + s2) {
    case 3313: return launch_k<P331, EPI_VAR, 0, 3>(P, st);
    case 4423: return launch_k<P442, EPI_VAR, 0, 3>(P, st);
    case 4424: return launch_k<P442, EPI_VAR, 0, 4>(P, st);
    case 5544: return launch_k<P554, EPI_VAR, 0, 4>(P, st);
    case 5545: return launch_k<P554, EPI_VAR, 0, 5>(P, st);
    case 6655: return launch_k<P665, EPI_VAR, 0, 5>(P, st);
    case 6656: return launch_k<P665, EPI_VAR, 0, 6>(P, st);
  }
  return bad_scheme();
}
// second contraction (EPI_DVAR or EPI_DACQ) with scheme `sch` for d input dimensions
template <int EPI, int DP>
static int launch_grad_d(int sch, const GemmParams& P, cudaStream_t st) {
  switch (sch) {
    case 331: return launch_k<P331, EPI, DP, 3>(P, st);
    case 442: return launch_k<P442, EPI, DP, 4>(P, st);
    case 554: return launch_k<P554, EPI, DP, 5>(P, st);
    case 665: return launch_k<P665, EPI, DP, 6>(P, st);
  }
  return bad_scheme();
}
template <int EPI>
static int launch_grad(int sch, int d, const GemmParams& P, cudaStream_t st) {
  if (d <= 4) return launch_grad_d<EPI, 4>(sch, P, st);
  if (d <= 6) return launch_grad_d<EPI, 6>(sch, P, st);
  if (d <= 8) return launch_grad_d<EPI, 8>(sch, P, st);
  if (d <= 10) return launch_grad_d<EPI, 10>(sch, P, st);
  if (d <= 12) return launch_grad_d<EPI, 12>(sch, P, st);
  return launch_grad_d<EPI, 16>(sch, P, st);
}

}  // namespace sg

// scheme of a symmetric "N digit planes" request (bocf_model_set_precision slices = 3..6)
int split_scheme_for_slices(int S) { return S == 3 ? 331 : S == 4 ? 442 : S == 5 ? 554 : S == 6 ? 665 : 0; }
int split_scheme_pairs(int sch) {
  sg::SchemeInfo si;
  return sg::scheme_info(sch, &si) ? si.pairs : 0;
}
// parts per candidate tile for a chunk of Nc candidates (Nc <= 0: what a large chunk gets -- the sizing figure; small
// chunks may use more parts, their scratch is sized exactly: chunk_bytes_per_candidate(M, grad, Nc))
int split_parts(const bocf_model* M, int64_t Nc) {
  int dev = 0, sms = 148, l2 = 126 << 20;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, dev);
  const int64_t a_tile = (int64_t)(M->S > M->S2 ? M->S : M->S2) * sg::TM * sg::KC * M->KCH;
  if (Nc <= 0) return sg::parts_for(sms, sms, a_tile, l2);               // what many units get
  return sg::parts_for((int)(M->m * (Nc / sg::TM)), sms, a_tile, l2);
}
int split_partials_var(const bocf_model* M, int64_t Nc) {      // partial sums per candidate and output written by the epilogues
  sg::SchemeInfo si;
  sg::scheme_info(M->sch1, &si);
  return si.EW / 4 * split_parts(M, Nc);
}
int split_partials_dvar(const bocf_model* M, int64_t Nc) {
  sg::SchemeInfo si;
  sg::scheme_info(M->sch2, &si);
  return si.EW / 4 * split_parts(M, Nc);
}

static void free_split(bocf_model* M) {
  auto fr = [](auto*& p) {
    if (p) cudaFree(p);
    p = nullptr;
  };
  fr(M->B1);
  fr(M->B2);
  fr(M->cs1);
  fr(M->cs2);
  fr(M->aq);
  fr(M->vq);
  M->split_ready = false;
}
void split_release(bocf_model* M) { free_split(M); }

// Largest |Linv| entry over all (h, j): drives the automatic choice of the digit-pair schemes.
int split_linv_absmax(bocf_model* M, double* out_host, cudaStream_t st) {
  double* d = nullptr;
  BOCF_CUDA_OK(cudaMalloc(&d, sizeof(double)));
  BOCF_CUDA_OK(cudaMemsetAsync(d, 0, sizeof(double), st));
  const size_t count = (size_t)M->H * M->m * M->n_pad * M->n_pad;
  sg::absmax_kernel<<<1024, 256, 0, st>>>(M->Linv, count, d);
  BOCF_LAUNCH_OK("absmax_kernel");
  BOCF_CUDA_OK(cudaMemcpyAsync(out_host, d, sizeof(double), cudaMemcpyDeviceToHost, st));
  BOCF_CUDA_OK(cudaStreamSynchronize(st));
  cudaFree(d);
  return 0;
}

// Digit planes of Linv for both contractions + all power-of-two scales.  Called after the factorisation.
// sch1: scheme of V = K* Linv^T;  sch2: scheme of Wt = V Linv (its SA is the number of planes V is re-split into).
int split_prepare(bocf_model* M, int sch1, int sch2, cudaStream_t st) {
  free_split(M);
  sg::SchemeInfo s1, s2;
  if (!sg::scheme_info(sch1, &s1) || !sg::scheme_info(sch2, &s2)) return sg::bad_scheme();
  const int Hm = M->H * M->m;
  M->sch1 = sch1;
  M->sch2 = sch2;
  M->S = s1.SA;
  M->S2 = s2.SA;
  M->NTs = s1.NT;
  M->NT2 = s2.NT;
  M->ncts = (int)ceil_div(M->n, s1.NT);
  M->nct2 = (int)ceil_div(M->n, s2.NT);
  M->KCH = (int)ceil_div(M->n, sg::KC);
  const int Rpad1 = M->ncts * s1.NT, Rpad2 = M->nct2 * s2.NT;
  const int Rmax = Rpad1 > Rpad2 ? Rpad1 : Rpad2;
  BOCF_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&M->B1), (size_t)Hm * M->ncts * M->KCH * s1.SB * s1.NT * sg::KC));
  BOCF_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&M->B2), (size_t)Hm * M->nct2 * M->KCH * s2.SB * s2.NT * sg::KC));
  BOCF_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&M->cs1), sizeof(double) * Hm * Rpad1));
  BOCF_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&M->cs2), sizeof(double) * Hm * Rpad2));
  BOCF_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&M->aq), sizeof(double) * Hm));
  BOCF_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&M->vq), sizeof(double) * Hm));
  int *exps = nullptr, *extra = nullptr;
  BOCF_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&exps), sizeof(int) * Hm * Rmax));
  BOCF_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&extra), sizeof(int) * 2 * Hm));
  // candidate-side scales: K* <= sigma_f^2 (stationary kernels), |V_k| <= sqrt(k**) = sigma_f
  std::vector<int> ex(2 * Hm);
  std::vector<double> aq(Hm), vq(Hm);
  for (int hj = 0; hj < Hm; ++hj) {
    int eA = 0, eV = 0;
    std::frexp(M->hyp_host[hj].variance * 1.02, &eA);
    std::frexp(std::sqrt(M->hyp_host[hj].variance) * 1.02, &eV);
    ex[hj] = eA;
    ex[Hm + hj] = eV;
    aq[hj] = std::ldexp(1.0, 8 * s1.SA - 2 - eA);
    vq[hj] = std::ldexp(1.0, 8 * s2.SA - 2 - eV);
  }
  BOCF_CUDA_OK(cudaMemcpyAsync(extra, ex.data(), sizeof(int) * 2 * Hm, cudaMemcpyHostToDevice, st));
  BOCF_CUDA_OK(cudaMemcpyAsync(M->aq, aq.data(), sizeof(double) * Hm, cudaMemcpyHostToDevice, st));
  BOCF_CUDA_OK(cudaMemcpyAsync(M->vq, vq.data(), sizeof(double) * Hm, cudaMemcpyHostToDevice, st));
  // output scale of a scheme: 2^(eA + eB) * 256^LMIN / (2^(8 SA - 2) 2^(8 SB - 2))
  const int base1 = -(8 * s1.SA - 2) - (8 * s1.SB - 2) + 8 * s1.LMIN;
  const int base2 = -(8 * s2.SA - 2) - (8 * s2.SB - 2) + 8 * s2.LMIN;
  const int64_t nn = (int64_t)M->n_pad * M->n_pad;
  int rc = 0;
  // first contraction: rows = factor row k, K = b      (element Linv[k][b])
  if (!rc) rc = sg::row_exps(M->Linv, nn, M->n_pad, 1, M->n, M->n, Rpad1, Hm, exps, M->cs1, extra, base1, st);
  if (!rc) rc = sg::pack_digits(s1.SB, M->Linv, nn, M->n_pad, 1, M->n, M->n, exps, Rpad1, s1.NT, M->ncts, M->KCH, Hm, M->B1, st);
  // second contraction: rows = factor column b, K = k  (element Linv[k][b])
  if (!rc) rc = sg::row_exps(M->Linv, nn, 1, M->n_pad, M->n, M->n, Rpad2, Hm, exps, M->cs2, extra + Hm, base2, st);
  if (!rc) rc = sg::pack_digits(s2.SB, M->Linv, nn, 1, M->n_pad, M->n, M->n, exps, Rpad2, s2.NT, M->nct2, M->KCH, Hm, M->B2, st);
  cudaError_t e = cudaStreamSynchronize(st);      // ex/aq/vq are host vectors going out of scope
  cudaFree(exps);
  cudaFree(extra);
  if (rc) return rc;
  if (e != cudaSuccess) {
    set_error(std::string("split_prepare: ") + cudaGetErrorString(e));
    return BOCF_ERR_CUDA;
  }
  M->split_ready = true;
  return 0;
}

uint64_t split_chunk_bytes_per_candidate(const bocf_model* M, bool grad, int64_t Nc) {
  uint64_t per = 0;
  per += (uint64_t)M->m * M->KCH * sg::KC * M->S;       // A1 digit planes of K*
  per += (uint64_t)M->m * split_partials_var(M, Nc) * 8; // part_var
  per += 2ull * M->m * 8;                               // mean, var
  if (grad) {
    per += (uint64_t)M->m * M->n16 * 8;                 // GsT
    per += (uint64_t)M->m * M->KCH * sg::KC * M->S2;    // A2 digit planes of V
    per += (uint64_t)M->m * split_partials_dvar(M, Nc) * (M->d + 1) * 8;  // part_dvar, part_s0
    per += 2ull * M->m * M->d * 8;                      // dmean, dvar
    per += 2ull * M->m * 8;                             // wa, wb (fused gradient path)
    per += (2ull * M->m * 4 + sg::TM - 1) / sg::TM;     // unit flags and unit list: one int each per (output, tile)
  }
  return per;
}

void split_carve_chunk(const bocf_model* M, void* base, int64_t Nc, bool grad, ChunkBuffers* cb) {
  uint8_t* p = reinterpret_cast<uint8_t*>(base);
  auto take = [&](uint64_t bytes) {
    uint8_t* r = p;
    p += round_up((int64_t)bytes, 1024);
    return r;
  };
  const uint64_t plane = (uint64_t)M->m * Nc * M->KCH * sg::KC;
  cb->Nc = Nc;
  cb->KsT = cb->V = nullptr;
  cb->A1 = take(plane * M->S);
  cb->part_var = reinterpret_cast<double*>(take((uint64_t)M->m * split_partials_var(M, Nc) * Nc * 8));
  cb->mean = reinterpret_cast<double*>(take((uint64_t)M->m * Nc * 8));
  cb->var = reinterpret_cast<double*>(take((uint64_t)M->m * Nc * 8));
  if (grad) {
    cb->GsT = reinterpret_cast<double*>(take((uint64_t)M->m * M->n16 * Nc * 8));
    cb->A2 = take(plane * M->S2);
    cb->part_dvar = reinterpret_cast<double*>(take((uint64_t)M->m * split_partials_dvar(M, Nc) * Nc * M->d * 8));
    cb->part_s0 = reinterpret_cast<double*>(take((uint64_t)M->m * split_partials_dvar(M, Nc) * Nc * 8));
    cb->dmean = reinterpret_cast<double*>(take((uint64_t)M->m * Nc * M->d * 8));
    cb->dvar = reinterpret_cast<double*>(take((uint64_t)M->m * Nc * M->d * 8));
    cb->wa = reinterpret_cast<double*>(take((uint64_t)M->m * Nc * 8));
    cb->wb = reinterpret_cast<double*>(take((uint64_t)M->m * Nc * 8));
    cb->unit_flags = reinterpret_cast<int*>(take((uint64_t)M->m * (Nc / sg::TM) * 4));
    cb->unit_list = reinterpret_cast<int*>(take((uint64_t)M->m * (Nc / sg::TM) * 4 + 4));
    cb->unit_count = cb->unit_list + M->m * (Nc / sg::TM);
  } else {
    cb->GsT = cb->part_dvar = cb->dmean = cb->dvar = nullptr;
    cb->A2 = nullptr;
  }
  cb->kpart = (kstar_ksplit(M, Nc) > 1) ? reinterpret_cast<double*>(take(kstar_part_bytes(M, Nc))) : nullptr;
}

static sg::GemmParams base_params(const bocf_model* M, int h, const ChunkBuffers& cb, int64_t Nvalid) {
  sg::GemmParams P;
  std::memset(&P, 0, sizeof(P));
  P.m = M->m;
  P.h = h;
  P.RT = (int)(cb.Nc / sg::TM);
  P.RTv = (Nvalid > 0 && Nvalid < cb.Nc) ? (int)ceil_div(Nvalid, sg::TM) : P.RT;
  P.Nvalid = Nvalid;
  P.KCH = M->KCH;
  P.n = M->n;
  P.Nc = cb.Nc;
  P.d = M->d;
  P.n16 = M->n16;
  P.n_pad = M->n_pad;
  P.hyp = M->hyp;
  P.np = split_parts(M, cb.Nc);
  return P;
}

int launch_split_var(bocf_model* M, int h, int64_t Nvalid, const ChunkBuffers& cb, bool need_dvar, cudaStream_t st) {
  sg::GemmParams P = base_params(M, h, cb, Nvalid);
  P.A = cb.A1;
  P.B = M->B1;
  P.cs = M->cs1;
  P.nct = M->ncts;
  P.tri = sg::TRI_K_LE_N;
  P.part_var = cb.part_var;
  P.A2 = need_dvar ? cb.A2 : nullptr;
  P.vq = M->vq;
  if (M->ncts < P.np)                      // parts without a column tile never write their partial
    BOCF_CUDA_OK(cudaMemsetAsync(cb.part_var, 0, sizeof(double) * M->m * split_partials_var(M, cb.Nc) * cb.Nc, st));
  ProfScope ps("split_var_kernel", st);
  return sg::launch_var(M->sch1, M->S2, P, st);
}

int launch_split_dvar(bocf_model* M, int h, const double* Xc, int64_t Nvalid, const ChunkBuffers& cb, bool fused_acq,
                      cudaStream_t st) {
  sg::GemmParams P = base_params(M, h, cb, Nvalid);
  P.A = cb.A2;
  P.B = M->B2;
  P.cs = M->cs2;
  P.nct = M->nct2;
  P.tri = sg::TRI_K_GE_N;
  P.part_dvar = cb.part_dvar;
  P.part_s0 = cb.part_s0;
  P.GsT = cb.GsT;
  P.Xc = Xc;
  P.Xs = M->Xs;
  if (fused_acq) {
    P.alpha = M->alpha;
    P.wa = cb.wa;
    P.wb = cb.wb;
    P.unit_list = cb.unit_list;
    P.unit_count = cb.unit_count;
  }
  if (M->nct2 < P.np) {
    BOCF_CUDA_OK(cudaMemsetAsync(cb.part_dvar, 0, sizeof(double) * M->m * split_partials_dvar(M, cb.Nc) * cb.Nc * M->d, st));
    BOCF_CUDA_OK(cudaMemsetAsync(cb.part_s0, 0, sizeof(double) * M->m * split_partials_dvar(M, cb.Nc) * cb.Nc, st));
  }
  ProfScope ps("split_dvar_kernel", st);
  return fused_acq ? sg::launch_grad<sg::EPI_DACQ>(M->sch2, M->d, P, st) : sg::launch_grad<sg::EPI_DVAR>(M->sch2, M->d, P, st);
}

// Test entry: out (R x N) = A (R x K) * B (N x K)^T through the digit-plane machinery.  All pointers [dev] fp64 row-major.
int split_debug_gemm(const double* A, const double* B, int R, int N, int K, int sch, int tri, double* out, cudaStream_t st) {
  sg::SchemeInfo si;
  if (!sg::scheme_info(sch, &si) || R < 1 || N < 1 || K < 1) {
    set_error("split_debug_gemm: invalid arguments");
    return BOCF_ERR_INVALID;
  }
  const int NT = si.NT;
  const int RT = (int)ceil_div(R, sg::TM), nct = (int)ceil_div(N, NT), KCH = (int)ceil_div(K, sg::KC);
  const int RpadA = RT * sg::TM, RpadB = nct * NT;
  uint8_t *pa = nullptr, *pb = nullptr;
  int *ea = nullptr, *eb = nullptr;
  double *rs = nullptr, *cs = nullptr, *tmp = nullptr;
  int rc = 0;
  do {
    if (cudaMalloc(reinterpret_cast<void**>(&pa), (size_t)RT * KCH * si.SA * sg::TM * sg::KC) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&pb), (size_t)nct * KCH * si.SB * NT * sg::KC) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&ea), sizeof(int) * RpadA) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&eb), sizeof(int) * RpadB) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&rs), sizeof(double) * RpadA) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&cs), sizeof(double) * RpadB) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&tmp), sizeof(double) * (size_t)RpadA * N) != cudaSuccess) {
      set_error("split_debug_gemm: out of device memory");
      rc = BOCF_ERR_CUDA;
      break;
    }
    const int base = -(8 * si.SA - 2) - (8 * si.SB - 2) + 8 * si.LMIN;
    if ((rc = sg::row_exps(A, 0, K, 1, R, K, RpadA, 1, ea, rs, nullptr, 0, st))) break;
    if ((rc = sg::row_exps(B, 0, K, 1, N, K, RpadB, 1, eb, cs, nullptr, base, st))) break;
    if ((rc = sg::pack_digits(si.SA, A, 0, K, 1, R, K, ea, RpadA, sg::TM, RT, KCH, 1, pa, st))) break;
    if ((rc = sg::pack_digits(si.SB, B, 0, K, 1, N, K, eb, RpadB, NT, nct, KCH, 1, pb, st))) break;
    sg::GemmParams P;
    std::memset(&P, 0, sizeof(P));
    P.A = pa;
    P.B = pb;
    P.cs = cs;
    P.m = 1;
    P.h = 0;
    P.np = 1;
    P.RT = RT;
    P.RTv = RT;
    P.nct = nct;
    P.KCH = KCH;
    P.n = K;
    P.tri = tri;
    P.Nc = RpadA;
    P.raw_out = tmp;
    P.raw_rs = rs;
    P.ldo = N;
    {
      ProfScope ps("split_raw_kernel", st);
      rc = sg::launch_raw(sch, P, st);
    }
    if (rc) break;
    if (cudaMemcpyAsync(out, tmp, sizeof(double) * (size_t)R * N, cudaMemcpyDeviceToDevice, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) {
      set_error(std::string("split_debug_gemm: ") + cudaGetErrorString(cudaGetLastError()));
      rc = BOCF_ERR_CUDA;
    }
  } while (0);
  cudaFree(pa);
  cudaFree(pb);
  cudaFree(ea);
  cudaFree(eb);
  cudaFree(rs);
  cudaFree(cs);
  cudaFree(tmp);
  return rc;
}

}  // namespace bocf
