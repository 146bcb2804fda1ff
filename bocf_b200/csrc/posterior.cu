// posterior.cu -- batched multi-output GP posterior at a chunk of candidates (north-star subsystems 1+2).
//
// For hyper-sample h and every output j, at Nc candidates (SURVEY.md 8a rows a9-a14):
//   kstar_kernel      K*  = K(x*, X)         stationary.py:104-166 / se.py:44-73      (CUDA cores + MUFU)
//                     mu  = K* alpha + ybar  posterior.py:299-305, gp.py:398-399
//                     dmu = gradients_X(alpha^T, x*, X)   gp.py:446, stationary.py:332-342, stationary_utils.c
//                     G*  = dK/dr / r        (weights for the variance gradient)
//   var_gemm_kernel   V   = K* Linv^T  (= L^-1 K(X,x*), the reference's dtrtrs route, posterior.py:312)
//                     var = k** - sum V^2 (+ noise), clipped 1e-10    posterior.py:313, gaussian.py:110, gpmodel.py:174
//   dvar_gemm_kernel  Wt  = V Linv     (= K* W^-1, gp.py:474)
//                     dvar = gradients_X(-2 Wt, x*, X)               gp.py:475
// The two contractions run on the fp64 tensor-core tile engine (DMMA.8x8x4, 256 x 64 tiles) and skip the
// zero blocks of the triangular factor; K*, G* and V live in a per-chunk HBM scratch, everything else
// (n x n factor, training inputs) is L2-resident and shared by all candidate tiles of one output.
#include <cstdlib>

#include "gemm_f64.cuh"
#include "kernfn.cuh"
#include "model.h"

namespace bocf {

using PT = gemm::TilePost;                 // 128 candidates x 64 factor columns, 128 threads, 2 CTAs / SM
constexpr int PT_MINBLOCKS = 2;
constexpr int64_t KSTAR_SPLIT_MAX = 1024;  // chunks up to this many candidates split the training points over blocks
constexpr int KSTAR_SPLIT = 8;

// K-split factor of the K* kernel for a chunk of Nc candidates (1 = none); also sizes the partial-sum scratch
int kstar_ksplit(const bocf_model* M, int64_t Nc) {
  if (Nc > KSTAR_SPLIT_MAX) return 1;
  const int blocks = (M->n16 + 127) / 128;
  return blocks < KSTAR_SPLIT ? (blocks < 1 ? 1 : blocks) : KSTAR_SPLIT;
}
constexpr int MI = PT::MI;                 // 8-row MMA tiles per warp (warp tile = 8*MI x 32)
constexpr int CT = PT::BM;                 // candidate tile
constexpr int NT = PT::BN;                 // column tile

// ===================================================================================================
// K*, mean, mean-gradient.  One thread per candidate, training points staged through shared memory.
// SPLIT: instead of the fp64 K* matrix, write the S balanced base-256 digit planes of round(K* 2^(8S-2-eA)) in the
// packed, 64-byte-swizzled tile layout the tcgen05 contraction streams (split_gemm.cu): plane t of K chunk kc of
// candidate tile rt holds, for row = candidate, the digits of 64 consecutive training points.
struct SplitOut {
  uint8_t* A1;
  const double* aq;    // [H*m] quantiser 2^(8S-2-eA)
  const double* gcs;   // [H*m][gcs_ld] power-of-two column scale of the second contraction, folded into G* here (exact)
  int gcs_ld;
  int KCH, S;
};

// SPL: 0 = fp64 K* output; 5 = exactly five digit planes (the common case, fewer registers); 6 = up to six (so.S);
//      -1 = no K* output at all: the mean-only pass that decides which candidates the acquisition sweep can skip (api.cu).
//      Every instantiation forms mu with the same per-pair arithmetic in the same order, so mu is bitwise the same.
// GRAD: 0 = value quantities only; 1 = also G* and the mean gradient; 2 = G* only -- the fused acquisition-gradient path
//       (api.cu) folds the mean-gradient contraction into the second contraction's epilogue, which saves the d + 2
//       fp64 operations per (candidate, training point) the mean gradient costs here.
template <int KIND, int DP, int GRAD, int SPL>
__global__ void __launch_bounds__(128, 1) kstar_kernel(const double* __restrict__ Xc, int64_t Nvalid, int64_t Nc, int d,
                                                    int n, int n16, int n_pad, int m, int h,
                                                    const OutHyp* __restrict__ hyp, const double* __restrict__ XsAll,
                                                    const double* __restrict__ xsqAll,
                                                    const double* __restrict__ alphaAll, double* __restrict__ KsT,
                                                    double* __restrict__ GsT, double* __restrict__ mean,
                                                    double* __restrict__ dmean, const SplitOut so, int j0) {
  // gridDim.z > 1: K-SPLIT for small batches.  One thread walks its candidate's training points serially -- ~120 us of
  // pure latency at n = 1000 however few candidates there are (the L-BFGS rounds of the acquisition optimiser evaluate
  // tens).  Block z then takes the 128-point blocks z, z + gridDim.z, ... and writes ADDITIVE partial sums of the mean
  // and its gradient (slab z of mean / dmean); kstar_reduce_kernel adds the slabs in fixed order.
  const int ks = (int)gridDim.z, kz = (int)blockIdx.z;
  if ((int64_t)blockIdx.x * 128 >= Nvalid) return;          // a tile of pure padding: nothing downstream reads it
  __shared__ double sX[128][DP];
  __shared__ double sxsq[128];
  __shared__ double salpha[128];
  __shared__ double sgcs[128];
  __shared__ double sexp[EXP_TAB_N];
  const int tid = threadIdx.x;
  // visible after the first __syncthreads of the tile loop; the output's signal variance rides in the table entries
  exp_table_fill(sexp, tid, hyp[h * m + j0 + blockIdx.y].variance);
  const int j = j0 + blockIdx.y;                 // this launch covers one run of outputs that share the kernel family
  const int hj = h * m + j;
  const int64_t i = (int64_t)blockIdx.x * 128 + tid;
  const OutHyp& hp = hyp[hj];

  // everything the kernel family multiplies the squared distance by (kernfn.cuh: KFast) is folded into the operands of
  // the distance itself:  q = SCALE r2 = SCALE (|x|^2 + |X_b|^2) + sum_q (-2 SCALE x_q) X_bq
  double xs[DP], xm2[DP];
  double xsq_i = 0.0;
#pragma unroll
  for (int q = 0; q < DP; ++q) {
    double v = 0.0;
    if (q < d && i < Nvalid) v = Xc[i * d + q] / hp.ls[q];
    xs[q] = v;
    xm2[q] = (-2.0 * KFast<KIND>::SCALE) * v;
    xsq_i += v * v;
  }
  xsq_i *= KFast<KIND>::SCALE;
  double mu = 0.0, wsum = 0.0;
  double gm[DP];       // sum_b w_b Xs_bq ;  dmean_q = (xs_q * sum_b w_b - gm_q) / l_q
#pragma unroll
  for (int q = 0; q < DP; ++q) gm[q] = 0.0;

  const double* Xs = XsAll + (int64_t)hj * n_pad * d;
  const double* xsq = xsqAll + (int64_t)hj * n_pad;
  const double* alpha = alphaAll + (int64_t)hj * n_pad;
  constexpr bool SPLIT = SPL > 0;
  constexpr bool GFOLD = SPLIT && GRAD == 2;
  double* Kout = (SPL == 0) ? KsT + (int64_t)j * n16 * Nc : nullptr;
  double* Gout = GRAD ? GsT + (int64_t)j * n16 * Nc : nullptr;
  // split mode: digit planes of this block's 128 candidates (row = tid) for output j
  constexpr int MAXS = SPLIT ? SPL : 1;
  uint32_t dv[MAXS][4];
  const double aq = SPLIT ? so.aq[hj] : 0.0;
  // rounding constant 1.5 * 2^52 plus the balanced-digit bias 0x80..80 (so.S bytes): both integers below 2^53, so the sum
  // is exact and the low bytes of the fused multiply-add's mantissa are digit + 128; the bias comes off with one XOR per
  // transposed word (a 64-bit add and a 64-bit XOR per training point before)
  const double magicb = SPLIT ? 6755399441055744.0 + (double)(0x808080808080ull >> (8 * (6 - so.S))) : 0.0;
  uint8_t* Aout = SPLIT ? so.A1 + ((size_t)((size_t)j * gridDim.x + blockIdx.x) * so.KCH) * so.S * (128 * 64) : nullptr;
  const uint32_t swz = (uint32_t)((tid >> 1) & 3);

  for (int b0 = kz * 128; b0 < n16; b0 += 128 * ks) {
    __syncthreads();
    for (int idx = tid; idx < 128 * DP; idx += 128) {
      int bb = idx / DP, q = idx - bb * DP;
      int b = b0 + bb;
      sX[bb][q] = (q < d && b < n) ? Xs[(int64_t)b * d + q] : 0.0;
    }
    {
      int b = b0 + tid;
      sxsq[tid] = (b < n) ? KFast<KIND>::SCALE * xsq[b] : 0.0;
      salpha[tid] = (b < n) ? alpha[b] : 0.0;
      // column scale of the second contraction times the 256 its epilogue's merged Horner leaves out (split_gemm.cu)
      // (and, when GFOLD, the constant factor of (dK/dr)/r that kern_eval_fast leaves out)
      if (SPL > 0) sgcs[tid] = (b < n) ? (GFOLD ? 256.0 * KFast<KIND>::GFAC : 256.0) * so.gcs[(size_t)hj * so.gcs_ld + b] : 0.0;
    }
    __syncthreads();
    const int bmax = min(128, n16 - b0);
    // 16 (split: one 16-byte piece of a digit-plane row) or 4 training points per trip, evaluated branch-free so the
    // independent chains interleave; padded points b >= n are evaluated like the others and masked at the end
    constexpr int UNR = (SPL != 0) ? 16 : 4;
    for (int bb0 = 0; bb0 < bmax; bb0 += UNR) {
      unsigned long long dg4[4];
#pragma unroll
      for (int e = 0; e < UNR; ++e) {
        const int bb = bb0 + e;
        const int b = b0 + bb;
        double kv, gv;
        {
          double r2;
          if (KIND == BOCF_KERN_SE) {
            double r2a = 0.0, r2b = 0.0;
#pragma unroll
            for (int q = 0; q < DP; q += 2) {
              const double d0 = xs[q] - sX[bb][q];
              r2a = fma(d0, d0, r2a);
              if (q + 1 < DP) {
                const double d1 = xs[q + 1] - sX[bb][q + 1];
                r2b = fma(d1, d1, r2b);
              }
            }
            r2 = KFast<KIND>::SCALE * (r2a + r2b);
          } else {
            // two chains (half the dependent-DFMA depth), seeded with the two squared norms: d DFMA + 1 DADD
            double dot0 = xsq_i, dot1 = sxsq[bb];
#pragma unroll
            for (int q = 0; q < DP; q += 2) {
              dot0 = fma(xm2[q], sX[bb][q], dot0);
              if (q + 1 < DP) dot1 = fma(xm2[q + 1], sX[bb][q + 1], dot1);
            }
            r2 = dot0 + dot1;
          }
          // clip at 0 (stationary.py:153) and the cap that replaces exp's clamp, on the integer pipe
          bool nz;
          const double qc = clamp_q<KIND>(r2, nz);
          kern_eval_fast<KIND, (GRAD != 0)>(qc, nz, kv, gv, sexp);
          if (GRAD && !GFOLD) gv *= KFast<KIND>::GFAC;
          // padded points b >= n need no mask: their alpha, column scale and factor rows / columns are zero, so whatever
          // finite K*, G* they produce is multiplied by an exact zero downstream (mean, both contractions, epilogues)
          const double a = salpha[bb];
          mu += kv * a;
          if (GRAD == 1) {
            const double w = gv * a;
            wsum += w;
#pragma unroll
            for (int q = 0; q < DP; ++q) gm[q] = fma(w, sX[bb][q], gm[q]);
          }
        }
        if (GRAD) Gout[(int64_t)b * Nc + i] = SPLIT ? gv * sgcs[bb] : gv;
        if (SPL == 0) {
          Kout[(int64_t)b * Nc + i] = kv;
        } else if (SPLIT) {
          dg4[e & 3] = (unsigned long long)__double_as_longlong(fma(kv, aq, magicb));
          if ((e & 3) == 3) {                                     // byte transpose of four points' digits
            uint32_t o[MAXS];
            digits_transpose4<MAXS>(dg4, o);
#pragma unroll
            for (int t = 0; t < MAXS; ++t) dv[t][e >> 2] = o[t] ^ 0x80808080u;
          }
        }
      }
      if (SPLIT) {
        const int k0 = b0 + bb0, kc = k0 >> 6, piece = (k0 & 63) >> 4;
        uint8_t* dst = Aout + (size_t)kc * so.S * (128 * 64) + tid * 64 + ((piece ^ swz) << 4);
#pragma unroll
        for (int t = 0; t < MAXS; ++t)
          if (t < so.S) *reinterpret_cast<uint4*>(dst + (size_t)t * (128 * 64)) = make_uint4(dv[t][0], dv[t][1], dv[t][2], dv[t][3]);
      }
    }
  }
  const int64_t slab = (int64_t)kz * m * Nc;                   // 0 without the K-split
  mean[slab + (int64_t)j * Nc + i] = (ks == 1) ? mu + hp.ybar : mu;
  if (GRAD == 1) {
#pragma unroll
    for (int q = 0; q < DP; ++q)
      if (q < d) dmean[(slab + (int64_t)j * Nc + i) * d + q] = (xs[q] * wsum - gm[q]) / hp.ls[q];
  }
}

// mean = ybar + sum_z slab_z, dmean = sum_z slab_z  (K-split partials, fixed order)
__global__ void kstar_reduce_kernel(const double* __restrict__ mean_part, const double* __restrict__ dmean_part, int ks,
                                    int64_t Nc, int m, int d, int h, const OutHyp* __restrict__ hyp, int grad,
                                    double* __restrict__ mean, double* __restrict__ dmean) {
  const int j = blockIdx.y;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t slab = (int64_t)m * Nc;
  if (idx < Nc) {
    double s = hyp[h * m + j].ybar;
    for (int z = 0; z < ks; ++z) s += mean_part[z * slab + (int64_t)j * Nc + idx];
    mean[(int64_t)j * Nc + idx] = s;
  }
  if (grad && idx < Nc * d) {
    double s = 0.0;
    for (int z = 0; z < ks; ++z) s += dmean_part[(z * slab + (int64_t)j * Nc) * d + idx];
    dmean[(int64_t)j * Nc * d + idx] = s;
  }
}

// ===================================================================================================
// V = K* Linv^T on the lower triangle; per column-tile partial sums of V^2.
// grid.x = m * nct * i_tiles, heaviest column tiles (largest K extent) first.
__global__ void __launch_bounds__(PT::NTHREADS, PT_MINBLOCKS) var_gemm_kernel(const double* __restrict__ KsT,
                                                                    const double* __restrict__ LinvAll,
                                                                    double* __restrict__ V,
                                                                    double* __restrict__ part_var, int64_t Nc, int n16,
                                                                    int n_pad, int nct, int m, int h, int store_v) {
  extern __shared__ __align__(16) double smem[];
  const int i_tiles = (int)(Nc / CT);
  int bid = blockIdx.x;
  const int it = bid % i_tiles;
  bid /= i_tiles;
  const int at = nct - 1 - (bid % nct);
  const int j = bid / nct;
  const int hj = h * m + j;

  const double* A = KsT + (int64_t)j * n16 * Nc + (int64_t)it * CT;                   // A(m,k) = KsT[k*Nc + m]
  const double* B = LinvAll + (int64_t)hj * n_pad * n_pad + (int64_t)at * NT * n_pad;   // B(k,n) = Linv[n*n_pad + k]
  const int k_end = min(n16, (at + 1) * NT);

  double acc[MI][4][2];
  gemm::zero_acc(acc);
  gemm::mainloop<PT, true, false, gemm::TRI_K_LE_N>(acc, A, Nc, B, n_pad, 0, k_end, smem, at * NT);

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const int wn = warp % PT::WN;
  const int mbase = (warp / PT::WN) * PT::WTM, nbase = wn * 32;
  double* red = smem;   // [WN][CT]
#pragma unroll
  for (int i = 0; i < MI; ++i) {
    double s = 0.0;
#pragma unroll
    for (int jn = 0; jn < 4; ++jn) s += acc[i][jn][0] * acc[i][jn][0] + acc[i][jn][1] * acc[i][jn][1];
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    if (t == 0) red[wn * CT + mbase + 8 * i + g] = s;
  }
  if (store_v) {
    double* Vt = V + ((int64_t)j * Nc + (int64_t)it * CT) * n_pad + (int64_t)at * NT;
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
      for (int jn = 0; jn < 4; ++jn) {
        int r = mbase + 8 * i + g, c = nbase + 8 * jn + 2 * t;
        *reinterpret_cast<double2*>(Vt + (int64_t)r * n_pad + c) = make_double2(acc[i][jn][0], acc[i][jn][1]);
      }
  }
  __syncthreads();
  if (threadIdx.x < CT) {
    const int r = threadIdx.x;
    double s = red[r];
#pragma unroll
    for (int w = 1; w < PT::WN; ++w) s += red[w * CT + r];
    part_var[((int64_t)j * nct + at) * Nc + (int64_t)it * CT + r] = s;
  }
}

// ===================================================================================================
// Wt = V Linv on the lower triangle; epilogue contracts  Wt * G* * (xs_i - Xs_b)  over the tile's
// columns into per column-tile partial variance gradients.   grid.x = m * nct * i_tiles.
__global__ void __launch_bounds__(PT::NTHREADS, PT_MINBLOCKS) dvar_gemm_kernel(
    const double* __restrict__ V, const double* __restrict__ LinvAll, const double* __restrict__ GsT,
    const double* __restrict__ Xc, int64_t Nvalid, const double* __restrict__ XsAll, const OutHyp* __restrict__ hyp,
    double* __restrict__ part_dvar, int64_t Nc, int n, int n16, int n_pad, int nct, int m, int d, int h) {
  extern __shared__ __align__(16) double smem[];
  const int i_tiles = (int)(Nc / CT);
  int bid = blockIdx.x;
  const int it = bid % i_tiles;
  bid /= i_tiles;
  const int bt = bid % nct;         // ascending: largest K extent first
  const int j = bid / nct;
  const int hj = h * m + j;

  const double* A = V + ((int64_t)j * Nc + (int64_t)it * CT) * n_pad;                   // A(m,k) = V[m*n_pad + k]
  const double* B = LinvAll + (int64_t)hj * n_pad * n_pad + (int64_t)bt * NT;             // B(k,n) = Linv[k*n_pad + n]
  double acc[MI][4][2];
  gemm::zero_acc(acc);
  if (bt * NT < n16)
    gemm::mainloop<PT, false, true, gemm::TRI_K_GE_N>(acc, A, n_pad, B, n_pad, bt * NT, n16, smem, bt * NT);

  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const int wn = warp % PT::WN;
  const int mbase = (warp / PT::WN) * PT::WTM, nbase = wn * 32;
  const OutHyp& hp = hyp[hj];

  // stage scaled candidate / training coordinates for this tile:  sxi[q][row], sxb[q][col]
  double* sxi = smem;                          // d x CT
  double* sxb = smem + d * CT;                 // d x NT
  double* red = smem + d * (CT + NT);          // WN x CT x d      (<= 56 KiB for d <= MAXD)
  for (int idx = tid; idx < d * CT; idx += PT::NTHREADS) {
    int r = idx / d, q = idx - r * d;
    int64_t i = (int64_t)it * CT + r;
    sxi[q * CT + r] = (i < Nvalid) ? Xc[i * d + q] / hp.ls[q] : 0.0;
  }
  for (int idx = tid; idx < d * NT; idx += PT::NTHREADS) {
    int c = idx / d, q = idx - c * d;
    int b = bt * NT + c;
    sxb[q * NT + c] = XsAll[((int64_t)hj * n_pad + b) * d + q];
  }
  // wg = Wt * G*
  const double* Gj = GsT + (int64_t)j * n16 * Nc + (int64_t)it * CT;
#pragma unroll
  for (int i = 0; i < MI; ++i) {
    const int r = mbase + 8 * i + g;
#pragma unroll
    for (int jn = 0; jn < 4; ++jn)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int b = bt * NT + nbase + 8 * jn + 2 * t + e;
        const double gv = (b < n) ? Gj[(int64_t)b * Nc + r] : 0.0;
        acc[i][jn][e] *= gv;
      }
  }
  __syncthreads();
  static_assert(MI == 4 || MI == 8, "the quad reduce-scatter below handles 4 or 8 row tiles per warp");
  for (int q = 0; q < d; ++q) {
    double xb[4][2];
#pragma unroll
    for (int jn = 0; jn < 4; ++jn) {
      xb[jn][0] = sxb[q * NT + nbase + 8 * jn + 2 * t];
      xb[jn][1] = sxb[q * NT + nbase + 8 * jn + 2 * t + 1];
    }
    double s[MI];
#pragma unroll
    for (int i = 0; i < MI; ++i) {
      const double xi = sxi[q * CT + mbase + 8 * i + g];
      double acc_s = 0.0;
#pragma unroll
      for (int jn = 0; jn < 4; ++jn) {
        acc_s += acc[i][jn][0] * (xi - xb[jn][0]);
        acc_s += acc[i][jn][1] * (xi - xb[jn][1]);
      }
      s[i] = acc_s;
    }
    // reduce over the 4 lanes of a quad AND scatter the MI row sums over them (3*MI/4 shuffles instead of 2*MI):
    // step 1 (lane ^ 1): a lane keeps rows (MI/2)*(t&1)+k, k < MI/2;  step 2 (lane ^ 2): rows ... + (MI/4)*(t>>1)+k
    constexpr int H1 = MI / 2, H2 = MI / 4;
    double u[H1], w2[H2];
#pragma unroll
    for (int k = 0; k < H1; ++k) {
      const double send = (t & 1) ? s[k] : s[k + H1];
      const double keep = (t & 1) ? s[k + H1] : s[k];
      u[k] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
    }
#pragma unroll
    for (int k = 0; k < H2; ++k) {
      const double send = (t & 2) ? u[k] : u[k + H2];
      const double keep = (t & 2) ? u[k + H2] : u[k];
      w2[k] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
#pragma unroll
    for (int k = 0; k < H2; ++k) {
      const int irow = H1 * (t & 1) + H2 * (t >> 1) + k;
      red[(wn * CT + mbase + 8 * irow + g) * d + q] = w2[k];
    }
  }
  __syncthreads();
  double* out = part_dvar + (((int64_t)j * nct + bt) * Nc + (int64_t)it * CT) * d;
  for (int idx = tid; idx < CT * d; idx += PT::NTHREADS) {
    double sum = red[idx];
#pragma unroll
    for (int w = 1; w < PT::WN; ++w) sum += red[w * CT * d + idx];
    out[idx] = sum;
  }
}

// ===================================================================================================
// var = clip(k** - sum_tiles part_var (+ noise), 1e-10);  dvar = (-2 / l_q) sum_tiles part_dvar
// split mode: part_dvar holds sum_b T_b Xs_bq and part_s0 holds sum_b T_b (T = Wt * G*), so that
//   sum_b T_b (xs_iq - Xs_bq) = xs_iq * S0 - ACC_q   with xs_i = x_i / l formed here, once per candidate.
__global__ void finalize_kernel(const double* __restrict__ part_var, const double* __restrict__ part_dvar,
                                const OutHyp* __restrict__ hyp, int64_t Nc, int nct, int nct_g, int m, int d, int h, int grad,
                                int noiseless, double* __restrict__ var, double* __restrict__ dvar,
                                const double* __restrict__ part_s0, const double* __restrict__ Xc, int64_t Nvalid) {
  // thread idx covers candidate idx (variance) and flat element idx = i*d + q (gradient): both coalesced
  const int j = blockIdx.y;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const OutHyp& hp = hyp[h * m + j];
  const int64_t Nv = min(Nc, (Nvalid + 127) / 128 * 128);     // candidate tiles beyond the valid ones were skipped upstream
  if (idx < Nv) {
    double s = 0.0;
    for (int tI = 0; tI < nct; ++tI) s += part_var[((int64_t)j * nct + tI) * Nc + idx];
    double v = hp.variance - s;
    if (!noiseless) v = hp.noise + v;
    var[(int64_t)j * Nc + idx] = (noiseless == 2) ? v : fmax(v, 1e-10);     // 2: the KG helpers' unclipped form (gp.py:543)
  }
  if (grad && idx < Nv * d) {
    const int q = (int)(idx % d);
    double gsum = 0.0;
    for (int tI = 0; tI < nct_g; ++tI) gsum += part_dvar[((int64_t)j * nct_g + tI) * Nc * d + idx];
    if (part_s0 != nullptr) {
      const int64_t i = idx / d;
      double s0 = 0.0;
      for (int tI = 0; tI < nct_g; ++tI) s0 += part_s0[((int64_t)j * nct_g + tI) * Nc + i];
      const double xs = (i < Nvalid) ? Xc[i * d + q] / hp.ls[q] : 0.0;
      gsum = xs * s0 - gsum;
    }
    dvar[(int64_t)j * Nc * d + idx] = -2.0 * gsum / hp.ls[q];
  }
}

// ===================================================================================================
int candidate_tile() { return CT; }
// scratch of the K-split partial sums (small chunks only; added on top of the per-candidate chunk bytes)
uint64_t kstar_part_bytes(const bocf_model* M, int64_t Nc) {
  const int ks = kstar_ksplit(M, Nc);
  return ks > 1 ? (uint64_t)ks * M->m * Nc * (1 + M->d) * sizeof(double) + 1024 : 0;
}

uint64_t chunk_bytes_per_candidate(const bocf_model* M, bool grad, int64_t Nc) {
  if (M->S > 0) return split_chunk_bytes_per_candidate(M, grad, Nc);
  const uint64_t nct = M->n_pad / NT;
  uint64_t per = 0;
  per += (uint64_t)M->m * M->n16;                       // KsT
  per += (uint64_t)M->m * nct;                          // part_var
  per += 2ull * M->m;                                   // mean, var
  if (grad) {
    per += (uint64_t)M->m * M->n16;                     // GsT
    per += (uint64_t)M->m * M->n_pad;                   // V
    per += (uint64_t)M->m * nct * M->d;                 // part_dvar
    per += 2ull * M->m * M->d;                          // dmean, dvar
  }
  return per * sizeof(double);
}

void carve_chunk(const bocf_model* M, void* base, int64_t Nc, bool grad, ChunkBuffers* cb) {
  cb->A1 = cb->A2 = nullptr;
  if (M->S > 0) {
    split_carve_chunk(M, base, Nc, grad, cb);
    return;
  }
  const uint64_t nct = M->n_pad / NT;
  double* p = reinterpret_cast<double*>(base);
  auto take = [&](uint64_t count) {
    double* r = p;
    p += round_up((int64_t)count, 32);
    return r;
  };
  cb->Nc = Nc;
  cb->KsT = take((uint64_t)M->m * M->n16 * Nc);
  cb->part_var = take((uint64_t)M->m * nct * Nc);
  cb->mean = take((uint64_t)M->m * Nc);
  cb->var = take((uint64_t)M->m * Nc);
  if (grad) {
    cb->GsT = take((uint64_t)M->m * M->n16 * Nc);
    cb->V = take((uint64_t)M->m * Nc * M->n_pad);
    cb->part_dvar = take((uint64_t)M->m * nct * Nc * M->d);
    cb->dmean = take((uint64_t)M->m * Nc * M->d);
    cb->dvar = take((uint64_t)M->m * Nc * M->d);
  } else {
    cb->GsT = cb->V = cb->part_dvar = cb->dmean = cb->dvar = nullptr;
  }
  cb->kpart = (kstar_ksplit(M, Nc) > 1) ? take((uint64_t)kstar_ksplit(M, Nc) * M->m * Nc * (1 + M->d)) : nullptr;
}

template <int KIND, int DP>
static int launch_kstar_t(bocf_model* M, int h, const double* Xc, int64_t Nvalid, int grad, const ChunkBuffers& cb,
                          OutRun run, cudaStream_t st) {
  SplitOut so;
  so.A1 = cb.A1;
  so.aq = M->aq;
  so.gcs = M->cs2;
  so.gcs_ld = M->nct2 * M->NT2;
  so.KCH = M->KCH;
  so.S = M->S;
  const int spl = (cb.A1 == nullptr) ? 0 : (M->S == 5 ? 5 : 6);
  // small batches: split the training points over gridDim.z blocks (latency), partial sums into cb.kpart
  const int ks = kstar_ksplit(M, cb.Nc);
  dim3 kgrid((unsigned)(cb.Nc / 128), (unsigned)run.cnt, (unsigned)ks);
  double* mean_out = (ks > 1) ? cb.kpart : cb.mean;
  double* dmean_out = (ks > 1) ? cb.kpart + (size_t)ks * M->m * cb.Nc : cb.dmean;
#define BOCF_KSTAR(G, SP)                                                                                               \
  kstar_kernel<KIND, DP, G, SP><<<kgrid, 128, 0, st>>>(Xc, Nvalid, cb.Nc, M->d, M->n, M->n16, M->n_pad, M->m, h, M->hyp, \
                                                       M->Xs, M->xsq, M->alpha, cb.KsT, cb.GsT, mean_out, dmean_out, so,     \
                                                       run.j0)
  if (grad < 0) BOCF_KSTAR(0, -1);
  else if (grad == 2 && spl == 5) BOCF_KSTAR(2, 5);
  else if (grad == 2 && spl == 6) BOCF_KSTAR(2, 6);
  else if (grad && spl == 5) BOCF_KSTAR(1, 5);
  else if (grad && spl == 6) BOCF_KSTAR(1, 6);
  else if (grad) BOCF_KSTAR(1, 0);
  else if (spl == 5) BOCF_KSTAR(0, 5);
  else if (spl == 6) BOCF_KSTAR(0, 6);
  else BOCF_KSTAR(0, 0);
#undef BOCF_KSTAR
  BOCF_LAUNCH_OK("kstar_kernel");
  return 0;
}

template <int KIND>
static int launch_kstar_k(bocf_model* M, int h, const double* Xc, int64_t Nvalid, int grad, const ChunkBuffers& cb,
                          OutRun run, cudaStream_t st) {
  const int d = M->d;
  if (d <= 4) return launch_kstar_t<KIND, 4>(M, h, Xc, Nvalid, grad, cb, run, st);
  if (d <= 6) return launch_kstar_t<KIND, 6>(M, h, Xc, Nvalid, grad, cb, run, st);
  if (d <= 8) return launch_kstar_t<KIND, 8>(M, h, Xc, Nvalid, grad, cb, run, st);
  if (d <= 10) return launch_kstar_t<KIND, 10>(M, h, Xc, Nvalid, grad, cb, run, st);
  if (d <= 12) return launch_kstar_t<KIND, 12>(M, h, Xc, Nvalid, grad, cb, run, st);
  return launch_kstar_t<KIND, MAXD>(M, h, Xc, Nvalid, grad, cb, run, st);
}

// grad: -1 = mean only (launch_posterior_mean_chunk); 0 / 1 / 2 = kstar_kernel's GRAD
static int launch_kstar(bocf_model* M, int h, const double* Xc, int64_t Nvalid, int grad, const ChunkBuffers& cb,
                        cudaStream_t st) {
  ProfScope ps(grad < 0 ? "kstar_mean_kernel" : "kstar_kernel", st);
  // one launch per run of outputs that share a kernel family (one launch when they all do)
  const int rc = for_each_kind_run(M, [&](int kind, OutRun run) -> int {
    switch (kind) {
      case BOCF_KERN_SE: return launch_kstar_k<BOCF_KERN_SE>(M, h, Xc, Nvalid, grad, cb, run, st);
      case BOCF_KERN_RBF: return launch_kstar_k<BOCF_KERN_RBF>(M, h, Xc, Nvalid, grad, cb, run, st);
      case BOCF_KERN_MATERN52: return launch_kstar_k<BOCF_KERN_MATERN52>(M, h, Xc, Nvalid, grad, cb, run, st);
      case BOCF_KERN_MATERN32: return launch_kstar_k<BOCF_KERN_MATERN32>(M, h, Xc, Nvalid, grad, cb, run, st);
    }
    set_error("unknown kernel kind");
    return -1;
  });
  if (rc) return rc;
  const int ks = kstar_ksplit(M, cb.Nc);
  if (ks > 1) {                                  // K-split partial sums of every output, added in fixed order
    double* mean_part = cb.kpart;
    double* dmean_part = cb.kpart + (size_t)ks * M->m * cb.Nc;
    dim3 rgrid((unsigned)ceil_div(grad == 1 ? cb.Nc * M->d : cb.Nc, 256), (unsigned)M->m);
    kstar_reduce_kernel<<<rgrid, 256, 0, st>>>(mean_part, dmean_part, ks, cb.Nc, M->m, M->d, h, M->hyp, grad == 1 ? 1 : 0,
                                               cb.mean, cb.dmean);
    BOCF_LAUNCH_OK("kstar_reduce_kernel");
  }
  return 0;
}

int launch_posterior_mean_chunk(bocf_model* M, int h, const double* Xc, int64_t Nvalid, const ChunkBuffers& cb,
                                cudaStream_t st) {
  return launch_kstar(M, h, Xc, Nvalid, -1, cb, st);
}

// ===================================================================================================
// Active units of the fused gradient's second contraction.  A unit (output j, candidate tile rt) whose gradient weights
// WA, WB are all exactly zero contributes exactly zero to the acquisition gradient (EI-CF: no base sample of its
// candidates passes the strict indicator U > f*).  Uniformly spread candidates almost never improve on the incumbent, so
// most units of a sweep are in this case and the EPI_DACQ contraction walks only the flagged ones.  The weights' producer
// does not matter (mc_acq_kernel, mc_acq_user_kernel, ma_acq_kernel).  A NaN weight counts as non-zero.
// flags[j * RTv + rt], one warp per unit; only valid candidates (i < Nvalid) are read.
__global__ void active_units_flag_kernel(const double* __restrict__ wa, const double* __restrict__ wb, int64_t Nc,
                                         int64_t Nvalid, int rtv, int units, int* __restrict__ flags) {
  const int unit = (int)blockIdx.x * (blockDim.x >> 5) + (int)(threadIdx.x >> 5);
  if (unit >= units) return;
  const int lane = threadIdx.x & 31;
  const int j = unit / rtv, rt = unit - j * rtv;
  bool act = false;
#pragma unroll
  for (int r = lane; r < CT; r += 32) {
    const int64_t i = (int64_t)rt * CT + r;
    if (i < Nvalid) act |= !(wa[(int64_t)j * Nc + i] == 0.0) || !(wb[(int64_t)j * Nc + i] == 0.0);
  }
  act = __any_sync(0xffffffffu, act);
  if (lane == 0) flags[unit] = act ? 1 : 0;
}

// The ids of the flagged units in ascending order and their number: one block of 1024 threads, 1024 flags per trip.
__global__ void __launch_bounds__(1024) active_units_list_kernel(const int* __restrict__ flags, int units,
                                                                 int* __restrict__ list, int* __restrict__ count) {
  __shared__ int s_warp[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int base = 0;
  for (int u0 = 0; u0 < units; u0 += 1024) {
    const int u = u0 + (int)threadIdx.x;
    const bool f = (u < units) && flags[u] != 0;
    const unsigned b = __ballot_sync(0xffffffffu, f);
    if (lane == 0) s_warp[warp] = __popc(b);
    __syncthreads();
    const int wc = s_warp[lane];                           // every warp scans the 32 warp counts itself
    int incl = wc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const int before = __shfl_sync(0xffffffffu, incl - wc, warp);
    if (f) list[base + before + __popc(b & ((1u << lane) - 1u))] = u;
    base += __shfl_sync(0xffffffffu, incl, 31);
    __syncthreads();                                       // s_warp is rewritten by the next trip
  }
  if (threadIdx.x == 0) *count = base;
}

// sum over outputs and partials of the fused gradient:  dacq[i][q] (+)= sum_j (xs_jq S0_j - ACC_jq) / l_jq
// (S0 / ACC: the weighted sums the EPI_DACQ epilogue leaves per output, split_gemm.cu).  Units without a flag were not
// computed: they contribute exactly zero, and their partial slots hold whatever an earlier chunk left there.
__global__ void finalize_grad_kernel(const double* __restrict__ part_dvar, const double* __restrict__ part_s0,
                                     const int* __restrict__ unit_flags, const OutHyp* __restrict__ hyp, int64_t Nc,
                                     int64_t Nvalid, int nparts, int m, int d, int h, const double* __restrict__ Xc,
                                     int accumulate, double* __restrict__ dacq) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= Nvalid * d) return;
  const int64_t i = idx / d;
  const int q = (int)(idx - i * d);
  const int rtv = (int)((Nvalid + CT - 1) / CT);
  const int* flag = unit_flags + i / CT;
  const double x = Xc[i * d + q];
  double g = 0.0;
  for (int j = 0; j < m; ++j) {
    if (flag[j * rtv] == 0) continue;
    const OutHyp& hp = hyp[h * m + j];
    double acc = 0.0, s0 = 0.0;
    for (int t = 0; t < nparts; ++t) {
      acc += part_dvar[(((int64_t)j * nparts + t) * Nc + i) * d + q];
      s0 += part_s0[((int64_t)j * nparts + t) * Nc + i];
    }
    g += ((x / hp.ls[q]) * s0 - acc) / hp.ls[q];
  }
  dacq[idx] = accumulate ? dacq[idx] + g : g;
}

// The same sum for tiny batches (the L-BFGS rounds: <= 128 candidates), where one thread per (candidate, dimension)
// walking m x nparts partials serially is pure latency (~50 us at m = 16, 12 partials): a WARP per (candidate, dimension),
// lanes striding over the (output, partial) pairs -- the sum is linear in them -- then one shuffle reduction.
// (one candidate tile: the unit flags are unit_flags[j])
__global__ void __launch_bounds__(256) finalize_grad_small_kernel(const double* __restrict__ part_dvar,
                                                                  const double* __restrict__ part_s0,
                                                                  const int* __restrict__ unit_flags,
                                                                  const OutHyp* __restrict__ hyp, int64_t Nc, int64_t Nvalid,
                                                                  int nparts, int m, int d, int h,
                                                                  const double* __restrict__ Xc, int accumulate,
                                                                  double* __restrict__ dacq) {
  const int64_t idx = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (idx >= Nvalid * d) return;
  const int lane = threadIdx.x & 31;
  const int64_t i = idx / d;
  const int q = (int)(idx - i * d);
  const double x = Xc[i * d + q];
  double g = 0.0;
  for (int p = lane; p < m * nparts; p += 32) {
    const int j = p / nparts;                                  // p = j * nparts + t
    if (unit_flags[j] == 0) continue;
    const double il = 1.0 / hyp[h * m + j].ls[q];
    g += (x * il * part_s0[(int64_t)p * Nc + i] - part_dvar[((int64_t)p * Nc + i) * d + q]) * il;
  }
  g = warp_sum(g);
  if (lane == 0) dacq[idx] = accumulate ? dacq[idx] + g : g;
}

// Fused acquisition-gradient sweep of one chunk and one hyper-sample (EI-CF / mean-utility with gradients, tensor-core
// contraction mode): K* (mean, digit planes, G*; no mean gradient) -> first contraction -> variance -> MC forward pass
// leaving the value and the per-(candidate, output) gradient weights WA, WB -> the units with a non-zero weight ->
// second contraction over those units, whose epilogue contracts G* (WA alpha - 2 WB Wt) against the training inputs ->
// sum over outputs.  The per-output mean / variance gradients (2 m d doubles per candidate) are never formed.
int launch_fused_grad_chunk(bocf_model* M, int h, const double* Xc, int64_t Nvalid, int noiseless, const ChunkBuffers& cb,
                            AcqParams P, double* acq, double* dacq, cudaStream_t st) {
  if (int rc = launch_kstar(M, h, Xc, Nvalid, 2, cb, st)) return rc;
  if (int rc = launch_split_var(M, h, Nvalid, cb, true, st)) return rc;
  {
    const int nct = split_partials_var(M, cb.Nc);
    dim3 fgrid((unsigned)ceil_div(cb.Nc, 256), (unsigned)M->m);
    ProfScope ps("finalize_kernel", st);
    finalize_kernel<<<fgrid, 256, 0, st>>>(cb.part_var, cb.part_dvar, M->hyp, cb.Nc, nct, 0, M->m, M->d, h, 0, noiseless,
                                           cb.var, cb.dvar, nullptr, Xc, Nvalid);
    BOCF_LAUNCH_OK("finalize_kernel");
  }
  P.wa = cb.wa;
  P.wb = cb.wb;
  if (int rc = launch_acq_chunk(P, cb, Nvalid, acq, nullptr, st)) return rc;
  {
    const int rtv = (int)ceil_div(Nvalid, CT);
    const int units = M->m * rtv;
    ProfScope ps("active_units_kernel", st);
    active_units_flag_kernel<<<(unsigned)ceil_div(units, 8), 256, 0, st>>>(cb.wa, cb.wb, cb.Nc, Nvalid, rtv, units,
                                                                           cb.unit_flags);
    BOCF_LAUNCH_OK("active_units_flag_kernel");
    active_units_list_kernel<<<1, 1024, 0, st>>>(cb.unit_flags, units, cb.unit_list, cb.unit_count);
    BOCF_LAUNCH_OK("active_units_list_kernel");
  }
  if (int rc = launch_split_dvar(M, h, Xc, Nvalid, cb, true, st)) return rc;
  {
    ProfScope ps("finalize_kernel", st);
    if (Nvalid <= 128)
      finalize_grad_small_kernel<<<(unsigned)ceil_div(Nvalid * M->d, 8), 256, 0, st>>>(cb.part_dvar, cb.part_s0, cb.unit_flags,
                                                                                     M->hyp, cb.Nc, Nvalid,
                                                                                     split_partials_dvar(M, cb.Nc), M->m, M->d,
                                                                                     h, Xc, P.accumulate, dacq);
    else
      finalize_grad_kernel<<<(unsigned)ceil_div(Nvalid * M->d, 256), 256, 0, st>>>(cb.part_dvar, cb.part_s0, cb.unit_flags,
                                                                                 M->hyp, cb.Nc, Nvalid,
                                                                                 split_partials_dvar(M, cb.Nc), M->m, M->d, h,
                                                                                 Xc, P.accumulate, dacq);
    BOCF_LAUNCH_OK("finalize_grad_kernel");
  }
  return 0;
}

int launch_posterior_chunk(bocf_model* M, int h, const double* Xc, int64_t Nvalid, bool grad, int noiseless,
                           const ChunkBuffers& cb, cudaStream_t st, bool need_var, bool need_dvar) {
  static bool attrs[64] = {false};               // per device: function attributes belong to the device's context
  if (M->device >= 0 && M->device < 64 && !attrs[M->device]) {
    BOCF_CUDA_OK(cudaFuncSetAttribute(var_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PT::SMEM_BYTES));
    BOCF_CUDA_OK(cudaFuncSetAttribute(dvar_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PT::SMEM_BYTES));
    attrs[M->device] = true;
  }
  need_dvar = need_dvar && grad;
  need_var = need_var || need_dvar;
  if (int rc = launch_kstar(M, h, Xc, Nvalid, grad ? 1 : 0, cb, st)) return rc;
  if (!need_var) return 0;      // mean (and mean gradient) only: no contraction against the factor
  const bool split = (cb.A1 != nullptr);
  const int nct = split ? split_partials_var(M, cb.Nc) : M->n_pad / NT;       // partial sums per candidate: variance
  const int nct_g = split ? split_partials_dvar(M, cb.Nc) : M->n_pad / NT;    //                             variance gradient
  const unsigned tiles = (unsigned)((cb.Nc / CT) * nct * M->m);
  if (split) {
    // tcgen05 kind::i8 digit-plane contractions (split_gemm.cu); same partial-sum layout, same finalize
    if (int rc2 = launch_split_var(M, h, Nvalid, cb, need_dvar, st)) return rc2;
    if (need_dvar)
      if (int rc2 = launch_split_dvar(M, h, Xc, Nvalid, cb, false, st)) return rc2;
  } else {
  {
    ProfScope ps("var_gemm_kernel", st);
    var_gemm_kernel<<<tiles, PT::NTHREADS, PT::SMEM_BYTES, st>>>(cb.KsT, M->Linv, cb.V, cb.part_var, cb.Nc, M->n16,
                                                                  M->n_pad, nct, M->m, h, need_dvar ? 1 : 0);
  }
  BOCF_LAUNCH_OK("var_gemm_kernel");
  if (need_dvar) {
    ProfScope ps("dvar_gemm_kernel", st);
    dvar_gemm_kernel<<<tiles, PT::NTHREADS, PT::SMEM_BYTES, st>>>(cb.V, M->Linv, cb.GsT, Xc, Nvalid, M->Xs, M->hyp,
                                                                  cb.part_dvar, cb.Nc, M->n, M->n16, M->n_pad, nct,
                                                                  M->m, M->d, h);
  }
  if (need_dvar) BOCF_LAUNCH_OK("dvar_gemm_kernel");
  }
  dim3 fgrid((unsigned)ceil_div(need_dvar ? cb.Nc * M->d : cb.Nc, 256), (unsigned)M->m);
  {
    ProfScope ps("finalize_kernel", st);
    finalize_kernel<<<fgrid, 256, 0, st>>>(cb.part_var, cb.part_dvar, M->hyp, cb.Nc, nct, nct_g, M->m, M->d, h,
                                           need_dvar ? 1 : 0, noiseless, cb.var, cb.dvar,
                                           split ? cb.part_s0 : nullptr, Xc, Nvalid);
  }
  BOCF_LAUNCH_OK("finalize_kernel");
  return 0;
}

}  // namespace bocf
