// chol.cu -- per-iteration model factorisation on device, fp64 (north-star subsystem 4, SURVEY K4).
//
// For every (hyper-sample h, output j):   Ky = K(X,X) + (sigma_n^2 + 1e-8 [+ jitter]) I
//   L = chol(Ky) (lower)          exact_gaussian_inference.py:43-49 -> linalg.py:52-83 (jitchol)
//   Linv = L^-1                   used by the candidate sweep instead of LAPACK dtrtrs (posterior.py:312)
//   alpha = Ky^-1 (y - ybar)      exact_gaussian_inference.py:51 (dpotrs)
// Blocked right-looking Cholesky with 128 x 128 blocks: the diagonal block is factorised and
// inverted by one CTA in shared memory, the panel solve and the trailing SYRK run on the DMMA
// tile engine (gemm_f64.cuh) batched over all H*m matrices.  L^-1 is then built block-row by
// block-row with the same engine.
#include "gemm_f64.cuh"
#include "kernfn.cuh"
#include "model.h"

namespace bocf {

// ---------------------------------------------------------------------------------------------------
// ybar / centred observations (GPy/util/normalizer.py:57-66: mean only, std == 1)
__global__ void ybar_kernel(const double* __restrict__ Y, int n, int n_pad, int m, int H, double* __restrict__ ybar,
                            double* __restrict__ yc, OutHyp* __restrict__ hyp) {
  __shared__ double red[32];
  __shared__ double mean_s;
  const int j = blockIdx.x;
  double s = 0.0;
  for (int b = threadIdx.x; b < n; b += blockDim.x) s += Y[(int64_t)j * n + b];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
    mean_s = tot / (double)n;
    ybar[j] = mean_s;
    for (int h = 0; h < H; ++h) hyp[h * m + j].ybar = mean_s;
  }
  __syncthreads();
  const double mu = mean_s;
  for (int b = threadIdx.x; b < n_pad; b += blockDim.x)
    yc[(int64_t)j * n_pad + b] = (b < n) ? (Y[(int64_t)j * n + b] - mu) / 1.0 : 0.0;
}

// Xs = X / lengthscale (stationary.py:161-164, se.py:86-89), xsq = sum_q Xs^2 (stationary.py:141-142)
__global__ void scale_inputs_kernel(const double* __restrict__ X, int n, int n_pad, int d,
                                    const OutHyp* __restrict__ hyp, double* __restrict__ Xs,
                                    double* __restrict__ xsq) {
  const int hj = blockIdx.y;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_pad) return;
  const OutHyp& hp = hyp[hj];
  double s = 0.0;
  for (int q = 0; q < d; ++q) {
    double v = (b < n) ? X[(int64_t)b * d + q] / hp.ls[q] : 0.0;
    Xs[((int64_t)hj * n_pad + b) * d + q] = v;
    s += v * v;
  }
  xsq[(int64_t)hj * n_pad + b] = s;
}

// Training Gram matrix + diagonal term (exact_gaussian_inference.py:43-47).
// Stationary kinds: r^2 = -2 Xs Xs^T + (xsq_a + xsq_b), diagonal forced to 0, clipped (stationary.py:134-139).
// SE: exact squared differences, diagonal = variance (se.py:56-58).
template <int KIND>
__global__ void gram_kernel(const double* __restrict__ Xs, const double* __restrict__ xsq,
                            const OutHyp* __restrict__ hyp, int n, int n_pad, int d, double* __restrict__ A, OutRun run,
                            int m) {
  if (blockIdx.x > blockIdx.y) return;             // only the lower triangle is ever read (potrf / trsm / syrk)
  const int hj = run_hj(blockIdx.z, run, m);
  const int a = blockIdx.y * 16 + threadIdx.y;
  const int b = blockIdx.x * 16 + threadIdx.x;
  __shared__ double sa[16][MAXD + 1], sb[16][MAXD + 1];
  const double* Xh = Xs + (int64_t)hj * n_pad * d;
  for (int q = threadIdx.x; q < d; q += 16) sa[threadIdx.y][q] = Xh[(int64_t)a * d + q];
  for (int q = threadIdx.y; q < d; q += 16) sb[threadIdx.x][q] = Xh[(int64_t)b * d + q];
  __syncthreads();
  const OutHyp& hp = hyp[hj];
  double val = 0.0;
  if (a < n && b < n) {
    double r2;
    if (KIND == BOCF_KERN_SE) {
      r2 = 0.0;
      for (int q = 0; q < d; ++q) {
        double df = sa[threadIdx.y][q] - sb[threadIdx.x][q];
        r2 += df * df;
      }
      if (a == b) r2 = 0.0;
    } else {
      double dot = 0.0;
      for (int q = 0; q < d; ++q) dot += sa[threadIdx.y][q] * sb[threadIdx.x][q];
      r2 = -2.0 * dot + (xsq[(int64_t)hj * n_pad + a] + xsq[(int64_t)hj * n_pad + b]);
      if (a == b) r2 = 0.0;
      r2 = fmax(r2, 0.0);
    }
    double k, gdummy;
    kern_eval<KIND, false>(r2, hp.variance, k, gdummy);
    if (a == b) k += hp.noise + 1e-8 + hp.jitter;
    val = k;
  }
  A[((int64_t)hj * n_pad + a) * n_pad + b] = val;
}

// ---------------------------------------------------------------------------------------------------
// Diagonal block: Cholesky + in-place triangular inverse of one 128 x 128 block in shared memory (one CTA / matrix).
// This step sits nb times on the critical path of every factorisation (only H*m CTAs can work on it), so it is organised
// around its dependency chain, in 32-wide sub-blocks (profiles/r2_fit_pass.md has the ncu history, 143 -> 46 us):
//   factor    the 32 x 32 diagonal sub-block by ONE warp, register resident (lane = row).  Per column the chain is
//             pivot shuffle -> rsqrt -> multiply -> multiply-add: the next pivot needs only lane k+1's own two values;
//             the finished column is parked in shared memory (column-major) and subtracted from the columns to its
//             right with independent multiply-adds fed by 16-byte broadcast loads;
//   solve     the rows below it by forward substitution, thread per row, from the parked columns -- and in the same
//             phase, by the same instructions, the rows of the IDENTITY, which gives the sub-block's inverse;
//   update    the trailing lower triangle on the fp64 tensor cores (DMMA 8x8x4, K = 32);
//   assemble  the 128 x 128 inverse from the four sub-block inverses recursively,  X21 = -X22 (L21 X11),  at 32 then 64
//             wide, again on DMMA.
// The dpotrf failure convention is kept: the first non-positive pivot is reported in info[] (1-based), replaced by 1.
constexpr int PSB = 32;                       // sub-block
constexpr int DLD = TILE + 4;                 // row stride == 4 mod 16 doubles: conflict-free 64-bit fragment loads
constexpr int WLD = 64 + 4;
constexpr int POTRF_SMEM = (TILE * DLD + 64 * WLD + TILE + (TILE / PSB) * PSB * PSB) * (int)sizeof(double);

// C[i0.., j0..] (8 x 8) = sum_k A[i0 + g][k] B(k, j0 + g), K a multiple of 4.  BT: B(k, n) = Bm[n * ldb + k] (rows of Bm
// are columns of B), else B(k, n) = Bm[k * ldb + n].  lane = 4 g + t.
template <bool BT>
__device__ __forceinline__ void dmma_tile(double& c0, double& c1, const double* __restrict__ A, int lda,
                                          const double* __restrict__ Bm, int ldb, int K, int g, int t) {
#pragma unroll 8
  for (int k = 0; k < K; k += 4) {
    const double a = A[g * lda + k + t];
    const double b = BT ? Bm[g * ldb + k + t] : Bm[(k + t) * ldb + g];
    dmma884(c0, c1, a, b);
  }
}

// The whole CTA (256 threads) factors and inverts block kb of matrix hj; T = POTRF_SMEM bytes of shared memory.  Called by
// potrf_diag_kernel (first block) and, as a look-ahead, by the CTA of the trailing update that owns the next diagonal tile.
__device__ __forceinline__ void potrf_block(double* __restrict__ T, double* __restrict__ Lmat, double* __restrict__ Dinv,
                                            int* __restrict__ info, int n, int n_pad, int nb, int kb, int hj) {
  double* W = T + TILE * DLD;                   // T[TILE][DLD] | W[64][WLD] | dinv[TILE] | Xb[4][32][32]
  double* dinv = W + 64 * WLD;
  double* Xb = dinv + TILE;                     // inverses of the four diagonal sub-blocks (row-major 32 x 32 each)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int k0 = kb * TILE;
  const int nrem = min(TILE, n - k0);
  double* Ablk = Lmat + (int64_t)hj * n_pad * n_pad + (int64_t)k0 * n_pad + k0;
  // lower triangle of the valid part, identity on the padding, zero above the diagonal; 16-byte async copies so the whole
  // 128 KB block is in flight at once (a scalar load loop cost ~19 us of exposed latency per launch)
  for (int idx = tid; idx < TILE * (TILE / 2); idx += 256) {
    const int r = idx >> 6, c = (idx & 63) * 2;
    double* dst = T + r * DLD + c;
    if (c > r) {
      dst[0] = 0.0;
      dst[1] = 0.0;
    } else if (r < nrem) {
      cp_async16(dst, Ablk + (int64_t)r * n_pad + c);
    } else {
      dst[0] = (r == c) ? 1.0 : 0.0;
      dst[1] = (r == c + 1) ? 1.0 : 0.0;
    }
  }
  cp_async_commit();
  cp_async_wait<0>();
  __syncthreads();
  if (tid < TILE / 2) T[(2 * tid) * DLD + 2 * tid + 1] = 0.0;      // the pair that straddles the diagonal
  __syncthreads();
  double* Lt = W;                                 // [4][32][32]: column k of sub-block s at Lt[s*1024 + k*32 + row]

  // ---------------- Cholesky ----------------
  for (int c0 = 0; c0 < TILE; c0 += PSB) {
    double* Ls = Lt + (c0 / PSB) * (PSB * PSB);
    if (warp == 0) {
      // lane = row of the diagonal sub-block, held in registers.  Right-looking: column k is finished (scaled by
      // 1 / sqrt(pivot)), parked in shared memory (Ls, column-major: the panel solve and the inverse below read it
      // again), and every lane subtracts its multiple from the columns to the right -- independent multiply-adds fed by
      // broadcast 16-byte loads.  Column k + 1 goes first so the next pivot's reciprocal square root overlaps the rest.
      double a[PSB];
#pragma unroll
      for (int q = 0; q < PSB; q += 2) {
        const double2 v = *reinterpret_cast<const double2*>(T + (c0 + lane) * DLD + c0 + q);
        a[q] = v.x;
        a[q + 1] = v.y;
      }
      double piv = __shfl_sync(0xffffffffu, a[0], 0);
#pragma unroll
      for (int k = 0; k < PSB; ++k) {
        double pk = piv;
        if (!(pk > 0.0)) {                       // dpotrf info != 0  -> jitchol retry on the host side
          if (lane == 0 && info[hj] == 0) info[hj] = k0 + c0 + k + 1;
          pk = 1.0;
        }
        // the dependency chain of the whole block runs through here, 128 times: pivot -> 1/sqrt -> scaled column ->
        // next pivot.  Only rsqrt and one multiply sit on it; the square root itself and the refined reciprocal are
        // needed by lane k's stores alone.
        const double rs = rsqrt(pk);
        const double ak = a[k] * rs;              // column k of L (meaningful for lanes > k)
        if (k + 1 < PSB) {
          // lane k + 1 owns both L[k+1][k] (its ak) and A[k+1][k+1]: the next pivot needs no other lane
          piv = __shfl_sync(0xffffffffu, fma(-ak, ak, a[k + 1]), k + 1);
        }
        double sq = pk * rs;
        sq = fma(fma(-sq, sq, pk), 0.5 * rs, sq);            // sqrt(pivot) to the last bit or so
        if (lane == k) dinv[c0 + k] = fma(fma(-sq, rs, 1.0), rs, rs);
        a[k] = (lane == k) ? sq : ak;
        Ls[k * PSB + lane] = a[k];
        __syncwarp();
        if (k + 1 < PSB) {
#pragma unroll
          for (int c2 = (k + 1) & ~1; c2 < PSB; c2 += 2) {  // lanes < c2 carry don't-care values, masked at the store
            const double2 l2 = *reinterpret_cast<const double2*>(Ls + k * PSB + c2);
            if (c2 >= k + 1) a[c2] = fma(-ak, l2.x, a[c2]);
            a[c2 + 1] = fma(-ak, l2.y, a[c2 + 1]);
          }
        }
      }
#pragma unroll
      for (int q = 0; q < PSB; q += 2)
        *reinterpret_cast<double2*>(T + (c0 + lane) * DLD + c0 + q) =
            make_double2((q <= lane) ? a[q] : 0.0, (q + 1 <= lane) ? a[q + 1] : 0.0);
    }
    __syncthreads();
    const int w0 = c0 + PSB;
    {
      // forward substitution  y L^T = b,  thread per right-hand side, in update form (the multiply-adds of a step are
      // independent), L broadcast from shared memory.  Warps 1 .. take the rows of the panel below the sub-block
      // (P = A L^-T); the next warp takes the rows of the identity, which gives the sub-block's INVERSE one column per
      // thread -- the same instruction stream, so it costs no extra phase (and no cold code) on the critical path.
      const int idx = tid - 32, nrows = TILE - w0;
      const bool is_row = tid >= 32 && idx < nrows;
      const bool is_inv = tid >= 32 && idx >= nrows && idx < nrows + PSB;
      if (is_row || is_inv) {
        const int r = w0 + idx;
        double a[PSB];
#pragma unroll
        for (int q = 0; q < PSB; q += 2) {
          double2 v = make_double2((q == idx - nrows) ? 1.0 : 0.0, (q + 1 == idx - nrows) ? 1.0 : 0.0);
          if (is_row) v = *reinterpret_cast<const double2*>(T + r * DLD + c0 + q);
          a[q] = v.x;
          a[q + 1] = v.y;
        }
#pragma unroll
        for (int k = 0; k < PSB; ++k) {
          a[k] *= dinv[c0 + k];
#pragma unroll
          for (int k2 = (k + 1) & ~1; k2 < PSB; k2 += 2) {
            const double2 l2 = *reinterpret_cast<const double2*>(Ls + k * PSB + k2);
            if (k2 >= k + 1) a[k2] = fma(-a[k], l2.x, a[k2]);
            a[k2 + 1] = fma(-a[k], l2.y, a[k2 + 1]);
          }
        }
        if (is_row) {
#pragma unroll
          for (int q = 0; q < PSB; q += 2) *reinterpret_cast<double2*>(T + r * DLD + c0 + q) = make_double2(a[q], a[q + 1]);
        } else {
          double* Xs = Xb + (c0 / PSB) * (PSB * PSB) + (idx - nrows);      // X[q][c]: exactly 0 above the diagonal
#pragma unroll
          for (int q = 0; q < PSB; ++q) Xs[q * PSB] = a[q];
        }
      }
    }
    if (w0 >= TILE) break;
    __syncthreads();
    {
      // trailing update  A[r][c] -= sum_k P[r][k] P[c][k]  on the lower triangle of [w0, TILE)^2: 8 x 8 DMMA tiles
      const int nt = (TILE - w0) >> 3;
      const int ntile = nt * (nt + 1) / 2;
      int bi = 0, bj = 0;
      for (int b = 0; b < warp; ++b)
        if (++bj > bi) { ++bi; bj = 0; }
      for (int b = warp; b < ntile; b += 8) {
        double x0 = 0.0, x1 = 0.0;
        dmma_tile<true>(x0, x1, T + (w0 + 8 * bi) * DLD + c0, DLD, T + (w0 + 8 * bj) * DLD + c0, DLD, PSB, g, t);
        double* Tt = T + (w0 + 8 * bi + g) * DLD + w0 + 8 * bj + 2 * t;
        Tt[0] -= x0;
        Tt[1] -= x1;
        for (int q = 0; q < 8; ++q)
          if (++bj > bi) { ++bi; bj = 0; }
      }
    }
    __syncthreads();
  }
  // write the factor back (lower triangle of the valid part; strict upper and padding -> 0)
  for (int idx = tid; idx < TILE * TILE; idx += 256) {
    const int r = idx >> 7, c = idx & 127;
    Ablk[(int64_t)r * n_pad + c] = (r < nrem && c <= r) ? T[r * DLD + c] : 0.0;
  }
  __syncthreads();

  // ---------------- the four sub-block inverses (Xb, from the solve phases) replace the factor's diagonal sub-blocks ----
  for (int idx = tid; idx < (TILE / PSB) * PSB * PSB; idx += 256) {
    const int sblk = idx >> 10, q = (idx >> 5) & 31, c = idx & 31;
    T[(sblk * PSB + q) * DLD + sblk * PSB + c] = Xb[idx];
  }
  __syncthreads();                                // Lt (in W) is dead from here on: W becomes the product scratch
  // ---------------- 64 x 64 inverses:  X21 = -X22 (L21 X11)  for the sub-block pairs (1,0) and (3,2) ----------------
  {
    const int p = warp >> 2, w4 = warp & 3;       // pair, warp within the pair: output tiles w4, w4 + 4, ... of 16
    const int o = 2 * PSB * p;
    double* Wp = W + p * PSB * WLD;
    double x0[4], x1[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int tt = w4 + 4 * q, ti = tt >> 2, tj = tt & 3;
      x0[q] = x1[q] = 0.0;
      dmma_tile<false>(x0[q], x1[q], T + (o + PSB + 8 * ti) * DLD + o, DLD, T + o * DLD + o + 8 * tj, DLD, PSB, g, t);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int tt = w4 + 4 * q, ti = tt >> 2, tj = tt & 3;
      Wp[(8 * ti + g) * WLD + 8 * tj + 2 * t] = x0[q];
      Wp[(8 * ti + g) * WLD + 8 * tj + 2 * t + 1] = x1[q];
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int tt = w4 + 4 * q, ti = tt >> 2, tj = tt & 3;
      x0[q] = x1[q] = 0.0;
      dmma_tile<false>(x0[q], x1[q], T + (o + PSB + 8 * ti) * DLD + o + PSB, DLD, Wp + 8 * tj, WLD, PSB, g, t);
    }
    __syncthreads();                              // L21 has been consumed by everyone (first product) before it is replaced
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int tt = w4 + 4 * q, ti = tt >> 2, tj = tt & 3;
      T[(o + PSB + 8 * ti + g) * DLD + o + 8 * tj + 2 * t] = -x0[q];
      T[(o + PSB + 8 * ti + g) * DLD + o + 8 * tj + 2 * t + 1] = -x1[q];
    }
  }
  __syncthreads();
  // ---------------- 128 x 128 inverse:  X21 = -X22 (L21 X11)  with 64 x 64 blocks; warp w owns row tile w ----------
  {
    double x0[8], x1[8];
#pragma unroll
    for (int tj = 0; tj < 8; ++tj) {
      x0[tj] = x1[tj] = 0.0;
      dmma_tile<false>(x0[tj], x1[tj], T + (64 + 8 * warp) * DLD, DLD, T + 8 * tj, DLD, 64, g, t);
    }
#pragma unroll
    for (int tj = 0; tj < 8; ++tj) {
      W[(8 * warp + g) * WLD + 8 * tj + 2 * t] = x0[tj];
      W[(8 * warp + g) * WLD + 8 * tj + 2 * t + 1] = x1[tj];
    }
    __syncthreads();
#pragma unroll
    for (int tj = 0; tj < 8; ++tj) {
      x0[tj] = x1[tj] = 0.0;
      dmma_tile<false>(x0[tj], x1[tj], T + (64 + 8 * warp) * DLD + 64, DLD, W + 8 * tj, WLD, 64, g, t);
    }
    // rows 64 + 8 warp .. of the (1,0) block are read only by this warp's own first product, which is complete
#pragma unroll
    for (int tj = 0; tj < 8; ++tj) {
      T[(64 + 8 * warp + g) * DLD + 8 * tj + 2 * t] = -x0[tj];
      T[(64 + 8 * warp + g) * DLD + 8 * tj + 2 * t + 1] = -x1[tj];
    }
  }
  __syncthreads();
  double* Dblk = Dinv + ((int64_t)hj * nb + kb) * TILE * TILE;
  for (int idx = tid; idx < TILE * TILE; idx += 256) {
    const int r = idx >> 7, c = idx & 127;
    Dblk[idx] = (r < nrem && c <= r) ? T[r * DLD + c] : 0.0;
  }
}

__global__ void __launch_bounds__(256) potrf_diag_kernel(double* __restrict__ Lmat, double* __restrict__ Dinv,
                                                         int* __restrict__ info, int n, int n_pad, int nb, int kb,
                                                         OutRun grp, int m) {
  extern __shared__ __align__(16) double T[];
  potrf_block(T, Lmat, Dinv, info, n, n_pad, nb, kb, run_hj(blockIdx.x, grp, m));
}

// ---------------------------------------------------------------------------------------------------
// Panel solve: A[I][K] <- A[I][K] . L_KK^-T  (= A . Dinv^T), I > K.   grid (nb-1-K, H*m)
__global__ void __launch_bounds__(gemm::Tile128::NTHREADS, 1) trsm_panel_kernel(double* __restrict__ Lmat,
                                                                      const double* __restrict__ Dinv, int n_pad,
                                                                      int nb, int kb, OutRun grp, int m) {
  extern __shared__ __align__(16) double smem[];
  const int hj = run_hj(blockIdx.y, grp, m);
  const int I = kb + 1 + blockIdx.x;
  double* Ablk = Lmat + (int64_t)hj * n_pad * n_pad + (int64_t)I * TILE * n_pad + (int64_t)kb * TILE;
  const double* D = Dinv + ((int64_t)hj * nb + kb) * TILE * TILE;
  double acc[8][4][2];
  gemm::zero_acc(acc);
  // A(m,k) = Ablk[m*n_pad + k] (m-major) ; B(k,n) = Dinv[n][k] (n-major)
  gemm::mainloop<gemm::Tile128, false, false>(acc, Ablk, n_pad, D, TILE, 0, TILE, smem);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const int mbase = (warp >> 2) * 64, nbase = (warp & 3) * 32;
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int r = mbase + 8 * i + g, c = nbase + 8 * j + 2 * t;
      *reinterpret_cast<double2*>(Ablk + (int64_t)r * n_pad + c) = make_double2(acc[i][j][0], acc[i][j][1]);
    }
}

// Trailing update: A[I][J] -= P_I . P_J^T for K < J <= I.   grid (#pairs, H*m)
__global__ void __launch_bounds__(gemm::Tile128::NTHREADS, 1) syrk_update_kernel(double* __restrict__ Lmat, int n_pad, int nb,
                                                                       int kb, OutRun grp, int m,
                                                                       double* __restrict__ Dinv, int* __restrict__ info,
                                                                       int n) {
  extern __shared__ __align__(16) double smem[];
  const int hj = run_hj(blockIdx.y, grp, m);
  // decode the lower-triangular pair index
  int p = blockIdx.x;
  int rr = (int)((sqrt(8.0 * (double)p + 1.0) - 1.0) * 0.5);
  while ((rr + 1) * (rr + 2) / 2 <= p) ++rr;
  while (rr * (rr + 1) / 2 > p) --rr;
  const int cc = p - rr * (rr + 1) / 2;
  const int I = kb + 1 + rr, J = kb + 1 + cc;
  double* base = Lmat + (int64_t)hj * n_pad * n_pad;
  const double* PI = base + (int64_t)I * TILE * n_pad + (int64_t)kb * TILE;
  const double* PJ = base + (int64_t)J * TILE * n_pad + (int64_t)kb * TILE;
  double* C = base + (int64_t)I * TILE * n_pad + (int64_t)J * TILE;
  // acc starts as -C and the product is added, so the tile is read BEFORE the contraction (its latency hides behind the
  // operand pipeline's own prologue) and the epilogue only stores: with K = 128 the read-modify-write after the loop was
  // a quarter of the kernel
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const int mbase = (warp >> 2) * 64, nbase = (warp & 3) * 32;
  double acc[8][4][2];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = mbase + 8 * i + g, c = nbase + 8 * j + 2 * t;
      const double2 old = *reinterpret_cast<const double2*>(C + (int64_t)r * n_pad + c);
      acc[i][j][0] = -old.x;
      acc[i][j][1] = -old.y;
    }
  gemm::mainloop<gemm::Tile128, false, false>(acc, PI, n_pad, PJ, n_pad, 0, TILE, smem);
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = mbase + 8 * i + g, c = nbase + 8 * j + 2 * t;
      *reinterpret_cast<double2*>(C + (int64_t)r * n_pad + c) = make_double2(-acc[i][j][0], -acc[i][j][1]);
    }
  // LOOK-AHEAD: tile 0 is the next diagonal block (kb+1, kb+1), now final.  Its owner factors and inverts it right here,
  // while the other CTAs of this launch are still updating the rest of the trailing matrix, so the diagonal-block step
  // (H*m CTAs, ~46 us, nb times on the chain of every factorisation) no longer has a launch of its own after the first.
  if (blockIdx.x == 0) {
    __syncthreads();                             // the tile's stores are visible to the whole CTA; smem is free (mainloop)
    potrf_block(smem, Lmat, Dinv, info, n, n_pad, nb, kb + 1, hj);
  }
}

// ---------------------------------------------------------------------------------------------------
// Blocked inverse of L.  Diagonal blocks come from Dinv; block row I is built from rows < I:
//   S[I][J]    = sum_{T=J}^{I-1} L[I][T] . Linv[T][J]          (step 1, stored in place of Linv[I][J])
//   Linv[I][J] = -Dinv_I . S[I][J]                              (step 2)
__global__ void linv_init_kernel(double* __restrict__ Linv, const double* __restrict__ Dinv, int n_pad, int nb, OutRun grp,
                                 int m) {
  const int hj = run_hj(blockIdx.y, grp, m), kb = blockIdx.x;
  const double* D = Dinv + ((int64_t)hj * nb + kb) * TILE * TILE;
  double* dst = Linv + (int64_t)hj * n_pad * n_pad + (int64_t)kb * TILE * n_pad + (int64_t)kb * TILE;
  for (int idx = threadIdx.x; idx < TILE * TILE; idx += blockDim.x) {
    int r = idx >> 7, c = idx & 127;
    dst[(int64_t)r * n_pad + c] = D[idx];
  }
}

// Merge step of the recursive inverse.  With L = [[L11, 0], [L21, L22]] and X11 = L11^-1, X22 = L22^-1 known,
//   X21 = -X22 (L21 X11).
// Level b (= 1, 2, 4, ... blocks of 128): the groups [o, o + 2b) of block rows, o = 0, 2b, ..., merge their halves, all
// groups and all matrices in one launch per product -- 2 ceil(log2 nb) launches whose tiles are all independent, instead
// of the 2 (nb - 1) launches of a row-by-row recursion whose longest tile grows with the row.
//   STEP 1:  Tm[I][J] = sum_{T = J}^{o+b-1} L[I][T] X[T][J]        (I in the lower half, J in the upper half)
//            kept TRANSPOSED in the unused mirror block (J, I) of Lmat (nothing reads Lmat above the diagonal)
//   STEP 2:  X[I][J]  = -sum_{T = o+b}^{I} X[I][T] Tm[T][J]
// grid.x = tile rank * Hm + hj, heaviest tiles (longest K) first.
template <int STEP>
__global__ void __launch_bounds__(gemm::Tile128::NTHREADS, 1) linv_merge_kernel(double* __restrict__ Lmat,
                                                                      double* __restrict__ Linv, int n_pad, int nb, int b,
                                                                      int Hm, OutRun grp, int m) {
  extern __shared__ __align__(16) double smem[];
  const int hj = run_hj(blockIdx.x % Hm, grp, m);              // Hm = matrices of this launch (H * grp.cnt)
  const int rank = blockIdx.x / Hm;
  const int ngroups = (nb - b + 2 * b - 1) / (2 * b);
  // rank -> (heavy index, group, light index): K depends on j for STEP 1 (small j heavy), on i for STEP 2 (large i heavy)
  const int hv = rank / (ngroups * b), rem = rank - hv * (ngroups * b);
  const int bg = rem / b, lt = rem - bg * b;      // block-row group of this level
  const int o = bg * 2 * b;
  const int i = (STEP == 1) ? lt : b - 1 - hv;
  const int j = (STEP == 1) ? hv : lt;
  const int I = o + b + i, J = o + j;
  if (I >= nb) return;                             // the last group may have a short lower half
  double* Lb = Lmat + (int64_t)hj * n_pad * n_pad;
  double* Li = Linv + (int64_t)hj * n_pad * n_pad;
  double acc[8][4][2];
  gemm::zero_acc(acc);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const int mbase = (warp >> 2) * 64, nbase = (warp & 3) * 32;
  if (STEP == 1) {
    // A(m,k) = L[I*128+m][k] (m-major) ; B(k,n) = X[k][J*128+n] (k-major) ; k in [J*128, (o+b)*128)
    gemm::mainloop<gemm::Tile128, false, true>(acc, Lb + (int64_t)I * TILE * n_pad, n_pad, Li + (int64_t)J * TILE, n_pad,
                                               J * TILE, (o + b) * TILE, smem);
    double* C = Lb + (int64_t)J * TILE * n_pad + (int64_t)I * TILE;      // Tm^T: element (r, c) at C[c * n_pad + r]
#pragma unroll
    for (int ii = 0; ii < 8; ++ii)
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        const int r = mbase + 8 * ii + g, c = nbase + 8 * jj + 2 * t;
        C[(int64_t)c * n_pad + r] = acc[ii][jj][0];
        C[(int64_t)(c + 1) * n_pad + r] = acc[ii][jj][1];
      }
  } else {
    // A(m,k) = X[I*128+m][k] (m-major) ; B(k,n) = Tm[k][J*128+n] = Lmat[(J*128+n)*n_pad + k] (n-major) ; k in [(o+b)*128, (I+1)*128)
    gemm::mainloop<gemm::Tile128, false, false>(acc, Li + (int64_t)I * TILE * n_pad, n_pad, Lb + (int64_t)J * TILE * n_pad, n_pad,
                                                (o + b) * TILE, (I + 1) * TILE, smem);
    double* C = Li + (int64_t)I * TILE * n_pad + (int64_t)J * TILE;
#pragma unroll
    for (int ii = 0; ii < 8; ++ii)
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        const int r = mbase + 8 * ii + g, c = nbase + 8 * jj + 2 * t;
        *reinterpret_cast<double2*>(C + (int64_t)r * n_pad + c) = make_double2(-acc[ii][jj][0], -acc[ii][jj][1]);
      }
  }
}

// t = Linv . yc   (warp per row)
__global__ void linv_matvec_kernel(const double* __restrict__ Linv, const double* __restrict__ yc, int m, int n_pad,
                                   double* __restrict__ tvec, OutRun grp) {
  const int hj = run_hj(blockIdx.y, grp, m), j = hj % m;
  const int a = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (a >= n_pad) return;
  const int lane = threadIdx.x & 31;
  const double* row = Linv + (int64_t)hj * n_pad * n_pad + (int64_t)a * n_pad;
  const double* y = yc + (int64_t)j * n_pad;
  double s = 0.0;
  for (int b = lane; b <= a; b += 32) s += row[b] * y[b];
  s = warp_sum(s);
  if (lane == 0) tvec[(int64_t)hj * n_pad + a] = s;
}

// alpha = Linv^T . t : CTA = 32 columns x 8 row groups (rows a = b0 + q, b0 + q + 8, ...: each row read is 256
// contiguous bytes), partial sums reduced through shared memory in fixed order
__global__ void __launch_bounds__(256) linv_t_matvec_kernel(const double* __restrict__ Linv, const double* __restrict__ tvec,
                                                            int n_pad, double* __restrict__ alpha, OutRun grp, int m) {
  __shared__ double red[8][33];
  const int hj = run_hj(blockIdx.y, grp, m);
  const int cl = threadIdx.x & 31, q = threadIdx.x >> 5;
  const int b0 = blockIdx.x * 32, b = b0 + cl;
  const double* Li = Linv + (int64_t)hj * n_pad * n_pad;
  const double* tv = tvec + (int64_t)hj * n_pad;
  double s0 = 0.0, s1 = 0.0;
  int a = b0 + q;                                   // rows a < b hold exact zeros above the diagonal
  for (; a + 8 < n_pad; a += 16) {
    s0 = fma(Li[(int64_t)a * n_pad + b], tv[a], s0);
    s1 = fma(Li[(int64_t)(a + 8) * n_pad + b], tv[a + 8], s1);
  }
  if (a < n_pad) s0 = fma(Li[(int64_t)a * n_pad + b], tv[a], s0);
  red[q][cl] = s0 + s1;
  __syncthreads();
  if (q == 0) {
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += red[k][cl];
    alpha[(int64_t)hj * n_pad + b] = s;
  }
}

// ---------------------------------------------------------------------------------------------------
// Appending ONE observation to a factorised model (SURVEY.md 8f rank 4): O(n^2) per output instead of the O(n^3)
// refactorisation.  With Ky' = [[Ky, k], [k^T, k** + noise + 1e-8 (+ jitter)]]:
//   L' = [[L, 0], [l^T, l_nn]],  l = L^-1 k,  l_nn = sqrt(k_nn - l^T l)
//   L'^-1 = [[L^-1, 0], [-(l^T L^-1) / l_nn, 1 / l_nn]]
// (the bordering form of the Cholesky update; GPy ships the rank-1 variant in util/linalg_cython.pyx:24-37).
__global__ void append_xy_kernel(const double* __restrict__ Xold, const double* __restrict__ Yold,
                                 const double* __restrict__ xnew, const double* __restrict__ ynew, int n, int d, int m,
                                 double* __restrict__ Xn, double* __restrict__ Yn) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < (int64_t)(n + 1) * d) Xn[idx] = (idx < (int64_t)n * d) ? Xold[idx] : xnew[idx - (int64_t)n * d];
  if (idx < (int64_t)m * (n + 1)) {
    const int j = (int)(idx / (n + 1)), b = (int)(idx % (n + 1));
    Yn[idx] = (b < n) ? Yold[(int64_t)j * n + b] : ynew[j];
  }
}

// one CTA per (h, j); n = number of points BEFORE the append; Xs / xsq already hold the scaled new point in row n
template <int KIND>
__global__ void __launch_bounds__(256) append_factor_kernel(double* __restrict__ LmatAll, double* __restrict__ LinvAll,
                                                            const double* __restrict__ XsAll,
                                                            const double* __restrict__ xsqAll,
                                                            const OutHyp* __restrict__ hyp, int n, int n_pad, int d,
                                                            int* __restrict__ info, double* __restrict__ work,
                                                            OutRun run, int m) {
  __shared__ double red[8];
  __shared__ double s_lnn;
  const int hj = run_hj(blockIdx.x, run, m), tid = threadIdx.x;
  const OutHyp& hp = hyp[hj];
  double* L = LmatAll + (int64_t)hj * n_pad * n_pad;
  double* Li = LinvAll + (int64_t)hj * n_pad * n_pad;
  const double* Xs = XsAll + (int64_t)hj * n_pad * d;
  const double* xsq = xsqAll + (int64_t)hj * n_pad;
  double* kvec = work + (int64_t)hj * 2 * n_pad;
  double* lvec = kvec + n_pad;
  const double* xn = Xs + (int64_t)n * d;
  for (int b = tid; b < n; b += 256) {                       // k = K(X, x_new)
    double r2;
    if (KIND == BOCF_KERN_SE) {
      r2 = 0.0;
      for (int q = 0; q < d; ++q) {
        const double df = xn[q] - Xs[(int64_t)b * d + q];
        r2 += df * df;
      }
    } else {
      double dot = 0.0;
      for (int q = 0; q < d; ++q) dot += xn[q] * Xs[(int64_t)b * d + q];
      r2 = fmax(-2.0 * dot + (xsq[n] + xsq[b]), 0.0);
    }
    double kv, gdummy;
    kern_eval<KIND, false>(r2, hp.variance, kv, gdummy);
    kvec[b] = kv;
  }
  __syncthreads();
  double ss = 0.0;
  for (int k = tid; k < n; k += 256) {                       // l = L^-1 k  (row k of the lower-triangular inverse)
    const double* row = Li + (int64_t)k * n_pad;
    double acc = 0.0;
    for (int b = 0; b <= k; ++b) acc += row[b] * kvec[b];
    lvec[k] = acc;
    L[(int64_t)n * n_pad + k] = acc;
    ss += acc * acc;
  }
  ss = warp_sum(ss);
  if ((tid & 31) == 0) red[tid >> 5] = ss;
  __syncthreads();
  if (tid == 0) {
    double tot = 0.0;
    for (int w = 0; w < 8; ++w) tot += red[w];
    double d2 = (hp.variance + (hp.noise + 1e-8 + hp.jitter)) - tot;
    if (!(d2 > 0.0)) {                                       // not positive definite: the caller refactorises (jitchol)
      info[hj] = n + 1;
      d2 = 1.0;
    }
    s_lnn = sqrt(d2);
    L[(int64_t)n * n_pad + n] = s_lnn;
    Li[(int64_t)n * n_pad + n] = 1.0 / s_lnn;
  }
  __syncthreads();
  const double inv = 1.0 / s_lnn;
  for (int b = tid; b < n; b += 256) {                       // new row of the inverse: -(l^T L^-1) / l_nn
    double acc = 0.0;
    for (int k = b; k < n; ++k) acc += lvec[k] * Li[(int64_t)k * n_pad + b];
    Li[(int64_t)n * n_pad + b] = -acc * inv;
  }
}

__global__ void copy_factor_kernel(const double* __restrict__ src, int n, int n_pad, int lower_only,
                                   double* __restrict__ dst) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)n * n) return;
  int r = (int)(idx / n), c = (int)(idx % n);
  double v = src[(int64_t)r * n_pad + c];
  if (lower_only && c > r) v = 0.0;
  dst[idx] = v;
}

// ===================================================================================================
int launch_prepare(bocf_model* M, cudaStream_t st) {
  const int Hm = M->H * M->m;
  ybar_kernel<<<M->m, 256, 0, st>>>(M->Y, M->n, M->n_pad, M->m, M->H, M->ybar, M->yc, M->hyp);
  BOCF_LAUNCH_OK("ybar_kernel");
  dim3 grid((unsigned)ceil_div(M->n_pad, 128), (unsigned)Hm);
  scale_inputs_kernel<<<grid, 128, 0, st>>>(M->X, M->n, M->n_pad, M->d, M->hyp, M->Xs, M->xsq);
  BOCF_LAUNCH_OK("scale_inputs_kernel");
  return 0;
}

int launch_gram(bocf_model* M, OutRun grp, cudaStream_t st) {
  const dim3 block(16, 16);
  return for_each_kind_run(M, grp, [&](int kind, OutRun run) -> int {
    const dim3 grid((unsigned)(M->n_pad / 16), (unsigned)(M->n_pad / 16), (unsigned)(M->H * run.cnt));
#define BOCF_GRAM(K) gram_kernel<K><<<grid, block, 0, st>>>(M->Xs, M->xsq, M->hyp, M->n, M->n_pad, M->d, M->Lmat, run, M->m)
    switch (kind) {
      case BOCF_KERN_SE: BOCF_GRAM(BOCF_KERN_SE); break;
      case BOCF_KERN_RBF: BOCF_GRAM(BOCF_KERN_RBF); break;
      case BOCF_KERN_MATERN52: BOCF_GRAM(BOCF_KERN_MATERN52); break;
      case BOCF_KERN_MATERN32: BOCF_GRAM(BOCF_KERN_MATERN32); break;
      default: set_error("unknown kernel kind"); return -1;
    }
#undef BOCF_GRAM
    BOCF_LAUNCH_OK("gram_kernel");
    return 0;
  });
}

// Two output groups on two streams when there are enough matrices for it to pay (see GroupStreams, model.h).
int for_each_output_group(bocf_model* M, cudaStream_t st, int (*f)(bocf_model*, OutRun, cudaStream_t, void*), void* ctx) {
  if (M->m < 4 || M->H * M->m < 8 || M->nb < 3) return f(M, OutRun{0, M->m}, st, ctx);
  GroupStreams& gs = M->gs;
  if (!gs.side) {
    BOCF_CUDA_OK(cudaStreamCreateWithFlags(&gs.side, cudaStreamNonBlocking));
    BOCF_CUDA_OK(cudaEventCreateWithFlags(&gs.fork, cudaEventDisableTiming));
    BOCF_CUDA_OK(cudaEventCreateWithFlags(&gs.join, cudaEventDisableTiming));
  }
  const int half = M->m / 2;
  BOCF_CUDA_OK(cudaEventRecord(gs.fork, st));
  BOCF_CUDA_OK(cudaStreamWaitEvent(gs.side, gs.fork, 0));
  int rc = f(M, OutRun{0, half}, st, ctx);
  const int rc2 = f(M, OutRun{half, M->m - half}, gs.side, ctx);
  BOCF_CUDA_OK(cudaEventRecord(gs.join, gs.side));             // always rejoin, also after a failed launch
  BOCF_CUDA_OK(cudaStreamWaitEvent(st, gs.join, 0));
  return rc ? rc : rc2;
}

constexpr int SYRK_SMEM = POTRF_SMEM > gemm::Tile128::SMEM_BYTES ? POTRF_SMEM : gemm::Tile128::SMEM_BYTES;
static int set_smem_attrs() {
  // per device: function attributes belong to the device's context (one process may drive several GPUs)
  static bool done_dev[64] = {false};
  int dev = 0;
  BOCF_CUDA_OK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) {
    set_error("unsupported device ordinal");
    return BOCF_ERR_INVALID;
  }
  bool& done = done_dev[dev];
  if (done) return 0;
  BOCF_CUDA_OK(cudaFuncSetAttribute(potrf_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, POTRF_SMEM));
  BOCF_CUDA_OK(cudaFuncSetAttribute(trsm_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm::Tile128::SMEM_BYTES));
  BOCF_CUDA_OK(cudaFuncSetAttribute(syrk_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SYRK_SMEM));
  BOCF_CUDA_OK(cudaFuncSetAttribute(linv_merge_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm::Tile128::SMEM_BYTES));
  BOCF_CUDA_OK(cudaFuncSetAttribute(linv_merge_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm::Tile128::SMEM_BYTES));
  done = true;
  return 0;
}

int launch_cholesky(bocf_model* M, OutRun grp, cudaStream_t st) {
  if (int rc = set_smem_attrs()) return rc;
  const int Hg = M->H * grp.cnt, nb = M->nb;
  // block 0 has its own launch; every later diagonal block is factored by the trailing update that completes it
  potrf_diag_kernel<<<Hg, 256, POTRF_SMEM, st>>>(M->Lmat, M->Dinv, M->info, M->n, M->n_pad, nb, 0, grp, M->m);
  BOCF_LAUNCH_OK("potrf_diag_kernel");
  for (int kb = 0; kb + 1 < nb; ++kb) {
    const int rem = nb - 1 - kb;
    trsm_panel_kernel<<<dim3(rem, Hg), gemm::Tile128::NTHREADS, gemm::Tile128::SMEM_BYTES, st>>>(M->Lmat, M->Dinv, M->n_pad, nb, kb, grp, M->m);
    BOCF_LAUNCH_OK("trsm_panel_kernel");
    syrk_update_kernel<<<dim3(rem * (rem + 1) / 2, Hg), gemm::Tile128::NTHREADS, SYRK_SMEM, st>>>(M->Lmat, M->n_pad, nb, kb, grp, M->m,
                                                                                                 M->Dinv, M->info, M->n);
    BOCF_LAUNCH_OK("syrk_update_kernel");
  }
  return 0;
}

int launch_inverse_and_alpha(bocf_model* M, OutRun grp, cudaStream_t st) {
  if (int rc = set_smem_attrs()) return rc;
  const int Hg = M->H * grp.cnt, nb = M->nb;
  // Linv above the block diagonal stays zero from its allocation (bocf_model_factorize); every block on or below it is
  // rewritten here
  linv_init_kernel<<<dim3(nb, Hg), 256, 0, st>>>(M->Linv, M->Dinv, M->n_pad, nb, grp, M->m);
  BOCF_LAUNCH_OK("linv_init_kernel");
  for (int b = 1; b < nb; b *= 2) {
    const int ngroups = (nb - b + 2 * b - 1) / (2 * b);
    const unsigned grid = (unsigned)(ngroups * b * b * Hg);
    linv_merge_kernel<1><<<grid, gemm::Tile128::NTHREADS, gemm::Tile128::SMEM_BYTES, st>>>(M->Lmat, M->Linv, M->n_pad, nb, b, Hg, grp, M->m);
    BOCF_LAUNCH_OK("linv_merge_kernel<1>");
    linv_merge_kernel<2><<<grid, gemm::Tile128::NTHREADS, gemm::Tile128::SMEM_BYTES, st>>>(M->Lmat, M->Linv, M->n_pad, nb, b, Hg, grp, M->m);
    BOCF_LAUNCH_OK("linv_merge_kernel<2>");
  }
  return launch_alpha(M, grp, st);
}

int launch_alpha(bocf_model* M, OutRun grp, cudaStream_t st) {
  const int Hg = M->H * grp.cnt;
  linv_matvec_kernel<<<dim3((unsigned)ceil_div(M->n_pad, 8), Hg), 256, 0, st>>>(M->Linv, M->yc, M->m, M->n_pad, M->tvec, grp);
  BOCF_LAUNCH_OK("linv_matvec_kernel");
  linv_t_matvec_kernel<<<dim3((unsigned)(M->n_pad / 32), Hg), 256, 0, st>>>(M->Linv, M->tvec, M->n_pad, M->alpha, grp, M->m);
  BOCF_LAUNCH_OK("linv_t_matvec_kernel");
  return 0;
}

// n_old = points before the append; M->n, M->X, M->Y already describe the n_old + 1 points
int launch_append(bocf_model* M, int n_old, double* work, cudaStream_t st) {
  const int Hm = M->H * M->m;
  BOCF_CUDA_OK(cudaMemsetAsync(M->info, 0, sizeof(int) * Hm, st));
  if (int rc = launch_prepare(M, st)) return rc;             // ybar, centred y, scaled inputs incl. the new row
  const int rc_runs = for_each_kind_run(M, [&](int kind, OutRun run) -> int {
    const int blocks = M->H * run.cnt;
#define BOCF_APPEND(K) \
  append_factor_kernel<K><<<blocks, 256, 0, st>>>(M->Lmat, M->Linv, M->Xs, M->xsq, M->hyp, n_old, M->n_pad, M->d, M->info, work, run, M->m)
    switch (kind) {
      case BOCF_KERN_SE: BOCF_APPEND(BOCF_KERN_SE); break;
      case BOCF_KERN_RBF: BOCF_APPEND(BOCF_KERN_RBF); break;
      case BOCF_KERN_MATERN52: BOCF_APPEND(BOCF_KERN_MATERN52); break;
      default: BOCF_APPEND(BOCF_KERN_MATERN32); break;
    }
#undef BOCF_APPEND
    BOCF_LAUNCH_OK("append_factor_kernel");
    return 0;
  });
  if (rc_runs) return rc_runs;
  return launch_alpha(M, OutRun{0, M->m}, st);
}

int launch_append_xy(const double* Xold, const double* Yold, const double* xnew, const double* ynew, int n, int d, int m,
                     double* Xn, double* Yn, cudaStream_t st) {
  const int64_t work = (int64_t)(n + 1) * (d > m ? d : m);
  append_xy_kernel<<<(unsigned)ceil_div(work, 256), 256, 0, st>>>(Xold, Yold, xnew, ynew, n, d, m, Xn, Yn);
  BOCF_LAUNCH_OK("append_xy_kernel");
  return 0;
}

int launch_copy_factor(bocf_model* M, int hj, double* L, double* Linv, double* alpha, cudaStream_t st) {
  const int64_t nn = (int64_t)M->n * M->n;
  const unsigned blocks = (unsigned)ceil_div(nn, 256);
  if (L) {
    copy_factor_kernel<<<blocks, 256, 0, st>>>(M->Lmat + (int64_t)hj * M->n_pad * M->n_pad, M->n, M->n_pad, 1, L);
    BOCF_LAUNCH_OK("copy_factor_kernel");
  }
  if (Linv) {
    copy_factor_kernel<<<blocks, 256, 0, st>>>(M->Linv + (int64_t)hj * M->n_pad * M->n_pad, M->n, M->n_pad, 1, Linv);
    BOCF_LAUNCH_OK("copy_factor_kernel");
  }
  if (alpha)
    BOCF_CUDA_OK(cudaMemcpyAsync(alpha, M->alpha + (int64_t)hj * M->n_pad, sizeof(double) * M->n, cudaMemcpyDeviceToDevice, st));
  return 0;
}

}  // namespace bocf
