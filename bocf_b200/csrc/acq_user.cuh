// acq_user.cuh -- the MC acquisition and utility kernels of a USER-DEFINED composite U(theta, y).
//
// Not compiled by nvcc: the text is embedded in libbocf_b200.so and compiled at run time by NVRTC (jit.cu), for
// sm_100a to a cubin, appended to the user's source, which defines
//   __device__ double bocf_U (const double* theta, const double* y);               // y[0 .. BOCF_M)
//   __device__ void   bocf_dU(const double* theta, const double* y, double* grad);  // grad[j] = dU / dy_j
// with BOCF_M (the number of outputs) given on the command line (include/bocf_b200.h).  It is self-contained: NVRTC
// compiles it without host or toolkit headers.
//
// mc_acq_user_kernel mirrors acq.cu's mc_acq_kernel -- the same MODE meanings, launch shapes (MCB, NW), sample walk,
// f* / PI-jitter / strict-indicator semantics, ragged S, scale / accumulate and gradient weights -- with the separable
// sum over comp_phi replaced by ONE call of bocf_U per (candidate, sample) on y = mu + sigma z, built in registers, and
// the per-output comp_dphi by ONE call of bocf_dU per active sample, whose gradient feeds the per-output sums
// A_j = sum_s 1 dU/dy_j and B_j = sum_s 1 dU/dy_j Z_sj exactly as the built-in kernel's do.

namespace bocf_user {

typedef long long i64;
constexpr int MC_WARPS = 8;    // as acq.cu
constexpr int MAXD = 16;       // as model.h
constexpr int MAXM = 64;
static_assert(BOCF_M >= 1 && BOCF_M <= MAXM, "BOCF_M must be in [1, 64]");

struct MuSigma {
  double mu, sg;
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// MODE: 0 = EI value only, 1 = EI value + gradient, 2 = PI value, 3 = mean utility value, 4 = mean utility value +
//       gradient, 5 / 6 = as 1 / 4 with the gradient left as per-(candidate, output) weights WA, WB (acq.cu)
template <int MODE, int MCB, int NW>
__global__ void __launch_bounds__(MC_WARPS * 32) mc_acq_user_kernel(
    const double* __restrict__ mean, const double* __restrict__ var, const double* __restrict__ dmean,
    const double* __restrict__ dvar, i64 Nc, i64 Nvalid, int d, const double* __restrict__ Zt, int S,
    const double* __restrict__ theta, int L, int p, const double* __restrict__ weight,
    const double* __restrict__ fstar, double scale, int accumulate, double* __restrict__ acq,
    double* __restrict__ dacq, double* __restrict__ wa_out, double* __restrict__ wb_out) {
  constexpr int M = BOCF_M;
  constexpr int MW = (M + 31) / 32;                            // weight slots per lane: lane (j & 31) keeps output j
  constexpr bool WITH_GRAD = (MODE == 1 || MODE == 4), WEIGHTS = (MODE == 5 || MODE == 6);
  constexpr bool PLAIN_U = (MODE == 3 || MODE == 4 || MODE == 6);
  static_assert(NW == 1 || (NW == MC_WARPS && MCB == 1), "a block shares one candidate or none");
  __shared__ MuSigma s_ms[MC_WARPS][M][MCB];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const i64 i0 = (NW == 1) ? ((i64)blockIdx.x * MC_WARPS + warp) * MCB : (i64)blockIdx.x;
  if (i0 >= Nvalid) return;
  const int nc = (Nvalid - i0 < MCB) ? (int)(Nvalid - i0) : MCB;
  for (int idx = lane; idx < M * MCB; idx += 32) {
    const int j = idx / MCB, c = idx - j * MCB;
    const i64 i = i0 + (c < nc - 1 ? c : nc - 1);            // ragged tail: replicate the last valid candidate
    s_ms[warp][j][c].mu = mean[(i64)j * Nc + i];
    s_ms[warp][j][c].sg = sqrt(var[(i64)j * Nc + i]);
  }
  __syncwarp();

  double val_total[MCB];
  double grad_q[MCB];
  double wa[MCB][MW], wb[MCB][MW];
#pragma unroll
  for (int c = 0; c < MCB; ++c) {
    val_total[c] = grad_q[c] = 0.0;
#pragma unroll
    for (int w = 0; w < MW; ++w) wa[c][w] = wb[c][w] = 0.0;
  }
  for (int l = 0; l < L; ++l) {
    const double* th = theta + (i64)l * p;
    const double wl = weight[l];
    const double fs = PLAIN_U ? 0.0 : ((MODE == 2) ? fstar[l] + 1e-6 : fstar[l]);
    double val_l[MCB];
#pragma unroll
    for (int c = 0; c < MCB; ++c) val_l[c] = 0.0;
    for (int sb = 0; sb < S; sb += 1024) {
      unsigned mask[MCB];
#pragma unroll
      for (int c = 0; c < MCB; ++c) mask[c] = 0u;
      const int kbeg = (NW == 1) ? 0 : warp * (32 / NW), kend = (NW == 1) ? 32 : kbeg + 32 / NW;
      // one sample per trip and one candidate per trip, neither unrolled, so bocf_U and bocf_dU are each inlined ONCE
      // (NVRTC's compile time and the register count grow with every inlined copy); the per-candidate accumulators
      // are selected with compile-time indices.  A sample's BOCF_M base-sample loads are in flight together.
#pragma unroll 1
      for (int k = kbeg; k < kend; ++k) {
        const int sidx = sb + k * 32 + lane;
        if (sidx >= S) continue;
        double z[M];
#pragma unroll
        for (int j = 0; j < M; ++j) z[j] = Zt[(i64)j * S + sidx];
#pragma unroll 1
        for (int c = 0; c < MCB; ++c) {
          double y[M];
#pragma unroll
          for (int j = 0; j < M; ++j) y[j] = s_ms[warp][j][c].mu + s_ms[warp][j][c].sg * z[j];
          const double U = bocf_U(th, y);
          double v;
          bool active;
          if (MODE == 2) {
            v = ((U - fs) > 0.0) ? 1.0 : 0.0;
            active = false;
          } else if (PLAIN_U) {
            v = U;
            active = true;
          } else {
            v = fmax(U - fs, 0.0);
            active = (U > fs);                                    // strict >
          }
#pragma unroll
          for (int cc = 0; cc < MCB; ++cc)
            if (cc == c) {
              val_l[cc] += v;
              if (active) mask[cc] |= (1u << k);
            }
        }
      }
      if (WITH_GRAD || WEIGHTS) {
#pragma unroll 1
        for (int c = 0; c < nc; ++c) {
          unsigned mk = 0u;
          double gq = 0.0;
#pragma unroll
          for (int cc = 0; cc < MCB; ++cc)
            if (cc == c) {
              mk = mask[cc];
              gq = grad_q[cc];
            }
          if (!__any_sync(0xffffffffu, mk != 0u)) continue;
          const i64 i = i0 + c;
          double A[M], B[M];
#pragma unroll
          for (int j = 0; j < M; ++j) A[j] = B[j] = 0.0;
          // this lane's active samples, in ascending order: one bocf_dU each
          for (unsigned rem = mk; rem != 0u; rem &= rem - 1u) {
            const int k = __ffs((int)rem) - 1;
            const int sidx = sb + k * 32 + lane;
            double y[M], g[M];
#pragma unroll
            for (int j = 0; j < M; ++j) y[j] = s_ms[warp][j][c].mu + s_ms[warp][j][c].sg * Zt[(i64)j * S + sidx];
            bocf_dU(th, y, g);
#pragma unroll
            for (int j = 0; j < M; ++j) {
              A[j] += g[j];
              B[j] += g[j] * Zt[(i64)j * S + sidx];
            }
          }
          __syncwarp();
#pragma unroll
          for (int j = 0; j < M; ++j) {
            const double Aj = warp_sum(A[j]);
            const double Bj = warp_sum(B[j]);
            const double sg = s_ms[warp][j][c].sg;
            if (WEIGHTS) {
              if (lane == (j & 31)) {
#pragma unroll
                for (int cc = 0; cc < MCB; ++cc)
                  if (cc == c) {
                    wa[cc][j >> 5] += wl * Aj;
                    wb[cc][j >> 5] += wl * (Bj * (0.5 / sg));
                  }
              }
            } else if (lane < d) {
              const i64 o = ((i64)j * Nc + i) * d + lane;
              gq += wl * (Aj * dmean[o] + Bj * (0.5 / sg) * dvar[o]);
            }
          }
          if (WITH_GRAD) {
#pragma unroll
            for (int cc = 0; cc < MCB; ++cc)
              if (cc == c) grad_q[cc] = gq;
          }
        }
      }
    }
#pragma unroll
    for (int c = 0; c < MCB; ++c) val_total[c] += wl * warp_sum(val_l[c]);
  }
  if (NW > 1) {
    // add the warps' partial sums in fixed order; warp 0 then writes like the single-warp path
    __shared__ double r_val[MC_WARPS], r_grad[MC_WARPS][MAXD], r_wa[MC_WARPS][MW * 32], r_wb[MC_WARPS][MW * 32];
    if (lane == 0) r_val[warp] = val_total[0];
    if (WITH_GRAD && lane < MAXD) r_grad[warp][lane] = grad_q[0];
    if (WEIGHTS) {
#pragma unroll
      for (int w = 0; w < MW; ++w) {
        r_wa[warp][w * 32 + lane] = wa[0][w];
        r_wb[warp][w * 32 + lane] = wb[0][w];
      }
    }
    __syncthreads();
    if (warp != 0) return;
    val_total[0] = 0.0;
    grad_q[0] = 0.0;
#pragma unroll
    for (int w = 0; w < MW; ++w) wa[0][w] = wb[0][w] = 0.0;
    for (int k = 0; k < MC_WARPS; ++k) {
      val_total[0] += r_val[k];
      if (WITH_GRAD && lane < MAXD) grad_q[0] += r_grad[k][lane];
      if (WEIGHTS) {
#pragma unroll
        for (int w = 0; w < MW; ++w) {
          wa[0][w] += r_wa[k][w * 32 + lane];
          wb[0][w] += r_wb[k][w * 32 + lane];
        }
      }
    }
  }
#pragma unroll
  for (int c = 0; c < MCB; ++c) {
    if (c >= nc) break;
    const i64 i = i0 + c;
    if (lane == 0) {
      const double v = val_total[c] * scale;
      acq[i] = accumulate ? acq[i] + v : v;
    }
    if (WITH_GRAD && lane < d) {
      const double gq = grad_q[c] * scale;
      dacq[i * d + lane] = accumulate ? dacq[i * d + lane] + gq : gq;
    }
    if (WEIGHTS) {
#pragma unroll
      for (int w = 0; w < MW; ++w) {
        const int j = w * 32 + lane;
        if (j < M) {
          wa_out[(i64)j * Nc + i] = wa[c][w] * scale;
          wb_out[(i64)j * Nc + i] = wb[c][w] * scale;
        }
      }
    }
  }
}

// out [L x N] = U(theta_l, Y[:, i]);  Y is BOCF_M x N.  grid (ceil(N / 256), L)
__global__ void utility_eval_user_kernel(const double* __restrict__ Y, i64 N, const double* __restrict__ theta, int p,
                                         double* __restrict__ out) {
  const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  const int l = blockIdx.y;
  if (i >= N) return;
  double y[BOCF_M];
#pragma unroll
  for (int j = 0; j < BOCF_M; ++j) y[j] = Y[(i64)j * N + i];
  out[(i64)l * N + i] = bocf_U(theta + (i64)l * p, y);
}

// out [L x BOCF_M x N] = dU / dy_j (theta_l, Y[:, i])
__global__ void utility_grad_eval_user_kernel(const double* __restrict__ Y, i64 N, const double* __restrict__ theta,
                                              int p, double* __restrict__ out) {
  const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  const int l = blockIdx.y;
  if (i >= N) return;
  double y[BOCF_M], g[BOCF_M];
#pragma unroll
  for (int j = 0; j < BOCF_M; ++j) y[j] = Y[(i64)j * N + i];
  bocf_dU(theta + (i64)l * p, y, g);
#pragma unroll
  for (int j = 0; j < BOCF_M; ++j) out[((i64)l * BOCF_M + j) * N + i] = g[j];
}

}  // namespace bocf_user
