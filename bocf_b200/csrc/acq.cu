// acq.cu -- acquisition kernels (north-star subsystem 3, SURVEY K3 / K3' / C1-local).
//
// mc_acq_kernel : EI-CF / PI-CF.  One warp per candidate; lanes split the S base samples (coalesced
//   reads of the transposed Z), h = mu + sigma*Z per output, separable composite U = sum_j phi_j(h_j),
//   improvement max(U - f*, 0) (or the PI indicator), warp-shuffle reduction over samples, and the
//   pathwise gradient  sum_s 1[U>f*] dU(h)^T (dmu + (Z/(2 sigma)) * dvar)  folded into per-output
//   sums A_j = sum_s 1 dphi_j, B_j = sum_s 1 dphi_j Z_sj  (uEI_noiseless.py:71-80,148-166; uPI.py:74-83).
//   MODE 3 / 4 drop the improvement: plain sum_s U(theta, mu + sigma Z_s) and its pathwise gradient, the 50-sample MC
//   branch of cbo._current_marginal_argmax (cbo.py:203-231).
// ma_acq_kernel : analytic EI / PI of theta^T y (maEI.py:81-126, maPI.py, EI.py, PI.py).
// psi_acq_kernel: closed-form E[U(theta, y)] under the posterior (the psi / psi_gradient pairs of test_1a.py:100-113,
//   test_2a.py:70-83, test_5a.py:64-77) and the posterior-mean branch for linear utilities (cbo.py:126-168,170-198).
// topk kernels  : local top-k of the acquisition (anchor_points_generator.py:59-64), deterministic ties.
#include <math_constants.h>

#include "model.h"
#include "common.cuh"

namespace bocf {

// ---------------------------------------------------------------------------------------------------
// separable composites: U(theta, y) = sum_j phi_j(y_j)
struct CompCtx {
  double th;     // theta entry relevant for output j (theta_j, or the scalar a for ROSEN)
  double c;      // EXP_COS coefficient c_j
  int lower;     // ROSEN: 1 if j < m/2, 0 if m/2 <= j < 2(m/2), -1 if unused
};

template <int COMP>
__device__ __forceinline__ CompCtx comp_ctx(const double* __restrict__ theta_l, int j, int m) {
  CompCtx c;
  c.th = 0.0;
  c.c = 0.0;
  c.lower = 0;
  if (COMP == BOCF_U_SUMSQ_TARGET || COMP == BOCF_U_LINEAR) c.th = theta_l[j];
  if (COMP == BOCF_U_EXP_COS) {
    const double cc[5] = {1., 2., 5., 2., 3.};
    c.c = cc[j % 5];
  }
  if (COMP == BOCF_U_ROSEN_COMPOSITE) {
    c.th = theta_l[0];
    const int hh = m / 2;
    c.lower = (j < hh) ? 1 : ((j < 2 * hh) ? 0 : -1);
  }
  return c;
}

template <int COMP>
__device__ __forceinline__ double comp_phi(const CompCtx& c, double y) {
  if (COMP == BOCF_U_SUMSQ_TARGET) {
    const double a = y - c.th;
    return -(a * a);
  } else if (COMP == BOCF_U_NEG_SUM_EXP) {
    return -exp(y);
  } else if (COMP == BOCF_U_EXP_COS) {
    return -(c.c * (exp(-y / CUDART_PI) * cos(CUDART_PI * y)));
  } else if (COMP == BOCF_U_ROSEN_COMPOSITE) {
    if (c.lower == 1) {
      const double a = c.th - y;
      return -(a * a);
    }
    if (c.lower == 0) return -(100.0 * (y * y));
    return 0.0;
  } else {
    return c.th * y;
  }
}

template <int COMP>
__device__ __forceinline__ double comp_dphi(const CompCtx& c, double y) {
  if (COMP == BOCF_U_SUMSQ_TARGET) {
    return -2.0 * (y - c.th);
  } else if (COMP == BOCF_U_NEG_SUM_EXP) {
    return -exp(y);
  } else if (COMP == BOCF_U_EXP_COS) {
    const double e = exp(-y / CUDART_PI);
    const double aux = -CUDART_PI * (e * sin(CUDART_PI * y)) - (e * cos(CUDART_PI * y)) / CUDART_PI;
    return -(c.c * aux);
  } else if (COMP == BOCF_U_ROSEN_COMPOSITE) {
    if (c.lower == 1) return 2.0 * (c.th - y);
    if (c.lower == 0) return -200.0 * y;
    return 0.0;
  } else {
    return c.th;
  }
}

// Upper bound of phi_j over the segment [lo, hi] (lo <= hi), and for LINEAR the magnitude max |phi_j| over it (the other
// three are <= 0 everywhere: their magnitude is -bound, formed by the caller).  Exact maxima of the segment, evaluated with
// the rounding error prune_bound_kernel's margin accounts for.
template <int COMP>
__device__ __forceinline__ double comp_seg_max(const CompCtx& c, double lo, double hi, double& mag) {
  mag = 0.0;
  if (COMP == BOCF_U_SUMSQ_TARGET || (COMP == BOCF_U_ROSEN_COMPOSITE && c.lower == 1)) {
    // -(distance from the target to the segment)^2; the negated compares let a NaN through
    const double d1 = lo - c.th, d2 = c.th - hi;
    const double dist = !(d1 <= 0.0) ? d1 : (!(d2 <= 0.0) ? d2 : 0.0);
    return -(dist * dist);
  } else if (COMP == BOCF_U_ROSEN_COMPOSITE) {
    if (c.lower != 0) return 0.0;
    const double dist = !(lo <= 0.0) ? lo : (!(hi >= 0.0) ? -hi : 0.0);
    return -(100.0 * (dist * dist));
  } else if (COMP == BOCF_U_NEG_SUM_EXP) {
    return -exp(lo);
  } else {                                                    // LINEAR
    mag = fabs(c.th) * fmax(fabs(lo), fabs(hi));
    return c.th * ((c.th >= 0.0) ? hi : lo);
  }
}

// ---------------------------------------------------------------------------------------------------
// Survivor flags of the pruned EI-CF / PI-CF sweep (bocf_acq_eval).  mc_acq_kernel forms, per base sample s,
// U_s = sum_j phi_j(mu_j + sigma_j z_sj) with sigma_j^2 the posterior variance (noise added, clipped at 1e-10), and a
// candidate contributes nothing -- value, gradient weights, PI count -- unless some U_s > f* (PI: f* + 1e-6).  Since the
// posterior variance never exceeds the prior one, sigma_j <= smax_j = sqrt(max(sigma_f,j^2 + noise_j, 1e-10)), so
//   U_s <= UB_s = sum_j max_{t in [0, 1]} phi_j(mu_j + t smax_j z_sj),
// a maximum over the segment between mu_j and mu_j + smax_j z_sj with a closed form (comp_seg_max).  A candidate is
// pruned when UB_s + margin <= f* for every hyper-sample, utility parameter and base sample; flags[i] = 1 keeps it.  mu is
// the mean-only pass's, bitwise the mean the sweep uses (posterior.cu); Zt, theta and f* are the sweep's own device slots.
//
// Why the floating-point comparison is safe (u = 2^-53, gamma_k = k u / (1 - k u)):
//  * The segment holds the sweep's y.  mc_acq_kernel computes y = fl(mu + sigma z), contracted to one FMA or not, with
//    sigma = sqrt(var) correctly rounded; its var <= max((sigma_f^2 + noise)(1 + u), 1e-10), so sigma <= smax (1 + 3.1 u).
//    Here smax is inflated by 2^-47 (>= 14 u after rounding), so with P = smax z the sweep's exact sigma z lies strictly
//    between 0 and fl(P), and by monotonicity of rounding y lies between mu and e = fl(mu + fl(P)).  e is formed with
//    __dmul_rn / __dadd_rn so the compiler cannot contract it.  Hence phi_j(y_j) <= the exact maximum over [lo, hi].
//  * SUMSQ_TARGET, ROSEN, NEG_SUM_EXP: every phi_j <= 0.  Each term of the sweep has a relative error <= gamma_3 (a
//    subtraction and a square, or exp within 1 ulp, fused or not) and the sum over m terms adds gamma_(m-1) of the sum of
//    magnitudes, so U_s(computed) <= (1 - gamma_(m+2)) U_s(exact) <= (1 - gamma_(m+2)) UB_s(exact).  The bound here is
//    evaluated the same way, UB(computed) = UB(exact)(1 + eta), |eta| <= gamma_(m+2), both <= 0, which gives
//    U_s(computed) <= UB + 2 gamma_(m+2) |UB| (computed UB).
//  * LINEAR: the sweep and the bound each err by <= gamma_m sum_j |theta_j| max(|lo_j|, |hi_j|) = gamma_m MAG, so
//    U_s(computed) <= UB + 2 gamma_m MAG / (1 - gamma_m) with MAG as computed here.
//  The margin is (4 m + 16) u MAG (MAG = -UB for the first three), over twice what is needed, which also covers the
//  rounding of UB + margin itself; the 1e-300 added to it covers results in the subnormal range, where errors are
//  absolute (<= m * 2^-1072 in all).  A NaN anywhere (input, mean, theta, f*) fails the <= and keeps the candidate.
constexpr int PB_WARPS = 8;
constexpr int PB_MCB = 4;      // candidates per warp (each base sample loaded is applied to all of them)
constexpr int PB_MCU = 4;      // sample groups per trip
// (LINEAR carries the magnitude sums as well, NEG_SUM_EXP sixteen inlined exp: one block per SM keeps them in registers)
template <int COMP>
__global__ void __launch_bounds__(PB_WARPS * 32, (COMP == BOCF_U_LINEAR || COMP == BOCF_U_NEG_SUM_EXP) ? 1 : 2)
    prune_bound_kernel(
    const double* __restrict__ mean, int64_t Nc, int64_t Nvalid, int m, const OutHyp* __restrict__ hyp,
    const double* __restrict__ Zt, int S, const double* __restrict__ theta, int L, int p,
    const double* __restrict__ fstar, int pi, int first, uint8_t* __restrict__ flags) {
  __shared__ double s_mu[PB_WARPS][MAXM][PB_MCB];
  __shared__ double s_sd[MAXM];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int j = threadIdx.x; j < m; j += blockDim.x)
    s_sd[j] = sqrt(fmax(hyp[j].variance + hyp[j].noise, 1e-10)) * (1.0 + 0x1p-47);
  const int64_t i0 = ((int64_t)blockIdx.x * PB_WARPS + warp) * PB_MCB;
  const int nc = (i0 < Nvalid) ? (int)min((int64_t)PB_MCB, Nvalid - i0) : 0;
  for (int idx = lane; idx < m * PB_MCB && nc > 0; idx += 32) {
    const int j = idx / PB_MCB, c = idx - j * PB_MCB;
    s_mu[warp][j][c] = mean[(int64_t)j * Nc + i0 + min(c, nc - 1)];    // ragged tail: replicate the last candidate
  }
  __syncthreads();
  if (nc == 0) return;
  const double cm = (4.0 * m + 16.0) * 0x1p-53;
  bool live[PB_MCB];                                        // warp-uniform
#pragma unroll
  for (int c = 0; c < PB_MCB; ++c) live[c] = (c >= nc);     // replicas count as decided
  bool done = false;
  for (int l = 0; l < L && !done; ++l) {
    const double* th = theta + (int64_t)l * p;
    const double fs = pi ? fstar[l] + 1e-6 : fstar[l];     // as mc_acq_kernel
#pragma unroll 1
    for (int s0 = 0; s0 < S && !done; s0 += 32 * PB_MCU) {
      double ub[PB_MCB][PB_MCU], mg[PB_MCB][PB_MCU];
#pragma unroll
      for (int c = 0; c < PB_MCB; ++c)
#pragma unroll
        for (int u = 0; u < PB_MCU; ++u) ub[c][u] = mg[c][u] = 0.0;
      for (int j = 0; j < m; ++j) {
        const CompCtx cx = comp_ctx<COMP>(th, j, m);
        const double sd = s_sd[j];
        const double* zr = Zt + (int64_t)j * S + s0 + lane;
        double z[PB_MCU];
#pragma unroll
        for (int u = 0; u < PB_MCU; ++u) z[u] = (s0 + u * 32 + lane < S) ? zr[u * 32] : 0.0;
#pragma unroll
        for (int c = 0; c < PB_MCB; ++c) {
          const double mu = s_mu[warp][j][c];
#pragma unroll
          for (int u = 0; u < PB_MCU; ++u) {
            const double e = __dadd_rn(mu, __dmul_rn(sd, z[u]));
            const bool up = z[u] >= 0.0;
            double mag;
            ub[c][u] += comp_seg_max<COMP>(cx, up ? mu : e, up ? e : mu, mag);
            if (COMP == BOCF_U_LINEAR) mg[c][u] += mag;
          }
        }
      }
#pragma unroll
      for (int c = 0; c < PB_MCB; ++c) {
        bool any = false;
#pragma unroll
        for (int u = 0; u < PB_MCU; ++u) {
          const double mag = (COMP == BOCF_U_LINEAR) ? mg[c][u] : -ub[c][u];
          if (s0 + u * 32 + lane < S) any |= !(ub[c][u] + fma(cm, mag, 1e-300) <= fs);
        }
        live[c] = live[c] || __any_sync(0xffffffffu, any);
      }
      done = true;
#pragma unroll
      for (int c = 0; c < PB_MCB; ++c) done = done && live[c];
    }
  }
  if (lane < nc) {
    bool v = false;
#pragma unroll
    for (int c = 0; c < PB_MCB; ++c)
      if (c == lane) v = live[c];
    const int64_t i = i0 + lane;
    flags[i] = (uint8_t)((first ? 0 : flags[i]) | (v ? 1 : 0));
  }
}

// ---------------------------------------------------------------------------------------------------
constexpr int MC_WARPS = 8;
constexpr int MCU = 4;         // sample groups per trip (independent base-sample loads in flight per lane)
// MCB = candidates per warp: every base sample loaded is applied to MCB candidates (the kernel was bound by its loads: one
// z + mu + sigma + theta fetch per 3 fp64 operations).  4 for sweeps; 1 for small batches, where the warp's serial walk over
// the samples is pure latency (83 -> ~25 us at 17 candidates, S = 1024) -- sums are per candidate, so results are identical.

// MODE: 0 = EI value only, 1 = EI value + gradient, 2 = PI value, 3 = mean utility (no improvement) value,
//       4 = mean utility value + gradient, 5 / 6 = as 1 / 4 but the gradient is left as per-(candidate, output) WEIGHTS
//       WA_j = scale sum_l w_l sum_s 1 dphi_j,  WB_j = scale sum_l w_l sum_s 1 dphi_j Z_sj / (2 sigma_j)
//       for the fused gradient path (the second contraction's epilogue applies them, split_gemm.cu EPI_DACQ)
// NW: warps per candidate.  1 for everything but tiny batches (the L-BFGS rounds of the acquisition optimiser: <= 128
// candidates), where a block of MC_WARPS warps shares ONE candidate: each warp takes a slice of every 1024-sample block
// and the per-warp partial sums -- every output of the kernel is linear in them -- are added through shared memory in
// fixed order at the end (93 -> ~25 us at 17 candidates, S = 1024: the warp's serial walk over the samples was latency).
template <int COMP, int MODE, int MCB, int NW = 1>
__global__ void __launch_bounds__(MC_WARPS * 32) mc_acq_kernel(
    const double* __restrict__ mean, const double* __restrict__ var, const double* __restrict__ dmean,
    const double* __restrict__ dvar, int64_t Nc, int64_t Nvalid, int m, int d, const double* __restrict__ Zt, int S,
    const double* __restrict__ theta, int L, int p, const double* __restrict__ weight,
    const double* __restrict__ fstar, double scale, int accumulate, double* __restrict__ acq,
    double* __restrict__ dacq, double* __restrict__ wa_out, double* __restrict__ wb_out) {
  constexpr bool WITH_GRAD = (MODE == 1 || MODE == 4), WEIGHTS = (MODE == 5 || MODE == 6);
  constexpr bool PLAIN_U = (MODE == 3 || MODE == 4 || MODE == 6);
  static_assert(NW == 1 || (NW == MC_WARPS && MCB == 1 && 32 % (NW * MCU) == 0), "a block shares one candidate or none");
  __shared__ double2 s_ms[MC_WARPS][MAXM][MCB];            // (mu, sigma) of the warp's MCB candidates, output-major
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t i0 = (NW == 1) ? ((int64_t)blockIdx.x * MC_WARPS + warp) * MCB : (int64_t)blockIdx.x;
  if (i0 >= Nvalid) return;
  const int nc = (int)min((int64_t)MCB, Nvalid - i0);       // valid candidates of this warp
  for (int idx = lane; idx < m * MCB; idx += 32) {
    const int j = idx / MCB, c = idx - j * MCB;
    const int64_t i = i0 + min(c, nc - 1);                  // ragged tail: replicate the last valid candidate
    s_ms[warp][j][c] = make_double2(mean[(int64_t)j * Nc + i], sqrt(var[(int64_t)j * Nc + i]));   // uEI_noiseless.py:74,151
  }
  __syncwarp();

  double val_total[MCB];     // sum_l w_l sum_s improvement
  double grad_q[MCB];        // lane q < d
  double wa[MCB][MAXM / 32], wb[MCB][MAXM / 32];   // WEIGHTS: lane (j & 31) keeps output j
#pragma unroll
  for (int c = 0; c < MCB; ++c) {
    val_total[c] = grad_q[c] = 0.0;
#pragma unroll
    for (int w = 0; w < MAXM / 32; ++w) wa[c][w] = wb[c][w] = 0.0;
  }
  for (int l = 0; l < L; ++l) {
    const double* th = theta + (int64_t)l * p;
    const double wl = weight[l];
    const double fs = PLAIN_U ? 0.0 : ((MODE == 2) ? fstar[l] + 1e-6 : fstar[l]);       // uPI.py:83 jitter
    double val_l[MCB];
#pragma unroll
    for (int c = 0; c < MCB; ++c) val_l[c] = 0.0;
    for (int sb = 0; sb < S; sb += 1024) {
      unsigned mask[MCB];
#pragma unroll
      for (int c = 0; c < MCB; ++c) mask[c] = 0u;
      // the 32 sample groups of this block of 1024: all of them (NW == 1) or this warp's slice
      const int kbeg = (NW == 1) ? 0 : warp * (32 / NW), kend = (NW == 1) ? 32 : kbeg + 32 / NW;
#pragma unroll 1
      for (int k0 = kbeg; k0 < kend; k0 += MCU) {
        double U[MCB][MCU];
#pragma unroll
        for (int c = 0; c < MCB; ++c)
#pragma unroll
          for (int u = 0; u < MCU; ++u) U[c][u] = 0.0;
        for (int j = 0; j < m; ++j) {
          const CompCtx cx = comp_ctx<COMP>(th, j, m);
          const double* zr = Zt + (int64_t)j * S + sb + lane;
          double z[MCU];
#pragma unroll
          for (int u = 0; u < MCU; ++u) z[u] = (sb + (k0 + u) * 32 + lane < S) ? zr[(k0 + u) * 32] : 0.0;
#pragma unroll
          for (int c = 0; c < MCB; ++c) {
            const double2 ms = s_ms[warp][j][c];
#pragma unroll
            for (int u = 0; u < MCU; ++u) U[c][u] += comp_phi<COMP>(cx, ms.x + ms.y * z[u]);
          }
        }
#pragma unroll
        for (int u = 0; u < MCU; ++u) {
          const int k = k0 + u;
          if (sb + k * 32 + lane < S) {
#pragma unroll
            for (int c = 0; c < MCB; ++c) {
              if (MODE == 2) {
                val_l[c] += ((U[c][u] - fs) > 0.0) ? 1.0 : 0.0;
              } else if (PLAIN_U) {
                val_l[c] += U[c][u];                                          // cbo.py:213,227: no max, no indicator
                mask[c] |= (1u << k);
              } else {
                val_l[c] += fmax(U[c][u] - fs, 0.0);                          // uEI_noiseless.py:80,161
                if (U[c][u] > fs) mask[c] |= (1u << k);                       // :162 strict >
              }
            }
          }
        }
      }
      if (WITH_GRAD || WEIGHTS) {
#pragma unroll
        for (int c = 0; c < MCB; ++c) {
          if (c >= nc) break;
          const unsigned mk = mask[c];
          if (!__any_sync(0xffffffffu, mk != 0u)) continue;
          const int64_t i = i0 + c;
          for (int j = 0; j < m; ++j) {
            const CompCtx cx = comp_ctx<COMP>(th, j, m);
            const double2 ms = s_ms[warp][j][c];
            double Aj = 0.0, Bj = 0.0;
            // this lane's active samples, in ascending order (set bits of its own mask; no warp-wide votes)
            for (unsigned rem = mk; rem != 0u; rem &= rem - 1u) {
              const int k = __ffs((int)rem) - 1;
              const int sidx = sb + k * 32 + lane;
              const double z = Zt[(int64_t)j * S + sidx];
              const double dp = comp_dphi<COMP>(cx, ms.x + ms.y * z);
              Aj += dp;
              Bj += dp * z;
            }
            __syncwarp();
            Aj = warp_sum(Aj);
            Bj = warp_sum(Bj);
            if (WEIGHTS) {
              if (lane == (j & 31)) {
#pragma unroll
                for (int w = 0; w < MAXM / 32; ++w)
                  if (w == (j >> 5)) {
                    wa[c][w] += wl * Aj;
                    wb[c][w] += wl * (Bj * (0.5 / ms.y));
                  }
              }
            } else if (lane < d) {
              const int64_t o = ((int64_t)j * Nc + i) * d + lane;
              grad_q[c] += wl * (Aj * dmean[o] + Bj * (0.5 / ms.y) * dvar[o]);   // :163-166
            }
          }
        }
      }
    }
#pragma unroll
    for (int c = 0; c < MCB; ++c) val_total[c] += wl * warp_sum(val_l[c]);
  }
  if (NW > 1) {
    // add the warps' partial sums in fixed order; warp 0 then writes like the single-warp path
    __shared__ double r_val[MC_WARPS], r_grad[MC_WARPS][MAXD], r_wa[MC_WARPS][MAXM], r_wb[MC_WARPS][MAXM];
    if (lane == 0) r_val[warp] = val_total[0];
    if (WITH_GRAD && lane < MAXD) r_grad[warp][lane] = grad_q[0];
    if (WEIGHTS) {
#pragma unroll
      for (int w = 0; w < MAXM / 32; ++w) {
        r_wa[warp][w * 32 + lane] = wa[0][w];
        r_wb[warp][w * 32 + lane] = wb[0][w];
      }
    }
    __syncthreads();
    if (warp != 0) return;
    val_total[0] = 0.0;
    grad_q[0] = 0.0;
#pragma unroll
    for (int w = 0; w < MAXM / 32; ++w) wa[0][w] = wb[0][w] = 0.0;
    for (int k = 0; k < MC_WARPS; ++k) {
      val_total[0] += r_val[k];
      if (WITH_GRAD && lane < MAXD) grad_q[0] += r_grad[k][lane];
      if (WEIGHTS) {
#pragma unroll
        for (int w = 0; w < MAXM / 32; ++w) {
          wa[0][w] += r_wa[k][w * 32 + lane];
          wb[0][w] += r_wb[k][w * 32 + lane];
        }
      }
    }
  }
#pragma unroll
  for (int c = 0; c < MCB; ++c) {
    if (c >= nc) break;
    const int64_t i = i0 + c;
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
      for (int w = 0; w < MAXM / 32; ++w) {
        const int j = w * 32 + lane;
        if (j < m) {
          wa_out[(int64_t)j * Nc + i] = wa[c][w] * scale;
          wb_out[(int64_t)j * Nc + i] = wb[c][w] * scale;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// analytic EI / PI of the linear scalarisation.  One thread per candidate.
// PI: 0 = maEI, 1 = maPI.   GRAD: 1 = with gradient; 2 = the gradient is left as per-(candidate, output) WEIGHTS of the
// posterior mean / variance gradients (wa_out, wb_out) for the fused gradient path, like the MC kernel's modes 5 / 6 (the
// second contraction's epilogue applies them, split_gemm.cu EPI_DACQ; needs m <= 16).  FORM (EI only): 1 = (mu-best)Phi + sigma phi (maEI.py:117-119,
// norm.cdf/pdf, sigma not clipped), 0 = sigma (u Phi + phi) with sigma clipped inside _get_quantiles (:95-96,147-163).
template <int PI, int GRAD>
__global__ void ma_acq_kernel(const double* __restrict__ mean, const double* __restrict__ var,
                              const double* __restrict__ dmean, const double* __restrict__ dvar, int64_t Nc,
                              int64_t Nvalid, int m, int d, const double* __restrict__ theta, int L, int p,
                              const double* __restrict__ weight, const double* __restrict__ best, int form,
                              double scale, int accumulate, double* __restrict__ acq, double* __restrict__ dacq,
                              double* __restrict__ wa_out, double* __restrict__ wb_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Nvalid) return;
  double val = 0.0;
  double g[MAXD];
#pragma unroll
  for (int q = 0; q < MAXD; ++q) g[q] = 0.0;
  constexpr int MREG = 16;
  if (m <= MREG) {
    // Few outputs (every shipped problem): the gradient is linear in the posterior gradients,
    //   grad_q = sum_j A_j dmu_jq + B_j dv_jq,   A_j = sum_l w_l a_l th_lj,   B_j = sum_l w_l b_l th_lj^2,
    // so the loop over the L parameter samples only builds the 2 m weights in registers and the m d posterior gradients
    // are read ONCE (the literal order below reads them L times: 8192 loads per candidate at L = 64, m = d = 8).
    double mj[MREG], vj[MREG], A[MREG], B[MREG];
#pragma unroll
    for (int j = 0; j < MREG; ++j) {
      mj[j] = (j < m) ? mean[(int64_t)j * Nc + i] : 0.0;
      vj[j] = (j < m) ? var[(int64_t)j * Nc + i] : 0.0;
      A[j] = B[j] = 0.0;
    }
    for (int l = 0; l < L; ++l) {
      const double* th = theta + (int64_t)l * p;
      double tj[MREG];
      double mu = 0.0, s2 = 0.0;
#pragma unroll
      for (int j = 0; j < MREG; ++j) {
        tj[j] = (j < m) ? th[j] : 0.0;
        mu += tj[j] * mj[j];
        s2 += (tj[j] * tj[j]) * vj[j];
      }
      const double sigma = sqrt(s2);
      const double b = best[l] + (PI ? 1e-6 : 0.0);                            // maPI.py:151
      double u;
      if (!PI && form == 1) {
        u = (mu - b) / sigma;                                                  // maEI.py:117-118 (scipy norm)
      } else {
        const double sc = (sigma < 1e-10) ? 1e-10 : sigma;                     // maEI.py:155-160
        u = (mu - b) / sc;
      }
      const double phi = exp(-0.5 * (u * u)) / sqrt(2.0 * CUDART_PI);
      const double Phi = 0.5 * erfc(-u / sqrt(2.0));
      double v;
      if (PI) v = Phi;                                                         // maPI.py:92,113
      else if (form == 1) v = (mu - b) * Phi + sigma * phi;                    // maEI.py:119
      else v = sigma * (u * Phi + phi);                                        // maEI.py:96
      const double wl = weight[l];
      val += wl * v;
      if (GRAD) {
        // maEI.py:120-122: dmu Phi + phi (0.5 dsg / sigma);  maPI.py:110-116: (phi / sigma)(dmu - u 0.5 dsg / sigma)
        const double a_l = PI ? wl * (phi / sigma) : wl * Phi;
        const double b_l = PI ? -wl * (phi / sigma) * u * (0.5 / sigma) : wl * phi * (0.5 / sigma);
#pragma unroll
        for (int j = 0; j < MREG; ++j) {
          A[j] = fma(a_l, tj[j], A[j]);
          B[j] = fma(b_l, tj[j] * tj[j], B[j]);
        }
      }
    }
    if (GRAD == 2) {
#pragma unroll
      for (int j = 0; j < MREG; ++j)
        if (j < m) {
          wa_out[(int64_t)j * Nc + i] = A[j] * scale;
          wb_out[(int64_t)j * Nc + i] = B[j] * scale;
        }
    } else if (GRAD) {
#pragma unroll
      for (int j = 0; j < MREG; ++j) {
        if (j < m) {
          const double* dm = dmean + ((int64_t)j * Nc + i) * d;
          const double* dv = dvar + ((int64_t)j * Nc + i) * d;
#pragma unroll
          for (int q = 0; q < MAXD; ++q)
            if (q < d) g[q] += A[j] * dm[q] + B[j] * dv[q];
        }
      }
    }
  } else
  for (int l = 0; l < L; ++l) {
    const double* th = theta + (int64_t)l * p;
    double mu = 0.0, s2 = 0.0;
    for (int j = 0; j < m; ++j) {
      const double t = th[j];
      mu += t * mean[(int64_t)j * Nc + i];
      s2 += (t * t) * var[(int64_t)j * Nc + i];
    }
    const double sigma = sqrt(s2);
    const double b = best[l] + (PI ? 1e-6 : 0.0);                            // maPI.py:151
    double phi, Phi, u;
    if (!PI && form == 1) {
      u = (mu - b) / sigma;                                                  // maEI.py:117-118 (scipy norm)
    } else {
      const double sc = (sigma < 1e-10) ? 1e-10 : sigma;                     // maEI.py:155-160
      u = (mu - b) / sc;
    }
    phi = exp(-0.5 * (u * u)) / sqrt(2.0 * CUDART_PI);
    Phi = 0.5 * erfc(-u / sqrt(2.0));
    double v;
    if (PI) v = Phi;                                                         // maPI.py:92,113
    else if (form == 1) v = (mu - b) * Phi + sigma * phi;                    // maEI.py:119
    else v = sigma * (u * Phi + phi);                                        // maEI.py:96
    const double wl = weight[l];
    val += wl * v;
    if (GRAD == 1) {
#pragma unroll
      for (int q = 0; q < MAXD; ++q) {
        if (q < d) {
          double dmu = 0.0, dsg = 0.0;
          for (int j = 0; j < m; ++j) {
            const double t = th[j];
            const int64_t o = ((int64_t)j * Nc + i) * d + q;
            dmu += t * dmean[o];
            dsg += (t * t) * dvar[o];
          }
          dsg = 0.5 * dsg / sigma;                                           // maEI.py:121
          if (PI) g[q] += wl * ((phi / sigma) * (dmu - u * dsg));            // maPI.py:116
          else g[q] += wl * (dmu * Phi + phi * dsg);                         // maEI.py:122
        }
      }
    }
  }
  const double v = val * scale;
  acq[i] = accumulate ? acq[i] + v : v;
  if (GRAD == 1) {
#pragma unroll
    for (int q = 0; q < MAXD; ++q)
      if (q < d) {
        const double gq = g[q] * scale;
        dacq[i * d + q] = accumulate ? dacq[i * d + q] + gq : gq;
      }
  }
}

// ---------------------------------------------------------------------------------------------------
// closed-form expectation of a separable composite under y_j ~ N(mu_j, v_j):  psi = sum_j psi_j(mu_j, v_j).
//   SUMSQ_TARGET  -(mu - th)^2 - v            test_1a.py:100-113, test_4a.py:96-107
//   NEG_SUM_EXP   -exp(mu + v / 2)            test_2a.py:70-83
//   ROSEN         -(a - mu)^2 - v  |  -100 mu^2 - 100 v      test_5a.py:64-77
//   LINEAR        th mu                        cbo.py:126-168 (posterior-mean branch; var / dvar are not read)
// One thread per candidate.  val = sum_l w_l psi(theta_l, .),  grad = sum_j dpsi/dmu_j dmu_j + dpsi/dv_j dv_j (cbo.py:196).
template <int COMP>
__device__ __forceinline__ void comp_psi(const CompCtx& c, double mu, double v, double& val, double& dmu, double& dv) {
  if (COMP == BOCF_U_SUMSQ_TARGET) {
    const double a = mu - c.th;
    val = -(a * a) - v;
    dmu = -2.0 * a;
    dv = -1.0;
  } else if (COMP == BOCF_U_NEG_SUM_EXP) {
    const double e = exp(mu + 0.5 * v);
    val = -e;
    dmu = -e;
    dv = -0.5 * e;
  } else if (COMP == BOCF_U_ROSEN_COMPOSITE) {
    if (c.lower == 1) {
      const double a = c.th - mu;
      val = -(a * a) - v;
      dmu = 2.0 * a;
      dv = -1.0;
    } else if (c.lower == 0) {
      val = -(100.0 * (mu * mu)) - 100.0 * v;
      dmu = -200.0 * mu;
      dv = -100.0;
    } else {
      val = dmu = dv = 0.0;
    }
  } else {
    val = c.th * mu;
    dmu = c.th;
    dv = 0.0;
  }
}

template <int COMP, int GRAD>
__global__ void psi_acq_kernel(const double* __restrict__ mean, const double* __restrict__ var,
                               const double* __restrict__ dmean, const double* __restrict__ dvar, int64_t Nc,
                               int64_t Nvalid, int m, int d, const double* __restrict__ theta, int L, int p,
                               const double* __restrict__ weight, double scale, int accumulate,
                               double* __restrict__ acq, double* __restrict__ dacq) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Nvalid) return;
  double val = 0.0;
  double g[MAXD];
#pragma unroll
  for (int q = 0; q < MAXD; ++q) g[q] = 0.0;
  for (int l = 0; l < L; ++l) {
    const double* th = theta + (int64_t)l * p;
    const double wl = weight[l];
    for (int j = 0; j < m; ++j) {
      const CompCtx cx = comp_ctx<COMP>(th, j, m);
      const double mu = mean[(int64_t)j * Nc + i];
      const double v = (COMP == BOCF_U_LINEAR) ? 0.0 : var[(int64_t)j * Nc + i];
      double pj, dm, dvv;
      comp_psi<COMP>(cx, mu, v, pj, dm, dvv);
      val += wl * pj;
      if (GRAD) {
        const int64_t o = ((int64_t)j * Nc + i) * d;
#pragma unroll
        for (int q = 0; q < MAXD; ++q)
          if (q < d) {
            double t = dm * dmean[o + q];
            if (COMP != BOCF_U_LINEAR) t += dvv * dvar[o + q];
            g[q] += wl * t;
          }
      }
    }
  }
  const double v = val * scale;
  acq[i] = accumulate ? acq[i] + v : v;
  if (GRAD == 1) {
#pragma unroll
    for (int q = 0; q < MAXD; ++q)
      if (q < d) {
        const double gq = g[q] * scale;
        dacq[i * d + q] = accumulate ? dacq[i * d + q] + gq : gq;
      }
  }
}

template <int COMP>
static int launch_psi_t(const AcqParams& P, const ChunkBuffers& cb, int64_t Nvalid, double* acq, double* dacq,
                        cudaStream_t st) {
  const unsigned grid = (unsigned)ceil_div(Nvalid, 128);
  if (dacq)
    psi_acq_kernel<COMP, 1><<<grid, 128, 0, st>>>(cb.mean, cb.var, cb.dmean, cb.dvar, cb.Nc, Nvalid, P.m, P.d, P.theta,
                                                  P.L, P.p, P.weight, P.scale, P.accumulate, acq, dacq);
  else
    psi_acq_kernel<COMP, 0><<<grid, 128, 0, st>>>(cb.mean, cb.var, cb.dmean, cb.dvar, cb.Nc, Nvalid, P.m, P.d, P.theta,
                                                  P.L, P.p, P.weight, P.scale, P.accumulate, acq, dacq);
  BOCF_LAUNCH_OK("psi_acq_kernel");
  return 0;
}

// ---------------------------------------------------------------------------------------------------
template <int COMP>
__global__ void utility_eval_kernel(int m, const double* __restrict__ Y, int64_t N, const double* __restrict__ theta,
                                    int L, int p, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int l = blockIdx.y;
  if (i >= N) return;
  const double* th = theta + (int64_t)l * p;
  double U = 0.0;
  for (int j = 0; j < m; ++j) {
    const CompCtx c = comp_ctx<COMP>(th, j, m);
    U += comp_phi<COMP>(c, Y[(int64_t)j * N + i]);
  }
  out[(int64_t)l * N + i] = U;
}

// out[l][j][i] = dU/dy_j (theta_l, Y[:, i]) = dphi_j (bocf_utility_grad_eval)
template <int COMP>
__global__ void utility_grad_eval_kernel(int m, const double* __restrict__ Y, int64_t N, const double* __restrict__ theta,
                                         int L, int p, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int l = blockIdx.y;
  if (i >= N) return;
  const double* th = theta + (int64_t)l * p;
  for (int j = 0; j < m; ++j) {
    const CompCtx c = comp_ctx<COMP>(th, j, m);
    out[((int64_t)l * m + j) * N + i] = comp_dphi<COMP>(c, Y[(int64_t)j * N + i]);
  }
}

// ---------------------------------------------------------------------------------------------------
// top-k (largest value, ties -> smaller index).  key order: a before b  <=>  va > vb || (va == vb && ia < ib)
__device__ __forceinline__ bool key_before(double va, int64_t ia, double vb, int64_t ib) {
  return (va > vb) || (va == vb && ia < ib);
}

constexpr int TOPK_THREADS = 256;
constexpr int TOPK_MAXK = 64;

// Each block selects the k best of its segment [seg0, seg1) by k rounds of arg-max under the previous pick.
// vals/idx describe the candidate pool: value = vals[t], index = idx ? idx[t] : t.
__global__ void __launch_bounds__(TOPK_THREADS) topk_select_kernel(const double* __restrict__ vals,
                                                                   const int64_t* __restrict__ idx, int64_t N,
                                                                   int64_t seg, int k, double* __restrict__ out_val,
                                                                   int64_t* __restrict__ out_idx) {
  __shared__ double sv[TOPK_THREADS / 32];
  __shared__ int64_t si[TOPK_THREADS / 32];
  __shared__ double pv;
  __shared__ int64_t pi;
  const int64_t seg0 = (int64_t)blockIdx.x * seg;
  const int64_t seg1 = min(N, seg0 + seg);
  double prev_v = CUDART_INF;
  int64_t prev_i = -1;
  for (int r = 0; r < k; ++r) {
    double bv = -CUDART_INF;
    int64_t bi = INT64_MAX;
    for (int64_t t = seg0 + threadIdx.x; t < seg1; t += TOPK_THREADS) {
      double v = vals[t];
      if (!(v == v)) v = -CUDART_INF;                       // NaN sorts last
      const int64_t id = idx ? idx[t] : t;
      if (id < 0) continue;                                 // empty slot
      // strictly after the previous pick, and better than the running best
      if (key_before(prev_v, prev_i, v, id) && key_before(v, id, bv, bi)) {
        bv = v;
        bi = id;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int64_t oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (key_before(ov, oi, bv, bi)) {
        bv = ov;
        bi = oi;
      }
    }
    if ((threadIdx.x & 31) == 0) {
      sv[threadIdx.x >> 5] = bv;
      si[threadIdx.x >> 5] = bi;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      double fv = sv[0];
      int64_t fi = si[0];
      for (int w = 1; w < TOPK_THREADS / 32; ++w)
        if (key_before(sv[w], si[w], fv, fi)) {
          fv = sv[w];
          fi = si[w];
        }
      pv = fv;
      pi = fi;
      out_val[(int64_t)blockIdx.x * k + r] = fv;
      out_idx[(int64_t)blockIdx.x * k + r] = (fi == INT64_MAX) ? -1 : fi;
    }
    __syncthreads();
    prev_v = pv;
    prev_i = pi;
    if (prev_i == INT64_MAX) {   // pool exhausted: fill the rest with empties
      for (int rr = r + 1 + threadIdx.x; rr < k; rr += TOPK_THREADS) {
        out_val[(int64_t)blockIdx.x * k + rr] = -CUDART_INF;
        out_idx[(int64_t)blockIdx.x * k + rr] = -1;
      }
      break;
    }
    __syncthreads();
  }
}

// record = (value, global index as double, x_0 .. x_{d-1})
__global__ void topk_gather_kernel(const double* __restrict__ val, const int64_t* __restrict__ idx,
                                   const double* __restrict__ Xc, int d, int k, int64_t index_offset,
                                   double* __restrict__ out_rec) {
  const int r = blockIdx.x;
  if (r >= k) return;
  const int64_t id = idx[r];
  double* rec = out_rec + (int64_t)r * (2 + d);
  if (threadIdx.x == 0) {
    rec[0] = (id >= 0) ? val[r] : -CUDART_INF;
    rec[1] = (id >= 0) ? (double)(id + index_offset) : -1.0;
  }
  for (int q = threadIdx.x; q < d; q += blockDim.x) rec[2 + q] = (id >= 0) ? Xc[id * d + q] : 0.0;
}

// ===================================================================================================
template <int COMP>
static int launch_mc_t(const AcqParams& P, const ChunkBuffers& cb, int64_t Nvalid, double* acq, double* dacq,
                       cudaStream_t st) {
  const bool small = (Nvalid <= 1024), tiny = (Nvalid <= 128);
  const unsigned grid = tiny ? (unsigned)Nvalid : (unsigned)ceil_div(Nvalid, (int64_t)MC_WARPS * (small ? 1 : 4));
  const bool weights = (P.wa != nullptr);
  const int mode = (P.variant == BOCF_ACQ_MEAN_UTILITY) ? (weights ? 6 : dacq ? 4 : 3)
                   : (P.variant == BOCF_ACQ_PI_CF)      ? 2
                                                         : (weights ? 5 : dacq ? 1 : 0);
#define BOCF_MC_ARGS                                                                                              \
  cb.mean, cb.var, cb.dmean, cb.dvar, cb.Nc, Nvalid, P.m, P.d, P.Zt, P.S, P.theta, P.L, P.p, P.weight, P.fstar, \
      P.scale, P.accumulate, acq, dacq, P.wa, P.wb
  {
  ProfScope ps("mc_acq_kernel", st);
#define BOCF_MC_LAUNCH(MD)                                                                       \
  do {                                                                                           \
    if (tiny) mc_acq_kernel<COMP, MD, 1, MC_WARPS><<<grid, MC_WARPS * 32, 0, st>>>(BOCF_MC_ARGS);     \
    else if (small) mc_acq_kernel<COMP, MD, 1><<<grid, MC_WARPS * 32, 0, st>>>(BOCF_MC_ARGS);    \
    else mc_acq_kernel<COMP, MD, 4><<<grid, MC_WARPS * 32, 0, st>>>(BOCF_MC_ARGS);               \
  } while (0)
  if (mode == 0) BOCF_MC_LAUNCH(0);
  else if (mode == 1) BOCF_MC_LAUNCH(1);
  else if (mode == 2) BOCF_MC_LAUNCH(2);
  else if (mode == 3) BOCF_MC_LAUNCH(3);
  else if (mode == 4) BOCF_MC_LAUNCH(4);
  else if (mode == 5) BOCF_MC_LAUNCH(5);
  else BOCF_MC_LAUNCH(6);
#undef BOCF_MC_LAUNCH
  }
#undef BOCF_MC_ARGS
  BOCF_LAUNCH_OK("mc_acq_kernel");
  return 0;
}

int launch_acq_chunk(const AcqParams& P, const ChunkBuffers& cb, int64_t Nvalid, double* acq, double* dacq,
                     cudaStream_t st) {
  if (Nvalid <= 0) return 0;
  if (P.variant == BOCF_ACQ_PSI) {
    switch (P.composite) {
      case BOCF_U_SUMSQ_TARGET: return launch_psi_t<BOCF_U_SUMSQ_TARGET>(P, cb, Nvalid, acq, dacq, st);
      case BOCF_U_NEG_SUM_EXP: return launch_psi_t<BOCF_U_NEG_SUM_EXP>(P, cb, Nvalid, acq, dacq, st);
      case BOCF_U_ROSEN_COMPOSITE: return launch_psi_t<BOCF_U_ROSEN_COMPOSITE>(P, cb, Nvalid, acq, dacq, st);
      case BOCF_U_LINEAR: return launch_psi_t<BOCF_U_LINEAR>(P, cb, Nvalid, acq, dacq, st);
      default:
        set_error("no closed-form expectation for this composite (the reference ships none for EXP_COS): use "
                  "BOCF_ACQ_MEAN_UTILITY");
        return BOCF_ERR_UNSUPPORTED;
    }
  }
  if (P.variant == BOCF_ACQ_EI_CF || P.variant == BOCF_ACQ_PI_CF || P.variant == BOCF_ACQ_MEAN_UTILITY) {
    if (P.m > MAXM) {
      set_error("mc acquisition: m exceeds MAXM");
      return -5;
    }
    if (is_user_composite(P.composite)) return launch_mc_user(P, cb, Nvalid, acq, dacq, st);
    switch (P.composite) {
      case BOCF_U_SUMSQ_TARGET: return launch_mc_t<BOCF_U_SUMSQ_TARGET>(P, cb, Nvalid, acq, dacq, st);
      case BOCF_U_NEG_SUM_EXP: return launch_mc_t<BOCF_U_NEG_SUM_EXP>(P, cb, Nvalid, acq, dacq, st);
      case BOCF_U_EXP_COS: return launch_mc_t<BOCF_U_EXP_COS>(P, cb, Nvalid, acq, dacq, st);
      case BOCF_U_ROSEN_COMPOSITE: return launch_mc_t<BOCF_U_ROSEN_COMPOSITE>(P, cb, Nvalid, acq, dacq, st);
      case BOCF_U_LINEAR: return launch_mc_t<BOCF_U_LINEAR>(P, cb, Nvalid, acq, dacq, st);
      default: set_error("unknown composite"); return -1;
    }
  }
  const unsigned grid = (unsigned)ceil_div(Nvalid, 128);
  const int pi = (P.variant == BOCF_ACQ_MA_PI) ? 1 : 0;
#define BOCF_MA_ARGS                                                                                         \
  cb.mean, cb.var, cb.dmean, cb.dvar, cb.Nc, Nvalid, P.m, P.d, P.theta, P.L, P.p, P.weight, P.fstar,        \
      P.with_grad_formula, P.scale, P.accumulate, acq, dacq, P.wa, P.wb
  if (P.wa != nullptr && P.m > 16) {
    set_error("analytic acquisition: the fused gradient path needs m <= 16");
    return BOCF_ERR_UNSUPPORTED;
  }
  if (pi) {
    if (P.wa) ma_acq_kernel<1, 2><<<grid, 128, 0, st>>>(BOCF_MA_ARGS);
    else if (dacq) ma_acq_kernel<1, 1><<<grid, 128, 0, st>>>(BOCF_MA_ARGS);
    else ma_acq_kernel<1, 0><<<grid, 128, 0, st>>>(BOCF_MA_ARGS);
  } else {
    if (P.wa) ma_acq_kernel<0, 2><<<grid, 128, 0, st>>>(BOCF_MA_ARGS);
    else if (dacq) ma_acq_kernel<0, 1><<<grid, 128, 0, st>>>(BOCF_MA_ARGS);
    else ma_acq_kernel<0, 0><<<grid, 128, 0, st>>>(BOCF_MA_ARGS);
  }
#undef BOCF_MA_ARGS
  BOCF_LAUNCH_OK("ma_acq_kernel");
  return 0;
}

// ---------------------------------------------------------------------------------------------------
// pruned sweep (bocf_acq_eval): bound, survivor list, gather, scatter
bool prune_supported(int variant, int composite) {
  return (variant == BOCF_ACQ_EI_CF || variant == BOCF_ACQ_PI_CF) &&
         (composite == BOCF_U_SUMSQ_TARGET || composite == BOCF_U_ROSEN_COMPOSITE || composite == BOCF_U_NEG_SUM_EXP ||
          composite == BOCF_U_LINEAR);
}

int launch_prune_bound(const AcqParams& P, const OutHyp* hyp_h, const ChunkBuffers& cb, int64_t Nvalid, bool first,
                       uint8_t* flags, cudaStream_t st) {
  if (Nvalid <= 0) return 0;
  if (P.m > MAXM) {
    set_error("prune bound: m exceeds MAXM");
    return BOCF_ERR_UNSUPPORTED;
  }
  const unsigned grid = (unsigned)ceil_div(Nvalid, (int64_t)PB_WARPS * PB_MCB);
  const int pi = (P.variant == BOCF_ACQ_PI_CF) ? 1 : 0;
  ProfScope ps("prune_bound_kernel", st);
#define BOCF_PB(C)                                                                                                     \
  prune_bound_kernel<C><<<grid, PB_WARPS * 32, 0, st>>>(cb.mean, cb.Nc, Nvalid, P.m, hyp_h, P.Zt, P.S, P.theta, P.L, P.p, \
                                                       P.fstar, pi, first ? 1 : 0, flags)
  switch (P.composite) {
    case BOCF_U_SUMSQ_TARGET: BOCF_PB(BOCF_U_SUMSQ_TARGET); break;
    case BOCF_U_ROSEN_COMPOSITE: BOCF_PB(BOCF_U_ROSEN_COMPOSITE); break;
    case BOCF_U_NEG_SUM_EXP: BOCF_PB(BOCF_U_NEG_SUM_EXP); break;
    case BOCF_U_LINEAR: BOCF_PB(BOCF_U_LINEAR); break;
    default: set_error("prune bound: no closed-form segment maximum for this composite"); return BOCF_ERR_UNSUPPORTED;
  }
#undef BOCF_PB
  BOCF_LAUNCH_OK("prune_bound_kernel");
  return 0;
}

// Survivor list: the indices i < N with flags[i] != 0, ascending, and their number.  Blocks of 256 threads own
// PL_TILE = 4096 consecutive flags (16 per thread): count -> exclusive scan of the block counts -> write.
constexpr int PL_THREADS = 256, PL_ITEMS = 16, PL_TILE = PL_THREADS * PL_ITEMS;

// exclusive prefix sum of v over the block (PL_THREADS threads); total into *tot
__device__ __forceinline__ int pl_block_scan(int v, int* tot) {
  __shared__ int s_w[PL_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s_w[warp] = incl;
  __syncthreads();
  int before = 0, all = 0;
#pragma unroll
  for (int w = 0; w < PL_THREADS / 32; ++w) {
    const int c = s_w[w];
    before += (w < warp) ? c : 0;
    all += c;
  }
  *tot = all;
  return before + incl - v;
}

__global__ void __launch_bounds__(PL_THREADS) prune_count_kernel(const uint8_t* __restrict__ flags, int64_t N,
                                                                 int64_t* __restrict__ blk) {
  const int64_t base = (int64_t)blockIdx.x * PL_TILE + (int64_t)threadIdx.x * PL_ITEMS;
  int c = 0;
#pragma unroll
  for (int k = 0; k < PL_ITEMS; ++k) c += (base + k < N && flags[base + k] != 0) ? 1 : 0;
  int tot;
  pl_block_scan(c, &tot);
  if (threadIdx.x == 0) blk[blockIdx.x] = tot;
}

// one block: blk[b] <- sum of blk[0 .. b), *count <- sum of all
__global__ void __launch_bounds__(PL_THREADS) prune_offsets_kernel(int64_t* __restrict__ blk, int nb,
                                                                   int64_t* __restrict__ count) {
  __shared__ int64_t s_w[PL_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int64_t base = 0;
  for (int b0 = 0; b0 < nb; b0 += PL_THREADS) {
    const int b = b0 + (int)threadIdx.x;
    const int64_t v = (b < nb) ? blk[b] : 0;
    int64_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    int64_t before = 0, all = 0;
#pragma unroll
    for (int w = 0; w < PL_THREADS / 32; ++w) {
      before += (w < warp) ? s_w[w] : 0;
      all += s_w[w];
    }
    if (b < nb) blk[b] = base + before + incl - v;
    base += all;
    __syncthreads();                                       // s_w is rewritten by the next trip
  }
  if (threadIdx.x == 0) *count = base;
}

__global__ void __launch_bounds__(PL_THREADS) prune_list_kernel(const uint8_t* __restrict__ flags, int64_t N,
                                                                const int64_t* __restrict__ blk, int64_t* __restrict__ list) {
  const int64_t base = (int64_t)blockIdx.x * PL_TILE + (int64_t)threadIdx.x * PL_ITEMS;
  bool f[PL_ITEMS];
  int c = 0;
#pragma unroll
  for (int k = 0; k < PL_ITEMS; ++k) {
    f[k] = base + k < N && flags[base + k] != 0;
    c += f[k] ? 1 : 0;
  }
  int tot;
  int64_t pos = blk[blockIdx.x] + pl_block_scan(c, &tot);
#pragma unroll
  for (int k = 0; k < PL_ITEMS; ++k)
    if (f[k]) list[pos++] = base + k;
}

uint64_t prune_list_work_bytes(int64_t N) { return (uint64_t)ceil_div(N, PL_TILE) * sizeof(int64_t); }

int launch_prune_list(const uint8_t* flags, int64_t N, int64_t* list, int64_t* count, void* work, cudaStream_t st) {
  const int nb = (int)ceil_div(N, PL_TILE);
  int64_t* blk = reinterpret_cast<int64_t*>(work);
  ProfScope ps("prune_list_kernel", st);
  prune_count_kernel<<<nb, PL_THREADS, 0, st>>>(flags, N, blk);
  BOCF_LAUNCH_OK("prune_count_kernel");
  prune_offsets_kernel<<<1, PL_THREADS, 0, st>>>(blk, nb, count);
  BOCF_LAUNCH_OK("prune_offsets_kernel");
  if (list) {
    prune_list_kernel<<<nb, PL_THREADS, 0, st>>>(flags, N, blk, list);
    BOCF_LAUNCH_OK("prune_list_kernel");
  }
  return 0;
}

// Xg[k] = Xc[list[min(k, last)]] for k < cnt (rows past the last survivor repeat it)
__global__ void prune_gather_kernel(const double* __restrict__ Xc, int d, const int64_t* __restrict__ list, int64_t last,
                                    int64_t cnt, double* __restrict__ Xg) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= cnt * d) return;
  const int64_t k = idx / d;
  const int q = (int)(idx - k * d);
  Xg[idx] = Xc[list[min(k, last)] * d + q];
}

// acq[list[k]] = acq_c[k], dacq[list[k]][.] = dacq_c[k][.] for k < cnt
__global__ void prune_scatter_kernel(const double* __restrict__ acq_c, const double* __restrict__ dacq_c,
                                     const int64_t* __restrict__ list, int64_t cnt, int d, double* __restrict__ acq,
                                     double* __restrict__ dacq) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= cnt * (d + 1)) return;
  const int64_t k = idx / (d + 1);
  const int q = (int)(idx - k * (d + 1));
  const int64_t i = list[k];
  if (q == d) acq[i] = acq_c[k];
  else if (dacq) dacq[i * d + q] = dacq_c[k * d + q];
}

// pruned candidates: acq = 0, dacq = 0
__global__ void prune_zero_kernel(const uint8_t* __restrict__ flags, int64_t N, int d, double* __restrict__ acq,
                                  double* __restrict__ dacq) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * (d + 1)) return;
  const int64_t i = idx / (d + 1);
  const int q = (int)(idx - i * (d + 1));
  if (flags[i] != 0) return;
  if (q == d) acq[i] = 0.0;
  else if (dacq) dacq[i * d + q] = 0.0;
}

int launch_prune_gather(const double* Xc, int d, const int64_t* list, int64_t last, int64_t cnt, double* Xg,
                        cudaStream_t st) {
  ProfScope ps("prune_gather_scatter_kernel", st);
  prune_gather_kernel<<<(unsigned)ceil_div(cnt * d, 256), 256, 0, st>>>(Xc, d, list, last, cnt, Xg);
  BOCF_LAUNCH_OK("prune_gather_kernel");
  return 0;
}

int launch_prune_scatter(const double* acq_c, const double* dacq_c, const int64_t* list, int64_t cnt, int d, double* acq,
                         double* dacq, cudaStream_t st) {
  ProfScope ps("prune_gather_scatter_kernel", st);
  prune_scatter_kernel<<<(unsigned)ceil_div(cnt * (d + 1), 256), 256, 0, st>>>(acq_c, dacq_c, list, cnt, d, acq, dacq);
  BOCF_LAUNCH_OK("prune_scatter_kernel");
  return 0;
}

int launch_prune_zero(const uint8_t* flags, int64_t N, int d, double* acq, double* dacq, cudaStream_t st) {
  ProfScope ps("prune_gather_scatter_kernel", st);
  prune_zero_kernel<<<(unsigned)ceil_div(N * (d + 1), 256), 256, 0, st>>>(flags, N, d, acq, dacq);
  BOCF_LAUNCH_OK("prune_zero_kernel");
  return 0;
}

template <int COMP>
static void launch_utility_grad_eval_t(dim3 grid, int m, const double* Y, int64_t N, const double* theta, int L, int p,
                                       double* out, cudaStream_t st) {
  utility_grad_eval_kernel<COMP><<<grid, 256, 0, st>>>(m, Y, N, theta, L, p, out);
}

int launch_utility_eval(int composite, int m, const double* Y, int64_t N, const double* theta, int L, int p,
                        double* out, bool grad, cudaStream_t st) {
  if (is_user_composite(composite)) return launch_utility_eval_user(composite, Y, N, theta, L, p, out, grad, st);
  dim3 grid((unsigned)ceil_div(N, 256), (unsigned)L);
  if (grad) {
    switch (composite) {
      case BOCF_U_SUMSQ_TARGET: launch_utility_grad_eval_t<BOCF_U_SUMSQ_TARGET>(grid, m, Y, N, theta, L, p, out, st); break;
      case BOCF_U_NEG_SUM_EXP: launch_utility_grad_eval_t<BOCF_U_NEG_SUM_EXP>(grid, m, Y, N, theta, L, p, out, st); break;
      case BOCF_U_EXP_COS: launch_utility_grad_eval_t<BOCF_U_EXP_COS>(grid, m, Y, N, theta, L, p, out, st); break;
      case BOCF_U_ROSEN_COMPOSITE: launch_utility_grad_eval_t<BOCF_U_ROSEN_COMPOSITE>(grid, m, Y, N, theta, L, p, out, st); break;
      case BOCF_U_LINEAR: launch_utility_grad_eval_t<BOCF_U_LINEAR>(grid, m, Y, N, theta, L, p, out, st); break;
      default: set_error("unknown composite"); return -1;
    }
    BOCF_LAUNCH_OK("utility_grad_eval_kernel");
    return 0;
  }
  switch (composite) {
    case BOCF_U_SUMSQ_TARGET: utility_eval_kernel<BOCF_U_SUMSQ_TARGET><<<grid, 256, 0, st>>>(m, Y, N, theta, L, p, out); break;
    case BOCF_U_NEG_SUM_EXP: utility_eval_kernel<BOCF_U_NEG_SUM_EXP><<<grid, 256, 0, st>>>(m, Y, N, theta, L, p, out); break;
    case BOCF_U_EXP_COS: utility_eval_kernel<BOCF_U_EXP_COS><<<grid, 256, 0, st>>>(m, Y, N, theta, L, p, out); break;
    case BOCF_U_ROSEN_COMPOSITE: utility_eval_kernel<BOCF_U_ROSEN_COMPOSITE><<<grid, 256, 0, st>>>(m, Y, N, theta, L, p, out); break;
    case BOCF_U_LINEAR: utility_eval_kernel<BOCF_U_LINEAR><<<grid, 256, 0, st>>>(m, Y, N, theta, L, p, out); break;
    default: set_error("unknown composite"); return -1;
  }
  BOCF_LAUNCH_OK("utility_eval_kernel");
  return 0;
}

static int64_t topk_blocks(int64_t N) {
  int64_t b = ceil_div(N, 8192);
  if (b > 1024) b = 1024;
  if (b < 1) b = 1;
  return b;
}

uint64_t topk_workspace_bytes(int64_t N, int k) {
  const int64_t B = topk_blocks(N);
  return (uint64_t)((B + 1) * k) * (sizeof(double) + sizeof(int64_t)) + 256;
}

int launch_topk(const double* acq, const double* Xc, int64_t N, int d, int k, int64_t index_offset, double* out_rec,
                void* workspace, cudaStream_t st) {
  if (k < 1 || k > TOPK_MAXK) {
    set_error("topk: k out of range");
    return -1;
  }
  const int64_t B = topk_blocks(N);
  const int64_t seg = ceil_div(N, B);
  double* v1 = reinterpret_cast<double*>(workspace);
  double* v2 = v1 + B * k;
  int64_t* i1 = reinterpret_cast<int64_t*>(v2 + k);
  int64_t* i2 = i1 + B * k;
  topk_select_kernel<<<(unsigned)B, TOPK_THREADS, 0, st>>>(acq, nullptr, N, seg, k, v1, i1);
  BOCF_LAUNCH_OK("topk_select_kernel");
  topk_select_kernel<<<1, TOPK_THREADS, 0, st>>>(v1, i1, B * k, B * k, k, v2, i2);
  BOCF_LAUNCH_OK("topk_select_kernel");
  topk_gather_kernel<<<k, 32, 0, st>>>(v2, i2, Xc, d, k, index_offset, out_rec);
  BOCF_LAUNCH_OK("topk_gather_kernel");
  return 0;
}

}  // namespace bocf
