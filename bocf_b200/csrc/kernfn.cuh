// kernfn.cuh -- covariance as a function of the (clipped) squared scaled distance, fp64.
//
//   k = K_of_r(r),   g = dK/dr(r) * (1/r)  with 1/r := 0 at r == 0   (Stationary._inv_dist, stationary.py:227-234)
// so that  gradients_X(D, x*, X)[q] = (1/l_q) * sum_b D_b * g_b * (xs*_q - Xs_bq)   in lengthscale-scaled inputs
// (stationary.py:332-342 + stationary_utils.c:1-14).  For SE the same form holds with g = -k (se.py:139-147).
//
// The reference evaluates dK/dr and then multiplies by 1/r; here the quotient is simplified algebraically
// (no division, no extra rounding step):
//   RBF       dK/dr / r = -k                                   (rbf.py:45-46:      dK/dr = -r k)
//   Matern52  dK/dr / r = -(5/3) s^2 (1 + sqrt5 r) e^{-sqrt5 r} (stationary.py:532-533: (10/3 r - 5 r - 5 sqrt5/3 r^2) e)
//   Matern32  dK/dr / r = -3 s^2 e^{-sqrt3 r}                   (stationary.py:443-444: -3 s^2 r e)
// with the reference's convention that the weight is exactly 0 where r == 0.  Differences are at the 1e-16 level.
//
// exp / sqrt: the arguments on this path are exp(x <= 0) and sqrt(r2 >= 0).  The generic libdevice routines spend
// most of their instructions on special cases (ncu: the K* kernel was issue-bound on non-fp64 instructions with the
// fp64 pipe 50 % busy), so branch-free versions restricted to these ranges are used: < 2 ulp from the libdevice
// results, far inside the 1e-6 / 1e-9 parity bars.
#pragma once
#include "model.h"

namespace bocf {

// exp(x) for x <= 0.  Cody-Waite reduction x = k ln2 + r, |r| <= ln2/2, degree-13 Taylor/Horner (remainder < 4e-18),
// scaling by 2^k through the exponent field.  The argument is clamped at -700: anything below returns e^-700 ~ 1e-304
// (the reference underflows to 0 below -745; the difference is invisible at any tolerance and saves a compare + select).
// Coefficients live in constant memory so every DFMA takes them as a constant-bank operand: as immediates each 64-bit
// literal costs two extra move instructions per use (the K* kernel was issue-bound on exactly those moves).
static __constant__ double EXPC[16] = {
    1.6059043836821613e-10,      // 1/13!
    2.08767569878681e-09,        // 1/12!
    2.505210838544172e-08,       // 1/11!
    2.755731922398589e-07,       // 1/10!
    2.7557319223985893e-06,      // 1/9!
    2.48015873015873e-05,        // 1/8!
    1.984126984126984e-04,       // 1/7!
    1.3888888888888889e-03,      // 1/6!
    8.333333333333333e-03,       // 1/5!
    4.1666666666666664e-02,      // 1/4!
    1.6666666666666666e-01,      // 1/3!
    1.4426950408889634074,       // [11] log2(e)
    6755399441055744.0,          // [12] 1.5 * 2^52
    6.93147180369123816490e-01,  // [13] ln2 high
    1.90821492927058770002e-10,  // [14] ln2 low
    -700.0};
// Kernel-family constants with a non-zero low word: as literals each use costs two register moves (see EXPC).
static __constant__ double KERC[8] = {
    2.23606797749978969641,      // [0] sqrt(5)
    5.0 / 3.0,                   // [1]
    -5.0 / 3.0,                  // [2]
    1.73205080756887729353,      // [3] sqrt(3)
    1e-300,                      // [4] keeps sqrt's seed finite at r2 == 0
    1.0 / 3.0,                   // [5]
    0.0, 0.0};
__device__ __forceinline__ double exp_nonpos(double x) {
  const double xc = fmax(x, EXPC[15]);
  // round-to-nearest integer of xc * log2(e) through the 1.5 * 2^52 shift: no FRND / F2I conversion instructions,
  // and the integer is available in the low word of the shifted value
  const double sh = fma(xc, EXPC[11], EXPC[12]);
  const double kf = sh - EXPC[12];
  double r = fma(-kf, EXPC[13], xc);
  r = fma(-kf, EXPC[14], r);
  double p = EXPC[0];
#pragma unroll
  for (int c = 1; c <= 10; ++c) p = fma(p, r, EXPC[c]);
  p = fma(p, r, 0.5);
  p = fma(p, r, 1.0);
  p = fma(p, r, 1.0);
  const int k = __double2loint(sh);
  return __hiloint2double(__double2hiint(p) + (k << 20), __double2loint(p));
}

// Table variant for the K* kernel: x = (128 k + j) ln2/128 + r, |r| <= ln2/256, exp(x) = 2^k * 2^(j/128) * p(r) with a
// degree-5 polynomial (remainder r^6/720 < 6e-19) -- 10 fp64 instructions instead of the Horner version's 17; `tab` =
// factor * 2^(j/128), j = 0..127, in SHARED memory (lanes index it independently; the factor is the kernel variance).
// (Round 2 started with 32 entries and degree 6: one DFMA more per evaluation.)
constexpr int EXP_TAB_N = 128;
// (16 interleaved copies, one per lane of a half-warp, make the lookup bank-conflict free: measured, no change --
// 69.8 vs 69.1 ms per step, profiles/r2_experiments.md section 8 -- so there is one copy)
static __constant__ double EXPT[8] = {
    184.6649652337873,           // [0] 128 log2(e)
    0.005415212348111709,        // [1] ln2/128 high (low 17 mantissa bits zero: n*hi is exact for |n| < 2^17; n >= -129272)
    1.2864023111638346e-14,      // [2] ln2/128 low
    8.333333333333333e-03,       // [3] 1/120
    4.1666666666666664e-02,      // [4] 1/24
    1.6666666666666666e-01,      // [5] 1/6
    0.0, 0.0};
// CLAMP = false: the caller guarantees -700.01 < x <= 0 (clamp_q below bounds the distance instead).
template <bool CLAMP = true>
__device__ __forceinline__ double exp_nonpos_tab(double x, const double* __restrict__ tab) {
  const double xc = CLAMP ? fmax(x, EXPC[15]) : x;
  const double sh = fma(xc, EXPT[0], EXPC[12]);
  const double kf = sh - EXPC[12];
  double r = fma(-kf, EXPT[1], xc);
  r = fma(-kf, EXPT[2], r);
  const int n = __double2loint(sh);
  const double t = tab[n & (EXP_TAB_N - 1)];
  double p = fma(EXPT[3], r, EXPT[4]);
  p = fma(p, r, EXPT[5]);
  p = fma(p, r, 0.5);
  p = fma(p, r, 1.0);
  p = fma(p, r, 1.0);
  p *= t;
  return __hiloint2double(__double2hiint(p) + ((n >> 7) << 20), __double2loint(p));
}
__device__ __forceinline__ void exp_table_fill(double* tab, int tid, double factor = 1.0) {   // factor * 2^(j/128)
  if (tid < EXP_TAB_N) tab[tid] = factor * exp2((double)tid * (1.0 / EXP_TAB_N));
}

// ---- the K* kernel's arithmetic (kern_eval_fast below) works on q = KFast<KIND>::SCALE * r2 ----
// SCALE is what the family multiplies r2 (or r) by before exp / sqrt -- Matern-5/2: sqrt5 r = sqrt(5 r2), Matern-3/2:
// sqrt(3 r2), RBF / SE: r2 / 2 -- folded into the scaled candidate and the squared norms once per thread / staged point,
// and GFAC is the constant factor of (dK/dr)/r, folded into the column scale G* is multiplied by anyway.
template <int KIND>
struct KFast {
  static constexpr double SCALE = (KIND == BOCF_KERN_MATERN52) ? 5.0 : (KIND == BOCF_KERN_MATERN32) ? 3.0 : 0.5;
  static constexpr double GFAC = (KIND == BOCF_KERN_MATERN52) ? -5.0 / 3.0 : (KIND == BOCF_KERN_MATERN32) ? -3.0 : -1.0;
  // high word of the largest q whose exponent argument stays above -700.01: Matern t = sqrt(q) <= 700, RBF / SE q <= 700
  static constexpr int HIMAX = (KIND == BOCF_KERN_MATERN52 || KIND == BOCF_KERN_MATERN32) ? 0x411DE840 : 0x4085E000;
};

// Clip of a finite scaled squared distance to [QMIN, QMAX] on the INTEGER pipe.  sm_100 has no fp64 min / max
// instruction: each fmax(double) is DSETP + 2 moves + 2 selects + a NaN fix-up (6 issue slots, one on the fp64 pipe), and
// the K* kernel paid that twice per (candidate, training point): the clip of the expanded distance at 0
// (stationary.py:153) and exp's clamp at -700.  For doubles >= 0 the order of the values is the order of their high
// words, so one signed min / max pair on the high word does both: anything negative (or below the smallest normal
// number, 2.2e-308) becomes ~2.2e-308 -- which stands for "r == 0": 1 + sqrt(2e-308) == 1, the rsqrt seed stays finite
// without sqrt_nonneg's 1e-300 bias, and `nz` tells the caller to zero the gradient weight like the reference's
// inv_dist -- and the cap keeps exp's argument above -700.01 (beyond it the covariance is < 1e-304 either way).
template <int KIND>
__device__ __forceinline__ double clamp_q(double q, bool& nz) {
  const int hi = __double2hiint(q);
  nz = hi >= 0x00100000;
  return __hiloint2double(min(max(hi, 0x00100000), KFast<KIND>::HIMAX), __double2loint(q));
}

// sqrt(a) for a >= 0 (finite).  libdevice's rsqrt(double) wraps the hardware seed (MUFU.RSQ64H, ~22 bits) in a range check
// with an out-of-line slow path; that branch (BSSY / CALL / BSYNC per evaluation) keeps ptxas from interleaving the
// independent distance -> kernel chains of an unrolled trip.  Here the seed is taken directly (rsqrt.approx.ftz.f64) and
// refined branch-free: y <- y (1 + e/2 + 3 e^2/8) with e = 1 - a y^2 (cubic, error ~e^3 ~ 1e-20), and the root is
// a y.  The argument is biased by 1e-300 (a no-op for a > 1e-284) so the seed stays finite at a == 0: sqrt(0) comes
// out as 1e-150 instead of 0, which no kernel value can see (1 + sqrt5 * 1e-150 == 1) -- one add instead of a compare and
// two selects.
__device__ __forceinline__ double sqrt_nonneg(double a0) {
  const double a = a0 + KERC[4];
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
  const double e = fma(-a * y, y, 1.0);
  const double p = fma(0.375, e, 0.5);
  y = fma(y * e, p, y);
  return a * y;                    // y carries ~1e-20 after the cubic step: a*y is within 1.5 ulp of sqrt(a)
}

#define BOCF_EXP(x) (variance * exp_nonpos(x))
template <int KIND, bool GRAD>
__device__ __forceinline__ void kern_eval(double r2, double variance, double& k, double& g) {
  if (KIND == BOCF_KERN_SE) {
    // se.py:60  variance * exp(-0.5 * sqdist)
    k = BOCF_EXP(-0.5 * r2);
    if (GRAD) g = -k;
  } else if (KIND == BOCF_KERN_RBF) {
    // rbf.py:42-46 (r*r of the rounded sqrt differs from r2 by <= 1 ulp)
    k = BOCF_EXP(-0.5 * r2);
    if (GRAD) g = (r2 != 0.0) ? -k : 0.0;
  } else if (KIND == BOCF_KERN_MATERN52) {
    // stationary.py:529-533
    const double r = sqrt_nonneg(r2);
    const double t = KERC[0] * r;               // sqrt(5) r
    const double e = BOCF_EXP(-t);
    const double lin = 1.0 + t;
    k = fma(KERC[1], r2, lin) * e;
    if (GRAD) g = (r2 != 0.0) ? KERC[2] * (lin * e) : 0.0;
  } else {
    // Matern32, stationary.py:440-444
    const double r = sqrt_nonneg(r2);
    const double t = KERC[3] * r;               // sqrt(3) r
    const double e = BOCF_EXP(-t);
    k = (1.0 + t) * e;
    if (GRAD) g = (r2 != 0.0) ? -3.0 * e : 0.0;
  }
}

// sqrt(a) for a >= 0 as a * rsqrt: only the root is refined (s0 = a y0, e = 1 - s0 y0, s = s0 (1 + e/2 + 3 e^2/8); the
// neglected 5 e^3 / 16 is ~3e-21), one fp64 instruction less than refining y first.  a >= 2.2e-308 (clamp_q): no bias.
__device__ __forceinline__ double sqrt_nonneg_root(double a) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
  const double s0 = a * y;
  const double e = fma(-s0, y, 1.0);
  const double p = fma(0.375, e, 0.5);
  return fma(s0 * e, p, s0);
}

// K* kernel only.  q, nz from clamp_q(SCALE * r2); `tab` = variance * 2^(j/32) (exp_table_fill with the output's
// variance).  Returns k and gp = (dK/dr)/r / GFAC (exactly 0 where the clipped distance is 0, the reference's inv_dist
// convention) -- same formulas as kern_eval with the constant factors moved to where they are free.
template <int KIND, bool GRAD>
__device__ __forceinline__ void kern_eval_fast(double q, bool nz, double& k, double& gp, const double* __restrict__ tab) {
  if (KIND == BOCF_KERN_SE || KIND == BOCF_KERN_RBF) {
    k = exp_nonpos_tab<false>(-q, tab);
    if (GRAD) gp = (KIND == BOCF_KERN_SE || nz) ? k : 0.0;
  } else if (KIND == BOCF_KERN_MATERN52) {
    const double t = sqrt_nonneg_root(q);        // sqrt(5) r
    const double e = exp_nonpos_tab<false>(-t, tab);
    const double lin = 1.0 + t;
    k = fma(KERC[5], q, lin) * e;                // 1 + sqrt5 r + (5 r2) / 3
    if (GRAD) gp = nz ? lin * e : 0.0;
  } else {
    const double t = sqrt_nonneg_root(q);        // sqrt(3) r
    const double e = exp_nonpos_tab<false>(-t, tab);
    k = (1.0 + t) * e;
    if (GRAD) gp = nz ? e : 0.0;
  }
}

}  // namespace bocf
