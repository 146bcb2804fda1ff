/*
 * bocf_b200.h -- C ABI of the B200-native EI-CF hot path (libbocf_b200.so).
 *
 * The reference (RaulAstudillo06/BOCF) has NO FFI boundary on this path: it is numpy/scipy
 * plus one C/OpenMP routine (GPy/kern/src/stationary_utils.c:_grad_X).  The entry points below
 * are what a binding of the reference's Python plugin surface calls instead of the numpy code;
 * each one cites the reference interface it replaces (paths relative to the reference checkout).
 * INTEGRATION.md shows the ctypes stub a maintainer would add on the reference side.
 *
 * Conventions
 *  - plain C, no torch types.  All matrices are row-major IEEE fp64.
 *  - pointers marked [dev] are device pointers on the model's device, owned by the caller;
 *    pointers marked [host] are host pointers.  The library owns only the handle's buffers.
 *  - every call is stream-ordered on `stream` (a cudaStream_t passed as void*; NULL = default).
 *  - return value: 0 on success, negative bocf_status otherwise; never throws across the ABI.
 *    bocf_last_error() returns a thread-local human-readable message for the last failure.
 *  - one handle per device; a handle is not thread-safe (the reference is single-threaded).
 */
#ifndef BOCF_B200_H_
#define BOCF_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bocf_model bocf_model;

enum bocf_status {
  BOCF_OK = 0,
  BOCF_ERR_INVALID = -1,      /* bad argument / call order                                    */
  BOCF_ERR_CUDA = -2,         /* CUDA runtime error (message in bocf_last_error)              */
  BOCF_ERR_NOT_PD = -3,       /* "not positive definite, even with jitter." GPy/util/linalg.py:71 */
  BOCF_ERR_NONPOS_DIAG = -4,  /* "not pd: non-positive diagonal elements"  GPy/util/linalg.py:60  */
  BOCF_ERR_UNSUPPORTED = -5
};

/* Covariance kernels on the path (SURVEY.md 8a rows a13/a14). */
enum bocf_kernel {
  BOCF_KERN_SE = 0,        /* GPy/kern/src/se.py:44-101,135-148 (exact-difference sq. distance) */
  BOCF_KERN_RBF = 1,       /* GPy/kern/src/rbf.py:42-46 on GPy/kern/src/stationary.py:104-166   */
  BOCF_KERN_MATERN52 = 2,  /* GPy/kern/src/stationary.py:529-533                                */
  BOCF_KERN_MATERN32 = 3   /* GPy/kern/src/stationary.py:440-444                                */
};

/* Composite utilities U(theta, y) found in the reference's scripts (SURVEY.md Appendix A). */
enum bocf_composite {
  BOCF_U_SUMSQ_TARGET = 0,     /* -sum_j (y_j-theta_j)^2          test_1a.py:89-96   p = m */
  BOCF_U_NEG_SUM_EXP = 1,      /* -sum_j exp(y_j)                 test_2a.py:60-65   p = 0 */
  BOCF_U_EXP_COS = 2,          /* -sum_j c_j e^{-y_j/pi}cos(pi y_j) test_3a.py:53-67 p = 0 */
  BOCF_U_ROSEN_COMPOSITE = 3,  /* -sum_{j<m/2} (theta-y_j)^2+100 y_{j+m/2}^2  test_5a.py:48-59 p = 1 */
  BOCF_U_LINEAR = 4,           /* theta . y                       test_1b.py:89-93   p = m */
  BOCF_U_USER = 1024           /* first id bocf_composite_register hands out                   */
};

/* User-defined composites.  bocf_composite_register compiles CUDA C++ source (fp64) that defines
 *
 *   __device__ double bocf_U (const double* theta, const double* y);               // y[0 .. BOCF_M)
 *   __device__ void   bocf_dU(const double* theta, const double* y, double* grad); // grad[j] = dU/dy_j, j < BOCF_M
 *
 * for m outputs: the library defines BOCF_M = m before the source.  theta points at ONE utility parameter of
 * theta_len entries (-1: one entry per output, theta_len = m).  The source is compiled with NVRTC for sm_100a, without
 * host or toolkit headers: the CUDA math functions NVRTC provides built in (exp, log, sin, sqrt, fma, ...) are
 * available; constants such as pi are written out.  Every entry that takes a composite accepts the returned id: the
 * MC variants of bocf_acq_eval / bocf_acq_eval_host (EI_CF, PI_CF, MEAN_UTILITY; not PSI, which needs a closed form),
 * bocf_utility_eval and bocf_utility_grad_eval, each with the registered m and p >= theta_len.
 *
 * The call compiles immediately (no GPU needed) and returns in *composite_out an id >= BOCF_U_USER; registering the
 * same (source, m, theta_len) again returns the same id.  The registry is process-wide and thread-safe; the compiled
 * module is loaded on each device at its first launch there.  Returns BOCF_ERR_INVALID for a source that does not
 * compile (the NVRTC log is in bocf_last_error()) or m outside [1, 64], and BOCF_ERR_UNSUPPORTED when libnvrtc.so.12
 * cannot be loaded (it is dlopen'ed at the first registration). */
int bocf_composite_register(const char* source, int m, int theta_len, int* composite_out);

/* Acquisition variants. */
enum bocf_acq_variant {
  BOCF_ACQ_EI_CF = 0,  /* uEI_noiseless.py:63-83,138-170  MC composite EI (+ pathwise gradient) */
  BOCF_ACQ_PI_CF = 1,  /* uPI.py:66-86                     MC composite PI, value only           */
  BOCF_ACQ_MA_EI = 2,  /* maEI.py:81-126 / EI.py:79-123    analytic EI of theta^T y              */
  BOCF_ACQ_MA_PI = 3,  /* maPI.py:80-120 / PI.py           analytic PI of theta^T y              */
  /* the two consumers of cbo._current_marginal_argmax (cbo.py:121-235): NOISELESS posterior variance, sums over the
   * hyper-samples and base samples NOT normalised (as in the reference), fstar ignored */
  BOCF_ACQ_MEAN_UTILITY = 4, /* cbo.py:203-231  sum_h sum_s U(theta, mu_h + sigma_h Z_s) + pathwise gradient    */
  BOCF_ACQ_PSI = 5     /* cbo.py:126-198  sum_h psi(theta, mu_h, var_h): closed-form E[U] of the composite (psi of
                          test_1a.py:100-113, test_2a.py:70-83, test_5a.py:64-77); LINEAR = posterior-mean branch  */
};

/* Arithmetic of the two candidate-side contractions  V = K* Linv^T,  Wt = V Linv  (posterior.py:312, gp.py:474).
 * Everything else (kernel evaluation, mean, MC acquisition, Cholesky) is always IEEE fp64. */
enum bocf_precision {
  BOCF_PREC_FP64_DMMA = 0,  /* fp64 tensor-core MMA (mma.sync m8n8k4.f64)                                          */
  BOCF_PREC_SPLIT_I8 = 1,   /* tcgen05.mma kind::i8: operands split into signed 8-bit digit planes, exact int32
                               accumulation in tensor memory.  `slices` = s (3..6): both contractions use the scheme of
                               s planes (3: 8 digit pairs, 4: 13, 5: 15, 6: 21);  `slices` = 10 s1 + s2: the first
                               contraction (variance) uses s1, the second (variance gradient) s2 = s1 or s1 - 1 >= 3
                               (33, 43, 44, 54, 55, 65, 66); other pairs return BOCF_ERR_INVALID                     */
  BOCF_PREC_AUTO = 2,       /* default: smallest variance scheme whose predicted relative error stays inside the fp64
                               bar (1e-6, element-wise) both away from the data (bound from max|L^-1|) and next to a
                               training input, where the variance drops to the noise level (bound from the smallest
                               noise / signal-variance ratio): 5 planes / 15 pairs for noise >= 3.6e-3 sigma_f^2, 6
                               planes below; variance gradient one scheme below (4 planes / 13 pairs: ~1e-7 on the
                               gradient); fp64 DMMA for ill-conditioned factors or noise < 1.7e-5 sigma_f^2        */
  BOCF_PREC_MIXED = 3       /* the north star's mixed mode (1e-4 on acq / grad acq): variance 4 planes / 13 pairs
                               (~1e-6), variance gradient 3 planes / 8 pairs (~1e-5); falls back towards AUTO when
                               max|L^-1| is large                                                                   */
};

const char* bocf_last_error(void);
/* Library / build identification ("bocf_b200 <ver> sm_100a"). */
const char* bocf_version(void);

/* ---- model: replaces multi_outputGP (multi_outputGP.py:9-348) + GPModel/GPModelFixedHyps prediction
 *      state (GPyOpt/models/gpmodel.py:136-175,259-271) -------------------------------------------- */

/* m independent outputs over d inputs, all with the kernel family `kernel` (see bocf_model_set_kernels). */
int bocf_model_create(bocf_model** out, int m, int d, int kernel, int device);
/* One kernel family per output: kinds[0..m) of enum bocf_kernel.  Replaces the `kernel` LIST multi_outputGP takes
 * (multi_outputGP.py:23,38-44: output j is built from kernel[j]).  Takes effect at the next bocf_model_factorize (the
 * factorised state is invalidated); the family is a compile-time parameter of every kernel that evaluates k(.,.), so
 * runs of consecutive outputs with the same family share one launch. */
int bocf_model_set_kernels(bocf_model* model, const int* kinds, int m);
int bocf_model_destroy(bocf_model* mdl);

/* Training data.  X [dev] n x d, Y [dev] m x n (row j = observations of output j).
 * Replaces GP.set_XY (GPy/core/gp.py:191-227) incl. the fork's mean-only normaliser
 * (GPy/util/normalizer.py:57-66). */
int bocf_model_set_data(bocf_model* mdl, int n, const double* X, const double* Y, void* stream);

/* H hyper-parameter samples.  variance [host] H x m, lengthscale [host] H x m x d, noise [host] H x m.
 * Replaces the per-sample GPRegression instances of GPModel (gpmodel.py:80-100,121-126). */
int bocf_model_set_hypers(bocf_model* mdl, int H, const double* variance, const double* lengthscale,
                          const double* noise);

/* Gram + Cholesky + L^-1 + alpha for every (h, j), fp64 on device.  Replaces
 * ExactGaussianInference.inference (exact_gaussian_inference.py:43-51), pdinv/jitchol/dpotrs
 * (GPy/util/linalg.py:52-83,112-121,189-210).  jitter_out [host, may be NULL] H x m receives the
 * jitter jitchol had to add (0 if none).  Synchronises the stream (needs the device info flag). */
int bocf_model_factorize(bocf_model* mdl, double* jitter_out, void* stream);

/* Append ONE observation (x_new [dev] d, y_new [dev] m) to a factorised model with unchanged hyper-parameters: bordered
 * update of L, L^-1 and alpha in O(n^2) per output instead of the O(n^3) refactorisation that multi_outputGP.updateModel
 * (multi_outputGP.py:97-102) triggers every BO iteration (SURVEY.md 8f rank 4; GPy's cholupdate, linalg_cython.pyx:24-37).
 * Returns BOCF_ERR_UNSUPPORTED when the factor buffers are full (n a multiple of 128) or the new pivot is not positive:
 * the data are in place then and bocf_model_factorize completes the update. */
int bocf_model_append_point(bocf_model* mdl, const double* x_new, const double* y_new, void* stream);

/* Log marginal likelihood of every (h, j) GP and its gradient w.r.t. the kernel variance, the ARD lengthscales and the
 * noise variance -- the objective / gradient pair of GPModel.updateModel's ML-II + HMC (gpmodel.py:117-119).  Replaces
 * ExactGaussianInference.inference's log_marginal and dL_dK (exact_gaussian_inference.py:53-63), Stationary /
 * SE.update_gradients_full (stationary.py:191-215, se.py:169-185, stationary_utils.c:34-48) and Gaussian.update_gradients
 * (gaussian.py:64-71).  All outputs [host]: lml H x m, g_variance H x m, g_lengthscale H x m x d, g_noise H x m
 * (gradient pointers may be NULL).  Synchronises the stream. */
int bocf_model_log_likelihood(bocf_model* mdl, double* lml, double* g_variance, double* g_lengthscale,
                              double* g_noise, void* stream);

/* Copy one factor out for inspection (tests): L, Linv n x n row-major, alpha n, [dev] or NULL. */
int bocf_model_get_factor(bocf_model* mdl, int h, int j, double* L, double* Linv, double* alpha,
                          void* stream);
/* Candidates the library evaluates per internal chunk for a call with N candidates (the K* / V scratch of one chunk
 * must fit the scratch limit); results never depend on it -- exposed so tests can place spot checks on chunk borders. */
int64_t bocf_model_chunk_candidates(bocf_model* mdl, int64_t N, int with_grad);

/* Of the latest bocf_acq_eval on the handle: the candidates, and how many of them the sweep evaluated.  Fewer when the
 * posterior mean proved the others' EI-CF / PI-CF exactly zero (pruned sweep); equal when the full sweep ran. */
int bocf_model_sweep_stats(const bocf_model* mdl, int64_t* candidates, int64_t* swept);
int bocf_model_n(const bocf_model* mdl);
int bocf_model_H(const bocf_model* mdl);

/* Select the contraction arithmetic (enum bocf_precision).  May be called before or after bocf_model_factorize; the
 * digit planes of L^-1 are (re)built when needed.  The environment variable BOCF_PRECISION (fp64 | auto | mixed | split3..6 | split<s1><s2>
 * with a pair set_precision accepts) sets the initial mode of new handles; bocf_model_create returns BOCF_ERR_INVALID
 * for any other non-empty value.  The planes are built lazily by the first posterior / acquisition call after a
 * factorisation (likelihood-only callers never pay for them).  bocf_model_active_slices: digit planes of the first contraction in use (0 = fp64);
 * bocf_model_active_scheme: 1000 * scheme of the first contraction + scheme of the second, a scheme being
 * 100 SA + 10 SB + LMIN (digit planes of the candidate side, of the factor side, lowest digit-pair weight kept);
 * 0 = fp64. */
int bocf_model_set_precision(bocf_model* mdl, int mode, int slices, void* stream);
int bocf_model_active_slices(bocf_model* mdl);
int bocf_model_active_scheme(bocf_model* mdl);

/* Test hook of the split-integer tensor-core GEMM: out (R x N) = A (R x K) * B (N x K)^T, all [dev] fp64 row-major,
 * through the same digit-plane packing, tcgen05 kernel and Horner epilogue the posterior uses.
 * tri: 0 full, 1 only K <= column (requires N == K), 2 only K >= column. */
int bocf_debug_split_gemm(const double* A, const double* B, int R, int N, int K, int slices, int tri, double* out,
                          void* stream);

/* Upper bound, in bytes, of the handle's per-chunk candidate scratch (default 4 GiB): it sets the chunk size of the
 * sweeps.  A pruned EI-CF / PI-CF sweep (bocf_acq_eval) adds, on top of it, 9 bytes per candidate of the call (survivor
 * flags and list) and one chunk of gathered candidates and results; it never changes the chunk size, so that a
 * candidate's result is the same whether the call was pruned or not. */
int bocf_model_set_scratch_limit(bocf_model* mdl, uint64_t bytes);

/* Posterior of hyper-sample h at N candidates Xc [dev] N x d.  Outputs [dev], any may be NULL:
 *   mean  m x N      GP.posterior_mean            gp.py:380-400 -> posterior.py:299-305
 *   var   m x N      GP.posterior_variance (+noise) gp.py:403-418 -> posterior.py:308-320, clipped at
 *                    1e-10 as GPModel.posterior_variance does (gpmodel.py:174); noiseless=1 omits the
 *                    likelihood variance (gp.py:421-435, gpmodel.py:183); noiseless=2 omits it and the clip
 *                    (the form the knowledge-gradient helpers use, gp.py:533-544)
 *   dmean m x N x d  GP.posterior_mean_gradient     gp.py:438-461 (Stationary.gradients_X / _grad_X)
 *   dvar  m x N x d  GP.posterior_variance_gradient gp.py:464-490 (not clipped, no noise term)
 * Stacking order is multi_outputGP's (multi_outputGP.py:165-191,284-306). */
int bocf_posterior(bocf_model* mdl, int h, const double* Xc, int64_t N, int noiseless, double* mean,
                   double* var, double* dmean, double* dvar, void* stream);

/* Posterior covariance of the latent functions between each of N candidates Xc [dev] N x d and ONE point x2 [dev] d,
 * under hyper-sample h:  cov [dev] m x N,  dcov [dev, may be NULL] m x N x d = its gradient w.r.t. the candidate.
 * Replaces GP.posterior_covariance_between_points[_partially_precomputed] (GPy/core/gp.py:577-599) and
 * GP.posterior_covariance_gradient[_partially_precomputed] (gp.py:601-627) for one column X2 = x2; the
 * conditioned-on-next-point variance helpers of gp.py:518-575 are built from it on the host side
 * (bocf_b200/model.py).  fp64 throughout (no digit planes). */
int bocf_posterior_cov_point(bocf_model* mdl, int h, const double* Xc, int64_t N, const double* x2, double* cov,
                             double* dcov, void* stream);

/* ---- acquisition: replaces _compute_acq / _compute_acq_withGradients ------------------------------
 * Xc   [dev] N x d candidates
 * Zt   [dev] m x S base samples, TRANSPOSED W_samples (uEI_noiseless.py:31), MC variants only
 * theta [host] L x p utility parameters; weight [host] L (prob_dist for full support, 1/L otherwise)
 * fstar [host] H x L: EI_CF/PI_CF: max_n U(theta_l, mu(X_n)) (uEI_noiseless.py:76; the reference
 *        evaluates it once with whichever hyper-sample is current, quirk q2 -- the caller decides);
 *        MA_EI/MA_PI: best_l per hyper-sample (maEI.py:129-136).  PI jitter 1e-6 is added inside.
 * H_use: number of hyper-samples averaged (min(10, n_samples), uEI_noiseless.py:32)
 * with_grad_formula: MA_EI only -- 1 uses the (mu-best)Phi+sigma*phi form of maEI.py:117-119, 0 the
 *        sigma(u Phi+phi) form of maEI.py:95-96; ignored elsewhere.
 * acq  [dev] N     ;  dacq [dev] N x d or NULL (value only). */
int bocf_acq_eval(bocf_model* mdl, int variant, int composite, const double* Xc, int64_t N,
                  const double* Zt, int S, const double* theta, int L, int p, const double* weight,
                  const double* fstar, int H_use, int with_grad_formula, double* acq, double* dacq,
                  void* stream);

/* Same call with HOST candidate / result buffers (pinned or pageable): copies Xc in, runs the sweep,
 * copies acq/dacq out, and synchronises.  This is the end-to-end entry bench.py times as `e2e`. */
int bocf_acq_eval_host(bocf_model* mdl, int variant, int composite, const double* Xc_host, int64_t N,
                       const double* Zt_dev, int S, const double* theta, int L, int p,
                       const double* weight, const double* fstar, int H_use, int with_grad_formula,
                       double* acq_host, double* dacq_host, void* stream);

/* U(theta_l, Y[:, i]) for a batch: Y [dev] m x N -> out [dev] L x N.  Used for f* (uEI_noiseless.py:76). */
int bocf_utility_eval(int composite, int m, const double* Y, int64_t N, const double* theta, int L,
                      int p, double* out, void* stream);
/* Its gradient twin: out [dev] L x m x N, out[l][j][i] = dU/dy_j (theta_l, Y[:, i]). */
int bocf_utility_grad_eval(int composite, int m, const double* Y, int64_t N, const double* theta, int L,
                           int p, double* out, void* stream);

/* Local top-k of the LARGEST acq values (anchor selection, anchor_points_generator.py:59-64 with
 * f = -acq).  Ties break on the smaller candidate index.  out_val [dev] k, out_idx [dev] k (int64,
 * index + index_offset), out_x [dev] k x d (gathered rows of Xc) -- laid out contiguously as one
 * k x (2 + d) fp64 record buffer `out_rec` (value, index-as-double, x...) ready for ncclAllGather. */
int bocf_topk(const double* acq, const double* Xc, int64_t N, int d, int k, int64_t index_offset,
              double* out_rec, void* stream);

/* Per-kernel device timing for bench.py's live roofline: when enabled, every kernel launch is bracketed by CUDA
 * events on its stream.  bocf_profile_report synchronises the device and writes "name count total_ms" lines. */
int bocf_profile_enable(int on);
int bocf_profile_report(char* buf, int buf_bytes);

/* Counters for bench.py's gpu_launches claim: number of kernels this library has launched. */
uint64_t bocf_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* BOCF_B200_H_ */
