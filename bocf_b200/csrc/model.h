// model.h -- internal handle layout and kernel-launcher prototypes (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <vector>

#include "../../include/bocf_b200.h"

namespace bocf {

constexpr int MAXD = 16;      // max input dimension (register / shared tiles are sized by this)
constexpr int MAXM = 64;      // max outputs handled by the MC kernel's per-warp staging
constexpr int TILE = 128;     // Cholesky block size (128 x 128 GEMM tiles)
constexpr int CAND_TILE = 256; // candidate tile of the posterior contractions (chunks are multiples of it)

// Per (hyper-sample, output) constants, resident in device memory.
struct OutHyp {
  double variance;            // sigma_f^2
  double noise;               // sigma_n^2 (Gaussian likelihood variance)
  double ybar;                // training mean of output j (Standardize, std == 1)
  double jitter;              // extra diagonal jitter added by the jitchol retry loop
  double ls[MAXD];            // lengthscale per input dimension
};

// A run of consecutive outputs j0 .. j0 + cnt - 1 that share one kernel family (multi_outputGP.py:23,38-44 takes a kernel
// LIST: the family may differ per output).  The family is a template parameter of every kernel that evaluates k(.,.), so
// the launchers issue one launch per run; kernels whose grid walks (hyper-sample, output) pairs decode through run_hj.
struct OutRun {
  int j0, cnt;
};
__host__ __device__ __forceinline__ int run_hj(int idx, OutRun r, int m) { return (idx / r.cnt) * m + r.j0 + idx % r.cnt; }

// The factorisation and the likelihood pass are chains of small, dependent launches (a 128-block Cholesky step keeps
// H*m of the 148 SMs busy): with enough outputs they are issued as TWO output groups on two streams, so one group's
// latency-bound steps run under the other's wide ones (fork / join around the groups with events; api.cu, lml.cu).
struct GroupStreams {
  cudaStream_t side = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
};

}  // namespace bocf

struct bocf_model {
  int m = 0, d = 0, kernel = 0, device = 0;
  std::vector<int> kinds;     // kernel family per output (bocf_model_set_kernels; all = `kernel` by default)
  int n = 0, n_pad = 0, n16 = 0, nb = 0, H = 0;
  bool has_data = false, has_hyp = false, factorized = false;

  double* X = nullptr;        // n x d
  double* Y = nullptr;        // m x n
  double* yc = nullptr;       // m x n_pad   centred observations (zero padded)
  double* ybar = nullptr;     // m
  bocf::OutHyp* hyp = nullptr;            // H*m
  std::vector<bocf::OutHyp> hyp_host;
  double* Xs = nullptr;       // H*m x n_pad x d   training inputs / lengthscale (zero padded rows)
  double* xsq = nullptr;      // H*m x n_pad
  double* Lmat = nullptr;     // H*m x n_pad x n_pad   Gram, then its lower Cholesky factor
  double* Linv = nullptr;     // H*m x n_pad x n_pad   L^-1 (lower, zero padded)
  double* Dinv = nullptr;     // H*m x nb x 128 x 128  inverses of L's diagonal blocks
  double* alpha = nullptr;    // H*m x n_pad
  double* tvec = nullptr;     // H*m x n_pad           L^-1 (y - ybar)
  int* info = nullptr;        // H*m                   first failing pivot (1-based) or 0

  // small per-call parameters (theta, weights, f*): ring of pinned host slots + device slots, one event per slot
  static constexpr int PAR_SLOTS = 8;
  void* par_host = nullptr;
  void* par_dev = nullptr;
  size_t par_slot_bytes = 0;
  int par_next = 0;
  cudaEvent_t par_event[PAR_SLOTS] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  double* io_buf = nullptr;   // grow-only staging of bocf_acq_eval_host (candidates in, acq / gradient out)
  size_t io_doubles = 0;
  int64_t* prune_count_host = nullptr;   // pinned: survivor count of the pruned sweep (bocf_acq_eval)
  int64_t swept_candidates = 0;          // latest bocf_acq_eval: candidates, and those the sweep evaluated (the rest
  int64_t swept_survivors = 0;           // were proven inactive)

  void* scratch = nullptr;
  uint64_t scratch_bytes = 0;
  uint64_t scratch_limit = 4ull << 30;

  // ---- split-integer tensor-core contraction (split_gemm.cu) ---------------------------------------
  int precision = 2;          // requested mode (bocf_precision); default BOCF_PREC_AUTO
  int slices_req = 5;         // requested digit planes for BOCF_PREC_SPLIT_I8
  int slices2_req = 0;        // ... of the second contraction (0: same as the first)
  int S = 0;                  // ACTIVE digit planes of K* (first contraction); 0 = fp64 DMMA contractions
  int S2 = 0;                 // ACTIVE digit planes of V  (second contraction)
  int sch1 = 0, sch2 = 0;     // digit-pair schemes (SA*100 + SB*10 + LMIN) of the two contractions
  int NTs = 0, ncts = 0, KCH = 0;   // first contraction: column tile, number of column tiles; 64-wide K chunks
  int NT2 = 0, nct2 = 0;      // second contraction: column tile, number of column tiles
  double linv_absmax = 0.0;   // max |Linv| over all (h, j), measured at factorisation
  uint8_t* B1 = nullptr;      // H*m x ncts x KCH x SB1 x NTs x 64  digit planes of Linv rows   (V  = K* Linv^T)
  uint8_t* B2 = nullptr;      // H*m x nct2 x KCH x SB2 x NT2 x 64  digit planes of Linv columns (Wt = V Linv)
  double* cs1 = nullptr;      // H*m x ncts*NTs   power-of-two output scale per column of the first contraction
  double* cs2 = nullptr;      // H*m x nct2*NT2   ... of the second
  double* aq = nullptr;       // H*m   2^(8 S  - 2 - eA): quantiser of K*   (K* <= sigma_f^2)
  double* vq = nullptr;       // H*m   2^(8 S2 - 2 - eV): quantiser of V    (|V| <= sigma_f)
  double* lml_ws = nullptr;   // workspace of the likelihood pass (per-tile partials + results), kept across calls: the
  size_t lml_ws_count = 0;    // fit loops call it thousands of times and cudaMalloc / cudaFree cost milliseconds each
  bocf::GroupStreams gs;      // second stream + events of the two-group factorisation / likelihood pass
  bool split_ready = false;
  bool precision_resolved = false;   // M->S and the digit planes match the current factor and requested mode
};

namespace bocf {

// f(kind, OutRun) for every maximal run of consecutive outputs with the same kernel family inside the output group
// `grp` (default: all outputs); stops at the first non-zero rc
template <class F>
inline int for_each_kind_run(const bocf_model* M, OutRun grp, F f) {
  int j0 = grp.j0;
  const int jend = grp.j0 + grp.cnt;
  while (j0 < jend) {
    const int kind = M->kinds.empty() ? M->kernel : M->kinds[j0];
    int j1 = j0 + 1;
    while (j1 < jend && (M->kinds.empty() ? M->kernel : M->kinds[j1]) == kind) ++j1;
    if (int rc = f(kind, OutRun{j0, j1 - j0})) return rc;
    j0 = j1;
  }
  return 0;
}
template <class F>
inline int for_each_kind_run(const bocf_model* M, F f) {
  return for_each_kind_run(M, OutRun{0, M->m}, f);
}

// ---- chol.cu ------------------------------------------------------------------------------------
int launch_prepare(bocf_model* M, cudaStream_t st);                       // ybar, yc, Xs, xsq
// `grp`: the outputs the launches cover (all hyper-samples of them)
int launch_gram(bocf_model* M, OutRun grp, cudaStream_t st);              // K + (noise+1e-8+jitter) I
int launch_cholesky(bocf_model* M, OutRun grp, cudaStream_t st);          // blocked potrf, info flags (info zeroed by the caller)
int launch_inverse_and_alpha(bocf_model* M, OutRun grp, cudaStream_t st); // Linv, alpha
// f(group, stream) for one group on `st`, or for two halves of the outputs on `st` and the model's side stream
int for_each_output_group(bocf_model* M, cudaStream_t st, int (*f)(bocf_model*, OutRun, cudaStream_t, void*), void* ctx);
int launch_copy_factor(bocf_model* M, int hj, double* L, double* Linv, double* alpha, cudaStream_t st);
int launch_alpha(bocf_model* M, OutRun grp, cudaStream_t st);              // alpha = Linv^T (Linv yc)
int launch_append_xy(const double* Xold, const double* Yold, const double* xnew, const double* ynew, int n, int d, int m,
                     double* Xn, double* Yn, cudaStream_t st);
int launch_append(bocf_model* M, int n_old, double* work, cudaStream_t st);   // bordered Cholesky / inverse update

// ---- lml.cu -------------------------------------------------------------------------------------
// out_host: H*m x (MAXD + 3) doubles [log p(y), d/dvariance, d/dnoise, d/dlengthscale[0..d)]
int launch_log_likelihood(bocf_model* M, double* out_host, cudaStream_t st);

// ---- posterior.cu -------------------------------------------------------------------------------
struct ChunkBuffers {          // scratch views for one candidate chunk (Nc rows, multiple of 128)
  int64_t Nc;
  double* KsT;                 // m x n16 x Nc      cross-covariance, transposed (row b, col i)
  double* GsT;                 // m x n16 x Nc      dK/dr * 1/r (gradient weights), transposed
  double* V;                   // m x Nc x n_pad    L^-1 k*
  double* part_var;            // m x nb x Nc       per column-tile partial sums of v^2
  double* part_dvar;           // m x nb x Nc x d   per column-tile partial variance gradients
  double* mean;                // m x Nc
  double* var;                 // m x Nc
  double* dmean;               // m x Nc x d
  double* dvar;                // m x Nc x d
  double* part_s0 = nullptr;   // split mode: m x parts x Nc  per column-tile partial sums of Wt * G*
  uint8_t* A1 = nullptr;       // split mode: m x Nc/128 x KCH x S x 128 x 64  digit planes of K* (replaces KsT)
  uint8_t* A2 = nullptr;       // split mode: same layout, digit planes of V   (replaces V)
  double* kpart = nullptr;     // K-split partial sums of mean / dmean for small chunks (posterior.cu: kstar_ksplit)
  double* wa = nullptr;        // split mode, fused gradient path: m x Nc weights of the mean gradient      (acq.cu)
  double* wb = nullptr;        //                                  m x Nc weights of the variance gradient
  int* unit_flags = nullptr;   //   m x RTv  unit (output j, candidate tile rt) has a non-zero weight (index j * RTv + rt)
  int* unit_list = nullptr;    //   ids j * RTv + rt of the flagged units, ascending
  int* unit_count = nullptr;   //   length of unit_list
};
int kstar_ksplit(const bocf_model* M, int64_t Nc);
uint64_t kstar_part_bytes(const bocf_model* M, int64_t Nc);
// Nc > 0: exact for a chunk of Nc candidates; Nc <= 0: the sizing figure of a LARGE chunk (pick_chunk divides the limit by it)
uint64_t chunk_bytes_per_candidate(const bocf_model* M, bool grad, int64_t Nc = 0);
void carve_chunk(const bocf_model* M, void* base, int64_t Nc, bool grad, ChunkBuffers* out);
// Posterior of hyper-sample h for candidates Xc[0..Nvalid) into the chunk buffers.
// grad: also K*-side gradient quantities (dmean, G*); need_var / need_dvar select the two contractions.
// noiseless: 0 = likelihood variance added, clipped at 1e-10; 1 = noiseless, clipped; 2 = noiseless, not clipped
int launch_posterior_chunk(bocf_model* M, int h, const double* Xc, int64_t Nvalid, bool grad, int noiseless,
                           const ChunkBuffers& cb, cudaStream_t st, bool need_var = true, bool need_dvar = true);
// Posterior mean of hyper-sample h only, into cb.mean: bitwise the mean launch_posterior_chunk / launch_fused_grad_chunk
// form for the same candidate (no K*, digit planes or G* are written)
int launch_posterior_mean_chunk(bocf_model* M, int h, const double* Xc, int64_t Nvalid, const ChunkBuffers& cb,
                                cudaStream_t st);

// ---- split_gemm.cu ------------------------------------------------------------------------------
int split_scheme_for_slices(int S);                 // 3..6 digit planes -> scheme code (331, 442, 554, 665)
int split_scheme_pairs(int sch);                     // int8 GEMM passes of a scheme
int split_parts(const bocf_model* M, int64_t Nc);    // parts per candidate tile for a chunk of Nc candidates (<= 0: a large chunk)
int split_partials_var(const bocf_model* M, int64_t Nc);    // partial sums per candidate the VAR / DVAR epilogues write
int split_partials_dvar(const bocf_model* M, int64_t Nc);
int split_prepare(bocf_model* M, int sch1, int sch2, cudaStream_t st);   // digit planes of Linv + scales
void split_release(bocf_model* M);
int split_linv_absmax(bocf_model* M, double* out_host, cudaStream_t st);
uint64_t split_chunk_bytes_per_candidate(const bocf_model* M, bool grad, int64_t Nc = 0);
void split_carve_chunk(const bocf_model* M, void* base, int64_t Nc, bool grad, ChunkBuffers* out);
int launch_split_var(bocf_model* M, int h, int64_t Nvalid, const ChunkBuffers& cb, bool need_dvar, cudaStream_t st);
// second contraction: per-output variance gradients, or with fused_acq the acquisition-gradient epilogue (weights
// cb.wa / cb.wb, alpha of the model)
int launch_split_dvar(bocf_model* M, int h, const double* Xc, int64_t Nvalid, const ChunkBuffers& cb, bool fused_acq,
                      cudaStream_t st);
int split_debug_gemm(const double* A, const double* B, int R, int N, int K, int sch, int tri, double* out, cudaStream_t st);

// ---- kg.cu --------------------------------------------------------------------------------------
// cov (m x N), dcov (m x N x d, may be NULL): posterior covariance between each candidate and the point x2 [dev, d];
// work [dev]: 3 * m * n_pad doubles
int launch_cov_point(bocf_model* M, int h, const double* Xc, int64_t N, const double* x2, double* cov, double* dcov,
                     double* work, cudaStream_t st);

// ---- acq.cu -------------------------------------------------------------------------------------
struct AcqParams {
  int variant, composite, m, d, S, L, p, with_grad_formula;
  const double* Zt;            // [dev] m x S
  const double* theta;         // [dev] L x p
  const double* weight;        // [dev] L
  const double* fstar;         // [dev] L    (already for this hyper-sample)
  double scale;                // 1 / (H * S)  or 1 / H
  int accumulate;              // 0: overwrite outputs, 1: add
  double* wa = nullptr;        // MC variants, fused gradient path: write the gradient weights (m x Nc each) instead of
  double* wb = nullptr;        // contracting them with dmean / dvar
};
int launch_fused_grad_chunk(bocf_model* M, int h, const double* Xc, int64_t Nvalid, int noiseless, const ChunkBuffers& cb,
                            AcqParams P, double* acq, double* dacq, cudaStream_t st);
int launch_acq_chunk(const AcqParams& P, const ChunkBuffers& cb, int64_t Nvalid, double* acq, double* dacq,
                     cudaStream_t st);
// Pruned EI-CF / PI-CF sweep (bocf_acq_eval).  prune_supported: variant and composite have the closed-form bound.
bool prune_supported(int variant, int composite);
// flags[i] (first: =, else |=) 1 unless candidate i < Nvalid of the chunk provably has a zero acquisition under the
// hyper-sample whose mean is in cb.mean, hyp_h = M->hyp + h m and P.fstar
int launch_prune_bound(const AcqParams& P, const OutHyp* hyp_h, const ChunkBuffers& cb, int64_t Nvalid, bool first,
                       uint8_t* flags, cudaStream_t st);
// ascending indices of the non-zero flags[0 .. N) into list (skipped when NULL), their number into *count [dev];
// work: prune_list_work_bytes(N)
uint64_t prune_list_work_bytes(int64_t N);
int launch_prune_list(const uint8_t* flags, int64_t N, int64_t* list, int64_t* count, void* work, cudaStream_t st);
int launch_prune_gather(const double* Xc, int d, const int64_t* list, int64_t last, int64_t cnt, double* Xg,
                        cudaStream_t st);
int launch_prune_scatter(const double* acq_c, const double* dacq_c, const int64_t* list, int64_t cnt, int d, double* acq,
                         double* dacq, cudaStream_t st);
int launch_prune_zero(const uint8_t* flags, int64_t N, int d, double* acq, double* dacq, cudaStream_t st);
// grad: out (L x m x N) = dU/dy_j instead of U
int launch_utility_eval(int composite, int m, const double* Y, int64_t N, const double* theta, int L, int p,
                        double* out, bool grad, cudaStream_t st);
int launch_topk(const double* acq, const double* Xc, int64_t N, int d, int k, int64_t index_offset,
                double* out_rec, void* workspace, cudaStream_t st);
uint64_t topk_workspace_bytes(int64_t N, int k);

// ---- jit.cu -------------------------------------------------------------------------------------
// user-defined composites (ids >= BOCF_U_USER, bocf_composite_register)
bool is_user_composite(int composite);
// registered outputs and parameter length (theta_len -1 resolved to m); BOCF_ERR_INVALID for an unknown id
int user_composite_info(int composite, int* m, int* theta_len);
int launch_mc_user(const AcqParams& P, const ChunkBuffers& cb, int64_t Nvalid, double* acq, double* dacq,
                   cudaStream_t st);
int launch_utility_eval_user(int composite, const double* Y, int64_t N, const double* theta, int L, int p, double* out,
                             bool grad, cudaStream_t st);

}  // namespace bocf
