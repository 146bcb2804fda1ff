// api.cu -- the C ABI of libbocf_b200 (include/bocf_b200.h): handle management, the jitchol retry
// loop, candidate chunking and the fused sweep  posterior -> acquisition  over all hyper-samples.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "common.cuh"
#include "model.h"

namespace bocf {
static thread_local std::string g_err;
static std::atomic<uint64_t> g_launches{0};
void set_error(const std::string& msg) { g_err = msg; }
void count_launch(uint64_t n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- per-kernel event timing ---------------------------------------------------------------------------------
struct ProfRec {
  const char* name;
  cudaEvent_t a, b;
};
static bool g_prof_on = false;
static std::vector<ProfRec*> g_prof;
ProfScope::ProfScope(const char* name, cudaStream_t stream) : st(stream) {
  if (!g_prof_on) return;
  ProfRec* r = new ProfRec();
  r->name = name;
  cudaEventCreate(&r->a);
  cudaEventCreate(&r->b);
  cudaEventRecord(r->a, st);
  rec = r;
}
ProfScope::~ProfScope() {
  if (!rec) return;
  ProfRec* r = static_cast<ProfRec*>(rec);
  cudaEventRecord(r->b, st);
  g_prof.push_back(r);
}

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur = -1;
    cudaGetDevice(&cur);
    if (prev >= 0 && cur != prev) cudaSetDevice(prev);
  }
};

template <typename T>
static int dev_alloc(T** p, size_t count) {
  *p = nullptr;
  if (count == 0) return 0;
  BOCF_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T)));
  return 0;
}
template <typename T>
static void dev_free(T*& p) {
  if (p) cudaFree(p);
  p = nullptr;
}

static void free_data(bocf_model* M) {
  dev_free(M->X);
  dev_free(M->Y);
  dev_free(M->yc);
  dev_free(M->ybar);
}
static void free_factor(bocf_model* M) {
  split_release(M);
  M->S = M->S2 = M->sch1 = M->sch2 = 0;
  dev_free(M->Xs);
  dev_free(M->xsq);
  dev_free(M->Lmat);
  dev_free(M->Linv);
  dev_free(M->Dinv);
  dev_free(M->alpha);
  dev_free(M->tvec);
  dev_free(M->info);
  dev_free(M->lml_ws);
  M->lml_ws_count = 0;
  M->factorized = false;
}

static int ensure_scratch(bocf_model* M, uint64_t bytes) {
  if (M->scratch_bytes >= bytes) return 0;
  if (M->scratch) cudaFree(M->scratch);
  M->scratch = nullptr;
  M->scratch_bytes = 0;
  BOCF_CUDA_OK(cudaMalloc(&M->scratch, bytes));
  M->scratch_bytes = bytes;
  return 0;
}

// Choose the candidate chunk (multiple of 128) so the per-chunk scratch fits the handle's limit.
static int64_t pick_chunk(const bocf_model* M, int64_t N, bool grad, uint64_t extra_per_cand) {
  const uint64_t per = chunk_bytes_per_candidate(M, grad) + extra_per_cand;
  int64_t nc = (int64_t)(M->scratch_limit / per);
  nc = nc / CAND_TILE * CAND_TILE;
  if (nc < CAND_TILE) nc = CAND_TILE;
  const int64_t need = round_up(N, CAND_TILE);
  if (nc > need) nc = need;
  if (nc > (1 << 17)) nc = 1 << 17;
  return nc;
}

// Resolve the requested contraction precision into the active digit-pair schemes (M->sch1 / M->sch2; M->S = 0 means
// fp64 DMMA) and build the split operands.  Error model (tests/test_split_numerics.py, tests/test_gpu_split.py):
//  (i)  for candidates away from the data the relative error of the variance stays below ~2000 * a^2 * 256^-5 for scheme
//       554 (15 digit pairs), ~2000 * a^2 * 256^-6 for 665 and ~150 * a^2 * 256^-4 for 442 (13 pairs), a = max|Linv|;
//  (ii) the ABSOLUTE error of sum V^2 is K_S * 256^-S * sigma_f^2 whatever the conditioning (K_4 < 60, K_5 < 1000,
//       K_6 < 1200 across kernels, sizes and noise levels 1e-1 ... 1e-6), while the variance itself drops to the noise
//       variance at candidates next to a training input -- the points the acquisition optimiser converges to, where
//       sigma enters the pathwise gradient as 0.5 / sigma.  The element-wise relative error of `posterior_variance`
//       there is K_S 256^-S sigma_f^2 / noise; the rule asks a quarter of the bar of it, so that the NOISELESS variance
//       of uEI_noiseless (which has no floor: it falls below the noise where many neighbours average) holds the bar
//       too wherever it is >= noise / 4.
// AUTO accepts a scheme when bound (i) is <= 5e-7 and bound (ii) <= 2.5e-7 for every output (the north-star fp64 bar of
// 1e-6, element-wise, at every candidate); the variance gradient runs one scheme below the variance (442 under 554: ~1e-7
// relative, norm-wise).  MIXED targets the 1e-4 bar on acq / grad acq instead: bounds 2e-5 / 1e-5, gradient two
// schemes down to 331 (8 pairs, ~1e-5).  Models too ill-conditioned or too noise-free for 665 stay on fp64.
static int apply_precision(bocf_model* M, cudaStream_t st) {
  int s1 = 0, s2 = 0;
  if (M->precision == BOCF_PREC_SPLIT_I8) {
    s1 = M->slices_req;
    s2 = M->slices2_req > 0 ? M->slices2_req : s1;
  } else if (M->precision == BOCF_PREC_AUTO || M->precision == BOCF_PREC_MIXED) {
    if (int rc = split_linv_absmax(M, &M->linv_absmax, st)) return rc;
    const double a2 = M->linv_absmax * M->linv_absmax;
    const double bound[7] = {0, 0, 0, 0, 150.0 * a2 * std::pow(256.0, -4), 2000.0 * a2 * std::pow(256.0, -5),
                             2000.0 * a2 * std::pow(256.0, -6)};
    const double target = (M->precision == BOCF_PREC_MIXED) ? 2e-5 : 5e-7;
    double vmin = 1e300;                                          // smallest noise-to-signal ratio over (hyper-sample, output)
    for (const auto& o : M->hyp_host) vmin = std::min(vmin, (o.noise + 1e-8 + o.jitter) / o.variance);
    const double near_data[7] = {0, 0, 0, 0, 60.0 * std::pow(256.0, -4) / (0.25 * vmin), 1000.0 * std::pow(256.0, -5) / (0.25 * vmin),
                                 1200.0 * std::pow(256.0, -6) / (0.25 * vmin)};
    for (int s = 4; s <= 6 && s1 == 0; ++s)
      if (bound[s] <= target && near_data[s] <= 2.0 * target) s1 = s;
    if (s1 > 0) s2 = (M->precision == BOCF_PREC_MIXED) ? (s1 == 4 ? 3 : s1 - 1) : (s1 > 4 ? s1 - 1 : 4);
  }
  if (s1 == 0) {
    split_release(M);
    M->S = M->S2 = M->sch1 = M->sch2 = 0;
    return 0;
  }
  const int sch1 = split_scheme_for_slices(s1), sch2 = split_scheme_for_slices(s2);
  if (M->split_ready && M->sch1 == sch1 && M->sch2 == sch2) return 0;
  return split_prepare(M, sch1, sch2, st);
}

// The split-integer plane pairs the first contraction is instantiated for (split_gemm.cu launch_var): the variance on
// s1 = 3..6 digit planes, its gradient on s2 = s1 or s1 - 1 >= 3 planes (s2 = 0: s1).
static bool split_pair_supported(int s1, int s2) {
  return s1 >= 3 && s1 <= 6 && (s2 == 0 || s2 == s1 || (s2 == s1 - 1 && s2 >= 3));
}

static int resolve_precision(bocf_model* M, cudaStream_t st) {
  if (M->precision_resolved) return 0;
  if (int rc = apply_precision(M, st)) return rc;
  M->precision_resolved = true;
  return 0;
}

// Pinned / device parameter ring of the handle (see bocf_acq_eval).
template <class Fill>
static int stage_params(bocf_model* M, size_t doubles, double** dev_out, cudaStream_t st, Fill fill) {
  const size_t bytes = doubles * sizeof(double);
  if (bytes > M->par_slot_bytes) {                       // (re)allocate: rare, synchronises
    cudaStreamSynchronize(st);
    for (int s = 0; s < bocf_model::PAR_SLOTS; ++s)
      if (M->par_event[s]) {
        cudaEventDestroy(M->par_event[s]);
        M->par_event[s] = nullptr;
      }
    if (M->par_host) cudaFreeHost(M->par_host);
    if (M->par_dev) cudaFree(M->par_dev);
    M->par_host = M->par_dev = nullptr;
    size_t slot = 4096;
    while (slot < bytes) slot *= 2;
    BOCF_CUDA_OK(cudaHostAlloc(reinterpret_cast<void**>(&M->par_host), slot * bocf_model::PAR_SLOTS, cudaHostAllocDefault));
    BOCF_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&M->par_dev), slot * bocf_model::PAR_SLOTS));
    M->par_slot_bytes = slot;
    M->par_next = 0;
  }
  const int s = M->par_next;
  M->par_next = (s + 1) % bocf_model::PAR_SLOTS;
  if (M->par_event[s]) BOCF_CUDA_OK(cudaEventSynchronize(M->par_event[s]));     // normally long complete
  else BOCF_CUDA_OK(cudaEventCreateWithFlags(&M->par_event[s], cudaEventDisableTiming));
  double* host = reinterpret_cast<double*>(reinterpret_cast<char*>(M->par_host) + (size_t)s * M->par_slot_bytes);
  double* dev = reinterpret_cast<double*>(reinterpret_cast<char*>(M->par_dev) + (size_t)s * M->par_slot_bytes);
  fill(host);
  BOCF_CUDA_OK(cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, st));
  // the DEVICE slot is read by kernels enqueued after this copy on the same stream; it is overwritten PAR_SLOTS calls
  // later by a copy that the stream orders behind them.  The event guards the HOST slot.
  BOCF_CUDA_OK(cudaEventRecord(M->par_event[s], st));
  *dev_out = dev;
  return 0;
}

static int check_ready(const bocf_model* M) {
  if (!M) {
    set_error("null model handle");
    return BOCF_ERR_INVALID;
  }
  if (!M->factorized) {
    set_error("model not factorized: call bocf_model_set_data, bocf_model_set_hypers, bocf_model_factorize first");
    return BOCF_ERR_INVALID;
  }
  return 0;
}
}  // namespace bocf

using namespace bocf;

extern "C" {

const char* bocf_last_error(void) { return g_err.c_str(); }
const char* bocf_version(void) { return "bocf_b200 0.3 sm_100a fp64-dmma + tcgen05-i8-split"; }
uint64_t bocf_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int bocf_profile_enable(int on) {
  for (ProfRec* r : g_prof) {
    cudaEventDestroy(r->a);
    cudaEventDestroy(r->b);
    delete r;
  }
  g_prof.clear();
  g_prof_on = (on != 0);
  return 0;
}

// Writes one line per kernel class "name count total_ms\n" into buf; returns bytes written (or needed size).
int bocf_profile_report(char* buf, int buf_bytes) {
  cudaDeviceSynchronize();
  std::vector<std::string> names;
  std::vector<uint64_t> counts;
  std::vector<double> totals;
  for (ProfRec* r : g_prof) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, r->a, r->b) != cudaSuccess) continue;
    size_t k = 0;
    for (; k < names.size(); ++k)
      if (names[k] == r->name) break;
    if (k == names.size()) {
      names.push_back(r->name);
      counts.push_back(0);
      totals.push_back(0.0);
    }
    counts[k] += 1;
    totals[k] += ms;
  }
  std::string out;
  for (size_t k = 0; k < names.size(); ++k)
    out += names[k] + " " + std::to_string(counts[k]) + " " + std::to_string(totals[k]) + "\n";
  if (buf && buf_bytes > 0) {
    size_t ncopy = out.size() < (size_t)buf_bytes - 1 ? out.size() : (size_t)buf_bytes - 1;
    std::memcpy(buf, out.data(), ncopy);
    buf[ncopy] = 0;
  }
  return (int)out.size() + 1;
}

int bocf_model_create(bocf_model** out, int m, int d, int kernel, int device) {
  if (!out || m < 1 || d < 1 || d > MAXD || kernel < 0 || kernel > BOCF_KERN_MATERN32) {
    set_error("bocf_model_create: invalid arguments (need m >= 1, 1 <= d <= 16, known kernel)");
    return BOCF_ERR_INVALID;
  }
  int precision = BOCF_PREC_AUTO, s1 = 0, s2 = 0;               // library default
  if (const char* env = std::getenv("BOCF_PRECISION")) {      // fp64 | auto | mixed | split3 .. split6 | split<s1><s2>
    const std::string v(env);
    const auto digit = [&](size_t k) { return (v.size() > k && v[k] >= '0' && v[k] <= '9') ? v[k] - '0' : -1; };
    if (v == "auto" || v.empty()) precision = BOCF_PREC_AUTO;
    else if (v == "mixed") precision = BOCF_PREC_MIXED;
    else if (v == "fp64") precision = BOCF_PREC_FP64_DMMA;
    else if (v.rfind("split", 0) == 0 && (v.size() == 6 || (v.size() == 7 && digit(6) > 0)) &&
             split_pair_supported(digit(5), v.size() == 7 ? digit(6) : 0)) {
      precision = BOCF_PREC_SPLIT_I8;
      s1 = digit(5);
      s2 = v.size() == 7 ? digit(6) : 0;
    } else {
      set_error("bocf_model_create: BOCF_PRECISION=" + v + " is not one of fp64, auto, mixed, split3 .. split6 or "
                "split<s1><s2> with 3 <= s1 <= 6 and s2 = s1 or s1 - 1 >= 3");
      return BOCF_ERR_INVALID;
    }
  }
  int ndev = 0;
  BOCF_CUDA_OK(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) {
    set_error("bocf_model_create: no such CUDA device");
    return BOCF_ERR_INVALID;
  }
  bocf_model* M = new (std::nothrow) bocf_model();
  if (!M) {
    set_error("out of host memory");
    return BOCF_ERR_INVALID;
  }
  M->m = m;
  M->d = d;
  M->kernel = kernel;
  M->kinds.assign((size_t)m, kernel);
  M->device = device;
  M->precision = precision;
  if (precision == BOCF_PREC_SPLIT_I8) {
    M->slices_req = s1;
    M->slices2_req = s2;
  }
  *out = M;
  return 0;
}

int bocf_model_set_kernels(bocf_model* M, const int* kinds, int m) {
  if (!M || !kinds || m != M->m) {
    set_error("bocf_model_set_kernels: need one kernel family per output (m entries)");
    return BOCF_ERR_INVALID;
  }
  for (int j = 0; j < m; ++j)
    if (kinds[j] < 0 || kinds[j] > BOCF_KERN_MATERN32) {
      set_error("bocf_model_set_kernels: unknown kernel family");
      return BOCF_ERR_INVALID;
    }
  M->kinds.assign(kinds, kinds + m);
  M->kernel = kinds[0];
  M->factorized = false;                                        // Gram, factor, alpha and the digit planes are stale
  M->split_ready = false;
  M->precision_resolved = false;
  return 0;
}

int bocf_model_set_precision(bocf_model* M, int mode, int slices, void* stream) {
  int s1 = slices, s2 = 0;
  if (slices >= 10) {
    s1 = slices / 10;
    s2 = slices % 10;
  }
  if (!M || mode < BOCF_PREC_FP64_DMMA || mode > BOCF_PREC_MIXED ||
      (mode == BOCF_PREC_SPLIT_I8 && !split_pair_supported(s1, s2))) {
    set_error("bocf_model_set_precision: mode must be 0 (fp64), 1 (split int8: slices = 3..6, or 10 s1 + s2 with "
              "3 <= s1 <= 6 and s2 = s1 or s1 - 1 >= 3), 2 (auto) or 3 (mixed)");
    return BOCF_ERR_INVALID;
  }
  M->precision = mode;
  if (mode == BOCF_PREC_SPLIT_I8) {
    M->slices_req = s1;
    M->slices2_req = s2;
  }
  M->precision_resolved = false;
  if (!M->factorized) return 0;
  DeviceGuard dg(M->device);
  return resolve_precision(M, static_cast<cudaStream_t>(stream));
}

int bocf_model_active_slices(bocf_model* M) {
  if (!M) return -1;
  if (M->factorized && !M->precision_resolved) {
    DeviceGuard dg(M->device);
    if (resolve_precision(M, nullptr)) return -1;
  }
  return M->S;
}

int bocf_model_active_scheme(bocf_model* M) {
  if (bocf_model_active_slices(M) < 0) return -1;
  return M->S > 0 ? M->sch1 * 1000 + M->sch2 : 0;
}

int bocf_debug_split_gemm(const double* A, const double* B, int R, int N, int K, int slices, int tri, double* out,
                          void* stream) {
  return split_debug_gemm(A, B, R, N, K, split_scheme_for_slices(slices), tri, out, static_cast<cudaStream_t>(stream));
}

int bocf_model_destroy(bocf_model* M) {
  if (!M) return 0;
  DeviceGuard dg(M->device);
  free_data(M);
  free_factor(M);
  dev_free(M->hyp);
  if (M->scratch) cudaFree(M->scratch);
  for (int s = 0; s < bocf_model::PAR_SLOTS; ++s)
    if (M->par_event[s]) cudaEventDestroy(M->par_event[s]);
  if (M->par_host) cudaFreeHost(M->par_host);
  if (M->par_dev) cudaFree(M->par_dev);
  if (M->io_buf) cudaFree(M->io_buf);
  if (M->prune_count_host) cudaFreeHost(M->prune_count_host);
  if (M->gs.side) cudaStreamDestroy(M->gs.side);
  if (M->gs.fork) cudaEventDestroy(M->gs.fork);
  if (M->gs.join) cudaEventDestroy(M->gs.join);
  delete M;
  return 0;
}

int bocf_model_sweep_stats(const bocf_model* M, int64_t* candidates, int64_t* swept) {
  if (!M || !candidates || !swept) {
    set_error("bocf_model_sweep_stats: invalid arguments");
    return BOCF_ERR_INVALID;
  }
  *candidates = M->swept_candidates;
  *swept = M->swept_survivors;
  return 0;
}

int64_t bocf_model_chunk_candidates(bocf_model* M, int64_t N, int with_grad) {
  if (check_ready(M) || N < 1) return -1;
  DeviceGuard dg(M->device);
  if (resolve_precision(M, nullptr)) return -1;
  return pick_chunk(M, N, with_grad != 0, 0);
}

int bocf_model_n(const bocf_model* M) { return M ? M->n : -1; }
int bocf_model_H(const bocf_model* M) { return M ? M->H : -1; }

int bocf_model_set_scratch_limit(bocf_model* M, uint64_t bytes) {
  if (!M || bytes < (64ull << 20)) {
    set_error("scratch limit must be at least 64 MiB");
    return BOCF_ERR_INVALID;
  }
  M->scratch_limit = bytes;
  return 0;
}

int bocf_model_set_data(bocf_model* M, int n, const double* X, const double* Y, void* stream) {
  if (!M || n < 1 || !X || !Y) {
    set_error("bocf_model_set_data: invalid arguments");
    return BOCF_ERR_INVALID;
  }
  DeviceGuard dg(M->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (n != M->n) {
    free_data(M);
    free_factor(M);
    M->n = n;
    M->n_pad = (int)round_up(n, TILE);
    M->n16 = (int)round_up(n, 16);
    M->nb = M->n_pad / TILE;
    if (int rc = dev_alloc(&M->X, (size_t)n * M->d)) return rc;
    if (int rc = dev_alloc(&M->Y, (size_t)n * M->m)) return rc;
    if (int rc = dev_alloc(&M->yc, (size_t)M->n_pad * M->m)) return rc;
    if (int rc = dev_alloc(&M->ybar, (size_t)M->m)) return rc;
  }
  BOCF_CUDA_OK(cudaMemcpyAsync(M->X, X, sizeof(double) * n * M->d, cudaMemcpyDeviceToDevice, st));
  BOCF_CUDA_OK(cudaMemcpyAsync(M->Y, Y, sizeof(double) * n * M->m, cudaMemcpyDeviceToDevice, st));
  M->has_data = true;
  M->factorized = false;
  return 0;
}

int bocf_model_set_hypers(bocf_model* M, int H, const double* variance, const double* lengthscale,
                          const double* noise) {
  if (!M || H < 1 || !variance || !lengthscale || !noise) {
    set_error("bocf_model_set_hypers: invalid arguments");
    return BOCF_ERR_INVALID;
  }
  DeviceGuard dg(M->device);
  const int Hm = H * M->m;
  std::vector<OutHyp> hv(Hm);
  for (int hj = 0; hj < Hm; ++hj) {
    OutHyp& o = hv[hj];
    std::memset(&o, 0, sizeof(o));
    o.variance = variance[hj];
    o.noise = noise[hj];
    for (int q = 0; q < MAXD; ++q) o.ls[q] = 1.0;
    for (int q = 0; q < M->d; ++q) o.ls[q] = lengthscale[(size_t)hj * M->d + q];
    if (!(o.variance > 0.0) || !(o.noise >= 0.0)) {
      set_error("bocf_model_set_hypers: variance must be > 0 and noise >= 0");
      return BOCF_ERR_INVALID;
    }
    for (int q = 0; q < M->d; ++q)
      if (!(o.ls[q] > 0.0)) {
        set_error("bocf_model_set_hypers: lengthscales must be > 0");
        return BOCF_ERR_INVALID;
      }
  }
  if (H != M->H) {
    free_factor(M);
    dev_free(M->hyp);
    M->H = H;
    if (int rc = dev_alloc(&M->hyp, (size_t)Hm)) return rc;
  }
  M->hyp_host = hv;
  M->has_hyp = true;
  M->factorized = false;
  return 0;
}

int bocf_model_factorize(bocf_model* M, double* jitter_out, void* stream) {
  if (!M || !M->has_data || !M->has_hyp) {
    set_error("bocf_model_factorize: set data and hyper-parameters first");
    return BOCF_ERR_INVALID;
  }
  DeviceGuard dg(M->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int Hm = M->H * M->m;
  const size_t nn = (size_t)M->n_pad * M->n_pad;
  if (!M->Lmat) {
    if (int rc = dev_alloc(&M->Xs, (size_t)Hm * M->n_pad * M->d)) return rc;
    if (int rc = dev_alloc(&M->xsq, (size_t)Hm * M->n_pad)) return rc;
    if (int rc = dev_alloc(&M->Lmat, (size_t)Hm * nn)) return rc;
    if (int rc = dev_alloc(&M->Linv, (size_t)Hm * nn)) return rc;
    // blocks above the block diagonal are never written afterwards and must read as zero (contractions, matvecs)
    BOCF_CUDA_OK(cudaMemsetAsync(M->Linv, 0, sizeof(double) * (size_t)Hm * nn, st));
    if (int rc = dev_alloc(&M->Dinv, (size_t)Hm * M->nb * TILE * TILE)) return rc;
    if (int rc = dev_alloc(&M->alpha, (size_t)Hm * M->n_pad)) return rc;
    if (int rc = dev_alloc(&M->tvec, (size_t)Hm * M->n_pad)) return rc;
    if (int rc = dev_alloc(&M->info, (size_t)Hm)) return rc;
  }
  for (auto& o : M->hyp_host) o.jitter = 0.0;
  std::vector<int> info(Hm, 0);
  std::vector<int> tries(Hm, 0);
  // jitchol (GPy/util/linalg.py:52-83): plain dpotrf first; on failure jitter = mean(diag) * 1e-6, then up to
  // maxtries = 5 attempts, jitter *= 10 after each failure.
  for (int attempt = 0; attempt <= 5; ++attempt) {
    BOCF_CUDA_OK(cudaMemcpyAsync(M->hyp, M->hyp_host.data(), sizeof(OutHyp) * Hm, cudaMemcpyHostToDevice, st));
    if (int rc = launch_prepare(M, st)) return rc;
    BOCF_CUDA_OK(cudaMemsetAsync(M->info, 0, sizeof(int) * Hm, st));
    // optimistic: the inverse and alpha are queued behind the factor without waiting for the pivot flags (a failed
    // factor carries unit pivots, so the work is finite and simply redone after the jitter retry): one host
    // synchronisation per factorisation instead of two -- the fit loops factorise thousands of times
    if (int rc = for_each_output_group(
            M, st,
            [](bocf_model* Mm, OutRun grp, cudaStream_t s, void*) -> int {
              if (int r = launch_gram(Mm, grp, s)) return r;
              if (int r = launch_cholesky(Mm, grp, s)) return r;
              return launch_inverse_and_alpha(Mm, grp, s);
            },
            nullptr))
      return rc;
    BOCF_CUDA_OK(cudaMemcpyAsync(info.data(), M->info, sizeof(int) * Hm, cudaMemcpyDeviceToHost, st));
    BOCF_CUDA_OK(cudaStreamSynchronize(st));
    bool any_fail = false;
    for (int hj = 0; hj < Hm; ++hj) {
      if (info[hj] == 0) continue;
      any_fail = true;
      OutHyp& o = M->hyp_host[hj];
      const double diag_mean = o.variance + o.noise + 1e-8;     // every diagonal entry of Ky is equal
      if (diag_mean <= 0.0) {
        set_error("not pd: non-positive diagonal elements");
        return BOCF_ERR_NONPOS_DIAG;
      }
      o.jitter = (tries[hj] == 0) ? diag_mean * 1e-6 : o.jitter * 10.0;
      tries[hj] += 1;
      if (tries[hj] > 5 || !std::isfinite(o.jitter)) {
        set_error("not positive definite, even with jitter.");
        return BOCF_ERR_NOT_PD;
      }
    }
    if (!any_fail) break;
  }
  if (jitter_out)
    for (int hj = 0; hj < Hm; ++hj) jitter_out[hj] = M->hyp_host[hj].jitter;
  // the digit planes belong to the previous factor: rebuilt lazily by the first posterior / acquisition call, so
  // likelihood-only users (ML-II, HMC: hundreds of factorisations per fit) never pay for them
  M->split_ready = false;
  M->precision_resolved = false;
  M->factorized = true;
  return 0;
}

int bocf_model_append_point(bocf_model* M, const double* x_new, const double* y_new, void* stream) {
  if (int rc = check_ready(M)) return rc;
  if (!x_new || !y_new) {
    set_error("bocf_model_append_point: invalid arguments");
    return BOCF_ERR_INVALID;
  }
  if (M->n + 1 > M->n_pad) {
    set_error("bocf_model_append_point: factor buffers are full (n is a multiple of 128); call bocf_model_set_data + "
              "bocf_model_factorize");
    return BOCF_ERR_UNSUPPORTED;
  }
  DeviceGuard dg(M->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int n_old = M->n, Hm = M->H * M->m;
  double *Xn = nullptr, *Yn = nullptr, *work = nullptr;
  if (int rc = dev_alloc(&Xn, (size_t)(n_old + 1) * M->d)) return rc;
  if (int rc = dev_alloc(&Yn, (size_t)(n_old + 1) * M->m)) {
    dev_free(Xn);
    return rc;
  }
  if (int rc = dev_alloc(&work, (size_t)Hm * 2 * M->n_pad)) {
    dev_free(Xn);
    dev_free(Yn);
    return rc;
  }
  int rc = launch_append_xy(M->X, M->Y, x_new, y_new, n_old, M->d, M->m, Xn, Yn, st);
  if (!rc) {
    cudaStreamSynchronize(st);
    dev_free(M->X);
    dev_free(M->Y);
    M->X = Xn;
    M->Y = Yn;
    Xn = Yn = nullptr;
    M->n = n_old + 1;
    M->n16 = (int)round_up(M->n, 16);
    rc = launch_append(M, n_old, work, st);
  }
  std::vector<int> info(Hm, 0);
  if (!rc && (cudaMemcpyAsync(info.data(), M->info, sizeof(int) * Hm, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
              cudaStreamSynchronize(st) != cudaSuccess)) {
    set_error("bocf_model_append_point: device error");
    rc = BOCF_ERR_CUDA;
  }
  dev_free(Xn);
  dev_free(Yn);
  dev_free(work);
  M->split_ready = false;                  // digit planes belong to the previous factor
  M->precision_resolved = false;
  if (rc) {
    M->factorized = false;
    return rc;
  }
  for (int hj = 0; hj < Hm; ++hj)
    if (info[hj] != 0) {
      M->factorized = false;               // data are in place: bocf_model_factorize (with its jitter schedule) recovers
      set_error("bocf_model_append_point: bordered pivot not positive; refactorise with bocf_model_factorize");
      return BOCF_ERR_UNSUPPORTED;
    }
  return 0;
}

int bocf_model_log_likelihood(bocf_model* M, double* lml, double* g_variance, double* g_lengthscale, double* g_noise,
                              void* stream) {
  if (int rc = check_ready(M)) return rc;
  if (!lml) {
    set_error("bocf_model_log_likelihood: lml must not be NULL");
    return BOCF_ERR_INVALID;
  }
  DeviceGuard dg(M->device);
  const int Hm = M->H * M->m;
  std::vector<double> buf((size_t)Hm * (MAXD + 3));
  if (int rc = launch_log_likelihood(M, buf.data(), static_cast<cudaStream_t>(stream))) return rc;
  for (int hj = 0; hj < Hm; ++hj) {
    const double* o = buf.data() + (size_t)hj * (MAXD + 3);
    lml[hj] = o[0];
    if (g_variance) g_variance[hj] = o[1];
    if (g_noise) g_noise[hj] = o[2];
    if (g_lengthscale)
      for (int q = 0; q < M->d; ++q) g_lengthscale[(size_t)hj * M->d + q] = o[3 + q];
  }
  return 0;
}

int bocf_model_get_factor(bocf_model* M, int h, int j, double* L, double* Linv, double* alpha, void* stream) {
  if (int rc = check_ready(M)) return rc;
  if (h < 0 || h >= M->H || j < 0 || j >= M->m) {
    set_error("bocf_model_get_factor: index out of range");
    return BOCF_ERR_INVALID;
  }
  DeviceGuard dg(M->device);
  return launch_copy_factor(M, h * M->m + j, L, Linv, alpha, static_cast<cudaStream_t>(stream));
}

// gather chunk-local (m x Nc [x d]) results into the caller's (m x N [x d]) arrays
static int scatter_out(const double* src, int64_t Nc, double* dst, int64_t N, int64_t off, int64_t cnt, int m,
                       int inner, cudaStream_t st) {
  if (!dst) return 0;
  BOCF_CUDA_OK(cudaMemcpy2DAsync(dst + off * inner, sizeof(double) * N * inner, src, sizeof(double) * Nc * inner,
                                 sizeof(double) * cnt * inner, m, cudaMemcpyDeviceToDevice, st));
  return 0;
}

int bocf_posterior(bocf_model* M, int h, const double* Xc, int64_t N, int noiseless, double* mean, double* var,
                   double* dmean, double* dvar, void* stream) {
  if (int rc = check_ready(M)) return rc;
  if (h < 0 || h >= M->H || !Xc || N < 0 || noiseless < 0 || noiseless > 2) {
    set_error("bocf_posterior: invalid arguments");
    return BOCF_ERR_INVALID;
  }
  if (N == 0) return 0;
  DeviceGuard dg(M->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = resolve_precision(M, st)) return rc;
  const bool grad = (dvar != nullptr) || (dmean != nullptr);
  const int64_t Nc = pick_chunk(M, N, grad, 0);
  if (int rc = ensure_scratch(M, chunk_bytes_per_candidate(M, grad, Nc) * Nc + kstar_part_bytes(M, Nc) + (1 << 16))) return rc;
  ChunkBuffers cb;
  carve_chunk(M, M->scratch, Nc, grad, &cb);
  for (int64_t off = 0; off < N; off += Nc) {
    const int64_t cnt = (N - off < Nc) ? N - off : Nc;
    // the mean alone: the mean-only K* pass (bitwise the same mean, nothing else written)
    if (int rc = (var || grad) ? launch_posterior_chunk(M, h, Xc + off * M->d, cnt, grad, noiseless, cb, st, var != nullptr,
                                                        dvar != nullptr)
                               : launch_posterior_mean_chunk(M, h, Xc + off * M->d, cnt, cb, st))
      return rc;
    if (int rc = scatter_out(cb.mean, Nc, mean, N, off, cnt, M->m, 1, st)) return rc;
    if (var)
      if (int rc = scatter_out(cb.var, Nc, var, N, off, cnt, M->m, 1, st)) return rc;
    if (dmean)
      if (int rc = scatter_out(cb.dmean, Nc, dmean, N, off, cnt, M->m, M->d, st)) return rc;
    if (dvar)
      if (int rc = scatter_out(cb.dvar, Nc, dvar, N, off, cnt, M->m, M->d, st)) return rc;
  }
  return 0;
}

int bocf_posterior_cov_point(bocf_model* M, int h, const double* Xc, int64_t N, const double* x2, double* cov,
                             double* dcov, void* stream) {
  if (int rc = check_ready(M)) return rc;
  if (h < 0 || h >= M->H || !Xc || !x2 || !cov || N < 0) {
    set_error("bocf_posterior_cov_point: invalid arguments");
    return BOCF_ERR_INVALID;
  }
  if (N == 0) return 0;
  DeviceGuard dg(M->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = ensure_scratch(M, sizeof(double) * 3 * (size_t)M->m * M->n_pad + 256)) return rc;
  return launch_cov_point(M, h, Xc, N, x2, cov, dcov, reinterpret_cast<double*>(M->scratch), st);
}

// Pruned sweep.  EI-CF and PI-CF are exactly zero, with a zero gradient, at a candidate none of whose base samples can
// beat the incumbent, and with uniformly spread candidates that is nearly all of them.  For composites whose maximum over
// a segment has a closed form, prune_bound_kernel (acq.cu) proves it from the posterior mean alone.  A call of at least
// PRUNE_MIN_N candidates then runs, chunk by chunk and for every hyper-sample, the mean-only K* pass and the bound over
// all candidates; lists the survivors on the device and reads their number (one stream synchronisation); and runs the
// unchanged chunk x hyper-sample sweep over the survivors, gathered into dense chunks of the size the full sweep uses, and
// scatters the results, zeros elsewhere.  Each survivor's result is bitwise the full sweep's, since no kernel's result for
// a candidate depends on where in its chunk it sits, with two exceptions that the sweep avoids: the chunk size, which sets
// the partial-sum split of the contractions, and a chunk of <= 128 candidates, which the MC pass and the gradient sum take
// through their latency-bound variants (the survivors' last chunk is padded past that; candidates that sit in such a
// last chunk in the full sweep can differ from it in the last bits).  The first chunk is a probe with a second
// synchronisation: when it keeps more than PRUNE_KEEP_MAX of its candidates (a pool concentrated near the incumbent) the
// call runs the full sweep and has lost only the probe.  Smaller calls, such as the acquisition optimiser's L-BFGS rounds
// of <= 128 candidates, never pay the synchronisations.
constexpr int64_t PRUNE_MIN_N = 16384;
constexpr double PRUNE_KEEP_MAX = 0.5;
static_assert(CAND_TILE > 128, "a survivor chunk padded to 129 candidates must fit the smallest chunk pick_chunk returns");

int bocf_acq_eval(bocf_model* M, int variant, int composite, const double* Xc, int64_t N, const double* Zt, int S,
                  const double* theta, int L, int p, const double* weight, const double* fstar, int H_use,
                  int with_grad_formula, double* acq, double* dacq, void* stream) {
  if (int rc = check_ready(M)) return rc;
  const bool mc = (variant == BOCF_ACQ_EI_CF || variant == BOCF_ACQ_PI_CF || variant == BOCF_ACQ_MEAN_UTILITY);
  const bool marginal = (variant == BOCF_ACQ_MEAN_UTILITY || variant == BOCF_ACQ_PSI);   // cbo._current_marginal_argmax
  if (!Xc || N < 0 || !acq || L < 1 || !weight || !fstar || H_use < 1 || H_use > M->H || variant < 0 ||
      variant > BOCF_ACQ_PSI || (mc && (!Zt || S < 1)) || (p > 0 && !theta)) {
    set_error("bocf_acq_eval: invalid arguments");
    return BOCF_ERR_INVALID;
  }
  if (variant == BOCF_ACQ_PI_CF && dacq) {
    set_error("uPI has no analytical gradient (uPI.py:19 analytical_gradient_prediction = False)");
    return BOCF_ERR_UNSUPPORTED;
  }
  if (!mc && !marginal && p != M->m) {
    set_error("maEI/maPI need theta of length m (linear scalarisation)");
    return BOCF_ERR_INVALID;
  }
  if (mc || marginal) {
    int need_p = (composite == BOCF_U_SUMSQ_TARGET || composite == BOCF_U_LINEAR) ? M->m
                 : (composite == BOCF_U_ROSEN_COMPOSITE ? 1 : 0);
    if (is_user_composite(composite)) {
      int um = 0;
      if (int rc = user_composite_info(composite, &um, &need_p)) return rc;
      if (variant == BOCF_ACQ_PSI) {
        set_error("bocf_acq_eval: a user-defined composite has no closed-form expectation: use BOCF_ACQ_MEAN_UTILITY");
        return BOCF_ERR_UNSUPPORTED;
      }
      if (um != M->m) {
        set_error("bocf_acq_eval: the composite was registered for " + std::to_string(um) + " outputs, the model has " +
                  std::to_string(M->m));
        return BOCF_ERR_INVALID;
      }
    }
    if (p < need_p) {
      set_error("bocf_acq_eval: theta has too few entries for this composite");
      return BOCF_ERR_INVALID;
    }
  }
  if (N == 0) return 0;
  DeviceGuard dg(M->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = resolve_precision(M, st)) return rc;
  const bool grad = (dacq != nullptr);
  M->swept_candidates = N;
  M->swept_survivors = N;

  // small host-side parameters (theta, weights, f*): staged through a handle-owned ring of PINNED slots and copied
  // to a matching ring of device slots, so the call never synchronises the stream (the L-BFGS rounds of the acquisition
  // optimiser are latency-bound: ~100 calls of <= 17 candidates per BO iteration).  A slot is reused only after the copy
  // that read it has completed (event per slot).
  const size_t n_theta = (size_t)L * (p > 0 ? p : 1);
  const size_t par_doubles = n_theta + (size_t)L + (size_t)H_use * L;
  const int64_t Nc = pick_chunk(M, N, grad, 0);
  const uint64_t chunk_bytes = chunk_bytes_per_candidate(M, grad, Nc) * Nc + kstar_part_bytes(M, Nc) + (1 << 16);
  const int d = M->d;
  bool prune = N >= PRUNE_MIN_N && prune_supported(variant, composite);
  for (int l = 0; l < L && prune; ++l) prune = std::isfinite(weight[l]);   // the full sweep's 0 * weight would be a NaN
  // pruned sweep, on top of the chunk: survivor flags, list-scan blocks, count, survivor list (N of each), gathered
  // candidates and compacted results (one chunk)
  const int64_t b_flags = round_up(N, 256), b_work = round_up((int64_t)prune_list_work_bytes(N), 256), b_count = 256;
  const int64_t b_list = round_up(N * 8, 256), b_x = Nc * d * 8, b_acq = Nc * 8, b_dacq = grad ? Nc * d * 8 : 0;
  const uint64_t prune_bytes = prune ? (uint64_t)(b_flags + b_work + b_count + b_list + b_x + b_acq + b_dacq) : 0;
  const uint64_t prune_off = (uint64_t)round_up((int64_t)chunk_bytes, 256);
  if (int rc = ensure_scratch(M, prune_off + prune_bytes + 256)) return rc;
  ChunkBuffers cb;
  carve_chunk(M, M->scratch, Nc, grad, &cb);
  double* par = nullptr;
  if (int rc = stage_params(M, par_doubles, &par, st, [&](double* host) {
        if (p > 0) std::memcpy(host, theta, sizeof(double) * L * p);
        else host[0] = 0.0;
        std::memcpy(host + n_theta, weight, sizeof(double) * L);
        std::memcpy(host + n_theta + L, fstar, sizeof(double) * H_use * L);
      }))
    return rc;

  AcqParams P;
  P.variant = variant;
  P.composite = composite;
  P.m = M->m;
  P.d = M->d;
  P.S = S;
  P.L = L;
  P.p = p;
  P.with_grad_formula = with_grad_formula;
  P.Zt = Zt;
  P.theta = par;
  P.weight = par + n_theta;
  // cbo.py:171 "the value of these functions is not normalized": plain sums over Z samples and hyper-samples
  P.scale = marginal ? 1.0 : (mc ? 1.0 / ((double)H_use * (double)S) : 1.0 / (double)H_use);
  const bool mean_only = (variant == BOCF_ACQ_PSI && composite == BOCF_U_LINEAR);   // posterior-mean branch: no contraction

  // Variants with gradients on the tensor-core contraction path: the fused gradient sweep (posterior.cu) -- the
  // per-output mean / variance gradients are never materialised (MC variants; the analytic ones up to 16 outputs, whose
  // weights live in registers).
  const bool fused = grad && M->S > 0 &&
                     (variant == BOCF_ACQ_EI_CF || variant == BOCF_ACQ_MEAN_UTILITY ||
                      ((variant == BOCF_ACQ_MA_EI || variant == BOCF_ACQ_MA_PI) && M->m <= 16));
  // cnt candidates X (one chunk) through every hyper-sample into a, g
  auto sweep = [&](const double* X, int64_t cnt, double* a, double* g) -> int {
    for (int h = 0; h < H_use; ++h) {
      P.fstar = par + n_theta + L + (size_t)h * L;
      P.accumulate = (h > 0) ? 1 : 0;
      if (fused) {
        if (int rc = launch_fused_grad_chunk(M, h, X, cnt, marginal ? 1 : 0, cb, P, a, g, st)) return rc;
        continue;
      }
      if (int rc = launch_posterior_chunk(M, h, X, cnt, grad, marginal ? 1 : 0, cb, st, !mean_only, !mean_only)) return rc;
      if (int rc = launch_acq_chunk(P, cb, cnt, a, g, st)) return rc;
    }
    return 0;
  };
  if (prune) {
    char* base = reinterpret_cast<char*>(M->scratch) + prune_off;
    uint8_t* flags = reinterpret_cast<uint8_t*>(base);
    void* work = base + b_flags;
    int64_t* count = reinterpret_cast<int64_t*>(base + b_flags + b_work);
    int64_t* list = reinterpret_cast<int64_t*>(base + b_flags + b_work + b_count);
    double* Xg = reinterpret_cast<double*>(base + b_flags + b_work + b_count + b_list);
    double* acq_c = Xg + Nc * d;
    double* dacq_c = grad ? acq_c + Nc : nullptr;
    if (!M->prune_count_host)
      BOCF_CUDA_OK(cudaHostAlloc(reinterpret_cast<void**>(&M->prune_count_host), sizeof(int64_t), cudaHostAllocDefault));
    auto bound = [&](int64_t off, int64_t cnt) -> int {
      for (int h = 0; h < H_use; ++h) {
        P.fstar = par + n_theta + L + (size_t)h * L;
        if (int rc = launch_posterior_mean_chunk(M, h, Xc + off * d, cnt, cb, st)) return rc;
        if (int rc = launch_prune_bound(P, M->hyp + (size_t)h * M->m, cb, cnt, h == 0, flags + off, st)) return rc;
      }
      return 0;
    };
    auto survivors = [&](int64_t n, int64_t* out_list, int64_t* kept) -> int {
      if (int rc = launch_prune_list(flags, n, out_list, count, work, st)) return rc;
      BOCF_CUDA_OK(cudaMemcpyAsync(M->prune_count_host, count, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
      BOCF_CUDA_OK(cudaStreamSynchronize(st));
      *kept = *M->prune_count_host;
      return 0;
    };
    const int64_t n0 = std::min(N, Nc);
    int64_t kept = 0;
    if (int rc = bound(0, n0)) return rc;
    if (int rc = survivors(n0, nullptr, &kept)) return rc;
    prune = kept <= PRUNE_KEEP_MAX * (double)n0;
    if (prune) {
      for (int64_t off = n0; off < N; off += Nc)
        if (int rc = bound(off, std::min(Nc, N - off))) return rc;
      if (int rc = survivors(N, list, &kept)) return rc;
      M->swept_survivors = kept;
      if (int rc = launch_prune_zero(flags, N, d, acq, dacq, st)) return rc;
      for (int64_t off = 0; off < kept; off += Nc) {
        const int64_t cnt = std::min(Nc, kept - off);
        const int64_t run = (cnt <= 128) ? 129 : cnt;     // fits: Nc >= CAND_TILE > 128 (pick_chunk, static_assert)
        if (int rc = launch_prune_gather(Xc, d, list + off, kept - 1 - off, run, Xg, st)) return rc;
        if (int rc = sweep(Xg, run, acq_c, dacq_c)) return rc;
        if (int rc = launch_prune_scatter(acq_c, dacq_c, list + off, cnt, d, acq, dacq, st)) return rc;
      }
      return 0;
    }
  }
  for (int64_t off = 0; off < N; off += Nc) {
    const int64_t cnt = (N - off < Nc) ? N - off : Nc;
    if (int rc = sweep(Xc + off * d, cnt, acq + off, grad ? dacq + off * d : nullptr)) return rc;
  }
  return 0;
}

int bocf_acq_eval_host(bocf_model* M, int variant, int composite, const double* Xc_host, int64_t N,
                       const double* Zt_dev, int S, const double* theta, int L, int p, const double* weight,
                       const double* fstar, int H_use, int with_grad_formula, double* acq_host, double* dacq_host,
                       void* stream) {
  if (int rc = check_ready(M)) return rc;
  if (!Xc_host || !acq_host || N < 0) {
    set_error("bocf_acq_eval_host: invalid arguments");
    return BOCF_ERR_INVALID;
  }
  if (N == 0) return 0;
  DeviceGuard dg(M->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // grow-only device staging owned by the handle (cudaMalloc / cudaFree per call cost more than a small sweep)
  const size_t need = (size_t)N * (2 * M->d + 1);
  if (M->io_doubles < need) {
    cudaStreamSynchronize(st);
    if (M->io_buf) cudaFree(M->io_buf);
    M->io_buf = nullptr;
    M->io_doubles = 0;
    if (int rc0 = dev_alloc(&M->io_buf, need)) return rc0;
    M->io_doubles = need;
  }
  double* dX = M->io_buf;
  double* dA = dX + (size_t)N * M->d;
  double* dG = dacq_host ? dA + N : nullptr;
  int rc = 0;
  do {
    if (cudaMemcpyAsync(dX, Xc_host, sizeof(double) * N * M->d, cudaMemcpyHostToDevice, st) != cudaSuccess) {
      set_error("H2D copy of candidates failed");
      rc = BOCF_ERR_CUDA;
      break;
    }
    if ((rc = bocf_acq_eval(M, variant, composite, dX, N, Zt_dev, S, theta, L, p, weight, fstar, H_use,
                            with_grad_formula, dA, dG, stream)))
      break;
    if (cudaMemcpyAsync(acq_host, dA, sizeof(double) * N, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        (dG && cudaMemcpyAsync(dacq_host, dG, sizeof(double) * N * M->d, cudaMemcpyDeviceToHost, st) != cudaSuccess) ||
        cudaStreamSynchronize(st) != cudaSuccess) {
      set_error("D2H copy of results failed");
      rc = BOCF_ERR_CUDA;
      break;
    }
  } while (0);
  return rc;
}

static int utility_eval(const char* fn, int composite, int m, const double* Y, int64_t N, const double* theta, int L,
                        int p, double* out, bool grad, void* stream) {
  if (!Y || !out || N < 0 || L < 1 || m < 1 || (p > 0 && !theta)) {
    set_error(std::string(fn) + ": invalid arguments");
    return BOCF_ERR_INVALID;
  }
  if (is_user_composite(composite)) {
    int um = 0, need_p = 0;
    if (int rc = user_composite_info(composite, &um, &need_p)) return rc;
    if (um != m || p < need_p) {
      set_error(std::string(fn) + ": the composite was registered for " + std::to_string(um) + " outputs and " +
                std::to_string(need_p) + " parameter entries (got m = " + std::to_string(m) + ", p = " +
                std::to_string(p) + ")");
      return BOCF_ERR_INVALID;
    }
  }
  if (N == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  double* dth = nullptr;
  const size_t n_theta = (size_t)L * (p > 0 ? p : 1);
  if (int rc = dev_alloc(&dth, n_theta)) return rc;
  int rc = 0;
  if (p > 0 && cudaMemcpyAsync(dth, theta, sizeof(double) * L * p, cudaMemcpyHostToDevice, st) != cudaSuccess) {
    set_error("H2D copy of theta failed");
    rc = BOCF_ERR_CUDA;
  }
  if (!rc) rc = launch_utility_eval(composite, m, Y, N, dth, L, p, out, grad, st);
  if (cudaStreamSynchronize(st) != cudaSuccess && !rc) {
    set_error(std::string(fn) + ": stream sync failed");
    rc = BOCF_ERR_CUDA;
  }
  dev_free(dth);
  return rc;
}

int bocf_utility_eval(int composite, int m, const double* Y, int64_t N, const double* theta, int L, int p,
                      double* out, void* stream) {
  return utility_eval("bocf_utility_eval", composite, m, Y, N, theta, L, p, out, false, stream);
}

int bocf_utility_grad_eval(int composite, int m, const double* Y, int64_t N, const double* theta, int L, int p,
                           double* out, void* stream) {
  return utility_eval("bocf_utility_grad_eval", composite, m, Y, N, theta, L, p, out, true, stream);
}

int bocf_topk(const double* acq, const double* Xc, int64_t N, int d, int k, int64_t index_offset, double* out_rec,
              void* stream) {
  if (!acq || !Xc || !out_rec || N < 1 || d < 1 || k < 1) {
    set_error("bocf_topk: invalid arguments");
    return BOCF_ERR_INVALID;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // grow-only workspace per device (stream-ordered pool allocations are trimmed back to the OS at every
  // synchronisation with the default release threshold, which stalls the device between steps)
  static void* ws_cache[64] = {nullptr};
  static uint64_t ws_bytes[64] = {0};
  int dev = 0;
  BOCF_CUDA_OK(cudaGetDevice(&dev));
  const uint64_t need = topk_workspace_bytes(N, k);
  if (dev < 0 || dev >= 64) {
    set_error("bocf_topk: unsupported device ordinal");
    return BOCF_ERR_INVALID;
  }
  if (ws_bytes[dev] < need) {
    if (ws_cache[dev]) cudaFree(ws_cache[dev]);
    ws_cache[dev] = nullptr;
    ws_bytes[dev] = 0;
    BOCF_CUDA_OK(cudaMalloc(&ws_cache[dev], need));
    ws_bytes[dev] = need;
  }
  return launch_topk(acq, Xc, N, d, k, index_offset, out_rec, ws_cache[dev], st);
}

}  // extern "C"
