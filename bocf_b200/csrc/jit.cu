// jit.cu -- user-defined composites (bocf_composite_register): the user's CUDA source, followed by the kernel template
// acq_user.cuh, is compiled by NVRTC to an sm_100a cubin; the cubin is loaded as a context-independent library at the
// first launch, so one registration serves every device of the process.
//
// NVRTC is reached through dlopen("libnvrtc.so.12") at the first registration: the library keeps no link-time
// dependency on it, and a process that never registers a composite never needs it.
#include <dlfcn.h>
#include <nvrtc.h>

#include <cstdio>
#include <memory>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "common.cuh"
#include "model.h"

namespace bocf {
namespace {

// acq_user.cuh as a raw string literal, generated at build time (__graft_entry__.build_library)
const char kTemplate[] =
#include "acq_user_src.inc"
    ;

struct Nvrtc {
  decltype(&nvrtcGetErrorString) error_string;
  decltype(&nvrtcCreateProgram) create;
  decltype(&nvrtcDestroyProgram) destroy;
  decltype(&nvrtcCompileProgram) compile;
  decltype(&nvrtcGetProgramLogSize) log_size;
  decltype(&nvrtcGetProgramLog) log;
  decltype(&nvrtcGetCUBINSize) cubin_size;
  decltype(&nvrtcGetCUBIN) cubin;
  decltype(&nvrtcAddNameExpression) add_name;
  decltype(&nvrtcGetLoweredName) lowered_name;
};

constexpr int MC_SHAPES = 3;                      // block per candidate / warp per candidate / 4 candidates per warp
constexpr int MC_MODES = 7;
constexpr int K_UEVAL = MC_MODES * MC_SHAPES;     // kernel slots: mc_acq_user_kernel [mode][shape], then the two
constexpr int K_UGRAD = K_UEVAL + 1;              // utility kernels
constexpr int K_COUNT = K_UGRAD + 1;

struct UserComposite {
  std::string source;
  int m = 0, theta_len = 0;
  std::vector<char> cubin;
  std::string names[K_COUNT];                     // lowered (mangled) kernel names
  cudaLibrary_t lib = nullptr;                    // loaded at the first launch
  cudaKernel_t k[K_COUNT] = {};
};

std::mutex g_register_mu;                         // serialises registrations (one compile per new composite)
std::mutex g_mu;                                  // guards g_reg and the lazy library loads
std::vector<std::unique_ptr<UserComposite>> g_reg;

std::string name_expression(int slot) {
  if (slot == K_UEVAL) return "&bocf_user::utility_eval_user_kernel";
  if (slot == K_UGRAD) return "&bocf_user::utility_grad_eval_user_kernel";
  static const int shape[MC_SHAPES][2] = {{1, 8}, {1, 1}, {4, 1}};   // <MCB, NW>
  const int mode = slot / MC_SHAPES, s = slot % MC_SHAPES;
  char buf[96];
  std::snprintf(buf, sizeof(buf), "&bocf_user::mc_acq_user_kernel<%d, %d, %d>", mode, shape[s][0], shape[s][1]);
  return buf;
}

// NVRTC entry points; nullptr (message set) when the library cannot be loaded.  Called under g_register_mu.
const Nvrtc* nvrtc() {
  static Nvrtc fn;
  static bool loaded = false;
  if (loaded) return &fn;
  void* h = dlopen("libnvrtc.so.12", RTLD_NOW | RTLD_GLOBAL);
  if (!h) {
    const char* e = dlerror();
    set_error(std::string("bocf_composite_register: NVRTC is not available (dlopen libnvrtc.so.12: ") +
              (e ? e : "not found") + ")");
    return nullptr;
  }
  bool ok = true;
  auto sym = [&](auto& f, const char* name) {
    f = reinterpret_cast<std::remove_reference_t<decltype(f)>>(dlsym(h, name));
    ok = ok && f != nullptr;
  };
  sym(fn.error_string, "nvrtcGetErrorString");
  sym(fn.create, "nvrtcCreateProgram");
  sym(fn.destroy, "nvrtcDestroyProgram");
  sym(fn.compile, "nvrtcCompileProgram");
  sym(fn.log_size, "nvrtcGetProgramLogSize");
  sym(fn.log, "nvrtcGetProgramLog");
  sym(fn.cubin_size, "nvrtcGetCUBINSize");
  sym(fn.cubin, "nvrtcGetCUBIN");
  sym(fn.add_name, "nvrtcAddNameExpression");
  sym(fn.lowered_name, "nvrtcGetLoweredName");
  if (!ok) {
    set_error("bocf_composite_register: libnvrtc.so.12 lacks an entry point this library uses");
    return nullptr;
  }
  loaded = true;
  return &fn;
}

// compile source + template for m outputs into e->cubin / e->names
int compile(const Nvrtc& nv, UserComposite* e) {
  const std::string src = e->source + "\n#line 1 \"acq_user.cuh\"\n" + kTemplate;
  nvrtcProgram prog = nullptr;
  nvrtcResult r = nv.create(&prog, src.c_str(), "user_composite.cu", 0, nullptr, nullptr);
  if (r != NVRTC_SUCCESS) {
    set_error(std::string("bocf_composite_register: nvrtcCreateProgram: ") + nv.error_string(r));
    return BOCF_ERR_INVALID;
  }
  for (int s = 0; s < K_COUNT; ++s) nv.add_name(prog, name_expression(s).c_str());
  const std::string mdef = "-DBOCF_M=" + std::to_string(e->m);
  const char* opts[] = {"--gpu-architecture=sm_100a", "-std=c++17", mdef.c_str()};
  r = nv.compile(prog, 3, opts);
  int rc = 0;
  if (r != NVRTC_SUCCESS) {
    size_t n = 0;
    nv.log_size(prog, &n);
    std::string log(n, '\0');
    if (n) nv.log(prog, &log[0]);
    set_error(std::string("bocf_composite_register: the composite does not compile (") + nv.error_string(r) + "):\n" +
              log.c_str());
    rc = BOCF_ERR_INVALID;
  } else {
    size_t n = 0;
    nv.cubin_size(prog, &n);
    e->cubin.resize(n);
    nv.cubin(prog, e->cubin.data());
    for (int s = 0; s < K_COUNT && !rc; ++s) {
      const char* lowered = nullptr;
      if (nv.lowered_name(prog, name_expression(s).c_str(), &lowered) != NVRTC_SUCCESS || !lowered) {
        set_error("bocf_composite_register: no lowered name for " + name_expression(s));
        rc = BOCF_ERR_INVALID;
      } else {
        e->names[s] = lowered;
      }
    }
  }
  nv.destroy(&prog);
  return rc;
}

UserComposite* lookup(int composite) {
  const int idx = composite - BOCF_U_USER;
  std::lock_guard<std::mutex> g(g_mu);
  if (idx < 0 || idx >= (int)g_reg.size()) return nullptr;
  return g_reg[idx].get();
}

// the composite's kernels, its library loaded on first use
int kernels(int composite, const UserComposite** out) {
  UserComposite* e = lookup(composite);
  if (!e) {
    set_error("unknown composite " + std::to_string(composite));
    return BOCF_ERR_INVALID;
  }
  std::lock_guard<std::mutex> g(g_mu);
  if (!e->lib) {
    cudaLibrary_t lib = nullptr;
    BOCF_CUDA_OK(cudaLibraryLoadData(&lib, e->cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0));
    for (int s = 0; s < K_COUNT; ++s) {
      const cudaError_t err = cudaLibraryGetKernel(&e->k[s], lib, e->names[s].c_str());
      if (err != cudaSuccess) {
        cudaLibraryUnload(lib);
        set_error("cudaLibraryGetKernel " + e->names[s] + ": " + cudaGetErrorString(err));
        return BOCF_ERR_CUDA;
      }
    }
    e->lib = lib;
  }
  *out = e;
  return 0;
}

int launch(cudaKernel_t k, dim3 grid, dim3 block, void** args, cudaStream_t st, const char* name) {
  cudaLaunchKernel(reinterpret_cast<const void*>(k), grid, block, args, 0, st);   // a failure is the last error
  BOCF_LAUNCH_OK(name);
  return 0;
}

}  // namespace

bool is_user_composite(int composite) { return composite >= BOCF_U_USER; }

int user_composite_info(int composite, int* m, int* theta_len) {
  const UserComposite* e = lookup(composite);
  if (!e) {
    set_error("unknown composite " + std::to_string(composite));
    return BOCF_ERR_INVALID;
  }
  *m = e->m;
  *theta_len = e->theta_len < 0 ? e->m : e->theta_len;
  return 0;
}

int launch_mc_user(const AcqParams& P, const ChunkBuffers& cb, int64_t Nvalid, double* acq, double* dacq,
                   cudaStream_t st) {
  const UserComposite* e = nullptr;
  if (int rc = kernels(P.composite, &e)) return rc;
  // launch shapes and modes of acq.cu launch_mc_t
  const bool small = (Nvalid <= 1024), tiny = (Nvalid <= 128);
  const unsigned grid = tiny ? (unsigned)Nvalid : (unsigned)ceil_div(Nvalid, (int64_t)8 * (small ? 1 : 4));
  const bool weights = (P.wa != nullptr);
  const int mode = (P.variant == BOCF_ACQ_MEAN_UTILITY) ? (weights ? 6 : dacq ? 4 : 3)
                   : (P.variant == BOCF_ACQ_PI_CF)      ? 2
                                                         : (weights ? 5 : dacq ? 1 : 0);
  const int shape = tiny ? 0 : small ? 1 : 2;
  int64_t Nc = cb.Nc;
  int d = P.d, S = P.S, L = P.L, p = P.p, accumulate = P.accumulate;
  double scale = P.scale;
  const double *mean = cb.mean, *var = cb.var, *dmean = cb.dmean, *dvar = cb.dvar, *Zt = P.Zt, *theta = P.theta,
               *weight = P.weight, *fstar = P.fstar;
  double *wa = P.wa, *wb = P.wb;
  void* args[] = {&mean, &var, &dmean, &dvar, &Nc, &Nvalid, &d, &Zt, &S, &theta, &L, &p, &weight, &fstar, &scale,
                  &accumulate, &acq, &dacq, &wa, &wb};
  ProfScope ps("mc_acq_user_kernel", st);
  return launch(e->k[mode * MC_SHAPES + shape], dim3(grid), dim3(8 * 32), args, st, "mc_acq_user_kernel");
}

int launch_utility_eval_user(int composite, const double* Y, int64_t N, const double* theta, int L, int p, double* out,
                             bool grad, cudaStream_t st) {
  const UserComposite* e = nullptr;
  if (int rc = kernels(composite, &e)) return rc;
  void* args[] = {&Y, &N, &theta, &p, &out};
  const dim3 grid((unsigned)ceil_div(N, 256), (unsigned)L);
  ProfScope ps("utility_eval_user_kernel", st);
  return launch(e->k[grad ? K_UGRAD : K_UEVAL], grid, dim3(256), args, st, "utility_eval_user_kernel");
}

}  // namespace bocf

extern "C" {

int bocf_composite_register(const char* source, int m, int theta_len, int* composite_out) {
  using namespace bocf;
  if (!source || !composite_out || m < 1 || m > MAXM || theta_len < -1) {
    set_error("bocf_composite_register: invalid arguments (source and composite_out non-NULL, 1 <= m <= 64, "
              "theta_len >= -1)");
    return BOCF_ERR_INVALID;
  }
  std::lock_guard<std::mutex> reg(g_register_mu);
  {
    std::lock_guard<std::mutex> g(g_mu);
    for (size_t i = 0; i < g_reg.size(); ++i)
      if (g_reg[i]->m == m && g_reg[i]->theta_len == theta_len && g_reg[i]->source == source) {
        *composite_out = BOCF_U_USER + (int)i;
        return 0;
      }
  }
  const Nvrtc* nv = nvrtc();
  if (!nv) return BOCF_ERR_UNSUPPORTED;
  std::unique_ptr<UserComposite> e(new UserComposite());
  e->source = source;
  e->m = m;
  e->theta_len = theta_len;
  if (int rc = compile(*nv, e.get())) return rc;
  std::lock_guard<std::mutex> g(g_mu);
  g_reg.push_back(std::move(e));
  *composite_out = BOCF_U_USER + (int)g_reg.size() - 1;
  return 0;
}

}  // extern "C"
