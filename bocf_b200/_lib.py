"""ctypes binding of libbocf_b200.so (C ABI in include/bocf_b200.h).

There is no CPU fallback: if the CUDA library is missing or a call fails, a
RuntimeError is raised with the library's own message.
"""
import ctypes
import os
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BOCF_LIB_PATH") or os.path.join(_HERE, "csrc", "libbocf_b200.so")   # override: kernel-variant experiments
_lib = None

KERNELS = {"se": 0, "rbf": 1, "matern52": 2, "matern32": 3}
COMPOSITES = {"sumsq_target": 0, "neg_sum_exp": 1, "exp_cos": 2, "rosen_composite": 3, "linear": 4}
COMPOSITE_USER_BASE = 1024      # BOCF_U_USER: ids of composites registered with bocf_composite_register
VARIANTS = {"ei_cf": 0, "pi_cf": 1, "ma_ei": 2, "ma_pi": 3, "mean_utility": 4, "psi": 5}

EXPORTS = [
    "bocf_last_error", "bocf_version", "bocf_launch_count",
    "bocf_model_create", "bocf_model_set_kernels", "bocf_model_destroy", "bocf_model_set_data", "bocf_model_set_hypers",
    "bocf_model_factorize", "bocf_model_get_factor", "bocf_model_n", "bocf_model_H",
    "bocf_model_set_scratch_limit", "bocf_posterior", "bocf_posterior_cov_point", "bocf_acq_eval", "bocf_acq_eval_host",
    "bocf_utility_eval", "bocf_utility_grad_eval", "bocf_composite_register", "bocf_topk", "bocf_profile_enable", "bocf_profile_report",
    "bocf_model_set_precision", "bocf_model_active_slices", "bocf_model_active_scheme", "bocf_model_chunk_candidates", "bocf_model_sweep_stats", "bocf_debug_split_gemm", "bocf_model_log_likelihood", "bocf_model_append_point",
]
# name -> (enum bocf_precision, slices).  "splitN": both contractions on the N-plane scheme; "splitNM": variance on N,
# variance gradient on M = N or N - 1 >= 3 planes, the pairs the library accepts (include/bocf_b200.h).
PRECISIONS = {"fp64": (0, 0), "auto": (2, 0), "mixed": (3, 0)}
for _s1 in range(3, 7):
    PRECISIONS["split%d" % _s1] = (1, _s1)
    for _s2 in range(max(3, _s1 - 1), _s1 + 1):
        PRECISIONS["split%d%d" % (_s1, _s2)] = (1, 10 * _s1 + _s2)


def parse_precision(name):
    try:
        return PRECISIONS[str(name).lower()]
    except KeyError:
        raise ValueError("precision must be one of %s" % sorted(PRECISIONS))


class BocfError(RuntimeError):
    def __init__(self, code, msg):
        super(BocfError, self).__init__("libbocf_b200 error %d: %s" % (code, msg))
        self.code = code


class NotPositiveDefiniteError(BocfError):
    """Mirrors numpy.linalg.LinAlgError('not positive definite, even with jitter.') of GPy/util/linalg.py:71."""


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libbocf_b200.so not built (%s). Run `python __graft_entry__.py` (nvcc, sm_100a). "
            "bocf_b200 has no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    c_dp = ctypes.c_void_p      # device or host double*; passed as raw addresses
    c_vp = ctypes.c_void_p
    i32, i64, u64 = ctypes.c_int, ctypes.c_int64, ctypes.c_uint64
    lib.bocf_last_error.restype = ctypes.c_char_p
    lib.bocf_version.restype = ctypes.c_char_p
    lib.bocf_launch_count.restype = u64
    lib.bocf_model_create.argtypes = [ctypes.POINTER(c_vp), i32, i32, i32, i32]
    lib.bocf_model_set_kernels.argtypes = [c_vp, ctypes.POINTER(i32), i32]
    lib.bocf_model_destroy.argtypes = [c_vp]
    lib.bocf_model_set_data.argtypes = [c_vp, i32, c_dp, c_dp, c_vp]
    lib.bocf_model_set_hypers.argtypes = [c_vp, i32, c_dp, c_dp, c_dp]
    lib.bocf_model_factorize.argtypes = [c_vp, c_dp, c_vp]
    lib.bocf_model_get_factor.argtypes = [c_vp, i32, i32, c_dp, c_dp, c_dp, c_vp]
    lib.bocf_model_n.argtypes = [c_vp]
    lib.bocf_model_H.argtypes = [c_vp]
    lib.bocf_model_set_scratch_limit.argtypes = [c_vp, u64]
    lib.bocf_posterior.argtypes = [c_vp, i32, c_dp, i64, i32, c_dp, c_dp, c_dp, c_dp, c_vp]
    lib.bocf_posterior_cov_point.argtypes = [c_vp, i32, c_dp, i64, c_dp, c_dp, c_dp, c_vp]
    lib.bocf_acq_eval.argtypes = [c_vp, i32, i32, c_dp, i64, c_dp, i32, c_dp, i32, i32, c_dp, c_dp, i32, i32,
                                  c_dp, c_dp, c_vp]
    lib.bocf_acq_eval_host.argtypes = lib.bocf_acq_eval.argtypes
    lib.bocf_utility_eval.argtypes = [i32, i32, c_dp, i64, c_dp, i32, i32, c_dp, c_vp]
    lib.bocf_utility_grad_eval.argtypes = lib.bocf_utility_eval.argtypes
    lib.bocf_composite_register.argtypes = [ctypes.c_char_p, i32, i32, ctypes.POINTER(i32)]
    lib.bocf_topk.argtypes = [c_dp, c_dp, i64, i32, i32, i64, c_dp, c_vp]
    lib.bocf_model_set_precision.argtypes = [c_vp, i32, i32, c_vp]
    lib.bocf_model_active_slices.argtypes = [c_vp]
    lib.bocf_model_active_scheme.argtypes = [c_vp]
    lib.bocf_model_chunk_candidates.argtypes = [c_vp, i64, i32]
    lib.bocf_model_chunk_candidates.restype = i64
    lib.bocf_model_sweep_stats.argtypes = [c_vp, ctypes.POINTER(i64), ctypes.POINTER(i64)]
    lib.bocf_debug_split_gemm.argtypes = [c_dp, c_dp, i32, i32, i32, i32, i32, c_dp, c_vp]
    lib.bocf_model_log_likelihood.argtypes = [c_vp, c_dp, c_dp, c_dp, c_dp, c_vp]
    lib.bocf_model_append_point.argtypes = [c_vp, c_dp, c_dp, c_vp]
    lib.bocf_profile_enable.argtypes = [i32]
    lib.bocf_profile_report.argtypes = [ctypes.c_char_p, i32]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name not in ("bocf_last_error", "bocf_version", "bocf_launch_count"):
            fn.restype = i32
    _lib = lib
    return lib


_nvrtc = None


def _nvrtc_candidates():
    yield "libnvrtc.so.12"
    for base in sys.path:                  # the copy bundled with the torch wheel, found without importing torch
        yield os.path.join(base, "nvidia", "cuda_nvrtc", "lib", "libnvrtc.so.12")
    for home in (os.environ.get("CUDA_HOME"), "/usr/local/cuda"):
        if home:
            yield os.path.join(home, "lib64", "libnvrtc.so.12")


def preload_nvrtc():
    """Load NVRTC with RTLD_GLOBAL, so the library's own dlopen("libnvrtc.so.12") at the first composite registration
    finds it by soname even when it is not on the loader's search path."""
    global _nvrtc
    if _nvrtc is None:
        for cand in _nvrtc_candidates():
            if os.path.isabs(cand) and not os.path.exists(cand):
                continue
            try:
                _nvrtc = ctypes.CDLL(cand, mode=ctypes.RTLD_GLOBAL)
                break
            except OSError:
                continue
    return _nvrtc


def register_composite(source, m, theta_len):
    """bocf_composite_register: compile a user composite for m outputs (theta_len -1 = m); returns its id."""
    lib = load_library()
    preload_nvrtc()
    out = ctypes.c_int(-1)
    check(lib.bocf_composite_register(source.encode("utf-8"), int(m), int(theta_len), ctypes.byref(out)))
    return out.value


def check(rc):
    if rc == 0:
        return
    msg = load_library().bocf_last_error().decode("utf-8", "replace")
    if rc == -3:
        raise NotPositiveDefiniteError(rc, msg)
    raise BocfError(rc, msg)


def profile_enable(on=True):
    load_library().bocf_profile_enable(1 if on else 0)


def profile_report():
    """{kernel class: (launches, total device ms)} since profile_enable(True); synchronises the device."""
    lib = load_library()
    buf = ctypes.create_string_buffer(1 << 16)
    lib.bocf_profile_report(buf, len(buf))
    out = {}
    for line in buf.value.decode().splitlines():
        name, cnt, ms = line.split()
        out[name] = (int(cnt), float(ms))
    return out


def launch_count():
    return int(load_library().bocf_launch_count())
