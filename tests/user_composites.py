"""User-defined composites for the CudaComposite tests: CUDA C++ sources (the contract of include/bocf_b200.h) with the
host callables of the same U(theta, y) / dU/dy.

RESTATED holds the five catalogued composites written as user source, in the built-in kernels' operation order (acq.cu
comp_phi / comp_dphi), so the user path can be held to the built-in one.  COUPLED_QUADRATIC and SOFTMIN are not
separable: no built-in composite can express them."""
import numpy as np

RESTATED = {
    "sumsq_target": ("m", r"""
__device__ double bocf_U(const double* th, const double* y) {
  double u = 0.0;
  for (int j = 0; j < BOCF_M; ++j) {
    const double a = y[j] - th[j];
    u += -(a * a);
  }
  return u;
}
__device__ void bocf_dU(const double* th, const double* y, double* g) {
  for (int j = 0; j < BOCF_M; ++j) g[j] = -2.0 * (y[j] - th[j]);
}
"""),
    "neg_sum_exp": (0, r"""
__device__ double bocf_U(const double* th, const double* y) {
  double u = 0.0;
  for (int j = 0; j < BOCF_M; ++j) u += -exp(y[j]);
  return u;
}
__device__ void bocf_dU(const double* th, const double* y, double* g) {
  for (int j = 0; j < BOCF_M; ++j) g[j] = -exp(y[j]);
}
"""),
    "exp_cos": (0, r"""
#define PI_ 3.1415926535897931
__device__ __forceinline__ double coef(int j) {
  const int k = j % 5;
  return k == 0 ? 1.0 : k == 1 ? 2.0 : k == 2 ? 5.0 : k == 3 ? 2.0 : 3.0;
}
__device__ double bocf_U(const double* th, const double* y) {
  double u = 0.0;
  for (int j = 0; j < BOCF_M; ++j) u += -(coef(j) * (exp(-y[j] / PI_) * cos(PI_ * y[j])));
  return u;
}
__device__ void bocf_dU(const double* th, const double* y, double* g) {
  for (int j = 0; j < BOCF_M; ++j) {
    const double e = exp(-y[j] / PI_);
    const double aux = -PI_ * (e * sin(PI_ * y[j])) - (e * cos(PI_ * y[j])) / PI_;
    g[j] = -(coef(j) * aux);
  }
}
"""),
    "rosen_composite": (1, r"""
__device__ double bocf_U(const double* th, const double* y) {
  const int h = BOCF_M / 2;
  double u = 0.0;
  for (int j = 0; j < BOCF_M; ++j) {
    if (j < h) {
      const double a = th[0] - y[j];
      u += -(a * a);
    } else if (j < 2 * h) {
      u += -(100.0 * (y[j] * y[j]));
    } else {
      u += 0.0;
    }
  }
  return u;
}
__device__ void bocf_dU(const double* th, const double* y, double* g) {
  const int h = BOCF_M / 2;
  for (int j = 0; j < BOCF_M; ++j) g[j] = (j < h) ? 2.0 * (th[0] - y[j]) : (j < 2 * h) ? -200.0 * y[j] : 0.0;
}
"""),
    "linear": ("m", r"""
__device__ double bocf_U(const double* th, const double* y) {
  double u = 0.0;
  for (int j = 0; j < BOCF_M; ++j) u += th[j] * y[j];
  return u;
}
__device__ void bocf_dU(const double* th, const double* y, double* g) {
  for (int j = 0; j < BOCF_M; ++j) g[j] = th[j];
}
"""),
}

RHO = 0.3

# -sum_j (y_j - theta_j)^2 - rho sum_j y_j y_{j+1}
COUPLED_QUADRATIC = r"""
__device__ double bocf_U(const double* th, const double* y) {
  double u = 0.0;
  for (int j = 0; j < BOCF_M; ++j) {
    const double a = y[j] - th[j];
    u -= a * a;
  }
  for (int j = 0; j + 1 < BOCF_M; ++j) u -= 0.3 * (y[j] * y[j + 1]);
  return u;
}
__device__ void bocf_dU(const double* th, const double* y, double* g) {
  for (int j = 0; j < BOCF_M; ++j) {
    double gj = -2.0 * (y[j] - th[j]);
    if (j > 0) gj -= 0.3 * y[j - 1];
    if (j + 1 < BOCF_M) gj -= 0.3 * y[j + 1];
    g[j] = gj;
  }
}
"""


# host callables take y as (m,) or as (m, N) columns (the oracle evaluates U over columns)
def coupled_quadratic_U(th, y):
    y = np.asarray(y, dtype=float)
    a = (y.T - np.asarray(th, dtype=float).reshape(-1)).T
    return -np.sum(a * a, axis=0) - RHO * np.sum(y[:-1] * y[1:], axis=0)


def coupled_quadratic_dU(th, y):
    y = np.asarray(y, dtype=float).reshape(-1)
    g = -2.0 * (y - np.asarray(th, dtype=float).reshape(-1))
    g[1:] -= RHO * y[:-1]
    g[:-1] -= RHO * y[1:]
    return g


TAU = 0.5

# soft minimum of the outputs, -tau log sum_j exp(-y_j / tau), in the stable log-sum-exp form; no parameter
SOFTMIN = r"""
__device__ double bocf_U(const double* th, const double* y) {
  double mn = y[0];
  for (int j = 1; j < BOCF_M; ++j) mn = fmin(mn, y[j]);
  double s = 0.0;
  for (int j = 0; j < BOCF_M; ++j) s += exp(-(y[j] - mn) / 0.5);
  return mn - 0.5 * log(s);
}
__device__ void bocf_dU(const double* th, const double* y, double* g) {
  double mn = y[0];
  for (int j = 1; j < BOCF_M; ++j) mn = fmin(mn, y[j]);
  double s = 0.0;
  for (int j = 0; j < BOCF_M; ++j) {
    g[j] = exp(-(y[j] - mn) / 0.5);
    s += g[j];
  }
  for (int j = 0; j < BOCF_M; ++j) g[j] /= s;
}
"""


def softmin_U(th, y):
    y = np.asarray(y, dtype=float)
    mn = y.min(axis=0)
    return mn - TAU * np.log(np.sum(np.exp(-(y - mn) / TAU), axis=0))


def softmin_dU(th, y):
    y = np.asarray(y, dtype=float).reshape(-1)
    w = np.exp(-(y - y.min()) / TAU)
    return w / w.sum()
