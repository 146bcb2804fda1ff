"""K* latency at small batches (kstar_kernel splits the training points over blocks for chunks up to 1024 candidates):
wall time per call and per-kernel times, K* alone and with the full posterior."""
import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bocf_b200 import _lib
from tests.helpers import make_problem, product_model
P = make_problem(m=16, d=10, n=1000, H=1, kind="matern52", N=64, S=8, seed=0)
pm = product_model(P, "cuda:0")
for N in (17, 256, 1024):
    X = torch.rand((N, 10), dtype=torch.float64, device="cuda")
    for what, kw in (("K* only", dict(want_dmean=True)), ("full posterior", dict(want_var=True, want_dmean=True, want_dvar=True))):
        for _ in range(5):
            pm._posterior(X, **kw)
        torch.cuda.synchronize()
        _lib.profile_enable(True)
        t0 = time.perf_counter()
        for _ in range(50):
            pm._posterior(X, **kw)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) / 50
        prof = _lib.profile_report(); _lib.profile_enable(False)
        print("N=%4d %-15s wall %7.1f us/call  kernels(us): %s" % (N, what, 1e6 * wall,
              {k: round(1e3 * v[1] / v[0], 1) for k, v in prof.items()}), flush=True)
