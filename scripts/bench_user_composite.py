"""Step time of a user-defined composite (CudaComposite, NVRTC-compiled mc_acq_user_kernel) against the built-in one.

Workload: bench.py's cfg3 (m=16, d=10, n=1000, Matern-5/2, S=1024, H=1, L=1) on 1M device-resident candidates, one step
= EI-CF value + gradient (the fused gradient path) + local top-16, as bench.py times it.  Three utilities:
  builtin   composite="sumsq_target" (acq.cu mc_acq_kernel)
  restated  the same U(theta, y) written as user source (tests/user_composites.py)
  coupled   -sum (y_j - theta_j)^2 - 0.3 sum y_j y_{j+1}: not separable, no built-in equivalent
on two candidate draws: `uniform` (bench.py's draw: almost no candidate improves on f*, so the gradient pass of the MC
kernel is nearly idle) and `focused` (make_problem's draw, 75 % of candidates next to the best observations, where the
gradient pass runs).  The utilities are alternated round by round in one process; a 256 MiB buffer is overwritten
between steps so no step reads the previous one's data from L2.  A separate profiled pass per utility reports the MC
kernel's device time (per-kernel CUDA events, bocf_profile_report).  Prints one JSON line.

  python scripts/bench_user_composite.py [--candidates 1000000] [--steps 3] [--rounds 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception:
        import torch
        return torch.cuda.get_device_name(), None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--candidates", type=int, default=1000000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import torch
    import bocf_b200
    from bocf_b200 import _lib, distributed as bd
    from bocf_b200.utility import _host_funcs
    from tests.helpers import make_problem, product_model
    from tests.user_composites import COUPLED_QUADRATIC, RESTATED, coupled_quadratic_U, coupled_quadratic_dU
    if not torch.cuda.is_available():
        raise RuntimeError("needs a CUDA device")
    dev = torch.device("cuda", 0)
    _lib.load_library()
    m, d, n, S = 16, 10, 1000, 1024
    P = make_problem(m=m, d=d, n=n, H=1, kind="matern52", composite="sumsq_target", N=args.candidates, S=S, L=1, seed=0)
    model = product_model(P, str(dev))
    pd = bocf_b200.ParameterDistribution(support=P.theta, prob_dist=P.prob)
    fu, dfu = _host_funcs("sumsq_target")
    utils = {
        "builtin": bocf_b200.Utility(parameter_dist=pd, composite="sumsq_target"),
        "restated": bocf_b200.Utility(func=fu, dfunc=dfu, parameter_dist=pd,
                                      composite=bocf_b200.CudaComposite(RESTATED["sumsq_target"][1])),
        "coupled": bocf_b200.Utility(func=coupled_quadratic_U, dfunc=coupled_quadratic_dU, parameter_dist=pd,
                                     composite=bocf_b200.CudaComposite(COUPLED_QUADRATIC)),
    }
    register_s = {}
    for name in ("restated", "coupled"):
        t0 = time.perf_counter()
        utils[name].composite.composite_id(m)                  # NVRTC compile of every instantiation
        register_s[name] = time.perf_counter() - t0
    acqs = {}
    for name, u in utils.items():
        a = bocf_b200.uEI_noiseless(model, None, utility=u)
        a.W_samples = P.Z
        acqs[name] = a
    draws = {"uniform": np.random.default_rng(7).uniform(size=(args.candidates, d)), "focused": P.Xc}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"config": "cfg3 m=16 d=10 n=1000 matern52 S=1024 H=1 L=1", "candidates": args.candidates,
           "steps": args.steps, "rounds": args.rounds, "register_s": register_s}
    for dname, Xn in draws.items():
        Xd = torch.from_numpy(np.ascontiguousarray(Xn)).to(dev)

        def step(name):
            model.set_hyperparameters(0)
            a, g = acqs[name]._compute_acq_withGradients(Xd)
            return bd.local_topk(a, Xd, 16)

        def timed(name):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            total = 0.0
            for _ in range(args.steps):
                e0.record()
                step(name)
                e1.record()
                flush.zero_()
                torch.cuda.synchronize()
                total += e0.elapsed_time(e1)
            return total / args.steps

        for name in utils:                                     # warm-up: module loads, allocations, f* caches
            step(name)
            step(name)
        ms = {name: [] for name in utils}
        for _ in range(args.rounds):
            for name in utils:
                ms[name].append(timed(name))
        prof = {}
        for name in utils:
            torch.cuda.synchronize()
            _lib.profile_enable(True)
            for _ in range(args.steps):
                step(name)
                flush.zero_()
            rep = _lib.profile_report()
            _lib.profile_enable(False)
            k = "mc_acq_kernel" if name == "builtin" else "mc_acq_user_kernel"
            prof[name] = {k + "_ms_per_step": rep.get(k, (0, 0.0))[1] / args.steps}
        with torch.no_grad():
            a, _ = acqs["builtin"]._compute_acq_withGradients(Xd)
            ei_pos = int((a > 0).sum().item()) if isinstance(a, torch.Tensor) else int(np.sum(a > 0))
        med = {name: float(np.median(v)) for name, v in ms.items()}
        out[dname] = {"step_ms_median": med, "step_ms_all": ms, "mc_kernel": prof,
                      "restated_over_builtin": med["restated"] / med["builtin"],
                      "coupled_over_builtin": med["coupled"] / med["builtin"], "candidates_with_ei_gt_0": ei_pos}
        del Xd
    name, power = gpu_info()
    out["gpu"] = name
    out["power_limit"] = power
    print(json.dumps(out))


if __name__ == "__main__":
    main()
