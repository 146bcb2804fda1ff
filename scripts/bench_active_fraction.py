"""Step time of the flagship sweep (cfg 3: m=16, d=10, n=1000, 1M candidates, S=1024, with gradients) against the share
of second-contraction units that carry a non-zero EI-CF gradient weight, for library builds compared in one run.

The fused gradient walks only the units (output, 128-candidate tile) with a non-zero weight.  Three candidate sets:
  uniform   U[0,1]^10, as bench.py draws them: almost no candidate improves on the incumbent
  focused   every candidate next to one of the 8 best training points (make_problem focus=1, scale 0.05): nearly every
            unit is active, so this is the set that shows the cost of the extra kernel and the listed walk
  mix       the first half uniform, the second half focused
Each build runs in its own process (BOCF_LIB_PATH); builds alternate for --rounds rounds.  Steps are timed with CUDA
events and a 256 MiB L2 flush between steps.  `active_tiles` is the share of 128-candidate tiles with a non-zero EI,
read from the outputs after the timed steps: for sumsq_target every output of an improving candidate has a non-zero
weight, so it is the share of units the second contraction walks.  `kernel_ms` are the library's per-kernel CUDA-event
times per step, from a separate profiled pass.  `pruned` is the share of the candidates the library proved inactive
from the posterior mean and left out of the sweep (bocf_model_sweep_stats; null for a build without it).  A library at
<tree>/bocf_b200/csrc/ runs with the Python package of <tree>, so builds with different bindings can be compared.

    python scripts/bench_active_fraction.py --libs parent.so branch.so [--rounds 2] [--steps 3] [--warmup 2]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CFG = dict(m=16, d=10, n=1000, kind="matern52", composite="sumsq_target", S=1024, H=1, L=1)
N = 1000000


def candidate_sets():
    from tests.helpers import make_problem
    uniform = np.random.default_rng(7).uniform(size=(N, CFG["d"]))
    focused = make_problem(N=N, seed=0, focus=1.0, focus_scale=0.05, **CFG).Xc
    mix = np.concatenate([uniform[:N // 2], focused[N // 2:]])
    return {"uniform": uniform, "focused": focused, "mix": mix}


def pruned_share(model):
    """1 - swept / candidates of the model's latest acquisition call, as the library counted them."""
    fn = getattr(model._lib, "bocf_model_sweep_stats", None)
    if fn is None:
        return None
    n, kept = ctypes.c_int64(0), ctypes.c_int64(0)
    fn(model._handle, ctypes.byref(n), ctypes.byref(kept))
    return 1.0 - kept.value / n.value


def child(args):
    tree = os.path.dirname(os.path.dirname(os.path.dirname(os.environ.get("BOCF_LIB_PATH", ""))))
    if os.path.exists(os.path.join(tree, "bocf_b200", "__init__.py")):
        sys.path.insert(0, tree)
    import torch
    import bocf_b200
    from bocf_b200 import _lib
    from tests.helpers import make_problem, product_model, product_utility
    _lib.load_library()
    dev = torch.device("cuda", 0)
    P = make_problem(N=4096, seed=0, **CFG)
    model = product_model(P, str(dev))
    acq = bocf_b200.uEI_noiseless(model, None, utility=product_utility(P))
    acq.W_samples = P.Z
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"lib": os.environ.get("BOCF_LIB_PATH", ""), "gpu": torch.cuda.get_device_name(0)}
    for name, X in candidate_sets().items():
        Xd = torch.from_numpy(X).to(dev)
        model.set_hyperparameters(0)
        for _ in range(args.warmup):
            a, g = acq._compute_acq_withGradients(Xd)
            flush.zero_()
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a, g = acq._compute_acq_withGradients(Xd)
            e1.record()
            flush.zero_()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        pruned = pruned_share(model)
        _lib.profile_enable(True)
        for _ in range(args.steps):
            acq._compute_acq_withGradients(Xd)
            flush.zero_()
        prof = _lib.profile_report()
        _lib.profile_enable(False)
        act = (a.reshape(-1) > 0).cpu().numpy()
        tiles = np.zeros(-(-N // 128), dtype=bool)
        np.logical_or.at(tiles, np.arange(N) // 128, act)
        out[name] = {"ms_per_step": float(np.median(ms)), "ms": ms, "active_candidates": float(act.mean()),
                     "active_tiles": float(tiles.mean()), "pruned": pruned,
                     "kernel_ms": {k: v[1] / args.steps for k, v in sorted(prof.items())}}
        del Xd, a, g
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--libs", nargs="+", default=[os.path.join(ROOT, "bocf_b200", "csrc", "libbocf_b200.so")])
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        return child(args)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True).stdout.strip()
    except OSError:
        q = "unknown"
    print(json.dumps({"gpu0": q}))
    for r in range(args.rounds):
        for lib in args.libs:
            env = dict(os.environ, BOCF_LIB_PATH=os.path.abspath(lib))
            res = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--steps", str(args.steps),
                                  "--warmup", str(args.warmup)], env=env, capture_output=True, text=True)
            if res.returncode != 0:
                sys.stderr.write(res.stderr)
                raise SystemExit("run with %s failed" % lib)
            rec = json.loads(res.stdout.strip().splitlines()[-1])
            rec["round"] = r
            print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
