#!/usr/bin/env python
"""bench.py -- EI-CF acquisition evaluations/sec WITH gradients (BASELINE.json metric) on N B200s.

One step = one pass of the hot path over one batch of synthetic candidates on every rank:
GP posterior (mean, variance, both gradients) of all m outputs -> fused MC composite EI and its
pathwise gradient over all S base samples -> local top-16 (+ NCCL all-gather of the top-k records
when N > 1, the path's only exchange).  Workload: BASELINE.json configs[2] (m=16, d=10, n=1000,
Matern-5/2 ARD, 1024 MC samples, sum-of-squares composite), 1M candidates per GPU per step.

    python bench.py [--gpus N] [--steps K] [--warmup W]          our CUDA path (one JSON line on rank 0)
    python bench.py --impl reference ...                          the reference's CPU algorithm (oracle port)
    python bench.py ... --dump-outputs DIR                        also write the last timed step's results to DIR/*.npy

`value`  : device-resident inputs, CUDA-event timed, max over ranks.
`e2e`    : the same sweep through the public plugin call acquisition_function_withGradients(numpy) with
           pinned HOST candidates in and HOST results out (H2D/D2H inside the timed region).
`roofline`: dominant kernel's algorithmic fp64 flops / its CUDA-event time, against an fp64 DGEMM peak
           measured in this run (MEASURED_PEAKS.json carries no fp64 figure).
`cpu_baseline`: the oracle port (reference loop structure) timed on this box's host cores, N=1 only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # BASELINE.json configs[2]: the configuration the metric is quoted on
    "cfg3": dict(m=16, d=10, n=1000, kind="matern52", composite="sumsq_target", S=1024, H=1, L=1, N=1000000),
    # BASELINE.json configs[4] (large-n stress; 4M candidates over 8 GPUs = 500k per GPU -- pass --candidates to scale)
    "cfg5": dict(m=32, d=10, n=4000, kind="matern52", composite="sumsq_target", S=512, H=1, L=1, N=500000),
    # BASELINE.json configs[1]
    "cfg2": dict(m=4, d=6, n=200, kind="rbf", composite="sumsq_target", S=256, H=1, L=1, N=100000),
    # BASELINE.json configs[3]: parameter-uncertain utility, 64 theta samples, analytic maEI of the linear scalarisation
    "cfg4": dict(m=8, d=8, n=500, kind="matern52", composite="linear", S=256, H=1, L=64, N=262144, variant="maEI"),
}
K_TOP = 16


def f_grad(c):
    """Algorithmic flops per evaluation with gradients, SURVEY.md 8(d) (analytic variants: L (4m + 2md + 30))."""
    m, n, d, S, H, L = c["m"], c["n"], c["d"], c["S"], c["H"], c["L"]
    acq = L * (4 * m + 2 * m * d + 30) if c.get("variant") in ("maEI", "maPI") else L * S * (12 * m + 2)
    return H * (m * (2 * n * n + n * (7 * d + 14)) + acq + 4 * m * d)


# ---- clocks ------------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, period_s=1.0):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.period = period_s
        self.nvml = None
        self._stop = threading.Event()

    def _nvml_loop(self):
        nv, h = self.nvml
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        try:
            smax = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception:
            smax = 0
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                flags = ["Active" if (reasons & b) else "Not Active" for b in
                         (bits["hw_slowdown"], bits["hw_thermal_slowdown"], bits["sw_thermal_slowdown"], bits["sw_power_cap"])]
                self.rows.append([str(self.gpu), str(sm), str(smax), "0", "0"] + flags)
            except Exception:
                pass
            self._stop.wait(self.period)

    def start(self):
        # in-process NVML at a low rate: `nvidia-smi -lms 200` was measured to slow the timed loop by ~15 %
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.gpu)
            self.nvml = (nv, h)
            self.th = threading.Thread(target=self._nvml_loop, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "1000"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self._stop.set()
            self.th.join(timeout=2)
        elif self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        else:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---- reference arm (CPU) -----------------------------------------------------------------------------------
def cpu_literal_rate(P, budget_s, chunk=32):
    """evals/s of the oracle port with the reference's loop structure (uEI_noiseless.py:138-170), gradients on."""
    from tests.helpers import oracle_model, oracle_acq
    om = oracle_model(P)
    done, t0 = 0, time.perf_counter()
    while True:
        lo = done % max(1, P.N - chunk)
        oracle_acq(P, grad=True, vectorised=False, Xc=P.Xc[lo:lo + chunk], model=om)
        done += chunk
        el = time.perf_counter() - t0
        if el > budget_s:
            break
    return done / el, done, el


def cpu_vectorised_rate(P, budget_s, chunk=2048):
    from tests.helpers import oracle_model, oracle_acq
    om = oracle_model(P)
    done, t0 = 0, time.perf_counter()
    while True:
        lo = done % max(1, P.N - chunk)
        oracle_acq(P, grad=True, vectorised=True, Xc=P.Xc[lo:lo + chunk], model=om)
        done += chunk
        el = time.perf_counter() - t0
        if el > budget_s:
            break
    return done / el, done, el


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from tests.helpers import make_problem, oracle_model, oracle_acq
    c = dict(cfg)
    sample = args.ref_sample
    P = make_problem(m=c["m"], d=c["d"], n=c["n"], H=c["H"], kind=c["kind"], composite=c["composite"], N=4096,
                     S=c["S"], L=c["L"], seed=0)
    om = oracle_model(P)
    for w in range(args.warmup):
        oracle_acq(P, grad=True, vectorised=False, Xc=P.Xc[:min(8, sample)], model=om)
    t0 = time.perf_counter()
    for k in range(args.steps):
        lo = (k * sample) % (P.N - sample)
        oracle_acq(P, grad=True, vectorised=False, Xc=P.Xc[lo:lo + sample], model=om)
    el = time.perf_counter() - t0
    val = args.steps * sample / el
    line = {
        "impl": "reference", "metric": "EI-CF acq evals/sec with grads", "value": val, "unit": "evals/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(c, sample),
        "cpu_baseline": {"value": val, "unit": "evals/s", "cores": os.cpu_count(), "kind": "port",
                         "sample": "%d candidates x %d MC samples per step; oracle port with the reference's loop "
                                   "structure (uEI_noiseless.py:138-170: Python loops over theta x Z x candidates, "
                                   "per-output LAPACK/BLAS posterior on all host threads)" % (sample, c["S"])},
        "e2e": {"value": val, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def workload_config(c, n_per_gpu):
    return {"workload": "BASELINE.json configs[%d]: synthetic independent multi-output GP m=%d d=%d n=%d %s-ARD, "
                        "%s composite, EI-CF with gradients, %d MC base samples, H=%d, L=%d"
                        % ({1000: 2, 200: 1, 4000: 4, 500: 3}.get(c["n"], 2), c["m"], c["d"], c["n"], c["kind"], c["composite"],
                           c["S"], c["H"], c["L"]),
            "candidates_per_gpu_per_step": int(n_per_gpu), "mc_samples": c["S"], "top_k": K_TOP,
            "l2": "256 MiB flush between steps; per-step K*/V scratch (GiBs) far exceeds the 126 MB L2"}


DUMP_ROWS = 1 << 18      # 2^18 candidates x (acq + d-gradient + index) x 8 B = 25 MB at d = 10


def dump_outputs(path, acq, grad_acq, topk):
    """Write one step's results as float64 .npy files under `path`: the top-K records (value, global index, x) and, for a
    fixed seeded sample of DUMP_ROWS candidates (all of them when there are fewer), acq, grad acq and the candidates'
    row indices.  Two builds run with the same arguments can then be compared output for output."""
    import torch
    n = acq.shape[0]
    idx = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    rows = torch.from_numpy(idx).to(acq.device)
    arrays = {"acq": acq.reshape(-1)[rows], "grad_acq": grad_acq[rows], "candidate_index": idx, "topk": topk}
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = a.cpu().numpy() if torch.is_tensor(a) else a
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float64))


def bf16_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops_sustained", 1400.0)), True
    except Exception:
        return 1400.0, False


def quick_sweep(cname, N, dev, precision, steps=2, warmup=2, e2e=True, seed=0):
    """A short device-resident (+ end-to-end) sweep of another BASELINE.json configuration or contraction mode on this
    rank's GPU: {value, ms_per_step, e2e, roofline of its dominant contraction}.  Same timing rules as the headline
    (CUDA events, L2 flushed between steps, per-kernel events in a separate pass)."""
    import torch
    import bocf_b200
    from bocf_b200 import _lib
    from tests.helpers import make_problem, product_model, product_utility
    c = dict(CONFIGS[cname])
    variant = c.get("variant", "uEI_noiseless")
    P = make_problem(m=c["m"], d=c["d"], n=c["n"], H=c["H"], kind=c["kind"], composite=c["composite"], N=4096,
                     S=c["S"], L=c["L"], seed=seed, prior_draw=c["n"] <= 2500)
    model = product_model(P, str(dev), precision=precision)
    acq = getattr(bocf_b200, variant)(model, None, utility=product_utility(P))
    if variant == "uEI_noiseless":
        acq.W_samples = P.Z
    else:                                  # the 64 theta samples as an explicit sample set (tests/test_gpu_fullsize.py)
        acq.use_full_support = False
        acq.utility.parameter_dist.sample = lambda k: P.theta
    Xh = torch.from_numpy(np.random.default_rng(7).uniform(size=(N, c["d"]))).pin_memory()
    Xd = Xh.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step_dev():
        model.set_hyperparameters(0)
        a, g = acq._compute_acq_withGradients(Xd)
        return a

    def timed(fn, k, profile=False):
        torch.cuda.synchronize()
        if profile:
            _lib.profile_enable(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(k):
            fn()
            flush.zero_()
        e1.record()
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        prof = _lib.profile_report() if profile else None
        if profile:
            _lib.profile_enable(False)
        return e0.elapsed_time(e1), wall, prof

    for _ in range(warmup):
        step_dev()
        flush.zero_()
    ms, _, _ = timed(step_dev, steps)
    _, _, prof = timed(step_dev, steps, profile=True)
    out = {"config": workload_config(c, N), "precision_mode": precision, "schemes": list(model.active_scheme()),
           "value": steps * N / (ms * 1e-3), "unit": "evals/s", "ms_per_step": ms / steps, "steps": steps, "warmup": warmup}
    gemms = [k for k in ("split_dvar_kernel", "split_var_kernel", "dvar_gemm_kernel", "var_gemm_kernel") if k in prof]
    if gemms:
        dom = max(gemms, key=lambda k: prof[k][1])
        cnt, tot = prof[dom]
        tf = c["m"] * float(c["n"]) ** 2 * (steps * N / cnt) / (tot / cnt * 1e-3) / 1e12
        peak, measured = bf16_peak()
        out["roofline"] = {"bound": "tensor", "kernel": dom, "achieved": tf, "unit": "TFLOP/s",
                           "peak": peak if model.active_slices() else None,
                           "frac": tf / peak if model.active_slices() else None,
                           "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if measured else "fallback 1400",
                           "kernel_ms_per_step": {k: v[1] / steps for k, v in prof.items()}}
    if e2e:
        def step_host():
            model.set_hyperparameters(0)
            return acq.acquisition_function_withGradients(Xh.numpy())
        step_host()
        _, wall, _ = timed(step_host, steps)
        out["e2e"] = {"value": steps * N / (wall * 1e-3), "unit": "evals/s", "h2d_bytes_per_step": int(N * c["d"] * 8),
                      "d2h_bytes_per_step": int(N * 8 + N * c["d"] * 8), "ms_per_step": wall / steps}
    del model, acq, Xd, flush
    torch.cuda.empty_cache()
    return out


# ---- our arm -----------------------------------------------------------------------------------------------
def run_ours(args, cfg):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on STDOUT when NCCL_DEBUG=VERSION/INFO; stdout must carry one JSON line
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "INFO", "TRACE") and not os.environ.get("BOCF_KEEP_NCCL_DEBUG"):
            os.environ["NCCL_DEBUG_FILE"] = os.environ.get("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    import bocf_b200
    from bocf_b200 import _lib, distributed as bd
    from tests.helpers import make_problem, product_model, product_utility
    # the library comes from `python __graft_entry__.py` / build(): the benchmark compiles nothing and writes nothing
    # into the tree, which may be read-only
    _lib.load_library()

    c = dict(cfg)
    N = args.candidates or c["N"]
    P = make_problem(m=c["m"], d=c["d"], n=c["n"], H=c["H"], kind=c["kind"], composite=c["composite"], N=4096,
                     S=c["S"], L=c["L"], seed=0)
    t_setup = time.perf_counter()
    model = product_model(P, str(dev), precision=args.precision)
    torch.cuda.synchronize()
    slices = model.active_slices()
    sch_var, sch_dvar = model.active_scheme()
    t_factor = time.perf_counter() - t_setup          # cold: library load, context, allocations, first launches
    t0 = time.perf_counter()
    model._upload_and_factorize(upload_data=False)      # warm: Gram + blocked Cholesky + L^-1 + alpha of all m outputs
    torch.cuda.synchronize()
    t_factor_warm = time.perf_counter() - t0
    # n^3/3 (Cholesky) + n^3/3 (triangular inverse) + 2 n^2 (alpha) per output, SURVEY.md 8a row a15
    factor_flops = c["H"] * c["m"] * (2.0 * c["n"] ** 3 / 3.0 + 2.0 * c["n"] ** 2)
    acq = bocf_b200.uEI_noiseless(model, None, utility=product_utility(P))
    acq.W_samples = P.Z
    # this rank's shard of the global candidate set (weak scaling: N per rank), seeded per rank
    Xh = torch.from_numpy(np.random.default_rng(7 + 1000 * rank).uniform(size=(N, c["d"]))).pin_memory()
    Xd = Xh.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    dbg = bool(os.environ.get("BOCF_BENCH_DEBUG"))
    last = {}                                           # results of the latest step, for --dump-outputs

    def step_device():
        model.set_hyperparameters(0)
        t0 = time.perf_counter()
        a, g = acq._compute_acq_withGradients(Xd)
        t1 = time.perf_counter()
        rec = bd.local_topk(a, Xd, K_TOP, index_offset=rank * N)
        t2 = time.perf_counter()
        out = bd.allgather_topk(rec, K_TOP) if world > 1 else rec
        if dbg and rank == 0:
            torch.cuda.synchronize()
            t3 = time.perf_counter()
            sys.stderr.write("    host: acq enqueue %.1f ms, topk enqueue %.1f ms, gather %.1f ms, drain %.1f ms\n"
                             % ((t1 - t0) * 1e3, (t2 - t1) * 1e3, 0.0, (t3 - t2) * 1e3))
        last.update(acq=a, grad_acq=g, topk=out)
        return out

    def step_host():
        model.set_hyperparameters(0)
        f, df = acq.acquisition_function_withGradients(Xh.numpy())
        return f, df

    def timed(fn, steps, profile=False):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if profile:
            _lib.profile_enable(True)
        l0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        marks = []
        for _ in range(steps):
            fn()
            flush.zero_()
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            marks.append((ev, time.perf_counter() - t0))
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        step_ms, prev = [], e0
        for ev, cpu_t in marks:
            step_ms.append(prev.elapsed_time(ev))
            if os.environ.get("BOCF_BENCH_DEBUG") and rank == 0:
                sys.stderr.write("  step gpu %.1f ms (cpu enqueue done at %.1f ms)\n" % (step_ms[-1], cpu_t * 1e3))
            prev = ev
        timed.last_step_ms = step_ms
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        launches = _lib.launch_count() - l0
        prof = _lib.profile_report() if profile else None
        if profile:
            _lib.profile_enable(False)
        t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), launches, prof

    for _ in range(args.warmup):
        step_device()
        flush.zero_()
    sampler = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get("BOCF_BENCH_NO_SAMPLER"):
        sampler.start()
    ms_dev, _, launches, _ = timed(step_device, args.steps)
    value_step_ms = list(timed.last_step_ms)
    clocks = sampler.stop() if (rank == 0 and not os.environ.get("BOCF_BENCH_NO_SAMPLER")) else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, **last)
    last.clear()
    # separate pass with per-kernel CUDA events (same steps, same data) for the roofline of the dominant kernel
    ms_prof, _, _, prof = timed(step_device, args.steps, profile=True)
    step_host()                                                     # warm the host path (pinned staging, allocator)
    _, ms_e2e, _, _ = timed(step_host, args.steps)

    # STRONG scaling next to the weak headline: BASELINE.json configs[2] as written -- 1M candidates in total, sharded
    # over the ranks (bocf_b200.distributed.shard_bounds), same exchange step
    strong = None
    if world > 1 and not args.no_strong:
        n_total = c["N"]
        lo, hi = bd.shard_bounds(n_total, world, rank)
        Xs = Xd[: hi - lo]

        def step_strong():
            model.set_hyperparameters(0)
            a, g = acq._compute_acq_withGradients(Xs)
            rec = bd.local_topk(a, Xs, K_TOP, index_offset=lo)
            return bd.allgather_topk(rec, K_TOP)
        for _ in range(2):
            step_strong()
            flush.zero_()
        ms_s, _, _, _ = timed(step_strong, args.steps)
        strong = {"scaling": "strong", "candidates_total_per_step": int(n_total), "candidates_per_gpu_per_step": int(hi - lo),
                  "value": args.steps * n_total / (ms_s * 1e-3), "unit": "evals/s", "ms_per_step": ms_s / args.steps}
    # BASELINE.json configs[4] on >= 4 GPUs: 4M candidates x 512 samples sharded over the ranks, m=32, n=4000 (the model
    # is replicated: 32 factors of 4000^2 per GPU, factorised on every rank -- 79 ms, cheaper than sharding + all-gather)
    cfg5 = None
    if world >= 4 and not args.no_cfg5:
        del Xd
        torch.cuda.empty_cache()
        c5 = dict(CONFIGS["cfg5"])
        n5 = 4000000 // world
        P5 = make_problem(m=c5["m"], d=c5["d"], n=c5["n"], H=1, kind=c5["kind"], composite=c5["composite"], N=4096,
                          S=c5["S"], L=1, seed=0, prior_draw=False)
        t0 = time.perf_counter()
        model5 = product_model(P5, str(dev), precision=args.precision)
        torch.cuda.synchronize()
        t_fac5 = time.perf_counter() - t0
        acq5 = bocf_b200.uEI_noiseless(model5, None, utility=product_utility(P5))
        acq5.W_samples = P5.Z
        X5 = torch.from_numpy(np.random.default_rng(7 + 1000 * rank).uniform(size=(n5, c5["d"]))).to(dev)

        def step5():
            model5.set_hyperparameters(0)
            a, g = acq5._compute_acq_withGradients(X5)
            rec = bd.local_topk(a, X5, K_TOP, index_offset=rank * n5)
            return bd.allgather_topk(rec, K_TOP)
        step5()
        flush.zero_()
        ms5, _, _, _ = timed(step5, 1)
        cfg5 = {"config": workload_config(c5, n5), "candidates_total_per_step": int(n5 * world), "value": n5 * world / (ms5 * 1e-3),
                "unit": "evals/s", "ms_per_step": ms5, "steps": 1, "warmup": 1, "schemes": list(model5.active_scheme()),
                "factorize_cold_s": t_fac5}
        del model5, acq5, X5
        torch.cuda.empty_cache()

    # fp64 peak: cuBLAS DGEMM 8192^3, best of 5, measured here because MEASURED_PEAKS.json has no fp64 entry
    peak_tf = None
    if rank == 0:
        A = torch.randn(8192, 8192, dtype=torch.float64, device=dev)
        B = torch.randn(8192, 8192, dtype=torch.float64, device=dev)
        torch.matmul(A, B)
        best = 1e30
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(A, B)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        peak_tf = 2 * 8192 ** 3 / (best * 1e-3) / 1e12
        del A, B

    # context for the int8 digit-plane path: what a library int8 GEMM reaches on this GPU (torch._int_mm -> cuBLASLt),
    # so the ISSUED int8 rate of the split contraction can be read against a measured, not a nominal, ceiling
    int8_tops = None
    if rank == 0 and slices:
        try:
            A8 = torch.randint(-100, 100, (8192, 8192), dtype=torch.int8, device=dev)
            B8 = torch.randint(-100, 100, (8192, 8192), dtype=torch.int8, device=dev)
            torch._int_mm(A8, B8)
            best = 1e30
            for _ in range(5):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                torch._int_mm(A8, B8)
                e1.record()
                torch.cuda.synchronize()
                best = min(best, e0.elapsed_time(e1))
            int8_tops = 2 * 8192 ** 3 / (best * 1e-3) / 1e12
            del A8, B8
        except Exception:
            int8_tops = None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    evals = args.steps * N * world
    value = evals / (ms_dev * 1e-3)
    e2e_value = evals / (ms_e2e * 1e-3)
    F = f_grad(c)
    # dominant kernel and its algorithmic flops: each of the two triangular contractions does n^2 flop per
    # (candidate, output) -- the 2 n^2 term of F_grad split evenly (DESIGN.md "kernels")
    gemm_names = ["split_dvar_kernel", "split_var_kernel"] if slices else ["dvar_gemm_kernel", "var_gemm_kernel"]
    dom = max(gemm_names, key=lambda k: prof.get(k, (0, 0.0))[1])
    cnt, tot_ms = prof[dom]
    cand_per_launch = args.steps * N / cnt
    flops_per_launch = c["m"] * float(c["n"]) ** 2 * cand_per_launch
    achieved_tf = flops_per_launch / (tot_ms / cnt * 1e-3) / 1e12
    total_kernel_ms = sum(v[1] for v in prof.values())
    if slices:
        # tcgen05 path: the roofline denominator is the measured dense bf16 tensor peak of MEASURED_PEAKS.json
        # (sustained figure: the kernel is timed inside a long step); algorithmic flops are counted ONCE -- the
        # S(S+1)/2 int8 digit-pair passes that buy fp64-level accuracy are overhead, not credit (SURVEY.md 8d).
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        bf16_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        def scheme_pairs(code):                      # digit pairs (= int8 GEMM passes) of scheme 100 SA + 10 SB + LMIN
            sa, sb, lmin = code // 100, (code // 10) % 10, code % 10
            return sum(1 for ta in range(sa) for tb in range(sb) if ta + tb >= lmin)
        dom_scheme = sch_dvar if dom == "split_dvar_kernel" else sch_var
        passes = scheme_pairs(dom_scheme)
        traffic = None
        try:     # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed ncu --set full capture
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))["kernels"][dom]
            if tj.get("scheme") == dom_scheme and c["n"] == 1000 and c["m"] == 16:
                traffic = tj["traffic_GB_per_launch"] * 1e9 * cand_per_launch / tj["candidates_per_launch"]
        except Exception:
            traffic = None
        roofline = {"bound": "tensor", "kernel": dom, "achieved": achieved_tf, "peak": bf16_peak, "unit": "TFLOP/s",
                    "frac": achieved_tf / bf16_peak, "traffic": traffic,
                    "traffic_note": "bytes per launch, scaled from the ncu --set full capture recorded in profiles/r2_traffic.json",
                    "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained (dense bf16 cuBLAS, measured)" if peaks else
                                    "fallback 1.4 PFLOP/s sustained bf16 (B200_PROFILING.md); MEASURED_PEAKS.json absent"),
                    "digit_planes": dom_scheme // 100, "scheme": dom_scheme, "int8_passes": passes,
                    "schemes": {"split_var_kernel": sch_var, "split_dvar_kernel": sch_dvar},
                    "issued_int8_tops": achieved_tf * passes,
                    "issued_frac_of_nominal_int8_4500": achieved_tf * passes / 4500.0,
                    "int8_gemm_tops_measured": int8_tops,
                    "issued_frac_of_measured_int8_gemm": (achieved_tf * passes / int8_tops) if int8_tops else None,
                    "fp64_dgemm_tflops_measured": peak_tf, "achieved_vs_fp64_dgemm": achieved_tf / peak_tf,
                    "launches": cnt, "avg_launch_ms": tot_ms / cnt, "kernel_share_of_step": tot_ms / total_kernel_ms,
                    "step_achieved": F * value / world / 1e12,
                    "kernel_ms": {k: v[1] for k, v in prof.items()}, "profiled_pass_ms_per_step": ms_prof / args.steps}
    else:
        roofline = {"bound": "tensor", "kernel": dom, "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": achieved_tf / peak_tf, "traffic": None,
                    "peak_source": "fp64 cuBLAS DGEMM 8192^3 best-of-5 measured in this run (MEASURED_PEAKS.json has no "
                                   "fp64 entry; fp64 contractions run on DMMA.8x8x4, there is no fp64 tcgen05 kind)",
                    "launches": cnt, "avg_launch_ms": tot_ms / cnt,
                    "kernel_share_of_step": tot_ms / total_kernel_ms,
                    "step_achieved": F * value / world / 1e12, "step_frac": F * value / world / 1e12 / peak_tf,
                    "kernel_ms": {k: v[1] for k, v in prof.items()}, "profiled_pass_ms_per_step": ms_prof / args.steps}

    # SURVEY.md 8(d): algorithmic HBM bytes per evaluation are 8 (2d + 1) (read x, write acq + gradient) -- reported to show
    # that HBM is not the binding roof of this path
    try:
        hbm_gbs = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6500.0))
    except Exception:
        hbm_gbs = 6500.0
    roofline["achieved_hbm_gbs"] = 8.0 * (2 * c["d"] + 1) * value / world / 1e9
    roofline["achieved_hbm_frac"] = roofline["achieved_hbm_gbs"] / hbm_gbs

    # the north star's MIXED-precision bar (1e-4 relative on the EI-CF value and gradient) is already met with four
    # digit planes (tests/test_gpu_split.py: split4); reported next to the headline, which runs the fp64-grade setting
    mixed = None
    if world == 1 and slices > 4 and not args.no_mixed:
        model.set_precision("mixed")
        for _ in range(2):
            step_device()
        ms4, _, _, _ = timed(step_device, args.steps)
        mixed = {"schemes": list(model.active_scheme()), "value": args.steps * N / (ms4 * 1e-3), "unit": "evals/s",
                 "ms_per_step": ms4 / args.steps,
                 "note": "same sweep in the library's mixed mode (variance 4 digit planes / 13 pairs, variance gradient "
                         "3 planes / 8 pairs): meets the north star's mixed-precision bar (<=1e-4 on acq / grad acq, "
                         "tests/test_gpu_split.py::test_auto_and_mixed_pick_their_schemes)"}
        model.set_precision(args.precision)

    # the other BASELINE.json configurations and the fp64 DMMA mode, each as a short sweep on the same GPU
    extras = None
    if world == 1 and not args.no_extras:
        del Xd
        torch.cuda.empty_cache()
        extras = {}
        for key, cname, n_x, prec, kw in (("fp64_dmma_mode", args.config, 262144, "fp64", dict(steps=2, warmup=1)),
                                          ("cfg2", "cfg2", 100000, args.precision, dict(steps=10, warmup=3)),
                                          ("cfg4_maEI_L64", "cfg4", 262144, args.precision, dict(steps=3, warmup=2)),
                                          ("cfg5_500k_share", "cfg5", 500000, args.precision, dict(steps=1, warmup=1, e2e=False))):
            try:
                extras[key] = quick_sweep(cname, n_x, dev, prec, **kw)
            except Exception as exc:                       # an extra must never cost the headline line
                extras[key] = {"error": "%s: %s" % (type(exc).__name__, exc)}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        rate_l, done_l, el_l = cpu_literal_rate(P, args.cpu_budget)
        rate_v, done_v, el_v = cpu_vectorised_rate(P, args.cpu_budget / 2)
        cpu = {"value": rate_l, "unit": "evals/s", "cores": os.cpu_count(), "kind": "port",
               "sample": "%d candidates x %d MC samples in %.1f s; oracle port with the reference's loop structure "
                         "(Python loops over theta x Z x candidates; LAPACK/BLAS posterior on all host threads); the same "
                         "oracle with the MC loops vectorised in numpy reaches %.0f evals/s on the same cores "
                         "(vectorised_numpy_value)" % (done_l, c["S"], el_l, rate_v),
               "vectorised_numpy_value": rate_v,
               "vectorised_sample": "%d candidates in %.1f s, chunks of 2048" % (done_v, el_v)}

    line = {
        "metric": "EI-CF acq evals/sec with grads", "value": value, "unit": "evals/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": ("f64 (kernel, mean, MC, Cholesky) + tcgen05 int8 digit planes x%d with exact int32 accumulation for "
                  "the two factor contractions (fp64-level: <=1e-6 rel. on mean/variance, tests/test_gpu_split.py)"
                  % slices) if slices else "f64",
        "schemes": [sch_var, sch_dvar],
        "data": "synthetic", "precision_mode": args.precision, "digit_planes": slices,
        "config": workload_config(c, N), "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "evals/s", "h2d_bytes_per_step": int(N * c["d"] * 8),
                "d2h_bytes_per_step": int(N * 8 + N * c["d"] * 8), "ms_per_step": ms_e2e / args.steps,
                "api": "uEI_noiseless.acquisition_function_withGradients(numpy (N,d)) -> numpy (N,1),(N,d)"},
        "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "mixed_precision_mode": mixed,
        "cand_x_samples_per_s": value * c["S"], "factorize_s": t_factor, "factorize_warm_s": t_factor_warm,
        "factorize_warm_tflops": factor_flops / t_factor_warm / 1e12, "step_ms": value_step_ms,
        "strong_scaling": strong, "cfg5_sharded": cfg5, "other_configs": extras,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg3", choices=sorted(CONFIGS))
    ap.add_argument("--candidates", type=int, default=0, help="candidates per GPU per step (default: the config's)")
    ap.add_argument("--ref-sample", type=int, default=96, help="candidates per step of the reference arm")
    ap.add_argument("--cpu-budget", type=float, default=16.0, help="seconds of CPU work for cpu_baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-mixed", action="store_true", help="skip the extra mixed-precision measurement")
    ap.add_argument("--no-extras", action="store_true", help="skip the short sweeps of the other configs / fp64 mode (N=1)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling pass (N>1)")
    ap.add_argument("--no-cfg5", action="store_true", help="skip the sharded configs[4] pass (N>=4)")
    ap.add_argument("--precision", default="auto", choices=["auto", "mixed", "fp64", "split3", "split4", "split5", "split6", "split54", "split43", "split53", "split44"],
                    help="arithmetic of the factor contractions (include/bocf_b200.h: enum bocf_precision)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the CUDA path (--impl ours)")
    cfg = CONFIGS[args.config]
    # stdout must carry exactly ONE JSON line: libraries (NCCL's version banner, build logs, ...) that write to
    # fd 1 are diverted to stderr for the whole run; print() below goes to the saved real stdout.
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    try:
        if args.impl == "reference":
            return run_reference(args, cfg)
        return run_ours(args, cfg)
    finally:
        real_stdout.flush()


if __name__ == "__main__":
    sys.exit(main())
