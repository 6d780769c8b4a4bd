"""bench.py -- collocation-points/sec for one residual+gradient evaluation (BASELINE.json metric) on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2] [--points P] [--impl ours|reference]
                  [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic collocation points: K0 pack -> K1 (forward jets +
residual + seeds) -> loss finalize -> K2 (reverse pass) -> K2b (reduce); with N > 1 GPUs every rank owns its own
shard of points (weak scaling: per-GPU points fixed) and the flat [grad | sum r^2] buffer is all-reduced once per
step over NCCL.  Workload = BASELINE.json configs[1]: Solver2D Laplace, DirichletBVP2D, FCNN(2-64-64-64-1, tanh),
16384 points per GPU, synthetic uniform points, PyTorch-default random init.

Timing: CUDA events on the launching stream around every step, L2 flushed (256 MiB memset) before every timed step,
max over ranks.  `value` = points/s with inputs resident in HBM; `e2e` = same metric through FusedProblem's public
call with pinned HOST coordinates copied in and the loss copied out inside the timed region.

`--impl reference` times the CPU oracle port of the reference's closure (oracle/reference_port.py, torch autograd,
float64 = the reference's default dtype) on this box's host cores for the same workload.

Besides the contract's keys the line carries, at N = 1: `cpu_baseline` (the same oracle closure on a bounded sample),
`gpu_autograd_baseline` (the reference algorithm through stock PyTorch CUDA autograd on this GPU -- what a user of the
reference gets on a B200 today) and `fit` (the product's Solver.fit end to end: host sampling, H2D, K0..K2b, Adam,
one loss read per epoch).  All three run AFTER the timed region.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import workloads  # noqa: E402

METRIC = "collocation-points/sec (residual+grad)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--points", type=int, default=0, help="points per GPU (default: the workload's BASELINE size)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--fit-epochs", type=int, default=200, help="epochs of the Solver.fit leg (0 = skip)")
    ap.add_argument("--no-gpu-comparator", action="store_true", help="skip the torch-CUDA-autograd comparator leg")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-strong", action="store_true", help="skip the C3 / C5 strong-scaling legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (grad.npy, sumsq.npy) under DIR")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference closure (only place outside tests/ that executes oracle/)
# ----------------------------------------------------------------------------------------------------------------------
def _oracle_step_fn(key, n_points, dtype, device="cpu"):
    """One reference closure (solvers.py:369-395) through the oracle port: host coordinates in, loss (host float) out."""
    from oracle import reference_port as oracle
    wl = workloads.build(oracle.NAMESPACE, key)
    torch.manual_seed(0)
    nets, conds = wl.make_nets(), wl.make_conditions()
    for m in oracle.distinct_modules(nets):
        m.to(device=device, dtype=dtype)
    coords_np = workloads.sample_coords(wl, n_points, seed=0)
    eqs = workloads.bundle_eq_wrapper(wl)

    def step():
        for m in oracle.distinct_modules(nets):
            for p in m.parameters():
                p.grad = None
        coords = [torch.as_tensor(c, dtype=dtype).to(device).reshape(-1, 1).requires_grad_(True) for c in coords_np]
        _, _, loss = oracle.closure(nets, conds, eqs, coords, backward=True)
        return float(loss.detach())
    return step


def gpu_autograd_comparator(key, n_points, dev, seconds=2.0):
    """Secondary comparator (SURVEY.md §8d): the SAME reference algorithm on the SAME GPU through stock PyTorch CUDA
    autograd (what a user of the reference gets on a B200 today).  Baseline only, measured after the timed region."""
    out = {}
    for name, dtype in (("f32", torch.float32), ("f64", torch.float64)):
        step = _oracle_step_fn(key, n_points, dtype, device=dev)
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        times, t_end = [], time.perf_counter() + seconds
        while time.perf_counter() < t_end or len(times) < 3:
            t0 = time.perf_counter()
            step()                      # ends with a host read of the loss, like the reference closure (:394)
            times.append(time.perf_counter() - t0)
        med = float(np.median(times))
        out[name] = {"value": n_points / med, "unit": "points/s", "ms_per_step": med * 1e3, "steps": len(times)}
    out["what"] = (f"oracle/reference_port.py closure on cuda via torch {torch.__version__} autograd (eager), "
                   f"{n_points} points, wall clock incl. the per-step loss read")
    return out


def cpu_reference_throughput(key, n_points, seconds, dtype=torch.float64, max_steps=None, warmup=1):
    step = _oracle_step_fn(key, n_points, dtype)

    # "all the host threads it can use": torch's intra-op pool degrades badly when oversubscribed on these small
    # matrices (128 threads: 18 s/closure on the GPU box vs 0.12 s with 8), so the reference arm gets the thread count
    # that is fastest for it, found by a short sweep, and that count is what `cores` reports.
    ncpu = os.cpu_count() or 1
    best_t, best_dt = 1, float("inf")
    for nt in sorted({t for t in (4, 8, 16, 32, 64, ncpu) if t <= ncpu}):
        torch.set_num_threads(nt)
        step()
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if dt < best_dt:
            best_t, best_dt = nt, dt
        if dt > 4 * best_dt:
            break
    torch.set_num_threads(best_t)
    for _ in range(warmup):
        step()
    times = []
    t_end = time.perf_counter() + seconds
    while True:
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if (max_steps and len(times) >= max_steps) or (not max_steps and time.perf_counter() > t_end):
            break
    med = float(np.median(times))
    return dict(value=n_points / med, unit="points/s", cores=torch.get_num_threads(), kind="port",
                sample=f"{len(times)} closures of {n_points} points, {str(dtype).replace('torch.', '')}, median "
                       f"{med * 1e3:.1f} ms, oracle/reference_port.py (torch {torch.__version__} autograd, CPU)",
                ms_per_step=med * 1e3, steps=len(times))


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = workloads.build(workloads.product_namespace(), args.workload)
    n = args.points or wl.default_n
    # The reference computes in torch's default dtype, float32 (it never calls set_default_dtype): that is the headline of
    # this arm.  float64 -- the precision of the parity oracle -- is timed beside it (BASELINE.md §3 asks for both).
    res = cpu_reference_throughput(args.workload, n, seconds=1e9, max_steps=max(args.steps, 1),
                                   warmup=max(args.warmup, 1), dtype=torch.float32)
    res64 = cpu_reference_throughput(args.workload, n, seconds=1e9, max_steps=max(min(args.steps, 5), 1), warmup=1,
                                     dtype=torch.float64)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": "points/s", "n_gpus": args.gpus,
        "steps": res["steps"], "warmup": max(args.warmup, 1), "ms_per_step": res["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{wl.name} {wl.solver} N={n} (reference closure solvers.py:369-395, CPU port)",
                   "points_per_step": n},
        "cpu_baseline": {**{k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
                         "f64": {k: res64[k] for k in ("value", "unit", "cores", "sample")}},
        "e2e": {"value": res["value"], "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------------
# clocks during the timed region
# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index):
        self.samples, self.reasons, self.power = [], set(), []
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                    nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            time.sleep(0.02)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(r for r in self.reasons if r != "gpu_idle"),
                "power_w_max": max(self.power) if self.power else None, "samples": len(self.samples)}


def _survey_generator(key, n, G):
    """Training generators of SURVEY.md §8d for the five workloads (host sampling, fresh points every epoch)."""
    if key == "c1":
        return G.Generator1D(n, 0.1, 12.0, "equally-spaced-noisy")
    if key in ("c2", "c3"):
        side = int(round(n ** 0.5))
        lo, hi = ((0.0, 0.0), (1.0, 1.0)) if key == "c2" else ((-1.0, 0.0), (1.0, 1.0))
        return G.Generator2D((side, side), lo, hi, "equally-spaced-noisy")
    if key == "c4":
        return G.GeneratorSpherical(n, 0.1, 3.0)
    if key == "c5":
        rng = ((0.0, 2 * np.pi), (0.05, 0.5), (0.5, 2.0), (-1.0, 1.0), (-1.0, 1.0))
        gens = [G.Generator1D(n, lo, hi, "uniform") for lo, hi in rng]
        g = gens[0]
        for h in gens[1:]:
            g = g * h
        return g
    raise KeyError(key)


def fit_throughput(key, n, epochs, warm=20, device_loop=False):
    """End-to-end ``Solver.fit`` of the product (SURVEY.md §8d "fit() epochs/s"), no validation batches.  Default loop: host
    sampling of a fresh batch, staging + H2D, K0..K2b (one graph replay), torch Adam, one loss read per epoch.
    ``device_loop=True`` (opt-in of the solvers): Philox sampling on the device, K0..K2b, best-parameter bookkeeping and
    Adam (optim.FlatAdam) replayed as ONE CUDA graph per epoch; the loss history is read back once at the end."""
    from neurodiffeq_b200 import solvers as S, generators as G
    nd = workloads.product_namespace()
    wl = workloads.build(nd, key)
    torch.manual_seed(0)
    nets, conds = wl.make_nets(), wl.make_conditions()
    gen = _survey_generator(key, n, G)
    kw = dict(nets=nets, train_generator=gen, valid_generator=gen, n_batches_valid=0)
    if device_loop:
        kw["device_loop"] = True
    kw["jit"] = os.environ.get("PINNJET_JIT", "1") != "0"
    if wl.solver == "BundleSolver1D":
        kw["eq_param_index"] = wl.eq_param_index
    solver = getattr(S, wl.solver)(wl.diff_eqs, conds, **kw)
    solver.fit(warm, tqdm_file=None)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    solver.fit(epochs, tqdm_file=None)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    hist = solver.metrics_history["train_loss"]
    return {"epochs_per_s": epochs / dt, "points_per_s": epochs * gen.size / dt, "ms_per_epoch": dt / epochs * 1e3,
            "epochs": epochs, "points_per_epoch": int(gen.size), "loss_first": hist[0], "loss_last": hist[-1],
            "what": (f"{wl.solver}.fit(device_loop=True): one CUDA-graph replay per epoch = Philox sampling "
                     f"({type(gen).__name__} law) + K0..K2b + best-parameter bookkeeping + FlatAdam; losses read once at "
                     f"the end; n_batches_valid=0, wall clock" if device_loop else
                     f"{wl.solver}.fit: host sampling ({type(gen).__name__}) + H2D + K0..K2b + torch Adam + 1 loss read "
                     f"per epoch, n_batches_valid=0, wall clock")}


def strong_scaling_leg(key, n_global, world, rank, dev, steps, warmup, flush_l2, align=None):
    """BASELINE configs 3 and 5 (C3 Burgers 65536 points, C5 bundle 131072 points): the GLOBAL batch is fixed and sharded
    over the ranks; step = pack + K1 + finalize + K2 + K2b + the collective, replayed as a CUDA graph, L2 flushed before each
    timed step, max over ranks.  Reported as an extra key of the bench line (the headline stays C2 weak scaling)."""
    import torch.distributed as dist
    from neurodiffeq_b200.parallel import GradBufReducer, shard_bounds
    wl, nets, conds, fp = workloads.build_fused(key, seed=0, device=dev)
    lo, hi = shard_bounds(n_global, rank, world)
    coords_np = workloads.sample_coords(wl, n_global, seed=2000)
    coords = [torch.from_numpy(c[lo:hi].copy()).to(dev) for c in coords_np]
    if os.environ.get("PINNJET_JIT", "1") != "0":
        fp.enable_jit()
    fp.gradbuf.zero_()
    fp.residual_grad(coords, n_global=n_global, sumsq_out=fp.sumsq)
    reducer = GradBufReducer(fp.gradbuf, dist) if world > 1 else None

    def body():
        fp.residual_grad(coords, n_global=n_global, sumsq_out=fp.sumsq, reducer=reducer, zero_gradbuf=True)

    for _ in range(max(warmup, 3)):
        body()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        body()
    torch.cuda.current_stream().wait_stream(side)
    if world > 1:
        dist.barrier()
    with torch.cuda.graph(graph):
        body()
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    total = 0.0
    for _ in range(steps):
        flush_l2()
        if align is not None:
            align()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        graph.replay()
        b.record()
        torch.cuda.synchronize()
        total += a.elapsed_time(b)
    if world > 1:
        t = torch.tensor([total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total = float(t.item())
    ms = total / steps
    info = fp.plan_info(hi - lo)
    out = {"workload": wl.name, "global_points": n_global, "points_per_gpu": hi - lo, "ms_per_step": ms,
           "points_per_s": n_global / (ms * 1e-3), "steps": steps, "loss": float(fp.sumsq.item()) / (n_global * fp.n_eq),
           "kernels": ("tensor-core" if info.get("tc") else "ffma") + " / " + ("tensor-core" if info.get("tc_bwd") else "ffma"),
           "collective": (reducer.mode + (" (fused with K2b)" if reducer.fused_args is not None else ""))
           if reducer is not None else "single"}
    del graph, fp
    torch.cuda.empty_cache()
    return out


def executed_flops(wl, tp):
    """F = sum over nets of 2*d0*h1 + C*2*(sum h_{l-1} h_l + h_L*d_out) with the channel count the kernels really carry."""
    c_exec, total = tp.n_channels, 0
    for widths, _ in wl.nets_spec:
        d0, h = widths[0], widths[1:]
        total += 2 * d0 * h[0] + c_exec * 2 * sum(a * b for a, b in zip(h[:-1], h[1:]))
    return total


def dump_outputs(out_dir, fp):
    """What a caller of the timed step receives, as float32 .npy files: ``grad`` = d mean(r^2) / d theta (flat, in the
    order of the networks' parameters) and ``sumsq`` = sum r^2 over the global batch.  Inputs are seeded (parameters:
    seed 0, points: seed 1000 + rank), so two builds given the same arguments can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "grad.npy"), fp.grad.detach().cpu().numpy())
    np.save(os.path.join(out_dir, "sumsq.npy"), fp.sumsq.detach().cpu().numpy())


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d.get("bf16_tflops", 1590.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 1590.0, 6650.0, "fallback (B200_PROFILING.md)"


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference_arm(args)

    import ctypes
    build_fused = workloads.build_fused
    from neurodiffeq_b200 import engine as E

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    wl, nets, conds, fp = build_fused(args.workload, seed=0, device=dev)
    n = args.points or wl.default_n                       # points per GPU (weak scaling)
    n_global = n * world
    coords_np = workloads.sample_coords(wl, n, seed=1000 + rank)
    coords = [torch.from_numpy(c).to(dev) for c in coords_np]
    host_coords = [torch.from_numpy(c).pin_memory() for c in coords_np]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flush_rd = torch.zeros(64 << 20, dtype=torch.float32, device=dev)   # 256 MiB, only read

    def flush_l2():
        """Write a 256 MiB buffer (evicts everything), then stream another 256 MiB through L2 by READING it so that the
        cache is left full of CLEAN lines: a memset alone leaves 126 MB of dirty lines whose write-back would be charged
        to the first kernel of the timed step."""
        flush.zero_()
        if os.environ.get("PINNJET_BENCH_DIRTY_FLUSH") != "1":
            flush_rd.sum()
    stream = torch.cuda.current_stream()

    jit_on = fp.enable_jit() if os.environ.get("PINNJET_JIT", "1") != "0" else False   # specialised forward kernel (jit.py)
    reducer, align = None, None

    def step_body():
        # K0 re-packs theta and clears [grad | sum r^2] (optimizer.zero_grad() + loss accumulator) in one launch; the loss
        # finalisation happens inside K1 (last-warp ticket).  N > 1: SUM of [grad | sum r^2] over the ranks (parallel.GradBufReducer) -- K2b and the one-shot NVLink collective
        # as ONE kernel (pj_backward_allreduce) when peer memory is available, K2b + the process group's all-reduce otherwise
        fp.residual_grad(coords, n_global=n_global, sumsq_out=fp.sumsq, reducer=reducer, zero_gradbuf=True)

    if world > 1:
        from neurodiffeq_b200.parallel import GradBufReducer
        fp.gradbuf.zero_()
        fp.residual_grad(coords, n_global=n_global, sumsq_out=fp.sumsq)   # allocates the buffers
        reducer = GradBufReducer(fp.gradbuf, dist)
        # the ranks flush their L2 independently before every timed step; a device-side barrier (the one-shot kernel on a dummy
        # buffer) after the flush lines the start events up, so that the flush's jitter is not charged to the step
        align_buf = torch.zeros(8, dtype=torch.float32, device=dev)
        aligner = GradBufReducer(align_buf, dist)
        if aligner.mode == "oneshot-nvlink" and os.environ.get("PINNJET_BENCH_ALIGN", "1") != "0":
            align = lambda: aligner(align_buf)            # noqa: E731
    fused_collective = reducer is not None and reducer.fused_args is not None

    # warm-up (also sizes buffers, sets kernel attributes)
    for _ in range(max(args.warmup, 3)):
        step_body()
    torch.cuda.synchronize()

    graph = None
    if not args.no_graph:   # the whole step (fill, K0..K2b and, for N > 1, the NCCL all-reduce) as one CUDA graph
        try:
            graph = torch.cuda.CUDAGraph()
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                step_body()
            torch.cuda.current_stream().wait_stream(s)
            with torch.cuda.graph(graph):
                step_body()
            for _ in range(3):
                graph.replay()
            torch.cuda.synchronize()
        except Exception as exc:   # noqa: BLE001  (e.g. a NCCL build that cannot be captured): time eager launches
            print(f"[bench] CUDA graph capture failed ({type(exc).__name__}: {exc}); timing eager launches",
                  file=sys.stderr)
            graph = None
            torch.cuda.synchronize()

    def run_step():
        if graph is not None:
            graph.replay()
        else:
            step_body()

    # pack (+ clear), K1 (+ loss finalisation), K2, K2b (or K2b + collective as one kernel); no torch launch inside the step
    ours_per_step = 4 + (1 if (reducer is not None and reducer.mode == "oneshot-nvlink" and not fused_collective) else 0)

    # ---- timed region: K steps, L2 flushed before each, CUDA events per step, max over ranks -------------------------
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    with ClockSampler(local_rank) as clk:
        t_wall0 = time.perf_counter()
        for a, b in ev:
            flush_l2()
            if align is not None:
                align()
            a.record()
            run_step()
            b.record()
        torch.cuda.synchronize()
        t_wall = time.perf_counter() - t_wall0
    step_ms = np.array([a.elapsed_time(b) for a, b in ev])
    total_ms = float(step_ms.sum())
    if world > 1:
        t = torch.tensor([total_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
        dist.barrier()
    ms_per_step = total_ms / args.steps
    value = n_global / (ms_per_step * 1e-3)
    loss = float(fp.sumsq.item()) / (n_global * fp.n_eq)
    if args.dump_outputs and rank == 0:   # before the per-kernel timing below overwrites the gradient
        dump_outputs(args.dump_outputs, fp)

    # ---- per-kernel timing for the roofline (events around each launch, same stream) ---------------------------------
    info = fp.plan_info(n)
    ptrs, keep = fp._coord_ptrs(coords, n)
    sp = ctypes.byref(fp.spec)
    cs = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731
    scale = ctypes.c_float(2.0 / (n_global * fp.n_eq))

    def k1_only():   # the forward kernel the step launches: the problem's specialised kernel when it is in use
        if jit_on and fp._jit_usable(n):
            E._check(fp.lib.pj_forward_train_jit(fp._jit.function, sp, fp.prog_train.data_ptr(), len(fp.tp.prog_train),
                                                 *fp._prog_w_args(), ptrs, n, fp.pack_buf.data_ptr(), scale, None, None,
                                                 fp.workspace.data_ptr(), fp.workspace.numel(), cs()), "k1 (specialised)")
        else:
            E._check(fp.lib.pj_forward_train(sp, fp.prog_train.data_ptr(), len(fp.tp.prog_train), *fp._prog_w_args(), ptrs, n,
                                             fp.pack_buf.data_ptr(), scale, None, None, None, fp.workspace.data_ptr(),
                                             fp.workspace.numel(), cs()), "k1")

    def k2_only():
        E._check(fp.lib.pj_backward(sp, ptrs, n, fp.pack_buf.data_ptr(), fp.grad.data_ptr(), fp.workspace.data_ptr(),
                                    fp.workspace.numel(), cs()), "k2")

    def time_kernel(fn, reps):
        ts = []
        for _ in range(reps):
            flush_l2()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.mean(ts)), float(np.min(ts))

    reps = min(max(args.steps, 10), 100)
    k1_ms, k1_min = time_kernel(k1_only, reps)
    k2_ms, k2_min = time_kernel(k2_only, reps)   # K2 + K2b (z-jets come from the preceding K1, L2 flushed in between)

    # ---- the collective alone (N > 1): our one-shot NVLink kernel and, beside it, the process group's NCCL all-reduce ---
    collective = None
    if world > 1:
        def time_collective(fn, reps=50):
            for _ in range(5):
                fn()
            torch.cuda.synchronize()
            dist.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            torch.cuda.synchronize()
            t = torch.tensor([a.elapsed_time(b) / reps], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        scratch = fp.gradbuf.clone()
        collective = {"mode": reducer.mode, "fallback_reason": reducer.why, "bytes": int(scratch.numel() * 4),
                      "ms_back_to_back": time_collective(lambda: reducer(fp.gradbuf)),
                      "nccl_all_reduce_ms_back_to_back": time_collective(lambda: dist.all_reduce(scratch)),
                      "fused_with_k2b": fused_collective,
                      "kernel": ("pj::reduce_allreduce_kernel (csrc/pinnjet_comm.cu, pj_backward_allreduce): the reverse kernel's "
                                 "per-CTA partials folded, published in the symmetric buffer and summed over the ranks in ONE "
                                 "launch; " if fused_collective else "") +
                                ("pj::allreduce_oneshot_kernel (stand-alone form, timed here back to back): peer loads over "
                                 "NVLink, flags with st.release.sys / ld.acquire.sys, sum in rank order"
                                 if reducer.mode == "oneshot-nvlink" else "torch.distributed.all_reduce"),
                      "rank_alignment": "device-side barrier after each L2 flush, before the start event" if align is not None
                                        else "none"}

    # ---- e2e: host coordinates in, loss out, through the public call -------------------------------------------------
    e2e_fold_zero = True

    def e2e_step():
        # the public call: host coordinates in (staged through pinned buffers, H2D inside), CUDA-graph replay of
        # K0..K2b (K0 also clears [grad | sum r^2]), loss read back to the host
        if e2e_fold_zero:
            fp.residual_grad_graphed(host_coords, n_global=n_global, zero_gradbuf=True)
        else:
            fp.gradbuf.zero_()
            fp.residual_grad_graphed(host_coords, n_global=n_global)
        if world > 1:
            reducer(fp.gradbuf)
        return fp.sumsq.item()   # device -> host read of the step's result

    try:   # the folded clear must give the loss the separate fill gives; otherwise (or on any error) keep the fill launch
        a_loss = e2e_step()
        e2e_fold_zero = False
        b_loss = e2e_step()
        e2e_fold_zero = abs(a_loss - b_loss) <= 1e-6 * abs(b_loss)
    except Exception as exc:  # noqa: BLE001
        print(f"[bench] e2e with the folded clear failed ({type(exc).__name__}: {exc}); using the separate fill", file=sys.stderr)
        e2e_fold_zero = False
    for _ in range(3):
        e2e_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e2e_steps = min(args.steps, 100)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(e2e_steps):
        e2e_step()
    b.record()
    torch.cuda.synchronize()
    e2e_ms = a.elapsed_time(b) / e2e_steps
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = n_global / (e2e_ms * 1e-3)
    h2d = int(sum(h.numel() * 4 for h in host_coords))

    # ---- roofline of the forward+jet kernel (K1), algorithmic FLOPs / measured launch time ----------------------------
    bf16_peak, hbm_peak, peak_src = load_peaks()
    clocks = clk.summary()
    flops_k1 = wl.flops_fwdjet * n
    ach_k1 = flops_k1 / (k1_ms * 1e-3) / 1e12
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    n_sms = torch.cuda.get_device_properties(dev).multi_processor_count
    fp32_peak = n_sms * 128 * 2 * sm_mhz * 1e6 / 1e12       # FFMA lanes x 2 flop x clock under load
    tc_fwd, tc_bwd = bool(info.get("tc")), bool(info.get("tc_bwd"))
    k1_name = "k1tc3_forward_kernel" if tc_fwd else "k1_forward_kernel"
    k2_name = "k2tc2_backward_kernel" if tc_bwd else "k2_backward_kernel"
    # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel, from the committed `ncu --set full`
    # capture of the same kernel variant (profiles/r02/traffic.json names the report it was read from); null if none.
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(args.workload, {}).get("pj_k1_jit" if (jit_on and tc_fwd) else k1_name, {}).get("dram_bytes")
    roofline = {
        "kernel": k1_name + (" specialised (pj_k1_jit: residual programs compiled in)" if jit_on else "") +
                  " (forward + jets + residual program)",
        "bound": "tensor", "achieved": ach_k1,
        "peak": bf16_peak, "unit": "TFLOP/s", "frac": ach_k1 / bf16_peak, "traffic": traffic,
        "peak_source": f"dense bf16 tensor, {peak_src}",
        "pipe": ("tcgen05.mma kind::f16, bf16x3 split operands (6 bf16 products per fp32 product, fp32 TMEM accumulators): "
                 "hidden-layer and output contractions on the tensor pipe; layer 0, activation jets and the residual program "
                 "on the CUDA cores" if tc_fwd else
                 "fp32 FFMA2 on CUDA cores (network not eligible for the tensor-core kernels: hidden width != 64, "
                 "or PINNJET_TC=0)"),
        "tensor_products_per_fp32_product": 6 if tc_fwd else 0,
        "fp32_ffma_peak": fp32_peak, "frac_of_fp32_ffma_peak": ach_k1 / fp32_peak,
        "algorithmic_flops_per_point": wl.flops_fwdjet, "launch_ms": k1_ms, "launch_ms_min": k1_min,
        # `achieved` counts the CANONICAL jet FLOPs (SURVEY.md §8d: one channel per needed partial derivative).  When the
        # tracer proves the residual affine in the pure second derivatives, the kernels carry ONE weighted second-order
        # channel instead (forward-Laplacian): fewer channels are executed for the same result.
        "channels_canonical": 1 + fp.tp.scheme.n1 + fp.tp.scheme.n2, "channels_executed": fp.tp.n_channels,
        "executed_flops_per_point": executed_flops(wl, fp.tp),
        "k2": {"kernel": k2_name + " + k2_reduce_kernel", "algorithmic_flops_per_point": 2 * wl.flops_fwdjet,
               "launch_ms": k2_ms, "achieved": 2 * flops_k1 / (k2_ms * 1e-3) / 1e12,
               "frac_of_fp32_ffma_peak": 2 * flops_k1 / (k2_ms * 1e-3) / 1e12 / fp32_peak},
    }

    cpu_base, fit, gpu_cmp = None, None, None
    if rank == 0 and world == 1:
        if args.fit_epochs > 0:
            try:
                fit = fit_throughput(args.workload, n, args.fit_epochs)
            except Exception as e:  # the fit leg is a secondary report: never lose the bench line over it
                fit = {"error": f"{type(e).__name__}: {e}"}
            try:
                fit["device_loop"] = fit_throughput(args.workload, n, 5 * args.fit_epochs, device_loop=True)
            except Exception as e:
                fit["device_loop"] = {"error": f"{type(e).__name__}: {e}"}
        if not args.no_gpu_comparator:
            try:
                gpu_cmp = gpu_autograd_comparator(args.workload, n, dev)
            except Exception as e:
                gpu_cmp = {"error": f"{type(e).__name__}: {e}"}
        cpu32 = cpu_reference_throughput(args.workload, n, seconds=args.cpu_seconds / 2, dtype=torch.float32)
        cpu64 = cpu_reference_throughput(args.workload, n, seconds=args.cpu_seconds / 2, dtype=torch.float64)
        cpu_base = {**{k: cpu32[k] for k in ("value", "unit", "cores", "kind", "sample")},   # float32 = the reference's dtype
                    "f64": {k: cpu64[k] for k in ("value", "unit", "cores", "sample")}}

    # ---- strong scaling of the two BASELINE configs that name it (C3: 65536 points, C5: 131072 points over the N GPUs) -----
    strong = None
    if args.workload == "c2" and not args.points and not args.no_strong:
        strong = {}
        for key, n_g in (("c3", 65536), ("c5", 131072)):
            try:
                strong[key] = strong_scaling_leg(key, n_g, world, rank, dev, steps=min(args.steps, 30), warmup=3, flush_l2=flush_l2,
                                                 align=align)
            except Exception as e:  # noqa: BLE001  (secondary report)
                strong[key] = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{wl.name}: {wl.solver}, nets {wl.nets_spec}, {n} points/GPU, "
                                   f"residual+grad step = K0 (pack + clear grad) + K1 (+ loss finalisation) + K2 + K2b"
                                   + (f" + all-reduce of [grad|loss] ({reducer.mode}"
                                      f"{', fused with K2b' if fused_collective else ''})" if world > 1 else ""),
                       "points_per_gpu": n, "global_points": n_global, "tile_points": info["T"],
                       "grid": info["grid"], "l2": "flushed before every timed step (256 MiB memset, then 256 MiB streamed read so the lines left are clean)",
                       "cuda_graph": graph is not None, "parallelism": f"dp{world} (points sharded)"},
            "e2e": {"value": e2e_value, "unit": "points/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 4},
            "gpu_launches": ours_per_step * args.steps,
            "roofline": roofline, "cpu_baseline": cpu_base, "clocks": clocks, "collective": collective,
            "strong_scaling": strong,
            "specialised_forward_kernel": {"in_use": bool(jit_on), "why_not": "" if jit_on else fp.jit_reason,
                                           "what": "residual programs compiled into k1tc3 (neurodiffeq_b200/jit.py, nvcc, "
                                                   "cached); PINNJET_JIT=0 keeps the in-kernel interpreter"},
            "fit": fit, "gpu_autograd_baseline": gpu_cmp,
            "loss": loss, "wall_s_timed_region": t_wall,
            "step_ms_stats": {"min": float(step_ms.min()), "median": float(np.median(step_ms)),
                              "max": float(step_ms.max()), "count": int(step_ms.size)},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tearing down a process group whose all-reduce was captured in a CUDA graph can block for minutes inside NCCL
        # (seen on 2 GPUs).  Every rank is done once rank 0 has printed: synchronise and leave without the teardown.
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
