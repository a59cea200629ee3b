#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's configurations.

    python bench.py --gpus N --steps K --warmup W [--workload W] [--path P] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

metric   : accepted RK steps/s x state elements, whole job (all ranks)
step     : ONE full odeint() solve (all accepted + rejected attempts, every output point) of the workload
workloads (BASELINE.json `configs`, SURVEY 8(d); per-GPU sizes, weak scaling -- every rank owns a shard of ONE system with
a shared step size, the per-attempt error-norm exchange runs inside the kernels over NVLink peer memory):
  cfg2       Lorenz 65 536 x 3 fp64, dopri5 (rtol 1e-7, atol 1e-9), 1 000 output points            [default]
  northstar  linear y @ A, 65 536 x 128 fp64, dopri5 -- the size north_star states its HBM target on (SURVEY row K)
  cfg3       spiral MLP 2 -> 50 -> 2, 131 072 x 2 fp32, rk4, 2 000 grid cells
  cfg4       Conv2dODEFunc(64) on 512 x 28 x 28 x 64 fp32 per GPU (4 096 at 8 GPUs), dopri5 1e-3, forward + adjoint
  cfg5       32 stacked Kepler orbits (DETEST D-class), 4 096 x 128 fp64 per GPU (16 384 at 4), dopri8 1e-9
Without --workload the line is cfg2 and carries short runs of the other four under `other_workloads`.

Every workload reports `parity`: at N = 1 the timed path against the oracle (oracle/np_ref.py) on what the oracle finishes
in about a second; at N > 1 each rank's shard of the sharded solve against a single-GPU solve of the WHOLE system (same
counts, values to 1e-9) -- so the scaling run carries multi-GPU parity.

`--impl reference` (and `cpu_baseline`): the oracle port on all host cores (oracle/par_ref.py: the batch split over
processes, the reference's global reductions combined across them), same workload, metric and unit.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "accepted_rk_steps_x_state_elements_per_s"
UNIT = "element-steps/s"


def peaks_json():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:                                           # noqa: BLE001
        return {}


def hbm_peak():
    d = peaks_json()
    if "hbm_gbs" in d:
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(kernel_key):
    """dram bytes per launch of a kernel from the committed ncu digest (profiles/ncu_traffic.json, written by
    scripts/summarize_ncu.py from a `--set full` capture); None when no capture of that kernel is on file."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        e = d.get(kernel_key)
        return (float(e["dram_bytes"]), e.get("source")) if e else (None, None)
    except Exception:                                           # noqa: BLE001
        return None, None


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (recipe in B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
            except (ValueError, IndexError):
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ======================================================================================================================
# workloads: inputs are numpy (seeded), shared by the GPU arm, the parity checks and the CPU arm
# ======================================================================================================================
class Workload(object):
    name = None
    dtype = "f64"
    np_dtype = np.float64
    method = "dopri5"
    rtol, atol = 1e-7, 1e-9
    solver_options = {}
    paths = ()                       # first = default primary
    adaptive = True
    tag = None

    def shape(self):                 # per-GPU state shape
        raise NotImplementedError

    def y0(self, rank):
        raise NotImplementedError

    def t(self):
        raise NotImplementedError

    def elements(self):
        return int(np.prod(self.shape()))

    def problem(self):               # (PROBLEMS key, kwargs) of the right-hand side for the oracle / external-func paths
        raise NotImplementedError

    def func(self, path, dev):
        """(callable, extra solver options) of a path."""
        from problems import PROBLEMS
        name, kw = self.problem()
        ext = PROBLEMS[name](backend="torch", dtype=np.dtype(self.np_dtype).name, device=dev, **kw)
        if path == "external_func_cuda_graph":
            return ext, {"cuda_graph": True}
        if path == "external_func_eager":
            return ext, {}
        raise KeyError(path)

    def torch_dtype(self):
        return torch.float64 if self.np_dtype == np.float64 else torch.float32

    # parity sample: (rows of the per-GPU batch, output times) the oracle finishes in about a second
    def parity_rows(self):
        return min(self.shape()[0], 2048)

    def parity_t(self):
        return self.t()[:3]

    def parity_tol(self):
        return 1e-6 if self.np_dtype == np.float64 else 1e-3


class Cfg2(Workload):
    name, tag = "cfg2", "lorenz_b65536x3_f64_dopri5_1000pts"
    paths = ("fused_rhs", "external_func_cuda_graph", "external_func_eager")
    B, NPTS = 65536, 1000

    def shape(self):
        return (self.B, 3)

    def y0(self, rank):
        return np.array([1.0, 1.0, 1.0]) + 0.1 * np.random.default_rng(rank).standard_normal((self.B, 3))

    def t(self):
        return np.arange(self.NPTS) * 0.01

    def problem(self):
        return "lorenz", {}

    def func(self, path, dev):
        if path == "fused_rhs":
            import tfdiffeq_b200 as tfd
            return tfd.rhs.Lorenz(), {}
        return Workload.func(self, path, dev)

    def parity_rows(self):
        return self.B

    def parity_t(self):
        return self.t()[:11]


class NorthStar(Workload):
    name, tag = "northstar", "linear_b65536x128_f64_dopri5_11pts"
    paths = ("external_func_eager", "external_func_cuda_graph")
    rtol, atol = 1e-6, 1e-9

    def shape(self):
        return (65536, 128)

    def y0(self, rank):
        return np.random.default_rng(100 + rank).standard_normal(self.shape())

    def t(self):
        return np.linspace(0., 2., 11)

    def problem(self):
        return "batched_linear", {"dim": 128, "seed": 0}


class Cfg3(Workload):
    name, tag = "cfg3", "spiral_mlp_b131072x2_f32_rk4_2000steps"
    dtype, np_dtype, method, adaptive = "f32", np.float32, "rk4", False
    paths = ("fused_rhs", "external_func_eager")

    def shape(self):
        return (131072, 2)

    def y0(self, rank):
        return (np.array([2., 0.]) + 0.1 * np.random.default_rng(300 + rank).standard_normal(self.shape())).astype(np.float32)

    def t(self):
        return np.linspace(0., 25., 2001).astype(np.float32)

    def problem(self):
        return "spiral_mlp", {"seed": 0, "hidden": 50}

    def func(self, path, dev):
        if path == "fused_rhs":
            import tfdiffeq_b200 as tfd
            from problems import PROBLEMS
            ref = PROBLEMS["spiral_mlp"](backend="numpy", dtype="float32", seed=0, hidden=50)
            m = tfd.rhs.CubicMLP(hidden=50, cube=True, dtype=torch.float32)
            with torch.no_grad():
                m.W1.copy_(torch.from_numpy(np.asarray(ref.W1, dtype=np.float32)))
                m.W2.copy_(torch.from_numpy(np.asarray(ref.W2, dtype=np.float32)))
            return m.to(dev), {}
        return Workload.func(self, path, dev)

    def parity_rows(self):
        return 32

    def parity_t(self):
        return self.t()


class Cfg5(Workload):
    name, tag = "cfg5", "kepler32_b4096x128_f64_dopri8_rtol1e-9_101pts"
    method, rtol, atol = "dopri8", 1e-9, 1e-9
    paths = ("builtin_rhs_stage_kernels_cuda_graph", "builtin_rhs_stage_kernels", "external_func_cuda_graph", "external_func_eager")

    def func(self, path, dev):
        if path.startswith("builtin_rhs"):
            import tfdiffeq_b200 as tfd
            return tfd.rhs.Kepler(), ({"cuda_graph": True} if path.endswith("cuda_graph") else {})
        return Workload.func(self, path, dev)

    def shape(self):
        return (4096, 128)

    def y0(self, rank):
        from problems import PROBLEMS
        return PROBLEMS["kepler"](backend="numpy").y0(4096, seed=500 + rank)

    def t(self):
        return np.linspace(0., 20., 101)

    def problem(self):
        return "kepler", {"orbits": 32}

    def parity_rows(self):
        return 256

    def parity_t(self):
        return self.t()[:3]


class Cfg4(Workload):
    """forward + adjoint backward; see run_cfg4 (its step is not a plain odeint call)."""
    name, tag = "cfg4", "conv2d_odefunc64_b512x28x28x64_f32_dopri5_tol1e-3_fwd+adjoint"
    dtype, np_dtype, rtol, atol = "f32", np.float32, 1e-3, 1e-3
    solver_options = {"max_num_steps": 1000}
    paths = ("tensor_cores_3xtf32", "torch_fp32")

    def shape(self):
        return (512, 28, 28, 64)

    def y0(self, rank):
        return np.random.default_rng(400 + rank).standard_normal(self.shape()).astype(np.float32)

    def t(self):
        return np.array([0., 1.])


WORKLOADS = {w.name: w for w in (Cfg2(), NorthStar(), Cfg3(), Cfg4(), Cfg5())}


# ======================================================================================================================
# reference arm / cpu baseline: the oracle port on all host cores (oracle/par_ref.py)
# ======================================================================================================================
def cpu_arm(w, budget_s, reps, warmup=0):
    """Time `reps` (+ `warmup`) solves of a bounded sample of workload `w` on the host cores.  The sample is the FULL
    per-GPU batch over the first `npts` output points, `npts` chosen from a short probe so that the whole call takes
    about `budget_s` seconds (the full horizon when that fits)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    if w.name == "cfg4":
        return cpu_arm_cfg4(w, budget_s, reps, warmup)
    import par_ref
    name, pkw = w.problem()
    y0, t = w.y0(0), w.t()
    kw = dict(rtol=w.rtol, atol=w.atol, method=w.method)
    cores = os.cpu_count() or 1
    n_probe = max(2, min(len(t), 13))
    # worker count: every logical core, or half of them when that is faster on a short probe (SMT siblings / the spin
    # barriers of the shared reductions)
    cand = sorted({max(1, cores), max(1, cores // 2)}, reverse=True)
    probe = {}
    for p in cand:
        r = par_ref.solve(name, y0, t[:n_probe], nproc=p, reps=2, pkw=pkw, **kw)
        probe[p] = min(r["seconds"])
    nproc = min(probe, key=probe.get)
    per_pt = probe[nproc] / (n_probe - 1)
    total = reps + warmup
    npts = int(min(len(t), max(n_probe, budget_s / max(total, 1) / max(per_pt, 1e-9))))
    r = par_ref.solve(name, y0, t[:npts], nproc=nproc, reps=total, pkw=pkw, **kw)
    secs = r["seconds"][warmup:]
    vals = [r["n_acc"] * w.elements() / s for s in secs]
    sample = "full %s batch, first %d of %d output points (%.0f%% of the time horizon), oracle port (numpy) on %d worker " \
             "processes of %d host cores, shared step via shared-memory reductions" % (
                 "x".join(str(v) for v in w.shape()), npts, len(t), 100.0 * (t[npts - 1] - t[0]) / (t[-1] - t[0]), nproc, cores)
    return dict(value=float(np.max(vals)), mean_value=float(np.mean(vals)), seconds=[float(s) for s in secs], cores=nproc,
                host_cores=cores, kind="port", sample=sample, n_acc=r["n_acc"], n_rej=r["n_rej"],
                probe_seconds={str(k): v for k, v in probe.items()})


def cpu_arm_cfg4(w, budget_s, reps, warmup):
    """Config 4 on the host: the oracle's dopri5 on torch-CPU tensors (all threads) with the same Conv2dODEFunc, forward
    solve of a 16-sample sub-batch (a conv net has no numpy form; the reference itself would run TF's CPU convolutions)."""
    import np_ref
    import tfdiffeq_b200  # noqa: F401  (only for the module definition; runs on CPU tensors here)
    from tfdiffeq_b200.rhs import Conv2dODEFunc
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    m = Conv2dODEFunc(64, tensor_cores=False)
    nb = 16
    x0 = torch.from_numpy(w.y0(0)[:nb])
    secs, acc = [], 0
    with torch.no_grad():
        for i in range(reps + warmup):
            st = np_ref.Stats()
            t0 = time.perf_counter()
            np_ref.odeint(lambda tt, y: m(torch.as_tensor(float(tt)), y), x0, w.t(), rtol=w.rtol, atol=w.atol, method="dopri5",
                          options=dict(max_num_steps=1000), stats=st)
            dt = time.perf_counter() - t0
            if i >= warmup:
                secs.append(dt)
                acc = st.n_acc
    elems = nb * 28 * 28 * 64
    vals = [acc * elems / s for s in secs]
    return dict(value=float(np.max(vals)), mean_value=float(np.mean(vals)), seconds=secs, cores=torch.get_num_threads(),
                host_cores=os.cpu_count(), kind="port", n_acc=acc, n_rej=None,
                sample="forward solve only, %d of 512 samples (16x28x28x64), oracle dopri5 on torch-CPU tensors, %d threads" % (
                    nb, torch.get_num_threads()))


def run_reference(args, rank, world):
    if rank != 0:
        return
    w = WORKLOADS[args.workload or "cfg2"]
    r = cpu_arm(w, budget_s=90.0, reps=max(args.steps, 1), warmup=args.warmup)
    v = r["mean_value"]
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(r["seconds"])), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": w.dtype, "data": "synthetic",
            "config": {"workload": w.tag, "sample": r["sample"], "best_step_value": r["value"],
                       "accepted": r["n_acc"], "rejected": r["n_rej"]},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ======================================================================================================================
# our arm
# ======================================================================================================================
class Ctx(object):
    """per-process state of the GPU arm"""

    def __init__(self, rank, world, local_rank):
        self.rank, self.world = rank, world
        self.dev = torch.device("cuda", local_rank)
        torch.cuda.set_device(self.dev)
        # page-locked staging buffers are allocated after this point: keep them (and this process) on the GPU's NUMA node
        from tfdiffeq_b200.comm import bind_to_gpu_numa
        self.numa_node = bind_to_gpu_numa(self.dev)
        self.group = None
        if world > 1:
            import torch.distributed as dist
            from tfdiffeq_b200.comm import SharedStepGroup
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
            dist.init_process_group("nccl", device_id=self.dev)
            self.group = SharedStepGroup()
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=self.dev)     # > 126 MB L2

    def barrier(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(self.dev)

    def reduce(self, ms, sums):
        """max over ranks of the time, sum over ranks of the work counters"""
        if self.world == 1:
            return ms, sums
        import torch.distributed as dist
        tt = torch.tensor([ms], dtype=torch.float64, device=self.dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ww = torch.tensor(list(sums), dtype=torch.float64, device=self.dev)
        dist.all_reduce(ww, op=dist.ReduceOp.SUM)
        return float(tt[0]), [float(x) for x in ww]

    def all_true(self, flag):
        if self.world == 1:
            return bool(flag)
        import torch.distributed as dist
        v = torch.tensor([0 if flag else 1], dtype=torch.int64, device=self.dev)
        dist.all_reduce(v)
        return int(v[0]) == 0


def timed(ctx, step_fn, steps, warmup):
    """W untimed + K timed steps, barrier + synchronize on both sides, CUDA events per step, L2 flushed between steps
    (untimed).  step_fn() -> (work_units, launches_in_graph)."""
    from tfdiffeq_b200 import _lib
    for _ in range(warmup):
        step_fn()
    torch.cuda.synchronize(ctx.dev)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    work = 0.0
    extra_launches = 0
    l0 = int(_lib.lib.b2ode_launch_count())
    ctx.barrier()
    w0 = time.perf_counter()
    for i in range(steps):
        ctx.flush.fill_(i & 0xFF)
        ev[i][0].record()
        wk, xl = step_fn()
        ev[i][1].record()
        work += wk
        extra_launches += xl
    ctx.barrier()
    wall = time.perf_counter() - w0
    launches = int(_lib.lib.b2ode_launch_count()) - l0 + extra_launches
    per_step = [a.elapsed_time(b) for a, b in ev]
    if os.environ.get("B2ODE_BENCH_DEBUG"):
        sys.stderr.write("rank %d per-step ms: %s\n" % (ctx.rank, " ".join("%.3f" % v for v in per_step)))
    ms = sum(per_step)
    ms, (work, launches) = ctx.reduce(ms, (work, launches))
    return dict(value=work / (ms * 1e-3), ms_per_step=ms / steps, launches=int(launches), wall=wall)


DUMP_BYTES = 60 * 1000 * 1000       # --dump-outputs: data of all files together, under 64 MB with room for the headers


def sample_outputs(arrays):
    """Host copies of the arrays a caller of the timed path received from its last step (--dump-outputs).  `arrays` maps
    a name to (tensor, batch axis or None).  Tensors with a batch axis keep the same rows: all of them when everything fits
    in DUMP_BYTES, otherwise a sorted sample drawn with np.random.default_rng(0), so that runs with the same arguments
    dump the same elements.  Tensors without a batch axis are kept whole."""
    fixed = sum(t.numel() * t.element_size() for t, ax in arrays.values() if ax is None)
    batched = [(t, ax) for t, ax in arrays.values() if ax is not None]
    idx = None
    if batched:
        n = batched[0][0].shape[batched[0][1]]
        assert all(t.shape[ax] == n for t, ax in batched)
        per_row = sum(t.numel() // n * t.element_size() for t, ax in batched)
        rows = min(n, (DUMP_BYTES - fixed) // per_row)
        if rows < n:
            idx = np.sort(np.random.default_rng(0).choice(n, size=rows, replace=False))
    out = {}
    for name, (t, ax) in arrays.items():
        t = t.detach()
        if ax is not None and idx is not None:
            t = t.index_select(ax, torch.from_numpy(idx).to(t.device))
        out[name] = t.cpu().numpy().astype(np.float64 if t.dtype == torch.float64 else np.float32, copy=False)
    return out


def make_solver(ctx, w, path, host_output=None):
    """Closures for one workload / path: solve(y_dev) -> solution, plus bookkeeping of accepted steps."""
    import tfdiffeq_b200 as tfd
    f, extra = w.func(path, ctx.dev)
    opts = dict(w.solver_options)
    opts.update(extra)
    if host_output is not None:
        opts["host_output"] = host_output
    if ctx.group is not None and w.adaptive:
        opts["shared_step_group"] = ctx.group
    kw = dict(rtol=w.rtol, atol=w.atol, method=w.method, options=opts)
    t_host = torch.from_numpy(np.asarray(w.t(), dtype=np.float64))

    def solve(y):
        return tfd.odeint(f, y, t_host, **kw)
    return solve, opts


def graph_launches(stats, n_k_minus_1_plus_2):
    """library kernels inside replayed CUDA graphs are not seen by the host-side launch counter"""
    if not stats.get("cuda_graph"):
        return 0
    return max(stats["n_accepted"] + stats["n_rejected"] - 2, 0) * n_k_minus_1_plus_2


def run_odeint_workload(ctx, w, path, steps, warmup, want_e2e=True, keep_output=False):
    import tfdiffeq_b200 as tfd
    solve, _ = make_solver(ctx, w, path)
    y0_host = torch.from_numpy(np.ascontiguousarray(w.y0(ctx.rank))).pin_memory()
    y0_dev = y0_host.to(ctx.dev)
    nk = {"dopri5": 8, "dopri8": 15, "rk4": 0}.get(w.method, 0)
    n_el = w.elements()
    stats_box = {}
    last = {}

    def step_dev():
        sol = solve(y0_dev)
        if keep_output:
            last["solution"] = sol
        s = tfd.last_stats
        stats_box.update(s)
        return float(s["n_accepted"]) * n_el, graph_launches(s, nk)
    res = timed(ctx, step_dev, steps, max(warmup, 3))
    if keep_output:
        res["outputs"] = sample_outputs({"solution": (last.pop("solution"), 1)})
    res["n_acc"], res["n_rej"] = stats_box.get("n_accepted"), stats_box.get("n_rejected")
    res["fused_rhs"] = bool(stats_box.get("fused_rhs"))
    if want_e2e:
        sol_shape = (len(w.t()),) + tuple(w.shape())
        out_host = torch.empty(sol_shape, dtype=w.torch_dtype()).pin_memory()

        solve_h, _ = make_solver(ctx, w, path, host_output=out_host)

        def step_e2e():
            y = y0_host.to(ctx.dev, non_blocking=True)           # H2D of the inputs inside the timed region
            sol = solve_h(y)                                     # the public API delivers the whole solution into out_host
            assert sol.data_ptr() == out_host.data_ptr()         # (D2H inside the timed region; streamed behind the solve
            torch.cuda.synchronize(ctx.dev)                      #  when the path supports it)
            s = tfd.last_stats
            return float(s["n_accepted"]) * n_el, graph_launches(s, nk)
        e = timed(ctx, step_e2e, max(1, min(steps, 5)), 1)
        res["e2e"] = {"value": e["value"], "unit": UNIT, "ms_per_step": e["ms_per_step"],
                      "h2d_bytes_per_step": int(y0_host.numel() * y0_host.element_size() + len(w.t()) * 8),
                      "d2h_bytes_per_step": int(out_host.numel() * out_host.element_size())}
        del out_host
    return res


# ---- parity -----------------------------------------------------------------------------------------------------------
def parity_odeint(ctx, w, path):
    """N = 1: the timed path vs the oracle on (parity_rows x parity_t).  N > 1: each rank's shard of the sharded solve vs a
    single-GPU solve of the WHOLE system (all ranks' rows), same short horizon."""
    import tfdiffeq_b200 as tfd
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    tp = np.asarray(w.parity_t(), dtype=np.float64)
    t_host = torch.from_numpy(tp)
    f, extra = w.func(path, ctx.dev)
    base_opts = dict(w.solver_options)
    base_opts.update(extra)
    kw = dict(rtol=w.rtol, atol=w.atol, method=w.method)
    tol = w.parity_tol()
    if ctx.world == 1 or not w.adaptive:
        import np_ref
        from problems import PROBLEMS
        rows = w.parity_rows()
        y0 = w.y0(ctx.rank)
        if w.adaptive:
            y0 = y0[:rows]                      # a sub-SYSTEM: shared step over these rows only, on both sides
            got = tfd.odeint(f, torch.from_numpy(np.ascontiguousarray(y0)).to(ctx.dev), t_host, options=base_opts, **kw)
            s = dict(tfd.last_stats)
            got = got.cpu().numpy()
        else:                                   # fixed grid: trajectories are independent -> compare a subset of the full solve
            full = tfd.odeint(f, torch.from_numpy(np.ascontiguousarray(y0)).to(ctx.dev), t_host, options=base_opts, **kw)
            s = dict(tfd.last_stats)
            idx = np.random.default_rng(7).choice(y0.shape[0], size=rows, replace=False)
            got = full[:, torch.from_numpy(idx).to(ctx.dev)].cpu().numpy()
            y0 = y0[idx]
            del full
        name, pkw = w.problem()
        st = np_ref.Stats()
        ref = np_ref.odeint(PROBLEMS[name](backend="numpy", dtype=np.dtype(w.np_dtype).name, **pkw), y0, tp, stats=st, **kw)
        err = float(np.max(np.abs(got - ref) / np.maximum(np.abs(ref), 1.0)))
        counts_ok = (not w.adaptive) or (s["n_accepted"], s["n_rejected"]) == (st.n_acc, st.n_rej)
        ok = bool(err <= tol and counts_ok)
        return {"ok": ctx.all_true(ok), "against": "oracle (np_ref) on %d rows x %d output points" % (y0.shape[0], len(tp)),
                "max_rel_err": err, "tol": tol, "counts": [s["n_accepted"], s["n_rejected"]],
                "counts_oracle": [st.n_acc, st.n_rej]}
    # ---- N > 1: sharded vs whole system on one GPU -------------------------------------------------------------------
    opts = dict(base_opts, shared_step_group=ctx.group)
    mine = tfd.odeint(f, torch.from_numpy(np.ascontiguousarray(w.y0(ctx.rank))).to(ctx.dev), t_host, options=opts, **kw)
    s = dict(tfd.last_stats)
    whole_y0 = np.concatenate([w.y0(r) for r in range(ctx.world)], 0)
    solo_opts = dict(base_opts)
    solo_opts.pop("cuda_graph", None)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")        # the whole system may exceed the fused kernel's co-residency limit
        whole = tfd.odeint(f, torch.from_numpy(whole_y0).to(ctx.dev), t_host, options=solo_opts, **kw)
    s1 = dict(tfd.last_stats)
    n = w.shape()[0]
    ref = whole[:, ctx.rank * n:(ctx.rank + 1) * n]
    err = float(((mine - ref).abs() / ref.abs().clamp_min(1.0)).max())
    ok = bool(err <= 1e-9 if w.np_dtype == np.float64 else err <= 1e-4) and \
        (s["n_accepted"], s["n_rejected"]) == (s1["n_accepted"], s1["n_rejected"])
    return {"ok": ctx.all_true(ok), "against": "single-GPU solve of the whole %d-row system (%d output points)" % (
        whole_y0.shape[0], len(tp)), "max_rel_err": err, "counts": [s["n_accepted"], s["n_rejected"]],
        "counts_single_gpu": [s1["n_accepted"], s1["n_rejected"]]}


# ---- config 4: forward + adjoint ---------------------------------------------------------------------------------------
def run_cfg4(ctx, w, path, steps, warmup, keep_output=False):
    import tfdiffeq_b200 as tfd
    from tfdiffeq_b200 import adjoint as adj
    torch.manual_seed(0)
    m = tfd.rhs.Conv2dODEFunc(64, tensor_cores=(True if path == "tensor_cores_3xtf32" else False)).to(ctx.dev)
    x_host = torch.from_numpy(w.y0(ctx.rank)).pin_memory()
    t_host = torch.tensor([0., 1.])
    opts = dict(w.solver_options)
    if ctx.group is not None:
        opts["shared_step_group"] = ctx.group
    n_el = w.elements()
    n_par = sum(p.numel() for p in m.parameters())
    n_aug = 2 * n_el + 1 + n_par
    gx_host = torch.empty(w.shape(), dtype=torch.float32).pin_memory()
    gp_host = torch.empty(n_par, dtype=torch.float32).pin_memory()
    box = {}

    def step(e2e):
        for p in m.parameters():
            p.grad = None
        x = (x_host.to(ctx.dev, non_blocking=True) if e2e else x_dev).detach().requires_grad_(True)
        with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
            out = tfd.odeint_adjoint(m, x, t_host, rtol=w.rtol, atol=w.atol, method="dopri5", options=opts)
            loss = (out[-1] ** 2).mean()
            loss.backward()
        if e2e:
            gx_host.copy_(x.grad, non_blocking=True)
            gp_host.copy_(torch.cat([p.grad.reshape(-1) for p in m.parameters()]), non_blocking=True)
            box["loss"] = float(loss)                               # D2H read of the step's result
            torch.cuda.synchronize(ctx.dev)
        elif keep_output:
            box["outputs"] = (out, x, [p.grad for p in m.parameters()])
        fwd, bwd = adj.last_stats["forward"], adj.last_stats["backward"]
        box.update(fwd_acc=fwd["n_accepted"], fwd_rej=fwd["n_rejected"], bwd_acc=sum(b["n_accepted"] for b in bwd),
                   bwd_rej=sum(b["n_rejected"] for b in bwd), nfe=m.nfe)
        return float(fwd["n_accepted"]) * n_el + float(sum(b["n_accepted"] for b in bwd)) * n_aug, 0
    x_dev = x_host.to(ctx.dev)
    res = timed(ctx, lambda: step(False), steps, warmup)
    if keep_output:
        out, x, grads = box.pop("outputs")
        res["outputs"] = sample_outputs({"solution": (out, 1), "input_grad": (x.grad, 0),
                                         "param_grad": (torch.cat([g.reshape(-1) for g in grads]), None)})
        del out, x, grads
    e = timed(ctx, lambda: step(True), max(1, min(steps, 3)), 1)
    res["e2e"] = {"value": e["value"], "unit": UNIT, "ms_per_step": e["ms_per_step"],
                  "h2d_bytes_per_step": int(x_host.numel() * 4), "d2h_bytes_per_step": int(gx_host.numel() * 4 + n_par * 4 + 4)}
    res.update(fwd_accepted=box["fwd_acc"], fwd_rejected=box["fwd_rej"], bwd_accepted=box["bwd_acc"],
               bwd_rejected=box["bwd_rej"], state_elements=n_el, augmented_state_elements=n_aug, parameters=n_par)
    # parity: the tensor-core path vs the same module in plain fp32 torch (cuDNN / cuBLAS, TF32 off), forward solution and
    # parameter gradient; at N > 1 additionally the sharded forward vs the whole batch on one GPU
    par = {}
    with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
        def fwd_bwd(mod, o):
            for p in mod.parameters():
                p.grad = None
            x = x_dev.detach().requires_grad_(True)
            out = tfd.odeint_adjoint(mod, x, t_host, rtol=w.rtol, atol=w.atol, method="dopri5", options=o)
            (out[-1] ** 2).mean().backward()
            return out[-1].detach(), torch.cat([p.grad.reshape(-1) for p in mod.parameters()]), x.grad
        a_out, a_gp, a_gx = fwd_bwd(m, opts)
        mode = m.tensor_cores
        m.tensor_cores = False
        old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        try:
            b_out, b_gp, b_gx = fwd_bwd(m, opts)
        finally:
            torch.backends.cuda.matmul.allow_tf32 = old
            m.tensor_cores = mode
        rel = lambda a, b: float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))   # noqa: E731
        par = {"against": "same module in plain fp32 torch (cuDNN/cuBLAS, TF32 off), same batch",
               "solution_rel_err": rel(a_out, b_out), "param_grad_rel_err": rel(a_gp, b_gp), "input_grad_rel_err": rel(a_gx, b_gx)}
        ok = par["solution_rel_err"] <= 1e-3 and par["param_grad_rel_err"] <= 1e-2 and par["input_grad_rel_err"] <= 1e-2
        if ctx.world > 1:
            with torch.no_grad():
                whole = torch.from_numpy(np.concatenate([w.y0(r) for r in range(ctx.world)], 0)).to(ctx.dev)
                solo = tfd.odeint(m, whole, t_host, rtol=w.rtol, atol=w.atol, method="dopri5", options=dict(w.solver_options))
                s1 = dict(tfd.last_stats)
                mine = tfd.odeint(m, x_dev, t_host, rtol=w.rtol, atol=w.atol, method="dopri5", options=opts)
                s = dict(tfd.last_stats)
            n = w.shape()[0]
            par["sharded_vs_single_gpu_rel_err"] = rel(mine[-1], solo[-1][ctx.rank * n:(ctx.rank + 1) * n])
            par["counts"] = [s["n_accepted"], s["n_rejected"]]
            par["counts_single_gpu"] = [s1["n_accepted"], s1["n_rejected"]]
            ok = ok and par["sharded_vs_single_gpu_rel_err"] <= 1e-4 and par["counts"] == par["counts_single_gpu"]
            del whole, solo
        par["ok"] = ctx.all_true(bool(ok))
    res["parity"] = par
    return res


# ---- per-kernel rooflines (CUDA events recorded by the library around its own launches) ---------------------------------
def family_times(fn, fams):
    import ctypes as C
    from tfdiffeq_b200 import _lib
    mask = 0
    for f in fams:
        mask |= 1 << f
    _lib.check(_lib.lib.b2ode_timing_enable(mask))
    fn()
    torch.cuda.synchronize()
    out = {}
    for f in fams:
        ms, cnt = C.c_double(), C.c_int()
        _lib.check(_lib.lib.b2ode_timing_read(f, C.byref(ms), C.byref(cnt)))
        out[f] = (ms.value, cnt.value)
    _lib.check(_lib.lib.b2ode_timing_enable(0))
    return out


def roofline_northstar(ctx, peak, peak_src):
    """k_rk_finalize / k_rk_stage at 65 536 x 128 fp64: 64 MiB per buffer, every launch streams far more than the 126 MB L2."""
    import tfdiffeq_b200 as tfd
    from tfdiffeq_b200 import _lib
    w = WORKLOADS["northstar"]
    solve, _ = make_solver(ctx, w, "external_func_eager")
    y0 = torch.from_numpy(w.y0(ctx.rank)).to(ctx.dev)
    solve(y0)
    st = {}

    def go():
        ctx.flush.fill_(5)
        solve(y0)
        st.update(tfd.last_stats)
    ft = family_times(go, (_lib.FAM_FINALIZE, _lib.FAM_STAGE, _lib.FAM_STAGE0, _lib.FAM_EMIT))
    n = w.elements()
    att = max(st["n_accepted"] + st["n_rejected"], 1)
    commit_frac = max(st["n_accepted"] - 1, 0) / float(att)
    per = {}
    for fam, name, elems in ((_lib.FAM_FINALIZE, "finalize", float(tfd_finalize_elems(st))), (_lib.FAM_STAGE, "stages_1_to_5", 29.0 / 5),
                             (_lib.FAM_STAGE0, "stage_0", 3.0 + 2.0 * commit_frac)):
        ms, cnt = ft[fam]
        if cnt:
            avg = ms / cnt
            gbs = elems * n * 8 / (avg * 1e-3) / 1e9
            per[name] = {"launches": cnt, "avg_ms": avg, "algorithmic_bytes": int(elems * n * 8), "achieved": gbs, "frac": gbs / peak}
    fin = per.get("finalize", {})
    traffic, src = ncu_traffic("k_rk_finalize_f64_northstar")
    return {"bound": "hbm", "kernel": "k_rk_finalize<double,6>: error combine + error norm + controller%s" % (
        " + dense output" if st.get("emit_fused") else ""), "workload": w.tag,
        "achieved": fin.get("achieved"), "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": fin.get("frac"),
        "traffic": traffic, "traffic_source": src, "algorithmic_bytes_per_launch": fin.get("algorithmic_bytes"),
        "avg_launch_ms": fin.get("avg_ms"), "launches_timed": fin.get("launches"), "per_kernel": per,
        "n_accepted": st.get("n_accepted"), "n_rejected": st.get("n_rejected"),
        "how": "CUDA events recorded by the library around each launch on its own stream (b2ode_timing_enable), L2 flushed before the solve"}


def tfd_finalize_elems(stats):
    """elements the finalize kernel reads per launch for Dopri5: y0, y1 and the six k's with a non-zero error weight"""
    return 8


def roofline_fused_cfg2(ctx, peak, peak_src):
    """The persistent kernel of the cfg2 headline: it keeps state and k's in registers, so HBM sees only the solution slab;
    its time is set by FP64 issue + one grid-wide barrier per attempted step, not by bandwidth."""
    import tfdiffeq_b200 as tfd
    from tfdiffeq_b200 import _lib
    w = WORKLOADS["cfg2"]
    solve, _ = make_solver(ctx, w, "fused_rhs")
    y0 = torch.from_numpy(w.y0(ctx.rank)).to(ctx.dev)
    solve(y0)
    st = {}

    def go():
        ctx.flush.fill_(6)
        solve(y0)
        st.update(tfd.last_stats)
    ft = family_times(go, (_lib.FAM_FUSED,))
    ms, cnt = ft[_lib.FAM_FUSED]
    if not cnt:
        return None
    avg = ms / cnt
    n = w.elements()
    slab = (len(w.t()) + 1) * n * 8                       # the (T, B, 3) fp64 solution written once + y0 read once
    att = st["n_accepted"] + st["n_rejected"]
    # arithmetic floor: ~410 FP64 instructions per trajectory-attempt (6 Lorenz evaluations, 6 stage combines, error,
    # norms) on 148 SMs x 64 FP64 lanes x 1.965 GHz = 18.6e12 DP instr/s
    dp_floor_us = 410.0 * w.shape()[0] / 18.6e12 * 1e6
    traffic, src = ncu_traffic("k_fused_adaptive_lorenz_f64")
    return {"bound": "fp64 issue + grid barrier (NOT hbm)", "kernel": "k_fused_adaptive<double, RhsLorenz, 7> (one launch = one whole solve)",
            "workload": w.tag, "achieved": slab / (avg * 1e-3) / 1e9, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
            "frac": slab / (avg * 1e-3) / 1e9 / peak, "traffic": traffic, "traffic_source": src,
            "algorithmic_bytes_per_launch": int(slab), "avg_launch_ms": avg, "launches_timed": cnt,
            "attempts_per_solve": att, "us_per_attempt": avg * 1e3 / max(att, 1), "fp64_floor_us_per_attempt": dp_floor_us,
            "fp64_pipe_frac_estimate": dp_floor_us / (avg * 1e3 / max(att, 1)),
            "note": "algorithmic bytes = the solution slab (all this kernel has to move); the 352 B/element-step of SURVEY 8(d) is the "
                    "traffic of a func-external design and does not apply. The limiter is latency: one grid-wide reduction per attempt."}


def tensor_core_block(ctx):
    """SURVEY 8(f)-3: the ODENet MLP func (dense_odenet.py:85-92, 64 -> 256 -> 256 -> 64, relu) on 131 072 rows inside dopri5
    (rtol = atol = 1e-3): default fp32-accurate 3xTF32 layers, opt-in single-pass TF32 chained kernel, cuBLAS baselines."""
    import tfdiffeq_b200 as tfd
    dev = ctx.dev
    Bm, Dm, Hm = 131072, 64, 256
    torch.manual_seed(0)
    m = tfd.rhs.DenseMLP(Dm, Hm, "relu").to(dev)
    y0 = torch.randn(Bm, Dm, device=dev)
    t = torch.tensor([0., 1.])
    kw = dict(rtol=1e-3, atol=1e-3, method="dopri5")

    def solve_ms(reps):
        ts = []
        for _ in range(reps):
            ctx.flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            tfd.odeint(m, y0, t, **kw)
            b.record()
            torch.cuda.synchronize(dev)
            ts.append(a.elapsed_time(b))
        return sorted(ts)[len(ts) // 2]

    def kernel_ms():
        x = torch.randn(Bm, Dm, device=dev)
        ev = []
        with torch.no_grad():
            for _ in range(3):
                m(0.0, x)
            for _ in range(10):
                ctx.flush.fill_(2)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                m(0.0, x)
                b.record()
                torch.cuda.synchronize(dev)
                ev.append(a.elapsed_time(b))
        return sorted(ev)[len(ev) // 2]
    out = {"workload": "odenet_mlp_64x256x256x64_relu_b131072_f32_dopri5"}
    flops = 2.0 * Bm * (Dm * Hm + Hm * Hm + Hm * Dm)
    bf16 = peaks_json().get("bf16_tflops")
    peak_tf32 = (float(bf16) / 2.0) if bf16 else 1125.0
    for mode, key in ((True, "3xtf32_default"), ("tf32", "tf32_opt_in")):
        m.tensor_cores = mode
        solve_ms(2)
        ms = solve_ms(5)
        st = dict(tfd.last_stats)
        k_ms = kernel_ms()
        mult = 3.0 if mode is True else 1.0
        tf = mult * flops / (k_ms * 1e-3) / 1e12
        out[key] = {"ms_per_solve": ms, "nfe": st.get("nfe"), "element_steps_per_s": st.get("n_accepted", 0) * Bm * Dm / (ms * 1e-3),
                    "ms_per_evaluation": k_ms,
                    "roofline": {"bound": "tensor", "achieved": tf, "peak": peak_tf32, "unit": "TFLOP/s", "frac": tf / peak_tf32,
                                 "peak_source": "half of MEASURED_PEAKS.json bf16_tflops (TF32 = bf16 / 2 on sm_100)" if bf16 else "fallback 1125",
                                 "flops_counted": "tensor-core flops actually issued (3 passes for 3xTF32)" if mode is True else "2*M*K*N per layer"}}
    m.tensor_cores = False
    torch.backends.cuda.matmul.allow_tf32 = False
    solve_ms(1)
    out["ms_per_solve_torch_fp32_matmul"] = solve_ms(3)
    torch.backends.cuda.matmul.allow_tf32 = True
    solve_ms(1)
    out["ms_per_solve_cublas_tf32_layers"] = solve_ms(3)
    torch.backends.cuda.matmul.allow_tf32 = False
    return out


def run_workload(ctx, name, path, steps, warmup, want_parity=True, keep_output=False):
    w = WORKLOADS[name]
    path = path or w.paths[0]
    if name == "cfg4":
        res = run_cfg4(ctx, w, path, steps, warmup, keep_output)
    else:
        res = run_odeint_workload(ctx, w, path, steps, warmup, keep_output=keep_output)
        if want_parity:
            res["parity"] = parity_odeint(ctx, w, path)
    res["path"] = path
    res["workload"] = w.tag
    res["dtype"] = w.dtype
    return res


def run_ours(args, rank, world, local_rank):
    import tfdiffeq_b200 as tfd  # noqa: F401
    ctx = Ctx(rank, world, local_rank)
    peak, peak_src = hbm_peak()
    primary_name = args.workload or "cfg2"
    w = WORKLOADS[primary_name]
    primary_path = args.path or w.paths[0]
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    main = run_workload(ctx, primary_name, primary_path, args.steps, max(args.warmup, 3),
                        keep_output=args.dump_outputs is not None)
    outputs = main.pop("outputs", {})
    if rank == 0 and outputs:                                      # at N > 1: rank 0's shard
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    del outputs
    others_paths = {}
    if primary_name != "cfg4":
        for p in w.paths:
            if p != primary_path:
                r = run_odeint_workload(ctx, w, p, max(1, min(args.steps, 2)), 1, want_e2e=False)
                others_paths[p] = {"value": r["value"], "unit": UNIT, "ms_per_step": r["ms_per_step"]}
    other_workloads = {}
    if args.workload is None and not args.quick:
        for name in ("northstar", "cfg3", "cfg4", "cfg5"):
            try:
                r = run_workload(ctx, name, None, 2, 1)
                other_workloads[name] = {k: r[k] for k in r if k not in ("wall",)}
            except Exception as e:                                 # noqa: BLE001  (never lose the main line)
                other_workloads[name] = {"error": repr(e)[:300]}
    clocks = sampler.stop() if rank == 0 else None

    roof = roof_primary = tc = cpu = None
    # per-kernel timing passes run on every rank (the kernels exchange over NVLink when a group is attached) ...
    try:
        roof = roofline_northstar(ctx, peak, peak_src)
    except Exception as e:                                         # noqa: BLE001
        roof = {"error": repr(e)[:300]}
    if primary_name == "cfg2" and primary_path == "fused_rhs":
        try:
            roof_primary = roofline_fused_cfg2(ctx, peak, peak_src)
        except Exception as e:                                     # noqa: BLE001
            roof_primary = {"error": repr(e)[:300]}
    if rank == 0 and world == 1 and not args.quick:
        try:
            tc = tensor_core_block(ctx)
        except Exception as e:                                     # noqa: BLE001
            tc = {"error": repr(e)[:300]}
        if not args.no_cpu_baseline:
            try:
                c = cpu_arm(w, budget_s=20.0, reps=2)
                cpu = {"value": c["value"], "unit": UNIT, "cores": c["cores"], "kind": c["kind"], "sample": c["sample"],
                       "seconds": c["seconds"], "host_cores": c["host_cores"]}
            except Exception as e:                                 # noqa: BLE001
                cpu = {"error": repr(e)[:300]}
    if rank == 0:
        line = {
            "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": w.dtype, "data": "synthetic",
            "config": {"workload": w.tag, "per_gpu_shape": list(w.shape()), "method": w.method, "rtol": w.rtol, "atol": w.atol,
                       "n_out": len(w.t()), "path": primary_path,
                       "l2": "flushed between timed iterations (256 MiB write)", "numa_node_bound": ctx.numa_node,
                       "parallelism": ("batch shards of one system, shared step via in-kernel NVLink mailbox exchange"
                                       if world > 1 else "single GPU"),
                       "accepted_per_solve": main.get("n_acc"), "rejected_per_solve": main.get("n_rej")},
            "parity": main.get("parity"),
            "roofline": roof,
            "roofline_primary_kernel": roof_primary,
            "cpu_baseline": cpu,
            "e2e": main.get("e2e"),
            "gpu_launches": main["launches"],
            "other_paths": others_paths,
            "other_workloads": other_workloads,
            "tensor_core_func": tc,
            "wall_s_timed_region": main["wall"],
            "clocks": clocks,
        }
        for k in ("fwd_accepted", "fwd_rejected", "bwd_accepted", "bwd_rejected", "state_elements", "augmented_state_elements"):
            if k in main:
                line["config"][k] = main[k]
        print(json.dumps(line))
    if ctx.group is not None:
        ctx.group.close()
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--path", default=None, help="which public-API path of the workload is the primary (timed) one")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="primary workload only: skip other_workloads / tensor_core_func / cpu_baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the primary path returned in its last timed step to DIR/<name>.npy (float32 / float64, "
                         "a seeded sample of the batch rows, under 64 MB in all), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
