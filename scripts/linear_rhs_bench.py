"""North-star workload (bench.py's NorthStar: 65 536 x 128 fp64, y' = y @ A, dopri5, rtol 1e-6 / atol 1e-9, 11 outputs) on
four paths in one process, alternating over the rounds:

  external_func_eager          BatchedLinear as an ordinary func (cuBLAS DGEMM per stage) -- what bench.py times
  external_func_cuda_graph     the same with one attempt captured in a CUDA graph and replayed
  linear_stages_eager          rhs.LinearSystem: every stage is one k_rk_stage_linear launch (stage combine + DMMA GEMM)
  linear_stages_cuda_graph     the same, replayed from a CUDA graph

Each solve is timed with CUDA events; a 256 MiB buffer is overwritten between solves (the 126 MB L2 starts cold); every
path is warmed up first.  A separate run with b2ode_timing_enable times the stage-GEMM launches alone (family
FAM_STAGE_GEMM) and sets the achieved FP64 FLOP/s and algorithmic bytes/s against the measured DMMA rate (--dmma-tflops,
from scripts/micro/dmma_rate.cu) and an HBM rate measured here (device-to-device copy of 2 GiB), naming the bound.  Both
paths' outputs are compared at full size (same accepted / rejected / NFE counts, 1e-10 relative).

    python scripts/linear_rhs_bench.py --rounds 5 --dmma-tflops X --out OUTDIR
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import bench  # noqa: E402  (make_solver, family_times, Ctx's L2-flush buffer)


def gpu_query():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True, timeout=60)
    return q.stdout.strip()


def hbm_rate(dev):
    """bytes/s of a 2 GiB device-to-device copy (read + write), best of 10"""
    n = 2 << 30
    a = torch.empty(n, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    a.fill_(1)
    best = 0.0
    for _ in range(12):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = max(best, 2.0 * n / (e0.elapsed_time(e1) * 1e-3))
    del a, b
    return best


def stage_bytes(tab, n_bytes):
    """algorithmic HBM bytes of the stage-GEMM launches of one attempt: stage 0's evaluation reads the stage input and
    writes k; stage i reads y0 and its nonzero-coefficient k's and writes k (the last one also writes y1)"""
    total = 2 * n_bytes
    for i in range(1, tab.n_k - 1):
        nnz = sum(1 for b in tab.beta[i] if b != 0.0)
        total += (1 + nnz + 1) * n_bytes + (n_bytes if i == tab.n_k - 2 else 0)
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--dmma-tflops", type=float, default=float("nan"), help="measured DMMA rate (scripts/micro/dmma_rate)")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("linear_rhs_bench.py needs a GPU")
    os.makedirs(args.out, exist_ok=True)
    import tfdiffeq_b200 as tfd
    from tfdiffeq_b200 import _lib, tableaus
    from problems import PROBLEMS

    ctx = bench.Ctx(0, 1, 0)
    w = bench.WORKLOADS["northstar"]
    dev = ctx.dev
    gpu = gpu_query()
    y0 = torch.tensor(w.y0(0), device=dev)
    t_host = torch.from_numpy(np.asarray(w.t(), dtype=np.float64))
    rows, D = w.shape()
    A = torch.as_tensor(PROBLEMS["batched_linear"](backend="numpy", **w.problem()[1]).A)
    lin = tfd.rhs.LinearSystem(A).to(dev)
    kw = dict(rtol=w.rtol, atol=w.atol, method=w.method)

    def lin_solver(graph):
        opts = {"fused_rhs": "stages", "cuda_graph": graph}
        return lambda y: tfd.odeint(lin, y, t_host, options=opts, **kw)
    paths = {
        "external_func_eager": bench.make_solver(ctx, w, "external_func_eager")[0],
        "external_func_cuda_graph": bench.make_solver(ctx, w, "external_func_cuda_graph")[0],
        "linear_stages_eager": lin_solver(False),
        "linear_stages_cuda_graph": lin_solver(True),
    }
    outs, stats = {}, {}
    for name, solve in paths.items():                      # warm-up (module load, cuBLAS heuristics, graph capture)
        outs[name] = solve(y0)
        stats[name] = dict(tfd.last_stats)
    torch.cuda.synchronize()
    ref = outs["external_func_eager"].cpu().numpy()
    check = {}
    for name in paths:
        got = outs[name].cpu().numpy()
        s, r = stats[name], stats["external_func_eager"]
        check[name] = dict(counts=[s["n_accepted"], s["n_rejected"], s["nfe"]],
                           counts_equal=(s["n_accepted"], s["n_rejected"], s["nfe"]) == (r["n_accepted"], r["n_rejected"], r["nfe"]),
                           max_rel_err=float(np.max(np.abs(got - ref)) / max(1.0, float(np.max(np.abs(ref))))),
                           stage_rhs=bool(s.get("stage_rhs")), cuda_graph=bool(s.get("cuda_graph")))
    outs.clear()

    times = {name: [] for name in paths}
    for rnd in range(args.rounds):
        order = list(paths) if rnd % 2 == 0 else list(reversed(list(paths)))
        for name in order:
            ctx.flush.fill_(rnd & 0xFF)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            sol = paths[name](y0)
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1))
            del sol

    # the stage-GEMM launches alone (eager path: events cannot be read back from a graph)
    attempts = stats["linear_stages_eager"]["n_accepted"] + stats["linear_stages_eager"]["n_rejected"]
    ctx.flush.fill_(7)
    fam = bench.family_times(lambda: paths["linear_stages_eager"](y0), (_lib.FAM_STAGE_GEMM, _lib.FAM_STAGE0, _lib.FAM_FINALIZE,
                                                                        _lib.FAM_EMIT))
    g_ms, g_cnt = fam[_lib.FAM_STAGE_GEMM]
    n_bytes = rows * D * 8
    flop = 2.0 * rows * D * D * g_cnt
    byt = 2 * (2 * n_bytes) + attempts * stage_bytes(tableaus.DOPRI5, n_bytes)   # f0 and the initial-step probe, then attempts
    hbm = hbm_rate(dev)
    dmma = args.dmma_tflops * 1e12
    t_s = g_ms * 1e-3
    t_compute, t_mem = flop / dmma if dmma == dmma else float("nan"), byt / hbm
    bound = "fp64 DMMA compute" if t_compute > t_mem else "HBM bandwidth"
    res = dict(
        workload=w.tag, gpu=gpu, rounds=args.rounds,
        ms_per_solve={k: dict(median=float(np.median(v)), min=float(np.min(v)), max=float(np.max(v)), all=v) for k, v in times.items()},
        check=check,
        stage_gemm=dict(launches=g_cnt, expected_launches=2 + (tableaus.DOPRI5.n_k - 1) * attempts, total_ms=g_ms,
                        avg_us=1e3 * g_ms / max(g_cnt, 1), flop=flop, algorithmic_bytes=byt,
                        achieved_tflops=flop / t_s * 1e-12, achieved_tbps=byt / t_s * 1e-12,
                        dmma_tflops_measured=args.dmma_tflops, hbm_tbps_measured=hbm * 1e-12,
                        time_at_dmma_rate_ms=t_compute * 1e3, time_at_hbm_rate_ms=t_mem * 1e3, bound=bound,
                        share_of_bound=max(t_compute, t_mem) / t_s),
        other_families_ms={"stage0": fam[_lib.FAM_STAGE0], "finalize": fam[_lib.FAM_FINALIZE], "emit": fam[_lib.FAM_EMIT]},
        attempts=attempts)
    with open(os.path.join(args.out, "linear_rhs_northstar.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
