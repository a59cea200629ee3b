"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/*.npz from the UNMODIFIED reference.

Run in the build container (needs /root/reference):   python oracle/make_golden.py
For every case of tests/cases.py the reference's own ``odeint`` (tfdiffeq/odeint.py:28, loaded over
oracle/tf_shim.py because TensorFlow is not installable here) is run on torch-CPU tensors, and the
solution (time axis subsampled by ``keep``), the accepted / rejected / NFE counts and the dt trace are
stored.  The fixtures travel to the GPU box; the reference does not.
The reference's literal Adams tables go to tests/golden/adams_tables.npz (``python oracle/make_golden.py adams_tables``
writes only those).
"""
import os
import signal
import sys
import time
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import ref_loader  # noqa: E402
from cases import CASES  # noqa: E402
from problems import PROBLEMS  # noqa: E402


CASE_TIMEOUT_S = 120


class CaseTimeout(Exception):
    pass


def _alarm(*a):
    raise CaseTimeout("reference did not finish in %d s" % CASE_TIMEOUT_S)


def keep_idx(T, keep):
    idx = list(range(0, T, keep))
    if idx[-1] != T - 1:
        idx.append(T - 1)
    return np.array(idx)


def run_case(c):
    tdt = {"float32": torch.float32, "float64": torch.float64}[c["dtype"]]
    prob = PROBLEMS[c["problem"]](backend="torch", dtype=c["dtype"], **c["pkw"])
    y0 = c["y0"]
    if isinstance(y0, tuple):
        y0_t = tuple(torch.tensor(np.asarray(v), dtype=tdt) for v in y0)
    else:
        y0_t = torch.tensor(np.asarray(y0), dtype=tdt)
    t_t = torch.from_numpy(np.ascontiguousarray(c["t"]))
    kw = dict(rtol=c["rtol"], atol=c["atol"])
    if c["method"] is not None:
        kw["method"] = c["method"]
    if c["options"] is not None:
        kw["options"] = c["options"]
    cnt = ref_loader.Counters()
    out = {"n_acc": -1, "n_rej": -1, "nfe": -1}
    err = ""
    warned = ""
    t0 = time.time()
    signal.signal(signal.SIGALRM, _alarm)
    signal.alarm(CASE_TIMEOUT_S)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        try:
            sol = ref_loader.run_reference(prob, y0_t, t_t, counters=cnt, **kw)
        except Exception as e:  # noqa: BLE001
            err = type(e).__name__ + ": " + str(e)[:200]
            sol = None
        finally:
            signal.alarm(0)
        for wi in w:
            if "Unexpected arguments" in str(wi.message):
                warned = str(wi.message)
    wall = time.time() - t0
    res = dict(t=c["t"], n_acc=cnt.n_acc, n_rej=cnt.n_rej, nfe=cnt.nfe, error=err, warned=warned,
               dt_trace=np.array(cnt.dt_trace[:4096], dtype=np.float64), wall=wall)
    if sol is not None:
        sols = sol if isinstance(sol, tuple) else (sol,)
        idx = keep_idx(len(c["t"]), c["keep"])
        res["idx"] = idx
        for i, s in enumerate(sols):
            res["sol%d" % i] = s.numpy()[idx]
        res["ncomp"] = len(sols)
    y0s = y0 if isinstance(y0, tuple) else (y0,)
    for i, v in enumerate(y0s):
        res["y0_%d" % i] = np.asarray(v)
    return res


def adams_tables():
    """The reference's literal Adams-Bashforth / Adams-Moulton tables and divisors (tfdiffeq/fixed_adams.py:8-145), one
    comma-separated row of decimal integers per order (index 0 is empty): the high orders do not fit in int64."""
    fa = ref_loader.load().fixed_adams
    row = lambda r: ",".join(str(int(x)) for x in r)                     # noqa: E731
    return dict(bashforth=np.array([row(r) for r in fa._BASHFORTH_COEFFICIENTS]),
                moulton=np.array([row(r) for r in fa._MOULTON_COEFFICIENTS]),
                divisor=np.array(["" if d is None else str(int(d)) for d in fa._DIVISOR]))


def main():
    outdir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(outdir, exist_ok=True)
    only = sys.argv[1:]
    if not only or "adams_tables" in only:
        np.savez_compressed(os.path.join(outdir, "adams_tables.npz"), **adams_tables())
    for c in CASES:
        if only and c["name"] not in only:
            continue
        res = run_case(c)
        np.savez_compressed(os.path.join(outdir, c["name"] + ".npz"), **res)
        print("%-28s acc %5d rej %5d nfe %6d  %6.2fs  %s%s" % (c["name"], res["n_acc"], res["n_rej"], res["nfe"],
                                                            res["wall"], res["error"][:60], res["warned"][:60]))


if __name__ == "__main__":
    main()
