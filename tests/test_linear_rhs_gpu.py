"""GPU: the linear built-in right-hand side (rhs.LinearSystem, B2ODE_RHS_LINEAR): k = s * (y @ A + b) evaluated inside the
stage kernels, the fp64 GEMM on the DMMA tensor cores.  Evaluation against torch, the stored stage input against the
plain stage kernel bit for bit, and whole solves against the cuBLAS func path, CUDA-graph replay, the numpy oracle and the
reference's golden vectors."""
import ctypes as C
import warnings

import numpy as np
import pytest
import torch

import np_ref
from golden_util import load_golden, max_rel_err
from problems import PROBLEMS
from tfdiffeq_b200 import _lib, tableaus

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def tfd():
    import tfdiffeq_b200
    return tfdiffeq_b200


def sm_count():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


def rhs_desc(A, b=None, sign=1.0):
    """(RhsDesc, staged data tensor): A row-major then b, in A's dtype."""
    rd = _lib.RhsDesc()
    rd.kind, rd.n_params = _lib.RHS_LINEAR, 2
    rd.params[0], rd.params[1] = float(A.shape[0]), 0.0 if b is None else 1.0
    data = torch.cat([A.reshape(-1)] + ([] if b is None else [b.reshape(-1)])).contiguous()
    rd.data = data.data_ptr()
    rd.time_sign = sign
    return rd, data


def rhs_eval(A, y, b=None, sign=1.0):
    rd, data = rhs_desc(A, b, sign)
    k = torch.empty_like(y)
    t = torch.zeros((), dtype=y.dtype, device=DEV)
    code = _lib.F64 if y.dtype == torch.float64 else _lib.F32
    _lib.check(_lib.lib.b2ode_rhs_eval(code, C.byref(rd), C.c_void_p(t.data_ptr()), C.c_void_p(y.data_ptr()),
                                       C.c_void_p(k.data_ptr()), y.numel(), sm_count(),
                                       C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)))
    torch.cuda.synchronize()
    del data
    return k


# ---- 1. evaluation -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [1, 3, 10, 16, 100, 128])
@pytest.mark.parametrize("rows", [1, 127, 129, 65537])
def test_eval_fp64_matches_torch(D, rows):
    g = torch.Generator(device=DEV).manual_seed(D * 1000 + rows)
    A = torch.randn(D, D, dtype=torch.float64, device=DEV, generator=g)
    b = torch.randn(D, dtype=torch.float64, device=DEV, generator=g)
    y = torch.randn(rows, D, dtype=torch.float64, device=DEV, generator=g)
    bound = 1e-13 * float(y.abs().max()) * float(A.abs().max()) * D
    for bias in (None, b):
        want = y @ A + (0 if bias is None else bias)
        got = rhs_eval(A, y, bias)
        assert float((got - want).abs().max()) <= bound, (D, rows, bias is not None)
    # deterministic: the same launch twice is bit-identical
    assert torch.equal(rhs_eval(A, y, b), rhs_eval(A, y, b))
    # reversed system: k = -(y @ A + b)
    assert torch.equal(rhs_eval(A, y, b, sign=-1.0), -rhs_eval(A, y, b))


@pytest.mark.parametrize("D", [1, 3, 10, 16, 100, 128])
@pytest.mark.parametrize("rows", [1, 127, 129, 65537])
def test_eval_fp32_matches_torch(D, rows):
    g = torch.Generator(device=DEV).manual_seed(D * 1000 + rows + 7)
    A = torch.randn(D, D, dtype=torch.float64, device=DEV, generator=g).float()
    b = torch.randn(D, dtype=torch.float64, device=DEV, generator=g).float()
    y = torch.randn(rows, D, dtype=torch.float64, device=DEV, generator=g).float()
    want = y.double() @ A.double() + b.double()
    got = rhs_eval(A, y, b).double()
    assert float((got - want).abs().max()) <= 1e-5 * float(want.abs().max()), (D, rows)


# ---- 2. the stored stage input is bit-identical to b2ode_rk_stage's -------------------------------------------------------
def _solver(y0, f0, ys, tstage, state, out, t_out, tab):
    d = _lib.AdaptiveDesc()
    d.dtype = _lib.F64 if y0.dtype == torch.float64 else _lib.F32
    d.nseg, d.n_k, d.fsal = 1, tab.n_k, 1 if tab.fsal else 0
    d.seg_len[0] = y0.numel()
    for i, row in enumerate(tab.beta):
        for j, v in enumerate(row):
            d.beta[i][j] = v
    for i, a in enumerate(tab.alpha):
        d.alpha[i] = a
    d.rtol[0], d.atol[0] = 1e-6, 1e-9
    d.safety, d.ifactor, d.dfactor, d.exponent = 0.9, 10.0, 0.2, 0.2
    d.max_num_steps, d.init_order, d.sm_count = 1000, 5, sm_count()
    h = C.c_void_p()
    _lib.check(_lib.lib.b2ode_adaptive_create(C.byref(h), C.byref(d)))
    ws = torch.zeros(max(int(_lib.lib.b2ode_workspace_bytes(C.byref(d))), 32), dtype=torch.uint8, device=DEV)
    _solver.keep = ws
    buf = _lib.AdaptiveBuffers()
    buf.state, buf.workspace, buf.workspace_bytes = state.data_ptr(), ws.data_ptr(), ws.numel()
    buf.y0[0], buf.f0[0], buf.ystage[0], buf.out[0] = y0.data_ptr(), f0.data_ptr(), ys.data_ptr(), out.data_ptr()
    buf.tstage, buf.t_out, buf.n_out = tstage.data_ptr(), t_out.data_ptr(), 2
    _lib.check(_lib.lib.b2ode_adaptive_bind(h, C.byref(buf), C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)))
    return h


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("tab", [tableaus.DOPRI5, tableaus.DOPRI8], ids=["dopri5", "dopri8"])
def test_last_stage_input_bit_identical_to_rk_stage(dtype, tab):
    rows, D = 1000, 100
    g = torch.Generator(device=DEV).manual_seed(11)
    mk = lambda: torch.randn(rows, D, dtype=torch.float64, device=DEV, generator=g).to(dtype)   # noqa: E731
    A = (0.1 * torch.randn(D, D, dtype=torch.float64, device=DEV, generator=g)).to(dtype)
    y0, f0 = mk(), mk()
    ks = [mk() for _ in range(tab.n_k - 1)]
    last = tab.n_k - 2
    res = []
    for fused in (True, False):
        ys = torch.zeros_like(y0)
        tstage = torch.zeros(tab.n_k, dtype=dtype, device=DEV)
        state = torch.zeros(256, dtype=torch.uint8, device=DEV)
        out = torch.zeros((2,) + y0.shape, dtype=dtype, device=DEV)
        t_out = torch.tensor([0.0, 1.0], dtype=torch.float64, device=DEV)
        h = _solver(y0, f0, ys, tstage, state, out, t_out, tab)
        try:
            _lib.check(_lib.lib.b2ode_adaptive_init(h, 0.0, 0.0123))
            P = C.c_void_p * _lib.MAXSEG
            for i in range(1, last):                      # register k_1 .. k_{last-1}
                _lib.check(_lib.lib.b2ode_set_k(h, i, P(ks[i - 1].data_ptr())))
            if fused:
                rd, data = rhs_desc(A)
                kout = torch.empty_like(y0)
                _lib.check(_lib.lib.b2ode_rk_stage_rhs(h, last, P(ks[last - 1].data_ptr()), C.byref(rd),
                                                       C.c_void_p(kout.data_ptr())))
                torch.cuda.synchronize()
                res.append((ys.clone(), kout))
            else:
                _lib.check(_lib.lib.b2ode_rk_stage(h, last, P(ks[last - 1].data_ptr())))
                torch.cuda.synchronize()
                res.append((ys.clone(), None))
        finally:
            torch.cuda.synchronize()
            _lib.lib.b2ode_adaptive_destroy(h)
    assert torch.equal(res[0][0], res[1][0])
    want = res[1][0].double() @ A.double()
    tol = 1e-12 if dtype == torch.float64 else 1e-5
    assert float((res[0][1].double() - want).abs().max()) <= tol * float(want.abs().max())


# ---- 3. three paths agree -------------------------------------------------------------------------------------------------
METHODS = [("dopri5", {}), ("dopri8", dict(rtol=1e-9, atol=1e-9)), ("bosh3", dict(rtol=1e-5, atol=1e-7)),
           ("tsit5", dict(rtol=1e-4, atol=1e-6)), ("adaptive_heun", dict(rtol=1e-4, atol=1e-6))]


def _batched(rows, D, seed=0):
    A = torch.as_tensor(PROBLEMS["batched_linear"](backend="numpy", dim=D, seed=seed).A)
    y0 = torch.tensor(np.random.default_rng(100).standard_normal((rows, D)), device=DEV)
    return A, y0


def _counts(s):
    return s["n_accepted"], s["n_rejected"], s["nfe"]


@pytest.mark.parametrize("method,kw", METHODS, ids=[m for m, _ in METHODS])
@pytest.mark.parametrize("D", [128, 10, 100])
def test_three_paths_agree(method, kw, D):
    A, y0 = _batched(2048, D)
    f = tfd().rhs.LinearSystem(A).to(DEV)
    t = torch.tensor(np.linspace(0., 2., 11)[:4])
    kw = dict(dict(rtol=1e-6, atol=1e-9), **kw)
    with warnings.catch_warnings():
        warnings.simplefilter("error", RuntimeWarning)   # no "co-resident" warning: the linear kind never tries the persistent kernel
        a = tfd().odeint(f, y0, t, method=method, **kw)
    sa = dict(tfd().last_stats)
    assert sa["stage_rhs"] and not sa["fused_rhs"]
    a2 = tfd().odeint(f, y0, t, method=method, options={"fused_rhs": "stages"}, **kw)
    assert torch.equal(a, a2) and tfd().last_stats["stage_rhs"]
    b = tfd().odeint(f, y0, t, method=method, options={"fused_rhs": False}, **kw)
    sb = dict(tfd().last_stats)
    assert not sb["stage_rhs"]
    c = tfd().odeint(f, y0, t, method=method, options={"cuda_graph": True}, **kw)
    sc = dict(tfd().last_stats)
    assert sc["stage_rhs"]
    assert _counts(sa) == _counts(sb) == _counts(sc)
    assert max_rel_err(a.cpu().numpy(), b.cpu().numpy()) <= 1e-10
    assert torch.equal(a, c)                        # graph replay of the same launches: bit-identical
    assert torch.equal(a, tfd().odeint(f, y0, t, method=method, **kw))    # run to run: bit-identical


# ---- 4. oracle and golden vectors -----------------------------------------------------------------------------------------
def test_batched_linear_vs_oracle():
    A, y0 = _batched(2048, 128)
    t = np.linspace(0., 2., 11)[:3]
    st = np_ref.Stats()
    ref = np_ref.odeint(PROBLEMS["batched_linear"](backend="numpy", dim=128, seed=0), y0.cpu().numpy(), t,
                        method="dopri5", rtol=1e-6, atol=1e-9, stats=st)
    sol = tfd().odeint(tfd().rhs.LinearSystem(A).to(DEV), y0, torch.tensor(t), method="dopri5", rtol=1e-6, atol=1e-9)
    s = tfd().last_stats
    assert s["stage_rhs"]
    assert (s["n_accepted"], s["n_rejected"]) == (st.n_acc, st.n_rej)
    assert max_rel_err(sol.cpu().numpy(), ref) <= 1e-6


@pytest.mark.parametrize("name,method,kw", [("linear_skew_dopri5", "dopri5", {}),
                                            ("linear_skew_dopri8", "dopri8", dict(rtol=1e-10, atol=1e-12))])
def test_golden_linear_skew(name, method, kw):
    """The reference's LinearODE (x' = A x on a (10,) state) is LinearSystem(A.T)."""
    g = load_golden(name)
    A = torch.as_tensor(PROBLEMS["linear"](backend="numpy", degenerate=False).A_np)
    f = tfd().rhs.LinearSystem(A.T.contiguous()).to(DEV)
    y0 = torch.tensor(g["y0_0"], device=DEV)
    t = torch.from_numpy(np.ascontiguousarray(g["t"]))
    sol = tfd().odeint(f, y0, t, method=method, **kw)
    s = tfd().last_stats
    assert s["stage_rhs"]
    assert max_rel_err(sol.cpu().numpy()[g["idx"]], g["sol0"]) <= 1e-6
    counts, want = (s["n_accepted"], s["n_rejected"], s["nfe"]), (g["n_acc"], g["n_rej"], g["nfe"])
    if kw.get("rtol", 1e-7) >= 1e-9:
        assert counts == want
    else:
        # the bar of tests/test_parity_gpu.py: at rtol <= 1e-10 the error estimate is rounding noise and the GEMM's
        # summation order is not the reference's, so a borderline accept may flip
        assert abs(counts[0] - want[0]) <= 2 and abs(counts[1] - want[1]) <= 2


# ---- 5. reverse time and bias ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_reverse_time_and_bias_match_func_path(dtype):
    A, y0 = _batched(3000, 64, seed=5)
    bvec = torch.linspace(-1., 1., 64, dtype=torch.float64)
    f = tfd().rhs.LinearSystem(A.to(dtype), bvec.to(dtype)).to(DEV)
    y0 = y0.to(dtype)
    kw = dict(rtol=1e-7, atol=1e-9) if dtype == torch.float64 else dict(rtol=1e-4, atol=1e-6)
    for t in (torch.tensor([2.0, 1.5, 1.0, 0.0], dtype=torch.float64), torch.tensor([0.0, 0.5, 1.0], dtype=torch.float64)):
        a = tfd().odeint(f, y0, t, method="dopri5", **kw)
        sa = dict(tfd().last_stats)
        assert sa["stage_rhs"]
        b = tfd().odeint(f, y0, t, method="dopri5", options={"fused_rhs": False}, **kw)
        sb = dict(tfd().last_stats)
        assert _counts(sa) == _counts(sb)
        tol = 1e-10 if dtype == torch.float64 else 1e-4
        assert max_rel_err(a.double().cpu().numpy(), b.double().cpu().numpy()) <= tol


# ---- 6. full size --------------------------------------------------------------------------------------------------------
def test_northstar_full_size_matches_func_path():
    A, _ = _batched(1, 128)
    y0 = torch.tensor(np.random.default_rng(100).standard_normal((65536, 128)), device=DEV)   # bench.py's NorthStar y0
    t = torch.tensor(np.linspace(0., 2., 11))
    f = tfd().rhs.LinearSystem(A).to(DEV)
    a = tfd().odeint(f, y0, t, method="dopri5", rtol=1e-6, atol=1e-9)
    sa = dict(tfd().last_stats)
    b = tfd().odeint(f, y0, t, method="dopri5", rtol=1e-6, atol=1e-9, options={"fused_rhs": False})
    sb = dict(tfd().last_stats)
    assert sa["stage_rhs"] and not sb["stage_rhs"]
    assert _counts(sa) == _counts(sb)
    assert max_rel_err(a.cpu().numpy(), b.cpu().numpy()) <= 1e-10


# ---- 7. fallbacks --------------------------------------------------------------------------------------------------------
def test_dim_above_128_warns_and_calls_forward():
    A, y0 = _batched(500, 129, seed=2)
    f = tfd().rhs.LinearSystem(0.1 * A).to(DEV)
    t = torch.tensor([0.0, 0.5, 1.0])
    with pytest.warns(RuntimeWarning, match="128"):
        a = tfd().odeint(f, y0, t, method="dopri5")
    sa = dict(tfd().last_stats)
    assert not sa["stage_rhs"]
    b = tfd().odeint(f, y0, t, method="dopri5", options={"fused_rhs": False})
    assert _counts(sa) == _counts(tfd().last_stats)
    assert torch.equal(a, b)


def test_fixed_grid_and_adams_call_forward():
    A, y0 = _batched(700, 32, seed=3)
    f = tfd().rhs.LinearSystem(A).to(DEV)
    t = torch.tensor(np.linspace(0., 1., 21))
    a = tfd().odeint(f, y0, t, method="rk4")
    assert not tfd().last_stats["fused_rhs"]
    b = tfd().odeint(f, y0, t, method="rk4", options={"fused_rhs": False})
    assert torch.equal(a, b)
    c = tfd().odeint(f, y0, t, method="adams", rtol=1e-6, atol=1e-8)
    d = tfd().odeint(lambda tt, yy: yy @ f.A, y0, t, method="adams", rtol=1e-6, atol=1e-8)
    assert torch.equal(c, d)
