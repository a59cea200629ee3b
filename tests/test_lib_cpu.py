"""CPU (no GPU needed): the C-ABI library loads and exports every symbol include/b2ode.h declares, rejects
bad arguments with the documented codes, and the host-side logic (tableaus, input handling, segment layout)
matches the oracle / the reference's semantics.  No compute kernels are launched here."""
import ctypes as C
import os
import re
import warnings

import numpy as np
import pytest
import torch

import np_ref
import tfdiffeq_b200 as tfd
from tfdiffeq_b200 import _lib, misc, solvers, tableaus

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "b2ode.h")).read()
    declared = set(re.findall(r"\b(b2ode_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no prototypes found"
    raw = C.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(raw, name), "libb2ode.so does not export %s" % name
    assert declared == set(_lib.EXPORTS)
    assert _lib.lib.b2ode_version() == 1
    assert _lib.lib.b2ode_state_bytes() == 256 == C.sizeof(_lib.State)


def _desc(nseg=1, n=10, dtype=_lib.F64, tab=tableaus.DOPRI5):
    d = _lib.AdaptiveDesc()
    d.dtype, d.nseg, d.n_k = dtype, nseg, tab.n_k
    for i in range(min(nseg, _lib.MAXSEG)):
        d.seg_len[i] = n
    d.fsal = 1
    return d


def test_argument_validation_codes():
    lib = _lib.lib
    h = C.c_void_p()
    d = _desc()
    assert lib.b2ode_adaptive_create(C.byref(h), C.byref(d)) == 0
    assert lib.b2ode_workspace_bytes(C.byref(d)) >= 32
    # not bound yet -> ESTATE (-2); nothing touches the GPU
    assert lib.b2ode_rk_stage(h, 0, None) == -2
    assert b"not bound" in lib.b2ode_last_error()
    assert lib.b2ode_rk_finalize(h, None) == -2
    lib.b2ode_adaptive_destroy(h)
    bad = _desc()
    bad.dtype = 7
    assert lib.b2ode_adaptive_create(C.byref(h), C.byref(bad)) == -1
    bad = _desc(nseg=_lib.MAXSEG + 1)
    assert lib.b2ode_adaptive_create(C.byref(h), C.byref(bad)) == -1
    bad = _desc()
    bad.n_k = 99
    assert lib.b2ode_adaptive_create(C.byref(h), C.byref(bad)) == -1
    assert lib.b2ode_adaptive_create(None, C.byref(d)) == -1
    with pytest.raises(_lib.B2odeError):
        _lib.check(-1)


def test_grid_geometry_scales_with_sm_count():
    lib = _lib.lib
    small = _desc(n=100)
    big = _desc(n=65536 * 128)
    big.sm_count = 148
    assert lib.b2ode_workspace_bytes(C.byref(small)) == 32          # one block, one 32-byte partial
    assert lib.b2ode_workspace_bytes(C.byref(big)) == 148 * 8 * 32  # capped at 8 blocks per SM


@pytest.mark.parametrize("name", ["dopri5", "tsit5", "bosh3", "bosh3_textbook", "adaptive_heun", "dopri8"])
def test_product_tableaus_equal_oracle_tableaus(name):
    """The oracle's tableaus are pinned against the reference through the golden vectors; the product's
    independently written tables must be the same floats."""
    a, b = tableaus.TABLEAUS[name], np_ref.TABLEAUS[name]
    assert list(a.alpha) == list(b.alpha)
    assert [list(r) for r in a.beta] == [list(r) for r in b.beta]
    assert list(a.c_sol) == list(b.c_sol)
    assert list(a.c_error) == list(b.c_error)
    if b.c_mid is None:
        assert a.c_mid is None
    else:
        assert list(a.c_mid) == list(b.c_mid)
    assert (a.init_order, a.ctrl_order, bool(a.fsal)) == (b.init_order, b.ctrl_order, bool(b.fsal))


def test_tf_f64_rounds_python_floats_through_float32():
    assert misc._tf_f64(0.9) == 0.8999999761581421
    assert misc._tf_f64(0.2) == 0.20000000298023224
    assert misc._tf_f64(10.0) == 10.0
    assert misc._tf_f64(3) == 3.0


def test_check_inputs_semantics():
    f = lambda t, y: y                                             # noqa: E731
    y0 = torch.ones(3, dtype=torch.float64)
    tensor_input, func, y, t = misc._check_inputs(f, y0, torch.tensor([0., 1., 2.]))
    assert tensor_input and isinstance(y, tuple) and len(y) == 1
    assert func(torch.tensor(0.), y)[0] is y0
    # decreasing t -> negated time and negated derivative (misc.py:318-321)
    _, func, _, t = misc._check_inputs(f, y0, torch.tensor([2., 1., 0.]))
    assert t.tolist() == [-2., -1., 0.]
    assert torch.equal(func(torch.tensor(0.), (y0,))[0], -y0)
    # a length-1 t counts as decreasing (empty reduce_all)
    _, _, _, t = misc._check_inputs(f, y0, torch.tensor([3.]))
    assert t.tolist() == [-3.]
    with pytest.raises(TypeError):
        misc._check_inputs(f, torch.ones(2, dtype=torch.bool), torch.tensor([0., 1.]))
    with pytest.raises(AssertionError):
        misc._check_inputs(f, [y0], torch.tensor([0., 1.]))
    with pytest.raises(AssertionError):
        misc._assert_increasing(torch.tensor([0., 2., 1.]))


def test_api_errors_without_gpu():
    f = lambda t, y: y                                             # noqa: E731
    y0 = torch.ones(3, dtype=torch.float64)
    t = torch.tensor([0., 1.])
    with pytest.raises(ValueError):
        tfd.odeint(f, y0, t, options=dict(first_step=0.1))
    with pytest.raises(KeyError):
        tfd.odeint(f, y0, t, method="nope")
    for m in ("adams", "fixed_adams", "explicit_adams"):           # multistep solvers: same loud failure on CPU tensors
        with pytest.raises(RuntimeError, match="CUDA tensors only"):
            tfd.odeint(f, y0, t, method=m)
    # the product has no CPU path: CPU tensors fail loudly instead of silently falling back
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        tfd.odeint(f, y0, t, method="dopri5")
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        tfd.odeint(f, y0, t, method="rk4")
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        with pytest.raises(RuntimeError):
            tfd.odeint(f, y0, t, method="dopri5", options=dict(bogus=1))
    assert any("Dopri5Solver: Unexpected arguments {'bogus': 1}" in str(x.message) for x in w)
    with pytest.raises(ValueError):
        tfd.odeint_adjoint(f, y0, t)                               # func must be an nn.Module
    assert set(tfd.SOLVERS) == {"tsit5", "dopri5", "dopri8", "bosh3", "euler", "midpoint", "rk4", "huen", "heun",
                                "adaptive_heun", "adams", "fixed_adams", "explicit_adams"}      # tfdiffeq/odeint.py:11-25


def test_missing_library_fails_loudly(tmp_path):
    import subprocess
    import sys
    code = "import os; os.environ['B2ODE_LIB']=%r; import tfdiffeq_b200" % str(tmp_path / "nope.so")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode != 0 and "no CPU fallback" in r.stderr


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "tfdiffeq_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "np_ref" not in src and "import oracle" not in src and "from oracle" not in src, fn


def test_adams_weights_are_exact_and_match_the_oracle(golden_dir):
    """The product regenerates the Adams-Bashforth / Adams-Moulton tables (tfdiffeq/fixed_adams.py:7-160) from their
    definition; the oracle does so independently.  Both are compared entry by entry with the reference's literal tables,
    stored by oracle/make_golden.py in tests/golden/adams_tables.npz as decimal strings."""
    from fractions import Fraction
    from tfdiffeq_b200.multistep import adams_weights
    for k in range(1, 21):
        for implicit in (False, True):
            c, d = adams_weights(k, implicit)
            assert (c, d) == tuple(np_ref._adams_weights(k, 1 if implicit else 0))
            assert sum(Fraction(x, d) for x in c) == 1                 # consistency: a constant derivative integrates exactly
    assert adams_weights(4, False) == ([55, -59, 37, -9], 24)
    assert adams_weights(4, True) == ([9, 19, -5, 1], 24)
    assert adams_weights(5, True) == ([251, 646, -264, 106, -19], 720)
    g = np.load(os.path.join(golden_dir, "adams_tables.npz"))
    ints = lambda s: [int(x) for x in str(s).split(",")]                # noqa: E731
    for k in range(2, 21):
        assert adams_weights(k, False) == (ints(g["bashforth"][k]), int(g["divisor"][k]))
        assert adams_weights(k, True) == (ints(g["moulton"][k]), int(g["divisor"][k]))


def test_multistep_host_controller_matches_the_oracle():
    """tfdiffeq/misc.py:267-287 restated twice (product host code for the Adams solver, oracle): same numbers."""
    from tfdiffeq_b200.multistep import _optimal_step_size
    rng = np.random.default_rng(0)
    for _ in range(300):
        dt = float(10 ** rng.uniform(-6, 0))
        ratios = [float(10 ** rng.uniform(-8, 3)) for _ in range(int(rng.integers(1, 4)))]
        order = int(rng.integers(1, 13))
        got = _optimal_step_size(dt, ratios, 0.9, 10.0, 0.2, order)
        want = float(np_ref.optimal_step_size(dt, tuple(np.float64(r) for r in ratios), 0.9, 10.0, 0.2, order=order))
        assert got == want or abs(got - want) <= 4e-16 * abs(want), (dt, ratios, order, got, want)
    assert _optimal_step_size(0.1, [0.0, 0.0], 0.9, 10.0, 0.2, 3) == 1.0
    assert np.isnan(_optimal_step_size(0.1, [float("nan"), 0.5], 0.9, 10.0, 0.2, 3))
