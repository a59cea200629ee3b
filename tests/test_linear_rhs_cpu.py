"""CPU (no GPU needed): the linear built-in right-hand side B2ODE_RHS_LINEAR (rhs.LinearSystem).

The C entry points reject bad linear descriptions with B2ODE_EINVAL before they touch the GPU, the module's forward is
``y @ A + b``, and the built library's fp64 stage kernels run their GEMM on the DMMA tensor cores without spilling to
local memory."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

import tfdiffeq_b200 as tfd
from tfdiffeq_b200 import _lib, tableaus

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(os.path.dirname(HERE), "tfdiffeq_b200", "libb2ode.so")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
EINVAL = -1
FAKE = 0x10000      # a 16-byte aligned address that the rejected calls never dereference


def _rd(D=4.0, has_bias=0.0, data=FAKE, n_params=2):
    rd = _lib.RhsDesc()
    rd.kind, rd.n_params = _lib.RHS_LINEAR, n_params
    rd.params[0], rd.params[1] = D, has_bias
    rd.data = data
    rd.time_sign = 1.0
    return rd


def _eval(rd, n, dtype=_lib.F64):
    return _lib.lib.b2ode_rhs_eval(dtype, C.byref(rd), C.c_void_p(FAKE), C.c_void_p(FAKE), C.c_void_p(FAKE), n, 148, None)


@pytest.mark.parametrize("rd,n,why", [
    (_rd(D=0.0), 8, "D < 1"),
    (_rd(D=129.0), 129, "D > 128"),
    (_rd(D=2.5), 10, "D not an integer"),
    (_rd(n_params=0), 8, "no D"),
    (_rd(data=None), 8, "no matrix"),
    (_rd(D=4.0), 10, "length not a multiple of D"),
    (_rd(D=3.0, has_bias=1.0), 7, "length not a multiple of D, with bias"),
])
def test_rhs_eval_rejects_bad_linear_description(rd, n, why):
    assert _eval(rd, n) == EINVAL, why
    assert _eval(rd, n, _lib.F32) == EINVAL, why


def _bound_solver(n, dtype=_lib.F64):
    """A solver bound to fake device addresses: binding is host-side bookkeeping, nothing is launched."""
    d = _lib.AdaptiveDesc()
    t = tableaus.DOPRI5
    d.dtype, d.nseg, d.n_k, d.fsal = dtype, 1, t.n_k, 1
    d.seg_len[0] = n
    d.sm_count = 148
    h = C.c_void_p()
    _lib.check(_lib.lib.b2ode_adaptive_create(C.byref(h), C.byref(d)))
    buf = _lib.AdaptiveBuffers()
    buf.state = buf.workspace = buf.tstage = buf.t_out = FAKE
    buf.workspace_bytes = 1 << 30
    buf.n_out = 2
    buf.y0[0] = buf.f0[0] = buf.ystage[0] = buf.out[0] = FAKE
    _lib.check(_lib.lib.b2ode_adaptive_bind(h, C.byref(buf), None))
    return h


@pytest.mark.parametrize("rd,n,why", [
    (_rd(D=0.0), 8, "D < 1"),
    (_rd(D=129.0), 129, "D > 128"),
    (_rd(data=None), 8, "no matrix"),
    (_rd(D=4.0), 10, "length not a multiple of D"),
])
def test_rk_stage_rhs_rejects_bad_linear_description(rd, n, why):
    h = _bound_solver(n)
    try:
        k = (C.c_void_p * _lib.MAXSEG)(FAKE)
        assert _lib.lib.b2ode_rk_stage_rhs(h, 1, k, C.byref(rd), C.c_void_p(FAKE)) == EINVAL, why
    finally:
        _lib.lib.b2ode_adaptive_destroy(h)


def test_no_persistent_or_fixed_grid_kernel_for_the_linear_kind():
    lib = _lib.lib
    d = _lib.AdaptiveDesc()
    d.dtype, d.nseg, d.n_k, d.fsal = _lib.F64, 1, 7, 1
    d.seg_len[0] = 128 * 1024
    assert lib.b2ode_fused_capacity(C.byref(d), _lib.RHS_LINEAR) == 0
    d.dtype = _lib.F32
    assert lib.b2ode_fused_capacity(C.byref(d), _lib.RHS_LINEAR) == 0
    prm = (C.c_double * 8)(4.0, 0.0)
    for method in range(4):
        rc = lib.b2ode_fused_fixed_solve(_lib.F64, method, _lib.RHS_LINEAR, prm, 2, C.c_void_p(FAKE), 1.0, C.c_void_p(FAKE),
                                         C.c_void_p(FAKE), 16, 0, 1, None, None, None, None, None, None, 148, None)
        assert rc == EINVAL
    fd = _lib.FusedDesc()
    fd.rhs_kind, fd.n_rhs_params = _lib.RHS_LINEAR, 2
    fd.rhs_params[0] = 4.0
    fd.rhs_data = fd.y0 = fd.out = fd.t_out = fd.state = fd.workspace = FAKE
    fd.n_out, fd.workspace_bytes = 2, 1 << 30
    d.dtype = _lib.F64
    assert lib.b2ode_fused_solve(C.byref(d), C.byref(fd)) == EINVAL


@pytest.mark.parametrize("bias", [False, True])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_linear_system_forward_on_cpu(bias, dtype):
    g = torch.Generator().manual_seed(0)
    A = torch.randn(7, 7, generator=g, dtype=dtype)
    b = torch.randn(7, generator=g, dtype=dtype) if bias else None
    f = tfd.rhs.LinearSystem(A, b)
    assert f.dim == 7 and f.kind == _lib.RHS_LINEAR and not f.persistent
    assert isinstance(f.A, torch.nn.Parameter) and (f.b is None) == (not bias)
    assert f.rhs_params() == [7.0, 1.0 if bias else 0.0]
    y = torch.randn(5, 3, 7, generator=g, dtype=dtype)
    want = y @ A + (b if bias else 0)
    assert torch.equal(f(0.0, y), want)
    data = f.rhs_data(torch.float64, "cpu")
    assert data.dtype == torch.float64 and data.numel() == 49 + (7 if bias else 0)
    assert torch.equal(data[:49], A.double().reshape(-1))
    # it trains: gradients reach A and b
    f(0.0, y).sum().backward()
    assert f.A.grad is not None and (not bias or f.b.grad is not None)


def test_linear_system_rejects_bad_shapes():
    with pytest.raises(ValueError):
        tfd.rhs.LinearSystem(torch.zeros(3, 4))
    with pytest.raises(ValueError):
        tfd.rhs.LinearSystem(torch.zeros(3, 3), torch.zeros(4))


# ---- SASS of the built library ---------------------------------------------------------------------------------------
FP64_KERNELS = ["_Z17k_rk_stage_linearIdLi%dEEv9LinParamsIXT0_EE" % nk for nk in range(14)]
FP32_KERNELS = ["_Z17k_rk_stage_linearIfLi%dEEv9LinParamsIXT0_EE" % nk for nk in range(14)]


def _sass(kernel):
    out = subprocess.run([CUOBJDUMP, "-sass", "-fun", kernel, LIB], capture_output=True, text=True, timeout=300).stdout
    return [m.group(1).strip() for m in re.finditer(r"/\*[0-9a-f]{4,}\*/\s+([^;]*);", out)]


@pytest.mark.skipif(not (os.path.exists(LIB) and os.path.exists(CUOBJDUMP)), reason="needs the built library and cuobjdump")
@pytest.mark.parametrize("kernel", FP64_KERNELS + FP32_KERNELS)
def test_linear_stage_kernel_sass(kernel):
    ins = _sass(kernel)
    assert ins, "kernel not found in the library: " + kernel
    ops = [t.split()[0] if not t.startswith("@") else t.split()[1] for t in ins]
    spills = [t for t, o in zip(ins, ops) if o.startswith("LDL") or o.startswith("STL")]
    assert not spills, "local-memory traffic (spills) in %s: %s" % (kernel, spills[:4])
    if "IdLi" in kernel:
        assert any(o.startswith("DMMA") for o in ops), "the fp64 GEMM is not on the DMMA tensor cores"
