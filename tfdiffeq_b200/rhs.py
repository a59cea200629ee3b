"""Built-in right-hand sides (SURVEY.md 8(f)-2).

Each class is an ordinary ``nn.Module`` -- ``forward(t, y)`` is written in plain torch ops and works anywhere
(on the generic path, on CPU, under autograd).  When an instance is handed to ``odeint`` with an adaptive
Runge-Kutta method and a single ``(..., k * dim)`` CUDA state, the solver recognises it and runs the WHOLE solve in
one persistent kernel (``b2ode_fused_solve``): every trajectory lives in one thread's registers, HBM traffic is
the solution slab only.  Batches that cannot stay co-resident (and tsit5, whose dense output needs all k's) take the
per-stage kernels with the right-hand side evaluated inside the stage kernel (``b2ode_rk_stage_rhs``): one launch per
stage, no ``forward`` call at all.  The kernel evaluates exactly the same IEEE operations in the same order as
``forward`` does, so both paths agree to the last bit per stage; ``options={'fused_rhs': False}`` forces the
generic path.
"""
import torch
import torch.nn as nn

from . import _lib


class BuiltinRHS(nn.Module):
    kind = None      # B2ODE_RHS_* code
    dim = None       # size of the last state axis
    persistent = True   # has a one-launch form (persistent adaptive kernel, fixed-grid kernel); else stage kernels only

    def rhs_params(self):
        raise NotImplementedError

    def rhs_data(self, dtype, device):
        """Device buffer of staged weights for the kernel (None for parameter-free systems)."""
        return None


class Lorenz(BuiltinRHS):
    """examples/lorenz_attractor.py:20-37, vectorised over leading batch axes: state (..., 3)."""
    kind, dim = _lib.RHS_LORENZ, 3

    def __init__(self, sigma=10.0, beta=8.0 / 3.0, rho=28.0):
        super(Lorenz, self).__init__()
        self.sigma, self.beta, self.rho = float(sigma), float(beta), float(rho)

    def rhs_params(self):
        return [self.sigma, self.beta, self.rho]

    def forward(self, t, y):
        x, yy, z = y[..., 0], y[..., 1], y[..., 2]
        return torch.stack([self.sigma * (yy - x), x * (self.rho - z) - yy, x * yy - self.beta * z], -1)


class LotkaVolterra(BuiltinRHS):
    """README.md:67-81: x' = a x - b x z, z' = -c z + d x z; state (..., 2)."""
    kind, dim = _lib.RHS_LOTKA_VOLTERRA, 2

    def __init__(self, a=1.5, b=1.0, c=3.0, d=1.0):
        super(LotkaVolterra, self).__init__()
        self.a, self.b, self.c, self.d = float(a), float(b), float(c), float(d)

    def rhs_params(self):
        return [self.a, self.b, self.c, self.d]

    def forward(self, t, y):
        x, z = y[..., 0], y[..., 1]
        return torch.stack([self.a * x - self.b * x * z, -self.c * z + self.d * x * z], -1)


class Kepler(BuiltinRHS):
    """DETEST class D (tests/DETEST/detest.py:263-283): two-body orbits, ``[x, y, vx, vy]`` per orbit, any number of orbits
    stacked along the last state axis (BASELINE config 5: 32 orbits = dim 128).  The kernels see the state as rows of 4."""
    kind, dim = _lib.RHS_KEPLER, 4

    def rhs_params(self):
        return []

    def forward(self, t, y):
        s = y.reshape(y.shape[:-1] + (y.shape[-1] // 4, 4))
        x, yy, vx, vy = s[..., 0], s[..., 1], s[..., 2], s[..., 3]
        r3 = (x * x + yy * yy) ** 1.5
        return torch.stack([vx, vy, -x / r3, -yy / r3], -1).reshape(y.shape)


class CubicMLP(BuiltinRHS):
    """examples/ode_demo.py:115-129 (BASELINE config 3): ``W2 . tanh(W1 . y**3 + b1) + b2`` with a 2 -> H -> 2
    network (H <= 128); ``cube=False`` drops the ``y**3``.  Weights are ordinary ``nn.Parameter`` s, so the module
    trains like any other (gradients come from the generic / adjoint path; the fused kernels are forward only).
    """
    kind, dim = _lib.RHS_CUBIC_MLP, 2

    def __init__(self, hidden=50, cube=True, std=0.1, dtype=torch.float32, generator=None):
        super(CubicMLP, self).__init__()
        if not 1 <= hidden <= 128:
            raise ValueError("hidden width must be in [1, 128]")
        self.hidden, self.cube = int(hidden), bool(cube)
        self.W1 = nn.Parameter(torch.randn(2, hidden, dtype=dtype, generator=generator) * std)
        self.b1 = nn.Parameter(torch.zeros(hidden, dtype=dtype))
        self.W2 = nn.Parameter(torch.randn(hidden, 2, dtype=dtype, generator=generator) * std)
        self.b2 = nn.Parameter(torch.zeros(2, dtype=dtype))

    def rhs_params(self):
        return [float(self.hidden), 1.0 if self.cube else 0.0]

    def rhs_data(self, dtype, device):
        with torch.no_grad():
            return torch.cat([self.W1.reshape(-1), self.b1.reshape(-1), self.W2.reshape(-1), self.b2.reshape(-1)]).to(
                device=device, dtype=dtype).contiguous()

    def forward(self, t, y):
        u = y ** 3 if self.cube else y
        return torch.tanh(u @ self.W1 + self.b1) @ self.W2 + self.b2


class LinearSystem(BuiltinRHS):
    """The linear system ``y' = y @ A (+ b)`` on a ``(..., D)`` state (the reference's ``LinearODE`` fixture,
    tests/problems.py:43-68, and the north-star ``BatchedLinear`` workload).  ``A`` (D x D) and ``b`` (D) are
    ``nn.Parameter`` s and ``forward`` is plain torch, so the module trains and runs anywhere.

    Note the side: unlike ``nn.Linear`` (``x @ W.T``) the state multiplies ``A`` from the LEFT, ``k[r, c] = sum_d
    y[r, d] A[d, c]`` -- as in ``BatchedLinear`` and ode_demo.py's ``y**3 @ A``.  A column-vector system ``x' = M x`` is
    ``LinearSystem(M.T)``.

    With an adaptive Runge-Kutta method on a CUDA state and ``D <= 128`` the solver runs every stage as ONE launch
    (``b2ode_rk_stage_rhs``): the stage combine forms the stage input tile by tile in shared memory and feeds it straight
    into an fp64 GEMM on the DMMA tensor cores with ``A`` resident in shared memory (fp32 states: fp32 FMAs), so the stage
    input never round-trips HBM and ``forward`` is never called.  There is no persistent one-kernel form (a row of up to 128
    values does not fit one thread's registers).  Fixed-grid and multistep methods, ``D > 128`` (with a warning) and
    ``options={'fused_rhs': False}`` call ``forward``."""
    kind = _lib.RHS_LINEAR
    persistent = False

    def __init__(self, A, b=None):
        super(LinearSystem, self).__init__()
        A = torch.as_tensor(A)
        if A.dim() != 2 or A.shape[0] != A.shape[1] or A.shape[0] < 1:
            raise ValueError("A must be a square (D, D) matrix")
        self.dim = int(A.shape[0])
        self.A = nn.Parameter(A.detach().clone())
        if b is not None:
            b = torch.as_tensor(b, dtype=A.dtype, device=A.device)
            if b.shape != (self.dim,):
                raise ValueError("b must have shape (D,)")
            self.b = nn.Parameter(b.detach().clone())
        else:
            self.b = None

    def rhs_params(self):
        return [float(self.dim), 0.0 if self.b is None else 1.0]

    def rhs_data(self, dtype, device):
        with torch.no_grad():
            parts = [self.A.reshape(-1)] + ([] if self.b is None else [self.b.reshape(-1)])
            return torch.cat([p.to(device=device, dtype=dtype) for p in parts]).contiguous()

    def forward(self, t, y):
        k = y @ self.A
        return k if self.b is None else k + self.b


_ACT = {None: 0, "none": 0, "relu": 1, "tanh": 2, "softplus": 3}

# numeric modes of the tensor-core func
#   "3xtf32" (default, also `True`): every product is split hi/lo and accumulated in fp32 -- as accurate as fp32 FMAs,
#            so solutions stay within north_star's 1e-3 fp32 bar of the reference's fp32 matmuls
#   "tf32"   (opt-in): single-pass TF32 (10-bit mantissa operands), the chained one-launch kernel; ~1e-3 relative error
#            per evaluation -- faster, but it does NOT meet the fp32 parity bar over a whole solve
#   False    : plain torch everywhere
_MODES = {True: "3xtf32", "3xtf32": "3xtf32", "tf32": "tf32", False: None, None: None}

# set by odeint_adjoint for the duration of its forward and backward solves: "tf32" is promoted to "3xtf32" so that the
# forward pass, the backward reconstruction of y (both under no_grad on the tensor cores) and the VJPs (autograd, fp32)
# integrate the same dynamics to fp32 rounding
_FORCE_ACCURATE = [0]


def _round_tf32(w):
    """Round-to-nearest (ties away from zero, what cvt.rna.tf32.f32 does) to TF32's 10 explicit mantissa bits."""
    i = w.contiguous().view(torch.int32)
    return ((i + 0x1000) & -0x2000).view(torch.float32)


class _WeightCache(object):
    """Derived images of a weight tensor (TF32-rounded copy, hi/lo split, packed shared-memory image), rebuilt when the
    weight changes.  Entries hold a weak reference to the weight they were built from and are only hit when that very
    object is still alive (`ref() is weight`) -- an `id()` recycled by a new tensor can never alias an old entry -- and
    are dropped when the weight is collected.  Validity is (data_ptr, _version, shape): in-place updates through
    autograd-visible ops (optimizer steps, `copy_`, `add_`) bump `_version`; writes through `.data` do NOT --
    call `invalidate(weight)` (or `DenseMLP.invalidate_tensor_core_cache()`) after those."""

    def __init__(self):
        self._d = {}

    @staticmethod
    def _key(ws):
        return tuple((w.data_ptr(), w._version, tuple(w.shape)) for w in ws)

    def get(self, tag, ws, build):
        ws = tuple(ws)
        slot = (tag,) + tuple(id(w) for w in ws)
        hit = self._d.get(slot)
        key = self._key(ws)
        if hit is not None and hit[0] == key and all(r() is w for r, w in zip(hit[1], ws)):
            return hit[2]
        import weakref
        d = self._d

        def _drop(_ref, slot=slot, d=d):
            d.pop(slot, None)
        with torch.no_grad():
            val = build(*[w.detach() for w in ws])
        d[slot] = (key, tuple(weakref.ref(w, _drop) for w in ws), val)
        return val

    def invalidate(self, weight=None):
        if weight is None:
            self._d.clear()
            return
        for slot in [s for s in self._d if id(weight) in s[1:]]:
            self._d.pop(slot, None)


_CACHE = _WeightCache()


def invalidate(weight=None):
    """Forget the cached tensor-core images of `weight` (all weights when None): needed after `.data` mutation."""
    _CACHE.invalidate(weight)


def _tf32_weight(weight):
    return _CACHE.get("tf32", (weight,), _round_tf32)


def _split_weight(weight):
    """(W_hi, W_lo) of the 3xTF32 split: W_hi = tf32(W), W_lo = tf32(W - W_hi) (the subtraction is exact in fp32)."""
    def build(w):
        hi = _round_tf32(w.reshape(w.shape[0], -1))
        lo = _round_tf32(w.reshape(w.shape[0], -1).contiguous() - hi)
        return hi, lo
    return _CACHE.get("x3", (weight,), build)


def _stage_args(stage):
    import ctypes as C
    if stage is None:
        return None, None, 0, None, None
    ks, coefs, state, ys = stage
    nk = len(ks)
    return (C.c_void_p * nk)(*[k.data_ptr() for k in ks]), (C.c_double * nk)(*coefs), nk, state, ys


def dense_layer(x, weight, bias, act="none", stage=None, mode="3xtf32"):
    """``act(x @ weight.T + bias)`` on the tcgen05 tensor cores, fp32 storage: ``b2ode_dense_layer_x3`` (mode "3xtf32",
    fp32-accurate products) or ``b2ode_dense_layer`` (mode "tf32").  ``weight`` is ``[N, K]`` (``nn.Linear.weight``; a 1x1
    convolution's ``[F, C, 1, 1]`` kernel is the same matrix) and ``x`` any contiguous tensor whose last axis is K.

    ``stage = (k_tensors, coefs, state_ptr, ystage_or_None)`` makes the Runge-Kutta stage combine the A-operand
    producer: A = x + sum_j (dt * coefs[j]) * k_tensors[j], dt read from the device state."""
    import ctypes as C
    K = x.shape[-1]
    M = x.numel() // K
    N = weight.shape[0]
    out = torch.empty(x.shape[:-1] + (N,), dtype=torch.float32, device=x.device)
    karr, carr, nk, state, ys = _stage_args(stage)

    def ptr(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None
    stream = C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)
    if mode == "3xtf32":
        hi, lo = _split_weight(weight)
        _lib.check(_lib.lib.b2ode_dense_layer_x3(ptr(x), karr, carr, nk, C.c_void_p(state) if state else None, ptr(ys),
                                                 ptr(hi), ptr(lo), ptr(bias), ptr(out), M, K, N, _ACT[act], stream))
    else:
        _lib.check(_lib.lib.b2ode_dense_layer(ptr(x), karr, carr, nk, C.c_void_p(state) if state else None, ptr(ys),
                                              ptr(_tf32_weight(weight)), ptr(bias), ptr(out), M, K, N, _ACT[act], stream))
    return out


def _mlp3_packed(fc1, fc2, fc3):
    """The three weights as ``b2ode_mlp3``'s shared-memory image, rebuilt only when a weight changes."""
    import ctypes as C

    def build(w1, w2, w3):
        H, D = w1.shape
        nbytes = _lib.lib.b2ode_mlp3_packed_bytes(D, H)
        if nbytes < 0:
            raise ValueError("mlp3 needs dim and hidden to be multiples of 16 in [16, 256]")
        packed = torch.empty(nbytes, dtype=torch.uint8, device=w1.device)
        cw = [w.contiguous() for w in (w1, w2, w3)]
        _lib.check(_lib.lib.b2ode_mlp3_pack(
            C.c_void_p(cw[0].data_ptr()), C.c_void_p(cw[1].data_ptr()), C.c_void_p(cw[2].data_ptr()), D, H,
            C.c_void_p(packed.data_ptr()), C.c_void_p(torch.cuda.current_stream(packed.device).cuda_stream)))
        return packed
    return _CACHE.get("mlp3", (fc1.weight, fc2.weight, fc3.weight), build)


def mlp3(x, fc1, fc2, fc3, act="relu", stage=None):
    """``fc3(act(fc2(act(fc1(x)))))`` in one launch (``b2ode_mlp3``, single-pass TF32): hidden activations never reach
    HBM.  ``stage`` as in :func:`dense_layer`."""
    import ctypes as C
    M, D = x.shape
    H = fc1.weight.shape[0]
    out = torch.empty((M, D), dtype=torch.float32, device=x.device)
    karr, carr, nk, state, ys = _stage_args(stage)

    def ptr(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None
    _lib.check(_lib.lib.b2ode_mlp3(
        ptr(x), karr, carr, nk, C.c_void_p(state) if state else None, ptr(ys),
        ptr(_mlp3_packed(fc1, fc2, fc3)), ptr(fc1.bias), ptr(fc2.bias), ptr(fc3.bias), ptr(out), M, D, H, _ACT[act],
        C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)))
    return out


class _TensorCoreFunc(nn.Module):
    """Shared mode handling of the GEMM-backed funcs."""

    def _mode(self):
        m = _MODES[self.tensor_cores]
        if m == "tf32" and _FORCE_ACCURATE[0]:
            m = "3xtf32"
        return m

    def invalidate_tensor_core_cache(self):
        for p in self.parameters():
            _CACHE.invalidate(p)


class DenseMLP(_TensorCoreFunc):
    """The reference's ``ODEFunc`` (tfdiffeq/models/dense_odenet.py:11-92, time-independent form): fc1 -> act ->
    fc2 -> act -> fc3 on a ``(batch, dim)`` state, counting ``nfe`` like the reference does (:78).

    Under ``torch.no_grad()`` on a CUDA fp32 state -- which is how ``odeint`` evaluates ``func`` -- the three layers
    run on the tcgen05 tensor cores, and the adaptive solvers feed the first layer straight from the stage combine (the
    stage input never round-trips HBM for the GEMM).  ``tensor_cores``: ``True`` / ``"3xtf32"`` (default) keeps fp32
    accuracy by splitting every operand into two TF32 halves (three tensor-core passes, fp32 accumulation), so the
    solution stays within the fp32 parity bar of the reference's fp32 matmuls; ``"tf32"`` opts into single-pass TF32
    and the chained one-launch kernel (faster, ~1e-3 relative error per evaluation); ``False`` is plain torch.  With
    autograd enabled (training, ``odeint_adjoint``'s VJPs) it is plain torch."""

    def __init__(self, dim, hidden, non_linearity="relu", tensor_cores=True, dtype=torch.float32, chain=True):
        super(DenseMLP, self).__init__()
        if non_linearity not in ("relu", "tanh", "softplus"):
            raise ValueError("non_linearity must be relu, tanh or softplus")
        if tensor_cores not in _MODES:
            raise ValueError("tensor_cores must be True, False, '3xtf32' or 'tf32'")
        self.dim, self.hidden, self.non_linearity, self.tensor_cores = int(dim), int(hidden), non_linearity, tensor_cores
        self.fc1 = nn.Linear(dim, hidden, dtype=dtype)
        self.fc2 = nn.Linear(hidden, hidden, dtype=dtype)
        self.fc3 = nn.Linear(hidden, dim, dtype=dtype)
        self.nfe = 0
        self.chain = chain

    def uses_tensor_cores(self, x):
        return (self._mode() is not None and x.is_cuda and x.dtype == torch.float32 and not torch.is_grad_enabled()
                and self.fc1.weight.dtype == torch.float32 and self.dim % 16 == 0 and self.hidden % 16 == 0
                and x.shape[-1] == self.dim)

    def chained(self):
        """One-launch form (``b2ode_mlp3``, single-pass TF32 only) when both widths fit the 128 KB activation tile."""
        return self._mode() == "tf32" and self.chain and self.dim <= 256 and self.hidden <= 256

    def _tail(self, h1):
        m = self._mode()
        h2 = dense_layer(h1, self.fc2.weight, self.fc2.bias, self.non_linearity, mode=m)
        return dense_layer(h2, self.fc3.weight, self.fc3.bias, "none", mode=m)

    def forward_from_stage(self, y0, ks, coefs, state_ptr, ystage):
        """First layer fed by the stage combine of y0 and the k's (all ``(batch, dim)`` fp32 CUDA tensors)."""
        self.nfe += 1
        if self.chained():
            return mlp3(y0, self.fc1, self.fc2, self.fc3, self.non_linearity, stage=(ks, coefs, state_ptr, ystage))
        h1 = dense_layer(y0, self.fc1.weight, self.fc1.bias, self.non_linearity, stage=(ks, coefs, state_ptr, ystage),
                         mode=self._mode())
        return self._tail(h1)

    def forward(self, t, x):
        self.nfe += 1
        if self.uses_tensor_cores(x):
            x2 = x.reshape(-1, self.dim)
            if not x2.is_contiguous():
                x2 = x2.contiguous()
            if self.chained():
                return mlp3(x2, self.fc1, self.fc2, self.fc3, self.non_linearity).reshape(x.shape)
            h1 = dense_layer(x2, self.fc1.weight, self.fc1.bias, self.non_linearity, mode=self._mode())
            return self._tail(h1).reshape(x.shape)
        act = {"relu": torch.relu, "tanh": torch.tanh, "softplus": torch.nn.functional.softplus}[self.non_linearity]
        return self.fc3(act(self.fc2(act(self.fc1(x)))))


class Conv2dODEFunc(_TensorCoreFunc):
    """The reference's ``Conv2dODEFunc`` (tfdiffeq/models/conv_odenet.py:45-143, BASELINE config 4): conv 1x1 -> act ->
    conv 3x3 'same' -> act -> conv 1x1 on an NHWC state ``(batch, height, width, channels)`` -- TensorFlow's default
    image layout, which is also what makes the 1x1 convolutions plain GEMMs over ``M = batch * height * width`` rows.

    Under ``torch.no_grad()`` on a CUDA fp32 state the two 1x1 convolutions run on the tcgen05 tensor cores through the
    same dense-layer kernel as :class:`DenseMLP` (``b2ode_dense_layer_x3`` / ``b2ode_dense_layer``), the first one fed
    straight from the Runge-Kutta stage combine; the 3x3 convolution stays on cuDNN (channels-last, no layout copies:
    the NHWC buffer *is* a channels-last NCHW tensor), with TF32 disabled in the accurate mode.  ``time_dependent=True``
    (conv_odenet.py:11-42: time appended as an extra input channel of every convolution) runs in plain torch.
    ``channels`` must be given up front (the reference builds conv3 lazily from the first input, :118-128)."""

    def __init__(self, num_filters, channels=None, time_dependent=False, non_linearity="relu", tensor_cores=True,
                 dtype=torch.float32):
        super(Conv2dODEFunc, self).__init__()
        if non_linearity not in ("relu", "tanh", "softplus"):
            raise ValueError("non_linearity must be relu, tanh or softplus")
        if tensor_cores not in _MODES:
            raise ValueError("tensor_cores must be True, False, '3xtf32' or 'tf32'")
        channels = num_filters if channels is None else channels
        self.num_filters, self.channels, self.time_dependent = int(num_filters), int(channels), bool(time_dependent)
        self.non_linearity, self.tensor_cores = non_linearity, tensor_cores
        extra = 1 if time_dependent else 0
        self.conv1 = nn.Conv2d(self.channels + extra, self.num_filters, 1, dtype=dtype)
        self.conv2 = nn.Conv2d(self.num_filters + extra, self.num_filters, 3, padding=1, dtype=dtype)
        self.conv3 = nn.Conv2d(self.num_filters + extra, self.channels, 1, dtype=dtype)
        self.nfe = 0

    def uses_tensor_cores(self, x):
        return (self._mode() is not None and not self.time_dependent and x.is_cuda and x.dtype == torch.float32
                and x.dim() == 4 and not torch.is_grad_enabled() and self.conv1.weight.dtype == torch.float32
                and self.channels % 16 == 0 and self.num_filters % 16 == 0 and x.shape[-1] == self.channels)

    def _act(self, v):
        return {"relu": torch.relu, "tanh": torch.tanh, "softplus": torch.nn.functional.softplus}[self.non_linearity](v)

    def _conv3x3(self, h):
        """h: NHWC contiguous -> NHWC contiguous; cuDNN channels-last, activation applied by the caller."""
        w = _CACHE.get("cl", (self.conv2.weight,), lambda w: w.contiguous(memory_format=torch.channels_last))
        with torch.backends.cudnn.flags(enabled=True, allow_tf32=(self._mode() == "tf32")):
            o = torch.nn.functional.conv2d(h.permute(0, 3, 1, 2), w, self.conv2.bias, padding=1)
        o = o.permute(0, 2, 3, 1)
        return o if o.is_contiguous() else o.contiguous()

    def _tail(self, h1):
        m = self._mode()
        h2 = self._act(self._conv3x3(h1))
        return dense_layer(h2, self.conv3.weight, self.conv3.bias, "none", mode=m)

    def forward_from_stage(self, y0, ks, coefs, state_ptr, ystage):
        self.nfe += 1
        h1 = dense_layer(y0, self.conv1.weight, self.conv1.bias, self.non_linearity, stage=(ks, coefs, state_ptr, ystage),
                         mode=self._mode())
        return self._tail(h1)

    def forward(self, t, x):
        self.nfe += 1
        if self.uses_tensor_cores(x):
            xc = x if x.is_contiguous() else x.contiguous()
            h1 = dense_layer(xc, self.conv1.weight, self.conv1.bias, self.non_linearity, mode=self._mode())
            return self._tail(h1)
        v = x.permute(0, 3, 1, 2)

        def tcat(u):
            if not self.time_dependent:
                return u
            tt = torch.ones_like(u[:, :1]) * t.to(u.dtype)                      # conv_odenet.py:30-40
            return torch.cat([tt, u], 1)
        out = self._act(self.conv1(tcat(v)))
        out = self._act(self.conv2(tcat(out)))
        out = self.conv3(tcat(out))
        return out.permute(0, 2, 3, 1)
