"""Host drivers: the reference's solver protocol (``__init__(func, y0, rtol=, atol=, **options)`` +
``integrate(t)``, tfdiffeq/odeint.py:77-78) on top of ``libb2ode``.

What stays in Python is what the reference keeps in Python: calling the user's ``func`` and sequencing the
stages.  Everything numeric is a kernel launch through the C ABI; the step size, the accept/reject decision
and the output cursor never leave the device, so the loop below enqueues whole attempts without reading
anything back, polling a 256-byte state asynchronously through pinned memory.
"""
import collections
import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from . import tableaus as tb
from .misc import _assert_increasing, _handle_unused_kwargs, _is_iterable, _tf_f64

_ITEM = {torch.float32: 4, torch.float64: 8}
_DT = {torch.float32: _lib.F32, torch.float64: _lib.F64}

# statistics of the most recent solve (the reference exposes none; `nfe` mirrors its model-side counters)
last_stats = {}


def _require_cuda(y0):
    dev = y0[0].device
    if dev.type != "cuda":
        raise RuntimeError(
            "tfdiffeq_b200 runs on CUDA tensors only (got device %s); there is no CPU code path." % dev)
    dt = y0[0].dtype
    if dt not in _ITEM:
        raise TypeError("state dtype must be float32 or float64, got %s" % dt)
    for y in y0:
        if y.device != dev or y.dtype != dt:
            raise TypeError("all state components must share one device and dtype")
    if len(y0) > _lib.MAXSEG:
        raise ValueError("at most %d state components are supported" % _lib.MAXSEG)
    return dev, dt


_PINNED_STATE = {}
_PINNED_BUSY = set()


def _pinned_acquire(dev, nbytes=256):
    """A reusable page-locked landing buffer for device-state polls, one per device and size (page-locking a fresh
    buffer costs more than launching the whole fused solve).  Returns (buffer, key); hand the key back to
    `_pinned_release`.  A nested solve on the same device (func calling odeint) gets a private buffer."""
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), int(nbytes))
    if key in _PINNED_BUSY:
        return torch.empty(int(nbytes), dtype=torch.uint8).pin_memory(), None
    buf = _PINNED_STATE.get(key)
    if buf is None:
        buf = _PINNED_STATE[key] = torch.empty(int(nbytes), dtype=torch.uint8).pin_memory()
    _PINNED_BUSY.add(key)
    return buf, key


_COPY_STREAMS = {}


def _copy_stream(dev):
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    st = _COPY_STREAMS.get(key)
    if st is None:
        st = _COPY_STREAMS[key] = torch.cuda.Stream(dev)
    return st


def _pinned_release(key):
    if key is not None:
        _PINNED_BUSY.discard(key)


class _Segments(object):
    """Engine-owned flat buffers: one allocation per role, tuple components at 16-byte aligned offsets."""

    def __init__(self, y0):
        self.device, self.dtype = _require_cuda(y0)
        self.item = _ITEM[self.dtype]
        self.shapes = [tuple(y.shape) for y in y0]
        self.lens = [int(y.numel()) for y in y0]
        al = 16 // self.item
        self.offs, off = [], 0
        for n in self.lens:
            self.offs.append(off)
            off += (n + al - 1) // al * al
        self.total = max(off, al)
        self.nseg = len(y0)

    def new(self):
        return torch.empty(self.total, dtype=self.dtype, device=self.device)

    def views(self, flat):
        return tuple(flat[o:o + n].view(s) for o, n, s in zip(self.offs, self.lens, self.shapes))

    def ptrs(self, flat):
        base = flat.data_ptr()
        return [base + o * self.item for o in self.offs]

    def fill(self, flat, tensors):
        for v, t in zip(self.views(flat), tensors):
            v.copy_(t)


def _ptr_array(ptrs):
    arr = _lib.PtrArray()
    for i, p in enumerate(ptrs):
        arr[i] = p
    return arr


class _FuncOutputs(object):
    """Normalises what ``func`` returns into per-segment contiguous tensors the kernels can read in place."""

    def __init__(self, seg, engine_flats):
        self.seg = seg
        self.ranges = [(f.data_ptr(), f.data_ptr() + f.numel() * seg.item) for f in engine_flats]
        self.arr = _lib.PtrArray()
        self.always_clone = False     # set once func is seen handing back the same storage twice
        self.alias_events = 0
        self._last = []               # outputs of the previous call, kept referenced so that pointer equality
                                      # with a new output can only mean shared storage, never allocator reuse

    def collect(self, outs, live):
        seg = self.seg
        if isinstance(outs, torch.Tensor):
            outs = (outs,)
        if len(outs) != seg.nseg:
            raise ValueError("func returned %d tensors for a state of %d components" % (len(outs), seg.nseg))
        res = []
        for s, o in enumerate(outs):
            if not isinstance(o, torch.Tensor):
                o = torch.as_tensor(o, dtype=seg.dtype, device=seg.device)
            if o.dtype != seg.dtype or o.device != seg.device:
                o = o.to(device=seg.device, dtype=seg.dtype)
            if o.numel() != seg.lens[s]:
                o = o.expand(seg.shapes[s])
            if not o.is_contiguous():
                o = o.contiguous()
            p = o.data_ptr()
            nbytes = seg.lens[s] * seg.item
            if nbytes:
                # a func that hands back the storage of its previous result (a preallocated output buffer) will
                # overwrite earlier k's: from the second call on, every result gets its own storage
                if not self.always_clone and (p in live or any(p == q.data_ptr() for q in self._last)):
                    self.always_clone = True
                    self.alias_events += 1
                # a func that returns (a view of) its input would be overwritten by the next stage
                if self.always_clone or any(p < hi and p + nbytes > lo for lo, hi in self.ranges):
                    o = o.clone()
                    p = o.data_ptr()
            live.add(p)
            res.append(o)
        self._last = res
        return res

    def pointers(self, tensors):
        for i, t in enumerate(tensors):
            self.arr[i] = t.data_ptr()
        return self.arr


class AdaptiveStepsizeODESolver(object):
    """Adaptive explicit Runge-Kutta driver (tfdiffeq/solvers.py:10-35 + the solver classes that follow it,
    e.g. tfdiffeq/dopri5.py:48-121), generic over the tableau."""

    tableau = None
    RUN_AHEAD = 8          # attempts the host may be ahead of the last state it has seen

    def __init__(self, func, y0, rtol, atol, first_step=None, safety=0.9, ifactor=10.0, dfactor=0.2,
                 max_num_steps=2 ** 31 - 1, **unused_kwargs):
        self.comm = unused_kwargs.pop("shared_step_group", None)     # extension: SURVEY 8(e)
        # with a group: tuple components every rank holds in full, bit-identical (odeint_adjoint's batch-summed adjoints)
        self.replicated = tuple(unused_kwargs.pop("replicated_components", ()))
        # extension: capture one attempt (the func calls included) into a CUDA graph and replay it.  Opt-in,
        # because python-side effects of func (e.g. an `nfe` counter on the module) happen once, at capture.
        self.cuda_graph = bool(unused_kwargs.pop("cuda_graph", False))
        # extension: a built-in right-hand side (tfdiffeq_b200/rhs.py) runs in one persistent kernel unless disabled
        # (True: persistent kernel when the batch fits, else the stage kernels with the right-hand side fused in; 'stages':
        # always the latter; False: call func like any other callable).  rhs.LinearSystem has no persistent kernel:
        # True and 'stages' both take its stage kernels
        fr = unused_kwargs.pop("fused_rhs", True)
        self.fused_rhs = fr if fr == "stages" else bool(fr)
        # extension: a page-locked host tensor of the solution's shape.  The solution is delivered THERE (and returned as
        # that tensor); with a built-in right-hand side the device-to-host copies are issued behind the running solve
        self.host_output = unused_kwargs.pop("host_output", None)
        _handle_unused_kwargs(self, unused_kwargs)
        del unused_kwargs
        self.func = func
        self.y0 = y0
        if self.tableau.controller == "tsit5":
            # tsit5.py:81-82 keeps scalars; iterables break its arithmetic
            self.rtol = [rtol] * len(y0)
            self.atol = [atol] * len(y0)
        else:
            self.rtol = list(rtol) if _is_iterable(rtol) else [rtol] * len(y0)
            self.atol = list(atol) if _is_iterable(atol) else [atol] * len(y0)
        self.first_step = first_step
        self.safety = _tf_f64(safety)
        self.ifactor = _tf_f64(ifactor)
        self.dfactor = _tf_f64(dfactor)
        self.max_num_steps = int(max_num_steps)
        self.stats = {}

    # -- construction of the native solver ---------------------------------------------------------
    def _describe(self, seg):
        t = self.tableau
        d = _lib.AdaptiveDesc()
        d.dtype = _DT[seg.dtype]
        d.nseg = seg.nseg
        for i, n in enumerate(seg.lens):
            d.seg_len[i] = n
        d.n_k = t.n_k
        d.fsal = 1 if t.fsal else 0
        for i, a in enumerate(t.alpha):
            d.alpha[i] = a
        for i, row in enumerate(t.beta):
            for j, v in enumerate(row):
                d.beta[i][j] = v
        for j in range(t.n_k):
            d.c_sol[j] = t.c_sol[j]
            d.c_error[j] = t.c_error[j]
            d.c_mid[j] = t.c_mid[j] if t.c_mid is not None else 0.0
        d.dense_kind = 0 if t.c_mid is not None else 1
        d.controller = _lib.CTRL_TSIT5 if t.controller == "tsit5" else _lib.CTRL_REFERENCE
        for i in range(seg.nseg):
            d.rtol[i] = float(self.rtol[i])
            d.atol[i] = float(self.atol[i])
        d.safety, d.ifactor, d.dfactor = self.safety, self.ifactor, self.dfactor
        if t.controller == "tsit5":
            d.exponent = 1.0 / t.ctrl_order                               # tsit5.py:59: exact float64
        else:
            d.exponent = float(np.float64(np.float32(1.0 / t.ctrl_order)))   # misc.py:281-282: via float32
        d.max_num_steps = min(self.max_num_steps, 2 ** 62)
        d.init_order = t.init_order
        d.sm_count = torch.cuda.get_device_properties(seg.device).multi_processor_count
        return d

    def integrate(self, t):
        _assert_increasing(t)
        seg = _Segments(self.y0)
        dev, dtype = seg.device, seg.dtype
        with torch.cuda.device(dev), torch.no_grad():
            fused = self._integrate_fused(t, seg, dev, dtype) if self.fused_rhs is True else None
            if fused is not None:
                return fused
            res = self._integrate(t, seg, dev, dtype)
            if self.host_output is not None:
                ho = self._check_host_output(res)
                for h, r in zip(ho, res):
                    h.copy_(r, non_blocking=True)
                torch.cuda.current_stream(dev).synchronize()
                return tuple(ho)
            return res

    def _check_host_output(self, outs):
        ho = self.host_output
        ho = (ho,) if isinstance(ho, torch.Tensor) else tuple(ho)
        if len(ho) != len(outs):
            raise ValueError("host_output must hold one tensor per state component")
        for h, o in zip(ho, outs):
            if h.device.type != "cpu" or not h.is_pinned() or h.shape != o.shape or h.dtype != o.dtype or not h.is_contiguous():
                raise ValueError("host_output must be page-locked, contiguous CPU tensors of the solution's shape and dtype")
        return ho

    def _integrate_fused(self, t, seg, dev, dtype):
        """Whole solve in one persistent kernel when func is a built-in right-hand side (rhs.py)."""
        from .rhs import BuiltinRHS
        base = getattr(self.func, "_b2ode_base", None)
        tab = self.tableau
        if (not isinstance(base, BuiltinRHS) or not base.persistent or seg.nseg != 1 or tab.c_mid is None
                or tab.n_k not in (2, 4, 7, 14)):
            return None
        shape = seg.shapes[0]
        if len(shape) < 1 or shape[-1] % base.dim != 0 or seg.lens[0] == 0:
            return None
        lib, check = _lib.lib, _lib.check
        n_traj = seg.lens[0] // base.dim
        t_host = t.detach().to("cpu", torch.float64).numpy()
        t_dev = torch.from_numpy(t_host).to(dev)
        n_out = int(t_host.shape[0])
        y0 = self.y0[0].contiguous()
        out = torch.empty((n_out,) + shape, dtype=dtype, device=dev)
        state_dev = torch.zeros(256, dtype=torch.uint8, device=dev)
        ws_bytes = int(lib.b2ode_fused_workspace_bytes(n_traj))
        workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        desc = self._describe(seg)
        prm = base.rhs_params()
        weights = base.rhs_data(dtype, dev)
        first = float("nan") if self.first_step is None else _tf_f64(self.first_step)
        fits = int(lib.b2ode_fused_capacity(C.byref(desc), base.kind)) >= n_traj
        fd = _lib.FusedDesc()
        fd.rank, fd.nranks = 0, 1
        if self.comm is not None:
            # the shards of a group must take the same path (the fused kernel and the generic kernels speak different
            # exchange protocols) and every rank derives every other rank's kernel grid from its shard size: agree on
            # "every shard fits" and learn all shard sizes in one cached collective
            sizes, fits = self.comm.agree_fused(n_traj, fits)
            fd.rank, fd.nranks = self.comm.rank, self.comm.world
            fd.mailboxes = C.cast(self.comm._ptrs, C.c_void_p)
            for r, n_r in enumerate(sizes):
                fd.n_traj_rank[r] = n_r
        if not fits:
            import warnings
            warnings.warn("tfdiffeq_b200: batch of %d trajectories per GPU exceeds what the persistent fused kernel can keep "
                          "co-resident; using the per-stage kernels with the right-hand side fused into them (one launch "
                          "per stage instead of one per solve)" % n_traj, RuntimeWarning)
            return None
        stream = torch.cuda.current_stream(dev)
        fd.rhs_kind, fd.n_rhs_params = base.kind, len(prm)
        for k_, v_ in enumerate(prm):
            fd.rhs_params[k_] = v_
        fd.rhs_data = weights.data_ptr() if weights is not None else None
        fd.time_sign = float(self.func._b2ode_sign)
        fd.y0, fd.out, fd.t_out, fd.n_out = y0.data_ptr(), out.data_ptr(), t_dev.data_ptr(), n_out
        fd.t_start, fd.first_step = float(t_host[0]), first
        fd.state, fd.workspace, fd.workspace_bytes = state_dev.data_ptr(), workspace.data_ptr(), ws_bytes
        fd.cuda_stream = stream.cuda_stream
        host_out = mark = mkey = None
        if self.host_output is not None:
            host_out = self._check_host_output((out,))[0]
            mark, mkey = _pinned_acquire(dev, 64)
            mark = mark[:4].view(torch.int32)
            mark.zero_()
            fd.host_mark = mark.data_ptr()      # page-locked memory is device-addressable at its host address (UVA)
        rc = lib.b2ode_fused_solve(C.byref(desc), C.byref(fd))
        check(rc)
        if host_out is not None:
            # stream the slab out behind the solve: the kernel keeps `mark` at the number of leading rows that are complete
            done = torch.cuda.Event()
            done.record(stream)
            cs = _copy_stream(dev)
            out.record_stream(cs)
            mark_np = mark.numpy()
            copied, chunk = 0, max(8, n_out // 64)
            while copied < n_out:
                fin = done.query()
                m = n_out if fin else min(int(mark_np[0]), n_out)
                if m - copied >= chunk or (fin and m > copied):
                    if fin:
                        cs.wait_event(done)
                    with torch.cuda.stream(cs):
                        host_out[copied:m].copy_(out[copied:m], non_blocking=True)
                    copied = m
        host, hkey = _pinned_acquire(dev)
        try:
            host.copy_(state_dev, non_blocking=True)
            stream.synchronize()
            final = _lib.State.from_buffer_copy(host.numpy().tobytes())
        finally:
            _pinned_release(hkey)
        if host_out is not None:
            cs.synchronize()
            _pinned_release(mkey)
            out = host_out
        attempts = int(final.n_acc + final.n_rej)
        nfe = 1 + (1 if self.first_step is None else 0) + (tab.n_k - 1) * attempts
        self.stats = dict(n_accepted=int(final.n_acc), n_rejected=int(final.n_rej), nfe=nfe, attempts_enqueued=attempts,
                          status=int(final.status), cuda_graph=False, fused_rhs=True)
        last_stats.clear()
        last_stats.update(self.stats)
        if final.status:
            self._raise(final, (out[0],), (y0,))
        return (out,)

    def _integrate(self, t, seg, dev, dtype):
        lib, check = _lib.lib, _lib.check
        tab = self.tableau
        nk = tab.n_k
        t_host = t.detach().to("cpu", torch.float64).numpy()                 # solvers.py:30: time is float64
        t_dev = torch.from_numpy(t_host).to(dev)
        n_out = int(t_host.shape[0])
        t_end = float(t_host[-1])

        Y0, F0, S = seg.new(), seg.new(), seg.new()
        outs = [torch.empty((n_out,) + shp, dtype=dtype, device=dev) for shp in seg.shapes]
        tstage = torch.zeros(nk, dtype=dtype, device=dev)
        state_dev = torch.zeros(256, dtype=torch.uint8, device=dev)
        desc = self._describe(seg)
        ws_bytes = int(lib.b2ode_workspace_bytes(C.byref(desc)))
        workspace = torch.empty(max(ws_bytes, 32), dtype=torch.uint8, device=dev)

        handle = C.c_void_p()
        check(lib.b2ode_adaptive_create(C.byref(handle), C.byref(desc)))
        stream = torch.cuda.current_stream(dev)
        try:
            buf = _lib.AdaptiveBuffers()
            buf.state = state_dev.data_ptr()
            buf.workspace = workspace.data_ptr()
            buf.workspace_bytes = workspace.numel()
            for i, (a, b, c) in enumerate(zip(seg.ptrs(Y0), seg.ptrs(F0), seg.ptrs(S))):
                buf.y0[i], buf.f0[i], buf.ystage[i] = a, b, c
                buf.out[i] = outs[i].data_ptr()
            buf.tstage = tstage.data_ptr()
            buf.t_out = t_dev.data_ptr()
            buf.n_out = n_out
            check(lib.b2ode_adaptive_bind(handle, C.byref(buf), C.c_void_p(stream.cuda_stream)))
            if self.comm is not None:
                self.comm.attach(handle, seg, self.replicated)

            fo = _FuncOutputs(seg, (Y0, F0, S))
            y0_views, s_views = seg.views(Y0), seg.views(S)
            nfe = 0

            # built-in right-hand side on the per-stage path: it is evaluated INSIDE the stage kernels
            # (b2ode_rk_stage_rhs / b2ode_rhs_eval), func's forward is never called; the k's live in engine buffers
            from .rhs import BuiltinRHS
            brhs = getattr(self.func, "_b2ode_base", None)
            if not (self.fused_rhs and isinstance(brhs, BuiltinRHS) and seg.nseg == 1 and len(seg.shapes[0]) >= 1
                    and seg.shapes[0][-1] % brhs.dim == 0 and seg.lens[0] > 0):
                brhs = None
            elif brhs.kind == _lib.RHS_LINEAR and (seg.shapes[0][-1] != brhs.dim or brhs.dim > _lib.LINEAR_MAX_DIM):
                if brhs.dim > _lib.LINEAR_MAX_DIM:
                    import warnings
                    warnings.warn("tfdiffeq_b200: LinearSystem of dimension %d exceeds the stage kernel's limit of %d (A must "
                                  "fit in shared memory); calling its forward" % (brhs.dim, _lib.LINEAR_MAX_DIM), RuntimeWarning)
                brhs = None
            if brhs is not None:
                rd = _lib.RhsDesc()
                prm = brhs.rhs_params()
                rd.kind, rd.n_params = brhs.kind, len(prm)
                for k_, v_ in enumerate(prm):
                    rd.params[k_] = v_
                rhs_weights = brhs.rhs_data(dtype, dev)
                rd.data = rhs_weights.data_ptr() if rhs_weights is not None else None
                rd.time_sign = float(getattr(self.func, "_b2ode_sign", 1.0))
                Kb = [seg.new() for _ in range(nk - 1)]
                Kp = [_ptr_array(seg.ptrs(kb)) for kb in Kb]
                dcode, n_el, sm_ = _DT[dtype], seg.lens[0], desc.sm_count

                def rhs_eval(t_ptr, y_flat, k_flat):
                    # on torch's CURRENT stream: inside a CUDA-graph capture that is the capture stream
                    check(lib.b2ode_rhs_eval(dcode, C.byref(rd), C.c_void_p(t_ptr), C.c_void_p(y_flat.data_ptr()),
                                             C.c_void_p(k_flat.data_ptr()), n_el, sm_,
                                             C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))

            # ---- before_integrate (dopri5.py:70-78) ----------------------------------------------
            seg.fill(Y0, self.y0)
            t0_state = t_dev[0].to(dtype)                                    # tf.cast(t[0], y0.dtype)
            if brhs is not None:
                rhs_eval(t0_state.data_ptr(), Y0, F0)
            else:
                f0 = fo.collect(self.func(t0_state, y0_views), set())
                seg.fill(F0, f0)
            nfe += 1
            if self.first_step is None:
                check(lib.b2ode_adaptive_init(handle, float(t_host[0]), float("nan")))
                check(lib.b2ode_initial_step_probe(handle))
                if brhs is not None:
                    rhs_eval(tstage.data_ptr(), S, Kb[0])
                    check(lib.b2ode_initial_step_finish(handle, Kp[0]))
                else:
                    f1 = fo.collect(self.func(tstage[0], s_views), set())
                    check(lib.b2ode_initial_step_finish(handle, fo.pointers(f1)))
                    del f1
                nfe += 1
            else:
                check(lib.b2ode_adaptive_init(handle, float(t_host[0]), _tf_f64(self.first_step)))
            if tab.controller == "tsit5":
                # tsit5.py:92-98: _select_initial_step computes its own f0 and the state f0 is evaluated
                # again (with the float64 t[0]); one redundant evaluation, kept so NFE matches
                if self.first_step is None:
                    if brhs is None:
                        self.func(t_dev[0], y0_views)
                    nfe += 1

            # ---- pinned ring for asynchronous state polls --------------------------------------------
            D = self.RUN_AHEAD
            pinned = torch.empty(256 * (D + 1), dtype=torch.uint8).pin_memory()
            slots = [_lib.State.from_address(pinned.data_ptr() + 256 * i) for i in range(D + 1)]
            events = [torch.cuda.Event() for _ in range(D + 1)]
            check(lib.b2ode_poll_sync(handle, C.c_void_p(pinned.data_ptr() + 256 * D)))
            known = _lib.State.from_buffer_copy(slots[D])     # snapshots: the ring slots get overwritten
            known_at = 0
            n_enq = 0
            pending = collections.deque()
            g = self.ifactor

            tstage_views = [tstage[i] for i in range(nk - 1)]
            func = self.func
            rk_stage, rk_finalize, poll_async = lib.b2ode_rk_stage, lib.b2ode_rk_finalize, lib.b2ode_poll_async

            # tensor-core func (rhs.DenseMLP): the stage combine becomes the A-operand producer of its first layer
            from .rhs import Conv2dODEFunc, DenseMLP
            dense = getattr(self.func, "_b2ode_base", None)
            if not (self.fused_rhs and seg.nseg == 1 and tab.fsal and getattr(self.func, "_b2ode_sign", 1.0) > 0
                    and ((isinstance(dense, DenseMLP) and len(seg.shapes[0]) == 2)
                         or (isinstance(dense, Conv2dODEFunc) and len(seg.shapes[0]) == 4))
                    and dense.uses_tensor_cores(s_views[0])):
                dense = None
            if dense is not None:
                f0_view = seg.views(F0)[0]
                rows = [[(j, b) for j, b in enumerate(tab.beta[i]) if b != 0.0] for i in range(nk - 1)]
                state_ptr = state_dev.data_ptr()

            def run_attempt():
                """Enqueue one attempt: stage i -> func -> ... -> finalize (+ dense output).  No kernel argument
                depends on dt / accept / the output cursor: they live in the device state."""
                if brhs is not None:
                    item_ = seg.item
                    check(rk_stage(handle, 0, None))
                    rhs_eval(tstage.data_ptr(), S, Kb[0])
                    for i in range(1, nk - 1):
                        check(lib.b2ode_rk_stage_rhs(handle, i, Kp[i - 1], C.byref(rd), C.c_void_p(Kb[i].data_ptr())))
                    if not tab.fsal:
                        check(rk_stage(handle, nk - 1, Kp[nk - 2]))
                    check(rk_finalize(handle, Kp[nk - 2]))
                    return Kb
                live = set()
                ks = []           # every k of the attempt stays referenced until its last reader is enqueued
                check(rk_stage(handle, 0, None))
                k = fo.collect(func(tstage_views[0], s_views), live)
                ks.append(k)
                for i in range(1, nk - 1):
                    if dense is not None and rows[i]:
                        # no stage kernel: y_i is formed inside the first GEMM's producer; only the last stage
                        # input (= y1, read by finalize / the dense output / the next commit) is also stored
                        check(lib.b2ode_set_k(handle, i, fo.pointers(k)))
                        kt = [f0_view if j == 0 else ks[j - 1][0] for j, _ in rows[i]]
                        out = dense.forward_from_stage(y0_views[0], kt, [b for _, b in rows[i]], state_ptr,
                                                       s_views[0] if i == nk - 2 else None)
                        k = fo.collect((out,), live)
                        ks.append(k)
                        continue
                    check(rk_stage(handle, i, fo.pointers(k)))
                    k = fo.collect(func(tstage_views[i], s_views), live)
                    ks.append(k)
                if not tab.fsal:
                    check(rk_stage(handle, nk - 1, fo.pointers(k)))
                check(rk_finalize(handle, fo.pointers(k)))
                return ks

            graph = None          # torch.cuda.CUDAGraph of one attempt (cuda_graph=True), captured after attempt 1
            graph_ks = None
            prev_last = None      # k_{s-1}: read once more by the next attempt's stage 0 (the commit)
            while not known.done:
                ahead = n_enq - known_at
                go = ahead == 0
                if not go and ahead < D:
                    # every attempt advances t1 by at most dt and grows dt by at most `ifactor`: if even that
                    # cannot reach the last output time, the next attempt is certainly needed -> no sync
                    reach = known.dt * (ahead if g == 1.0 else (g ** ahead - 1.0) / (g - 1.0))
                    go = (known.t1 + reach) < t_end and known.status == 0
                if go:
                    if graph is not None:
                        graph.replay()
                    elif self.cuda_graph and n_enq >= 1:
                        # attempt 1 ran eagerly (warm-up); capture attempt 2 and replay it from now on
                        # (capture_begin/capture_end directly: torch.cuda.graph() would also run gc.collect() and
                        # empty the allocator cache on entry, tens of milliseconds per solve)
                        graph = torch.cuda.CUDAGraph()
                        cap = torch.cuda.Stream(dev)
                        cap.wait_stream(stream)
                        try:
                            with torch.cuda.stream(cap):
                                check(lib.b2ode_set_stream(handle, C.c_void_p(cap.cuda_stream)))
                                graph.capture_begin()
                                try:
                                    graph_ks = run_attempt()
                                finally:
                                    graph.capture_end()
                        finally:
                            check(lib.b2ode_set_stream(handle, C.c_void_p(stream.cuda_stream)))
                        stream.wait_stream(cap)
                        graph.replay()
                    else:
                        prev_last = run_attempt()[-1]
                    nfe += nk - 1
                    slot = n_enq % D
                    n_enq += 1
                    check(poll_async(handle, C.c_void_p(pinned.data_ptr() + 256 * slot)))
                    events[slot].record(stream)
                    pending.append((n_enq, slot))
                    while pending and events[pending[0][1]].query():
                        known_at, slot = pending.popleft()
                        known = _lib.State.from_buffer_copy(slots[slot])
                else:
                    known_at, slot = pending.popleft()
                    events[slot].synchronize()
                    known = _lib.State.from_buffer_copy(slots[slot])
            final = known
            self.stats = dict(n_accepted=int(final.n_acc), n_rejected=int(final.n_rej), nfe=nfe,
                              attempts_enqueued=n_enq, status=int(final.status), cuda_graph=graph is not None,
                              fused_rhs=False, stage_rhs=brhs is not None)
            last_stats.clear()
            last_stats.update(self.stats)
            if final.status:
                self._raise(final, s_views, y0_views)
            del prev_last, graph_ks, graph
        finally:
            # also on the error paths (status != 0 seen early, func raising mid-attempt): attempts and raw
            # cudaMemcpyAsync polls into `pinned` may still be in flight -- drain them before the pinned ring, the
            # engine buffers and the native handle are released
            stream.synchronize()
            lib.b2ode_adaptive_destroy(handle)
        return tuple(outs)

    def _raise(self, st, s_views, y0_views):
        """Re-raise the device status word with the reference's assertion messages."""
        if st.status & _lib.ST_NONFINITE:
            raise AssertionError('non-finite values in state `y`: {}'.format(y0_views[0]))   # dopri5.py:100
        if st.status & _lib.ST_MAXSTEPS:
            raise AssertionError('max_num_steps exceeded ({}>={})'.format(                  # dopri5.py:85
                int(st.n_steps_adv), self.max_num_steps))
        if st.status & _lib.ST_UNDERFLOW:
            raise AssertionError('underflow in dt {}'.format(st.dt))                         # dopri5.py:98
        raise AssertionError('solver status {}'.format(st.status))


class Dopri5Solver(AdaptiveStepsizeODESolver):
    """tfdiffeq/dopri5.py:48 (the ``tableau=`` option of :53 is honoured)"""
    tableau = tb.DOPRI5

    def __init__(self, func, y0, rtol, atol, tableau=None, **kw):
        if tableau is not None:
            self.tableau = tableau
        super(Dopri5Solver, self).__init__(func, y0, rtol, atol, **kw)


class Dopri8Solver(AdaptiveStepsizeODESolver):
    """tfdiffeq/dopri8.py:100"""
    tableau = tb.DOPRI8


class Bosh3Solver(AdaptiveStepsizeODESolver):
    """tfdiffeq/bosh3.py:33; ``options={'textbook_tableau': True}`` selects the tableau the reference meant."""
    tableau = tb.BOSH3

    def __init__(self, func, y0, rtol, atol, textbook_tableau=False, **kw):
        if textbook_tableau:
            self.tableau = tb.BOSH3_TEXTBOOK
        super(Bosh3Solver, self).__init__(func, y0, rtol, atol, **kw)


class AdaptiveHeunSolver(AdaptiveStepsizeODESolver):
    """tfdiffeq/adaptive_huen.py:47"""
    tableau = tb.ADAPTIVE_HEUN


class Tsit5Solver(AdaptiveStepsizeODESolver):
    """tfdiffeq/tsit5.py:69 (pooled error, sqrt-free controller, k-based dense output as written)"""
    tableau = tb.TSIT5


# ----------------------------------------------------------------------------------------------------
# fixed grid
# ----------------------------------------------------------------------------------------------------
class FixedGridODESolver(object):
    """tfdiffeq/solvers.py:38-115"""

    method = None
    order = None

    def __init__(self, func, y0, step_size=None, grid_constructor=None, eps=0.0, **unused_kwargs):
        unused_kwargs.pop('rtol', None)
        unused_kwargs.pop('atol', None)
        unused_kwargs.pop('shared_step_group', None)     # a fixed grid needs no exchange between shards
        unused_kwargs.pop('replicated_components', None)
        unused_kwargs.pop('cuda_graph', None)
        self.fused_rhs = bool(unused_kwargs.pop("fused_rhs", True))
        self.host_output = unused_kwargs.pop("host_output", None)
        _handle_unused_kwargs(self, unused_kwargs)
        del unused_kwargs
        self.func = func
        self.y0 = y0
        self.eps = eps
        # tfdiffeq/solvers.py:49-56 raises "exclusive arguments" whenever a grid_constructor is given at all (its
        # last `else`), which makes the option unusable; the evident intent (both given -> error) is implemented
        if step_size is not None and grid_constructor is not None:
            raise ValueError("step_size and grid_constructor are exclusive arguments.")
        if step_size is not None:
            self.grid_constructor = self._grid_constructor_from_step_size(step_size)
        elif grid_constructor is None:
            self.grid_constructor = lambda f, y0, t: t
        else:
            self.grid_constructor = grid_constructor
        self.stats = {}

    @staticmethod
    def _grid_constructor_from_step_size(step_size):
        # tfdiffeq/solvers.py:58-71 cannot run under TF2 (`tf.ceil`, item assignment); this is its evident
        # intent: a uniform grid from t[0] whose last point is clamped to t[-1]  (SURVEY App. A-9)
        def _grid_constructor(func, y0, t):
            start_time, end_time = t[0], t[-1]
            niters = int(math.ceil(float((end_time - start_time) / step_size + 1)))
            t_infer = torch.arange(0, niters, dtype=t.dtype, device=t.device) * step_size + start_time
            if t_infer[-1] > t[-1]:
                t_infer[-1] = t[-1]
            return t_infer
        return _grid_constructor

    # stage recipes: (time offset as a function of (t0, dt) in the state dtype, kernel op, operand indices)
    def integrate(self, t):
        _assert_increasing(t)
        seg = _Segments(self.y0)
        with torch.cuda.device(seg.device), torch.no_grad():
            res = self._integrate(t, seg)
            if self.host_output is not None:
                ho = AdaptiveStepsizeODESolver._check_host_output(self, res)
                for h, r in zip(ho, res):
                    h.copy_(r, non_blocking=True)
                torch.cuda.current_stream(seg.device).synchronize()
                return tuple(ho)
            return res

    def _integrate(self, t, seg):
        lib, check = _lib.lib, _lib.check
        dev, dtype = seg.device, seg.dtype
        npdt = np.float32 if dtype == torch.float32 else np.float64
        t = t.to(dtype)                                                        # solvers.py:84
        time_grid = self.grid_constructor(self.func, self.y0, t)
        t_np = t.detach().cpu().numpy().astype(npdt)
        g_np = time_grid.detach().cpu().numpy().astype(npdt)
        assert g_np[0] == t_np[0] and g_np[-1] == t_np[-1]                     # solvers.py:86
        n_out, n_steps = int(t_np.shape[0]), int(g_np.shape[0]) - 1
        outs = [torch.empty((n_out,) + shp, dtype=dtype, device=dev) for shp in seg.shapes]
        for o, y in zip(outs, self.y0):
            o[0].copy_(y)
        stream = torch.cuda.current_stream(dev)
        sm = torch.cuda.get_device_properties(dev).multi_processor_count
        dcode = _DT[dtype]
        lens = _lib.LenArray(*seg.lens)
        nseg = seg.nseg
        item = seg.item
        sptr = C.c_void_p(stream.cuda_stream)

        # stage times for every step, computed on the host in the state dtype with the reference's operation
        # order, uploaded once; func receives 0-dim device views
        eps = npdt(self.eps)
        t0s, dts = g_np[:-1], g_np[1:] - g_np[:-1]
        m = self.method
        if m == "euler":
            times = np.stack([t0s + eps], 1)                                   # fixed_grid.py:7
        elif m == "midpoint":
            times = np.stack([t0s + eps, t0s + dts / npdt(2)], 1)              # fixed_grid.py:17-18
        elif m == "heun":
            times = np.stack([t0s + eps, t0s + dts], 1)                        # fixed_grid.py:29-31
        else:
            te = t0s + eps                                                     # fixed_grid.py:42
            times = np.stack([te, te + dts / npdt(3), te + dts * npdt(2) / npdt(3), te + dts], 1)  # rk_common.py:76-79
        times_dev = torch.from_numpy(np.ascontiguousarray(times.astype(npdt))).to(dev)

        # ---- built-in right-hand side: the whole grid in one launch (b2ode_fused_fixed_solve) -----------------------
        from .rhs import BuiltinRHS
        base = getattr(self.func, "_b2ode_base", None)
        if (self.fused_rhs and isinstance(base, BuiltinRHS) and base.persistent and seg.nseg == 1
                and len(seg.shapes[0]) >= 1 and seg.shapes[0][-1] % base.dim == 0 and seg.lens[0] > 0):
            n_traj = seg.lens[0] // base.dim
            j0 = np.zeros(n_steps + 1, dtype=np.int32)
            ends = np.zeros(max(n_steps, 1), dtype=np.uint8)
            s2 = np.zeros(n_out, dtype=npdt)
            j = 1
            for i in range(n_steps):
                j0[i] = j
                while j < n_out and g_np[i + 1] >= t_np[j]:          # solvers.py:97
                    s2[j] = npdt(t_np[j]) - npdt(g_np[i])
                    j += 1
                ends[i] = 1 if (j > j0[i] and t_np[j - 1] == g_np[i + 1]) else 0
            j0[n_steps] = j
            times4 = np.zeros((max(n_steps, 1), 4), dtype=npdt)
            times4[:n_steps, :times.shape[1]] = times
            up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)                                  # noqa: E731
            times_d, dts_d, j0_d, ends_d, s1_d, s2_d = up(times4), up(dts.astype(npdt)), up(j0), up(ends), up(dts.astype(npdt)), up(s2)
            prm = base.rhs_params()
            prm_arr = (C.c_double * 8)(*(prm + [0.0] * (8 - len(prm))))
            weights = base.rhs_data(dtype, dev)
            y0c = self.y0[0].contiguous()
            mcode = {"euler": 0, "midpoint": 1, "heun": 2, "rk4": 3}[m]
            check(lib.b2ode_fused_fixed_solve(dcode, mcode, base.kind, prm_arr, len(prm),
                                              C.c_void_p(weights.data_ptr()) if weights is not None else None,
                                              float(self.func._b2ode_sign), C.c_void_p(y0c.data_ptr()),
                                              C.c_void_p(outs[0].data_ptr()), n_traj, n_steps, n_out,
                                              C.c_void_p(times_d.data_ptr()), C.c_void_p(dts_d.data_ptr()),
                                              C.c_void_p(j0_d.data_ptr()), C.c_void_p(ends_d.data_ptr()),
                                              C.c_void_p(s1_d.data_ptr()), C.c_void_p(s2_d.data_ptr()), sm, sptr))
            per_step = {"euler": 1, "midpoint": 2, "heun": 2, "rk4": 4}[m]
            self.stats = dict(n_accepted=n_steps, n_rejected=0, nfe=per_step * n_steps, status=0, fused_rhs=True)
            last_stats.clear()
            last_stats.update(self.stats)
            stream.synchronize()
            return tuple(outs)

        # two scratch states: the stage input, and y1 for grid cells whose end is not an output time
        S, Y1a, Y1b = seg.new(), seg.new(), seg.new()
        fo = _FuncOutputs(seg, (S, Y1a, Y1b) + tuple(outs))
        s_views, s_ptrs = seg.views(S), _ptr_array(seg.ptrs(S))
        scratch = [(seg.views(Y1a), _ptr_array(seg.ptrs(Y1a))), (seg.views(Y1b), _ptr_array(seg.ptrs(Y1b)))]

        def op(code, out_p, y_p, a, b=None, c=None, d=None, dt=0.0, s1=0.0, s2=0.0):
            check(lib.b2ode_fixed_op(dcode, code, nseg, lens, out_p, y_p, a, b, c, d, float(dt), float(s1), float(s2),
                                     sm, sptr))

        def row_ptrs(j):
            return _ptr_array([o.data_ptr() + j * n * item for o, n in zip(outs, seg.lens)])

        def row_views(j):
            return tuple(o[j] for o in outs)

        y_views, y_ptrs = row_views(0), row_ptrs(0)
        j = 1
        nfe = 0
        func = self.func
        flip = 0
        for i in range(n_steps):
            t0, t1, dt = g_np[i], g_np[i + 1], dts[i]
            # outputs inside this cell (solvers.py:97): t0 < t[j] <= t1
            j_hi = j
            while j_hi < n_out and t1 >= t_np[j_hi]:
                j_hi += 1
            ends_on_output = j_hi > j and t_np[j_hi - 1] == t1
            if ends_on_output:
                y1_views, y1_ptrs = row_views(j_hi - 1), row_ptrs(j_hi - 1)   # y1 lands straight in the slab
            else:
                y1_views, y1_ptrs = scratch[flip]
                flip ^= 1
            tv = times_dev[i]
            while True:
                live = set()
                alias0 = fo.alias_events
                if m == "euler":
                    k1 = fo.collect(func(tv[0], y_views), live)
                    op(_lib.OP_EULER, y1_ptrs, y_ptrs, fo.pointers(k1), dt=dt)
                    nfe += 1
                elif m == "midpoint":
                    k1 = fo.collect(func(tv[0], y_views), live)
                    op(_lib.OP_HALF_STEP, s_ptrs, y_ptrs, fo.pointers(k1), dt=dt)
                    k2 = fo.collect(func(tv[1], s_views), live)
                    op(_lib.OP_EULER, y1_ptrs, y_ptrs, fo.pointers(k2), dt=dt)
                    nfe += 2
                elif m == "heun":
                    k1 = fo.collect(func(tv[0], y_views), live)
                    op(_lib.OP_EULER, s_ptrs, y_ptrs, fo.pointers(k1), dt=dt)
                    k2 = fo.collect(func(tv[1], s_views), live)
                    op(_lib.OP_HEUN_FINAL, y1_ptrs, y_ptrs, _ptr_array([x.data_ptr() for x in k1]),
                       _ptr_array([x.data_ptr() for x in k2]), dt=dt)
                    nfe += 2
                else:   # rk4, 3/8 rule (rk_common.py:73-81)
                    k1 = fo.collect(func(tv[0], y_views), live)
                    p1 = _ptr_array([x.data_ptr() for x in k1])
                    op(_lib.OP_RK4_S2, s_ptrs, y_ptrs, p1, dt=dt)
                    k2 = fo.collect(func(tv[1], s_views), live)
                    p2 = _ptr_array([x.data_ptr() for x in k2])
                    op(_lib.OP_RK4_S3, s_ptrs, y_ptrs, p1, p2, dt=dt)
                    k3 = fo.collect(func(tv[2], s_views), live)
                    p3 = _ptr_array([x.data_ptr() for x in k3])
                    op(_lib.OP_RK4_S4, s_ptrs, y_ptrs, p1, p2, p3, dt=dt)
                    k4 = fo.collect(func(tv[3], s_views), live)
                    p4 = _ptr_array([x.data_ptr() for x in k4])
                    op(_lib.OP_RK4_FINAL, y1_ptrs, y_ptrs, p1, p2, p3, p4, dt=dt)
                    nfe += 4
                if fo.alias_events == alias0:
                    break
                # func turned out to reuse its output storage inside this step: earlier k's were overwritten;
                # from now on results are cloned -- redo the step once (y0 of the cell is untouched)
            # interior outputs: linear interpolation (solvers.py:106-115)
            for jj in range(j, j_hi - (1 if ends_on_output else 0)):
                op(_lib.OP_LERP, row_ptrs(jj), y_ptrs, y1_ptrs, s1=npdt(t1) - npdt(t0), s2=npdt(t_np[jj]) - npdt(t0))
            j = j_hi
            y_views, y_ptrs = y1_views, y1_ptrs
        self.stats = dict(n_accepted=n_steps, n_rejected=0, nfe=nfe, status=0, fused_rhs=False)
        last_stats.clear()
        last_stats.update(self.stats)
        stream.synchronize()
        return tuple(outs)


class Euler(FixedGridODESolver):
    """tfdiffeq/fixed_grid.py:4"""
    method, order = "euler", 1


class Midpoint(FixedGridODESolver):
    """tfdiffeq/fixed_grid.py:14"""
    method, order = "midpoint", 2


class Heun(FixedGridODESolver):
    """tfdiffeq/fixed_grid.py:26"""
    method, order = "heun", 2


class RK4(FixedGridODESolver):
    """tfdiffeq/fixed_grid.py:39 (the 3/8 rule, rk_common.py:73-81)"""
    method, order = "rk4", 4
