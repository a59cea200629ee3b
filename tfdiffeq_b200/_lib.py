"""ctypes binding of ``libb2ode.so`` (C ABI declared in ``include/b2ode.h``).

The product path has NO fallback: if the shared library is missing or does not export the ABI this
module raises ``ImportError``/``OSError`` loudly.  Nothing here imports ``oracle/``.
"""
import ctypes as C
import os

MAXSEG = 12
MAXK = 14
MAXPEERS = 8
F32, F64 = 0, 1
ST_UNDERFLOW, ST_NONFINITE, ST_MAXSTEPS = 1, 2, 4
CTRL_REFERENCE, CTRL_TSIT5 = 0, 1
FAM_STAGE0, FAM_STAGE, FAM_FINALIZE, FAM_EMIT, FAM_INIT, FAM_FIXED, FAM_FUSED, FAM_STAGE_GEMM = range(8)
RHS_LORENZ, RHS_LOTKA_VOLTERRA, RHS_CUBIC_MLP, RHS_KEPLER, RHS_LINEAR = 0, 1, 2, 3, 4
LINEAR_MAX_DIM = 128      # largest D of RHS_LINEAR (A stays in shared memory: 128 x 128 fp64 = 128 KB)
OP_EULER, OP_HALF_STEP, OP_HEUN_FINAL, OP_RK4_S2, OP_RK4_S3, OP_RK4_S4, OP_RK4_FINAL, OP_LERP = range(8)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B2ODE_LIB", os.path.join(_HERE, "libb2ode.so"))


class State(C.Structure):
    """mirror of ``b2ode_state`` (256 bytes)"""
    _fields_ = [("t0", C.c_double), ("t1", C.c_double), ("dt", C.c_double), ("dt_last", C.c_double),
                ("msr_max", C.c_double), ("h0", C.c_double), ("reserved_d", C.c_double * 2),
                ("n_acc", C.c_uint64), ("n_rej", C.c_uint64), ("attempt", C.c_uint64), ("n_steps_adv", C.c_int64),
                ("accept", C.c_int32), ("done", C.c_int32), ("status", C.c_uint32), ("cursor", C.c_int32),
                ("emit_j0", C.c_int32), ("emit_j1", C.c_int32), ("ticket", C.c_uint32), ("reserved_u", C.c_uint32),
                ("xseq", C.c_uint64), ("klast", C.c_uint64 * MAXSEG), ("reserved_t", C.c_double * 3)]


class AdaptiveDesc(C.Structure):
    """mirror of ``b2ode_adaptive_desc``"""
    _fields_ = [("dtype", C.c_int32), ("nseg", C.c_int32), ("seg_len", C.c_int64 * MAXSEG),
                ("n_k", C.c_int32), ("fsal", C.c_int32), ("alpha", C.c_double * MAXK),
                ("beta", (C.c_double * MAXK) * MAXK), ("c_sol", C.c_double * MAXK), ("c_error", C.c_double * MAXK),
                ("c_mid", C.c_double * MAXK), ("dense_kind", C.c_int32), ("controller", C.c_int32),
                ("rtol", C.c_double * MAXSEG), ("atol", C.c_double * MAXSEG),
                ("safety", C.c_double), ("ifactor", C.c_double), ("dfactor", C.c_double), ("exponent", C.c_double),
                ("max_num_steps", C.c_int64), ("init_order", C.c_int32), ("sm_count", C.c_int32)]


class AdaptiveBuffers(C.Structure):
    """mirror of ``b2ode_adaptive_buffers``"""
    _fields_ = [("state", C.c_void_p), ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
                ("y0", C.c_void_p * MAXSEG), ("f0", C.c_void_p * MAXSEG), ("ystage", C.c_void_p * MAXSEG),
                ("tstage", C.c_void_p), ("t_out", C.c_void_p), ("n_out", C.c_int32),
                ("out", C.c_void_p * MAXSEG)]


class RhsDesc(C.Structure):
    """mirror of ``b2ode_rhs_desc``"""
    _fields_ = [("kind", C.c_int32), ("n_params", C.c_int32), ("params", C.c_double * 8), ("data", C.c_void_p),
                ("time_sign", C.c_double)]


class FusedDesc(C.Structure):
    """mirror of ``b2ode_fused_desc``"""
    _fields_ = [("rhs_kind", C.c_int32), ("n_rhs_params", C.c_int32), ("rhs_params", C.c_double * 8), ("rhs_data", C.c_void_p),
                ("time_sign", C.c_double), ("y0", C.c_void_p), ("out", C.c_void_p), ("t_out", C.c_void_p), ("n_out", C.c_int32),
                ("t_start", C.c_double), ("first_step", C.c_double), ("state", C.c_void_p), ("workspace", C.c_void_p),
                ("workspace_bytes", C.c_size_t), ("rank", C.c_int32), ("nranks", C.c_int32), ("mailboxes", C.c_void_p),
                ("n_traj_rank", C.c_int64 * MAXPEERS), ("cuda_stream", C.c_void_p), ("host_mark", C.c_void_p)]


assert C.sizeof(State) == 256

PtrArray = C.c_void_p * MAXSEG
LenArray = C.c_int64 * MAXSEG

_SIGNATURES = {
    "b2ode_version": (C.c_int, []),
    "b2ode_last_error": (C.c_char_p, []),
    "b2ode_state_bytes": (C.c_size_t, []),
    "b2ode_mailbox_bytes": (C.c_size_t, []),
    "b2ode_workspace_bytes": (C.c_size_t, [C.POINTER(AdaptiveDesc)]),
    "b2ode_adaptive_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(AdaptiveDesc)]),
    "b2ode_adaptive_destroy": (None, [C.c_void_p]),
    "b2ode_adaptive_bind": (C.c_int, [C.c_void_p, C.POINTER(AdaptiveBuffers), C.c_void_p]),
    "b2ode_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b2ode_adaptive_init": (C.c_int, [C.c_void_p, C.c_double, C.c_double]),
    "b2ode_initial_step_probe": (C.c_int, [C.c_void_p]),
    "b2ode_initial_step_finish": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "b2ode_rk_stage": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "b2ode_rk_finalize": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "b2ode_poll_async": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b2ode_poll_sync": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b2ode_comm_attach": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "b2ode_comm_set_global_len": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "b2ode_comm_set_replicated": (C.c_int, [C.c_void_p, C.c_uint]),
    "b2ode_mailbox_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_char_p]),
    "b2ode_mailbox_open": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "b2ode_mailbox_close": (C.c_int, [C.c_void_p]),
    "b2ode_mailbox_destroy": (C.c_int, [C.c_void_p]),
    "b2ode_fused_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "b2ode_fused_capacity": (C.c_int64, [C.POINTER(AdaptiveDesc), C.c_int]),
    "b2ode_fused_fixed_solve": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_void_p, C.c_double,
                                          C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "b2ode_fused_solve": (C.c_int, [C.POINTER(AdaptiveDesc), C.c_void_p]),
    "b2ode_rhs_eval": (C.c_int, [C.c_int, C.POINTER(RhsDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "b2ode_rk_stage_rhs": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(RhsDesc), C.c_void_p]),
    "b2ode_set_k": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "b2ode_dense_layer": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_double), C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "b2ode_dense_layer_x3": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_double), C.c_int, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int,
                                       C.c_void_p]),
    "b2ode_mlp3_packed_bytes": (C.c_int64, [C.c_int, C.c_int]),
    "b2ode_mlp3_pack": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "b2ode_mlp3": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_double), C.c_int, C.c_void_p, C.c_void_p,
                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                             C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "b2ode_lincomb": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_double,
                                C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_double), C.c_int, C.c_void_p]),
    "b2ode_reduce_workspace_bytes": (C.c_size_t, [C.c_int]),
    "b2ode_reduce": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                               C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p, C.c_void_p, C.c_size_t, C.c_int,
                               C.c_void_p]),
    "b2ode_launch_count": (C.c_ulonglong, []),
    "b2ode_timing_enable": (C.c_int, [C.c_uint]),
    "b2ode_timing_read": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "b2ode_fixed_op": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_void_p),
                                 C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                 C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_double, C.c_double, C.c_double,
                                 C.c_int, C.c_void_p]),
}

EXPORTS = tuple(sorted(_SIGNATURES))


class B2odeError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "tfdiffeq_b200: %s not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C tfdiffeq_b200/csrc`). There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError if the ABI is incomplete -- loud on purpose
        fn.restype = res
        fn.argtypes = args
    if lib.b2ode_version() != 1:
        raise ImportError("libb2ode.so ABI version %d != 1" % lib.b2ode_version())
    return lib


lib = _load()


def check(rc):
    if rc != 0:
        raise B2odeError("libb2ode call failed (%d): %s" % (rc, lib.b2ode_last_error().decode("utf-8", "replace")))
RED_ABSMAX2, RED_RATIO_SUMSQ, RED_NOT_CONVERGED = 0, 1, 2
