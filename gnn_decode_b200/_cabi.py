"""ctypes binding of the C ABI declared in include/gnn_decode.h.

The product has NO CPU fallback: if the CUDA library is missing this module raises, loudly.
"""
import ctypes as C
import os

from .build import LIB_PATH

GD_OK, GD_ERR_INVALID, GD_ERR_CUDA, GD_ERR_UNSUPPORTED = 0, 1, 2, 3
PROG_CGNNI, PROG_QGNNI, PROG_V2_4, PROG_BP_QUANTUM, PROG_BP_CLASSICAL = 0, 1, 2, 3, 4
PROG_NEURAL_BP, PROG_GRU_CA = 5, 6
PROG_V3_0, PROG_V1_2_2, PROG_V2_4_1 = 7, 8, 9
FLAG_ALL_ITERS = 1
PHASE_VAR, PHASE_CHK = 0, 1
ABI_VERSION = 2


class GdModel(C.Structure):
    _fields_ = [("program", C.c_int32), ("hidden", C.c_int32), ("iters", C.c_int32), ("flags", C.c_int32)]


class GdLaunchInfo(C.Structure):
    _fields_ = [("tile", C.c_int32), ("threads", C.c_int32), ("grid", C.c_int32), ("smem_bytes", C.c_int32),
                ("resident", C.c_int32), ("n_tiles", C.c_int32)]


class GdAdam(C.Structure):
    _fields_ = [("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double),
                ("weight_decay", C.c_double), ("step", C.c_int32)]


_p = C.c_void_p
_SIGNATURES = {
    # name: (restype, argtypes)
    "gd_last_error": (C.c_char_p, []),
    "gd_abi_version": (C.c_int, []),
    "gd_weights_size": (C.c_int64, [C.POINTER(GdModel)]),
    "gd_graph_create": (C.c_int, [_p, C.c_int64, C.c_int32, C.c_int32, C.c_int, C.POINTER(_p)]),
    "gd_graph_destroy": (None, [_p]),
    "gd_graph_dims": (C.c_int, [_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int64),
                                C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "gd_graph_tables": (C.c_int, [_p, _p, _p, _p, _p, _p, _p]),
    "gd_graph_check_batched": (C.c_int, [_p, _p, C.c_int64, C.c_int32, _p, C.POINTER(C.c_int64)]),
    "gd_propagate_features": (C.c_int, [C.c_int32, C.c_int32]),
    "gd_propagate_fwd": (C.c_int, [_p, C.POINTER(GdModel), C.c_int32, C.c_int32, _p, _p, _p, _p, C.c_int64, _p]),
    "gd_decode_fwd": (C.c_int, [_p, C.POINTER(GdModel), _p, _p, _p, _p, _p, C.c_int64, _p]),
    "gd_decode_fwd_aux": (C.c_int, [_p, C.POINTER(GdModel), _p, _p, _p, _p, _p, _p, _p, C.c_int64, _p]),
    "gd_decode_packed_fwd": (C.c_int, [_p, C.POINTER(GdModel), _p, _p, _p, _p, _p, C.c_int64, _p]),
    "gd_pipeline_create": (C.c_int, [_p, C.POINTER(GdModel), _p, C.c_int64, C.c_int32, C.POINTER(_p)]),
    "gd_pipeline_destroy": (None, [_p]),
    "gd_pipeline_set_weights": (C.c_int, [_p, _p]),
    "gd_pipeline_submit": (C.c_int, [_p, _p, _p, _p, C.c_int64, C.POINTER(C.c_int32)]),
    "gd_pipeline_submit_packed": (C.c_int, [_p, _p, _p, _p, _p, C.c_int64, C.POINTER(C.c_int32)]),
    "gd_pipeline_wait": (C.c_int, [_p, C.c_int32]),
    "gd_pipeline_drain": (C.c_int, [_p]),
    "gd_decode_host": (C.c_int, [_p, C.POINTER(GdModel), _p, _p, _p, _p, C.c_int64]),
    "gd_decode_tables_info": (C.c_int, [_p, C.POINTER(GdModel), C.c_int64, C.POINTER(C.c_int32)]),
    "gd_decode_launch_info": (C.c_int, [_p, C.POINTER(GdModel), C.c_int64, C.POINTER(GdLaunchInfo)]),
    "gd_decode_autotune": (C.c_int, [_p, C.POINTER(GdModel), _p, _p, C.c_int64, C.c_int32, _p, C.POINTER(GdLaunchInfo)]),
    "gd_sample": (C.c_int, [_p, C.c_int32, _p, C.c_int32, C.c_uint64, C.c_uint64, _p, _p, C.c_int64, _p]),
    "gd_eval_failures": (C.c_int, [_p, _p, C.c_int32, _p, _p, C.c_int64, _p, _p]),
    "gd_microbench": (C.c_int, [C.c_int32, C.c_int32, C.c_int, C.POINTER(C.c_double)]),
    "gd_set_option": (C.c_int, [C.c_char_p, C.c_int64, C.c_int32]),
    "gd_stash_floats": (C.c_int64, [_p, C.POINTER(GdModel), C.c_int64]),
    "gd_decode_fwd_train": (C.c_int, [_p, C.POINTER(GdModel), _p, _p, _p, _p, _p, C.c_int64, _p]),
    "gd_bwd_workspace_floats": (C.c_int64, [_p, C.POINTER(GdModel), C.c_int64]),
    "gd_decode_bwd": (C.c_int, [_p, C.POINTER(GdModel), _p, _p, _p, _p, _p, _p, C.c_int32, C.c_int64, _p]),
    "gd_loss_v2_4": (C.c_int, [_p, _p, C.c_int32, _p, _p, _p, _p, _p, C.c_int64, _p]),
    "gd_p2p_buffer_floats": (C.c_int64, [C.c_int32]),
    "gd_p2p_allreduce": (C.c_int, [_p, C.c_int32, C.c_int32, _p, _p, C.c_int32, C.c_uint32, C.c_float, _p, _p]),
    "gd_adam_step": (C.c_int, [C.POINTER(GdAdam), _p, _p, _p, _p, C.c_int64, C.c_float, _p]),
    "gd_p2p_allreduce_adam": (C.c_int, [_p, C.c_int32, C.c_int32, _p, _p, C.c_int32, C.c_uint32, C.c_float, _p,
                                        C.POINTER(GdAdam), _p, _p, _p, _p]),
}
# entry points added after ABI v1 froze; bound when present (tests assert the header/.so agree)
_OPTIONAL = {}

_lib = None


class GdError(RuntimeError):
    pass


def lib():
    """Load the CUDA library (once).  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GdError(
            "gnn_decode_b200: CUDA library %s is missing. Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
            "There is no CPU fallback." % LIB_PATH)
    l = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(l, name)
        fn.restype, fn.argtypes = res, args
    for name, (res, args) in _OPTIONAL.items():
        if hasattr(l, name):
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
    if l.gd_abi_version() != ABI_VERSION:
        raise GdError("ABI version mismatch: library %d, binding %d" % (l.gd_abi_version(), ABI_VERSION))
    _lib = l
    return l


def check(rc, what=""):
    """Map a C status to the exception the reference's Python would raise."""
    if rc == GD_OK:
        return
    msg = lib().gd_last_error().decode("utf-8", "replace")
    if rc == GD_ERR_INVALID:
        raise ValueError(msg or what)
    raise GdError(msg or what)


def exported_symbols():
    return list(_SIGNATURES) + [n for n in _OPTIONAL if hasattr(lib(), n)]
