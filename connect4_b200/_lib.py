"""ctypes binding of libc4b200.so (include/c4b200.h).  There is no CPU fallback: if the library is missing, or a
compute entry point is called without a usable GPU, the call raises."""
import ctypes as C
import os
import threading

from . import _build

_lib = None

u64p = C.c_void_p
vp = C.c_void_p


class C4Error(RuntimeError):
    pass


class MCTSConfigC(C.Structure):
    _fields_ = [("simulations", C.c_int32), ("pb_c_base", C.c_double), ("pb_c_init", C.c_double),
                ("root_dirichlet_alpha", C.c_double), ("root_exploration_fraction", C.c_double),
                ("num_sampling_moves", C.c_int32)]


class RecordC(C.Structure):
    _fields_ = [("c0", C.c_uint64), ("c1", C.c_uint64), ("policy", C.c_float * 7), ("result_value", C.c_float),
                ("search_value", C.c_float), ("game_id", C.c_int32), ("move", C.c_int8), ("ply", C.c_int8),
                ("n_moves", C.c_int8), ("result", C.c_int8), ("reserved", C.c_int32)]


assert C.sizeof(RecordC) == 64

# c4_eval_fn: the evaluator of a caller-served network (c4_net_create_external)
EVAL_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p)

# every symbol declared in include/c4b200.h : (restype, argtypes)
SIGNATURES = {
    "c4_last_error": (C.c_char_p, []),
    "c4_abi_version": (C.c_int, []),
    "c4_device_count": (C.c_int, []),
    "c4_board_legal_mask": (C.c_int, [vp, vp, vp, vp, C.c_int64, vp]),
    "c4_board_drop": (C.c_int, [vp, vp, vp, vp, C.c_int64, vp]),
    "c4_board_has_win": (C.c_int, [vp, vp, C.c_int64, vp]),
    "c4_board_result": (C.c_int, [vp, vp, vp, C.c_int64, vp]),
    "c4_board_fliplr": (C.c_int, [vp, vp, vp, vp, C.c_int64, vp]),
    "c4_board_to_planes": (C.c_int, [vp, vp, vp, C.c_int, C.c_int64, vp]),
    "c4_board_from_planes": (C.c_int, [vp, vp, vp, vp, C.c_int64, vp]),
    "c4_board_evaluate_centre": (C.c_int, [vp, vp, vp, C.c_int64, vp]),
    "c4_net_create": (C.c_int, [C.c_int, vp, C.c_int64, C.POINTER(vp)]),
    "c4_net_create_external": (C.c_int, [C.c_int, EVAL_FN, vp, C.POINTER(vp)]),
    "c4_net_destroy": (C.c_int, [vp]),
    "c4_net_forward": (C.c_int, [vp, vp, vp, C.c_int64, vp, vp, vp]),
    "c4_net_flops_per_position": (C.c_double, [vp]),
    "c4_net_get": (C.c_double, [vp, C.c_int]),
    "c4_ctx_create": (C.c_int, [C.c_int, C.c_int32, C.POINTER(MCTSConfigC), C.POINTER(vp)]),
    "c4_ctx_destroy": (C.c_int, [vp]),
    "c4_ctx_set_config": (C.c_int, [vp, C.POINTER(MCTSConfigC)]),
    "c4_ctx_set_net": (C.c_int, [vp, vp]),
    "c4_ctx_get": (C.c_int, [vp, C.c_int]),
    "c4_ctx_set_rng": (C.c_int, [vp, C.c_int, C.c_uint64, vp, vp, C.c_int]),
    "c4_search_begin": (C.c_int, [vp, vp, vp, C.c_int32, vp]),
    "c4_search_pending": (C.c_int, [vp, vp, vp, vp, C.POINTER(C.c_int32), vp]),
    "c4_search_supply": (C.c_int, [vp, vp, vp, C.c_int, C.c_int32, vp]),
    "c4_search_run": (C.c_int, [vp, C.c_int, vp]),
    "c4_search_readout": (C.c_int, [vp, C.c_int32] + [vp] * 11 + [vp]),
    "c4_search_export_tree": (C.c_int, [vp, C.c_int32, vp, C.c_int64, C.POINTER(C.c_int64), vp]),
    "c4_selfplay_run": (C.c_int, [vp, C.c_int, C.c_int64, C.c_int64, C.c_int64, vp, vp, vp, C.c_int64,
                                  C.POINTER(C.c_int64), vp]),
    "c4_selfplay_bench": (C.c_int, [vp, C.c_int, C.c_int64] + [C.POINTER(C.c_int64)] * 4 +
                          [C.POINTER(C.c_float)] * 3 + [vp]),
    "c4_selfplay_reset": (C.c_int, [vp, vp]),
    "c4_selfplay_stream": (C.c_int, [vp, C.c_int, C.c_int, C.c_int64, C.c_double] + [C.POINTER(C.c_int64)] * 4 +
                           [C.POINTER(C.c_float), C.POINTER(C.c_int32), vp]),
    "c4_ctx_clear_memo": (C.c_int, [vp, vp]),
    "c4_records_augment_pack": (C.c_int, [vp, C.c_int64, vp, vp, vp, vp]),
}

EVAL_EXTERNAL, EVAL_CENTRE, EVAL_NET = 0, 1, 2
RNG_NONE, RNG_PHILOX, RNG_INJECTED = 0, 1, 2


def lib_path():
    # C4_LIB: an alternative build of the SAME library (tools/build_variant.sh; kernel-variant experiments)
    return os.environ.get("C4_LIB") or _build.LIB


def load():
    """Load libc4b200.so (never builds implicitly on a GPU box: the .so travels in-tree; __graft_entry__.build() or
    `python -m connect4_b200._build` creates it)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise C4Error("libc4b200.so not found at %s -- run `python -m connect4_b200._build` (nvcc, sm_100a). "
                      "There is no CPU fallback." % path)
    L = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    if L.c4_abi_version() != 1:
        raise C4Error("libc4b200.so ABI version mismatch")
    _lib = L
    return L


_callback_error = threading.local()


def set_callback_error(exc):
    """remember the exception a Python evaluator raised inside a c4_eval_fn callback (which can only return non-zero);
    the failing engine call re-raises it as the cause of its C4Error"""
    _callback_error.exc = exc


def check(rc):
    if rc != 0:
        msg = load().c4_last_error().decode() or "libc4b200 error %d" % rc
        cause, _callback_error.exc = getattr(_callback_error, "exc", None), None
        if cause is None:
            raise C4Error(msg)
        raise C4Error("%s: %s: %s" % (msg, type(cause).__name__, cause)) from cause


def require_gpu():
    import torch
    if not torch.cuda.is_available() or load().c4_device_count() <= 0:
        raise C4Error("connect4_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def ptr(t):
    """device/host pointer of a torch tensor (or None)"""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
