"""ctypes binding of libagcn_sm100.so (C ABI declared in include/agcn_sgcll.h).

There is no CPU fallback and no alternative backend: if the library is missing or a call fails,
an exception is raised.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libagcn_sm100.so")

AGCN_OK = 0
VARIANT = {"SGC_LL": 0, "SGC_LL_Reslap": 1}
LAPLACIAN = {"reference_literal": 0, "paper": 1}
METRIC_GRAD = {"reference": 0, "full": 1}
ACT = {"linear": 0, "relu": 1}
LOSS = {"sigmoid_ce": 0, "softmax_ce": 1, "weighted_l2": 2}      # the graph heads (AGCN_LOSS_*)
NODE_LOSS = {"node_softmax_ce": 4}                                 # the per-node head (AGCN_PER_NODE_*)
ADJ_RULE = {"mean_distance": 0, "cutoff": 1}
NODE = {"sgcll": 0, "block_end": 1}
NOTIFY_FN = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p)
OUT_RES_L, OUT_RES_W, OUT_L_ALL, SAVE_FOR_BACKWARD = 1, 2, 4, 8


class AgcnError(RuntimeError):
    pass


def loss_code(name):
    """The loss_kind value of agcn_stack_create(_nodes) for a loss name of LOSS or NODE_LOSS."""
    if name in LOSS:
        return LOSS[name]
    if name in NODE_LOSS:
        return NODE_LOSS[name]
    raise ValueError("loss must be one of %s" % sorted(list(LOSS) + list(NODE_LOSS)))


class Desc(ctypes.Structure):
    _fields_ = [("F", ctypes.c_int32), ("Fo", ctypes.c_int32), ("K", ctypes.c_int32), ("variant", ctypes.c_int32),
                ("laplacian_mode", ctypes.c_int32), ("metric_grad", ctypes.c_int32), ("activation", ctypes.c_int32),
                ("flags", ctypes.c_uint32)]


class StackNode(ctypes.Structure):
    """agcn_stack_node: one node of agcn_stack_create_nodes."""
    _fields_ = [("kind", ctypes.c_int32), ("desc", Desc), ("src", ctypes.c_int32)]


_P = ctypes.c_void_p
_SIGNATURES = {
    "agcn_version": (ctypes.c_int, []),
    "agcn_last_error": (ctypes.c_char_p, []),
    "agcn_launch_count": (ctypes.c_uint64, []),
    "agcn_plan_create": (ctypes.c_int, [_P, ctypes.c_int32, ctypes.c_int32, _P, ctypes.POINTER(_P)]),
    "agcn_plan_destroy": (ctypes.c_int, [_P]),
    "agcn_plan_total_nodes": (ctypes.c_int64, [_P]),
    "agcn_plan_total_lap": (ctypes.c_int64, [_P]),
    "agcn_plan_node_off_host": (_P, [_P]),
    "agcn_plan_lap_off_host": (_P, [_P]),
    "agcn_fused_tiles_host": (ctypes.c_int, [_P, ctypes.c_int32, _P, ctypes.c_int32, _P, ctypes.c_int32, _P, _P]),
    "agcn_profile_enable": (ctypes.c_int, [ctypes.c_int]),
    "agcn_profile_read": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]),
    "agcn_profile_timeline": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]),
    "agcn_probe_fp32_fma": (ctypes.c_int, [_P, ctypes.c_int32, _P]),
    "agcn_pack_nodes": (ctypes.c_int, [_P, _P, _P, ctypes.c_int32, _P]),
    "agcn_unpack_nodes": (ctypes.c_int, [_P, _P, _P, ctypes.c_int32, _P]),
    "agcn_pack_lap": (ctypes.c_int, [_P, _P, _P, _P]),
    "agcn_capture_begin": (ctypes.c_int, [_P]),
    "agcn_capture_end_launch": (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_int32)]),
    "agcn_capture_abort": (ctypes.c_int, [_P]),
    "agcn_step_graph_destroy": (ctypes.c_int, [_P]),
    "agcn_unpack_lap": (ctypes.c_int, [_P, _P, _P, _P]),
    "agcn_debug_grouped_product": (ctypes.c_int, [_P, _P, _P, _P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                                  ctypes.c_float, ctypes.c_int32, _P]),
    "agcn_pack_lap_csr": (ctypes.c_int, [_P, _P, _P, _P, _P, _P]),
    "agcn_point_laplacian_workspace_bytes": (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_size_t)]),
    "agcn_point_laplacian": (ctypes.c_int, [_P, _P, ctypes.c_int32, ctypes.c_int32, ctypes.c_float, _P, _P,
                                            ctypes.c_size_t, _P]),
    "agcn_graph_pool": (ctypes.c_int, [_P, _P, _P, _P, _P, ctypes.c_int32, _P]),
    "agcn_graph_pool_backward": (ctypes.c_int, [_P, _P, _P, _P, ctypes.c_int32, _P]),
    "agcn_sgcll_workspace_bytes": (ctypes.c_int, [ctypes.POINTER(Desc), _P, ctypes.POINTER(ctypes.c_size_t),
                                                  ctypes.POINTER(ctypes.c_size_t)]),
    "agcn_sgcll_forward": (ctypes.c_int, [ctypes.POINTER(Desc), _P] + [_P] * 14 + [ctypes.c_size_t, _P]),
    "agcn_sgcll_backward": (ctypes.c_int, [ctypes.POINTER(Desc), _P] + [_P] * 19 + [ctypes.c_size_t, _P]),
    "agcn_gemm_tn_scratch_bytes": (ctypes.c_size_t, [ctypes.c_int32] * 4),
    "agcn_gemm_tn": (ctypes.c_int, [_P, _P, _P, _P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                    _P, ctypes.c_int32, _P]),
    "agcn_node_gemm_scratch_bytes": (ctypes.c_size_t, [ctypes.c_int32, ctypes.c_int32]),
    "agcn_node_gemm": (ctypes.c_int, [_P, ctypes.c_int32, _P, ctypes.c_int32, ctypes.c_int32, _P, ctypes.c_int32,
                                      ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _P, _P, ctypes.c_int32,
                                      ctypes.c_int32, _P, _P]),
    "agcn_dropout": (ctypes.c_int, [_P, _P, ctypes.c_int64, ctypes.c_float, ctypes.c_uint64, _P]),
    "agcn_expand_labels": (ctypes.c_int, [_P, _P, ctypes.c_int32, ctypes.c_int32, _P, _P, _P]),
    "agcn_head_workspace_bytes": (ctypes.c_int, [_P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                                  ctypes.POINTER(ctypes.c_size_t)]),
    "agcn_head_loss_grad": (ctypes.c_int, [_P] * 8 + [ctypes.c_float, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32] +
                            [_P] * 7 + [ctypes.c_size_t, _P]),
    "agcn_head_loss_grad_ex": (ctypes.c_int, [_P] * 8 + [ctypes.c_float, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                                     ctypes.c_int32] + [_P] * 7 + [ctypes.c_size_t, _P]),
    "agcn_head_predict_workspace_bytes": (ctypes.c_int, [_P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                                          ctypes.POINTER(ctypes.c_size_t)]),
    "agcn_head_predict": (ctypes.c_int, [_P] * 8 + [ctypes.c_float, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                                ctypes.c_int32] + [_P] * 3 + [ctypes.c_size_t, _P]),
    "agcn_node_head_workspace_bytes": (ctypes.c_int, [_P, ctypes.c_int32, ctypes.c_int32,
                                                       ctypes.POINTER(ctypes.c_size_t)]),
    "agcn_node_head_loss_grad": (ctypes.c_int, [_P] * 6 + [ctypes.c_float, ctypes.c_int32, ctypes.c_int32] + [_P] * 5 +
                                 [ctypes.c_size_t, _P]),
    "agcn_node_head_predict_workspace_bytes": (ctypes.c_int, [_P, ctypes.c_int32, ctypes.c_int32,
                                                               ctypes.POINTER(ctypes.c_size_t)]),
    "agcn_node_head_predict": (ctypes.c_int, [_P] * 6 + [ctypes.c_float, ctypes.c_int32, ctypes.c_int32] + [_P] * 3 +
                               [ctypes.c_size_t, _P]),
    "agcn_stack_create": (ctypes.c_int, [_P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _P,
                                         ctypes.POINTER(_P)]),
    "agcn_stack_create_nodes": (ctypes.c_int, [_P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _P,
                                               ctypes.POINTER(_P)]),
    "agcn_stack_destroy": (ctypes.c_int, [_P]),
    "agcn_stack_workspace_bytes": (ctypes.c_int, [_P, _P, ctypes.POINTER(ctypes.c_size_t)]),
    "agcn_stack_loss_grad": (ctypes.c_int, [_P] * 6 + [ctypes.c_float] + [_P] * 4 + [ctypes.c_size_t, _P, _P, _P]),
    "agcn_stack_predict_workspace_bytes": (ctypes.c_int, [_P, _P, ctypes.POINTER(ctypes.c_size_t)]),
    "agcn_stack_predict": (ctypes.c_int, [_P] * 6 + [ctypes.c_float] + [_P] * 4 + [ctypes.c_size_t, _P]),
    "agcn_adam_step": (ctypes.c_int, [_P] * 5 + [ctypes.c_int64] + [ctypes.c_float] * 4 + [_P]),
    "agcn_sgcll_host_scratch_bytes": (ctypes.c_int, [ctypes.POINTER(Desc), _P, ctypes.POINTER(ctypes.c_size_t)]),
    "agcn_sgcll_forward_host": (ctypes.c_int, [ctypes.POINTER(Desc), _P] + [_P] * 8 + [ctypes.c_size_t, _P]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def lib():
    """The loaded library; raises if it has not been built (python build_ext.py)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise AgcnError("libagcn_sm100.so is missing: run `python %s` (no CPU fallback exists)"
                            % os.path.join(HERE, "build_ext.py"))
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc):
    if rc != AGCN_OK:
        raise AgcnError("libagcn_sm100 error %d: %s" % (rc, lib().agcn_last_error().decode()))


def launch_count():
    return int(lib().agcn_launch_count())


def profile_enable(on):
    check(lib().agcn_profile_enable(1 if on else 0))


def profile_timeline():
    """[(kernel name, start ms, end ms)] of the launches recorded since the last read, relative to the first one."""
    buf = ctypes.create_string_buffer(1 << 18)
    check(lib().agcn_profile_timeline(buf, len(buf), None))
    out = []
    for line in buf.value.decode().splitlines():
        name, t0, t1 = line.split("\t")
        out.append((name, float(t0), float(t1)))
    return out


def profile_read():
    """{kernel name: (launches, milliseconds)} of the launches recorded since the last read (waits for them)."""
    buf = ctypes.create_string_buffer(1 << 16)
    check(lib().agcn_profile_read(buf, len(buf), None))
    out = {}
    for line in buf.value.decode().splitlines():
        name, n, ms = line.split("\t")
        out[name] = (int(n), float(ms))
    return out
