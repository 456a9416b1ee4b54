"""ctypes prototypes of include/gaz_net.h."""
import ctypes as C

_P = C.c_void_p


class GazNetBuf(C.Structure):
    _fields_ = [("kind", C.c_int32), ("width", C.c_int32)]


class GazNetOp(C.Structure):
    _fields_ = [("type", C.c_int32), ("in_buf", C.c_int32), ("res_buf", C.c_int32), ("out_raw", C.c_int32),
                ("out_a", C.c_int32), ("out_b", C.c_int32), ("cin", C.c_int32), ("cout", C.c_int32),
                ("ksize", C.c_int32), ("act", C.c_int32), ("flags", C.c_int32), ("pad", C.c_int32),
                ("w", C.c_int64), ("bias", C.c_int64), ("scale_a", C.c_int64), ("shift_a", C.c_int64),
                ("scale_b", C.c_int64), ("shift_b", C.c_int64), ("w2", C.c_int64), ("bias2", C.c_int64),
                ("w3", C.c_int64), ("bias3", C.c_int64)]


class GazNetDesc(C.Structure):
    _fields_ = [("game", C.c_int32), ("max_batch", C.c_int32), ("n_bufs", C.c_int32), ("n_ops", C.c_int32),
                ("policy_mode", C.c_int32), ("device", C.c_int32), ("bufs", C.POINTER(GazNetBuf)),
                ("ops", C.POINTER(GazNetOp)), ("wf", _P), ("n_wf", C.c_int64), ("wh", _P), ("n_wh", C.c_int64)]


SYMBOLS = {
    "gaz_net_create": (C.c_int, [C.POINTER(GazNetDesc), C.POINTER(_P)]),
    "gaz_net_create_shared": (C.c_int, [C.POINTER(GazNetDesc), _P, C.POINTER(_P)]),
    "gaz_net_destroy": (None, [_P]),
    "gaz_net_forward_host": (C.c_int, [_P, _P, C.c_int, _P, _P, _P]),
    "gaz_attach_net": (C.c_int, [_P, _P]),
    "gaz_attach_nets": (C.c_int, [_P, _P, C.c_int]),
    "gaz_set_tree_nets": (C.c_int, [_P, _P]),
    "gaz_set_eval_symmetry": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, C.c_uint64]),
    "gaz_eval_net": (C.c_int, [_P]),
    "gaz_rounds_net": (C.c_int, [_P, C.c_int]),
    "gaz_rounds_net_async": (C.c_int, [_P, C.c_int]),
    "gaz_net_bytes": (C.c_int64, [_P]),
    "gaz_net_launches_per_forward": (C.c_int, [_P]),
    "gaz_net_op_blocks": (C.c_int, [_P, C.c_int]),
    "gaz_net_profile": (C.c_int, [_P, C.c_int]),
    "gaz_net_profile_read": (C.c_int, [_P, _P, _P, _P]),
    "gaz_net_time_forward": (C.c_int, [_P, C.c_int, C.c_int, _P]),
}
