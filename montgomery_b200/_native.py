"""ctypes binding of libmontgomery_b200.so (the C ABI in include/montgomery_b200.h).

There is deliberately no fallback: if the CUDA library is missing or fails to load, importing
this module raises.  The oracle under oracle/ is never imported from here.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# MGB_LIB: an experiment build of the same library (montgomery_b200.build --variant); never a different backend
LIB_PATH = os.environ.get("MGB_LIB") or os.path.join(_HERE, "libmontgomery_b200.so")

BLS12_377_G1, PALLAS, ED_ON_BLS12_377, BLS12_381_G1 = 0, 1, 2, 3


class MgbOpts(ctypes.Structure):
    _fields_ = [("c", ctypes.c_int), ("unsafe", ctypes.c_int), ("verbose", ctypes.c_int), ("projective", ctypes.c_int),
                ("affine_reduction", ctypes.c_int)]


class MgbTiming(ctypes.Structure):
    _fields_ = [
        ("h2d_scalars", ctypes.c_float), ("decompose_slice", ctypes.c_float), ("sort", ctypes.c_float),
        ("accumulate", ctypes.c_float), ("reduce", ctypes.c_float), ("final_sum", ctypes.c_float),
        ("total", ctypes.c_float), ("c", ctypes.c_int), ("K", ctypes.c_int), ("rounds", ctypes.c_int),
        ("max_bucket", ctypes.c_uint32), ("n_pairs", ctypes.c_uint64), ("n_launches", ctypes.c_uint32),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


EXPORTS = [
    "mgb_create", "mgb_set_points", "mgb_set_points_checked", "mgb_random_points", "mgb_get_points", "mgb_msm", "mgb_msm_prefetch", "mgb_msm_device",
    "mgb_partial_bytes", "mgb_msm_partial", "mgb_combine_partials", "mgb_field_op", "mgb_microbench",
    "mgb_last_error", "mgb_destroy",
    "mgb_comm_unique_id", "mgb_comm_init", "mgb_comm_info", "mgb_msm_sharded",
    "mgb_multi_create", "mgb_multi_set_points", "mgb_multi_set_points_checked", "mgb_multi_random_points", "mgb_multi_get_points", "mgb_multi_msm",
    "mgb_multi_last_error", "mgb_multi_destroy",
]
COMM_ID_BYTES = 128
E_INVALID, E_CUDA, E_NOMEM, E_STATE, E_COMM = -1, -2, -3, -4, -5
PT_NONCANONICAL, PT_OFF_CURVE, PT_NOT_IN_SUBGROUP = 1, 2, 4      # status bits of mgb_set_points_checked


def load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "montgomery_b200: %s is missing -- build it with `python -m montgomery_b200.build` "
            "(nvcc, sm_100a).  There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, sz, ci = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int
    lib.mgb_create.argtypes = [ctypes.POINTER(vp), ci, ci, sz]
    lib.mgb_set_points.argtypes = [vp, vp, vp, sz]
    lib.mgb_set_points_checked.argtypes = [vp, vp, vp, sz, vp, ctypes.POINTER(ctypes.c_uint64)]
    lib.mgb_random_points.argtypes = [vp, ctypes.c_uint64, sz]
    lib.mgb_get_points.argtypes = [vp, sz, sz, vp, vp]
    lib.mgb_msm.argtypes = [vp, vp, sz, ctypes.POINTER(MgbOpts), vp, ctypes.POINTER(ci), ctypes.POINTER(MgbTiming)]
    lib.mgb_msm_device.argtypes = lib.mgb_msm.argtypes
    lib.mgb_msm_prefetch.argtypes = [vp, vp, sz]
    lib.mgb_partial_bytes.argtypes = [vp]
    lib.mgb_partial_bytes.restype = sz
    lib.mgb_msm_partial.argtypes = [vp, vp, ci, sz, ctypes.POINTER(MgbOpts), vp, ctypes.POINTER(MgbTiming)]
    lib.mgb_combine_partials.argtypes = [vp, vp, ci, vp, ctypes.POINTER(ci)]
    lib.mgb_field_op.argtypes = [ci, ci, ci, vp, vp, vp, sz]
    lib.mgb_microbench.argtypes = [ci, ci, ci, ci, ci, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_float)]
    lib.mgb_last_error.argtypes = [vp]
    lib.mgb_last_error.restype = ctypes.c_char_p
    lib.mgb_destroy.argtypes = [vp]
    lib.mgb_destroy.restype = None
    pi = ctypes.POINTER(ci)
    lib.mgb_comm_unique_id.argtypes = [vp]
    lib.mgb_comm_init.argtypes = [vp, vp, ci, ci]
    lib.mgb_comm_info.argtypes = [vp, pi, pi, pi]
    lib.mgb_msm_sharded.argtypes = [vp, vp, ci, sz, ctypes.POINTER(MgbOpts), vp, pi, ctypes.POINTER(MgbTiming)]
    lib.mgb_multi_create.argtypes = [ctypes.POINTER(vp), ci, pi, ci, sz]
    lib.mgb_multi_set_points.argtypes = [vp, vp, vp, sz]
    lib.mgb_multi_set_points_checked.argtypes = [vp, vp, vp, sz, vp, ctypes.POINTER(ctypes.c_uint64)]
    lib.mgb_multi_random_points.argtypes = [vp, ctypes.c_uint64, sz]
    lib.mgb_multi_get_points.argtypes = [vp, sz, sz, vp, vp]
    lib.mgb_multi_msm.argtypes = [vp, vp, sz, ctypes.POINTER(MgbOpts), vp, pi, ctypes.POINTER(MgbTiming)]
    lib.mgb_multi_last_error.argtypes = [vp]
    lib.mgb_multi_last_error.restype = ctypes.c_char_p
    lib.mgb_multi_destroy.argtypes = [vp]
    lib.mgb_multi_destroy.restype = None
    for name in EXPORTS:
        if name not in ("mgb_partial_bytes", "mgb_last_error", "mgb_destroy", "mgb_multi_last_error", "mgb_multi_destroy"):
            getattr(lib, name).restype = ci
    return lib


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = load()
    return _lib
