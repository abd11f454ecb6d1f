"""ctypes binding of libgenpc_b200.so (the C ABI in include/genpc_b200.h).

There is NO CPU fallback: if the CUDA library is missing or a call fails, this module raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# GENPC_LIB: an alternative build of the same library (same-box A/B runs of compile-time variants, tools/); default: in-tree
LIB_PATH = os.path.abspath(os.environ["GENPC_LIB"]) if os.environ.get("GENPC_LIB") else os.path.join(_HERE, "libgenpc_b200.so")
_lib = None

_vp = ctypes.c_void_p
_int = ctypes.c_int
_flt = ctypes.c_float
_dbl = ctypes.c_double
_sz = ctypes.c_size_t


class GenpcError(RuntimeError):
    pass


class ChamferFuse(ctypes.Structure):
    """genpc_chamfer_fuse_t (include/genpc_b200.h)."""
    _fields_ = [("workspace_armed", _int), ("use_sqrt", _int), ("w1", _flt), ("w2", _flt), ("loss_out", _vp),
                ("loss_workspace", _vp), ("loss_workspace_bytes", _sz), ("zero1", _vp), ("zero2", _vp)]


_SIGNATURES = {
    "genpc_version": (ctypes.c_char_p, []),
    "genpc_set_tunable": (_int, [ctypes.c_char_p, ctypes.c_char_p]),
    "genpc_get_tunable": (ctypes.c_char_p, [ctypes.c_char_p]),
    "genpc_chamfer_workspace_bytes": (_sz, [_int, _int, _int]),
    "genpc_chamfer_forward": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _int, _vp, _sz, _vp]),
    "genpc_chamfer_prune_stats": (_int, [_vp]),
    "genpc_chamfer_scan_kind": (_int, [_int, _int, _int]),
    "genpc_chamfer_sort_layout": (_int, [_int, _int, _int, _int, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    "genpc_host_feed_create": (_int, [ctypes.POINTER(_vp)]),
    "genpc_host_feed_destroy": (_int, [_vp]),
    "genpc_host_feed_error": (_int, [_vp, _vp]),
    "genpc_host_feed_inject_error": (_int, [_vp, _vp]),
    "genpc_chamfer_forward_host": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _int, _int, _vp, _sz,
                                          _vp]),
    "genpc_chamfer_fuse_workspace_bytes": (_sz, [_int, _int, _int]),
    "genpc_chamfer_forward_fused": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _int, _vp, _sz,
                                           ctypes.POINTER(ChamferFuse), _vp]),
    "genpc_chamfer_forward_host_fused": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _int, _int, _vp,
                                                _sz, ctypes.POINTER(ChamferFuse), _vp]),
    "genpc_chamfer_forward_ragged": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _int, _vp, _sz,
                                            ctypes.POINTER(ChamferFuse), _vp]),
    "genpc_chamfer_loss_backward_ragged": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _flt, _flt, _vp, _vp,
                                                  _int, _int, _int, _vp]),
    "genpc_chamfer_backward": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _int, _vp]),
    "genpc_chamfer_loss_workspace_bytes": (_sz, []),
    "genpc_chamfer_loss": (_int, [_vp, _vp, _sz, _sz, _int, _flt, _flt, _vp, _vp, _sz, _vp]),
    "genpc_chamfer_loss_backward": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _flt, _flt, _vp, _vp, _int, _int,
                                           _int, _vp]),
    "genpc_nn_partial_packed": (_int, [_vp, _vp, _vp, _int, _int, _int, _int, _int, _vp]),
    "genpc_nn_unpack": (_int, [_vp, _vp, _vp, _sz, _vp]),
    "genpc_chamfer_sym_partial": (_int, [_vp, _vp, _vp, _vp, _int, _int, _int, _int, _int, _vp]),
    "genpc_chamfer_sym_fixup": (_int, [_vp, _vp, _vp, _int, _int, _int, _vp, _vp, _vp]),
    "genpc_icp_step": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _int, _int, _flt, _flt, _flt, _int, _vp]),
    "genpc_icp_step_ragged": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _int, _int, _flt, _flt,
                                     _flt, _int, _vp]),
    "genpc_knn_mean_distance": (_int, [_vp, _int, _int, _int, _vp, _vp]),
    "genpc_knn_mean_distance_ragged": (_int, [_vp, _vp, _int, _int, _int, _int, _vp, _vp]),
    "genpc_mesh_face_areas": (_int, [_vp, _vp, _int, _int, _vp, _vp]),
    "genpc_mesh_sample": (_int, [_vp, _vp, _vp, _vp, _int, _int, ctypes.c_ulonglong, _vp, _vp, _vp, _vp]),
    "genpc_fps_workspace_bytes": (_sz, [_int, _int, _int]),
    "genpc_fps": (_int, [_vp, _int, _int, _int, _int, _vp, _vp, _vp, _sz, _vp]),
    "genpc_depth_workspace_bytes": (_sz, [_int]),
    "genpc_project_uv": (_int, [_vp, _vp, _int, _int, _int, _flt, _vp, _vp, _vp, _vp, _sz, _vp]),
    "genpc_zbuffer_render": (_int, [_vp, _vp, _vp, _vp, _int, _int, _int, _int, _vp, _vp, _vp, _vp, _vp, _vp, _sz,
                                    _vp]),
    "genpc_unproject": (_int, [_vp, _vp, _int, _vp, _vp, _int, _int, _int, _vp, _vp, _vp, _vp]),
    "genpc_emd_workspace_bytes": (_sz, [_int]),
    "genpc_emd_workspace_bytes_n": (_sz, [_int, _int]),
    "genpc_emd_forward": (_int, [_vp] * 12 + [_int, _int, _int, _flt, _int, _vp, _sz, _vp]),
    "genpc_emd_backward": (_int, [_vp, _vp, _vp, _vp, _vp, _int, _int, _vp]),
    "genpc_register_workspace_bytes": (_sz, [_int, _int, _int]),
    "genpc_register_launches_per_iter": (_int, [_int, _int, _int]),
    "genpc_register_run": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _int, _int, _int, _int, _int,
                                  _dbl, _dbl, _dbl, _flt, _flt, _flt, _vp, _sz, _int, _vp]),
    "genpc_register_run_ragged": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _int, _int, _int, _int,
                                         _int, _dbl, _dbl, _dbl, _flt, _flt, _flt, _vp, _sz, _int, _vp]),
}


def lib():
    """Load the shared library (built by `python -m genpc_b200.csrc.build` / __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GenpcError(
                f"{LIB_PATH} is missing: build it with `python -m genpc_b200.csrc.build` "
                "(genpc_b200 has no CPU fallback)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class tunable:
    """Context manager: set an experiment knob of the library (GENPC_* name) for the duration of a block.  The library reads
    the environment only once, at load time, so tests / tools flip knobs through this instead of os.environ."""

    def __init__(self, **knobs):
        self.knobs = {k: (None if v is None else str(v)) for k, v in knobs.items()}
        self.old = {}

    def __enter__(self):
        L = lib()
        for k, v in self.knobs.items():
            self.old[k] = L.genpc_get_tunable(k.encode())
            check(L.genpc_set_tunable(k.encode(), None if v is None else v.encode()), f"genpc_set_tunable({k})")
        return self

    def __exit__(self, *exc):
        L = lib()
        for k, v in self.old.items():
            L.genpc_set_tunable(k.encode(), v)
        return False


def check(rc, what):
    if rc != 0:
        if rc > 0:
            raise GenpcError(f"{what}: CUDA error {rc}")
        names = {-1: "shape violation", -2: "workspace missing/too small", -3: "index range"}
        raise GenpcError(f"{what}: {names.get(rc, rc)}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def current_stream(device):
    import torch

    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if not t.is_cuda:
            raise GenpcError("genpc_b200 runs on CUDA tensors only (no CPU fallback); got a CPU tensor")
