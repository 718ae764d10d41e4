"""ctypes binding of libdinotrk.so (include/dinotrk.h).  There is NO fallback: if the CUDA library is
missing or fails to load, importing the product path raises."""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_size_t, c_ulonglong, c_void_p

import torch

from . import build as _build

_LIB = None


class Geom(Structure):
    _fields_ = [("H", c_int), ("W", c_int), ("patch", c_int), ("stride", c_int), ("radius", c_int),
                ("h", c_int), ("w", c_int)]


class HeadWeights(Structure):
    _fields_ = [("w1", c_float * 9 * 16), ("b1", c_float * 16), ("w2", c_float * 9 * 16), ("b2", c_float)]


class Features(Structure):
    _fields_ = [("tpc", c_void_p), ("norms", c_void_p), ("hi", c_void_p), ("lo", c_void_p), ("T", c_int), ("C", c_int)]


class VitConfig(Structure):
    _fields_ = [("depth", c_int), ("dim", c_int), ("heads", c_int), ("tap_layer", c_int), ("patch", c_int), ("stride", c_int),
                ("attn_materialized", c_int), ("gemm_f16", c_int), ("gemm_pair", c_int)]


class VitWeights(Structure):
    _fields_ = [("patch_w", c_void_p), ("patch_b", c_void_p), ("cls_pos", c_void_p), ("pos", c_void_p),
                ("blocks", POINTER(c_void_p))]


class DinotrkError(RuntimeError):
    pass


# every exported symbol of include/dinotrk.h: name -> (restype, argtypes)
_P = c_void_p
SIGNATURES = {
    "dinotrk_version": (c_int, []),
    "dinotrk_last_error": (c_char_p, []),
    "dinotrk_launch_count": (c_ulonglong, []),
    "dinotrk_make_geom": (c_int, [c_int, c_int, c_int, c_int, c_int, POINTER(Geom)]),
    "dinotrk_pack_features": (c_int, [_P, _P, _P, c_int, c_int, c_int, _P]),
    "dinotrk_unpack_features": (c_int, [_P, _P, c_int, c_int, c_int, _P]),
    "dinotrk_token_norms": (c_int, [_P, _P, c_int, c_int, c_int, _P]),
    "dinotrk_sample_descriptors": (c_int, [_P, c_int, c_int, POINTER(Geom), _P, c_int, _P, c_int, c_int, _P, _P, _P]),
    "dinotrk_split_fp16": (c_int, [_P, _P, _P, c_size_t, _P]),
    "dinotrk_corr_track_workspace_bytes": (c_size_t, [c_int, c_int, c_int, POINTER(Geom)]),
    "dinotrk_corr_track": (c_int, [POINTER(Features), POINTER(Geom), POINTER(HeadWeights), _P, _P, _P, _P, _P, _P,
                                   c_int, c_int, c_int, _P, _P, c_int, c_int, _P, c_size_t, _P]),
    "dinotrk_corr_maps_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "dinotrk_map_stride": (c_int, [POINTER(Geom)]),
    "dinotrk_corr_maps": (c_int, [POINTER(Features), POINTER(Geom), _P, _P, _P, _P, _P, _P, c_int, c_int, c_int,
                                  _P, _P, c_size_t, _P]),
    "dinotrk_head": (c_int, [_P, c_int, POINTER(Geom), POINTER(HeadWeights), _P, _P, c_int, c_int, _P, _P, _P]),
    "dinotrk_sample_backward": (c_int, [c_int, c_int, POINTER(Geom), _P, c_int, _P, c_int, c_int, _P, _P, _P]),
    "dinotrk_track_backward_workspace_bytes": (c_size_t, [c_int, c_int, POINTER(Geom)]),
    "dinotrk_track_backward": (c_int, [POINTER(Features), POINTER(Geom), POINTER(HeadWeights), _P, _P, c_int, _P, _P, _P, _P, _P,
                                       _P, c_int, _P, _P, _P, c_size_t, _P]),
    "dinotrk_infer_workspace_bytes": (c_size_t, [c_int, c_int, POINTER(Geom), c_int, c_int]),
    "dinotrk_infer_set_overlap": (c_int, [c_int]),
    "dinotrk_infer_set_path": (c_int, [c_int]),
    "dinotrk_infer_last_stats": (c_int, [POINTER(ctypes.c_longlong), c_int]),
    "dinotrk_infer_max_chunks": (c_size_t, [c_int, c_int, c_int]),
    "dinotrk_infer_plan": (c_int, [c_int, c_int, c_int, _P, c_int, _P, _P, c_int, _P]),
    "dinotrk_infer": (c_int, [POINTER(Features), POINTER(Geom), POINTER(HeadWeights), _P, c_int, c_float, c_float,
                              c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, c_size_t, _P]),
    "dinotrk_traj_cos_sims": (c_int, [_P, c_int, c_int, POINTER(Geom), _P, _P, c_int, _P, _P, c_size_t, _P]),
    "dinotrk_delta_workspace_bytes": (c_size_t, [c_int, c_int, c_int, POINTER(c_int)]),
    "dinotrk_delta_refine": (c_int, [_P, c_int, c_int, c_int, POINTER(c_int), POINTER(c_void_p), POINTER(c_void_p), _P,
                                     _P, _P, c_int, c_int, _P, _P, _P, c_size_t, _P]),
    "dinotrk_vit_workspace_bytes": (c_size_t, [POINTER(VitConfig), POINTER(Geom), c_int]),
    "dinotrk_vit_attention": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "dinotrk_vit_forward": (c_int, [_P, c_int, POINTER(Geom), POINTER(VitConfig), POINTER(VitWeights), _P, _P, c_size_t, _P]),
    "dinotrk_best_buddies_workspace_bytes": (c_size_t, [c_int, c_int]),
    "dinotrk_best_buddies_pairs": (c_int, [POINTER(Features), POINTER(Geom), _P, _P, c_int, _P, _P, _P, c_size_t, _P]),
    "dinotrk_bb_mutual": (c_int, [_P, _P, c_int, c_int, _P, _P]),
    "dinotrk_bb_nms": (c_int, [_P, c_int, POINTER(Geom), c_float, c_float, c_int, _P, _P, _P]),
    "dinotrk_profile_classes": (c_int, []),
    "dinotrk_profile_class_name": (c_char_p, [c_int]),
    "dinotrk_profile_enable": (None, [c_int]),
    "dinotrk_profile_collect": (c_int, [POINTER(ctypes.c_double), POINTER(c_ulonglong), c_int]),
    "dinotrk_delta_refine_allgather": (c_int, [_P, c_int, c_int, c_int, POINTER(c_int), POINTER(c_void_p), POINTER(c_void_p), _P,
                                               _P, _P, c_int, c_int, _P, _P, _P, c_size_t, POINTER(c_void_p), c_int, c_size_t, _P]),
    "dinotrk_delta_refine_tc": (c_int, [_P, c_int, c_int, c_int, POINTER(c_int), POINTER(c_void_p), POINTER(c_void_p),
                                        POINTER(c_void_p), _P, _P, _P, c_int, c_int, _P, _P, _P, c_size_t, POINTER(c_void_p),
                                        c_int, c_size_t, _P]),
    "dinotrk_peer_alloc": (c_int, [c_size_t, POINTER(c_void_p), ctypes.c_char_p]),
    "dinotrk_peer_open": (c_int, [ctypes.c_char_p, POINTER(c_void_p)]),
    "dinotrk_peer_close": (c_int, [_P]),
    "dinotrk_peer_free": (c_int, [_P]),
    "dinotrk_occlusion": (c_int, [_P, _P, _P, c_int, c_int, c_float, c_float, _P, _P]),
}


def lib_path():
    return _build.LIB_PATH


def load(build_if_missing=True):
    """Load (building in-tree if needed) libdinotrk.so.  Raises if that is impossible."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        if not build_if_missing:
            raise DinotrkError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
        _build.build()
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.dinotrk_version() < 100:
        raise DinotrkError("libdinotrk.so is older than the Python binding")
    _LIB = lib
    return lib


def check(rc, what="dinotrk"):
    if rc != 0:
        raise DinotrkError(f"{what} failed ({rc}): {load().dinotrk_last_error().decode()}")


def ptr(t):
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "device pointers must come from contiguous CUDA tensors"
    return c_void_p(t.data_ptr())


def stream_ptr(device=None):
    """Current torch stream of ``device`` (default: the current device).  The library launches on the CURRENT device,
    so callers that own a device wrap their calls in ``torch.cuda.device(dev)`` (see ``on_device``)."""
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def on_device(fn):
    """Method decorator: run with ``self._dev`` as the current CUDA device (kernels, streams and the library's
    per-device state then all belong to the model's device, whatever the caller's current device is)."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *a, **kw):
        with torch.cuda.device(self._dev):
            return fn(self, *a, **kw)
    return wrapped


def require_cuda(device):
    if not torch.cuda.is_available():
        raise DinotrkError("dino_tracker_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    dev = torch.device(device)
    if dev.type != "cuda":
        raise DinotrkError(f"dino_tracker_b200 runs on CUDA only, got device={device!r}")
    return dev


def make_features(tpc, norms, hi=None, lo=None):
    f = Features()
    f.tpc, f.norms = tpc.data_ptr(), norms.data_ptr()
    f.hi = hi.data_ptr() if hi is not None else None
    f.lo = lo.data_ptr() if lo is not None else None
    f.T, f.C = tpc.shape[0], tpc.shape[2]
    f._keep = (tpc, norms, hi, lo)  # keep the tensors alive as long as the struct
    return f


def make_geom(H, W, patch=14, stride=7, radius=35):
    g = Geom()
    check(load().dinotrk_make_geom(H, W, patch, stride, radius, ctypes.byref(g)), "make_geom")
    return g


def profile_enable(on=True):
    load().dinotrk_profile_enable(1 if on else 0)


def profile_collect():
    """-> {class name: (total ms, launches)} since the previous collect."""
    lib = load()
    n = lib.dinotrk_profile_classes()
    ms = (ctypes.c_double * n)()
    cnt = (c_ulonglong * n)()
    check(lib.dinotrk_profile_collect(ms, cnt, n), "profile_collect")
    return {lib.dinotrk_profile_class_name(i).decode(): (ms[i], int(cnt[i])) for i in range(n) if cnt[i]}


def infer_stats():
    """{anchor-phase maps, finished by the exact-window path, re-done by the full-map path, pipeline} of the last infer,
    plus the re-done maps queued by the certificate and the exact-window cells by the part count of their token box."""
    a = (ctypes.c_longlong * 8)()
    check(load().dinotrk_infer_last_stats(a, 8), "infer_last_stats")
    return {"anchor_maps": int(a[0]), "exact_window": int(a[1]), "full_map": int(a[2]), "pipeline": "exact-window" if a[3] else "full-map",
            "full_map_by_certificate": int(a[4]), "exact_window_cells_by_parts": {p: int(a[3 + p]) for p in (2, 3, 4)}}


def launch_count():
    return int(load().dinotrk_launch_count())
