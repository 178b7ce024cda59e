"""ctypes binding of libmpn_b200.so (include/mpn_abi.h).

This is the Python twin of the LuaJIT `ffi.cdef` shim in lua/mpn_ffi.lua: the reference
binds its only native code the same way (utils.lua:15-26: cdef + ffi.load of ./libnms.so).
There is NO fallback: if the CUDA library is missing or no B200 is present, loading or
context creation raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmpn_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "mpn_abi.h")

MPN_LAYER_CONV, MPN_LAYER_MAXPOOL, MPN_LAYER_AVGPOOL, MPN_LAYER_FLATTEN = 1, 2, 3, 4
MPN_MAX_DET, MPN_REC_FLOATS, MPN_DIST_ID_BYTES, MPN_MAX_BATCH = 128, 769, 128, 64      # include/mpn_abi.h
MPN_LAYER_LRN = 5       # CaffeNet local response norm: CPU-oracle plumbing config only (BASELINE configs[0]), not on the B200 path


class MpnError(RuntimeError):
    pass


class CLayer(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "kind", "in_slot", "out_slot", "cin", "cout", "kh", "kw", "stride", "pad", "relu",
        "residual_slot", "ceil_mode", "weight", "bias")]


class CTower(C.Structure):
    _fields_ = [("region", C.c_int32), ("n_levels", C.c_int32), ("level_slot", C.c_int32 * 3),
                ("level_scale", C.c_float * 3), ("pooled_w", C.c_int32), ("pooled_h", C.c_int32),
                ("normalize", C.c_int32), ("n_layers", C.c_int32), ("first_layer", C.c_int32),
                ("out_slot", C.c_int32)]


class CHead(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("col_begin", "col_len", "cout", "weight", "bias")]


class CImageTransform(C.Structure):
    """mpn_image_transform: fbcoco.ImageTransformer(mean, std, scale, swap) as plain data"""
    _fields_ = [("swap", C.c_int32 * 3), ("scale", C.c_float), ("mean", C.c_float * 3), ("std", C.c_float * 3), ("has_std", C.c_int32)]

    @staticmethod
    def of(kind: str) -> "CImageTransform":
        from . import workloads as wl
        t = CImageTransform()
        if kind == "ross":                                   # utils.RossTransformer, model_utils.lua:138-140
            t.swap[:] = [3, 2, 1]; t.scale = 255.0; t.mean[:] = wl.ROSS_MEAN; t.std[:] = [1, 1, 1]; t.has_std = 0
        elif kind == "imagenet":                             # utils.ImagenetTransformer, model_utils.lua:143-155
            t.swap[:] = [1, 2, 3]; t.scale = 1.0; t.mean[:] = wl.IMAGENET_MEAN; t.std[:] = wl.IMAGENET_STD; t.has_std = 1
        else:
            raise ValueError(f"unknown transformer {kind!r}")
        return t


class CTestOpts(C.Structure):
    """mpn_test_opts: the test-time options of Tester_FRCNN:testOne"""
    _fields_ = [("num_iter", C.c_int32), ("use_rbox_scores", C.c_int32), ("bbox_voting", C.c_int32), ("score_thresh", C.c_float),
                ("nms_thr", C.c_float), ("vote_thr", C.c_float), ("vote_score_pow", C.c_float)]


class CModelDesc(C.Structure):
    _fields_ = [("n_trunk_layers", C.c_int32), ("trunk_layers", C.POINTER(CLayer)),
                ("n_towers", C.c_int32), ("towers", C.POINTER(CTower)),
                ("n_tower_layers", C.c_int32), ("tower_layers", C.POINTER(CLayer)),
                ("n_cls_heads", C.c_int32), ("cls_heads", C.POINTER(CHead)),
                ("bbox_head", CHead), ("num_classes", C.c_int32), ("roi_variant", C.c_int32),
                ("no_softmax", C.c_int32), ("has_bbox_norm", C.c_int32),
                ("bbox_mean", C.c_float * 4), ("bbox_std", C.c_float * 4),
                ("max_rois", C.c_int32), ("max_h", C.c_int32), ("max_w", C.c_int32)]


_f32p = C.POINTER(C.c_float)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_vp = C.c_void_p

# name -> (restype, argtypes). Mirrors include/mpn_abi.h one to one (tests check the symbol set).
SIGNATURES = {
    "mpn_ctx_create": (C.c_int, [C.c_int, _vp, C.POINTER(_vp)]),
    "mpn_ctx_create_stream": (C.c_int, [C.c_int, C.c_int, C.POINTER(_vp)]),
    "mpn_ctx_stream": (_vp, [_vp]),
    "mpn_ctx_wait_ctx": (C.c_int, [_vp, _vp]),
    "mpn_ctx_destroy": (None, [_vp]),
    "mpn_last_error": (C.c_char_p, [_vp]),
    "mpn_ctx_synchronize": (C.c_int, [_vp]),
    "mpn_ctx_launch_count": (C.c_int64, [_vp]),
    "mpn_version": (C.c_char_p, []),
    "mpn_ctx_set_option": (C.c_int, [_vp, C.c_char_p, C.c_int64]),
    "mpn_ctx_profile_begin": (C.c_int, [_vp]),
    "mpn_ctx_profile_end": (C.c_int, [_vp, C.POINTER(C.c_double), _i64p]),
    "mpn_ctx_timeline_begin": (C.c_int, [_vp, C.c_int32]),
    "mpn_ctx_timeline_end": (C.c_int, [_vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), _i32p]),
    "mpn_nms": (C.c_int, [_vp, _vp, C.c_int64, C.c_float, _vp, _i64p]),
    "mpn_nms_batched": (C.c_int, [_vp, _vp, _i64p, C.c_int64, C.c_float, _vp, _i64p]),
    "mpn_nms_batched_dev": (C.c_int, [_vp, _vp, _i64p, C.c_int64, C.c_float, _vp, _vp]),
    "mpn_nms_dense": (C.c_int, [_vp, _vp, C.c_int64, C.c_float, _vp, _i64p]),
    "mpn_bbox_vote": (C.c_int, [_vp, _vp, C.c_int64, _vp, C.c_int64, C.c_float, _vp]),
    "mpn_foveal": (C.c_int, [_vp, _vp, C.c_int64, _vp]),
    "mpn_context_region": (C.c_int, [_vp, _vp, C.c_int64, C.c_float, _vp]),
    "mpn_bbox_norm": (C.c_int, [_vp, _vp, C.c_int64, C.c_int64, _vp, _vp]),
    "mpn_foveal_dev": (C.c_int, [_vp, _vp, C.c_int64, _vp]),
    "mpn_context_region_dev": (C.c_int, [_vp, _vp, C.c_int64, C.c_float, _vp]),
    "mpn_bbox_norm_dev": (C.c_int, [_vp, _vp, C.c_int64, C.c_int64, _vp, _vp]),
    "mpn_bbox_decode": (C.c_int, [_vp, _vp, _vp, C.c_int64, C.c_int64, _vp]),
    "mpn_roi_pool": (C.c_int, [_vp, _vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, _vp, C.c_int64,
                               C.c_int32, C.c_int32, C.c_float, C.c_int32, _vp, _vp]),
    "mpn_roi_pool_dev": (C.c_int, [_vp, _vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, _vp, C.c_int64,
                                   C.c_int32, C.c_int32, C.c_float, C.c_int32, _vp, _vp]),
    "mpn_get_images_size": (C.c_int, [C.c_int32, C.c_int32, C.c_double, C.c_double, _i32p, _i32p, C.POINTER(C.c_double)]),
    "mpn_get_images": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_int32, C.c_int32, _vp]),
    "mpn_get_images_dev": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_int32, C.c_int32, _vp]),
    "mpn_get_images_u8": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_int32, C.c_int32, _vp]),
    "mpn_get_images_u8_dev": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_int32, C.c_int32, _vp]),
    "mpn_get_images_batch_size": (C.c_int, [C.c_int32, _i32p, _i32p, C.c_double, C.c_double, _i32p, _i32p, C.POINTER(C.c_double), _i32p,
                                            _i32p]),
    "mpn_get_images_batch_u8": (C.c_int, [_vp, _vp, C.c_int32, _i32p, _i32p, _vp, C.c_double, C.c_double, _vp]),
    "mpn_get_images_batch_u8_dev": (C.c_int, [_vp, _vp, C.c_int32, _i32p, _i32p, _vp, C.c_double, C.c_double, _vp]),
    "mpn_model_detect_nms_batch_submit_u8": (C.c_int, [_vp, _vp, C.c_int32, _i32p, _i32p, _vp, C.c_double, C.c_double, _vp, _i64p, C.c_float,
                                                       C.c_float, _vp, _vp, _vp, _vp, _i32p]),
    "mpn_model_detect_nms_submit_u8": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_double, C.c_double, _vp, C.c_int64, C.c_float, C.c_float,
                                                 _vp, _vp, _vp, _vp, _i32p]),
    "mpn_model_trunk_image": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_double, C.c_double, C.POINTER(C.c_double), _i32p, _i32p]),
    "mpn_model_create": (C.c_int, [_vp, C.POINTER(CModelDesc), C.POINTER(_vp), _i64p, C.c_int32, C.POINTER(_vp)]),
    "mpn_model_destroy": (None, [_vp]),
    "mpn_model_trunk": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32]),
    "mpn_model_trunk_dev": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32]),
    "mpn_model_trunk_batch": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, C.c_int32]),
    "mpn_model_trunk_batch_dev": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, C.c_int32]),
    "mpn_model_detect_nms_batch": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, C.c_int32, _vp, _i64p, _vp, _vp, _vp, C.c_float, C.c_float,
                                             _vp, _vp, _vp, _vp]),
    "mpn_model_detect_nms_batch_dev": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, C.c_int32, _vp, _i64p, _vp, _vp, _vp, C.c_float,
                                                 C.c_float, _vp, _vp, _vp, _vp]),
    "mpn_model_heads": (C.c_int, [_vp, _vp, C.c_int64, _vp, _vp]),
    "mpn_model_heads_dev": (C.c_int, [_vp, _vp, C.c_int64, _vp, _vp]),
    "mpn_model_detect": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_int64, C.c_float, C.c_int32, _vp, _vp]),
    "mpn_model_detect_nms": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_int64, C.c_float, C.c_float,
                                       C.c_float, C.c_float, C.c_float, _vp, _vp, _vp, _vp]),
    "mpn_model_detect_nms_submit": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_int64, C.c_float, C.c_float,
                                              C.c_float, C.c_float, C.c_float, _vp, _vp, _vp, _vp, _i32p]),
    "mpn_model_detect_nms_wait": (C.c_int, [_vp, C.c_int32]),
    "mpn_model_test_one": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_int64, C.c_float, C.c_float, C.c_float, C.POINTER(CTestOpts),
                                     _vp, _vp, _vp, _vp, _vp]),
    "mpn_model_detect_nms_dev": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_int64, C.c_float, C.c_float,
                                           C.c_float, C.c_float, C.c_float, _vp, _vp, _vp, _vp]),
    "mpn_post_detect_dev": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int64, C.c_int32, _vp, _vp, C.c_float, C.c_float, C.c_float, C.c_float,
                                      C.c_int32, C.c_int32, _vp, _vp, _vp]),
    "mpn_pack_detections_dev": (C.c_int, [_vp, _vp, _vp, C.c_int64, C.c_int32, _vp, _vp, C.c_int64, C.c_int32, _vp]),
    "mpn_pack_detections": (C.c_int, [_vp, _vp, _vp, C.c_int64, C.c_int32, _vp, _vp, C.c_int64, C.c_int32, _vp]),
    "mpn_select_boxes": (C.c_int, [_vp, _vp, _vp, C.c_int64, C.c_int32, _vp, _vp, _vp]),
    "mpn_select_boxes_dev": (C.c_int, [_vp, _vp, _vp, C.c_int64, C.c_int32, _vp, _vp, _vp]),
    "mpn_model_set_detection_sink": (C.c_int, [_vp, _vp, C.c_int64, C.c_int32]),
    "mpn_model_detection_sink_count": (C.c_int, [_vp, _i64p]),
    "mpn_dist_unique_id": (C.c_int, [_vp, _vp]),
    "mpn_dist_init": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32]),
    "mpn_dist_world": (C.c_int, [_vp, _i32p, _i32p]),
    "mpn_dist_all_gather_dev": (C.c_int, [_vp, _vp, C.c_int64, _vp]),
    "mpn_dist_all_gather": (C.c_int, [_vp, _vp, C.c_int64, _vp]),
    "mpn_dist_destroy": (C.c_int, [_vp]),
    "mpn_dist_nccl_version": (C.c_int, [_vp, _i32p]),
    "mpn_model_get_pooled": (C.c_int, [_vp, C.c_int32, C.c_int64, C.c_int64, _vp, C.c_int64, _i64p, _i32p, _i32p]),
    "mpn_model_get_trunk_slot": (C.c_int, [_vp, C.c_int32, _vp, C.c_int64, _i32p, _i32p, _i32p]),
    "mpn_model_set_conv_impl": (C.c_int, [_vp, C.c_int32]),
    "mpn_model_last_flops": (C.c_int, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "mpn_gemm_bench": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.POINTER(C.c_double), _i32p, _i32p, _i32p]),
    "mpn_conv_bench": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                 C.POINTER(C.c_double), _i32p, _i32p, _i32p, C.POINTER(C.c_uint64)]),
    "mpn_debug_plan": (C.c_int, [C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _i32p]),
    "mpn_debug_segwalk": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _i32p, C.c_int32, _i32p]),
    "mpn_gemm_check": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, _vp]),
    "mpn_conv_check": (C.c_int, [_vp, _vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, _vp, _vp, C.c_int64,
                                 C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _vp]),
}

_lib = None


def load_library():
    """dlopen libmpn_b200.so and bind every symbol of the ABI. Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MpnError(
            f"{LIB_PATH} is missing: build it with `make` (or `python -c 'import __graft_entry__ as g; g.build()'`). "
            "There is no CPU or PyTorch fallback for this path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)     # AttributeError if the .so does not export what the header declares
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(a) -> Optional[int]:
    """Raw address of a numpy array / torch tensor / int / None."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    raise TypeError(f"cannot take the address of {type(a)}")


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def _raw_batch(ims, scale: float, max_size: float):
    """host-side checks of N raw images for the batched getImages -> (list of contiguous H0 x W0 x 3 uint8 arrays,
    H0 int32 N, W0 int32 N, [(h_i, w_i, im_scale_i)], canvas (H, W)); raises ValueError before any library call. The sizes
    follow image_detect's rule, which tests/test_batch_raw_cpu.py pins to mpn_get_images_batch_size."""
    from .image_detect import _get_images_size
    if not isinstance(ims, (list, tuple)) or not 1 <= len(ims) <= MPN_MAX_BATCH:
        raise ValueError(f"expected a list of 1..{MPN_MAX_BATCH} raw images")
    out = []
    for i, im in enumerate(ims):
        if not isinstance(im, np.ndarray) or im.dtype != np.uint8 or im.ndim != 3 or im.shape[2] != 3 or im.shape[0] < 1 or im.shape[1] < 1:
            raise ValueError(f"image {i}: expected an H0 x W0 x 3 uint8 array")
        out.append(np.ascontiguousarray(im))
    if not (scale > 0 and max_size > 0):
        raise ValueError("scale and max_size must be > 0")
    H0 = np.array([im.shape[0] for im in out], np.int32)
    W0 = np.array([im.shape[1] for im in out], np.int32)
    sizes = [_get_images_size(int(h), int(w), scale, max_size) for h, w in zip(H0, W0)]
    H, W = max(h for h, _, _ in sizes), max(w for _, w, _ in sizes)
    if min(min(h, w) for h, w, _ in sizes) < 1 or H > 65535:
        raise ValueError(f"scaled sizes out of range: canvas {H} x {W}")
    return out, H0, W0, sizes, (H, W)


class Context:
    """One mpn_ctx: (thread, device, stream). Mirrors the one-replica-per-thread model of
    test_runner.lua:55-66."""

    def __init__(self, device: int = 0, stream: Optional[int] = None, own_stream: bool = False, priority: int = 0):
        """stream: a cudaStream_t handle of the caller's (None = the legacy default stream); own_stream=True: the ctx
        creates a non-blocking stream of its own (mpn_ctx_create_stream) — what several replicas on one GPU use"""
        self.lib = load_library()
        h = _vp()
        if own_stream:
            rc = self.lib.mpn_ctx_create_stream(int(device), int(priority), C.byref(h))
        else:
            rc = self.lib.mpn_ctx_create(int(device), _vp(stream) if stream else None, C.byref(h))
        if rc != 0:
            raise MpnError(f"mpn_ctx_create failed ({rc}): {self.lib.mpn_last_error(None).decode()}")
        self.h = h
        self.device = device
        self._models = []          # weak references to the live Models: closed before the ctx (they dereference it)

    def check(self, rc: int, what: str = ""):
        if rc != 0:
            raise MpnError(f"{what} failed ({rc}): {self.lib.mpn_last_error(self.h).decode()}")

    def synchronize(self):
        self.check(self.lib.mpn_ctx_synchronize(self.h), "synchronize")

    @property
    def stream_handle(self) -> int:
        """the ctx's cudaStream_t as an integer (0 = the legacy default stream)"""
        return int(self.lib.mpn_ctx_stream(self.h) or 0)

    def wait_ctx(self, other: "Context"):
        """everything enqueued on this ctx from now on waits for what `other` has enqueued so far (mpn_ctx_wait_ctx)"""
        self.check(self.lib.mpn_ctx_wait_ctx(self.h, other.h), "mpn_ctx_wait_ctx")

    def set_option(self, name: str, value: int):
        self.check(self.lib.mpn_ctx_set_option(self.h, name.encode(), int(value)), "mpn_ctx_set_option")

    @property
    def launch_count(self) -> int:
        return int(self.lib.mpn_ctx_launch_count(self.h))

    PROFILE_CATS = ("conv_gemm_tc", "conv_direct", "roi_pool", "nms", "elementwise", "pool")

    def profile_begin(self):
        self.check(self.lib.mpn_ctx_profile_begin(self.h), "profile_begin")

    def profile_end(self):
        ms = (C.c_double * 6)()
        n = (C.c_int64 * 6)()
        self.check(self.lib.mpn_ctx_profile_end(self.h, ms, n), "profile_end")
        return {k: (ms[i], int(n[i])) for i, k in enumerate(self.PROFILE_CATS)}

    def close(self):
        if getattr(self, "h", None):
            for ref in list(getattr(self, "_models", [])):      # mpn_model_destroy touches the ctx: models go first
                m = ref()
                if m is not None:
                    m.close()
            self._models = []
            self.lib.mpn_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- the end-of-run collective (SURVEY 8e) ----------------------------------------------
    def dist_unique_id(self) -> bytes:
        buf = (C.c_uint8 * MPN_DIST_ID_BYTES)()
        self.check(self.lib.mpn_dist_unique_id(self.h, buf), "mpn_dist_unique_id")
        return bytes(buf)

    def dist_init(self, unique_id: bytes, rank: int, world: int):
        assert len(unique_id) == MPN_DIST_ID_BYTES
        buf = (C.c_uint8 * MPN_DIST_ID_BYTES).from_buffer_copy(unique_id)
        self.check(self.lib.mpn_dist_init(self.h, buf, int(rank), int(world)), "mpn_dist_init")

    def dist_world(self):
        r, w = C.c_int32(), C.c_int32()
        self.check(self.lib.mpn_dist_world(self.h, C.byref(r), C.byref(w)), "mpn_dist_world")
        return r.value, w.value

    def dist_all_gather_dev(self, send_dev, n_floats: int, recv_dev):
        self.check(self.lib.mpn_dist_all_gather_dev(self.h, _ptr(send_dev), int(n_floats), _ptr(recv_dev)), "mpn_dist_all_gather_dev")

    def dist_all_gather(self, send_dev, n_floats: int) -> np.ndarray:
        """device records of this rank -> host array world x n_floats (synchronous)"""
        _, w = self.dist_world()
        out = np.empty((w, int(n_floats)), np.float32)
        self.check(self.lib.mpn_dist_all_gather(self.h, _ptr(send_dev), int(n_floats), _ptr(out)), "mpn_dist_all_gather")
        return out

    def dist_destroy(self):
        self.check(self.lib.mpn_dist_destroy(self.h), "mpn_dist_destroy")

    # ---- after NMS ---------------------------------------------------------------------------
    def pack_detections(self, scores, bboxes, keep_idx, keep_counts, top_k: int = 100) -> np.ndarray:
        """utils.keep_top_k + the fixed-size record (include/mpn_abi.h): scores R x C, bboxes R x 4C, keep_idx (C-1) x cap,
        keep_counts C-1 -> MPN_REC_FLOATS floats"""
        s, b = _f32(scores), _f32(bboxes)
        k = np.ascontiguousarray(keep_idx, dtype=np.int32); c = np.ascontiguousarray(keep_counts, dtype=np.int32)
        rec = np.empty(MPN_REC_FLOATS, np.float32)
        self.check(self.lib.mpn_pack_detections(self.h, _ptr(s), _ptr(b), s.shape[0], s.shape[1], _ptr(k), _ptr(c), k.shape[1],
                                                int(top_k), _ptr(rec)), "mpn_pack_detections")
        return rec

    def select_boxes(self, classes, ys, mean=None, std=None) -> np.ndarray:
        """nn.SelectBoxes:updateOutput (modules/SelectBoxes.lua:26-56)"""
        s, y = _f32(classes), _f32(ys)
        out = np.empty((s.shape[0], 4), np.float32)
        m = None if mean is None else _f32(mean).reshape(4)
        sd = None if std is None else _f32(std).reshape(4)
        self.check(self.lib.mpn_select_boxes(self.h, _ptr(s), _ptr(y), s.shape[0], s.shape[1], _ptr(m), _ptr(sd), _ptr(out)),
                   "mpn_select_boxes")
        return out

    # ---- NMS family -------------------------------------------------------------------------
    def nms(self, scored_boxes, thr: float) -> np.ndarray:
        sb = _f32(scored_boxes).reshape(-1, 5)
        n = sb.shape[0]
        keep = np.empty(max(n, 1), dtype=np.int32)
        cnt = C.c_int64(0)
        self.check(self.lib.mpn_nms(self.h, _ptr(sb), n, float(thr), _ptr(keep), C.byref(cnt)), "mpn_nms")
        return keep[: cnt.value].copy()

    def nms_batched(self, scored_boxes, seg_offsets: Sequence[int], thr: float) -> List[np.ndarray]:
        sb = _f32(scored_boxes).reshape(-1, 5)
        offs = np.ascontiguousarray(seg_offsets, dtype=np.int64)
        nseg = len(offs) - 1
        keep = np.empty(max(sb.shape[0], 1), dtype=np.int32)
        counts = np.zeros(max(nseg, 1), dtype=np.int64)
        self.check(self.lib.mpn_nms_batched(self.h, _ptr(sb), offs.ctypes.data_as(_i64p), nseg, float(thr), _ptr(keep),
                                            counts.ctypes.data_as(_i64p)), "mpn_nms_batched")
        return [keep[offs[s]: offs[s] + counts[s]].copy() for s in range(nseg)]

    def nms_dense(self, scored_boxes, thr: float) -> np.ndarray:
        sb = _f32(scored_boxes).reshape(-1, 5)
        n = sb.shape[0]
        pick = np.empty(max(n, 1), dtype=np.int32)
        cnt = C.c_int64(0)
        self.check(self.lib.mpn_nms_dense(self.h, _ptr(sb), n, float(thr), _ptr(pick), C.byref(cnt)), "mpn_nms_dense")
        return pick[: cnt.value].copy()

    def bbox_vote(self, nms_boxes, scored_boxes, thr: float) -> np.ndarray:
        nb = _f32(nms_boxes).reshape(-1, 5)
        sb = _f32(scored_boxes).reshape(-1, 5)
        res = np.zeros_like(nb)
        self.check(self.lib.mpn_bbox_vote(self.h, _ptr(nb), nb.shape[0], _ptr(sb), sb.shape[0], float(thr), _ptr(res)),
                   "mpn_bbox_vote")
        return res

    # ---- region modules ---------------------------------------------------------------------
    def foveal(self, rois) -> np.ndarray:
        r = _f32(rois)
        out = np.empty((r.shape[0] * 4, 5), dtype=np.float32)
        self.check(self.lib.mpn_foveal(self.h, _ptr(r), r.shape[0], _ptr(out)), "mpn_foveal")
        return out

    def context_region(self, rois, scale: float) -> np.ndarray:
        r = _f32(rois)
        out = np.empty_like(r)
        self.check(self.lib.mpn_context_region(self.h, _ptr(r), r.shape[0], float(scale), _ptr(out)), "mpn_context_region")
        return out

    # device-resident module ops (torch CUDA tensors or raw addresses in, stream-ordered, nothing copied)
    def foveal_dev(self, rois_dev, R: int, out_dev):
        self.check(self.lib.mpn_foveal_dev(self.h, _ptr(rois_dev), int(R), _ptr(out_dev)), "mpn_foveal_dev")

    def context_region_dev(self, rois_dev, R: int, scale: float, out_dev):
        self.check(self.lib.mpn_context_region_dev(self.h, _ptr(rois_dev), int(R), float(scale), _ptr(out_dev)), "mpn_context_region_dev")

    def bbox_norm_dev(self, deltas_dev, R: int, C4: int, mean, std):
        m, s = _f32(mean).reshape(4), _f32(std).reshape(4)
        self.check(self.lib.mpn_bbox_norm_dev(self.h, _ptr(deltas_dev), int(R), int(C4), _ptr(m), _ptr(s)), "mpn_bbox_norm_dev")

    def get_images(self, im, kind: str, scale: float = 600, max_size: float = 1000):
        """getImages on the device (ImageDetect.lua:22-52): raw 3 x H0 x W0 image -> (transformed + scaled image, im_scale)"""
        im = _f32(im)
        if im.ndim != 3 or im.shape[0] != 3:
            raise ValueError("ImageTransformer expects a 3 x H x W image")
        h, w, s = C.c_int32(), C.c_int32(), C.c_double()
        self.check(self.lib.mpn_get_images_size(im.shape[1], im.shape[2], float(scale), float(max_size), C.byref(h), C.byref(w), C.byref(s)),
                   "mpn_get_images_size")
        out = np.empty((3, h.value, w.value), np.float32)
        tf = CImageTransform.of(kind)
        self.check(self.lib.mpn_get_images(self.h, _ptr(im), im.shape[1], im.shape[2], C.addressof(tf), h.value, w.value, _ptr(out)),
                   "mpn_get_images")
        return out, float(s.value)

    def get_images_u8(self, im_hwc_u8, kind: str, scale: float = 600, max_size: float = 1000):
        """getImages on the device from the decoder's bytes (H0 x W0 x 3 uint8 RGB) -> (transformed + scaled image, im_scale)"""
        im = np.ascontiguousarray(im_hwc_u8, dtype=np.uint8)
        if im.ndim != 3 or im.shape[2] != 3:
            raise ValueError("expected an H x W x 3 uint8 image")
        h, w, s = C.c_int32(), C.c_int32(), C.c_double()
        self.check(self.lib.mpn_get_images_size(im.shape[0], im.shape[1], float(scale), float(max_size), C.byref(h), C.byref(w), C.byref(s)),
                   "mpn_get_images_size")
        out = np.empty((3, h.value, w.value), np.float32)
        tf = CImageTransform.of(kind)
        self.check(self.lib.mpn_get_images_u8(self.h, _ptr(im), im.shape[0], im.shape[1], C.addressof(tf), h.value, w.value, _ptr(out)),
                   "mpn_get_images_u8")
        return out, float(s.value)

    def get_images_batch_u8(self, ims, kind: str, scale: float = 600, max_size: float = 1000):
        """getImages of N raw H0 x W0 x 3 uint8 images of any sizes into one zero-padded canvas on the device (one launch)
        -> (batch N x 3 x H x W, [im_scale_i], [(h_i, w_i)]); image i fills [0, h_i) x [0, w_i) of its plane, the rest is 0"""
        ims, H0, W0, sizes, (H, W) = _raw_batch(ims, scale, max_size)
        tf = CImageTransform.of(kind)
        raw = np.concatenate([im.reshape(-1) for im in ims])
        out = np.empty((len(ims), 3, H, W), np.float32)
        self.check(self.lib.mpn_get_images_batch_u8(self.h, _ptr(raw), len(ims), H0.ctypes.data_as(_i32p), W0.ctypes.data_as(_i32p),
                                                    C.addressof(tf), float(scale), float(max_size), _ptr(out)), "mpn_get_images_batch_u8")
        return out, [s for _, _, s in sizes], [(h, w) for h, w, _ in sizes]

    def bbox_norm(self, deltas, mean, std) -> np.ndarray:
        d = _f32(deltas).copy()
        m, s = _f32(mean).reshape(4), _f32(std).reshape(4)
        self.check(self.lib.mpn_bbox_norm(self.h, _ptr(d), d.shape[0], d.shape[1], _ptr(m), _ptr(s)), "mpn_bbox_norm")
        return d

    def bbox_decode(self, deltas, boxes) -> np.ndarray:
        d, b = _f32(deltas), _f32(boxes)
        out = np.empty_like(d)
        self.check(self.lib.mpn_bbox_decode(self.h, _ptr(d), _ptr(b), d.shape[0], d.shape[1] // 4, _ptr(out)), "mpn_bbox_decode")
        return out

    def roi_pool(self, fmap, rois, pw: int, ph: int, scale: float, variant: int = 2, with_argmax: bool = False):
        f, r = _f32(fmap), _f32(rois)
        n, c, h, w = f.shape
        out = np.empty((r.shape[0], c, ph, pw), dtype=np.float32)
        am = np.empty(out.shape, dtype=np.int32) if with_argmax else None
        self.check(self.lib.mpn_roi_pool(self.h, _ptr(f), n, c, h, w, _ptr(r), r.shape[0], pw, ph, float(scale), variant,
                                         _ptr(out), _ptr(am)), "mpn_roi_pool")
        return (out, am) if with_argmax else out

    # ---- engine checks ----------------------------------------------------------------------
    def gemm_check(self, A, B, bias=None, relu=False, impl=0) -> np.ndarray:
        A, B = _f32(A), _f32(B)
        m, k = A.shape
        n = B.shape[0]
        bias = None if bias is None else _f32(bias)
        out = np.empty((m, n), dtype=np.float32)
        self.check(self.lib.mpn_gemm_check(self.h, _ptr(A), _ptr(B), _ptr(bias), m, n, k, int(relu), impl, _ptr(out)), "mpn_gemm_check")
        return out

    def gemm_bench(self, M, N, K, iters=20):
        ms = C.c_double(); bn = C.c_int32(); cg = C.c_int32(); sk = C.c_int32()
        self.check(self.lib.mpn_gemm_bench(self.h, M, N, K, iters, C.byref(ms), C.byref(bn), C.byref(cg), C.byref(sk)), "mpn_gemm_bench")
        return ms.value, bn.value, cg.value, sk.value

    def conv_bench(self, N, Cin, H, W, Cout, k=3, stride=1, pad=1, iters=20):
        ms = C.c_double(); bn = C.c_int32(); cg = C.c_int32(); mode = C.c_int32(); dbg = (C.c_uint64 * 16)()
        self.check(self.lib.mpn_conv_bench(self.h, N, Cin, H, W, Cout, k, stride, pad, iters, C.byref(ms), C.byref(bn), C.byref(cg),
                                           C.byref(mode), dbg), "mpn_conv_bench")
        return ms.value, bn.value, cg.value, mode.value, [int(x) for x in dbg]

    def conv_check(self, x, w, bias=None, stride=1, pad=0, relu=False, impl=0) -> np.ndarray:
        x, w = _f32(x), _f32(w)
        n, cin, h, ww = x.shape
        cout, _, kh, kw = w.shape
        bias = None if bias is None else _f32(bias)
        ho, wo = (h + 2 * pad - kh) // stride + 1, (ww + 2 * pad - kw) // stride + 1
        y = np.empty((n, cout, ho, wo), dtype=np.float32)
        self.check(self.lib.mpn_conv_check(self.h, _ptr(x), n, cin, h, ww, _ptr(w), _ptr(bias), cout, kh, kw, stride, pad,
                                           int(relu), impl, _ptr(y)), "mpn_conv_check")
        return y


# ------------------------------------------------------------------------------------------
# model description (Python twin of mpn_model_desc) — built by multipathnet_b200.models
@dataclass
class Layer:
    kind: int
    in_slot: int
    out_slot: int
    cin: int = 0
    cout: int = 0
    kh: int = 1
    kw: int = 1
    stride: int = 1
    pad: int = 0
    relu: int = 0
    residual_slot: int = -1
    ceil_mode: int = 0
    weight: int = -1
    bias: int = -1
    groups: int = 1          # grouped conv (CaffeNet conv2/4/5): CPU-oracle plumbing config only

    def to_c(self) -> CLayer:
        if self.groups != 1 or self.kind == MPN_LAYER_LRN:
            raise MpnError("grouped convolution / LRN (CaffeNet, BASELINE configs[0]) is the CPU plumbing configuration; "
                           "it is not part of the B200 path")
        return CLayer(self.kind, self.in_slot, self.out_slot, self.cin, self.cout, self.kh, self.kw, self.stride,
                      self.pad, self.relu, self.residual_slot, self.ceil_mode, self.weight, self.bias)


@dataclass
class Tower:
    region: int
    levels: List[tuple]            # [(trunk_slot, spatial_scale), ...] channel-concat order
    pooled_w: int
    pooled_h: int
    normalize: int
    layers: List[Layer]
    out_slot: int


@dataclass
class Head:
    col_begin: int
    col_len: int
    cout: int
    weight: int
    bias: int

    def to_c(self) -> CHead:
        return CHead(self.col_begin, self.col_len, self.cout, self.weight, self.bias)


@dataclass
class ModelSpec:
    name: str
    trunk_layers: List[Layer]
    towers: List[Tower]
    cls_heads: List[Head]
    bbox_head: Head
    num_classes: int
    weights: List[np.ndarray]
    roi_variant: int = 2
    no_softmax: int = 0
    has_bbox_norm: int = 1
    bbox_mean: tuple = (0.0, 0.0, 0.0, 0.0)
    bbox_std: tuple = (0.1, 0.1, 0.2, 0.2)
    transformer: str = "ross"      # "ross" | "imagenet"  (model_utils.lua:138-155)
    taps: dict = field(default_factory=dict)   # name -> trunk slot, for tests


class Model:
    """mpn_model handle: the B200 replacement for the nn.Sequential graph a model file returns."""

    @staticmethod
    def build_desc(spec: ModelSpec, max_rois: int = 2048, max_h: int = 1024, max_w: int = 1344):
        """ModelSpec -> (mpn_model_desc, keep-alive objects). Pure host code (no GPU needed)."""
        trunk = (CLayer * len(spec.trunk_layers))(*[l.to_c() for l in spec.trunk_layers])
        tl: List[Layer] = []
        ctowers = []
        for t in spec.towers:
            ct = CTower()
            ct.region, ct.n_levels = t.region, len(t.levels)
            for i, (slot, sc) in enumerate(t.levels):
                ct.level_slot[i] = slot
                ct.level_scale[i] = sc
            ct.pooled_w, ct.pooled_h, ct.normalize = t.pooled_w, t.pooled_h, t.normalize
            ct.n_layers, ct.first_layer, ct.out_slot = len(t.layers), len(tl), t.out_slot
            tl.extend(t.layers)
            ctowers.append(ct)
        towers = (CTower * len(ctowers))(*ctowers)
        tower_layers = (CLayer * max(len(tl), 1))(*[l.to_c() for l in tl])
        heads = (CHead * len(spec.cls_heads))(*[h.to_c() for h in spec.cls_heads])
        d = CModelDesc()
        d.n_trunk_layers, d.trunk_layers = len(spec.trunk_layers), trunk
        d.n_towers, d.towers = len(ctowers), towers
        d.n_tower_layers, d.tower_layers = len(tl), tower_layers
        d.n_cls_heads, d.cls_heads = len(spec.cls_heads), heads
        d.bbox_head = spec.bbox_head.to_c()
        d.num_classes, d.roi_variant = spec.num_classes, spec.roi_variant
        d.no_softmax, d.has_bbox_norm = spec.no_softmax, spec.has_bbox_norm
        for i in range(4):
            d.bbox_mean[i] = spec.bbox_mean[i]
            d.bbox_std[i] = spec.bbox_std[i]
        d.max_rois, d.max_h, d.max_w = max_rois, max_h, max_w
        return d, (trunk, towers, tower_layers, heads)

    def __init__(self, ctx: Context, spec: ModelSpec, max_rois: int = 2048, max_h: int = 1024, max_w: int = 1344):
        self.ctx, self.spec = ctx, spec
        lib = ctx.lib
        d, self._keep = Model.build_desc(spec, max_rois, max_h, max_w)
        ws = [np.ascontiguousarray(w, dtype=np.float32) for w in spec.weights]
        wptrs = (_vp * len(ws))(*[w.ctypes.data for w in ws])
        wn = np.array([w.size for w in ws], dtype=np.int64)
        h = _vp()
        ctx.check(lib.mpn_model_create(ctx.h, C.byref(d), wptrs, wn.ctypes.data_as(_i64p), len(ws), C.byref(h)),
                  "mpn_model_create")
        self.h = h
        self.C = spec.num_classes
        self.max_rois = int(max_rois)
        self.max_h, self.max_w = int(max_h), int(max_w)
        self._trunk_n = 1                  # images of the last trunk forward (the leading size of trunk_slot)
        import weakref
        ctx._models.append(weakref.ref(self))

    def close(self):
        if getattr(self, "h", None):
            if getattr(self.ctx, "h", None):               # a closed ctx has already closed its models
                self.ctx.lib.mpn_model_destroy(self.h)
            self.h = None

    def set_detection_sink(self, records_dev, capacity: int, top_k: int = 100):
        """every later detect_nms* call appends the image's packed record to records_dev (a CUDA tensor / address)"""
        self.ctx.check(self.ctx.lib.mpn_model_set_detection_sink(self.h, _ptr(records_dev), int(capacity), int(top_k)),
                       "mpn_model_set_detection_sink")

    def detection_sink_count(self) -> int:
        n = C.c_int64()
        self.ctx.check(self.ctx.lib.mpn_model_detection_sink_count(self.h, C.byref(n)), "mpn_model_detection_sink_count")
        return int(n.value)

    def pooled(self, tower: int, r0: int = 0, n: Optional[int] = None) -> np.ndarray:
        """rows [r0, r0+n) of the pooled tensor the last heads/detect call fed to `tower`: n x bins x Ctot fp32"""
        R, bins, ct = C.c_int64(), C.c_int32(), C.c_int32()
        self.ctx.check(self.ctx.lib.mpn_model_get_pooled(self.h, tower, 0, 0, None, 0, C.byref(R), C.byref(bins), C.byref(ct)), "get_pooled")
        n = R.value - r0 if n is None else n
        out = np.empty((n, bins.value, ct.value), np.float32)
        self.ctx.check(self.ctx.lib.mpn_model_get_pooled(self.h, tower, r0, n, _ptr(out), out.size, C.byref(R), C.byref(bins), C.byref(ct)),
                       "get_pooled")
        return out

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_conv_impl(self, impl: int):
        self.ctx.check(self.ctx.lib.mpn_model_set_conv_impl(self.h, impl), "set_conv_impl")

    def trunk(self, image_chw):
        im = _f32(image_chw)
        assert im.ndim == 3 and im.shape[0] == 3
        self._trunk_n = 1
        self.ctx.check(self.ctx.lib.mpn_model_trunk(self.h, _ptr(im), im.shape[1], im.shape[2]), "mpn_model_trunk")

    def trunk_batch(self, images_nchw):
        """model:get(1):forward on N x 3 x H x W images of one (padded) size; ROI rows then pick their image by column 0"""
        im = _f32(images_nchw)
        if im.ndim != 4 or im.shape[1] != 3 or im.shape[0] < 1 or im.shape[0] > MPN_MAX_BATCH:
            raise ValueError(f"trunk_batch expects N x 3 x H x W images with 1 <= N <= {MPN_MAX_BATCH}")
        self._trunk_n = im.shape[0]
        self.ctx.check(self.ctx.lib.mpn_model_trunk_batch(self.h, _ptr(im), im.shape[0], im.shape[2], im.shape[3]), "mpn_model_trunk_batch")

    def trunk_image(self, raw_image_chw, kind: str, scale: float = 600, max_size: float = 1000):
        """getImages + trunk on the device from the RAW image (SURVEY 8f-1) -> (im_scale, h, w)"""
        im = _f32(raw_image_chw)
        if im.ndim != 3 or im.shape[0] != 3:
            raise ValueError("ImageTransformer expects a 3 x H x W image")
        h, w, s = C.c_int32(), C.c_int32(), C.c_double()
        tf = CImageTransform.of(kind)
        self._trunk_n = 1
        self.ctx.check(self.ctx.lib.mpn_model_trunk_image(self.h, _ptr(im), im.shape[1], im.shape[2], C.addressof(tf), float(scale),
                                                          float(max_size), C.byref(s), C.byref(h), C.byref(w)), "mpn_model_trunk_image")
        return float(s.value), h.value, w.value

    def heads(self, rois):
        r = _f32(rois)
        n = r.shape[0]
        cls = np.empty((n, self.C), dtype=np.float32)
        bbox = np.empty((n, 4 * self.C), dtype=np.float32)
        self.ctx.check(self.ctx.lib.mpn_model_heads(self.h, _ptr(r), n, _ptr(cls), _ptr(bbox)), "mpn_model_heads")
        return cls, bbox

    def forward(self, images, rois):
        """model:forward{images, rois} (eval mode): images 3 x H x W, or N x 3 x H x W with ROI rows [n, x1, y1, x2, y2]
        naming their image by the 1-based n."""
        if np.ndim(images) == 4:
            self.trunk_batch(images)
        else:
            self.trunk(images)
        return self.heads(rois)

    def detect(self, image_chw, boxes, im_scale: float, recompute_features: bool = True):
        b = _f32(boxes)
        n = b.shape[0]
        im = None if image_chw is None else _f32(image_chw)
        scores = np.empty((n, self.C), dtype=np.float32)
        bboxes = np.empty((n, 4 * self.C), dtype=np.float32)
        H, W = (im.shape[1], im.shape[2]) if im is not None else (0, 0)
        if recompute_features:
            self._trunk_n = 1
        self.ctx.check(self.ctx.lib.mpn_model_detect(self.h, _ptr(im), H, W, _ptr(b), n, float(im_scale),
                                                     int(recompute_features), _ptr(scores), _ptr(bboxes)), "mpn_model_detect")
        return scores, bboxes

    def detect_nms(self, image_chw, boxes, im_scale: float, W0: float, H0: float, score_thresh: float = -1.5,
                   nms_thr: float = 0.3, want_raw: bool = True):
        im, b = _f32(image_chw), _f32(boxes)
        n = b.shape[0]
        scores = np.empty((n, self.C), dtype=np.float32) if want_raw else None
        bboxes = np.empty((n, 4 * self.C), dtype=np.float32) if want_raw else None
        keep = np.empty((self.C - 1, n), dtype=np.int32)
        counts = np.empty(self.C - 1, dtype=np.int32)
        self._trunk_n = 1
        self.ctx.check(self.ctx.lib.mpn_model_detect_nms(
            self.h, _ptr(im), im.shape[1], im.shape[2], _ptr(b), n, float(im_scale), float(W0), float(H0),
            float(score_thresh), float(nms_thr), _ptr(scores), _ptr(bboxes), _ptr(keep), _ptr(counts)), "mpn_model_detect_nms")
        return scores, bboxes, [keep[j, : counts[j]].copy() for j in range(self.C - 1)]

    def test_one(self, image_chw, boxes, im_scale: float, W0: float, H0: float, num_iter: int = 1, use_rbox_scores: bool = False,
                 bbox_voting: bool = False, score_thresh: float = -1.5, nms_thr: float = 0.3, vote_thr: float = 0.5, vote_score_pow: float = 1.0):
        """Tester_FRCNN:testOne on the device (mpn_model_test_one): -> (scores n_out x C, bboxes n_out x 4C,
        [keep rows per class], [voted K_j x 5 per class] or None)"""
        im, b = _f32(image_chw), _f32(boxes)
        n = b.shape[0]
        n_out = n * (num_iter - (1 if use_rbox_scores else 0))
        o = CTestOpts(int(num_iter), int(bool(use_rbox_scores)), int(bool(bbox_voting)), float(score_thresh), float(nms_thr), float(vote_thr),
                      float(vote_score_pow))
        scores = np.empty((n_out, self.C), np.float32); bboxes = np.empty((n_out, 4 * self.C), np.float32)
        keep = np.empty((self.C - 1, n_out), np.int32); counts = np.empty(self.C - 1, np.int32)
        voted = np.empty((self.C - 1, n_out, 5), np.float32) if bbox_voting else None
        self._trunk_n = 1
        self.ctx.check(self.ctx.lib.mpn_model_test_one(self.h, _ptr(im), im.shape[1], im.shape[2], _ptr(b), n, float(im_scale), float(W0), float(H0),
                                                       C.byref(o), _ptr(scores), _ptr(bboxes), _ptr(keep), _ptr(counts), _ptr(voted)), "mpn_model_test_one")
        keeps = [keep[j, :counts[j]].copy() for j in range(self.C - 1)]
        return scores, bboxes, keeps, ([voted[j, :counts[j]].copy() for j in range(self.C - 1)] if bbox_voting else None)

    def detect_nms_submit(self, image_chw, boxes, im_scale: float, W0: float, H0: float, score_thresh: float = -1.5,
                          nms_thr: float = 0.3):
        """Pipelined detect_nms (at most two in flight): returns a ticket; `detect_nms_wait(ticket)` returns the results.
        The host->device copy overlaps the previous submission's kernels (pass pinned arrays for real overlap)."""
        im, b = _f32(image_chw), _f32(boxes)
        n = b.shape[0]
        out = dict(im=im, b=b, scores=np.empty((n, self.C), dtype=np.float32), bboxes=np.empty((n, 4 * self.C), dtype=np.float32),
                   keep=np.empty((self.C - 1, n), dtype=np.int32), counts=np.empty(self.C - 1, dtype=np.int32))
        t = C.c_int32(-1)
        self._trunk_n = 1
        self.ctx.check(self.ctx.lib.mpn_model_detect_nms_submit(
            self.h, _ptr(im), im.shape[1], im.shape[2], _ptr(b), n, float(im_scale), float(W0), float(H0), float(score_thresh),
            float(nms_thr), _ptr(out["scores"]), _ptr(out["bboxes"]), _ptr(out["keep"]), _ptr(out["counts"]), C.byref(t)),
            "mpn_model_detect_nms_submit")
        self._inflight = getattr(self, "_inflight", {})
        self._inflight[t.value] = out              # keeps the host buffers alive until wait()
        return t.value

    def detect_nms_submit_u8(self, im_hwc_u8, boxes, kind: str, scale: float = 600, max_size: float = 1000, score_thresh: float = -1.5,
                             nms_thr: float = 0.3):
        """pipelined detect_nms from the RAW uint8 H0 x W0 x 3 image: getImages runs on the device (mpn_model_detect_nms_submit_u8)"""
        im, b = np.ascontiguousarray(im_hwc_u8, dtype=np.uint8), _f32(boxes)
        n = b.shape[0]
        out = dict(im=im, b=b, scores=np.empty((n, self.C), dtype=np.float32), bboxes=np.empty((n, 4 * self.C), dtype=np.float32),
                   keep=np.empty((self.C - 1, n), dtype=np.int32), counts=np.empty(self.C - 1, dtype=np.int32), tf=CImageTransform.of(kind))
        t = C.c_int32(-1)
        self._trunk_n = 1
        self.ctx.check(self.ctx.lib.mpn_model_detect_nms_submit_u8(
            self.h, _ptr(im), im.shape[0], im.shape[1], C.addressof(out["tf"]), float(scale), float(max_size), _ptr(b), n, float(score_thresh),
            float(nms_thr), _ptr(out["scores"]), _ptr(out["bboxes"]), _ptr(out["keep"]), _ptr(out["counts"]), C.byref(t)),
            "mpn_model_detect_nms_submit_u8")
        self._inflight = getattr(self, "_inflight", {})
        self._inflight[t.value] = out
        return t.value

    def detect_nms_batch_submit_u8(self, ims, boxes_list, kind: str, scale: float = 600, max_size: float = 1000,
                                   score_thresh: float = -1.5, nms_thr: float = 0.3):
        """pipelined detect_nms_batch from N RAW uint8 H0 x W0 x 3 images of any sizes (mpn_model_detect_nms_batch_submit_u8):
        getImages pads them into one canvas on the device. boxes_list[i]: R_i x 4 in image i's ORIGINAL coordinates.
        Returns a ticket; detect_nms_wait(ticket) returns one (scores, bboxes, keeps) per image, as detect_nms_batch."""
        ims, H0, W0, sizes, (H, W) = _raw_batch(ims, scale, max_size)
        N = len(ims)
        if len(boxes_list) != N:
            raise ValueError(f"{N} images need {N} box arrays, got {len(boxes_list)}")
        boxes = [_f32(b) for b in boxes_list]
        if any(b.ndim != 2 or b.shape[1] != 4 for b in boxes):
            raise ValueError("every box array must be R_i x 4")
        if H > self.max_h or W > self.max_w:
            raise ValueError(f"padded canvas {H} x {W} larger than the model's max_h x max_w = {self.max_h} x {self.max_w}")
        offs, _, _, _ = self._batch_args(N, [b.shape[0] for b in boxes], [s for _, _, s in sizes], [(int(w), int(h)) for h, w in zip(H0, W0)])
        Rt, Cn = int(offs[-1]), self.C
        out = dict(im=np.concatenate([im.reshape(-1) for im in ims]), b=np.ascontiguousarray(np.concatenate(boxes, 0)), H0=H0, W0=W0,
                   offs=offs, scores=np.empty((Rt, Cn), np.float32), bboxes=np.empty((Rt, 4 * Cn), np.float32),
                   keep=np.empty((Cn - 1) * Rt, np.int32), counts=np.empty((N, Cn - 1), np.int32), tf=CImageTransform.of(kind))
        t = C.c_int32(-1)
        self._trunk_n = N
        self.ctx.check(self.ctx.lib.mpn_model_detect_nms_batch_submit_u8(
            self.h, _ptr(out["im"]), N, H0.ctypes.data_as(_i32p), W0.ctypes.data_as(_i32p), C.addressof(out["tf"]), float(scale),
            float(max_size), _ptr(out["b"]), offs.ctypes.data_as(_i64p), float(score_thresh), float(nms_thr), _ptr(out["scores"]),
            _ptr(out["bboxes"]), _ptr(out["keep"]), _ptr(out["counts"]), C.byref(t)), "mpn_model_detect_nms_batch_submit_u8")
        self._inflight = getattr(self, "_inflight", {})
        self._inflight[t.value] = out
        return t.value

    def detect_nms_wait(self, ticket: int):
        """results of a submission: (scores, bboxes, keeps) for a single image, one such tuple per image for a batch"""
        self.ctx.check(self.ctx.lib.mpn_model_detect_nms_wait(self.h, int(ticket)), "mpn_model_detect_nms_wait")
        o = self._inflight.pop(ticket)
        if "offs" in o:
            return self._split_batch(o["offs"], o["scores"], o["bboxes"], o["keep"], o["counts"])
        return o["scores"], o["bboxes"], [o["keep"][j, : o["counts"][j]].copy() for j in range(self.C - 1)]

    def _split_batch(self, offs, scores, bboxes, keep, counts):
        """the flat outputs of a batch call -> [(scores R_i x C, bboxes R_i x 4C, [keep rows per class])] per image"""
        Cn, out = self.C, []
        for i in range(len(offs) - 1):
            r0, r1 = int(offs[i]), int(offs[i + 1])
            k = keep[(Cn - 1) * r0:(Cn - 1) * r1].reshape(Cn - 1, r1 - r0)
            out.append((scores[r0:r1], bboxes[r0:r1], [k[j, :counts[i, j]].copy() for j in range(Cn - 1)]))
        return out

    def detect_nms_dev(self, image_dev, H: int, W: int, boxes_dev, R: int, im_scale: float, W0: float, H0: float,
                       score_thresh: float, nms_thr: float, scores_dev=None, bboxes_dev=None, keep_idx_dev=None,
                       keep_counts_dev=None):
        """Fully device-resident, asynchronous (arguments are torch CUDA tensors or raw addresses)."""
        self._trunk_n = 1
        self.ctx.check(self.ctx.lib.mpn_model_detect_nms_dev(
            self.h, _ptr(image_dev), H, W, _ptr(boxes_dev), R, float(im_scale), float(W0), float(H0), float(score_thresh),
            float(nms_thr), _ptr(scores_dev), _ptr(bboxes_dev), _ptr(keep_idx_dev), _ptr(keep_counts_dev)),
            "mpn_model_detect_nms_dev")

    def _batch_args(self, N: int, R: Sequence[int], im_scales, sizes):
        """host-side checks of a batch description -> (img_offsets int64 N+1, im_scale, W0, H0 float32 N)"""
        if not 1 <= N <= MPN_MAX_BATCH:
            raise ValueError(f"batch size must be in 1..{MPN_MAX_BATCH}, got {N}")
        R = [int(r) for r in R]
        if len(R) != N or len(im_scales) != N or len(sizes) != N:
            raise ValueError(f"{N} images need {N} box arrays, im_scales and (W0, H0) sizes; got {len(R)}, {len(im_scales)}, {len(sizes)}")
        if min(R) < 1:
            raise ValueError("every image needs at least one proposal")
        offs = np.zeros(N + 1, np.int64)
        offs[1:] = np.cumsum(R)
        if offs[-1] > self.max_rois:
            raise ValueError(f"{int(offs[-1])} proposals in the batch exceed max_rois = {self.max_rois}")
        sz = np.asarray(sizes, np.float32).reshape(N, 2)
        return offs, np.asarray(im_scales, np.float32).reshape(N), np.ascontiguousarray(sz[:, 0]), np.ascontiguousarray(sz[:, 1])

    def detect_nms_batch(self, images_nchw, boxes_list, im_scales, sizes, score_thresh: float = -1.5, nms_thr: float = 0.3):
        """detect_nms for N images of one padded size in one pass: boxes_list[i] R_i x 4 in image i's ORIGINAL coordinates,
        im_scales[i] and sizes[i] = (W0, H0) as getImages gave them. -> one (scores, bboxes, keeps) per image, as detect_nms."""
        im = _f32(images_nchw)
        if im.ndim != 4 or im.shape[1] != 3:
            raise ValueError("detect_nms_batch expects N x 3 x H x W images")
        N = im.shape[0]
        boxes = [_f32(b).reshape(-1, 4) for b in boxes_list]
        offs, sc, w0, h0 = self._batch_args(N, [b.shape[0] for b in boxes], im_scales, sizes)
        Rt, Cn = int(offs[-1]), self.C
        b = np.ascontiguousarray(np.concatenate(boxes, 0))
        scores = np.empty((Rt, Cn), np.float32); bboxes = np.empty((Rt, 4 * Cn), np.float32)
        keep = np.empty((Cn - 1) * Rt, np.int32); counts = np.empty((N, Cn - 1), np.int32)
        self._trunk_n = N
        self.ctx.check(self.ctx.lib.mpn_model_detect_nms_batch(
            self.h, _ptr(im), N, im.shape[2], im.shape[3], _ptr(b), offs.ctypes.data_as(_i64p), _ptr(sc), _ptr(w0), _ptr(h0),
            float(score_thresh), float(nms_thr), _ptr(scores), _ptr(bboxes), _ptr(keep), _ptr(counts)), "mpn_model_detect_nms_batch")
        return self._split_batch(offs, scores, bboxes, keep, counts)

    def detect_nms_batch_dev(self, images_dev, N: int, H: int, W: int, boxes_dev, R_list: Sequence[int], im_scales, sizes,
                             score_thresh: float, nms_thr: float, scores_dev=None, bboxes_dev=None, keep_idx_dev=None,
                             keep_counts_dev=None):
        """detect_nms_batch fully device-resident and asynchronous (arguments are torch CUDA tensors or raw addresses):
        boxes_dev R_total x 4, image i owning R_list[i] consecutive rows; keep_idx_dev (C-1) * R_total, image i's
        (C-1) x R_i block at (C-1) * offset_i; keep_counts_dev N x (C-1)."""
        offs, sc, w0, h0 = self._batch_args(int(N), R_list, im_scales, sizes)
        self._trunk_n = int(N)
        self.ctx.check(self.ctx.lib.mpn_model_detect_nms_batch_dev(
            self.h, _ptr(images_dev), int(N), int(H), int(W), _ptr(boxes_dev), offs.ctypes.data_as(_i64p), _ptr(sc), _ptr(w0),
            _ptr(h0), float(score_thresh), float(nms_thr), _ptr(scores_dev), _ptr(bboxes_dev), _ptr(keep_idx_dev),
            _ptr(keep_counts_dev)), "mpn_model_detect_nms_batch_dev")

    def trunk_slot(self, slot: int) -> np.ndarray:
        """trunk slot `slot` of the last trunk forward as N x C x H x W fp32 (N = its images)"""
        c, h, w = C.c_int32(), C.c_int32(), C.c_int32()
        self.ctx.check(self.ctx.lib.mpn_model_get_trunk_slot(self.h, slot, None, 0, C.byref(c), C.byref(h), C.byref(w)), "get_trunk_slot")
        out = np.empty((self._trunk_n, c.value, h.value, w.value), dtype=np.float32)
        self.ctx.check(self.ctx.lib.mpn_model_get_trunk_slot(self.h, slot, _ptr(out), out.size, C.byref(c), C.byref(h), C.byref(w)),
                       "get_trunk_slot")
        return out

    def last_flops(self):
        a, b = C.c_double(), C.c_double()
        self.ctx.check(self.ctx.lib.mpn_model_last_flops(self.h, C.byref(a), C.byref(b)), "last_flops")
        return a.value, b.value
