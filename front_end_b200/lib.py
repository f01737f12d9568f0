"""ctypes binding of libfe_b200.so (the C-ABI declared in include/fe_abi.h).

This is plumbing only: every computation happens in the CUDA library.  There is no CPU fallback;
if the shared library has not been built (``python -c "import __graft_entry__ as g; g.build()"`` or
``make -C front_end_b200/csrc``) importing this module raises ImportError.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfe_b200.so")

FE_OK, FE_ERR_BAD_ARG, FE_ERR_CAPACITY, FE_ERR_CUDA, FE_ERR_NO_DEVICE, FE_ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5
FAST_9_16, FAST_7_12, FAST_5_8 = 16, 12, 8
DESC_ORB256, DESC_SURF64, DESC_SURF128 = 0, 1, 2
DESC_BRIEF16, DESC_BRIEF32, DESC_BRIEF64 = 3, 4, 5
DESC_FREAK = 6
NORM_HAMMING, NORM_HAMMING2, NORM_L2 = 6, 7, 4
MATCH_RATIO, MATCH_CROSSCHECK = 0, 1
MASK_NONE, MASK_EPIPOLAR, MASK_WINDOW = 0, 1, 2

# msg/kPoint.msg and msg/cvMatch.msg wire layouts
KPOINT = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"),
                   ("octave", "<i4"), ("class_id", "<i4")])
MATCH = np.dtype([("queryIdx", "<u4"), ("trainIdx", "<u4"), ("imgIdx", "<u4"), ("distance", "<f4")])
assert KPOINT.itemsize == 28 and MATCH.itemsize == 16


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("max_width", C.c_int32), ("max_height", C.c_int32),
                ("max_images", C.c_int32), ("max_keypoints", C.c_int32), ("fast_threshold", C.c_int32),
                ("fast_type", C.c_int32), ("nonmax", C.c_int32), ("n_features", C.c_int32),
                ("edge_threshold", C.c_int32), ("orientation", C.c_int32), ("surf_upright", C.c_int32),
                ("stream", C.c_void_p)]


class MatchCfg(C.Structure):
    _fields_ = [("ratio", C.c_double), ("mode", C.c_int32), ("mask", C.c_int32), ("norm", C.c_int32),
                ("epi_threshold", C.c_float), ("q_y_offset", C.c_float), ("t_y_offset", C.c_float),
                ("win_w", C.c_int32), ("win_h", C.c_int32), ("max_dy", C.c_float)]


class GridCfg(C.Structure):
    _fields_ = [("roi_x", C.c_int32), ("roi_y", C.c_int32), ("roi_w", C.c_int32), ("roi_h", C.c_int32),
                ("rows", C.c_int32), ("cols", C.c_int32), ("variant", C.c_int32), ("fast_type", C.c_int32),
                ("set_point", C.c_int32), ("min_threshold", C.c_int32), ("max_threshold", C.c_int32),
                ("subpix", C.c_int32), ("update", C.c_int32)]


class WindowCfg(C.Structure):
    _fields_ = [("length", C.c_int32), ("variant", C.c_int32)]


class SurfParams(C.Structure):
    _fields_ = [("hessian_threshold", C.c_float), ("n_octaves", C.c_int32), ("n_octave_layers", C.c_int32),
                ("extended", C.c_int32), ("upright", C.c_int32)]


def match_cfg(mode=MATCH_RATIO, mask=MASK_EPIPOLAR, norm=NORM_HAMMING, epi_threshold=2.0, ratio=0.8,
              q_y_offset=0.0, t_y_offset=0.0, win_w=100, win_h=100, max_dy=0.7):
    return MatchCfg(ratio, mode, mask, norm, epi_threshold, q_y_offset, t_y_offset, win_w, win_h, max_dy)


EXPORTS = {
    # name: (restype, argtypes)
    "fe_abi_version": (C.c_int32, []),
    "fe_default_config": (None, [C.POINTER(Config)]),
    "fe_set_orb_score_type": (C.c_int32, [C.c_void_p, C.c_int32]),
    "fe_surf_detect_batch": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(SurfParams), C.c_void_p,
                                         C.c_void_p, C.c_int32, C.c_void_p]),
    "fe_set_brief_pattern": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32]),
    "fe_set_freak": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_int32, C.c_void_p]),
    "fe_window_update": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                     C.POINTER(MatchCfg), C.POINTER(WindowCfg), C.c_void_p, C.c_int32, C.POINTER(C.c_int32),
                                     C.POINTER(C.c_int32)]),
    "fe_create": (C.c_int32, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "fe_destroy": (None, [C.c_void_p]),
    "fe_last_error": (C.c_char_p, [C.c_void_p]),
    "fe_device_count": (C.c_int32, []),
    "fe_set_detection": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]),
    "fe_detect": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                              C.POINTER(C.c_int32)]),
    "fe_grid_detect": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.POINTER(GridCfg),
                                   C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_void_p]),
    "fe_corner_subpix": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32]),
    "fe_surf_detect_and_compute": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                               C.POINTER(SurfParams), C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]),
    "fe_describe": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                C.POINTER(C.c_int32), C.c_void_p, C.c_int32]),
    "fe_knn2": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                            C.c_int32, C.POINTER(MatchCfg), C.c_void_p, C.c_void_p]),
    "fe_stereo_match": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_int32, C.c_int32, C.POINTER(MatchCfg), C.c_void_p, C.c_int32,
                                    C.POINTER(C.c_int32)]),
    "fe_window_match": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_int32, C.c_int32, C.POINTER(MatchCfg), C.c_void_p, C.c_int32,
                                    C.POINTER(C.c_int32)]),
    "fe_stereo_features": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                       C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.c_void_p,
                                       C.c_void_p, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_double)]),
    "fe_pipeline_batch": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                      C.POINTER(MatchCfg), C.POINTER(MatchCfg), C.c_int32, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fe_measure_popc_peak": (C.c_int32, [C.c_void_p, C.POINTER(C.c_double)]),
    "fe_window_batch": (C.c_int32, [C.c_void_p, C.POINTER(MatchCfg), C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_void_p]),
    "fe_set_orb_patch_size": (C.c_int32, [C.c_void_p, C.c_int32]),
    "fe_set_orb_pyramid": (C.c_int32, [C.c_void_p, C.c_int32, C.c_float]),
    "fe_set_orb_wta_k": (C.c_int32, [C.c_void_p, C.c_int32]),
    "fe_batch_landmarks": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]),
    "fe_set_chunk_pairs": (C.c_int32, [C.c_void_p, C.c_int32]),
    "fe_set_batch_descriptor": (C.c_int32, [C.c_void_p, C.c_int32]),
    "fe_set_batch_detector": (C.c_int32, [C.c_void_p, C.POINTER(SurfParams)]),
    "fe_batch_upload": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    "fe_batch_run": (C.c_int32, [C.c_void_p, C.POINTER(MatchCfg), C.POINTER(MatchCfg), C.c_int32]),
    "fe_batch_download": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]),
    "fe_host_alloc": (C.c_void_p, [C.c_size_t]),
    "fe_host_free": (None, [C.c_void_p]),
    "fe_sync": (C.c_int32, [C.c_void_p]),
    "fe_stream": (C.c_void_p, [C.c_void_p]),
    "fe_profile_enable": (C.c_int32, [C.c_void_p, C.c_int32]),
    "fe_profile_reset": (C.c_int32, [C.c_void_p]),
    "fe_stage_times": (C.c_int32, [C.c_void_p, C.c_int32, C.POINTER(C.c_char_p), C.POINTER(C.c_double),
                                   C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "fe_kernel_launches": (C.c_int64, [C.c_void_p]),
    "fe_transfer_bytes": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
}


def load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "front_end_b200: %s is missing -- build it with `make -C front_end_b200/csrc` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)   # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib


class FeError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("fe status %d: %s" % (code, msg))
        self.code = code


class PinnedArray:
    """numpy view over cudaHostAlloc memory (freed on close / garbage collection)."""

    def __init__(self, lib, shape, dtype):
        self._lib = lib
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        self.ptr = lib.fe_host_alloc(max(n, 1))
        if not self.ptr:
            raise MemoryError("fe_host_alloc(%d) failed" % n)
        buf = (C.c_uint8 * max(n, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def close(self):
        if self.ptr:
            self.array = None
            self._lib.fe_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
