"""ctypes binding of libmanuscript_b200.so (include/manuscript_b200.h).

The library is built in-tree by manuscript-ocr_b200/build.py (nvcc, sm_100a).  Nothing here computes:
if the shared object is missing or no CUDA device is present the calls raise, they never fall back.
"""
import ctypes as C
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_NAME = "libmanuscript_b200.so"

MS_OK = 0
MS_ERR_INVALID = -1
MS_ERR_CUDA = -2
MS_ERR_CAPACITY = -3
MS_ERR_INDEX = -4
MS_ERR_NO_DEVICE = -5

MS_FLAG_CAND_OVERFLOW = 1
MS_FLAG_INDEX_ERROR = 2
MS_FLAG_EDGE_OVERFLOW = 4
MS_FLAG_ORDER_OVERFLOW = 8

MS_JPEG_OK = 0
MS_JPEG_NOT_JPEG = 1
MS_JPEG_PROGRESSIVE = 2
MS_JPEG_UNSUPPORTED_CODING = 3
MS_JPEG_COLOR = 4
MS_JPEG_SAMPLING = 5
MS_JPEG_ORIENTATION = 6
MS_JPEG_SCAN = 7
MS_JPEG_BAD_ENTROPY = 16

MS_DTYPE_F32 = 0
MS_DTYPE_F16 = 1
MS_DTYPE_BF16 = 2


class CABIError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"manuscript_b200 error {code}: {msg}")
        self.code = code


class EastParams(C.Structure):
    """ms_east_params: the EAST constructor kwargs that shape the path (reference infer.py:28-43)."""

    _fields_ = [
        ("score_thresh", C.c_float),
        ("scale", C.c_double),
        ("quantization", C.c_int),
        ("iou_threshold", C.c_double),
        ("expand_ratio_w", C.c_double),
        ("expand_ratio_h", C.c_double),
        ("target_size", C.c_int),
        ("axis_aligned_output", C.c_int),
        ("remove_area_anomalies", C.c_int),
        ("anomaly_sigma_threshold", C.c_double),
        ("anomaly_min_box_count", C.c_int),
        ("sort_reading_order", C.c_int),
    ]

    @classmethod
    def default(cls, **overrides):
        p = cls()
        load_library().ms_east_params_default(C.byref(p))
        for k, v in overrides.items():
            if not hasattr(p, k):
                raise TypeError(f"unknown EAST parameter {k!r}")
            setattr(p, k, v)
        return p


class MsMaps(C.Structure):
    """ms_maps: the score and geometry maps of a batch, one element type, each at its own element strides."""

    _fields_ = [
        ("score", C.c_void_p),
        ("geo", C.c_void_p),
        ("dtype", C.c_int32),
        ("score_strides", C.c_int64 * 3),
        ("geo_strides", C.c_int64 * 4),
    ]


_vp = C.c_void_p
_i = C.c_int
_i64 = C.c_int64
_d = C.c_double
_f = C.c_float

# name -> (restype, argtypes); must list every symbol include/manuscript_b200.h declares
SIGNATURES = {
    "ms_version": (C.c_char_p, []),
    "ms_last_error": (C.c_char_p, []),
    "ms_east_params_default": (None, [C.POINTER(EastParams)]),
    "ms_create": (_i, [_i, C.POINTER(_vp)]),
    "ms_destroy": (None, [_vp]),
    "ms_device_count": (_i, []),
    "ms_launch_count": (_i64, [_vp]),
    "ms_set_edge_factor": (_i, [_vp, _i]),
    "ms_get_edge_factor": (_i, [_vp]),
    "ms_stage_timing": (_i, [_vp, _i]),
    "ms_stage_times": (_i, [_vp, C.POINTER(_d)]),
    "ms_decode_quads_host": (_i, [_vp, _vp, _vp, _i, _i, _f, _d, _i, _vp, _i64, C.POINTER(_i64)]),
    "ms_decode_rbox_host": (_i, [_vp, _vp, _vp, _i, _i, _f, _d, _i, _vp, _i64, C.POINTER(_i64)]),
    "ms_decode_rbox": (_i, [_vp, _vp, _vp, _i, _i, _i, _f, _d, _i, _vp, _i, _vp, _vp, _vp]),
    "ms_lanms_host": (_i, [_vp, _vp, _i64, _d, _vp, C.POINTER(_i64)]),
    "ms_standard_nms_host": (_i, [_vp, _vp, _vp, _i64, _d, _vp, C.POINTER(_i64)]),
    "ms_polygon_iou_host": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "ms_quad_crop_last_counts": (_i, [_vp, _vp]),
    "ms_crop_last_counts": (_i, [_vp, _vp]),
    "ms_test_iou_proved_host": (_i, [_vp, _vp, _vp, _i64, _d, _vp]),
    "ms_test_resize_tables_host": (_i, [_vp, _i, _i, _vp, _i64, _vp, _vp, _i64, _vp, _i64]),
    "ms_test_np_sum_host": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "ms_expand_boxes_host": (_i, [_vp, _vp, _i64, _d, _d, _vp]),
    "ms_east_boxes_host": (_i, [_vp, _vp, _i64, C.POINTER(EastParams), _i, _i, _vp, C.POINTER(_i64)]),
    "ms_word_rects_host": (_i, [_vp, _vp, _i64, _i, _i, _i, _vp, _vp]),
    "ms_reading_order_host": (_i, [_vp, _vp, _i64, _vp]),
    "ms_reading_order": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "ms_crop_resize_pad_host": (_i, [_vp, _vp, _i, _i, _vp, _i64, _i, _i, _vp, _vp]),
    "ms_quad_crop_resize_pad_host": (_i, [_vp, _vp, _i, _i, _vp, _i64, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "ms_warp_quad_host": (_i, [_vp, _vp, _i, _i, _vp, _i, _i, _vp, _i64, C.POINTER(_i), C.POINTER(_i)]),
    "ms_quad_crop_resize_pad": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _vp, _i64, _i, _i, _i, _i, _i, _vp, _vp, _vp,
                                     _vp]),
    "ms_detector_input": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "ms_detector_input_batch": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _i, _vp]),
    "ms_tps_rectify": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "ms_decode_quads": (_i, [_vp, _vp, _vp, _i, _i, _i, _f, _d, _i, _vp, _i, _vp, _vp, _vp]),
    "ms_lanms": (_i, [_vp, _vp, _vp, _i, _i, _d, _vp, _vp, _vp, _vp]),
    "ms_east_boxes": (_i, [_vp, _vp, _vp, _i, _i, C.POINTER(EastParams), _vp, _vp, _vp, _vp]),
    "ms_word_rects": (_i, [_vp, _vp, _vp, _i, _i, _vp, _i, _i, _i, _vp, _i64, _vp, _vp]),
    "ms_crop_resize_pad": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i64, _i, _i, _vp, _vp, _vp]),
    "ms_page_batch": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, C.POINTER(EastParams), _i, _i, _i, _i, _vp, _vp,
                           _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "ms_page_batch_ragged": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, C.POINTER(EastParams), _i, _i, _i, _i, _vp, _vp,
                                  _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "ms_page_batch_ragged_host": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, C.POINTER(EastParams), _i, _i, _i, _i, _vp,
                                       _vp, _vp, _i64, _vp, _vp, C.POINTER(_vp), _vp]),
    "ms_page_batch_host": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, C.POINTER(EastParams), _i, _i, _i, _i, _vp,
                                _vp, _vp, _i64, _vp, _vp, C.POINTER(_vp), _vp]),
    # the same entry points with the batch in an MS_DTYPE_* element type (void *batch, int batch_dtype)
    "ms_crop_resize_pad_ex": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i64, _i, _i, _vp, _i, _vp, _vp]),
    "ms_quad_crop_resize_pad_ex": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _vp, _i64, _i, _i, _i, _i, _i, _vp, _i, _vp,
                                        _vp, _vp]),
    "ms_page_batch_ex": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, C.POINTER(EastParams), _i, _i, _i, _i, _vp, _vp,
                              _vp, _i64, _vp, _vp, _i, _vp, _vp, _vp]),
    "ms_page_batch_ragged_ex": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, C.POINTER(EastParams), _i, _i, _i, _i, _vp,
                                     _vp, _vp, _i64, _vp, _vp, _i, _vp, _vp, _vp]),
    "ms_page_batch_host_ex": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, C.POINTER(EastParams), _i, _i, _i, _i, _vp,
                                   _vp, _vp, _i64, _vp, _vp, _i, C.POINTER(_vp), _vp]),
    "ms_page_batch_ragged_host_ex": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, C.POINTER(EastParams), _i, _i, _i, _i,
                                          _vp, _vp, _vp, _i64, _vp, _vp, _i, C.POINTER(_vp), _vp]),
    # EXTENSION: page batches whose crop stage is the rectified crop of every final quad (border_mode, border_value
    # after min_text_size)
    "ms_page_batch_quads": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, C.POINTER(EastParams), _i, _i, _i, _i, _i,
                                 _i, _vp, _vp, _vp, _i64, _vp, _vp, _i, _vp, _vp, _vp]),
    "ms_page_batch_ragged_quads": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, C.POINTER(EastParams), _i, _i, _i, _i, _i,
                                        _i, _vp, _vp, _vp, _i64, _vp, _vp, _i, _vp, _vp, _vp]),
    # EXTENSION: the same entry points on an ms_maps descriptor (maps in float32 / float16 / bfloat16, any strides)
    "ms_decode_quads_maps": (_i, [_vp, C.POINTER(MsMaps), _i, _i, _i, _f, _d, _i, _vp, _i, _vp, _vp, _vp]),
    "ms_page_batch_maps": (_i, [_vp, C.POINTER(MsMaps), _vp, _i, _i, _i, _i, _i, C.POINTER(EastParams), _i, _i, _i,
                                _i, _vp, _vp, _vp, _i64, _vp, _vp, _i, _vp, _vp, _vp]),
    "ms_page_batch_ragged_maps": (_i, [_vp, C.POINTER(MsMaps), _vp, _vp, _i, _i, _i, C.POINTER(EastParams), _i, _i,
                                       _i, _i, _vp, _vp, _vp, _i64, _vp, _vp, _i, _vp, _vp, _vp]),
    "ms_page_batch_quads_maps": (_i, [_vp, C.POINTER(MsMaps), _vp, _i, _i, _i, _i, _i, C.POINTER(EastParams), _i,
                                      _i, _i, _i, _i, _i, _vp, _vp, _vp, _i64, _vp, _vp, _i, _vp, _vp, _vp]),
    "ms_page_batch_ragged_quads_maps": (_i, [_vp, C.POINTER(MsMaps), _vp, _vp, _i, _i, _i, C.POINTER(EastParams), _i,
                                             _i, _i, _i, _i, _i, _vp, _vp, _vp, _i64, _vp, _vp, _i, _vp, _vp, _vp]),
    # EXTENSION: baseline-JPEG decode on the device (ms_jpeg_info *, host files -> device pages)
    "ms_jpeg_inspect_host": (_i, [_vp, _i64, _vp]),
    "ms_jpeg_decode_batch": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp]),
}


def batch_dtype_code(dtype):
    """torch.float32 / torch.float16 / torch.bfloat16 -> MS_DTYPE_F32 / _F16 / _BF16 (the `batch_dtype` argument of
    the *_ex entry points).  Any other dtype raises ValueError."""
    import torch

    codes = {torch.float32: MS_DTYPE_F32, torch.float16: MS_DTYPE_F16, torch.bfloat16: MS_DTYPE_BF16}
    if dtype not in codes:
        raise ValueError(f"the recogniser batch can be float32, float16 or bfloat16, not {dtype}")
    return codes[dtype]


def maps_descriptor(score, geo):
    """MsMaps of a (P, H, W) score and a (P, 8, H, W) geometry CUDA tensor, both float32, float16 or bfloat16, at the
    strides they have.  The descriptor holds the tensors' addresses: the caller keeps them alive."""
    import torch

    codes = {torch.float32: MS_DTYPE_F32, torch.float16: MS_DTYPE_F16, torch.bfloat16: MS_DTYPE_BF16}
    if score.dtype != geo.dtype or score.dtype not in codes:
        raise ValueError(f"score and geometry maps must both be float32, float16 or bfloat16, got {score.dtype} and "
                         f"{geo.dtype}")
    if score.dim() != 3 or geo.dim() != 4:
        raise ValueError(f"maps must be (P, H, W) and (P, 8, H, W), got {tuple(score.shape)} and {tuple(geo.shape)}")
    return MsMaps(score.data_ptr(), geo.data_ptr(), codes[score.dtype], (C.c_int64 * 3)(*score.stride()),
                  (C.c_int64 * 4)(*geo.stride()))


_lib = None
_lock = threading.Lock()


def library_path():
    # MS_B200_LIB: an experiment build of the same library (manuscript-ocr_b200/build.py --variant), for A/B timing
    return os.environ.get("MS_B200_LIB") or os.path.join(HERE, _LIB_NAME)


def load_library():
    """dlopen the in-tree library and type every entry point.  Raises if it has not been built."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = library_path()
        if not os.path.exists(path):
            raise ImportError(
                f"{path} is missing: build it with `python manuscript-ocr_b200/build.py` "
                "(there is no CPU fallback for this path)")
        lib = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError here == ABI drift between header and library
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def last_error():
    return load_library().ms_last_error().decode("utf-8", "replace")


def check(rc):
    if rc == MS_OK:
        return
    msg = last_error()
    if rc == MS_ERR_INDEX:
        raise IndexError(msg)  # what the reference raises at utils.py:370
    raise CABIError(rc, msg)


class Context:
    """ms_ctx: one per (thread, device).  Holds the device scratch arenas reused across calls."""

    def __init__(self, device=0):
        lib = load_library()
        h = _vp()
        check(lib.ms_create(int(device), C.byref(h)))
        self._h = h
        self.device = int(device)
        self.lib = lib

    @property
    def handle(self):
        if self._h is None:
            raise RuntimeError("context destroyed")
        return self._h

    @property
    def launches(self):
        return int(self.lib.ms_launch_count(self.handle))

    @property
    def edge_factor(self):
        return int(self.lib.ms_get_edge_factor(self.handle))

    @edge_factor.setter
    def edge_factor(self, k):
        check(self.lib.ms_set_edge_factor(self.handle, int(k)))

    def grow_edge_factor(self):
        """x4 (the policy of the *_host entry points); False once the limit is reached."""
        k = self.edge_factor
        if k >= 4096:
            return False
        self.edge_factor = min(4096, k * 4)
        return True

    STAGES = ("decode", "lanms", "east_boxes", "word_rects", "crop")

    def stage_timing(self, enable=True):
        check(self.lib.ms_stage_timing(self.handle, int(bool(enable))))

    def stage_times(self):
        """(n_batches, {stage: summed ms}) since the last read; waits for the recorded batches."""
        ms = (_d * len(self.STAGES))()
        n = self.lib.ms_stage_times(self.handle, ms)
        if n < 0:
            check(n)
        return n, dict(zip(self.STAGES, [float(v) for v in ms]))

    def close(self):
        if getattr(self, "_h", None) is not None:
            self.lib.ms_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx = {}


def default_context(device=0):
    key = (threading.get_ident(), int(device))
    ctx = _default_ctx.get(key)
    if ctx is None:
        ctx = _default_ctx[key] = Context(device)
    return ctx
