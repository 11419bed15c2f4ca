"""ctypes binding of libb2chips.so (the C ABI declared in include/b2chips.h).

There is NO CPU fallback: if the shared library is missing or no B200 is visible, every entry point
raises.  torch is used only as plumbing (device allocations, streams); the arithmetic is in the .so.
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B2CHIPS_LIB") or os.path.join(_HERE, "libb2chips.so")   # override: development builds only

# element type codes (b2chips.h)
B2_U8, B2_U16, B2_I16, B2_U32, B2_I32, B2_F32, B2_F64, B2_I8 = range(8)
SINK_NONE, SINK_RAW, SINK_NORM_ONEHOT, SINK_NORM_ONEHOT_F32 = 0, 1, 2, 3


class B2Error(RuntimeError):
    pass


class ExampleIndex(ctypes.Structure):
    _fields_ = [("img_off", ctypes.c_uint64), ("img_len", ctypes.c_uint64),
                ("tgt_off", ctypes.c_uint64), ("tgt_len", ctypes.c_uint64),
                ("id_off", ctypes.c_uint64), ("id_len", ctypes.c_uint64),
                ("img_kind", ctypes.c_int32), ("tgt_kind", ctypes.c_int32),
                ("height", ctypes.c_int32), ("width", ctypes.c_int32), ("channels", ctypes.c_int32),
                ("tgt_height", ctypes.c_int32), ("tgt_width", ctypes.c_int32), ("status", ctypes.c_int32)]


class ParseSink(ctypes.Structure):
    _fields_ = [("mode", ctypes.c_int32), ("verify_crc", ctypes.c_int32),
                ("img_out", ctypes.c_void_p), ("img_stride", ctypes.c_uint64),
                ("tgt_out", ctypes.c_void_p), ("tgt_stride", ctypes.c_uint64),
                ("mean", ctypes.c_void_p), ("std", ctypes.c_void_p),
                ("channels", ctypes.c_int32), ("num_classes", ctypes.c_int32)]


class BuildDesc(ctypes.Structure):
    _fields_ = [("out_off", ctypes.c_uint64), ("example_len", ctypes.c_uint64), ("scaffold_off", ctypes.c_uint64),
                ("piece_len", ctypes.c_uint32 * 3), ("src_dtype", ctypes.c_int32), ("tgt_dtype", ctypes.c_int32),
                ("kind", ctypes.c_int32),
                ("img_src", ctypes.c_void_p), ("img_count", ctypes.c_uint64),
                ("tgt_src", ctypes.c_void_p), ("tgt_count", ctypes.c_uint64)]


EXAMPLE_INDEX_DTYPE = [("img_off", "<u8"), ("img_len", "<u8"), ("tgt_off", "<u8"), ("tgt_len", "<u8"),
                       ("id_off", "<u8"), ("id_len", "<u8"), ("img_kind", "<i4"), ("tgt_kind", "<i4"),
                       ("height", "<i4"), ("width", "<i4"), ("channels", "<i4"), ("tgt_height", "<i4"),
                       ("tgt_width", "<i4"), ("status", "<i4")]
BUILD_DESC_DTYPE = [("out_off", "<u8"), ("example_len", "<u8"), ("scaffold_off", "<u8"), ("piece_len", "<u4", (3,)),
                    ("src_dtype", "<i4"), ("tgt_dtype", "<i4"), ("kind", "<i4"),
                    ("img_src", "<u8"), ("img_count", "<u8"), ("tgt_src", "<u8"), ("tgt_count", "<u8")]

_vp, _i, _u64, _i32, _f = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64, ctypes.c_int32, ctypes.c_float

# name -> (restype, argtypes); every symbol declared in include/b2chips.h
SIGNATURES = {
    "b2_version": (_i, []),
    "b2_last_error": (ctypes.c_char_p, []),
    "b2_ctx_create": (_i, [_i, ctypes.POINTER(_vp)]),
    "b2_ctx_destroy": (_i, [_vp]),
    "b2_ctx_launch_count": (_u64, [_vp]),
    "b2_ctx_sm_count": (_i, [_vp]),
    "b2_median_composite_u16": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "b2_nearest_date_mosaic": (_i, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _f, _i, _i, _i, _i, _i, _i,
                                    _vp, _vp, _vp, _vp, _vp, _vp]),
    "b2_normalise_onehot": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp, _u64, _i, _i, _vp, _vp, _vp]),
    "b2_band_stats": (_i, [_vp, _vp, _i, _vp, _u64, _i, _vp, _vp]),
    "b2_crc32c": (_i, [_vp, _vp, _vp, _vp, _i, _u64, _vp, _vp]),
    "b2_tfrecord_scan": (_i, [_vp, _vp, _u64, _u64, _vp, _vp, _vp, _vp]),
    "b2_tfrecord_index": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "b2_tfrecord_table_bytes": (_u64, [_u64, _u64]),
    "b2_tfrecord_table_layout": (_i, [_u64, _u64, ctypes.POINTER(_u64)]),
    "b2_tfrecord_open": (_i, [_vp, _vp, _u64, _u64, _vp, _vp]),
    "b2_tfrecord_parse_table": (_i, [_vp, _vp, _u64, _u64, _vp, ctypes.POINTER(ParseSink), _vp, _vp]),
    "b2_tfrecord_parse": (_i, [_vp, _vp, _u64, _vp, _vp, _vp, _i, _u64, ctypes.POINTER(ParseSink), _vp, _vp]),
    "b2_example_layout": (_i, [_i, _u64, _u64, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64,
                               ctypes.c_int64, _vp, _u64, _vp, _u64, ctypes.POINTER(ctypes.c_uint32),
                               ctypes.POINTER(_u64)]),
    "b2_example_layout_batch": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _u64, ctypes.POINTER(_u64), ctypes.POINTER(_u64), ctypes.POINTER(_u64)]),
    "b2_tfrecord_build": (_i, [_vp, _vp, _i, _u64, _vp, _vp, _vp]),
    "b2_rasterize_polygons": (_i, [_vp, _vp, _vp, _vp, _vp, ctypes.c_uint32, _vp, _vp, ctypes.c_uint32, _vp, _i, _i, _i, _i,
                                   ctypes.c_uint32, _vp, _vp, _vp, _vp]),
}

_lib = None
_lock = threading.Lock()


def register_signatures(extra):
    """Later modules (codec) add their entry points here before the library is first loaded."""
    SIGNATURES.update(extra)
    if _lib is not None:
        for name, (res, args) in extra.items():
            fn = getattr(_lib, name)
            fn.restype = res
            fn.argtypes = args


def lib():
    """Load libb2chips.so (once).  Raises if it has not been built — the product has no CPU path."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise B2Error(
                        "libb2chips.so not found at %s: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(or `make -C dl_image_segmentation_b200/csrc`). There is no CPU fallback." % LIB_PATH)
                L = ctypes.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(L, name)
                    fn.restype = res
                    fn.argtypes = args
                _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise B2Error(lib().b2_last_error().decode("utf-8", "replace"))


class Context:
    """One b2_ctx per (process, device)."""

    def __init__(self, device):
        import torch
        if not torch.cuda.is_available():
            raise B2Error("no CUDA device visible: dl_image_segmentation_b200 runs on B200 GPUs only (no CPU fallback)")
        self.device = torch.device("cuda", device if device is not None else torch.cuda.current_device())
        h = ctypes.c_void_p()
        check(lib().b2_ctx_create(self.device.index, ctypes.byref(h)))
        self.handle = h

    @property
    def launches(self):
        return int(lib().b2_ctx_launch_count(self.handle))

    @property
    def sm_count(self):
        return int(lib().b2_ctx_sm_count(self.handle))

    def stream(self):
        import torch
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)


_ctxs = {}


def get_ctx(device=None) -> Context:
    import torch
    if isinstance(device, torch.device):
        device = device.index
    if isinstance(device, str):
        device = torch.device(device).index
    if device is None:
        if not torch.cuda.is_available():
            raise B2Error("no CUDA device visible: dl_image_segmentation_b200 runs on B200 GPUs only (no CPU fallback)")
        device = torch.cuda.current_device()
    with _lock:
        c = _ctxs.get(device)
    if c is None:
        c = Context(device)
        with _lock:
            _ctxs[device] = c
    return c


def ptr(t):
    """Device (or host) pointer of a torch tensor / numpy array, None -> NULL."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return ctypes.c_void_p(t.data_ptr())
    return ctypes.c_void_p(t.ctypes.data)
