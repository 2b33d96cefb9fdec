"""ctypes binding of ``libb2ocr.so`` (C-ABI in include/b2ocr.h).

There is deliberately no fallback: if the shared library is missing or the device is not a
B200-class GPU, importing/creating fails loudly.  PyTorch is used by the callers only to own
device memory and streams; only raw pointers cross this boundary.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B2O_LIB") or os.path.join(_HERE, "libb2ocr.so")      # B2O_LIB: development builds only

CONV_AUTO, CONV_SIMT, CONV_TC_GENERIC = 0, 1, 2
MAX_CLASSES = 1024            # B2O_MAX_CLASSES in include/b2ocr.h
CRNN_HEIGHTS = (16, 64)       # B2O_CRNN_MIN_HEIGHT / B2O_CRNN_MAX_HEIGHT: supported recognizer crop heights
CRNN_WIDTHS = (32, 800)       # B2O_CRNN_MIN_WIDTH / B2O_CRNN_MAX_WIDTH: ... and widths


class B2OError(RuntimeError):
    pass


class _Tensor(ctypes.Structure):
    _fields_ = [("name", ctypes.c_char_p), ("data", ctypes.POINTER(ctypes.c_float)),
                ("ndim", ctypes.c_int32), ("shape", ctypes.c_int64 * 4)]


_c = ctypes
_vp, _i, _f, _sz = _c.c_void_p, _c.c_int, _c.c_float, _c.c_size_t

# name -> (restype, argtypes); mirrors include/b2ocr.h one to one
SIGNATURES = {
    "b2o_version": (_i, []),
    "b2o_create": (_i, [_i, _c.POINTER(_vp)]),
    "b2o_destroy": (None, [_vp]),
    "b2o_last_error": (_c.c_char_p, [_vp]),
    "b2o_set_conv_engine": (_i, [_vp, _i]),
    "b2o_launch_count": (_c.c_int64, [_vp]),
    "b2o_profile_enable": (_i, [_vp, _i]),
    "b2o_profile_read": (_i, [_vp, _c.POINTER(_c.c_double), _c.POINTER(_c.c_double), _c.POINTER(_c.c_int64)]),
    "b2o_load_craft": (_i, [_vp, _c.POINTER(_Tensor), _i]),
    "b2o_load_crnn": (_i, [_vp, _c.POINTER(_Tensor), _i]),
    "b2o_set_crnn_geometry": (_i, [_vp, _i, _i, _i]),
    "b2o_resize_pad": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _i, _i, _vp]),
    "b2o_resize_pad_batch": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _i, _i, _vp, _vp]),
    "b2o_jpeg_info": (_i, [_vp, _vp, _sz, _c.POINTER(_i), _c.POINTER(_i), _c.POINTER(_i)]),
    "b2o_decode_jpeg": (_i, [_vp, _vp, _sz, _vp, _i, _i, _vp]),
    "b2o_rgb_to_gray": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "b2o_craft_workspace_bytes": (_sz, [_i, _i, _i]),
    "b2o_craft_forward": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "b2o_boxes_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "b2o_get_boxes": (_i, [_vp, _vp, _i, _i, _i, _f, _f, _f, _i, _vp, _vp, _i, _vp, _sz, _vp]),
    "b2o_compact_boxes": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "b2o_record_floats": (_sz, [_i]),
    "b2o_record_floats_steps": (_sz, [_i, _i]),
    "b2o_pack_records": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "b2o_pack_records_steps": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "b2o_warp_boxes": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp]),
    "b2o_warp_boxes_color": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp]),
    "b2o_crops_to_input_color": (_i, [_vp, _vp, _i, _vp, _vp]),
    "b2o_fit_crops": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "b2o_crnn_workspace_bytes": (_sz, [_i]),
    "b2o_crnn_workspace_bytes_for": (_sz, [_vp, _i]),
    "b2o_crops_to_input": (_i, [_vp, _vp, _i, _vp, _vp]),
    "b2o_crnn_forward": (_i, [_vp, _vp, _i, _vp, _vp, _sz, _vp]),
    "b2o_set_debug_taps": (_i, [_vp, _i]),
    "b2o_crnn_tap": (_i, [_vp, _c.c_char_p, _vp, _i, _vp, _sz, _vp]),
    "b2o_conv2d_test": (_i, [_vp, _vp, _i, _i, _i, _i, _c.POINTER(_c.c_float), _i, _i, _i,
                             _c.POINTER(_c.c_float), _c.POINTER(_c.c_float), _i,
                             _c.POINTER(_c.c_float), _c.POINTER(_c.c_float), _vp, _i, _vp]),
}

_lib = None


def load_library():
    """dlopen libb2ocr.so and type every export of include/b2ocr.h (no GPU needed for this)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B2OError(f"{LIB_PATH} not found: build it with `python keras-ocr_b200/build.py` "
                       "(there is no CPU fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export the symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _tensor_array(weights):
    keep = []
    arr = (_Tensor * len(weights))()
    for k, (name, value) in enumerate(weights.items()):
        a = np.ascontiguousarray(np.asarray(value), dtype=np.float32)
        keep.append(a)
        arr[k].name = name.encode()
        arr[k].data = a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
        arr[k].ndim = a.ndim
        for d in range(a.ndim):
            arr[k].shape[d] = a.shape[d]
    return arr, keep


def _fptr(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float)) if a is not None else None


class Context:
    """One b2o_ctx per device.  All methods take raw device pointers (ints) and a stream (int)."""

    def __init__(self, device=0):
        self.lib = load_library()
        handle = _vp()
        rc = self.lib.b2o_create(int(device), ctypes.byref(handle))
        if rc != 0 or not handle:
            raise B2OError(f"b2o_create(device={device}) failed with status {rc}: an sm_100 (B200) GPU is "
                           "required and there is no CPU fallback")
        self.handle = handle
        self.device = device

    def close(self):
        if getattr(self, "handle", None):
            self.lib.b2o_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # pragma: no cover - interpreter shutdown
            pass

    def _check(self, rc, what):
        if rc != 0:
            msg = self.lib.b2o_last_error(self.handle)
            raise B2OError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")

    def set_conv_engine(self, engine):
        self._check(self.lib.b2o_set_conv_engine(self.handle, engine), "b2o_set_conv_engine")

    def launch_count(self):
        return int(self.lib.b2o_launch_count(self.handle))

    def profile_enable(self, on):
        self._check(self.lib.b2o_profile_enable(self.handle, int(on)), "b2o_profile_enable")

    def profile_read(self):
        ms, flop, n = ctypes.c_double(), ctypes.c_double(), ctypes.c_int64()
        self._check(self.lib.b2o_profile_read(self.handle, ctypes.byref(ms), ctypes.byref(flop), ctypes.byref(n)),
                    "b2o_profile_read")
        return ms.value, flop.value, n.value

    def load_craft(self, weights):
        arr, keep = _tensor_array(weights)
        self._check(self.lib.b2o_load_craft(self.handle, arr, len(weights)), "b2o_load_craft")

    def set_crnn_geometry(self, height, width, rnn_steps_to_discard):
        self._check(self.lib.b2o_set_crnn_geometry(self.handle, int(height), int(width), int(rnn_steps_to_discard)),
                    "b2o_set_crnn_geometry")

    def load_crnn(self, weights):
        arr, keep = _tensor_array(weights)
        self._check(self.lib.b2o_load_crnn(self.handle, arr, len(weights)), "b2o_load_crnn")

    def resize_pad(self, src, hs, ws, hr, wr, dst, index, hp, wp, stream):
        self._check(self.lib.b2o_resize_pad(self.handle, src, hs, ws, hr, wr, dst, index, hp, wp, stream), "b2o_resize_pad")

    def resize_pad_batch(self, src, n, hs, ws, hr, wr, dst, hp, wp, gray, stream):
        self._check(self.lib.b2o_resize_pad_batch(self.handle, src, n, hs, ws, hr, wr, dst, hp, wp, gray, stream),
                    "b2o_resize_pad_batch")

    def jpeg_info(self, data):
        """(height, width, components) of a JPEG byte string, or None if nvJPEG is missing / refuses the stream."""
        buf = (ctypes.c_ubyte * len(data)).from_buffer_copy(data)
        h, w, c = _i(), _i(), _i()
        rc = self.lib.b2o_jpeg_info(self.handle, buf, len(data), ctypes.byref(h), ctypes.byref(w), ctypes.byref(c))
        return (h.value, w.value, c.value) if rc == 0 else None

    def decode_jpeg(self, data, rgb, h, w, stream):
        buf = (ctypes.c_ubyte * len(data)).from_buffer_copy(data)
        return self.lib.b2o_decode_jpeg(self.handle, buf, len(data), rgb, h, w, stream) == 0

    def rgb_to_gray(self, img, n, h, w, gray, stream):
        self._check(self.lib.b2o_rgb_to_gray(self.handle, img, n, h, w, gray, stream), "b2o_rgb_to_gray")

    def craft_workspace_bytes(self, n, h, w):
        return int(self.lib.b2o_craft_workspace_bytes(n, h, w))

    def craft_forward(self, img, n, h, w, scores, ws, ws_bytes, stream):
        self._check(self.lib.b2o_craft_forward(self.handle, img, n, h, w, scores, ws, ws_bytes, stream), "b2o_craft_forward")

    def boxes_workspace_bytes(self, n, hs, ws, max_boxes):
        return int(self.lib.b2o_boxes_workspace_bytes(n, hs, ws, max_boxes))

    def get_boxes(self, scores, n, hs, ws, det, text, link, size, boxes, counts, max_boxes, wsp, ws_bytes, stream):
        self._check(self.lib.b2o_get_boxes(self.handle, scores, n, hs, ws, det, text, link, size, boxes, counts,
                                           max_boxes, wsp, ws_bytes, stream), "b2o_get_boxes")

    def compact_boxes(self, boxes, counts, n, max_boxes, flat, image_index, stream):
        self._check(self.lib.b2o_compact_boxes(self.handle, boxes, counts, n, max_boxes, flat, image_index, stream),
                    "b2o_compact_boxes")

    def record_floats(self, rec_boxes, steps=None):
        if steps is None:
            return int(self.lib.b2o_record_floats(rec_boxes))
        return int(self.lib.b2o_record_floats_steps(rec_boxes, int(steps)))

    def pack_records(self, boxes, counts, labels, inv_scale, n, max_boxes, rows, rec_boxes, records, stream, steps=None):
        if steps is None:
            self._check(self.lib.b2o_pack_records(self.handle, boxes, counts, labels, inv_scale, n, max_boxes, rows,
                                                  rec_boxes, records, stream), "b2o_pack_records")
        else:
            self._check(self.lib.b2o_pack_records_steps(self.handle, boxes, counts, labels, inv_scale, n, max_boxes, rows,
                                                        rec_boxes, int(steps), records, stream), "b2o_pack_records_steps")

    def warp_boxes(self, gray, n, h, w, boxes, image_index, n_boxes, crops, crnn_in, stream, color=False):
        fn = self.lib.b2o_warp_boxes_color if color else self.lib.b2o_warp_boxes
        self._check(fn(self.handle, gray, n, h, w, boxes, image_index, n_boxes, crops, crnn_in, stream), "b2o_warp_boxes")

    def crnn_workspace_bytes(self, b):
        """Workspace of b2o_crnn_forward at this context's crop geometry (b2o_crnn_workspace_bytes_for)."""
        return int(self.lib.b2o_crnn_workspace_bytes_for(self.handle, b))

    def crops_to_input(self, crops, b, crnn_in, stream, color=False):
        fn = self.lib.b2o_crops_to_input_color if color else self.lib.b2o_crops_to_input
        self._check(fn(self.handle, crops, b, crnn_in, stream), "b2o_crops_to_input")

    def fit_crops(self, srcs, dims, b, crops, crnn_in, stream):
        """srcs: device array of b crop pointers; dims: device (b, 4) int32 (sh, sw, rh, rw); crops nullable."""
        self._check(self.lib.b2o_fit_crops(self.handle, srcs, dims, b, crops, crnn_in, stream), "b2o_fit_crops")

    def crnn_forward(self, crnn_in, b, labels, ws, ws_bytes, stream):
        self._check(self.lib.b2o_crnn_forward(self.handle, crnn_in, b, labels, ws, ws_bytes, stream), "b2o_crnn_forward")

    def set_debug_taps(self, on):
        self._check(self.lib.b2o_set_debug_taps(self.handle, int(on)), "b2o_set_debug_taps")

    def crnn_tap(self, name, ws, b, out, out_bytes, stream):
        self._check(self.lib.b2o_crnn_tap(self.handle, name.encode(), ws, b, out, out_bytes, stream), "b2o_crnn_tap")

    def conv2d_test(self, x, n, h, w, cin, wgt, cout, ksize, dilation, s1, t1, relu, s2, t2, out, engine, stream):
        wgt = np.ascontiguousarray(wgt, np.float32)
        s1 = np.ascontiguousarray(s1, np.float32)
        t1 = np.ascontiguousarray(t1, np.float32)
        s2 = None if s2 is None else np.ascontiguousarray(s2, np.float32)
        t2 = None if t2 is None else np.ascontiguousarray(t2, np.float32)
        self._check(self.lib.b2o_conv2d_test(self.handle, x, n, h, w, cin, _fptr(wgt), cout, ksize, dilation, _fptr(s1),
                                             _fptr(t1), int(relu), _fptr(s2), _fptr(t2), out, engine, stream),
                    "b2o_conv2d_test")


_contexts = {}


def get_context(device=0):
    """Process-wide context cache (weights are loaded per owner object, see Detector/Recognizer)."""
    if device not in _contexts:
        _contexts[device] = Context(device)
    return _contexts[device]
