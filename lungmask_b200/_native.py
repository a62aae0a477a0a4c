"""ctypes binding of liblungmask_b200.so (include/lungmask_b200.h).  No torch types cross this boundary."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblungmask_b200.so")

NET_RES = 256
FLAG_NO_POSTPROCESS = 1

_lib = None


class NativeError(RuntimeError):
    pass


def lib():
    """Loads the CUDA library; fails loudly when it has not been built (there is no CPU fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            "%s is missing: build it with `python -m lungmask_b200.build` (needs nvcc, sm_100a). "
            "lungmask_b200 has no CPU or eager-PyTorch fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32, u8p, i16p, i32p, f32p = C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p
    sig = {
        "lm_create": ([i32, i32, C.POINTER(vp)], i32),
        "lm_destroy": ([vp], None),
        "lm_last_error": ([], C.c_char_p),
        "lm_device": ([vp], i32),
        "lm_batch_capacity": ([vp], i32),
        "lm_weight_blob_floats": ([i32], C.c_size_t),
        "lm_load_weights": ([vp, i32, f32p, C.c_size_t, i32], i32),
        "lm_apply_volume": ([vp, i32, i16p, i32, i32, i32, i32, u8p], i32),
        "lm_apply_volume_dev": ([vp, i32, i16p, i32, i32, i32, i32, u8p], i32),
        "lm_apply_fused": ([vp, i32, i32, i16p, i32, i32, i32, i32, u8p], i32),
        "lm_apply_fused_dev": ([vp, i32, i32, i16p, i32, i32, i32, i32, u8p], i32),
        "lm_apply_volume_float": ([vp, i32, i32, vp, i32, i32, i32, i32, i32, u8p], i32),
        "lm_preprocess_float": ([vp, vp, i32, i32, i32, i32, f32p, i32p], i32),
        "lm_apply_volume_oriented": ([vp, i32, i32, i16p, i32, i32, i32, vp, vp, i32, u8p], i32),
        "lm_shard_init": ([vp, i32, i32, i32], i32),
        "lm_shard_handle_bytes": ([], C.c_size_t),
        "lm_shard_export": ([vp, vp], i32),
        "lm_shard_connect": ([vp, vp], i32),
        "lm_shard_labels": ([vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_size_t)], i32),
        "lm_apply_volume_sharded": ([vp, i32, i16p, i32, i32, i32, i32, u8p], i32),
        "lm_apply_volume_sharded_dev": ([vp, i32, i16p, i32, i32, i32, i32, u8p], i32),
        "lm_fuse": ([vp, u8p, u8p, i32, i32, i32, u8p, C.POINTER(i32)], i32),
        "lm_preprocess": ([vp, i16p, i32, i32, i32, i32, i32, i32, i16p, i32p], i32),
        "lm_simple_bodymask": ([vp, i16p, i32, i32, u8p], i32),
        "lm_forward": ([vp, i32, i16p, i32, u8p, f32p], i32),
        "lm_forward_dev": ([vp, i32, i16p, i32, u8p, C.POINTER(C.c_float)], i32),
        "lm_postprocess": ([vp, u8p, i32, i32, i32, i32p, i32, i32, u8p], i32),
        "lm_reshape_masks": ([vp, u8p, i32, i32, i32p, i32, i32, i32, u8p], i32),
        "lm_keep_largest_component": ([vp, u8p, i32, i32, i32, u8p], i32),
        "lm_last_timings": ([vp, C.POINTER(C.c_float), C.POINTER(C.c_int64)], i32),
        "lm_set_option": ([vp, C.c_char_p, i32], i32),
        "lm_debug_activation_info": ([i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)], i32),
        "lm_debug_read_activation": ([vp, i32, i32, f32p], i32),
        "lm_last_conv_timing": ([vp, C.POINTER(C.c_float), C.POINTER(C.c_int64)], i32),
        "lm_decode_frames": ([i32, u8p, C.c_size_t, vp, i32, vp, i32p], i32),
    }
    for name, (argtypes, restype) in sig.items():
        fn = getattr(L, name)  # AttributeError here = header / library mismatch
        fn.argtypes, fn.restype = argtypes, restype
    _lib = L
    return L


EXPORTS = ["lm_create", "lm_destroy", "lm_last_error", "lm_device", "lm_batch_capacity", "lm_weight_blob_floats",
           "lm_load_weights", "lm_apply_volume", "lm_apply_volume_dev", "lm_apply_fused", "lm_apply_fused_dev", "lm_apply_volume_oriented", "lm_apply_volume_float", "lm_preprocess_float", "lm_fuse", "lm_preprocess",
           "lm_shard_init", "lm_shard_handle_bytes", "lm_shard_export", "lm_shard_connect", "lm_shard_labels",
           "lm_apply_volume_sharded", "lm_apply_volume_sharded_dev",
           "lm_simple_bodymask", "lm_forward", "lm_forward_dev", "lm_postprocess", "lm_reshape_masks",
           "lm_keep_largest_component",
           "lm_last_timings", "lm_set_option", "lm_last_conv_timing",
           "lm_debug_activation_info", "lm_debug_read_activation", "lm_decode_frames"]


CODEC_JPEG_LOSSLESS, CODEC_RLE = 1, 2
DECODE_ERRORS = {-60: "unsupported or malformed JPEG marker segments or RLE header",
                 -61: "malformed entropy-coded data",
                 -62: "the data ends before Rows x Columns samples or does not match the restart intervals"}
FRAME_DTYPE = np.dtype([("offset", "<u8"), ("length", "<u8"), ("codec", "<i4"), ("rows", "<i4"), ("cols", "<i4"),
                        ("is_signed", "<i4")])   # lm_frame


def decode_frames(data, frames, device=0):
    """lm_decode_frames: `data` bytes, `frames` a FRAME_DTYPE array -> (list of (rows, cols) uint16 arrays, int32 status
    per frame).  Needs no Engine."""
    frames = np.ascontiguousarray(frames, dtype=FRAME_DTYPE)
    buf = np.frombuffer(data, dtype=np.uint8) if len(data) else np.zeros(1, np.uint8)
    sizes = frames["rows"].astype(np.int64) * frames["cols"].astype(np.int64)
    out = np.empty(int(sizes.sum()), np.uint16)
    status = np.zeros(len(frames), np.int32)
    _check(lib().lm_decode_frames(int(device), _ptr(buf), len(data), _ptr(frames), len(frames), _ptr(out), _ptr(status)))
    ends = np.cumsum(sizes)
    return [out[e - n:e].reshape(int(r), int(c)) for e, n, r, c in zip(ends, sizes, frames["rows"], frames["cols"])], status


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


def _check(rc):
    if rc != 0:
        raise NativeError("lungmask_b200 native call failed (%d): %s" % (rc, lib().lm_last_error().decode()))


def _as(a, dtype, ndim=None):
    """C-contiguous array of `dtype` for the C ABI.  Only value-preserving conversions happen here: a float volume is
    never truncated and an int32 / uint16 volume never wraps silently (integers of another width are range-checked);
    LMInferer / utils do the reference-compatible dtype handling before they get here."""
    a = np.asarray(a)
    dtype = np.dtype(dtype)
    if a.dtype != dtype:
        if a.dtype == bool or np.can_cast(a.dtype, dtype, casting="safe"):
            pass
        elif np.issubdtype(a.dtype, np.integer) and np.issubdtype(dtype, np.integer):
            info = np.iinfo(dtype)
            if a.size and (a.min() < info.min or a.max() > info.max):
                raise TypeError("values of the %s array do not fit %s" % (a.dtype, dtype))
        else:
            raise TypeError("refusing to convert %s to %s (lossy); convert explicitly" % (a.dtype, dtype))
    a = np.ascontiguousarray(a, dtype=dtype)
    if ndim is not None and a.ndim != ndim:
        raise ValueError("expected %d-d array, got shape %s" % (ndim, a.shape))
    return a


class Engine:
    """One engine = one CUDA device (see lm_create)."""

    def __init__(self, device=0, batch_capacity=20):
        self._h = C.c_void_p()
        _check(lib().lm_create(int(device), int(batch_capacity), C.byref(self._h)))
        self.device, self.batch_capacity = int(device), int(batch_capacity)
        self.n_classes = {}

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib().lm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- weights
    def load_weights(self, slot, blob, n_classes):
        blob = _as(blob, np.float32, 1)
        _check(lib().lm_load_weights(self._h, slot, _ptr(blob), blob.size, int(n_classes)))
        self.n_classes[slot] = int(n_classes)

    # ---- whole path
    def apply_volume(self, slot, vol, postprocess=True, out=None):
        vol = _as(vol, np.int16, 3)
        if out is None:
            out = np.empty(vol.shape, np.uint8)
        assert out.dtype == np.uint8 and out.shape == vol.shape and out.flags.c_contiguous
        S, H, W = vol.shape
        _check(lib().lm_apply_volume(self._h, slot, _ptr(vol), S, H, W, 0 if postprocess else FLAG_NO_POSTPROCESS, _ptr(out)))
        return out

    def apply_volume_dev(self, slot, d_vol_ptr, shape, d_out_ptr, postprocess=True):
        S, H, W = shape
        _check(lib().lm_apply_volume_dev(self._h, slot, C.c_void_p(d_vol_ptr), S, H, W,
                                         0 if postprocess else FLAG_NO_POSTPROCESS, C.c_void_p(d_out_ptr)))

    def apply_fused(self, slot_base, slot_fill, vol, postprocess=True):
        """`postprocess` = LMInferer.volume_postprocessing: it reaches the two inner inferences only (mask.py:191-194);
        the fusion post-processing (mask.py:232) always runs."""
        vol = _as(vol, np.int16, 3)
        out = np.empty(vol.shape, np.uint8)
        S, H, W = vol.shape
        _check(lib().lm_apply_fused(self._h, slot_base, slot_fill, _ptr(vol), S, H, W,
                                    0 if postprocess else FLAG_NO_POSTPROCESS, _ptr(out)))
        return out

    def apply_fused_dev(self, slot_base, slot_fill, d_vol_ptr, shape, d_out_ptr, postprocess=True):
        S, H, W = shape
        _check(lib().lm_apply_fused_dev(self._h, slot_base, slot_fill, C.c_void_p(d_vol_ptr), S, H, W,
                                        0 if postprocess else FLAG_NO_POSTPROCESS, C.c_void_p(d_out_ptr)))

    def apply_volume_float(self, slot, vol, slot_fill=-1, postprocess=True):
        """float32 / float64 HU volume (the dtype is kept through pre-processing and normalisation, as the reference does)."""
        vol = np.asarray(vol)
        if vol.dtype not in (np.float32, np.float64):
            raise TypeError("apply_volume_float expects float32 or float64, got %s" % vol.dtype)
        vol = _as(vol, vol.dtype, 3)
        out = np.empty(vol.shape, np.uint8)
        S, H, W = vol.shape
        _check(lib().lm_apply_volume_float(self._h, slot, int(slot_fill), _ptr(vol), 1 if vol.dtype == np.float64 else 0, S, H, W,
                                           0 if postprocess else FLAG_NO_POSTPROCESS, _ptr(out)))
        return out

    def preprocess_float(self, vol):
        vol = np.asarray(vol)
        if vol.dtype not in (np.float32, np.float64):
            raise TypeError("preprocess_float expects float32 or float64, got %s" % vol.dtype)
        vol = _as(vol, vol.dtype, 3)
        S, H, W = vol.shape
        norm = np.empty((S, NET_RES, NET_RES), np.float32)
        boxes = np.empty((S, 4), np.int32)
        _check(lib().lm_preprocess_float(self._h, _ptr(vol), 1 if vol.dtype == np.float64 else 0, S, H, W, _ptr(norm), _ptr(boxes)))
        return norm, boxes

    def apply_volume_oriented(self, slot, vol, perm, flip, slot_fill=-1, postprocess=True):
        """`vol` in its native orientation; (perm, flip) = lungmask_b200.orient.array_transform_to_lps(code)."""
        vol = _as(vol, np.int16, 3)
        out = np.empty(vol.shape, np.uint8)
        pa = (C.c_int * 3)(*[int(x) for x in perm])
        fa = (C.c_int * 3)(*[1 if x else 0 for x in flip])
        n0, n1, n2 = vol.shape
        _check(lib().lm_apply_volume_oriented(self._h, slot, int(slot_fill), _ptr(vol), n0, n1, n2, pa, fa,
                                              0 if postprocess else FLAG_NO_POSTPROCESS, _ptr(out)))
        return out

    # ---- one volume over several GPUs (one engine per rank; see include/lungmask_b200.h)
    def shard_init(self, rank, world, max_slices):
        _check(lib().lm_shard_init(self._h, int(rank), int(world), int(max_slices)))
        self.shard_rank, self.shard_world = int(rank), int(world)

    def shard_export(self):
        buf = C.create_string_buffer(int(lib().lm_shard_handle_bytes()))
        _check(lib().lm_shard_export(self._h, C.cast(buf, C.c_void_p)))
        return buf.raw

    def shard_connect(self, handles):
        """`handles`: the ranks' shard_export() results in rank order."""
        blob = b"".join(bytes(h) for h in handles)
        if len(blob) != self.shard_world * int(lib().lm_shard_handle_bytes()):
            raise ValueError("shard_connect expects %d handles" % self.shard_world)
        buf = C.create_string_buffer(blob, len(blob))
        _check(lib().lm_shard_connect(self._h, C.cast(buf, C.c_void_p)))

    def shard_labels(self):
        """(device pointer of the gathered boxes, device pointer of the gathered labels, slice capacity)"""
        b, l, cap = C.c_void_p(), C.c_void_p(), C.c_size_t(0)
        _check(lib().lm_shard_labels(self._h, C.byref(b), C.byref(l), C.byref(cap)))
        return b.value, l.value, int(cap.value)

    def apply_volume_sharded(self, slot, vol, postprocess=True, want_output=True):
        vol = _as(vol, np.int16, 3)
        S, H, W = vol.shape
        out = np.empty(vol.shape, np.uint8) if want_output else None
        _check(lib().lm_apply_volume_sharded(self._h, slot, _ptr(vol), S, H, W, 0 if postprocess else FLAG_NO_POSTPROCESS,
                                             _ptr(out) if out is not None else None))
        return out

    def apply_volume_sharded_dev(self, slot, d_vol_ptr, shape, d_out_ptr, postprocess=True):
        S, H, W = shape
        _check(lib().lm_apply_volume_sharded_dev(self._h, slot, C.c_void_p(d_vol_ptr), S, H, W,
                                                 0 if postprocess else FLAG_NO_POSTPROCESS, C.c_void_p(d_out_ptr)))

    def fuse(self, res_l, res_r):
        """mask.py:228-230 -> (fused uint8 volume before the post-processing, spare value)."""
        res_l, res_r = _as(res_l, np.uint8, 3), _as(res_r, np.uint8, 3)
        if res_l.shape != res_r.shape:
            raise ValueError("fuse: shapes differ")
        out = np.empty(res_l.shape, np.uint8)
        spare = C.c_int(0)
        S, H, W = res_l.shape
        _check(lib().lm_fuse(self._h, _ptr(res_l), _ptr(res_r), S, H, W, _ptr(out), C.byref(spare)))
        return out, int(spare.value)

    # ---- stages
    def preprocess(self, vol, out_h=NET_RES, out_w=NET_RES, clip=True):
        vol = _as(vol, np.int16, 3)
        S, H, W = vol.shape
        resized = np.empty((S, out_h, out_w), np.int16)
        boxes = np.empty((S, 4), np.int32)
        _check(lib().lm_preprocess(self._h, _ptr(vol), S, H, W, out_h, out_w, 1 if clip else 0, _ptr(resized), _ptr(boxes)))
        return resized, boxes

    def simple_bodymask(self, img):
        img = _as(img, np.int16, 2)
        out = np.empty(img.shape, np.uint8)
        _check(lib().lm_simple_bodymask(self._h, _ptr(img), img.shape[0], img.shape[1], _ptr(out)))
        return out

    def forward(self, slot, resized, return_scores=False):
        resized = _as(resized, np.int16, 3)
        S = resized.shape[0]
        if resized.shape[1:] != (NET_RES, NET_RES):
            raise ValueError("forward expects (S,256,256) slices")
        labels = np.empty((S, NET_RES, NET_RES), np.uint8)
        scores = None
        if return_scores:
            scores = np.empty((S, self.n_classes[slot], NET_RES, NET_RES), np.float32)
        _check(lib().lm_forward(self._h, slot, _ptr(resized), S, _ptr(labels), _ptr(scores) if scores is not None else None))
        return (labels, scores) if return_scores else labels

    def forward_dev(self, slot, d_resized_ptr, S, d_labels_ptr):
        ms = C.c_float(0)
        _check(lib().lm_forward_dev(self._h, slot, C.c_void_p(d_resized_ptr), S, C.c_void_p(d_labels_ptr), C.byref(ms)))
        return float(ms.value)

    def postprocess(self, labels, spare=(), skip_below=3):
        labels = _as(labels, np.uint8, 3)
        S, H, W = labels.shape
        sp = np.asarray(list(spare), dtype=np.int32)
        out = np.empty(labels.shape, np.uint8)
        _check(lib().lm_postprocess(self._h, _ptr(labels), S, H, W, _ptr(sp) if sp.size else None, int(sp.size), int(skip_below), _ptr(out)))
        return out

    def keep_largest_component(self, mask):
        mask = _as(mask, np.uint8, 3)
        out = np.empty(mask.shape, np.uint8)
        _check(lib().lm_keep_largest_component(self._h, _ptr(mask), mask.shape[0], mask.shape[1], mask.shape[2], _ptr(out)))
        return out

    def reshape_masks(self, masks, boxes, H, W):
        masks = _as(masks, np.uint8, 3)
        boxes = _as(boxes, np.int32, 2)
        S = masks.shape[0]
        out = np.empty((S, H, W), np.uint8)
        _check(lib().lm_reshape_masks(self._h, _ptr(masks), masks.shape[1], masks.shape[2], _ptr(boxes), S, H, W, _ptr(out)))
        return out

    def read_activation(self, act_id, n):
        lv, ch, sp = C.c_int(0), C.c_int(0), C.c_int(0)
        _check(lib().lm_debug_activation_info(act_id, C.byref(lv), C.byref(ch), C.byref(sp)))
        hw = NET_RES >> lv.value
        out = np.empty((n, hw, hw, ch.value), np.float32)
        _check(lib().lm_debug_read_activation(self._h, act_id, n, _ptr(out)))
        return out

    def set_option(self, key, value):
        _check(lib().lm_set_option(self._h, key.encode(), int(value)))

    def last_conv_timing(self):
        ms, n = C.c_float(0), C.c_int64(0)
        _check(lib().lm_last_conv_timing(self._h, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def last_timings(self):
        ms = (C.c_float * 7)()
        n = C.c_int64(0)
        _check(lib().lm_last_timings(self._h, ms, C.byref(n)))
        keys = ["h2d", "preprocess", "forward", "postprocess", "reshape", "d2h", "total"]
        d = {k: float(v) for k, v in zip(keys, ms)}
        d["kernel_launches"] = int(n.value)
        return d
