"""ctypes binding to the libjpeg-turbo that Pillow bundles (test oracle): lossless JPEG (SOF3) of 2- to 16-bit
grayscale, written and read by an implementation that shares nothing with this project.

    encode(img, P, predictor, pt=0, restart_in_rows=0) -> bytes     input samples must be < 2^P; their low pt bits
                                                                    are dropped, as the point transform does
    decode(stream) -> (rows, cols) uint16                           any lossless stream
    encode_many / decode_many_with_header                           the same for a list, in one child process
    available() / version()

The API follows the precision: jpeg_*_scanlines for P <= 8, jpeg12_* for P <= 12, jpeg16_* above.  libjpeg's default
error handler calls exit(), so every libjpeg call runs in a child process (this file run as a script); a stream it
rejects raises LibjpegError in the caller instead of ending it.

The binding writes struct fields at fixed offsets of jpeg_compress_struct / jpeg_decompress_struct as libjpeg-turbo
3.x lays them out on LP64 (JPEG_LIB_VERSION 62); jpeg_Create* checks the struct sizes, and
tests/test_dicom_conformance.py pins the offsets with round trips (SOF3 / DRI fields and the decoded header).
"""
import ctypes as C
import glob
import importlib.util
import os
import pickle
import struct
import subprocess
import sys

import numpy as np

JPEG_LIB_VERSION = 62
COMPRESS_SIZE, DECOMPRESS_SIZE = 520, 632
# jpeg_compress_struct
C_IMAGE_WIDTH, C_IMAGE_HEIGHT, C_INPUT_COMPONENTS, C_IN_COLOR_SPACE, C_DATA_PRECISION = 48, 52, 56, 60, 72
C_RESTART_IN_ROWS = 284
# jpeg_decompress_struct
D_IMAGE_WIDTH, D_IMAGE_HEIGHT, D_NUM_COMPONENTS, D_OUTPUT_WIDTH, D_OUTPUT_HEIGHT, D_OUTPUT_COMPONENTS = 48, 52, 56, 136, 140, 148
D_DATA_PRECISION = 296
JCS_GRAYSCALE = 1


class LibjpegError(RuntimeError):
    pass


def library_path():
    """libjpeg.so.62 from Pillow's wheel (pillow.libs next to the PIL package), or None."""
    spec = importlib.util.find_spec("PIL")
    if spec is None or not spec.submodule_search_locations:
        return None
    libs = os.path.join(os.path.dirname(list(spec.submodule_search_locations)[0]), "pillow.libs")
    found = sorted(glob.glob(os.path.join(libs, "libjpeg-*.so*")))
    return found[0] if found else None


def _load():
    p = library_path()
    if p is None:
        return None
    try:
        L = C.CDLL(p)
    except OSError:
        return None
    needed = ["jpeg_std_error", "jpeg_CreateCompress", "jpeg_CreateDecompress", "jpeg_enable_lossless", "jpeg_mem_dest",
              "jpeg_mem_src"] + ["jpeg%s_%s_scanlines" % (b, rw) for b in ("", "12", "16") for rw in ("read", "write")]
    return L if all(hasattr(L, s) for s in needed) else None


def available():
    return _load() is not None


def version():
    """Pillow's report of its libjpeg-turbo version, e.g. '3.1.4.1'."""
    from PIL import features
    return features.version("libjpeg_turbo")


def _api(P):
    return ("", np.uint8) if P <= 8 else ("12", np.int16) if P <= 12 else ("16", np.uint16)


def _rows(a):
    base = a.ctypes.data
    return (C.c_void_p * a.shape[0])(*[base + r * a.strides[0] for r in range(a.shape[0])])


def _new(L, size):
    err = C.create_string_buffer(1024)                      # jpeg_error_mgr (168 bytes in 3.1), with room to spare
    L.jpeg_std_error.restype = C.c_void_p
    L.jpeg_std_error(err)
    info = C.create_string_buffer(size)
    struct.pack_into("<Q", info, 0, C.addressof(err))       # jpeg_common_fields: err first
    return info, err


def _child_encode(L, P, predictor, pt, restart_in_rows, H, W, raw):
    info, err = _new(L, COMPRESS_SIZE)
    L.jpeg_CreateCompress(info, JPEG_LIB_VERSION, COMPRESS_SIZE)
    outbuf, outsize = C.c_void_p(), C.c_ulong()
    L.jpeg_mem_dest(info, C.byref(outbuf), C.byref(outsize))
    struct.pack_into("<IIii", info, C_IMAGE_WIDTH, W, H, 1, JCS_GRAYSCALE)
    struct.pack_into("<i", info, C_DATA_PRECISION, P)
    L.jpeg_set_defaults(info)
    struct.pack_into("<i", info, C_DATA_PRECISION, P)
    L.jpeg_enable_lossless(info, predictor, pt)
    struct.pack_into("<i", info, C_RESTART_IN_ROWS, restart_in_rows)
    L.jpeg_start_compress(info, 1)
    suffix, dt = _api(P)
    a = np.ascontiguousarray(np.frombuffer(raw, "<u2").reshape(H, W).astype(dt))
    rows = _rows(a)
    write = getattr(L, "jpeg%s_write_scanlines" % suffix)
    done = 0
    while done < H:
        done += write(info, C.byref(rows, done * C.sizeof(C.c_void_p)), H - done)
    L.jpeg_finish_compress(info)
    out = C.string_at(outbuf, outsize.value)
    L.jpeg_destroy_compress(info)
    return out


def _child_decode(L, stream):
    info, err = _new(L, DECOMPRESS_SIZE)
    L.jpeg_CreateDecompress(info, JPEG_LIB_VERSION, DECOMPRESS_SIZE)
    src = C.create_string_buffer(stream, len(stream))
    L.jpeg_mem_src(info, src, C.c_ulong(len(stream)))
    L.jpeg_read_header(info, 1)
    W, H, nc = struct.unpack_from("<IIi", info, D_IMAGE_WIDTH)
    P = struct.unpack_from("<i", info, D_DATA_PRECISION)[0]
    if nc != 1:
        raise SystemExit("%d components" % nc)
    L.jpeg_start_decompress(info)
    ow, oh = struct.unpack_from("<II", info, D_OUTPUT_WIDTH)
    oc = struct.unpack_from("<i", info, D_OUTPUT_COMPONENTS)[0]
    if (ow, oh, oc) != (W, H, 1):
        raise SystemExit("output %d x %d x %d" % (oh, ow, oc))
    suffix, dt = _api(P)
    a = np.zeros((H, W), dt)
    rows = _rows(a)
    read = getattr(L, "jpeg%s_read_scanlines" % suffix)
    done = 0
    while done < H:
        done += read(info, C.byref(rows, done * C.sizeof(C.c_void_p)), H - done)
    L.jpeg_finish_decompress(info)
    L.jpeg_destroy_decompress(info)
    return struct.pack("<III", H, W, P) + a.astype("<u2").tobytes()


def _run(op, items):
    """Runs the jobs in one child process; if it fails, once more one job per child, so that a stream libjpeg-turbo
    rejects raises only for itself."""
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], input=pickle.dumps((op, items)), capture_output=True,
                       timeout=600)
    if r.returncode == 0:
        return pickle.loads(r.stdout)
    if len(items) > 1:
        return [_run(op, [it])[0] for it in items]
    raise LibjpegError("libjpeg-turbo %s: exit %d: %s" % (op, r.returncode, r.stderr.decode(errors="replace").strip()))


def encode_many(jobs):
    """jobs: (img, P, predictor, pt, restart_in_rows) tuples -> list of streams."""
    items = []
    for img, P, predictor, pt, restart_in_rows in jobs:
        img = np.asarray(img)
        assert img.ndim == 2 and 2 <= P <= 16 and 1 <= predictor <= 7 and 0 <= pt < P
        assert img.min(initial=0) >= 0 and img.max(initial=0) < (1 << P)
        items.append((P, predictor, pt, restart_in_rows, img.shape[0], img.shape[1], img.astype("<u2").tobytes()))
    return _run("encode", items)


def encode(img, P, predictor, pt=0, restart_in_rows=0):
    return encode_many([(img, P, predictor, pt, restart_in_rows)])[0]


def decode_many_with_header(streams):
    """-> list of (samples (rows, cols) uint16, data_precision as libjpeg-turbo read it); LibjpegError if any fails."""
    out = []
    for res in _run("decode", [bytes(s) for s in streams]):
        H, W, P = struct.unpack_from("<III", res)
        out.append((np.frombuffer(res, "<u2", offset=12).reshape(H, W).astype(np.uint16), P))
    return out


def decode(stream):
    return decode_many_with_header([stream])[0][0]


if __name__ == "__main__":
    lib = _load()
    if lib is None:
        raise SystemExit("libjpeg-turbo unavailable")
    op, items = pickle.loads(sys.stdin.buffer.read())
    if op == "encode":
        res = [_child_encode(lib, *it) for it in items]
    else:
        res = [_child_decode(lib, it) for it in items]
    sys.stdout.buffer.write(pickle.dumps(res))
