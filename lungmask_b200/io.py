"""Volume ingest and write-back without SimpleITK / pydicom (the reference's `utils.read_dicoms`, `utils.load_input_image`
and the `sitk.WriteImage` of `__main__.py`: lungmask/utils.py:132-269, lungmask/__main__.py:119-144).

The reference leans on SimpleITK (ITK / GDCM) and pydicom for this; neither is in this image, and the accelerated path
only needs three things from a file: the voxel array (z, y, x), the 3x3 direction cosines (for the orientation
handling of mask.py:157-164) and enough geometry to write the mask back next to the input.  So this module reads

  * DICOM series (a directory tree): uncompressed little-endian transfer syntaxes (implicit / explicit VR), and JPEG
    Lossless (.4.57, .4.70) and RLE Lossless (.5) single-frame encapsulated pixel data, decoded on the GPU by
    lm_decode_frames in one call per series; 16-bit pixels, RescaleSlope / RescaleIntercept applied as ITK does; slices grouped by SeriesInstanceUID, de-duplicated by
    (study, series, position) and sorted by the z component of ImagePositionPatient exactly like utils.py:196-214;
    the largest series wins (utils.py:262-268); ImageType filters `primary` / `original` as in utils.py:152-170;
  * NIfTI-1 single files (.nii, .nii.gz): sform, else qform, else pixdim; RAS -> LPS like ITK's NIfTI reader;
  * MetaImage (.mha, and .mhd + raw), uncompressed;
  * .npy (array only, identity geometry);

and writes masks as .nii / .nii.gz / .mha / .npy with the input's geometry.  DICOM tags are never copied into the
output (what `--removemetadata` asks for is therefore always the case here).
"""
import gzip
import os
import struct
from dataclasses import dataclass, field

import numpy as np

from .logger import logger


@dataclass
class Volume:
    array: np.ndarray                      # (z, y, x)
    spacing: tuple = (1.0, 1.0, 1.0)       # (x, y, z) mm
    origin: tuple = (0.0, 0.0, 0.0)        # LPS mm
    direction: tuple = (1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0)   # row-major 3x3, columns = image axes x, y, z in LPS
    meta: dict = field(default_factory=dict)

    def GetDirection(self):                # the two SimpleITK accessors LMInferer.apply needs
        return tuple(self.direction)

    def GetSize(self):
        return tuple(int(n) for n in self.array.shape[::-1])


# --------------------------------------------------------------------------------------------------------------
# DICOM
# --------------------------------------------------------------------------------------------------------------
_LONG_VR = {b"OB", b"OW", b"OF", b"SQ", b"UT", b"UN", b"OD", b"OL", b"UC", b"UR", b"OV", b"SV", b"UV"}
_EXPLICIT_LE, _IMPLICIT_LE = "1.2.840.10008.1.2.1", "1.2.840.10008.1.2"
_CODECS = {"1.2.840.10008.1.2.4.57": 1, "1.2.840.10008.1.2.4.70": 1, "1.2.840.10008.1.2.5": 2}   # lm_frame.codec
_WANTED = {(0x0008, 0x0008): "ImageType", (0x0020, 0x000D): "StudyInstanceUID", (0x0020, 0x000E): "SeriesInstanceUID",
           (0x0020, 0x0032): "ImagePositionPatient", (0x0020, 0x0037): "ImageOrientationPatient", (0x0028, 0x0010): "Rows",
           (0x0028, 0x0011): "Columns", (0x0028, 0x0030): "PixelSpacing", (0x0028, 0x0100): "BitsAllocated",
           (0x0028, 0x0103): "PixelRepresentation", (0x0028, 0x1052): "RescaleIntercept", (0x0028, 0x1053): "RescaleSlope",
           (0x0028, 0x0002): "SamplesPerPixel", (0x0018, 0x0050): "SliceThickness", (0x0028, 0x0008): "NumberOfFrames"}


class DicomError(ValueError):
    pass


def _skip_sequence(b, pos, explicit):
    """Skips an undefined-length sequence / item: walks items until the matching delimiter."""
    while pos + 8 <= len(b):
        g, e, ln = struct.unpack_from("<HHI", b, pos)
        pos += 8
        if (g, e) == (0xFFFE, 0xE0DD):      # sequence delimiter
            return pos
        if (g, e) == (0xFFFE, 0xE000):      # item
            if ln != 0xFFFFFFFF:
                pos += ln
            else:
                pos = _skip_items(b, pos, explicit)
        else:
            raise DicomError("malformed sequence")
    return pos


def _skip_items(b, pos, explicit):
    """Inside an undefined-length item: walks data elements until the item delimiter."""
    while pos + 8 <= len(b):
        g, e = struct.unpack_from("<HH", b, pos)
        if (g, e) == (0xFFFE, 0xE00D):
            return pos + 8
        pos, _, _ = _read_element(b, pos, explicit, want_value=False)
    return pos


def _read_fragments(b, pos):
    """Encapsulated pixel data (PS3.5 A.4) from the first item on: Basic Offset Table item, fragment items, sequence
    delimiter -> (fragment spans, position after the delimiter)."""
    items = []
    while True:
        if pos + 8 > len(b):
            raise DicomError("encapsulated pixel data without a sequence delimiter")
        g, e, ln = struct.unpack_from("<HHI", b, pos)
        pos += 8
        if (g, e) == (0xFFFE, 0xE0DD):
            break
        if (g, e) != (0xFFFE, 0xE000) or ln == 0xFFFFFFFF or pos + ln > len(b):
            raise DicomError("malformed encapsulated pixel data")
        items.append((pos, ln))
        pos += ln
    if len(items) < 2:
        raise DicomError("encapsulated pixel data without a fragment")
    if items[0][1] > 4:
        raise DicomError("multi-frame objects are not supported")
    return items[1:], pos


def _read_element(b, pos, explicit, want_value=True, encapsulated=False):
    g, e = struct.unpack_from("<HH", b, pos)
    if explicit and g != 0xFFFE:
        vr = b[pos + 4:pos + 6]
        if vr in _LONG_VR:
            ln = struct.unpack_from("<I", b, pos + 8)[0]
            vpos = pos + 12
        else:
            ln = struct.unpack_from("<H", b, pos + 6)[0]
            vpos = pos + 8
    else:
        vr = None
        ln = struct.unpack_from("<I", b, pos + 4)[0]
        vpos = pos + 8
    if ln == 0xFFFFFFFF:                    # undefined length: a sequence (or encapsulated pixel data)
        if (g, e) == (0x7FE0, 0x0010):
            if not encapsulated:
                raise DicomError("encapsulated (compressed) pixel data is not supported")
            frags, end = _read_fragments(b, vpos)
            return end, (g, e), (frags if want_value else None)
        return _skip_sequence(b, vpos, explicit), (g, e), None
    return vpos + ln, (g, e), ((vpos, ln) if want_value else None)


def _read_dicom(path, stop_before_pixels=False):
    """read_dicom_file without the decode: a compressed frame is left in '_frame' = (codec, bytes)."""
    with open(path, "rb") as f:
        b = f.read()
    pos, syntax = 0, _IMPLICIT_LE
    if len(b) >= 132 and b[128:132] == b"DICM":
        pos = 132
        while pos + 8 <= len(b) and struct.unpack_from("<H", b, pos)[0] == 0x0002:   # file meta group: explicit VR LE
            pos, tag, val = _read_element(b, pos, True)
            if tag == (0x0002, 0x0010) and val:
                syntax = b[val[0]:val[0] + val[1]].decode("ascii", "ignore").strip("\x00 ")
    elif len(b) < 8:
        raise DicomError("not a DICOM file")
    codec = _CODECS.get(syntax)
    if syntax not in (_EXPLICIT_LE, _IMPLICIT_LE) and codec is None:
        raise DicomError("transfer syntax %s is not supported (uncompressed little endian, JPEG Lossless and RLE Lossless "
                         "only)" % syntax)
    explicit = syntax != _IMPLICIT_LE
    out = {}
    while pos + 8 <= len(b):
        g, e = struct.unpack_from("<HH", b, pos)
        if (g, e) == (0x7FE0, 0x0010) and stop_before_pixels:
            break
        pos, tag, val = _read_element(b, pos, explicit, encapsulated=codec is not None)
        if val is None:
            continue
        if tag in _WANTED:
            raw = b[val[0]:val[0] + val[1]]
            name = _WANTED[tag]
            if name in ("Rows", "Columns", "BitsAllocated", "PixelRepresentation", "SamplesPerPixel"):
                out[name] = struct.unpack_from("<H", raw)[0]
            else:
                out[name] = raw.decode("ascii", "ignore").strip("\x00 ")
        elif tag == (0x7FE0, 0x0010):
            out["_pixel_span"] = val
            break
    if not stop_before_pixels:
        if "_pixel_span" not in out or "Rows" not in out or "Columns" not in out:
            raise DicomError("no pixel data")
        if out.get("BitsAllocated", 16) != 16 or out.get("SamplesPerPixel", 1) != 1:
            raise DicomError("only 16-bit single-sample images are supported")
        if codec is not None:
            if int(out.get("NumberOfFrames", "1") or 1) != 1:
                raise DicomError("multi-frame objects are not supported")
            span = out.pop("_pixel_span")
            if not isinstance(span, list):              # a (vpos, length) tuple: native pixel data
                raise DicomError("%s: transfer syntax %s requires encapsulated pixel data" % (path, syntax))
            out["_frame"] = (codec, b"".join(b[p:p + n] for p, n in span))
            return out
        vpos, ln = out.pop("_pixel_span")
        n = out["Rows"] * out["Columns"]
        if ln < 2 * n:
            raise DicomError("pixel data shorter than Rows x Columns")
        dt = "<i2" if out.get("PixelRepresentation", 0) == 1 else "<u2"
        out["pixels"] = np.frombuffer(b, dtype=dt, count=n, offset=vpos).reshape(out["Rows"], out["Columns"])
    else:
        out.pop("_pixel_span", None)
    return out


def _decode_device(device):
    return int(os.environ.get("LOCAL_RANK", 0)) if device is None else int(device)


def _decode_pending(slices, names, device=None):
    """Decodes the compressed frames among `slices` (dicts of _read_dicom) in one lm_decode_frames call and stores each
    as 'pixels' (int16 when PixelRepresentation is 1, else uint16, as for uncompressed data)."""
    todo = [k for k, s in enumerate(slices) if "_frame" in s]
    if not todo:
        return
    from . import _native
    frames = np.zeros(len(todo), _native.FRAME_DTYPE)
    blobs, off = [], 0
    for i, k in enumerate(todo):
        s = slices[k]
        codec, blob = s["_frame"]
        frames[i] = (off, len(blob), codec, s["Rows"], s["Columns"], 1 if s.get("PixelRepresentation", 0) == 1 else 0)
        blobs.append(blob)
        off += len(blob)
    arrays, status = _native.decode_frames(b"".join(blobs), frames, _decode_device(device))
    for i, k in enumerate(todo):
        if status[i]:
            raise DicomError("%s: cannot decode the compressed pixel data: %s (%d)"
                             % (names[k], _native.DECODE_ERRORS.get(int(status[i]), "error"), int(status[i])))
        s = slices[k]
        del s["_frame"]
        s["pixels"] = arrays[i].view(np.int16) if s.get("PixelRepresentation", 0) == 1 else arrays[i]


def read_dicom_file(path, stop_before_pixels=False, device=None):
    """-> dict of the tags this module needs (+ 'pixels': int16/uint16 2-D array unless stop_before_pixels).  Compressed
    pixel data is decoded on CUDA device `device` (default: LOCAL_RANK, else 0)."""
    out = _read_dicom(path, stop_before_pixels)
    _decode_pending([out], [path], device)
    return out


def _floats(s, n):
    v = [float(x) for x in s.split("\\") if x.strip() != ""]
    if len(v) != n:
        raise DicomError("expected %d numbers, got %r" % (n, s))
    return v


def read_dicoms(path, primary=True, original=True, disable_tqdm=False, read_metadata=False, device=None):
    """utils.read_dicoms (utils.py:132-232): every series under `path` as a Volume.  The compressed frames of a series
    are decoded in one call on CUDA device `device` (default: LOCAL_RANK, else 0)."""
    files = [os.path.join(d, f) for d, _, fs in os.walk(path) for f in fs]
    infos, seen = [], set()
    for fname in files:
        if os.path.splitext(os.path.basename(fname))[0] == "DICOMDIR":
            continue
        try:
            h = _read_dicom(fname, stop_before_pixels=True)
        except Exception:
            logger.warning("Doesn't seem to be DICOM, will be skipped: %s", fname)
            continue
        if "ImageType" not in h or "SeriesInstanceUID" not in h or "ImagePositionPatient" not in h:
            continue
        itype = h["ImageType"].split("\\")
        if (primary and "PRIMARY" not in itype) or (original and "ORIGINAL" not in itype) or "LOCALIZER" in itype:
            continue
        key = (h.get("StudyInstanceUID", ""), h["SeriesInstanceUID"], h["ImagePositionPatient"])
        if key in seen:                     # duplicates of one slice under different names (utils.py:139-141,183-185)
            continue
        seen.add(key)
        infos.append((h["SeriesInstanceUID"], fname, _floats(h["ImagePositionPatient"], 3)))
    series = {}
    for uid, fname, ipp in infos:
        series.setdefault(uid, []).append((ipp, fname))
    n = len(series)
    logger.info("There %s %d volume%s in the study", "is" if n == 1 else "are", n, "" if n == 1 else "s")
    vols = []
    for uid in sorted(series):
        items = sorted(series[uid], key=lambda t: t[0][2])          # np.argsort of the z positions (utils.py:211-214)
        names = [f for _, f in items]
        slices = [_read_dicom(f) for f in names]
        _decode_pending(slices, names, device)
        first = slices[0]
        iop = _floats(first.get("ImageOrientationPatient", "1\\0\\0\\0\\1\\0"), 6)
        px = _floats(first.get("PixelSpacing", "1\\1"), 2)           # row spacing (y), column spacing (x)
        rx, ry = np.asarray(iop[:3]), np.asarray(iop[3:])
        normal = np.cross(rx, ry)
        pos = np.asarray([ipp for ipp, _ in items], dtype=np.float64)
        if len(items) > 1:
            step = pos[-1] - pos[0]
            dz = float(np.linalg.norm(step)) / (len(items) - 1)
            zdir = step / max(np.linalg.norm(step), 1e-12)
            if abs(float(np.dot(zdir, normal))) > 0.5:                # snap to the in-plane normal, keep the slice order's sign
                zdir = normal if np.dot(zdir, normal) > 0 else -normal
        else:
            dz, zdir = float(first.get("SliceThickness", "1") or 1), normal
        arr = np.stack([s["pixels"] for s in slices])
        slope, inter = float(first.get("RescaleSlope", "1") or 1), float(first.get("RescaleIntercept", "0") or 0)
        if slope != 1.0 or inter != 0.0:
            resc = arr.astype(np.float64) * slope + inter
            arr = resc.astype(np.int16) if float(slope).is_integer() and float(inter).is_integer() and \
                resc.min() >= -32768 and resc.max() <= 32767 else resc.astype(np.float32)
        elif arr.dtype == np.uint16 and arr.max() <= 32767:
            arr = arr.astype(np.int16)
        direction = np.stack([rx, ry, zdir], axis=1)                  # columns = image axes
        vols.append(Volume(np.ascontiguousarray(arr), (px[1], px[0], dz if dz > 0 else 1.0), tuple(float(x) for x in pos[0]),
                           tuple(float(x) for x in direction.ravel()), {"SeriesInstanceUID": uid, "files": [f for _, f in items]}))
    return vols


# --------------------------------------------------------------------------------------------------------------
# NIfTI-1, MetaImage, npy
# --------------------------------------------------------------------------------------------------------------
_NII_DTYPES = {2: np.uint8, 4: np.int16, 8: np.int32, 16: np.float32, 64: np.float64, 256: np.int8, 512: np.uint16, 768: np.uint32}
_LPS_FLIP = np.diag([-1.0, -1.0, 1.0])


def _read_nifti(path):
    raw = (gzip.open(path, "rb") if path.endswith(".gz") else open(path, "rb")).read()
    if len(raw) < 352 or struct.unpack_from("<i", raw, 0)[0] != 348:
        raise ValueError("%s: not a little-endian NIfTI-1 file" % path)
    dim = struct.unpack_from("<8h", raw, 40)
    datatype = struct.unpack_from("<h", raw, 70)[0]
    pixdim = struct.unpack_from("<8f", raw, 76)
    vox_offset = int(struct.unpack_from("<f", raw, 108)[0])
    slope, inter = struct.unpack_from("<2f", raw, 112)
    qform, sform = struct.unpack_from("<2h", raw, 252)
    if datatype not in _NII_DTYPES or dim[0] < 3:
        raise ValueError("%s: unsupported NIfTI datatype %d / dim %s" % (path, datatype, dim[:4]))
    nx, ny, nz = dim[1], dim[2], dim[3]
    arr = np.frombuffer(raw, dtype=np.dtype(_NII_DTYPES[datatype]).newbyteorder("<"), count=nx * ny * nz, offset=max(vox_offset, 352))
    arr = arr.reshape(nz, ny, nx)
    if slope not in (0.0, 1.0) or inter != 0.0:
        resc = arr.astype(np.float64) * (slope if slope != 0 else 1.0) + inter
        arr = resc.astype(np.int16) if np.all(resc == np.rint(resc)) and resc.min() >= -32768 and resc.max() <= 32767 else resc.astype(np.float32)
    if sform > 0:
        A = np.asarray([struct.unpack_from("<4f", raw, 280), struct.unpack_from("<4f", raw, 296), struct.unpack_from("<4f", raw, 312)], dtype=np.float64)
        M, t = A[:, :3], A[:, 3]
    elif qform > 0:
        b, c, d = struct.unpack_from("<3f", raw, 256)
        t = np.asarray(struct.unpack_from("<3f", raw, 268), dtype=np.float64)
        a = np.sqrt(max(0.0, 1.0 - (b * b + c * c + d * d)))
        R = np.asarray([[a * a + b * b - c * c - d * d, 2 * (b * c - a * d), 2 * (b * d + a * c)],
                        [2 * (b * c + a * d), a * a + c * c - b * b - d * d, 2 * (c * d - a * b)],
                        [2 * (b * d - a * c), 2 * (c * d + a * b), a * a + d * d - b * b - c * c]])
        qfac = -1.0 if pixdim[0] < 0 else 1.0
        M = R * np.asarray([pixdim[1], pixdim[2], pixdim[3] * qfac])
    else:
        M, t = np.diag([pixdim[1] or 1.0, pixdim[2] or 1.0, pixdim[3] or 1.0]), np.zeros(3)
    spacing = np.linalg.norm(M, axis=0)
    spacing[spacing == 0] = 1.0
    direction = _LPS_FLIP @ (M / spacing)                             # NIfTI is RAS, ITK / DICOM are LPS
    return Volume(np.ascontiguousarray(arr), tuple(float(s) for s in spacing), tuple(float(x) for x in _LPS_FLIP @ t),
                  tuple(float(x) for x in direction.ravel()), {"format": "nifti"})


def _write_nifti(path, arr, like):
    arr = np.ascontiguousarray(arr)
    code = {v: k for k, v in _NII_DTYPES.items()}[arr.dtype.type]
    nz, ny, nx = arr.shape
    D = np.asarray(like.direction, dtype=np.float64).reshape(3, 3)
    M = _LPS_FLIP @ (D * np.asarray(like.spacing, dtype=np.float64))
    t = _LPS_FLIP @ np.asarray(like.origin, dtype=np.float64)
    hdr = bytearray(352)
    struct.pack_into("<i", hdr, 0, 348)
    struct.pack_into("<8h", hdr, 40, 3, nx, ny, nz, 1, 1, 1, 1)
    struct.pack_into("<hh", hdr, 70, code, arr.dtype.itemsize * 8)
    struct.pack_into("<8f", hdr, 76, 1.0, *[float(s) for s in like.spacing], 0.0, 0.0, 0.0, 0.0)
    struct.pack_into("<f", hdr, 108, 352.0)
    struct.pack_into("<2f", hdr, 112, 1.0, 0.0)
    hdr[123] = 2                                                       # xyzt_units: mm
    struct.pack_into("<2h", hdr, 252, 0, 1)                            # sform only
    for r in range(3):
        struct.pack_into("<4f", hdr, 280 + 16 * r, *[float(x) for x in M[r]], float(t[r]))
    hdr[344:348] = b"n+1\x00"
    data = bytes(hdr) + arr.astype(arr.dtype.newbyteorder("<"), copy=False).tobytes()
    with (gzip.open(path, "wb", compresslevel=1) if path.endswith(".gz") else open(path, "wb")) as f:
        f.write(data)


_MHA_TYPES = {"MET_UCHAR": np.uint8, "MET_CHAR": np.int8, "MET_SHORT": np.int16, "MET_USHORT": np.uint16, "MET_INT": np.int32,
              "MET_UINT": np.uint32, "MET_FLOAT": np.float32, "MET_DOUBLE": np.float64}


def _read_mha(path):
    raw = open(path, "rb").read()
    hdr, pos = {}, 0
    while True:
        end = raw.index(b"\n", pos)
        line = raw[pos:end].decode("ascii", "ignore").strip()
        pos = end + 1
        if "=" in line:
            k, v = [x.strip() for x in line.split("=", 1)]
            hdr[k] = v
            if k == "ElementDataFile":
                break
    if hdr.get("CompressedData", "False").lower() == "true" or hdr.get("BinaryDataByteOrderMSB", "False").lower() == "true":
        raise ValueError("%s: compressed / big-endian MetaImage is not supported" % path)
    dims = [int(x) for x in hdr["DimSize"].split()]
    dt = np.dtype(_MHA_TYPES[hdr["ElementType"]]).newbyteorder("<")
    src = raw[pos:] if hdr["ElementDataFile"] == "LOCAL" else open(os.path.join(os.path.dirname(path), hdr["ElementDataFile"]), "rb").read()
    arr = np.frombuffer(src, dtype=dt, count=int(np.prod(dims))).reshape(dims[::-1])
    spacing = tuple(float(x) for x in hdr.get("ElementSpacing", "1 1 1").split())
    origin = tuple(float(x) for x in hdr.get("Offset", hdr.get("Position", "0 0 0")).split())
    tm = [float(x) for x in hdr.get("TransformMatrix", "1 0 0 0 1 0 0 0 1").split()]
    direction = tuple(float(x) for x in np.asarray(tm).reshape(3, 3).T.ravel())          # MetaImage stores the axes as rows
    return Volume(np.ascontiguousarray(arr), spacing, origin, direction, {"format": "mha"})


def _write_mha(path, arr, like):
    arr = np.ascontiguousarray(arr)
    et = {v: k for k, v in _MHA_TYPES.items()}[arr.dtype.type]
    D = np.asarray(like.direction, dtype=np.float64).reshape(3, 3)
    hdr = ("ObjectType = Image\nNDims = 3\nBinaryData = True\nBinaryDataByteOrderMSB = False\nCompressedData = False\n"
           "TransformMatrix = %s\nOffset = %s\nCenterOfRotation = 0 0 0\nElementSpacing = %s\nDimSize = %d %d %d\n"
           "ElementType = %s\nElementDataFile = LOCAL\n") % (
        " ".join("%.17g" % x for x in D.T.ravel()), " ".join("%.17g" % x for x in like.origin),
        " ".join("%.17g" % x for x in like.spacing), arr.shape[2], arr.shape[1], arr.shape[0], et)
    with open(path, "wb") as f:
        f.write(hdr.encode("ascii"))
        f.write(arr.tobytes())


def load_input_image(path, disable_tqdm=False, read_metadata=False, device=None):
    """utils.load_input_image (utils.py:235-269): a file is read as is, a directory as a DICOM series (the largest one).
    `device`: the CUDA device that decodes compressed DICOM (default: LOCAL_RANK, else 0)."""
    if os.path.isfile(path):
        logger.info("Read input: %s", path)
        low = path.lower()
        if low.endswith(".npy"):
            return Volume(np.load(path))
        if low.endswith((".nii", ".nii.gz")):
            return _read_nifti(path)
        if low.endswith((".mha", ".mhd")):
            return _read_mha(path)
        h = read_dicom_file(path, device=device)                        # a single DICOM slice
        px = _floats(h.get("PixelSpacing", "1\\1"), 2)
        iop = _floats(h.get("ImageOrientationPatient", "1\\0\\0\\0\\1\\0"), 6)
        rx, ry = np.asarray(iop[:3]), np.asarray(iop[3:])
        arr = h["pixels"][None]
        slope, inter = float(h.get("RescaleSlope", "1") or 1), float(h.get("RescaleIntercept", "0") or 0)
        if slope != 1.0 or inter != 0.0:
            arr = (arr.astype(np.float64) * slope + inter).astype(np.float32)
        return Volume(np.ascontiguousarray(arr), (px[1], px[0], float(h.get("SliceThickness", "1") or 1)),
                      tuple(_floats(h.get("ImagePositionPatient", "0\\0\\0"), 3)),
                      tuple(float(x) for x in np.stack([rx, ry, np.cross(rx, ry)], axis=1).ravel()))
    logger.info("Looking for dicoms in %s", path)
    vols = read_dicoms(path, original=False, primary=False, disable_tqdm=disable_tqdm, read_metadata=read_metadata,
                       device=device)
    if len(vols) < 1:
        raise SystemExit("No dicoms found!")
    if len(vols) > 1:
        logger.warning("There are more than one volume in the path, will take the largest one")
    return vols[int(np.argmax([np.prod(v.GetSize()) for v in vols]))]


def save_mask(path, mask, like=None):
    """Writes the uint8 mask with the geometry of `like` (what sitk.WriteImage(result_out, output) does after
    CopyInformation, __main__.py:129-144); the format follows the extension."""
    like = like if like is not None else Volume(mask)
    low = path.lower()
    if low.endswith(".npy"):
        np.save(path, mask)
    elif low.endswith((".nii", ".nii.gz")):
        _write_nifti(path, mask, like)
    elif low.endswith(".mha"):
        _write_mha(path, mask, like)
    else:
        raise SystemExit("unsupported output format (use .nii, .nii.gz, .mha or .npy): %s" % path)
