"""Compressed DICOM series (JPEG Lossless .4.57 / .4.70, RLE Lossless .5): the oracle encoders, the encapsulation parser
and the transfer-syntax handling on the CPU; lm_decode_frames (csrc/decode.cu) bit-exact, batched, on malformed input
and end to end on the GPU."""
import io
import os
import struct

import numpy as np
import pytest

from lungmask_b200 import io as lio
from oracle import dicom_codecs as dc

gpu = pytest.mark.gpu
SYNTAXES = [dc.JPEG_LOSSLESS, dc.JPEG_LOSSLESS_SV1, dc.RLE_LOSSLESS]


def _encode(img, syntax, **kw):
    return dc.rle_encode(img) if syntax == dc.RLE_LOSSLESS else dc.jpeg_lossless_encode(img, **kw)


# --------------------------------------------------------------------------------------------------------------
# CPU
# --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("predictor", range(1, 8))
@pytest.mark.parametrize("pt", [0, 2])
@pytest.mark.parametrize("restart_rows", [0, 3])
def test_jpeg_encoder_matches_libjpeg_turbo(predictor, pt, restart_rows):
    Image = pytest.importorskip("PIL.Image")
    rng = np.random.default_rng(predictor * 10 + pt + restart_rows)
    img = rng.integers(0, 256, (19, 23)).astype(np.uint16)
    img[4:9, 3:] = 255                                           # flat and saturated areas: 0xFF bytes, long zero runs
    img = (img >> pt) << pt
    b = dc.jpeg_lossless_encode(img, P=8, predictor=predictor, pt=pt, restart_rows=restart_rows)
    assert (b"\xff\xdd" in b) == (restart_rows > 0)
    assert np.array_equal(np.asarray(Image.open(io.BytesIO(b))), img)


@pytest.mark.parametrize("bot", ["empty", "filled"])
@pytest.mark.parametrize("fragments", [1, 3])
def test_encapsulated_frame_is_reassembled(tmp_path, bot, fragments):
    rng = np.random.default_rng(1)
    frame = b""
    while len(frame) % 2 == 0:                                   # an odd-length stream: one pad byte after EOI
        img = rng.integers(-1000, 1000, (9, 7)).astype(np.int16)
        frame = dc.jpeg_lossless_encode(img)
    p = str(tmp_path / "f.dcm")
    dc.write_encapsulated(p, frame, dc.JPEG_LOSSLESS_SV1, *img.shape, "1.2.9", (0, 0, 0), fragments=fragments, bot=bot)
    h = lio._read_dicom(p)
    assert h["_frame"] == (1, frame + b"\x00")
    assert h["Rows"] == img.shape[0] and h["Columns"] == img.shape[1] and h["SeriesInstanceUID"] == "1.2.9"


def test_multiframe_and_undefined_length_uncompressed_stay_rejected(tmp_path):
    p = str(tmp_path / "m.dcm")
    item = lambda v: struct.pack("<HHI", 0xFFFE, 0xE000, len(v)) + v
    pix = (struct.pack("<HH2sHI", 0x7FE0, 0x0010, b"OB", 0, 0xFFFFFFFF) + item(struct.pack("<2I", 0, 8)) + item(b"\xff\xd8" * 4)
           + item(b"\xff\xd8" * 4) + struct.pack("<HHI", 0xFFFE, 0xE0DD, 0))
    dc.write_encapsulated(p, None, dc.RLE_LOSSLESS, 2, 2, "1.2.9", (0, 0, 0), pixel_data=pix)
    with pytest.raises(lio.DicomError, match="multi-frame"):
        lio.read_dicom_file(p)
    dc.write_encapsulated(p, dc.rle_encode(np.zeros((2, 2), np.int16)), "1.2.840.10008.1.2.1", 2, 2, "1.2.9", (0, 0, 0))
    with pytest.raises(lio.DicomError, match="encapsulated"):
        lio.read_dicom_file(p)


@pytest.mark.parametrize("syntax", SYNTAXES)
def test_native_pixel_data_under_a_compressed_syntax_is_rejected(tmp_path, syntax):
    img = np.zeros((2, 2), np.int16)
    native = struct.pack("<HH2sHI", 0x7FE0, 0x0010, b"OW", 0, img.nbytes) + img.tobytes()
    d = tmp_path / "series"
    d.mkdir()
    p = str(d / "n.dcm")
    dc.write_encapsulated(p, None, syntax, 2, 2, "1.2.9", (0, 0, 0), pixel_data=native)
    with pytest.raises(lio.DicomError, match=r"n\.dcm.*requires encapsulated"):
        lio.read_dicom_file(p)
    with pytest.raises(lio.DicomError, match=r"n\.dcm"):
        lio.load_input_image(str(d))


@pytest.mark.parametrize("syntax", ["1.2.840.10008.1.2.4.50", "1.2.840.10008.1.2.4.51", "1.2.840.10008.1.2.4.80",
                                    "1.2.840.10008.1.2.4.90", "1.2.840.10008.1.2.1.99", "1.2.840.10008.1.2.2"])
def test_unsupported_syntaxes_are_rejected(tmp_path, syntax):
    p = str(tmp_path / "u.dcm")
    dc.write_encapsulated(p, b"\xff\xd8\xff\xd9", syntax, 2, 2, "1.2.9", (0, 0, 0))
    with pytest.raises(lio.DicomError, match=syntax.replace(".", r"\.")):
        lio.read_dicom_file(p)


@pytest.mark.parametrize("syntax", SYNTAXES)
def test_series_header_stage_and_one_decode_call(tmp_path, monkeypatch, syntax):
    """Grouping, sorting and geometry run on the headers; the frames of the series reach the decoder in one call."""
    vol = np.random.default_rng(2).integers(-1000, 1000, (4, 6, 5)).astype(np.int16)
    for k in range(vol.shape[0]):                                # reversed file order
        dc.write_encapsulated(str(tmp_path / ("im%d.dcm" % (9 - k))), _encode(vol[k], syntax), syntax, 6, 5, "1.2.7",
                              (-8.0, -9.0, 2.5 * k))
    calls = []

    def fake_decode(slices, names, device=None):
        calls.append([os.path.basename(n) for n in names])
        for k, s in enumerate(slices):
            s["pixels"] = np.full((s["Rows"], s["Columns"]), k, np.int16)
            del s["_frame"]
    monkeypatch.setattr(lio, "_decode_pending", fake_decode)
    vols = lio.read_dicoms(str(tmp_path), primary=False, original=False)
    assert len(vols) == 1 and calls == [["im9.dcm", "im8.dcm", "im7.dcm", "im6.dcm"]]
    v = vols[0]
    assert np.array_equal(v.array[:, 0, 0], np.arange(4)) and v.array.dtype == np.int16
    assert np.allclose(v.spacing, (0.75, 0.5, 2.5)) and np.allclose(v.origin, (-8.0, -9.0, 0.0))


# --------------------------------------------------------------------------------------------------------------
# GPU
# --------------------------------------------------------------------------------------------------------------
def _decode(streams, shapes, codecs, signed):
    from lungmask_b200 import _native
    frames = np.zeros(len(streams), _native.FRAME_DTYPE)
    off = 0
    for i, (s, (h, w), c, sg) in enumerate(zip(streams, shapes, codecs, signed)):
        frames[i] = (off, len(s), c, h, w, int(sg))
        off += len(s)
    return _native.decode_frames(b"".join(streams), frames, 0)


def _roundtrip_jpeg(img, signed, **kw):
    arrays, status = _decode([dc.jpeg_lossless_encode(img, **kw)], [img.shape], [1], [signed])
    assert status.tolist() == [0]
    got = arrays[0].view(np.int16) if signed else arrays[0]
    assert np.array_equal(got, img), kw


@gpu
def test_jpeg_known_answer_category_16():
    kat = bytes.fromhex("ff d8 ff c3 00 0b 10 00 01 00 02 01 01 11 00 ff c4 00 14 00 01 00 00 00 00 00 00 00 00 00 00 00 00 "
                        "00 00 00 10 ff da 00 08 01 01 00 01 00 00 3f ff d9")
    arrays, status = _decode([kat], [(1, 2)], [1], [False])
    assert status.tolist() == [0] and arrays[0].tolist() == [[0, 32768]]


def _ct_like(rng, shape):
    from oracle import synth
    return synth.phantom(1, *shape, seed=int(rng.integers(1 << 30)))[0]


@gpu
@pytest.mark.parametrize("predictor", range(1, 8))
@pytest.mark.parametrize("pt", [0, 3])
def test_jpeg_roundtrip_predictors(predictor, pt):
    rng = np.random.default_rng(predictor + 10 * pt)
    u = rng.integers(0, 65536, (67, 45)).astype(np.uint16)          # P = 16 unsigned noise: every category
    _roundtrip_jpeg((u >> pt) << pt, False, P=16, predictor=predictor, pt=pt)
    ct = _ct_like(rng, (96, 80))                                    # CT-like int16, P = 16 signed
    _roundtrip_jpeg((ct >> pt) << pt, True, P=16, predictor=predictor, pt=pt, restart_rows=7)
    s12 = np.clip(ct, -2048, 2047).astype(np.int16)                 # P = 12 signed: sign extension from bit 11
    _roundtrip_jpeg((s12 >> pt) << pt, True, P=12, predictor=predictor, pt=pt)
    _roundtrip_jpeg((s12 >> pt) << pt, True, P=12, predictor=predictor, pt=pt, restart_rows=1)


@gpu
@pytest.mark.parametrize("shape", [(1, 1), (1, 700), (700, 1), (511, 509)])
def test_jpeg_roundtrip_odd_sizes_and_long_streams(shape):
    rng = np.random.default_rng(shape[0] + shape[1])
    img = rng.integers(-32768, 32768, shape).astype(np.int16)
    for predictor in (1, 4, 7):
        _roundtrip_jpeg(img, True, P=16, predictor=predictor)
    if shape == (511, 509):                                         # ~2.3 Mbit: thousands of synchronisation chunks
        _roundtrip_jpeg(img, True, P=16, predictor=1, restart_rows=73)


@gpu
def test_jpeg_roundtrip_ff_bytes_and_32768_differences():
    row = (np.arange(4000, dtype=np.int64) * 32767) & 0xFFFF         # difference +32767: category 15, extra bits all ones
    img = row.reshape(40, 100).astype(np.uint16)
    b = dc.jpeg_lossless_encode(img, P=16, predictor=1)
    assert b.count(b"\xff\x00") > 2000
    _roundtrip_jpeg(img, False, P=16, predictor=1)
    alt = np.zeros((33, 65), np.uint16)                             # differences of +-32768 everywhere: category 16
    alt[::2, ::2] = alt[1::2, 1::2] = 32768
    for predictor in (1, 2, 3):
        _roundtrip_jpeg(alt, False, P=16, predictor=predictor)


@gpu
def test_jpeg_and_rle_roundtrip_ct_slice(ct_slice):
    img = np.asarray(ct_slice).astype(np.int16)
    for predictor in (1, 6):
        _roundtrip_jpeg(img, True, P=16, predictor=predictor)
    arrays, status = _decode([dc.rle_encode(img)], [img.shape], [2], [True])
    assert status.tolist() == [0] and np.array_equal(arrays[0].view(np.int16), img)


@gpu
def test_rle_roundtrip():
    rng = np.random.default_rng(5)
    cases = {
        "literal": rng.integers(0, 65536, (31, 37)).astype(np.uint16),
        "replicate": np.full((64, 64), 0x1234, np.uint16),          # runs far beyond 128 bytes
        "mixed": np.repeat(rng.integers(0, 4, (40, 50)), rng.integers(1, 300, 40 * 50)).astype(np.uint16)[:77 * 53].reshape(77, 53),
        "odd": rng.integers(0, 3, (3, 5)).astype(np.uint16),
    }
    for name, img in cases.items():
        enc = dc.rle_encode(img)
        segs = struct.unpack_from("<3I", enc)
        if name == "odd":
            assert (segs[2] - segs[1]) % 2 == 0                     # segments are padded to even lengths
        arrays, status = _decode([enc], [img.shape], [2], [False])
        assert status.tolist() == [0] and np.array_equal(arrays[0], img), name


@gpu
def test_batched_decode_equals_per_frame():
    rng = np.random.default_rng(9)
    imgs = [_ct_like(rng, (96, 80)), rng.integers(-500, 500, (33, 47)).astype(np.int16), _ct_like(rng, (64, 128)),
            np.zeros((5, 5), np.int16), rng.integers(-3000, 3000, (200, 1)).astype(np.int16)]
    streams = [dc.jpeg_lossless_encode(imgs[0], predictor=1), dc.rle_encode(imgs[1]),
               dc.jpeg_lossless_encode(imgs[2], predictor=5, restart_rows=4), dc.rle_encode(imgs[3]),
               dc.jpeg_lossless_encode(imgs[4], predictor=2)]
    codecs = [1, 2, 1, 2, 1]
    arrays, status = _decode(streams, [i.shape for i in imgs], codecs, [True] * 5)
    assert status.tolist() == [0] * 5
    for k, img in enumerate(imgs):
        one, st = _decode([streams[k]], [img.shape], [codecs[k]], [True])
        assert st.tolist() == [0] and np.array_equal(one[0], arrays[k]) and np.array_equal(arrays[k].view(np.int16), img)


def _rst_markers(first, n):
    """n RSTm markers in sequence, the first one RST(first mod 8)."""
    codes = 0xD0 + (np.arange(first, first + n) & 7)
    return np.stack([np.full(n, 0xFF), codes], axis=1).astype(np.uint8).tobytes()


@gpu
def test_more_restart_markers_than_intervals_is_a_length_error():
    rng = np.random.default_rng(11)
    img = _ct_like(rng, (24, 20))
    jpg = dc.jpeg_lossless_encode(img, restart_rows=1)               # 24 intervals: RST0..RST22 in the stream
    extra = jpg[:-2] + _rst_markers(23, 3 * 24) + b"\xff\xd9"          # 72 more, in sequence, before EOI
    arrays, status = _decode([jpg, extra], [img.shape] * 2, [1, 1], [True, True])
    assert status.tolist() == [0, -62] and np.array_equal(arrays[0].view(np.int16), img)
    # 2^24 + 5 markers in one frame between two valid ones: the marker count has the full 32 bits of the scan word
    small = dc.jpeg_lossless_encode(img[:1])
    many = small[:-2] + _rst_markers(0, (1 << 24) + 5) + b"\xff\xd9"
    arrays, status = _decode([jpg, many, jpg], [img.shape, (1, 20), img.shape], [1, 1, 1], [True] * 3)
    assert status.tolist() == [0, -62, 0]
    assert np.array_equal(arrays[0].view(np.int16), img) and np.array_equal(arrays[2].view(np.int16), img)


@gpu
def test_codewords_beyond_the_last_sample_are_ignored():
    """As libjpeg-turbo does: data left before EOI after rows x cols samples does not fail the frame; too few samples do."""
    img = _ct_like(np.random.default_rng(12), (30, 26))
    for kw in ({}, {"restart_rows": 5}):
        jpg = dc.jpeg_lossless_encode(img, **kw)
        surplus = jpg[:-2] + bytes(16) + b"\xff\xd9"
        arrays, status = _decode([surplus], [img.shape], [1], [True])
        assert status.tolist() == [0] and np.array_equal(arrays[0].view(np.int16), img), kw


def _replace_sof(stream, nf):
    i = stream.index(b"\xff\xc3")
    P, H, W = struct.unpack_from(">BHH", stream, i + 4)
    body = struct.pack(">BHHB", P, H, W, nf) + b"".join(bytes([c + 1, 0x11, 0]) for c in range(nf))
    return stream[:i] + b"\xff\xc3" + struct.pack(">H", len(body) + 2) + body + stream[i + 13:]


@gpu
def test_malformed_frames_raise_dicom_error_naming_the_file(tmp_path):
    img = _ct_like(np.random.default_rng(3), (24, 20))
    jpg = dc.jpeg_lossless_encode(img)
    rle = dc.rle_encode(img)
    sos = jpg.index(b"\xff\xda") + 10
    undefined = dc.jpeg_lossless_encode(np.zeros((1, 16), np.uint16), table=([1] + [0] * 15, [0]))
    undefined = undefined[:undefined.index(b"\xff\xda") + 10] + b"\x80\x00\x00\x00\xff\xd9"   # only code: 0
    n1 = struct.unpack_from("<I", rle, 8)[0]
    cases = {
        "truncated": (jpg[:sos + (len(jpg) - sos) // 2] + b"\xff\xd9", dc.JPEG_LOSSLESS_SV1, img.shape),
        "no_eoi": (jpg[:-2], dc.JPEG_LOSSLESS_SV1, img.shape),
        "undefined_code": (undefined, dc.JPEG_LOSSLESS, (1, 16)),
        "sof0": (jpg.replace(b"\xff\xc3", b"\xff\xc0", 1), dc.JPEG_LOSSLESS_SV1, img.shape),
        "nf3": (_replace_sof(jpg, 3), dc.JPEG_LOSSLESS_SV1, img.shape),
        "size": (jpg, dc.JPEG_LOSSLESS_SV1, (img.shape[0], img.shape[1] + 1)),
        "rle_3_segments": (struct.pack("<I", 3) + rle[4:], dc.RLE_LOSSLESS, img.shape),
        "rle_short_segment": (rle[:n1 + (len(rle) - n1) // 3], dc.RLE_LOSSLESS, img.shape),
    }
    for name, (frame, syntax, shape) in cases.items():
        p = str(tmp_path / (name + ".dcm"))
        dc.write_encapsulated(p, frame, syntax, shape[0], shape[1], "1.2.3", (0, 0, 0))
        with pytest.raises(lio.DicomError, match=name + r"\.dcm"):
            lio.read_dicom_file(p)
    # a series with one bad slice names that slice
    sdir = tmp_path / "series"
    sdir.mkdir()
    for k in range(3):
        frame = jpg if k != 1 else jpg[:-2]
        dc.write_encapsulated(str(sdir / ("s%d.dcm" % k)), frame, dc.JPEG_LOSSLESS_SV1, *img.shape, "1.2.3", (0, 0, k))
    with pytest.raises(lio.DicomError, match=r"s1\.dcm"):
        lio.load_input_image(str(sdir))


@gpu
def test_compressed_series_end_to_end(tmp_path):
    import torch
    from _dicom_writer import _write_dicom
    from lungmask_b200.__main__ import main
    from oracle import synth
    vol = synth.phantom(40, 160, 176, seed=31)
    dirs = {}
    for name in ("raw", "jpeg", "rle"):
        d = tmp_path / name
        d.mkdir()
        dirs[name] = str(d)
        for k in range(vol.shape[0]):                                # reversed file order: the reader sorts by position
            p, ipp = str(d / ("im%02d.dcm" % (99 - k))), (-80.0, -90.0, 1.5 * k)
            if name == "raw":
                _write_dicom(p, vol[k], "1.2.840.5", ipp)
            else:
                syntax = dc.JPEG_LOSSLESS_SV1 if name == "jpeg" else dc.RLE_LOSSLESS
                dc.write_encapsulated(p, _encode(vol[k], syntax), syntax, *vol.shape[1:], "1.2.840.5", ipp,
                                      fragments=1 + k % 3)
    loaded = {n: lio.load_input_image(d) for n, d in dirs.items()}
    for n in ("jpeg", "rle"):
        a, b = loaded["raw"], loaded[n]
        assert a.array.dtype == b.array.dtype and np.array_equal(a.array, b.array), n
        assert (a.spacing, a.origin, a.direction) == (b.spacing, b.origin, b.direction)
    assert np.array_equal(loaded["raw"].array, vol)
    w = str(tmp_path / "w.pth")
    torch.save(synth.random_state_dict(3, seed=13, head_gain=0.3), w)
    masks = {}
    for n, d in dirs.items():
        out = str(tmp_path / (n + ".nii.gz"))
        main([d, out, "--modelpath", w, "--noprogress", "--batchsize", "8"])
        masks[n] = lio.load_input_image(out).array
    assert masks["raw"].max() > 0
    assert np.array_equal(masks["raw"], masks["jpeg"]) and np.array_equal(masks["raw"], masks["rle"])
