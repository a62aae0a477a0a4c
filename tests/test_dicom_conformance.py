"""lm_decode_frames (csrc/decode.cu) and the oracle encoder checked against implementations outside this project:
libjpeg-turbo (Pillow's, through oracle/libjpeg_turbo.py) and the sequential T.81 / PackBits reference decoders of
oracle/ljpeg_ref.py.  The GPU tests read tests/golden/codec_conformance.npz (oracle/make_codec_golden.py) and the
oracle only, so they need no Pillow."""
import re
import time

import numpy as np
import pytest

from oracle import dicom_codecs as dc
from oracle import libjpeg_turbo as lj
from oracle import ljpeg_ref as ref
from oracle import make_codec_golden as mcg

gpu = pytest.mark.gpu
needs_libjpeg_turbo = pytest.mark.skipif(not lj.available(), reason="Pillow's libjpeg-turbo is not installed")


def _reference_decode(c):
    if c["codec"] == 1:
        return ref.jpeg_lossless_decode(c["stream"])
    return ref.rle_decode(c["stream"], c["rows"], c["cols"])


@pytest.fixture(scope="module")
def golden():
    """The fixture's frames; the expected samples of each valid one are the sequential reference's decode, checked
    against the digest stored with the frame (libjpeg-turbo's decode, or the reference decode libjpeg-turbo agreed with
    when the fixture was written)."""
    z = np.load(mcg.OUT)
    data = z["data"].tobytes()
    cases = []
    for k, f in enumerate(z["frames"]):
        c = dict(name=str(z["name"][k]), origin=str(z["origin"][k]), codec=int(f["codec"]), rows=int(f["rows"]),
                 cols=int(f["cols"]), P=int(f["P"]), status=int(f["status"]), ljt=int(f["ljt"]),
                 stream=data[f["offset"]:f["offset"] + f["length"]], sha256=str(z["sha256"][k]), expected=None)
        if not c["status"]:
            c["expected"] = _reference_decode(c)
            assert mcg.digest(c["expected"]) == c["sha256"], c["name"]
        cases.append(c)
    return cases


def _by_name(cases, name):
    return next(c for c in cases if c["name"] == name)


# --------------------------------------------------------------------------------------------------------------
# CPU: the reference decoders, the libjpeg-turbo binding, the fixture
# --------------------------------------------------------------------------------------------------------------
def test_fixture_covers_the_documented_cases(golden):
    names = {c["name"] for c in golden}
    for p in ("J1_", "J2_", "J3_", "J4_", "J5_", "J6_", "J7_", "J8_", "J9_", "J10_", "J11_", "J12_", "R1_", "R2_", "R3_",
              "R4_", "R5_"):
        assert any(n.startswith(p) for n in names), p
    for P in (2, 8, 12, 15, 16):
        assert sum(re.fullmatch(r"ljt_P%d_p[1-7]_pt[0-3]_r[03]" % P, n) is not None for n in names) == 28
    assert sorted({c["status"] for c in golden if c["origin"] == "malformed"}) == [-62, -61, -60]
    assert all(c["ljt"] == 1 for c in golden if c["origin"] in ("libjpeg-turbo", "hand"))


def test_reference_decodes_every_fixture_frame(golden):
    """libjpeg-turbo's decodes of its own streams (by digest), and the documented status of every malformed frame."""
    for c in golden:
        if c["status"]:
            with pytest.raises(ref.DecodeError) as e:
                _reference_decode(c)
            assert e.value.status == c["status"], c["name"]
        else:
            assert mcg.digest(_reference_decode(c)) == c["sha256"] != "", c["name"]


def test_sync_worst_case_is_one_3_bit_code():
    """J11 needs codewords that resynchronise never: one code, 3 bits long, 1024 % 3 != 0, ~300 chunks."""
    s = next(s for n, s, *_ in mcg.hand_jpeg_cases() if n == mcg.SYNC_WORST_CASE)
    h = ref.parse_jpeg(s)
    assert h["table"].maxcode[3] == 0 and max(h["table"].maxcode) == 0 and h["pt"] == 0
    assert len(ref.split_entropy(h["entropy"])[0]) * 8 // 1024 >= 300 and 1024 % 3


@needs_libjpeg_turbo
def test_libjpeg_turbo_binding_writes_the_fields_it_sets():
    """The struct offsets of oracle/libjpeg_turbo.py: what it wrote shows in SOF3 / DRI / SOS, what it read in the header."""
    rng = np.random.default_rng(3)
    jobs = [(rng.integers(0, 1 << P, (h, w)).astype(np.uint16), P, pred, 0, rr)
            for P, pred, rr, (h, w) in [(2, 3, 0, (5, 9)), (9, 5, 2, (13, 7)), (13, 7, 1, (3, 300)), (16, 2, 5, (37, 11))]]
    streams = lj.encode_many(jobs)
    for (img, P, pred, pt, rr), s, (dec, Pd) in zip(jobs, streams, lj.decode_many_with_header(streams)):
        h = ref.parse_jpeg(s)
        assert (h["P"], h["rows"], h["cols"], h["pred"], h["ri"]) == (P, *img.shape, pred, rr * img.shape[1])
        assert Pd == P and np.array_equal(dec, img) and np.array_equal(ref.jpeg_lossless_decode(s), img)


@needs_libjpeg_turbo
@pytest.mark.parametrize("predictor, restart_in_rows", [(1, 0), (6, 64)])
def test_reference_equals_libjpeg_turbo_on_the_ct_slice(ct_slice, predictor, restart_in_rows):
    """The whole 512^2 CT slice (the fixture holds a 96^2 crop of it): written by libjpeg-turbo, read by both."""
    img = np.asarray(ct_slice).astype(np.int16).view(np.uint16)
    s = lj.encode(img, 16, predictor, 0, restart_in_rows)
    assert np.array_equal(lj.decode(s), img) and np.array_equal(ref.jpeg_lossless_decode(s), img)


@needs_libjpeg_turbo
def test_libjpeg_turbo_failure_is_an_exception():
    with pytest.raises(lj.LibjpegError):
        lj.decode(b"\xff\xd8\xff\xc3\x00\x0b\x10")


@needs_libjpeg_turbo
@pytest.mark.parametrize("predictor", range(1, 8))
def test_reference_equals_libjpeg_turbo_on_oracle_encoder_streams(predictor):
    rng = np.random.default_rng(predictor)
    streams, imgs = [], []
    for P in range(2, 17):
        for pt, rr in ((0, 0), (min(3, P - 1), 4)):
            img = ((rng.integers(0, 1 << P, (21, 17)) >> pt) << pt).astype(np.uint16)
            img[3:6] = ((1 << P) - 1) >> pt << pt
            streams.append(dc.jpeg_lossless_encode(img, P=P, predictor=predictor, pt=pt, restart_rows=rr))
            imgs.append(img)
    for s, img, (dec, P) in zip(streams, imgs, lj.decode_many_with_header(streams)):
        assert np.array_equal(dec, img) and np.array_equal(ref.jpeg_lossless_decode(s), img), P


@pytest.mark.parametrize("min_rep", [1, 2, 3])
def test_packbits_reference_inverts_rle_encode(min_rep):
    rng = np.random.default_rng(min_rep)
    for shape in ((1, 1), (1, 300), (37, 41)):
        img = np.repeat(rng.integers(0, 4, shape[0] * shape[1]), rng.integers(1, 400, shape[0] * shape[1]))
        img = (img[:shape[0] * shape[1]].reshape(shape) * 0x0101 + (rng.random(shape) < 0.1)).astype(np.uint16)
        assert np.array_equal(ref.rle_decode(dc.rle_encode(img, min_rep), *shape), img)


@needs_libjpeg_turbo
def test_codec_golden_is_up_to_date():
    mcg.main(["--check"])


# --------------------------------------------------------------------------------------------------------------
# GPU
# --------------------------------------------------------------------------------------------------------------
def _decode(cases, signed):
    """One lm_decode_frames call; signed: one flag for all frames, or one per frame."""
    from lungmask_b200 import _native
    signed = [signed] * len(cases) if isinstance(signed, bool) else signed
    frames = np.zeros(len(cases), _native.FRAME_DTYPE)
    off = 0
    for i, c in enumerate(cases):
        frames[i] = (off, len(c["stream"]), c["codec"], c["rows"], c["cols"], int(signed[i]))
        off += len(c["stream"])
    return _native.decode_frames(b"".join(c["stream"] for c in cases), frames, 0)


def _want(c, signed):
    return mcg.sign_extend(c["expected"], c["P"]) if signed and c["codec"] == 1 else c["expected"]


def _check(c, got, status, signed):
    assert status == c["status"], (c["name"], status)
    if not c["status"]:
        assert np.array_equal(got, _want(c, signed)), (c["name"], signed)


@gpu
@pytest.mark.parametrize("signed", [False, True])
def test_every_fixture_frame_alone(golden, signed):
    for c in golden:
        arrays, status = _decode([c], signed)
        _check(c, arrays[0], int(status[0]), signed)


@gpu
def test_all_fixture_frames_in_one_shuffled_call(golden):
    """Frames of every origin in one call, malformed ones between them: each frame's result as when decoded alone."""
    order = np.random.default_rng(17).permutation(len(golden))
    cases = [golden[k] for k in order]
    assert any(cases[k]["status"] and not cases[k + 1]["status"] for k in range(len(cases) - 1))
    signed = [bool(k % 2) for k in range(len(cases))]
    arrays, status = _decode(cases, signed)
    for c, a, st, sg in zip(cases, arrays, status, signed):
        _check(c, a, int(st), sg)


@gpu
def test_sync_worst_case_decodes_exactly(golden):
    c = _by_name(golden, mcg.SYNC_WORST_CASE)
    _decode([_by_name(golden, "ljt_1x1")], False)            # CUDA context and module load out of the timed call
    t = time.perf_counter()
    arrays, status = _decode([c], False)
    dt = time.perf_counter() - t
    assert status.tolist() == [0] and np.array_equal(arrays[0], c["expected"])
    assert np.all(arrays[0] == 1 << 15)
    print("%s: %d x %d decoded in %.1f ms (host clock, one call)" % (c["name"], c["rows"], c["cols"], dt * 1e3))


def _random_table(rng):
    """A random valid DC table over a random subset of the categories, in random HUFFVAL order, with a 16-bit code."""
    n = int(rng.integers(3, 17))
    cats = rng.permutation(17)[:n]
    bits = [0] * 16
    lengths = sorted(rng.integers(1, 16, n - 1).tolist()) + [16]
    for l in lengths:
        bits[l - 1] += 1
    while True:                                             # Kraft sum < 1 keeps the all-ones code free (T.81 C)
        kraft = sum(b / (1 << (l + 1)) for l, b in enumerate(bits))
        if kraft < 1:
            return bits, [int(c) for c in cats]
        l = max(l for l in range(15) if bits[l])
        bits[l] -= 1
        bits[l + 1] += 1


@gpu
@pytest.mark.parametrize("seed", range(4))
def test_generated_streams_equal_the_reference(seed):
    """Seeded random tables (with 16-bit codes) and marker layouts; the expected samples from oracle/ljpeg_ref.py."""
    rng = np.random.default_rng(1000 + seed)
    bits, vals = _random_table(rng)
    h, w = int(rng.integers(1, 90)), int(rng.integers(1, 90))
    cats = rng.choice([c for c in vals if c != 16], (h, w))
    img = mcg.image_from_differences(mcg.differences_of_categories(rng, cats), 16)
    parts = mcg.split_stream(dc.jpeg_lossless_encode(img, P=16, predictor=1, table=(bits, vals)))
    th = int(rng.integers(0, 4))
    parts[0xDA] = parts[0xDA][:2] + bytes([th << 4]) + parts[0xDA][3:]
    extras = [mcg.seg(0xE0 + int(rng.integers(0, 16)), rng.bytes(int(rng.integers(0, 20)))), b"\xff\x01",
              mcg.seg(0xFE, b"generated"), mcg.dht((th, [1] + [0] * 15, [0]))]   # a decoy table, redefined below
    layout = [extras[k] for k in rng.permutation(len(extras))]
    layout.insert(int(rng.integers(0, len(layout) + 1)), 0xC3)
    layout.append(mcg.dht((th, bits, vals)))
    layout.insert(int(rng.integers(0, len(layout) + 1)), b"\xff" * int(rng.integers(1, 4)))   # fill bytes
    stream = mcg.assemble(parts, *layout, 0xDA)
    expected = ref.jpeg_lossless_decode(stream)
    assert np.array_equal(expected, img)
    c = dict(name="generated%d" % seed, codec=1, rows=h, cols=w, P=16, status=0, stream=stream, expected=expected)
    arrays, status = _decode([c], False)
    _check(c, arrays[0], int(status[0]), False)


@gpu
def test_libjpeg_turbo_series_loads_like_the_uncompressed_one(golden, tmp_path):
    from _dicom_writer import _write_dicom
    from lungmask_b200 import io as lio
    slices = sorted((c for c in golden if c["name"].startswith("ljt_series_")), key=lambda c: c["name"])
    assert len(slices) == 4 and ref.parse_jpeg(slices[0]["stream"])["entropy"]
    assert slices[0]["stream"][2:4] == b"\xff\xe0"                  # libjpeg-turbo's APP0 (JFIF) before SOF3
    vol = np.stack([c["expected"].view(np.int16) for c in slices])
    for name in ("raw", "jpeg"):
        (tmp_path / name).mkdir()
    for k, c in enumerate(slices):
        ipp = (-20.0, -24.0, 2.0 * k)
        _write_dicom(str(tmp_path / "raw" / ("im%d.dcm" % k)), vol[k], "1.2.840.9", ipp)
        dc.write_encapsulated(str(tmp_path / "jpeg" / ("im%d.dcm" % k)), c["stream"], dc.JPEG_LOSSLESS_SV1, c["rows"],
                              c["cols"], "1.2.840.9", ipp, fragments=1 + k % 2)
    a, b = lio.load_input_image(str(tmp_path / "raw")), lio.load_input_image(str(tmp_path / "jpeg"))
    assert a.array.dtype == b.array.dtype and np.array_equal(a.array, b.array) and np.array_equal(a.array, vol)
    assert (a.spacing, a.origin, a.direction) == (b.spacing, b.origin, b.direction)


@gpu
def test_abi_edges():
    from lungmask_b200 import _native
    arrays, status = _native.decode_frames(b"", np.zeros(0, _native.FRAME_DTYPE), 0)
    assert arrays == [] and status.size == 0
    kat = bytes.fromhex("ff d8 ff c3 00 0b 10 00 01 00 02 01 01 11 00 ff c4 00 14 00 01 00 00 00 00 00 00 00 00 00 00 00 "
                        "00 00 00 00 10 ff da 00 08 01 01 00 01 00 00 3f ff d9")
    frames = np.zeros(5, _native.FRAME_DTYPE)
    frames[0] = (0, len(kat), 1, 1, 2, 0)
    frames[1] = (len(kat), 0, 1, 3, 3, 0)                   # zero-length JPEG frame
    frames[2] = (len(kat), 0, 2, 3, 3, 0)                   # zero-length RLE frame
    frames[3] = (0, len(kat), 3, 1, 2, 0)                   # unknown codecs
    frames[4] = (0, len(kat), 0, 1, 2, 0)
    arrays, status = _native.decode_frames(kat, frames, 0)
    assert status.tolist() == [0, -60, -60, -60, -60] and arrays[0].tolist() == [[0, 32768]]
