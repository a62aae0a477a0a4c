"""Writes tests/golden/codec_conformance.npz: JPEG Lossless and RLE frames with the samples (or the status) that
lm_decode_frames must give for them, so that the GPU suite checks csrc/decode.cu against libjpeg-turbo and against the
sequential reference decoder (oracle/ljpeg_ref.py) without either being present where it runs.

    python -m oracle.make_codec_golden            regenerate the fixture (needs Pillow's libjpeg-turbo)
    python -m oracle.make_codec_golden --check    regenerate it in memory and compare with the committed file

Origins of the frames:
  libjpeg-turbo  written by libjpeg-turbo (oracle/libjpeg_turbo.py); expected = libjpeg-turbo's own decode, which must
                 also equal the input
  hand           JPEG streams valid per T.81 that exercise one marker layout, table shape or synchronisation case each
                 (J1-J12); expected = the sequential reference, and libjpeg-turbo's decode must agree where it accepts
                 the stream (column ljt: 1 accepted and equal, 0 rejected)
  rle            hand-built PackBits segments (R1-R5, edge shapes); expected = the PackBits reference
  malformed      one deterministic stream per defect; expected = the LM_ERR_DECODE_* status include/lungmask_b200.h
                 documents, which the sequential reference raises too

The expected samples are stored as the SHA-256 of their little-endian uint16 bytes, not as samples: the sequential
reference regenerates them wherever the tests run, and the digest ties that regeneration to libjpeg-turbo's decode (or,
for hand-built frames, to the reference decode checked against libjpeg-turbo here), which keeps the file small.
"""
import hashlib
import os
import struct
import sys

import numpy as np

from oracle import dicom_codecs as dc
from oracle import libjpeg_turbo as lj
from oracle import ljpeg_ref as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "codec_conformance.npz")
CASE_DTYPE = np.dtype([("offset", "<u8"), ("length", "<u8"), ("codec", "<i4"), ("rows", "<i4"), ("cols", "<i4"),
                       ("is_signed", "<i4"), ("P", "<i4"), ("status", "<i4"), ("ljt", "<i4")])
JPEG, RLE = 1, 2
SYNC_WORST_CASE = "J11_sync_worst_case"


# --------------------------------------------------------------------------------------------------------------
# stream surgery: a JPEG stream as its marker segments
# --------------------------------------------------------------------------------------------------------------
def seg(m, body):
    return bytes([0xFF, m]) + struct.pack(">H", len(body) + 2) + body


def dht(*tables):
    """One DHT segment defining (th, bits, vals) tables."""
    return seg(0xC4, b"".join(bytes([th]) + bytes(bits) + bytes(vals) for th, bits, vals in tables))


def split_stream(b):
    """oracle.dicom_codecs output -> dict of its segment bodies (SOF3, DHT, DRI, SOS) and the entropy-coded data."""
    p, out = 2, {}
    while True:
        m, L = b[p + 1], struct.unpack_from(">H", b, p + 2)[0]
        out[m] = b[p + 4:p + 2 + L]
        p += 2 + L
        if m == 0xDA:
            out["ent"] = b[p:-2]
            return out


def assemble(parts, *layout):
    """SOI + the layout (raw bytes, or 0xC3 / 0xDD / 0xDA for the stream's own segment) + entropy data + EOI."""
    out = b"\xff\xd8"
    for x in layout:
        out += seg(x, parts[x]) if isinstance(x, int) else x
    return out + parts["ent"] + b"\xff\xd9"


def image_from_differences(d, P):
    """The predictor-1 image whose differences (no restarts, Pt 0) are d (|d| < 32768)."""
    x = np.array(d, np.int64)
    x[0, 0] += 1 << (P - 1)
    x[:, 0] = np.cumsum(x[:, 0])
    return (np.cumsum(x, axis=1) & 0xFFFF).astype(np.uint16)


def differences_of_categories(rng, cats):
    """A random difference of each given category (T.81 Table H.2), random sign; category 0 -> 0."""
    cats = np.asarray(cats, np.int64)
    lo = np.where(cats > 0, 1 << np.maximum(cats - 1, 0), 0)
    mag = lo + (rng.random(cats.shape) * lo).astype(np.int64)
    return np.where(rng.random(cats.shape) < 0.5, -mag, mag)


# --------------------------------------------------------------------------------------------------------------
# PackBits writer for hand-built RLE frames
# --------------------------------------------------------------------------------------------------------------
def lit(bs):
    bs = bytes(bs)
    assert 1 <= len(bs) <= 128
    return bytes([len(bs) - 1]) + bs


def rep(v, n):
    assert 2 <= n <= 128
    return bytes([257 - n, v])


NOOP = b"\x80"


def packbits_runs(plane, min_rep=3, row=0, noop=False):
    """Greedy PackBits of one plane: replicate runs of >= min_rep equal bytes, literal runs of <= 128 bytes, runs
    broken at every multiple of `row` bytes when row > 0, a -128 byte between runs when noop."""
    plane = bytes(plane)
    out, i, n = [], 0, len(plane)
    while i < n:
        stop = min(n, (i // row + 1) * row) if row else n
        j = i
        while j < stop and plane[j] == plane[i] and j - i < 128:
            j += 1
        if j - i >= min_rep:
            out.append(rep(plane[i], j - i))
            i = j
            continue
        j = i + 1
        while j < stop and j - i < 128:
            k = j
            while k < stop and plane[k] == plane[j] and k - j < min_rep:
                k += 1
            if k - j >= min_rep:
                break
            j += 1
        out.append(lit(plane[i:j]))
        i = j
    return (NOOP if noop else b"").join(out)


def rle_frame(hi, lo):
    """Header + two segments (each padded to an even length)."""
    hi += b"\x00" * (len(hi) & 1)
    lo += b"\x00" * (len(lo) & 1)
    return struct.pack("<16I", 2, 64, 64 + len(hi), *([0] * 13)) + hi + lo


def planes(img):
    u = np.asarray(img, np.uint16).ravel()
    return (u >> 8).astype(np.uint8).tobytes(), (u & 0xFF).astype(np.uint8).tobytes()


# --------------------------------------------------------------------------------------------------------------
# cases
# --------------------------------------------------------------------------------------------------------------
def noise_with_bands(rng, P, shape=(32, 32)):
    """Full-range noise in the top quarter (every difference category up to P), small noise on a ramp below it, and
    flat bands: long zero-difference runs and 0xFF bytes."""
    h, w = shape
    amp = 1 << (P // 2)
    ramp = (np.arange(h)[:, None] * 3 + np.arange(w)[None, :] * 5) * max(1, (1 << P) // 256)
    img = (ramp + rng.integers(0, amp, shape)) % (1 << P)
    img[:h // 4] = rng.integers(0, 1 << P, (h // 4, w))
    img[h // 4 + 2:h // 4 + 5, :] = (1 << P) - 1
    img[:, w // 2:w // 2 + 3] = rng.integers(0, 1 << P)
    img[3 * h // 4:3 * h // 4 + 3, 2:w - 4] = 0
    return img.astype(np.uint16)


def libjpeg_turbo_cases():
    """(name, img, P, predictor, pt, restart_in_rows)"""
    rng = np.random.default_rng(2026)
    jobs = []
    for P in (2, 8, 12, 15, 16):
        for pred in range(1, 8):
            for pt in (0, min(3, P - 1)):
                for rr in (0, 3):
                    img = noise_with_bands(rng, P)
                    jobs.append(("ljt_P%d_p%d_pt%d_r%d" % (P, pred, pt, rr), (img >> pt) << pt, P, pred, pt, rr))
    img = noise_with_bands(rng, 12)
    jobs.append(("ljt_P12_p4_pt11", (img >> 11) << 11, 12, 4, 11, 2))
    alt = np.zeros((33, 65), np.uint16)
    alt[::2, ::2] = alt[1::2, 1::2] = 32768
    jobs.append(("ljt_category16", alt, 16, 1, 0, 0))
    jobs.append(("ljt_1x1", rng.integers(0, 65536, (1, 1)).astype(np.uint16), 16, 1, 0, 0))
    jobs.append(("ljt_1x4096", rng.integers(0, 65536, (1, 4096)).astype(np.uint16), 16, 7, 0, 0))
    jobs.append(("ljt_4096x1", rng.integers(0, 4096, (4096, 1)).astype(np.uint16), 12, 2, 0, 0))
    ct = np.load(os.path.join(ROOT, "tests", "golden", "ct_slice_512.npz"))["slice"].astype(np.int16).view(np.uint16)
    ct = np.ascontiguousarray(ct[200:296, 40:136])          # 96^2 of the real slice: lung and soft tissue
    jobs += [("ljt_ct96_p1", ct, 16, 1, 0, 0), ("ljt_ct96_p6", ct, 16, 6, 0, 0), ("ljt_ct96_p6_r16", ct, 16, 6, 0, 16)]
    from oracle import synth                                # a CT-like series for the end-to-end test
    vol = synth.phantom(4, 48, 40, seed=41).astype(np.int16).view(np.uint16)
    jobs += [("ljt_series_%d" % k, vol[k], 16, 1, 0, 0) for k in range(vol.shape[0])]
    return jobs


def hand_jpeg_cases():
    """(name, stream, rows, cols, P): J1-J12, valid per T.81."""
    rng = np.random.default_rng(7)
    out = []
    img = noise_with_bands(rng, 12, (24, 20))
    parts = split_stream(dc.jpeg_lossless_encode(img, P=12, predictor=4))
    parts_r = split_stream(dc.jpeg_lossless_encode(img, P=12, predictor=5, restart_rows=4))
    t0 = parts[0xC4]
    other = (0, [0, 0, 1] + [1] * 13, list(range(16, 2, -1)))      # a valid table that decodes this data differently
    bits, vals = list(t0[1:17]), list(t0[17:])
    out.append(("J1_dht_before_sof", assemble(parts, 0xC4, 0xC3, 0xDA), 24, 20, 12))
    two_tables = dht((0, *other[1:]), (1, *other[1:]), (2, bits, vals), (3, *other[1:]))
    sos2 = {**parts, 0xDA: parts[0xDA][:2] + b"\x20" + parts[0xDA][3:]}
    out.append(("J2_tables_0_to_3_td2", assemble(sos2, 0xC3, two_tables, 0xDA), 24, 20, 12))
    out.append(("J3_table_redefined", assemble(parts, dht(other), 0xC3, 0xC4, 0xDA), 24, 20, 12))
    app0 = seg(0xE0, b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00")
    app14 = seg(0xEE, b"Adobe\x00\x64\x00\x00\x00\x00\x00")
    com = seg(0xFE, b"lungmask_b200 conformance")
    dqt = seg(0xDB, b"\x00" + bytes(range(1, 65)))
    tem = b"\xff\x01"
    out.append(("J4_app_com_dqt_tem", assemble(parts_r, app0, tem, 0xC3, app14, 0xC4, tem, com, dqt, 0xDD, tem, 0xDA),
                24, 20, 12))
    fill = b"\xff" * 3
    ent = parts_r["ent"]
    filled = bytearray()
    for i, c in enumerate(ent):                             # fill before every RSTm (0xFF then 0xD0-0xD7)
        if c == 0xFF and i + 1 < len(ent) and 0xD0 <= ent[i + 1] <= 0xD7:
            filled += fill
        filled.append(c)
    s = b"\xff\xd8" + fill + seg(0xC3, parts_r[0xC3]) + fill + seg(0xC4, parts_r[0xC4]) + fill + seg(0xDD, parts_r[0xDD])
    s += fill + seg(0xDA, parts_r[0xDA]) + bytes(filled) + fill + b"\xff\xd9"
    out.append(("J5_fill_bytes", s, 24, 20, 12))
    for cid in (0, 255):
        sof = parts[0xC3][:6] + bytes([cid]) + parts[0xC3][7:]
        sos = bytes([1, cid]) + parts[0xDA][2:]
        out.append(("J6_component_id_%d" % cid, assemble({**parts, 0xC3: sof, 0xDA: sos}, 0xC3, 0xC4, 0xDA), 24, 20, 12))
    # J7: one code of every length 1-16; the frequent categories 10-15 on the 11-16-bit codes (31-bit codewords)
    cats = np.where(rng.random((64, 64)) < 0.9, rng.integers(10, 16, (64, 64)), rng.integers(0, 10, (64, 64)))
    img7 = image_from_differences(differences_of_categories(rng, cats), 16)
    t7 = ([1] * 16, list(range(16)))
    out.append(("J7_long_codes", dc.jpeg_lossless_encode(img7, P=16, predictor=1, table=t7), 64, 64, 16))
    # J8: HUFFVAL in no particular order, categories 7-16 absent
    img8 = image_from_differences(differences_of_categories(rng, rng.integers(0, 7, (30, 50))), 16)
    t8 = ([0, 2, 2, 3] + [0] * 12, [5, 0, 3, 6, 1, 4, 2])
    out.append(("J8_unsorted_huffval", dc.jpeg_lossless_encode(img8, P=16, predictor=1, table=t8), 30, 50, 16))
    # J9: DRI 0, and DRI of at least rows x cols (no RSTm at all)
    out.append(("J9_dri_0", assemble(parts, 0xC3, 0xC4, seg(0xDD, b"\x00\x00"), 0xDA), 24, 20, 12))
    out.append(("J9_dri_480", assemble(parts, 0xC3, 0xC4, seg(0xDD, struct.pack(">H", 480)), 0xDA), 24, 20, 12))
    out.append(("J9_dri_65520", assemble(parts, 0xC3, 0xC4, seg(0xDD, struct.pack(">H", 65520)), 0xDA), 24, 20, 12))
    # J10: one-row restart intervals on 1- and 2-row frames
    for h in (1, 2):
        im = noise_with_bands(rng, 16, (h, 37))
        out.append(("J10_ri1_rows%d" % h, dc.jpeg_lossless_encode(im, P=16, predictor=6, restart_rows=1), h, 37, 16))
    # J11: the synchronisation worst case: every codeword the 3-bit code 000 (category 0), 1024 not a multiple of 3
    img11 = np.full((320, 320), 1 << 15, np.uint16)
    out.append((SYNC_WORST_CASE, dc.jpeg_lossless_encode(img11, P=16, predictor=1, table=([0, 0, 1] + [0] * 13, [0])),
                320, 320, 16))
    # J12: codes 00 (category 0) and 01 (category 1) only; every difference +1, so codewords 011: a chunk decoded out
    # of phase meets the undefined code 11 or 10 at once
    img12 = image_from_differences(np.ones((64, 64), np.int64), 16)
    out.append(("J12_undefined_out_of_phase", dc.jpeg_lossless_encode(img12, P=16, predictor=1,
                                                                       table=([0, 2] + [0] * 14, [0, 1])), 64, 64, 16))
    return out


def rle_cases():
    """(name, frame, rows, cols, img): R1-R5 and edge shapes."""
    rng = np.random.default_rng(11)
    out = []
    img = np.repeat(rng.integers(0, 6, 300), rng.integers(1, 9, 300))[:24 * 30].reshape(24, 30).astype(np.uint16) * 257
    hi, lo = planes(img)
    out.append(("R1_noop_bytes", rle_frame(NOOP + packbits_runs(hi, noop=True) + NOOP, packbits_runs(lo, noop=True)), 24, 30, img))
    hi, hseg = b"", b""
    for k in range(4):                                      # 4 x (128 literal bytes, a 2-byte replicate run), 80 literal
        lits = rng.permutation(256)[:128].astype(np.uint8).tobytes()
        hi += lits + bytes([k + 1]) * 2
        hseg += lit(lits) + rep(k + 1, 2)
    tail = rng.integers(0, 256, 80).astype(np.uint8).tobytes()
    hi, hseg = hi + tail, hseg + lit(tail)
    lo = rng.integers(0, 256, 600).astype(np.uint8).tobytes()
    img = ((np.frombuffer(hi, np.uint8).astype(np.uint16) << 8) | np.frombuffer(lo, np.uint8)).reshape(20, 30)
    out.append(("R2_rep2_lit128", rle_frame(hseg, packbits_runs(lo, min_rep=2)), 20, 30, img))
    img = np.repeat(rng.integers(0, 3, (17, 1)), 45, axis=1).astype(np.uint16) * 0x0101
    img[::4] = 0x7777                                       # runs would cross rows: the encoder stops them at row ends
    hi, lo = planes(img)
    out.append(("R3_rows", rle_frame(packbits_runs(hi, row=45), packbits_runs(lo, row=45, min_rep=2)), 17, 45, img))
    img = rng.integers(0, 65536, (9, 13)).astype(np.uint16)
    hi, lo = planes(img)
    out.append(("R4_bytes_after_last_run", rle_frame(packbits_runs(hi) + b"\x05\x01\x02\x03", packbits_runs(lo) + b"\xfe\x09\x80"),
                9, 13, img))
    img = np.full((16, 16), 0xABCD, np.uint16)
    out.append(("R5_rep128_at_end", rle_frame(rep(0xAB, 128) * 2, rep(0xCD, 128) + NOOP + rep(0xCD, 128)), 16, 16, img))
    one = np.array([[0xBEEF]], np.uint16)
    out.append(("R_1x1", rle_frame(lit(b"\xbe"), NOOP + lit(b"\xef")), 1, 1, one))
    img = rng.integers(0, 4, (1, 301)).astype(np.uint16) * 0x0102
    hi, lo = planes(img)
    out.append(("R_1x301", rle_frame(packbits_runs(hi, min_rep=2), packbits_runs(lo)), 1, 301, img))
    return out


def malformed_cases():
    """(name, stream, codec, rows, cols, status)"""
    img = noise_with_bands(np.random.default_rng(5), 12, (24, 20))
    parts = split_stream(dc.jpeg_lossless_encode(img, P=12, predictor=1))
    parts_r = split_stream(dc.jpeg_lossless_encode(img, P=12, predictor=1, restart_rows=4))
    out = []
    sos1 = {**parts, 0xDA: parts[0xDA][:2] + b"\x10" + parts[0xDA][3:]}
    out.append(("M_sos_undefined_table", assemble(sos1, 0xC3, 0xC4, 0xDA), JPEG, 24, 20, ref.HEADER))
    over = dht((0, [3] + [0] * 15, [0, 1, 2]))                    # three 1-bit codes
    out.append(("M_bits_overfill", assemble(parts, 0xC3, over, 0xDA), JPEG, 24, 20, ref.HEADER))
    dri = {**parts_r, 0xDD: struct.pack(">H", 30)}
    out.append(("M_dri_not_whole_rows", assemble(dri, 0xC3, 0xC4, 0xDD, 0xDA), JPEG, 24, 20, ref.HEADER))
    i = parts_r["ent"].index(b"\xff\xd0")
    rst = dict(parts_r, ent=parts_r["ent"][:i] + b"\xff\xd1" + parts_r["ent"][i + 2:])
    out.append(("M_rst_out_of_sequence", assemble(rst, 0xC3, 0xC4, 0xDD, 0xDA), JPEG, 24, 20, ref.DATA))
    ent = parts["ent"]
    i = len(ent) // 2
    while ent[i - 1] == 0xFF:
        i += 1
    app = dict(parts, ent=ent[:i] + b"\xff\xe1" + ent[i:])
    out.append(("M_marker_in_entropy_data", assemble(app, 0xC3, 0xC4, 0xDA), JPEG, 24, 20, ref.DATA))
    out.append(("M_rle_runs_past_frame", rle_frame(rep(1, 128), rep(2, 100)), RLE, 10, 10, ref.LENGTH))
    out.append(("M_rle_literal_past_segment", rle_frame(rep(1, 100), b"\x7f\x01\x02\x03"), RLE, 10, 10, ref.LENGTH))
    fr = rle_frame(rep(1, 100), rep(2, 100))
    out.append(("M_rle_offsets_out_of_order", fr[:4] + struct.pack("<2I", 64, 60) + fr[12:], RLE, 10, 10, ref.HEADER))
    return out


def sign_extend(u, P):
    """The stored values a decoder with is_signed gives: bit P - 1 extended (P < 16), as a uint16 bit pattern."""
    u = np.asarray(u, np.uint16)
    if P >= 16:
        return u
    neg = (u >> (P - 1)) & 1
    return np.where(neg == 1, u | np.uint16((0xFFFF << P) & 0xFFFF), u).astype(np.uint16)


def digest(samples):
    return hashlib.sha256(np.ascontiguousarray(samples, "<u2").tobytes()).hexdigest()


def generate():
    cases = []                                              # (name, origin, stream, codec, rows, cols, P, status, ljt, expected)
    jobs = libjpeg_turbo_cases()
    streams = lj.encode_many([j[1:] for j in jobs])
    for (name, img, P, pred, pt, rr), s, (dec, Pd) in zip(jobs, streams, lj.decode_many_with_header(streams)):
        assert Pd == P and np.array_equal(dec, img), name
        cases.append((name, "libjpeg-turbo", s, JPEG, *img.shape, P, 0, 1, dec))
    for name, s, h, w, P in hand_jpeg_cases():
        exp = ref.jpeg_lossless_decode(s)
        try:
            assert np.array_equal(lj.decode(s), exp), "libjpeg-turbo disagrees with the reference on " + name
            agrees = 1
        except lj.LibjpegError:
            agrees = 0
        cases.append((name, "hand", s, JPEG, h, w, P, 0, agrees, exp))
    for name, s, h, w, img in rle_cases():
        exp = ref.rle_decode(s, h, w)
        assert np.array_equal(exp, img), name
        cases.append((name, "rle", s, RLE, h, w, 16, 0, -1, exp))
    for name, s, codec, h, w, status in malformed_cases():
        try:
            ref.jpeg_lossless_decode(s) if codec == JPEG else ref.rle_decode(s, h, w)
            raise AssertionError("the reference accepts " + name)
        except ref.DecodeError as e:
            assert e.status == status, (name, e)
        cases.append((name, "malformed", s, codec, h, w, 16, status, -1, None))

    table = np.zeros(len(cases), CASE_DTYPE)
    off = 0
    for k, (name, origin, s, codec, h, w, P, status, ljt, exp) in enumerate(cases):
        table[k] = (off, len(s), codec, h, w, 0, P, status, ljt)
        off += len(s)
    return dict(data=np.frombuffer(b"".join(c[2] for c in cases), np.uint8), frames=table,
                name=np.array([c[0] for c in cases]), origin=np.array([c[1] for c in cases]),
                sha256=np.array(["" if c[9] is None else digest(c[9]) for c in cases]),
                libjpeg_turbo_version=np.array(lj.version()))


def main(argv):
    new = generate()
    if "--check" in argv:
        old = np.load(OUT)
        bad = [k for k in new if k not in old or not np.array_equal(old[k], new[k])]
        if bad:
            sys.exit("%s differs from what oracle/make_codec_golden.py generates: %s (libjpeg-turbo here %s, in the "
                     "fixture %s)" % (os.path.relpath(OUT, ROOT), bad, new["libjpeg_turbo_version"], old["libjpeg_turbo_version"]))
        print("%s: up to date (%d frames)" % (os.path.relpath(OUT, ROOT), len(new["frames"])))
        return
    np.savez_compressed(OUT, **new)
    print("wrote %s: %d frames, %d bytes" % (OUT, len(new["frames"]), os.path.getsize(OUT)))


if __name__ == "__main__":
    main(sys.argv[1:])
