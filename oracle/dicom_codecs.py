"""Encoders for the compressed DICOM transfer syntaxes lungmask_b200 reads (test infrastructure, numpy only).

  * jpeg_lossless_encode  ITU-T T.81 process 14 (SOF3): precision P <= 16, predictors 1-7, point transform Pt, optional
                          restart interval of whole rows, a Huffman table fitted to the data that codes every
                          difference category 0-16 (syntaxes 1.2.840.10008.1.2.4.57 / .4.70)
  * rle_encode            DICOM PS3.5 Annex G for 16-bit samples: two PackBits segments (most significant bytes first)
                          with literal and replicate runs, replicate runs of more than 128 bytes split
  * write_encapsulated    a Part-10 file with encapsulated pixel data (PS3.5 A.4): Basic Offset Table item (empty or
                          filled), the frame split over one or more fragments, sequence delimiter

Both encoders are vectorised (bit packing by cumulative code lengths), so a 300 x 512^2 series encodes in seconds.  At
P = 8 the JPEG encoder is pinned against libjpeg-turbo through Pillow (tests/test_dicom_compressed.py).
"""
import heapq
import struct

import numpy as np

JPEG_LOSSLESS_SV1 = "1.2.840.10008.1.2.4.70"
JPEG_LOSSLESS = "1.2.840.10008.1.2.4.57"
RLE_LOSSLESS = "1.2.840.10008.1.2.5"


# --------------------------------------------------------------------------------------------------------------
# JPEG Lossless
# --------------------------------------------------------------------------------------------------------------
def predict(x, P, predictor, pt, restart_rows):
    """The prediction of every sample of x (values already point-transformed), T.81 H.1.2.1 with restarts."""
    x = x.astype(np.int64)
    H, W = x.shape
    Ra = np.zeros_like(x)
    Rb = np.zeros_like(x)
    Rc = np.zeros_like(x)
    Ra[:, 1:] = x[:, :-1]
    Rb[1:, :] = x[:-1, :]
    Rc[1:, 1:] = x[:-1, :-1]
    pred = {1: Ra, 2: Rb, 3: Rc, 4: Ra + Rb - Rc, 5: Ra + ((Rb - Rc) >> 1), 6: Rb + ((Ra - Rc) >> 1),
            7: (Ra + Rb) >> 1}[predictor].copy()
    pred[:, 0] = Rb[:, 0]                                   # first column: Rb
    step = restart_rows or H
    for r0 in range(0, H, step):                            # first row of the scan and of every restart interval: Ra
        pred[r0, 1:] = x[r0, :-1]
        pred[r0, 0] = 1 << (P - pt - 1)
    return pred


def categories(d):
    """Difference (modulo 2^16) -> (SSSS, additional bits value).  SSSS 16 stands for 32768 and has no additional bits."""
    d = d & 0xFFFF
    s = np.where(d >= 32768, d - 65536, d)
    cat = np.zeros(d.shape, np.int64)
    a = np.abs(s)
    nz = a > 0
    cat[nz] = np.floor(np.log2(a[nz])).astype(np.int64) + 1
    cat[d == 32768] = 16
    extra = np.where(s < 0, s + (1 << cat) - 1, s)
    extra[cat == 16] = 0
    return cat, extra


def huffman_table(freq):
    """(BITS[1..16], HUFFVAL) of a code for the 17 categories, at most 16 bits, no all-ones code (T.81 K.2 / K.3 with
    a reserved pseudo-symbol as libjpeg does); every category gets a code."""
    freq = [int(f) + 1 for f in freq[:17]] + [0]            # + 1: categories absent from the data keep a code
    freq[17] = 0
    syms = list(range(17)) + [256]
    weights = freq[:17] + [1]                               # the pseudo-symbol takes the all-ones code
    heap = [(w, i, [s]) for i, (w, s) in enumerate(zip(weights, syms))]
    heapq.heapify(heap)
    length = {s: 0 for s in syms}
    tie = len(heap)
    while len(heap) > 1:
        w1, _, a = heapq.heappop(heap)
        w2, _, b = heapq.heappop(heap)
        for s in a + b:
            length[s] += 1
        heapq.heappush(heap, (w1 + w2, tie, a + b))
        tie += 1
    bits = [0] * 33
    for s in syms:
        bits[length[s]] += 1
    for i in range(32, 16, -1):                             # K.3 Adjust_BITS: limit to 16 bits
        while bits[i] > 0:
            j = i - 2
            while bits[j] == 0:
                j -= 1
            bits[i] -= 2
            bits[i - 1] += 1
            bits[j + 1] += 2
            bits[j] -= 1
    i = 16
    while bits[i] == 0:
        i -= 1
    bits[i] -= 1                                            # drop the pseudo-symbol (the longest, last code)
    order = sorted(range(17), key=lambda s: (-freq[s], s))  # most frequent first = shortest codes
    return bits[1:17], order


def canonical_codes(bits, vals):
    """symbol -> (code, length), T.81 Annex C."""
    out, code, k = {}, 0, 0
    for l in range(1, 17):
        for _ in range(bits[l - 1]):
            out[vals[k]] = (code, l)
            code += 1
            k += 1
        code <<= 1
    return out


def pack_bits(values, lengths):
    """Concatenates the MSB-first bit strings (value, length <= 32) and pads with 1-bits to whole bytes."""
    values = np.asarray(values, np.uint64).ravel()
    lengths = np.asarray(lengths, np.int64).ravel()
    total = int(lengths.sum())
    nbytes = (total + 7) // 8
    bits = np.ones(nbytes * 8, np.uint8)
    ends = np.cumsum(lengths)
    starts = ends - lengths
    for k in range(int(lengths.max()) if lengths.size else 0):
        m = lengths > k
        b = (values[m] >> (lengths[m] - 1 - k).astype(np.uint64)) & np.uint64(1)
        bits[starts[m] + k] = b.astype(np.uint8)
    return np.packbits(bits)


def stuff(b):
    """0xFF in entropy-coded data is followed by a stuffed 0x00."""
    b = np.asarray(b, np.uint8)
    idx = np.flatnonzero(b == 0xFF)
    return np.insert(b, idx + 1, 0).tobytes()


def jpeg_lossless_encode(img, P=16, predictor=1, pt=0, restart_rows=0, table=None):
    """img: 2-D array of stored values (int16 / uint16; signed data as its P-bit two's complement pattern) -> bytes.
    restart_rows: restart interval in rows (0: none).  table: (BITS, HUFFVAL), default fitted to the data."""
    img = np.asarray(img)
    H, W = img.shape
    assert 2 <= P <= 16 and 1 <= predictor <= 7 and 0 <= pt < P
    x = (img.astype(np.int64) & ((1 << P) - 1)) >> pt
    d = x - predict(x, P, predictor, pt, restart_rows)
    cat, extra = categories(d)
    bits, vals = table if table is not None else huffman_table(np.bincount(cat.ravel(), minlength=17))
    codes = canonical_codes(bits, vals)
    cl = np.zeros(17, np.int64)
    cv = np.zeros(17, np.int64)
    for s, (c, l) in codes.items():
        cv[s], cl[s] = c, l
    xl = np.where(cat == 16, 0, cat)
    value = (cv[cat] << xl) | extra
    length = cl[cat] + xl
    step = restart_rows or H
    ent = b""
    for k, r0 in enumerate(range(0, H, step)):
        if k:
            ent += bytes([0xFF, 0xD0 + (k - 1) % 8])
        ent += stuff(pack_bits(value[r0:r0 + step], length[r0:r0 + step]))
    seg = lambda m, body: bytes([0xFF, m]) + struct.pack(">H", len(body) + 2) + body
    out = b"\xff\xd8"
    out += seg(0xC3, struct.pack(">BHHB", P, H, W, 1) + bytes([1, 0x11, 0]))
    out += seg(0xC4, bytes([0x00]) + bytes(bits) + bytes(vals))
    if restart_rows:
        out += seg(0xDD, struct.pack(">H", restart_rows * W))
    out += seg(0xDA, bytes([1, 1, 0x00, predictor, 0, pt]))
    return out + ent + b"\xff\xd9"


# --------------------------------------------------------------------------------------------------------------
# RLE Lossless
# --------------------------------------------------------------------------------------------------------------
def packbits(b, min_rep=3):
    """PackBits of one byte plane: replicate runs for repeats of >= min_rep bytes (split at 128), literal runs of <= 128
    bytes for the rest.  Padded to an even length with a zero byte."""
    b = np.asarray(b, np.uint8).ravel()
    n = b.size
    brk = np.flatnonzero(np.diff(b.astype(np.int16)) != 0) + 1
    rs = np.concatenate([[0], brk])
    rl = np.diff(np.concatenate([rs, [n]]))
    rep = rl >= min_rep
    # literal stretches: maximal groups of consecutive non-replicate runs
    lit_run = ~rep
    grp_start = lit_run & np.concatenate([[True], ~lit_run[:-1]])
    gid = np.cumsum(grp_start) - 1
    ls = rs[grp_start]
    ll = np.bincount(gid[lit_run], weights=rl[lit_run], minlength=int(grp_start.sum())).astype(np.int64)
    # pieces of <= 128 bytes
    def split(starts, lens):
        cnt = (lens + 127) // 128
        idx = np.repeat(np.arange(starts.size), cnt)
        k = np.arange(idx.size) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        st = starts[idx] + 128 * k
        return st, np.minimum(128, lens[idx] - 128 * k)
    ps_r, pl_r = split(rs[rep], rl[rep])
    ps_l, pl_l = split(ls, ll)
    starts = np.concatenate([ps_r, ps_l])
    lens = np.concatenate([pl_r, pl_l])
    is_rep = np.concatenate([np.ones(ps_r.size, bool), np.zeros(ps_l.size, bool)])
    order = np.argsort(starts, kind="stable")
    starts, lens, is_rep = starts[order], lens[order], is_rep[order]
    size = np.where(is_rep, 2, 1 + lens)
    off = np.cumsum(size) - size
    total = int(size.sum())
    out = np.zeros(total + (total & 1), np.uint8)
    out[off] = np.where(is_rep, (257 - lens) & 0xFF, lens - 1).astype(np.uint8)
    out[off[is_rep] + 1] = b[starts[is_rep]]
    lit = ~is_rep
    cnt = lens[lit]
    src = np.repeat(starts[lit], cnt) + (np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt))
    dst = np.repeat(off[lit] + 1, cnt) + (np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt))
    out[dst] = b[src]
    return out.tobytes()


def rle_encode(img, min_rep=3):
    """16-bit frame (stored values) -> RLE Lossless frame: 64-byte header + MSB segment + LSB segment."""
    u = np.ascontiguousarray(np.asarray(img).astype(np.uint16) if np.asarray(img).dtype != np.int16
                             else np.asarray(img).view(np.uint16))
    segs = [packbits(u >> 8, min_rep), packbits(u & 0xFF, min_rep)]
    hdr = struct.pack("<16I", 2, 64, 64 + len(segs[0]), *([0] * 13))
    return hdr + segs[0] + segs[1]


# --------------------------------------------------------------------------------------------------------------
# DICOM Part-10 with encapsulated pixel data (explicit VR little endian, the tags lungmask_b200.io reads)
# --------------------------------------------------------------------------------------------------------------
def _elem(tag, vr, value):
    if isinstance(value, str):
        value = value.encode("ascii")
        if len(value) % 2:
            value += b"\x00" if vr == "UI" else b" "
    g, e = tag
    if vr in ("OB", "OW", "SQ", "UN"):
        return struct.pack("<HH2sHI", g, e, vr.encode(), 0, len(value)) + value
    return struct.pack("<HH2sH", g, e, vr.encode(), len(value)) + value


def encapsulate(frame, fragments=1, bot="empty"):
    """(7FE0,0010) with undefined length: Basic Offset Table item ("empty" or "filled"), the frame over `fragments`
    even-length fragments (an odd frame gets one pad byte), sequence delimiter."""
    if len(frame) % 2:
        frame = frame + b"\x00"
    n = len(frame) // 2
    cuts = [2 * (n * k // fragments) for k in range(fragments + 1)]
    item = lambda v: struct.pack("<HHI", 0xFFFE, 0xE000, len(v)) + v
    out = struct.pack("<HH2sHI", 0x7FE0, 0x0010, b"OB", 0, 0xFFFFFFFF)
    out += item(struct.pack("<I", 0) if bot == "filled" else b"")
    for a, b in zip(cuts[:-1], cuts[1:]):
        out += item(frame[a:b])
    return out + struct.pack("<HHI", 0xFFFE, 0xE0DD, 0)


def write_encapsulated(path, frame, syntax, rows, cols, series, ipp, signed=True, image_type="ORIGINAL\\PRIMARY\\AXIAL",
                       slope=1, intercept=0, iop="1\\0\\0\\0\\1\\0", study="1.2.3", fragments=1, bot="empty",
                       pixel_data=None):
    """A single-frame Part-10 file whose pixel data is `frame` (an encoded JPEG Lossless / RLE frame) under `syntax`.
    The tags and values are those of tests/_dicom_writer.py, so both writers describe the same geometry.
    pixel_data: the raw (7FE0,0010) element instead of encapsulate(frame, fragments, bot)."""
    meta = _elem((0x0002, 0x0010), "UI", syntax)
    meta = _elem((0x0002, 0x0000), "UL", struct.pack("<I", len(meta))) + meta
    body = _elem((0x0008, 0x0008), "CS", image_type)
    body += _elem((0x0020, 0x000D), "UI", study)
    body += _elem((0x0020, 0x000E), "UI", series)
    body += _elem((0x0020, 0x0032), "DS", "\\".join("%g" % v for v in ipp))
    body += _elem((0x0020, 0x0037), "DS", iop)
    body += _elem((0x0028, 0x0002), "US", struct.pack("<H", 1))
    body += _elem((0x0028, 0x0010), "US", struct.pack("<H", rows))
    body += _elem((0x0028, 0x0011), "US", struct.pack("<H", cols))
    body += _elem((0x0028, 0x0030), "DS", "0.5\\0.75")
    body += _elem((0x0028, 0x0100), "US", struct.pack("<H", 16))
    body += _elem((0x0028, 0x0103), "US", struct.pack("<H", 1 if signed else 0))
    body += _elem((0x0028, 0x1052), "DS", "%g" % intercept)
    body += _elem((0x0028, 0x1053), "DS", "%g" % slope)
    body += pixel_data if pixel_data is not None else encapsulate(frame, fragments, bot)
    with open(path, "wb") as f:
        f.write(b"\x00" * 128 + b"DICM" + meta + body)
