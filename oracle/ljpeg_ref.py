"""Sequential reference decoders for the compressed pixel data lungmask_b200 reads (test oracle, Python and numpy).

  * jpeg_lossless_decode  ITU-T T.81 process 14 (SOF3) transcribed directly: marker segments per Annex B (fill bytes,
                          APPn / COM / DQT / TEM, several DHT segments, a table redefined by a later DHT), Huffman tables
                          per Annex C and F.2.2.3 (HUFFSIZE / HUFFCODE, MINCODE / MAXCODE / VALPTR), DECODE (F.16) one
                          bit at a time, prediction per H.1.2.1 with restart intervals and the point transform
  * packbits_decode       one PackBits segment, byte by byte per DICOM PS3.5 G.3.2, including the -128 no-op byte
  * rle_decode            a 16-bit single-sample RLE Lossless frame (PS3.5 Annex G): header and two segments

These share no code with oracle/dicom_codecs.py: they check that encoder and the CUDA decoder (csrc/decode.cu) from
outside.  Malformed input raises DecodeError carrying the LM_ERR_DECODE_* status include/lungmask_b200.h documents for
it.  One sample at a time in Python: meant for test-sized frames (a 512 x 512 frame takes seconds).
"""
import struct

import numpy as np

HEADER, DATA, LENGTH = -60, -61, -62        # LM_ERR_DECODE_HEADER / _DATA / _LENGTH


class DecodeError(ValueError):
    def __init__(self, status, msg):
        super().__init__("%s (status %d)" % (msg, status))
        self.status = status


def _need(cond, status, msg):
    if not cond:
        raise DecodeError(status, msg)


# --------------------------------------------------------------------------------------------------------------
# JPEG Lossless
# --------------------------------------------------------------------------------------------------------------
class HuffTable:
    """One DC table (Tc = 0): the decoder tables of T.81 F.2.2.3, built from BITS and HUFFVAL per Annex C."""

    def __init__(self, bits, huffval):
        self.huffval = list(huffval)
        huffsize = []                                       # C.1 (Figure C.1)
        for l in range(1, 17):
            huffsize += [l] * bits[l - 1]
        huffcode, code, si, k = [], 0, huffsize[0] if huffsize else 0, 0   # C.2 (Figure C.2)
        while k < len(huffsize):
            while k < len(huffsize) and huffsize[k] == si:
                huffcode.append(code)
                code += 1
                k += 1
            _need(code <= (1 << si), HEADER, "DHT: BITS overfill the code space of length %d" % si)
            code <<= 1
            si += 1
        self.maxcode, self.mincode, self.valptr = [-1] * 17, [0] * 17, [0] * 17   # F.2.2.3 (Figure F.15)
        j = 0
        for l in range(1, 17):
            if bits[l - 1]:
                self.valptr[l] = j
                self.mincode[l] = huffcode[j]
                j += bits[l - 1]
                self.maxcode[l] = huffcode[j - 1]


class _Bits:
    """NEXTBIT over one entropy-coded segment with stuffing and markers already removed."""

    def __init__(self, data):
        self.bits = np.unpackbits(np.frombuffer(bytes(data), np.uint8)).tolist()
        self.pos = 0

    def nextbit(self):
        _need(self.pos < len(self.bits), LENGTH, "a restart interval ends before its samples")
        b = self.bits[self.pos]
        self.pos += 1
        return b

    def receive(self, ssss):                                # F.2.2.4 RECEIVE
        v = 0
        for _ in range(ssss):
            v = (v << 1) | self.nextbit()
        return v


def _decode(br, t):                                         # F.2.2.3 DECODE (Figure F.16)
    i = 1
    code = br.nextbit()
    while code > t.maxcode[i]:
        i += 1
        _need(i <= 16, DATA, "undefined Huffman code")
        code = (code << 1) | br.nextbit()
    return t.huffval[t.valptr[i] + code - t.mincode[i]]


def _difference(br, t):                                     # H.1.2.2: SSSS, then EXTEND (F.12) of the extra bits
    s = _decode(br, t)
    _need(s <= 16, DATA, "difference category %d" % s)
    if s == 0:
        return 0
    if s == 16:
        return 32768
    v = br.receive(s)
    return v - (1 << s) + 1 if v < (1 << (s - 1)) else v


def parse_jpeg(data):
    """Marker segments SOI .. SOS (T.81 Annex B) -> dict(P, rows, cols, table, pred, pt, ri, entropy=bytes after SOS)."""
    b = bytes(data)
    _need(b[:2] == b"\xff\xd8", HEADER, "no SOI")
    p, tables, sof, ri = 2, {}, None, 0
    while True:
        _need(p < len(b) and b[p] == 0xFF, HEADER, "no marker at byte %d" % p)
        while p < len(b) and b[p] == 0xFF:                  # B.1.1.2: fill bytes before any marker
            p += 1
        _need(p < len(b), HEADER, "data ends in fill bytes")
        m = b[p]
        p += 1
        if m == 0x01:                                       # TEM: a marker without a length
            continue
        _need(m not in (0xD8, 0xD9) and not 0xD0 <= m <= 0xD7, HEADER, "marker 0x%02X before SOS" % m)
        _need(p + 2 <= len(b), HEADER, "truncated marker segment")
        L = struct.unpack_from(">H", b, p)[0]
        _need(L >= 2 and p + L <= len(b), HEADER, "marker segment length %d" % L)
        body = b[p + 2:p + L]
        if m == 0xC3:                                       # SOF3 (B.2.2)
            _need(sof is None and len(body) >= 6, HEADER, "SOF3")
            P, Y, X, Nf = struct.unpack_from(">BHHB", body)
            _need(Nf == 1 and len(body) == 6 + 3 * Nf and 2 <= P <= 16, HEADER, "SOF3: P %d, Nf %d" % (P, Nf))
            sof = dict(P=P, rows=Y, cols=X, comp=body[6])
        elif 0xC0 <= m <= 0xCF and m not in (0xC4, 0xC8, 0xCC):
            raise DecodeError(HEADER, "frame type SOF%d" % (m - 0xC0))
        elif m == 0xC4:                                     # DHT (B.2.4.2), any number of tables
            q = 0
            while q < len(body):
                _need(q + 17 <= len(body), HEADER, "DHT: truncated BITS")
                tc, th = body[q] >> 4, body[q] & 15
                bits = list(body[q + 1:q + 17])
                n = sum(bits)
                _need(tc == 0 and th <= 3 and q + 17 + n <= len(body), HEADER, "DHT: Tc %d Th %d" % (tc, th))
                tables[th] = HuffTable(bits, body[q + 17:q + 17 + n])
                q += 17 + n
        elif m == 0xDD:                                     # DRI (B.2.4.4)
            _need(len(body) == 2, HEADER, "DRI length")
            ri = struct.unpack(">H", body)[0]
        elif m == 0xDA:                                     # SOS (B.2.3)
            _need(sof is not None and len(body) == 6 and body[0] == 1, HEADER, "SOS")
            cs, td, ss, se, ah, al = body[1], body[2] >> 4, body[3], body[4], body[5] >> 4, body[5] & 15
            _need(cs == sof["comp"], HEADER, "SOS selects component %d" % cs)
            _need(td in tables, HEADER, "SOS selects undefined table %d" % td)
            _need(1 <= ss <= 7 and se == 0 and ah == 0 and al < sof["P"], HEADER, "SOS: Ss %d Se %d Ah %d Al %d" % (ss, se, ah, al))
            _need(ri == 0 or ri % sof["cols"] == 0, HEADER, "restart interval %d is not whole rows" % ri)
            return dict(sof, table=tables[td], pred=ss, pt=al, ri=ri, entropy=b[p + L:])
        else:
            _need(0xE0 <= m <= 0xEF or m in (0xFE, 0xDB), HEADER, "marker 0x%02X" % m)
        p += L


def split_entropy(ent):
    """Entropy-coded data after SOS -> list of restart intervals' bytes (B.1.1.5: stuffed zero bytes removed, fill
    bytes before markers dropped, RSTm in sequence), ending at EOI; one pad byte may follow EOI."""
    segs, cur, i, n = [], bytearray(), 0, len(ent)
    while True:
        _need(i < n, HEADER, "no EOI")
        c = ent[i]
        if c != 0xFF:
            cur.append(c)
            i += 1
            continue
        j = i + 1
        while j < n and ent[j] == 0xFF:
            j += 1
        _need(j < n, HEADER, "no EOI")
        m = ent[j]
        if m == 0x00 and j == i + 1:
            cur.append(0xFF)
            i = j + 1
        elif 0xD0 <= m <= 0xD7:
            _need(m == 0xD0 + len(segs) % 8, DATA, "RST%d out of sequence" % (m - 0xD0))
            segs.append(bytes(cur))
            cur = bytearray()
            i = j + 1
        elif m == 0xD9:
            _need(n - (j + 1) <= 1, HEADER, "data after EOI")
            segs.append(bytes(cur))
            return segs
        else:
            raise DecodeError(DATA, "marker 0x%02X in entropy-coded data" % m)


def _predict(x, r, c, r0, W, pred, init):                  # H.1.2.1, restart intervals starting afresh at row r0
    if r == r0:
        return init if c == 0 else x[r * W + c - 1]
    if c == 0:
        return x[(r - 1) * W]
    Ra, Rb, Rc = x[r * W + c - 1], x[(r - 1) * W + c], x[(r - 1) * W + c - 1]
    if pred == 1:
        return Ra
    if pred == 2:
        return Rb
    if pred == 3:
        return Rc
    if pred == 4:
        return Ra + Rb - Rc
    if pred == 5:
        return Ra + ((Rb - Rc) >> 1)
    if pred == 6:
        return Rb + ((Ra - Rc) >> 1)
    return (Ra + Rb) >> 1


def jpeg_lossless_decode(data):
    """A JPEG Lossless (SOF3, one component) stream -> (rows, cols) uint16: the P-bit samples, point transform undone.
    Codewords after an interval's last sample are ignored; an interval short of samples raises (status -62)."""
    h = parse_jpeg(data)
    H, W, P, pt, pred, t = h["rows"], h["cols"], h["P"], h["pt"], h["pred"], h["table"]
    step = h["ri"] // W if h["ri"] else H
    segs = split_entropy(h["entropy"])
    _need(len(segs) == -(-H // step), LENGTH, "%d restart intervals, %d expected" % (len(segs), -(-H // step)))
    init = 1 << (P - pt - 1)
    x = [0] * (H * W)
    for k, seg in enumerate(segs):
        br = _Bits(seg)
        r0 = k * step
        for r in range(r0, min(r0 + step, H)):
            for c in range(W):
                d = _difference(br, t)
                x[r * W + c] = (_predict(x, r, c, r0, W, pred, init) + d) & 0xFFFF   # modulo 2^16 (H.1.2.1)
    out = np.array(x, np.uint32).reshape(H, W)
    return ((out << pt) & 0xFFFF).astype(np.uint16)


# --------------------------------------------------------------------------------------------------------------
# RLE Lossless
# --------------------------------------------------------------------------------------------------------------
def packbits_decode(seg, n):
    """One PackBits segment -> its first n bytes (PS3.5 G.3.2); bytes after the n-th are ignored."""
    seg = bytes(seg)
    out, i = bytearray(), 0
    while len(out) < n:
        _need(i < len(seg), LENGTH, "segment ends after %d of %d bytes" % (len(out), n))
        h = seg[i] - 256 if seg[i] >= 128 else seg[i]
        i += 1
        if h >= 0:                                          # literal run: the next h + 1 bytes
            _need(i + h + 1 <= len(seg), LENGTH, "literal run past the segment end")
            out += seg[i:i + h + 1]
            i += h + 1
        elif h >= -127:                                     # replicate run: the next byte -h + 1 times
            _need(i < len(seg), LENGTH, "replicate run past the segment end")
            out += bytes([seg[i]]) * (1 - h)
            i += 1
        # h == -128: no operation
        _need(len(out) <= n, LENGTH, "runs past %d bytes" % n)
    return bytes(out)


def rle_decode(frame, rows, cols):
    """A 16-bit single-sample RLE Lossless frame -> (rows, cols) uint16 (segment 1 = most significant bytes)."""
    frame = bytes(frame)
    _need(len(frame) >= 64, HEADER, "RLE header")
    hdr = struct.unpack_from("<16I", frame)
    _need(hdr[0] == 2, HEADER, "%d RLE segments, 2 expected" % hdr[0])
    o0, o1 = hdr[1], hdr[2]
    _need(o0 == 64 and o0 < o1 < len(frame), HEADER, "RLE segment offsets %d, %d" % (o0, o1))
    n = rows * cols
    hi = np.frombuffer(packbits_decode(frame[o0:o1], n), np.uint8).astype(np.uint16)
    lo = np.frombuffer(packbits_decode(frame[o1:], n), np.uint8).astype(np.uint16)
    return ((hi << 8) | lo).reshape(rows, cols)
