// lm_decode_frames (include/lungmask_b200.h): JPEG Lossless (ITU-T T.81 process 14, SOF3) and DICOM RLE Lossless
// (PS3.5 Annex G) frames decoded on the GPU.  The host side of the call parses the JPEG marker segments and the RLE
// header; every byte of entropy-coded or run-length data is handled by the kernels below.
//
// JPEG:   lm_jpeg_classify   one thread per entropy byte: keep / drop (0xFF00 stuffing, fill bytes) / RSTm, scanned
//         lm_jpeg_compact    scatter of the kept bytes, restart-segment starts, RSTm sequence check
//         lm_jpeg_sync       self-synchronising chunk decode (Weissenberger & Schmidt, ICPP 2018): every CHUNK_BITS chunk
//                            decodes speculatively; repeated until each chunk starts where its predecessor left off
//         lm_jpeg_emit       after a scan of the per-chunk codeword counts: writes the differences
//         lm_jpeg_check      per restart segment: at least the expected samples decoded (codewords beyond them are
//                            ignored, as libjpeg-turbo does)
//         lm_undiff_rows / lm_undiff_cols / lm_undiff_diag / lm_undiff_wave   reconstruction (modular scans for the
//                            linear predictors 1-4, a row-pipelined wavefront for 5-7)
//         lm_jpeg_finish     point transform and sign extension
// RLE:    lm_rle_runs        one thread per segment walks the PackBits control bytes and records the runs
//         lm_rle_expand      the runs expanded in parallel into the byte planes
//
// Every device read of input data is bounded by its frame's [offset, offset + length); malformed data sets the frame's
// status and never traps.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "../../include/lungmask_b200.h"

namespace lm_impl {
int fail(int code, const char* fmt, ...);
}
using lm_impl::fail;

namespace lm_decode {

constexpr int LUT_BITS = 10;                   // first-level Huffman lookup: codes up to 10 bits in one shared-memory read
constexpr uint32_t CHUNK_BITS = 1024;          // self-synchronisation chunk
constexpr uint32_t NO_EXIT = 0xFFFFFFFFu;      // a speculative decode met an undefined code
constexpr int MAX_SYNC_ROUNDS_EXTRA = 2;

struct HuffDev {                               // built on the host from DHT BITS / HUFFVAL (T.81 Annex C)
  uint16_t lut[1 << LUT_BITS];                 // (length << 8) | symbol, 0 = longer than LUT_BITS or undefined
  int32_t maxcode[18];                         // largest code of each length, -1 if none
  int32_t valoff[17];                          // index into val = valoff[l] + code
  uint8_t val[256];
};
static_assert(sizeof(HuffDev) % 4 == 0, "HuffDev is copied as 32-bit words");

struct JFrame {
  uint64_t ent_begin, ent_end;                 // entropy-coded bytes in the input buffer
  uint64_t e_off;                              // offset in the flat index space of all entropy bytes
  uint64_t out_base;                           // first sample in the output
  uint32_t rows, cols, ivl_rows;               // ivl_rows = rows per restart interval (rows without DRI)
  int32_t P, Pt, pred, is_signed, idx;         // idx = position in the caller's frame list
  uint32_t chunk_begin, chunk_end;
};

struct JSeg {                                  // one restart interval
  uint32_t byte_begin, byte_end;               // in the compacted entropy buffer
  uint32_t first_chunk, n_chunks;
  uint64_t sample_begin;                       // in the output
  uint32_t n_samples, frame;                   // frame = JFrame index
};

struct RSeg {                                  // one RLE byte plane
  uint64_t begin, end;                         // in the input buffer
  uint64_t out_base;
  uint32_t n_samples, plane, run_base, run_cap;
  int32_t idx;
};

struct Run {
  uint32_t out, src, len;                      // src: literal bytes' offset in the segment, or the repeated value
};

// ---------------------------------------------------------------------------------------------------------------
// scan (exclusive, in place, uint64)
// ---------------------------------------------------------------------------------------------------------------
constexpr int SCAN_THREADS = 256, SCAN_ITEMS = 4, SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__global__ void __launch_bounds__(SCAN_THREADS) lm_scan_tiles(uint64_t* d, size_t n, uint64_t* tile_sums) {
  __shared__ uint64_t s[SCAN_THREADS];
  const size_t base = (size_t)blockIdx.x * SCAN_TILE + (size_t)threadIdx.x * SCAN_ITEMS;
  uint64_t v[SCAN_ITEMS], t = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    v[k] = base + k < n ? d[base + k] : 0;
    const uint64_t x = v[k];
    v[k] = t;
    t += x;
  }
  s[threadIdx.x] = t;
  __syncthreads();
  for (int off = 1; off < SCAN_THREADS; off <<= 1) {
    const uint64_t add = threadIdx.x >= off ? s[threadIdx.x - off] : 0;
    __syncthreads();
    s[threadIdx.x] += add;
    __syncthreads();
  }
  const uint64_t excl = s[threadIdx.x] - t;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k)
    if (base + k < n) d[base + k] = v[k] + excl;
  if (threadIdx.x == SCAN_THREADS - 1) tile_sums[blockIdx.x] = s[threadIdx.x];
}

__global__ void lm_scan_add(uint64_t* d, size_t n, const uint64_t* tile_offsets) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) d[i] += tile_offsets[i / SCAN_TILE];
}

// ---------------------------------------------------------------------------------------------------------------
// JPEG: entropy bytes -> compacted bit stream per restart segment
// ---------------------------------------------------------------------------------------------------------------
// Scan value = kept bytes (low 32 bits) | RST markers (high 32 bits).  Every entropy byte adds to at most one field and
// a call holds fewer than 2^32 - 1 entropy bytes (checked on the host), so neither field can carry into the other.
constexpr int RST_SHIFT = 32;
constexpr uint64_t RST_ONE = 1ull << RST_SHIFT, KEPT_MASK = RST_ONE - 1;

__device__ __forceinline__ int frame_of(const JFrame* fr, int n, uint64_t t) {   // last frame with e_off <= t
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (fr[mid].e_off <= t) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// 1 = data byte, 0 = dropped (stuffing 0x00, fill 0xFF, 0xFF of an RST), 2 = RSTm code byte, -1 = not allowed here
__device__ __forceinline__ int classify(const uint8_t* d, uint64_t pos, uint64_t begin, uint64_t end) {
  const uint32_t b = d[pos];
  const uint32_t prev = pos > begin ? d[pos - 1] : 0u;
  if (b != 0xFF) {
    if (prev != 0xFF) return 1;
    if (b == 0x00) return 0;
    return (b >= 0xD0 && b <= 0xD7) ? 2 : -1;
  }
  const uint32_t next = pos + 1 < end ? d[pos + 1] : 0x100u;
  if (next == 0x00) return 1;
  if (next == 0xFF || (next >= 0xD0 && next <= 0xD7)) return 0;
  return -1;
}

__global__ void lm_jpeg_classify(const uint8_t* data, const JFrame* fr, int nf, uint64_t total, uint64_t* v,
                                 int32_t* status) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t > total) return;
  if (t == total) { v[t] = 0; return; }
  const int f = frame_of(fr, nf, t);
  const JFrame F = fr[f];
  const int c = classify(data, F.ent_begin + (t - F.e_off), F.ent_begin, F.ent_end);
  if (c < 0) status[F.idx] = LM_ERR_DECODE_DATA;
  v[t] = c == 1 ? 1ull : c == 2 ? RST_ONE : 0ull;
}

__global__ void lm_jpeg_frame_offsets(const JFrame* fr, int nf, const uint64_t* v, uint64_t total, uint64_t* out) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f <= nf) out[f] = v[f < nf ? fr[f].e_off : total];
}

__global__ void lm_jpeg_compact(const uint8_t* data, const JFrame* fr, int nf, uint64_t total, const uint64_t* v,
                                const uint64_t* frame_v, uint8_t* comp, uint32_t* seg_begin, uint64_t n_seg_begin,
                                int32_t* status) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int f = frame_of(fr, nf, t);
  const JFrame F = fr[f];
  const uint64_t pos = F.ent_begin + (t - F.e_off);
  const int c = classify(data, pos, F.ent_begin, F.ent_end);
  const uint64_t s = v[t];
  if (c == 1) {
    comp[s & KEPT_MASK] = data[pos];
  } else if (c == 2) {
    const uint64_t k = s >> RST_SHIFT;                      // RST markers before this one, all frames
    const uint64_t local = k - (frame_v[f] >> RST_SHIFT);
    if (data[pos] != 0xD0 + (local & 7)) status[F.idx] = LM_ERR_DECODE_DATA;
    if (k + f + 1 < n_seg_begin)                            // always true; the bound is kept next to the write
      seg_begin[k + f + 1] = (uint32_t)(s & KEPT_MASK);     // the next data byte starts segment local + 1 of frame f
  }
}

// ---------------------------------------------------------------------------------------------------------------
// JPEG: Huffman decode
// ---------------------------------------------------------------------------------------------------------------
struct BitReader {                             // MSB-first; bits past the segment end read as 1 (JPEG pad bits)
  const uint8_t* p;
  uint32_t nbytes, nbits, base;
  uint64_t win;
  __device__ void load(uint32_t pos) {
    base = pos & ~7u;
    const uint32_t b = base >> 3;
    win = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) win = (win << 8) | (b + k < nbytes ? p[b + k] : 0xFFu);
  }
  __device__ uint32_t peek32(uint32_t pos) {
    if (pos < base || pos + 32 > base + 64) load(pos);
    return (uint32_t)((win << (pos - base)) >> 32);
  }
};

// Decodes the codeword (Huffman code + SSSS extra bits) at pos.  > 0: its length in bits, diff = the difference;
// 0: the codeword does not fit before the segment end (the end of the segment's data); -1: undefined code.
__device__ __forceinline__ int decode_one(BitReader& br, uint32_t pos, const HuffDev& h, int32_t& diff) {
  const uint32_t w = br.peek32(pos);
  int len = 0, sym = 0;
  const uint32_t e = h.lut[w >> (32 - LUT_BITS)];
  if (e) {
    len = (int)(e >> 8);
    sym = (int)(e & 0xFF);
  } else {
    for (int l = LUT_BITS + 1; l <= 16; ++l) {
      const int32_t code = (int32_t)(w >> (32 - l));
      if (code <= h.maxcode[l]) {
        len = l;
        sym = h.val[h.valoff[l] + code];
        break;
      }
    }
    if (!len) return pos + 16 > br.nbits ? 0 : -1;
  }
  if (sym > 16) return pos + (uint32_t)len > br.nbits ? 0 : -1;
  const int extra = sym == 16 ? 0 : sym;
  if (pos + (uint32_t)(len + extra) > br.nbits) return 0;
  if (sym == 0) {
    diff = 0;
  } else if (sym == 16) {
    diff = 32768;                                           // H.1.2.2: category 16 has no additional bits
  } else {
    const int32_t x = (int32_t)((w << len) >> (32 - sym));
    diff = x < (1 << (sym - 1)) ? x - ((1 << sym) - 1) : x;
  }
  return len + extra;
}

__device__ void load_table(HuffDev& dst, const HuffDev* src) {
  const uint32_t* s = reinterpret_cast<const uint32_t*>(src);
  uint32_t* d = reinterpret_cast<uint32_t*>(&dst);
  for (int i = threadIdx.x; i < (int)(sizeof(HuffDev) / 4); i += blockDim.x) d[i] = s[i];
  __syncthreads();
}

constexpr int DEC_THREADS = 128;

// One round of the chunk synchronisation.  Round 0 decodes every chunk from its first bit; later rounds re-decode a
// chunk only when its predecessor now exits at another bit than where the chunk last started.
__global__ void __launch_bounds__(DEC_THREADS) lm_jpeg_sync(const uint8_t* comp, const JFrame* fr, const JSeg* segs,
                                                            const uint32_t* chunk_seg, const HuffDev* tables,
                                                            uint32_t* start, uint32_t* exitp, uint64_t* count,
                                                            int first_round, int* changed) {
  __shared__ HuffDev h;
  const JFrame F = fr[blockIdx.y];
  load_table(h, tables + blockIdx.y);
  const uint32_t c = F.chunk_begin + blockIdx.x * DEC_THREADS + threadIdx.x;
  if (c >= F.chunk_end) return;
  const JSeg S = segs[chunk_seg[c]];
  const uint32_t cbeg = (c - S.first_chunk) * CHUNK_BITS;
  uint32_t s;
  if (first_round) {
    s = cbeg;
  } else {
    if (c == S.first_chunk) return;
    s = *(volatile const uint32_t*)(exitp + c - 1);
    if (s == NO_EXIT || s == start[c]) return;
  }
  BitReader br{comp + S.byte_begin, S.byte_end - S.byte_begin, (S.byte_end - S.byte_begin) * 8u, 0xFFFFFFF0u, 0};
  const uint32_t cend = min(cbeg + CHUNK_BITS, br.nbits);
  uint32_t pos = s, n = 0;
  while (pos < cend) {
    int32_t diff;
    const int l = decode_one(br, pos, h, diff);
    if (l < 0) { pos = NO_EXIT; break; }
    if (l == 0) break;
    pos += (uint32_t)l;
    ++n;
  }
  start[c] = s;
  count[c] = n;
  *(volatile uint32_t*)(exitp + c) = pos;
  if (!first_round) *changed = 1;
}

// Writes the differences of every codeword (count scanned: count[c] = codewords before chunk c, all segments).  The
// first sample of each restart interval carries the initial prediction 2^(P-Pt-1).
__global__ void __launch_bounds__(DEC_THREADS) lm_jpeg_emit(const uint8_t* comp, const JFrame* fr, const JSeg* segs,
                                                            const uint32_t* chunk_seg, const HuffDev* tables,
                                                            const uint32_t* start, const uint64_t* count, uint16_t* out,
                                                            int32_t* status) {
  __shared__ HuffDev h;
  const JFrame F = fr[blockIdx.y];
  load_table(h, tables + blockIdx.y);
  const uint32_t c = F.chunk_begin + blockIdx.x * DEC_THREADS + threadIdx.x;
  if (c >= F.chunk_end) return;
  const JSeg S = segs[chunk_seg[c]];
  const uint32_t cbeg = (c - S.first_chunk) * CHUNK_BITS;
  BitReader br{comp + S.byte_begin, S.byte_end - S.byte_begin, (S.byte_end - S.byte_begin) * 8u, 0xFFFFFFF0u, 0};
  const uint32_t cend = min(cbeg + CHUNK_BITS, br.nbits);
  uint64_t li = count[c] - count[S.first_chunk];
  const int32_t init = 1 << (F.P - F.Pt - 1);
  uint16_t* o = out + S.sample_begin;
  for (uint32_t pos = start[c]; pos < cend;) {
    int32_t diff;
    const int l = decode_one(br, pos, h, diff);
    if (l < 0) { status[F.idx] = LM_ERR_DECODE_DATA; return; }
    if (l == 0) return;
    if (li < S.n_samples) o[li] = (uint16_t)(diff + (li == 0 ? init : 0));
    ++li;
    pos += (uint32_t)l;
  }
}

__global__ void lm_jpeg_check(const JFrame* fr, const JSeg* segs, uint32_t nseg, const uint64_t* count, int32_t* status) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nseg) return;
  const JSeg S = segs[s];
  if (count[S.first_chunk + S.n_chunks] - count[S.first_chunk] < S.n_samples) status[fr[S.frame].idx] = LM_ERR_DECODE_LENGTH;
}

// ---------------------------------------------------------------------------------------------------------------
// JPEG: reconstruction.  x = difference + prediction, modulo 2^16; restart intervals start afresh (their first
// sample holds the initial prediction already), their first row predicts from Ra, their first column from Rb.
// ---------------------------------------------------------------------------------------------------------------
// Prefix sums along rows (one warp per row): all rows, or only the first row of each restart interval.
__global__ void lm_undiff_rows(const JFrame* fr, const uint32_t* list, uint16_t* out, int first_rows_only) {
  const JFrame F = fr[list[blockIdx.y]];
  const uint32_t warp = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32, lane = threadIdx.x & 31;
  const uint32_t r = first_rows_only ? warp * F.ivl_rows : warp;
  if (r >= F.rows) return;
  uint16_t* row = out + F.out_base + (uint64_t)r * F.cols;
  uint32_t carry = 0;
  for (uint32_t c0 = 0; c0 < F.cols; c0 += 32) {
    const uint32_t c = c0 + lane;
    uint32_t v = c < F.cols ? row[c] : 0u;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, v, off);
      if (lane >= (uint32_t)off) v += u;
    }
    v += carry;
    if (c < F.cols) row[c] = (uint16_t)v;
    carry = __shfl_sync(0xFFFFFFFFu, v, 31);
  }
}

// Prefix sums down the columns of each restart interval (one thread per interval and column): all columns, or only
// the first.
__global__ void lm_undiff_cols(const JFrame* fr, const uint32_t* list, uint16_t* out, int first_col_only) {
  const JFrame F = fr[list[blockIdx.y]];
  const uint32_t ncol = first_col_only ? 1u : F.cols;
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t ivl = t / ncol, c = t % ncol;
  const uint32_t r0 = ivl * F.ivl_rows;
  if (r0 >= F.rows) return;
  const uint32_t r1 = min(r0 + F.ivl_rows, F.rows);
  uint16_t* p = out + F.out_base + (uint64_t)r0 * F.cols + c;
  uint32_t acc = 0;
  for (uint32_t r = r0; r < r1; ++r, p += F.cols) {
    acc += *p;
    *p = (uint16_t)acc;
  }
}

// Predictor 3 (Rc): after the interval's first row and first column, sums along the diagonals.
__global__ void lm_undiff_diag(const JFrame* fr, const uint32_t* list, uint16_t* out) {
  const JFrame F = fr[list[blockIdx.y]];
  const uint32_t nd = F.cols + F.ivl_rows - 1;
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t ivl = t / nd, j = t % nd;
  const uint32_t r0 = ivl * F.ivl_rows;
  if (r0 >= F.rows) return;
  const uint32_t r1 = min(r0 + F.ivl_rows, F.rows);
  uint32_t r = j < F.cols ? r0 : r0 + (j - F.cols + 1), c = j < F.cols ? j : 0;
  if (r >= r1) return;
  uint16_t* base = out + F.out_base;
  uint32_t acc = base[(uint64_t)r * F.cols + c];
  for (++r, ++c; r < r1 && c < F.cols; ++r, ++c) {
    uint16_t* p = base + (uint64_t)r * F.cols + c;
    acc += *p;
    *p = (uint16_t)acc;
  }
}

// Predictors 5-7 (non-linear): one block per restart interval, one thread per row, the rows offset by one column
// each (a wavefront), bands of blockDim rows one after the other.
__global__ void lm_undiff_wave(const JFrame* fr, const uint32_t* list, uint16_t* out) {
  const JFrame F = fr[list[blockIdx.y]];
  const uint32_t r0 = blockIdx.x * F.ivl_rows;
  if (r0 >= F.rows) return;
  const uint32_t r1 = min(r0 + F.ivl_rows, F.rows);
  uint16_t* base = out + F.out_base;
  const uint32_t W = F.cols;
  for (uint32_t band = r0; band < r1; band += blockDim.x) {
    const uint32_t nb = min((uint32_t)blockDim.x, r1 - band);
    const uint32_t r = band + threadIdx.x;
    for (uint32_t step = 0; step < W + nb - 1; ++step) {
      const int32_t c = (int32_t)step - (int32_t)threadIdx.x;
      if (threadIdx.x < nb && c >= 0 && c < (int32_t)W) {
        uint16_t* p = base + (uint64_t)r * W + c;
        int32_t pred;
        if (r == r0) {
          pred = c == 0 ? 0 : p[-1];
        } else if (c == 0) {
          pred = p[-(int64_t)W];
        } else {
          const int32_t Ra = p[-1], Rb = p[-(int64_t)W], Rc = p[-(int64_t)W - 1];
          switch (F.pred) {
            case 1: pred = Ra; break;
            case 2: pred = Rb; break;
            case 3: pred = Rc; break;
            case 4: pred = Ra + Rb - Rc; break;
            case 5: pred = Ra + ((Rb - Rc) >> 1); break;
            case 6: pred = Rb + ((Ra - Rc) >> 1); break;
            default: pred = (Ra + Rb) >> 1; break;
          }
        }
        *p = (uint16_t)(*p + pred);
      }
      __syncthreads();
    }
  }
}

__global__ void lm_jpeg_finish(const JFrame* fr, const uint32_t* list, uint16_t* out) {
  const JFrame F = fr[list[blockIdx.y]];
  const uint64_t n = (uint64_t)F.rows * F.cols;
  uint16_t* o = out + F.out_base;
  const uint32_t sign = F.is_signed && F.P < 16 ? 1u << (F.P - 1) : 0u;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t v = ((uint32_t)o[i] << F.Pt) & 0xFFFFu;
    if (v & sign) v |= 0xFFFFu & ~((sign << 1) - 1);
    o[i] = (uint16_t)v;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// RLE
// ---------------------------------------------------------------------------------------------------------------
__global__ void lm_rle_runs(const uint8_t* data, const RSeg* segs, int nseg, Run* runs, uint32_t* n_runs, int32_t* status) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nseg) return;
  const RSeg S = segs[s];
  Run* r = runs + S.run_base;
  uint64_t pos = S.begin;
  uint32_t produced = 0, k = 0;
  int err = 0;
  while (produced < S.n_samples) {
    if (pos >= S.end) { err = LM_ERR_DECODE_LENGTH; break; }
    const int n = (int8_t)data[pos++];
    if (n == -128) continue;
    const uint32_t len = n >= 0 ? (uint32_t)n + 1 : (uint32_t)(1 - n);
    const uint64_t need = n >= 0 ? len : 1;
    if (pos + need > S.end || produced + len > S.n_samples || k >= S.run_cap) { err = LM_ERR_DECODE_LENGTH; break; }
    r[k++] = Run{produced, n >= 0 ? (uint32_t)(pos - S.begin) : 0x80000000u | data[pos], len};
    pos += need;
    produced += len;
  }
  n_runs[s] = err ? 0 : k;
  if (err) status[S.idx] = err;
}

__global__ void lm_rle_expand(const uint8_t* data, const RSeg* segs, const Run* runs, const uint32_t* n_runs, uint16_t* out) {
  const RSeg S = segs[blockIdx.x];
  const uint32_t nr = n_runs[blockIdx.x];
  const uint8_t* src = data + S.begin;
  uint8_t* dst = reinterpret_cast<uint8_t*>(out + S.out_base) + (S.plane == 0 ? 1 : 0);   // plane 0 = most significant bytes
  for (uint32_t i = threadIdx.x; i < nr; i += blockDim.x) {
    const Run R = runs[S.run_base + i];
    uint8_t* d = dst + 2ull * R.out;
    if (R.src & 0x80000000u) {
      const uint8_t v = (uint8_t)R.src;
      for (uint32_t k = 0; k < R.len; ++k) d[2 * k] = v;
    } else {
      for (uint32_t k = 0; k < R.len; ++k) d[2 * k] = src[R.src + k];
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
struct Scratch {                                // device allocations and the stream of one call, released on every path
  std::vector<void*> ptrs;
  cudaStream_t st = nullptr;
  ~Scratch() {
    if (st) cudaStreamSynchronize(st);
    for (void* p : ptrs) cudaFree(p);
    if (st) cudaStreamDestroy(st);
  }
  template <typename T>
  cudaError_t alloc(T** p, size_t n) {
    *p = nullptr;
    cudaError_t e = cudaMalloc((void**)p, std::max<size_t>(n, 1) * sizeof(T));
    if (e == cudaSuccess) ptrs.push_back(*p);
    return e;
  }
};

#define CU(x)                                                                                                        \
  do {                                                                                                               \
    cudaError_t e_ = (x);                                                                                            \
    if (e_ != cudaSuccess) return fail((int)e_, "%s failed: %s (%s:%d)", #x, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

static int scan_exclusive(Scratch& sc, uint64_t* d, size_t n) {
  if (n == 0) return 0;
  const size_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  uint64_t* sums;
  CU(sc.alloc(&sums, tiles));
  lm_scan_tiles<<<(unsigned)tiles, SCAN_THREADS, 0, sc.st>>>(d, n, sums);
  CU(cudaGetLastError());
  if (tiles > 1) {
    if (int rc = scan_exclusive(sc, sums, tiles)) return rc;
    lm_scan_add<<<(unsigned)((n + 255) / 256), 256, 0, sc.st>>>(d, n, sums);
    CU(cudaGetLastError());
  }
  return 0;
}

struct JHost {
  JFrame f;
  HuffDev table;
};

static uint32_t be16(const uint8_t* p) { return (uint32_t)p[0] << 8 | p[1]; }
static uint32_t le32(const uint8_t* p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }

static bool build_table(const uint8_t bits[17], const uint8_t* vals, int nvals, HuffDev& h) {
  memset(&h, 0, sizeof(h));
  memcpy(h.val, vals, nvals);
  uint32_t code = 0;
  int k = 0;
  for (int l = 1; l <= 16; ++l) {
    h.valoff[l] = k - (int32_t)code;
    for (int i = 0; i < bits[l]; ++i, ++k, ++code) {
      if (l <= LUT_BITS) {
        const uint32_t lo = code << (LUT_BITS - l), hi = (code + 1) << (LUT_BITS - l);
        for (uint32_t j = lo; j < hi && j < (1u << LUT_BITS); ++j) h.lut[j] = (uint16_t)(l << 8 | vals[k]);
      }
    }
    h.maxcode[l] = bits[l] ? (int32_t)code - 1 : -1;
    if (code > (1u << l)) return false;                     // more codes than the code space of this length
    code <<= 1;
  }
  h.maxcode[17] = 0x7FFFFFFF;
  return true;
}

// Parses SOI .. SOS and locates EOI; fills the frame's prediction parameters, entropy range and Huffman table.
static int parse_jpeg(const uint8_t* d, uint64_t off, uint64_t len, const lm_frame& fm, JHost& j) {
  const uint64_t end = off + len;
  if (len < 4 || d[off] != 0xFF || d[off + 1] != 0xD8) return LM_ERR_DECODE_HEADER;
  uint64_t p = off + 2;
  bool have_sof = false;
  int P = 0, comp_id = -1, ri = 0;
  uint32_t Y = 0, X = 0;
  bool have_table[4] = {false, false, false, false};
  static thread_local HuffDev tables[4];
  for (;;) {
    if (p >= end || d[p] != 0xFF) return LM_ERR_DECODE_HEADER;
    while (p < end && d[p] == 0xFF) ++p;                    // fill bytes
    if (p >= end) return LM_ERR_DECODE_HEADER;
    const uint32_t m = d[p++];
    if (m == 0x01) continue;                                // TEM: no length
    if (m == 0xD8 || m == 0xD9 || (m >= 0xD0 && m <= 0xD7) || p + 2 > end) return LM_ERR_DECODE_HEADER;
    const uint32_t L = be16(d + p);
    if (L < 2 || p + L > end) return LM_ERR_DECODE_HEADER;
    const uint8_t* s = d + p + 2;
    const uint32_t n = L - 2;
    if (m == 0xC3) {                                        // SOF3: lossless, Huffman
      if (have_sof || n < 6) return LM_ERR_DECODE_HEADER;
      P = s[0];
      Y = be16(s + 1);
      X = be16(s + 3);
      const int Nf = s[5];
      if (Nf != 1 || n != 6u + 3u * Nf || P < 2 || P > 16) return LM_ERR_DECODE_HEADER;
      if (Y != (uint32_t)fm.rows || X != (uint32_t)fm.cols) return LM_ERR_DECODE_HEADER;
      comp_id = s[6];
      have_sof = true;
    } else if ((m >= 0xC0 && m <= 0xCF) && m != 0xC4 && m != 0xC8 && m != 0xCC) {
      return LM_ERR_DECODE_HEADER;                          // any other frame type: DCT or arithmetic coding
    } else if (m == 0xC4) {                                 // DHT
      uint32_t q = 0;
      while (q < n) {
        if (q + 17 > n) return LM_ERR_DECODE_HEADER;
        const int tc = s[q] >> 4, th = s[q] & 15;
        uint8_t bits[17] = {0};
        int count = 0;
        for (int l = 1; l <= 16; ++l) count += bits[l] = s[q + l];
        q += 17;
        if (tc != 0 || th > 3 || count > 256 || q + count > n) return LM_ERR_DECODE_HEADER;
        if (!build_table(bits, s + q, count, tables[th])) return LM_ERR_DECODE_HEADER;
        have_table[th] = true;
        q += count;
      }
    } else if (m == 0xDD) {                                 // DRI
      if (n != 2) return LM_ERR_DECODE_HEADER;
      ri = (int)be16(s);
    } else if (m == 0xDA) {                                 // SOS
      if (!have_sof || n < 1 || s[0] != 1 || n != 6) return LM_ERR_DECODE_HEADER;
      const int cs = s[1], td = s[2] >> 4, ss = s[3], se = s[4], ah = s[5] >> 4, al = s[5] & 15;
      if (cs != comp_id || td > 3 || !have_table[td] || ss < 1 || ss > 7 || se != 0 || ah != 0 || al >= P)
        return LM_ERR_DECODE_HEADER;
      if (ri && ri % X != 0) return LM_ERR_DECODE_HEADER;   // restart intervals of whole rows only
      j.table = tables[td];
      j.f.P = P;
      j.f.Pt = al;
      j.f.pred = ss;
      j.f.rows = Y;
      j.f.cols = X;
      j.f.ivl_rows = ri ? (uint32_t)(ri / X) : Y;
      p += L;
      break;
    } else if (!((m >= 0xE0 && m <= 0xEF) || m == 0xFE || m == 0xDB)) {
      return LM_ERR_DECODE_HEADER;                          // DNL, DHP, EXP, arithmetic conditioning, ...
    }
    p += L;
  }
  // EOI ends the frame; the DICOM fragment may add one pad byte after it
  uint64_t e = end;
  if (e - p >= 3 && d[e - 1] != 0xD9) --e;
  if (e - p < 2 || d[e - 2] != 0xFF || d[e - 1] != 0xD9) return LM_ERR_DECODE_HEADER;
  e -= 2;
  while (e > p && d[e - 1] == 0xFF) --e;                    // fill bytes before EOI
  j.f.ent_begin = p;
  j.f.ent_end = e;
  return 0;
}

static int parse_rle(const uint8_t* d, uint64_t off, uint64_t len, uint64_t& b0, uint64_t& b1) {
  if (len < 64) return LM_ERR_DECODE_HEADER;
  const uint8_t* h = d + off;
  if (le32(h) != 2) return LM_ERR_DECODE_HEADER;            // 16-bit single-sample frames: exactly 2 byte planes
  const uint64_t o0 = le32(h + 4), o1 = le32(h + 8);
  if (o0 != 64 || o1 <= o0 || o1 >= len) return LM_ERR_DECODE_HEADER;
  b0 = o0;
  b1 = o1;
  return 0;
}

static int decode(const uint8_t* data, size_t n_bytes, const lm_frame* frames, int nf, uint16_t* out, int32_t* status) {
  std::vector<int32_t> hstat(nf, 0);
  std::vector<uint64_t> out_base(nf + 1, 0);
  for (int i = 0; i < nf; ++i) {
    const lm_frame& fm = frames[i];
    if (fm.rows <= 0 || fm.cols <= 0 || fm.rows > 65535 || fm.cols > 65535) return fail(-1, "lm_decode_frames: frame %d has size %d x %d", i, fm.rows, fm.cols);
    out_base[i + 1] = out_base[i] + (uint64_t)fm.rows * fm.cols;
    if (fm.offset > n_bytes || fm.length > n_bytes - fm.offset) return fail(-1, "lm_decode_frames: frame %d lies outside the data", i);
    if (fm.codec != LM_CODEC_JPEG_LOSSLESS && fm.codec != LM_CODEC_RLE) hstat[i] = LM_ERR_DECODE_HEADER;
  }
  const uint64_t n_out = out_base[nf];

  // ---- host parsing
  std::vector<JHost> jh;
  std::vector<RSeg> rsegs;
  uint64_t e_total = 0;
  uint32_t run_total = 0;
  for (int i = 0; i < nf; ++i) {
    if (hstat[i]) continue;
    const lm_frame& fm = frames[i];
    if (fm.codec == LM_CODEC_JPEG_LOSSLESS) {
      JHost j;
      memset(&j, 0, sizeof(j));
      if ((hstat[i] = parse_jpeg(data, fm.offset, fm.length, fm, j))) continue;
      j.f.is_signed = fm.is_signed ? 1 : 0;
      j.f.idx = i;
      j.f.out_base = out_base[i];
      j.f.e_off = e_total;
      e_total += j.f.ent_end - j.f.ent_begin;
      jh.push_back(j);
    } else {
      uint64_t b0, b1;
      if ((hstat[i] = parse_rle(data, fm.offset, fm.length, b0, b1))) continue;
      const uint32_t n = (uint32_t)((uint64_t)fm.rows * fm.cols);
      const uint64_t bounds[3] = {fm.offset + b0, fm.offset + b1, fm.offset + fm.length};
      for (int pl = 0; pl < 2; ++pl) {
        RSeg s;
        s.begin = bounds[pl];
        s.end = bounds[pl + 1];
        s.out_base = out_base[i];
        s.n_samples = n;
        s.plane = pl;
        s.run_cap = (uint32_t)std::min<uint64_t>(n, (s.end - s.begin) / 2 + 1);
        s.run_base = run_total;
        if ((uint64_t)run_total + s.run_cap > 0xFFFFFFFFull) return fail(-1, "lm_decode_frames: too many RLE runs in one call");
        run_total += s.run_cap;
        s.idx = i;
        rsegs.push_back(s);
      }
    }
  }
  if (e_total >= (1ull << 32) - 1) return fail(-1, "lm_decode_frames: more than 4 GB of entropy-coded data in one call");

  Scratch sc;
  CU(cudaStreamCreateWithFlags(&sc.st, cudaStreamNonBlocking));
  uint8_t* d_data;
  uint16_t* d_out;
  int32_t* d_stat;
  CU(sc.alloc(&d_data, n_bytes));
  CU(sc.alloc(&d_out, n_out));
  CU(sc.alloc(&d_stat, nf));
  CU(cudaMemcpyAsync(d_data, data, n_bytes, cudaMemcpyHostToDevice, sc.st));
  CU(cudaMemsetAsync(d_out, 0, n_out * sizeof(uint16_t), sc.st));
  CU(cudaMemsetAsync(d_stat, 0, nf * sizeof(int32_t), sc.st));

  // ---- JPEG
  const int nj = (int)jh.size();
  if (nj > 0) {
    std::vector<JFrame> jf(nj);
    std::vector<HuffDev> jt(nj);
    for (int k = 0; k < nj; ++k) { jf[k] = jh[k].f; jt[k] = jh[k].table; }
    JFrame* d_jf;
    HuffDev* d_jt;
    uint64_t *d_v, *d_fv;
    CU(sc.alloc(&d_jf, nj));
    CU(sc.alloc(&d_jt, nj));
    CU(sc.alloc(&d_v, e_total + 1));
    CU(sc.alloc(&d_fv, nj + 1));
    CU(cudaMemcpyAsync(d_jt, jt.data(), nj * sizeof(HuffDev), cudaMemcpyHostToDevice, sc.st));
    CU(cudaMemcpyAsync(d_jf, jf.data(), nj * sizeof(JFrame), cudaMemcpyHostToDevice, sc.st));
    lm_jpeg_classify<<<(unsigned)((e_total + 1 + 255) / 256), 256, 0, sc.st>>>(d_data, d_jf, nj, e_total, d_v, d_stat);
    CU(cudaGetLastError());
    if (int rc = scan_exclusive(sc, d_v, e_total + 1)) return rc;
    lm_jpeg_frame_offsets<<<(nj + 1 + 255) / 256, 256, 0, sc.st>>>(d_jf, nj, d_v, e_total, d_fv);
    CU(cudaGetLastError());
    std::vector<uint64_t> fv(nj + 1);
    CU(cudaMemcpyAsync(fv.data(), d_fv, (nj + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, sc.st));
    CU(cudaStreamSynchronize(sc.st));
    const uint64_t kept = fv[nj] & KEPT_MASK, n_rst = fv[nj] >> RST_SHIFT;
    const uint64_t nseg_all = n_rst + nj;
    uint8_t* d_comp;
    uint32_t* d_segb;
    CU(sc.alloc(&d_comp, kept + 8));
    CU(sc.alloc(&d_segb, nseg_all));
    if (e_total > 0) {
      lm_jpeg_compact<<<(unsigned)((e_total + 255) / 256), 256, 0, sc.st>>>(d_data, d_jf, nj, e_total, d_v, d_fv, d_comp, d_segb, nseg_all, d_stat);
      CU(cudaGetLastError());
    }
    std::vector<uint32_t> segb(nseg_all);
    CU(cudaMemcpyAsync(segb.data(), d_segb, nseg_all * sizeof(uint32_t), cudaMemcpyDeviceToHost, sc.st));
    CU(cudaStreamSynchronize(sc.st));

    // restart segments and chunks; a frame whose segment count is not ceil(samples / interval) is not decoded
    std::vector<JSeg> segs;
    std::vector<uint32_t> chunk_seg;
    uint32_t max_chunks_frame = 0, max_chunks_seg = 1;
    for (int k = 0; k < nj; ++k) {
      JFrame& F = jf[k];
      const uint64_t rst0 = fv[k] >> RST_SHIFT, rst1 = fv[k + 1] >> RST_SHIFT;
      const uint64_t first = rst0 + k, nseg = rst1 - rst0 + 1;
      const uint32_t frame_end = (uint32_t)(fv[k + 1] & KEPT_MASK);
      const uint64_t n = (uint64_t)F.rows * F.cols, ivl = (uint64_t)F.ivl_rows * F.cols;
      F.chunk_begin = F.chunk_end = (uint32_t)chunk_seg.size();
      if (nseg != (n + ivl - 1) / ivl) {                    // more or fewer RSTm markers than restart intervals
        hstat[F.idx] = LM_ERR_DECODE_LENGTH;
        continue;
      }
      if (rst1 < rst0 || first + nseg > nseg_all) return fail(-1, "lm_decode_frames: restart marker count out of range (internal error)");
      segb[first] = (uint32_t)(fv[k] & KEPT_MASK);
      for (uint64_t s = 0; s < nseg; ++s) {
        JSeg S;
        S.byte_begin = segb[first + s];
        S.byte_end = s + 1 < nseg ? segb[first + s + 1] : frame_end;
        if (S.byte_end < S.byte_begin || (uint64_t)(S.byte_end - S.byte_begin) * 8 >= (1ull << 32) - CHUNK_BITS)
          return fail(-1, "lm_decode_frames: a restart interval exceeds 512 MB");
        const uint32_t nbits = (S.byte_end - S.byte_begin) * 8u;
        S.first_chunk = (uint32_t)chunk_seg.size();
        S.n_chunks = std::max(1u, (nbits + CHUNK_BITS - 1) / CHUNK_BITS);
        S.sample_begin = F.out_base + s * ivl;
        S.n_samples = (uint32_t)std::min(ivl, n - s * ivl);
        S.frame = (uint32_t)k;
        max_chunks_seg = std::max(max_chunks_seg, S.n_chunks);
        chunk_seg.insert(chunk_seg.end(), S.n_chunks, (uint32_t)segs.size());
        segs.push_back(S);
      }
      F.chunk_end = (uint32_t)chunk_seg.size();
      max_chunks_frame = std::max(max_chunks_frame, F.chunk_end - F.chunk_begin);
    }
    const uint32_t nchunks = (uint32_t)chunk_seg.size(), nseg = (uint32_t)segs.size();
    if (nchunks > 0) {
      JSeg* d_segs;
      uint32_t *d_cseg, *d_start, *d_exit;
      uint64_t* d_cnt;
      int* d_changed;
      CU(sc.alloc(&d_segs, nseg));
      CU(sc.alloc(&d_cseg, nchunks));
      CU(sc.alloc(&d_start, nchunks));
      CU(sc.alloc(&d_exit, nchunks));
      CU(sc.alloc(&d_cnt, nchunks + 1));
      CU(sc.alloc(&d_changed, 1));
      CU(cudaMemcpyAsync(d_jf, jf.data(), nj * sizeof(JFrame), cudaMemcpyHostToDevice, sc.st));
      CU(cudaMemcpyAsync(d_segs, segs.data(), nseg * sizeof(JSeg), cudaMemcpyHostToDevice, sc.st));
      CU(cudaMemcpyAsync(d_cseg, chunk_seg.data(), nchunks * sizeof(uint32_t), cudaMemcpyHostToDevice, sc.st));
      CU(cudaMemsetAsync(d_cnt + nchunks, 0, sizeof(uint64_t), sc.st));
      const dim3 grid((max_chunks_frame + DEC_THREADS - 1) / DEC_THREADS, nj);
      // Round r leaves at least the first r + 1 chunks of every segment synchronised, so the loop ends by
      // max_chunks_seg rounds; in practice a Huffman code resynchronises within a few codewords and 1-2 rounds do.
      for (uint32_t round = 0; round <= max_chunks_seg + MAX_SYNC_ROUNDS_EXTRA; ++round) {
        int changed = 0;
        CU(cudaMemsetAsync(d_changed, 0, sizeof(int), sc.st));
        lm_jpeg_sync<<<grid, DEC_THREADS, 0, sc.st>>>(d_comp, d_jf, d_segs, d_cseg, d_jt, d_start, d_exit, d_cnt, round == 0, d_changed);
        CU(cudaGetLastError());
        if (round == 0) continue;
        CU(cudaMemcpyAsync(&changed, d_changed, sizeof(int), cudaMemcpyDeviceToHost, sc.st));
        CU(cudaStreamSynchronize(sc.st));
        if (!changed) break;
      }
      if (int rc = scan_exclusive(sc, d_cnt, nchunks + 1)) return rc;
      lm_jpeg_emit<<<grid, DEC_THREADS, 0, sc.st>>>(d_comp, d_jf, d_segs, d_cseg, d_jt, d_start, d_cnt, d_out, d_stat);
      CU(cudaGetLastError());
      lm_jpeg_check<<<(nseg + 255) / 256, 256, 0, sc.st>>>(d_jf, d_segs, nseg, d_cnt, d_stat);
      CU(cudaGetLastError());

      // reconstruction, grouped by predictor
      std::vector<uint32_t> lists[8];
      uint32_t max_rows = 1, max_cols = 1, max_ivl = 1, max_diag = 1;
      for (int k = 0; k < nj; ++k) {
        const JFrame& F = jf[k];
        if (F.chunk_end == F.chunk_begin) continue;
        lists[F.pred].push_back((uint32_t)k);
        const uint32_t nivl = (F.rows + F.ivl_rows - 1) / F.ivl_rows;
        max_rows = std::max(max_rows, F.rows);
        max_cols = std::max(max_cols, F.cols * nivl);
        max_ivl = std::max(max_ivl, nivl);
        max_diag = std::max(max_diag, (F.cols + F.ivl_rows - 1) * nivl);
      }
      std::vector<uint32_t> all;
      for (int p = 1; p <= 7; ++p) all.insert(all.end(), lists[p].begin(), lists[p].end());
      uint32_t* d_lists;
      CU(sc.alloc(&d_lists, all.size()));
      CU(cudaMemcpyAsync(d_lists, all.data(), all.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, sc.st));
      uint32_t at = 0;
      for (int p = 1; p <= 7; ++p) {
        const uint32_t n = (uint32_t)lists[p].size();
        if (!n) continue;
        const uint32_t* L = d_lists + at;
        at += n;
        const dim3 g_rows((max_rows + 7) / 8, n), g_first((max_ivl + 7) / 8, n);
        const dim3 g_col0((max_ivl + 127) / 128, n), g_cols((max_cols + 127) / 128, n), g_diag((max_diag + 127) / 128, n);
        switch (p) {
          case 1:   // column 0 down each interval, then every row
            lm_undiff_cols<<<g_col0, 128, 0, sc.st>>>(d_jf, L, d_out, 1);
            lm_undiff_rows<<<g_rows, 256, 0, sc.st>>>(d_jf, L, d_out, 0);
            break;
          case 2:   // the interval's first row, then every column
            lm_undiff_rows<<<g_first, 256, 0, sc.st>>>(d_jf, L, d_out, 1);
            lm_undiff_cols<<<g_cols, 128, 0, sc.st>>>(d_jf, L, d_out, 0);
            break;
          case 3:   // first row, first column, then the diagonals
            lm_undiff_rows<<<g_first, 256, 0, sc.st>>>(d_jf, L, d_out, 1);
            lm_undiff_cols<<<g_col0, 128, 0, sc.st>>>(d_jf, L, d_out, 1);
            lm_undiff_diag<<<g_diag, 128, 0, sc.st>>>(d_jf, L, d_out);
            break;
          case 4:   // Ra + Rb - Rc is linear: a 2-D prefix sum per interval
            lm_undiff_rows<<<g_rows, 256, 0, sc.st>>>(d_jf, L, d_out, 0);
            lm_undiff_cols<<<g_cols, 128, 0, sc.st>>>(d_jf, L, d_out, 0);
            break;
          default:
            lm_undiff_wave<<<dim3(max_ivl, n), 256, 0, sc.st>>>(d_jf, L, d_out);
            break;
        }
        CU(cudaGetLastError());
      }
      lm_jpeg_finish<<<dim3(64, (unsigned)all.size()), 256, 0, sc.st>>>(d_jf, d_lists, d_out);
      CU(cudaGetLastError());
    }
  }

  // ---- RLE
  const int nr = (int)rsegs.size();
  if (nr > 0) {
    RSeg* d_rs;
    Run* d_runs;
    uint32_t* d_nruns;
    CU(sc.alloc(&d_rs, nr));
    CU(sc.alloc(&d_runs, run_total));
    CU(sc.alloc(&d_nruns, nr));
    CU(cudaMemcpyAsync(d_rs, rsegs.data(), nr * sizeof(RSeg), cudaMemcpyHostToDevice, sc.st));
    lm_rle_runs<<<(nr + 63) / 64, 64, 0, sc.st>>>(d_data, d_rs, nr, d_runs, d_nruns, d_stat);
    CU(cudaGetLastError());
    lm_rle_expand<<<nr, 256, 0, sc.st>>>(d_data, d_rs, d_runs, d_nruns, d_out);
    CU(cudaGetLastError());
  }

  std::vector<int32_t> dstat(nf);
  CU(cudaMemcpyAsync(out, d_out, n_out * sizeof(uint16_t), cudaMemcpyDeviceToHost, sc.st));
  CU(cudaMemcpyAsync(dstat.data(), d_stat, nf * sizeof(int32_t), cudaMemcpyDeviceToHost, sc.st));
  CU(cudaStreamSynchronize(sc.st));
  for (int i = 0; i < nf; ++i) status[i] = hstat[i] ? hstat[i] : dstat[i];
  return 0;
}

}  // namespace lm_decode

extern "C" int lm_decode_frames(int device, const uint8_t* data, size_t n_bytes, const lm_frame* frames, int n_frames,
                                uint16_t* out, int32_t* frame_status) {
  if (n_frames < 0 || n_frames > 65535 || (n_frames > 0 && (!data || !frames || !out || !frame_status)))
    return fail(-1, "lm_decode_frames: invalid arguments (n_frames %d)", n_frames);
  if (n_frames == 0) return 0;
  int prev = -1;
  cudaError_t e = cudaGetDevice(&prev);
  if (e != cudaSuccess) return fail((int)e, "lm_decode_frames: cudaGetDevice failed: %s", cudaGetErrorString(e));
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail((int)e, "lm_decode_frames: cudaSetDevice(%d) failed: %s", device, cudaGetErrorString(e));
  const int rc = lm_decode::decode(data, n_bytes, frames, n_frames, out, frame_status);
  cudaSetDevice(prev);
  return rc;
}
