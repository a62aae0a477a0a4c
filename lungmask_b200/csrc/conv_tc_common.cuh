// Pieces of the tensor-core convolution kernel (conv_tc.cu): tile geometry, shared-memory budget and the epilogue warps'
// code - chunk drains out of TMEM with round-to-nearest fp32 accumulation, then bias / ReLU / BatchNorm, operand-plane split,
// 2x2 average pool, 1x1 head with log-softmax + argmax, and the TMA stores.
// The including file defines LM_PROF_T0 / LM_PROF_ADD / LM_EXP (instrumentation of tools/conv_probe) first.
// Staged rows leave through cp.async.bulk.tensor stores out of a 4 KB buffer per epilogue warp.  (Round 2 measured coalesced
// 16-byte stores out of the same buffer: equal within 0.5 % per wave, profiles/r02_call5_summary.md; 8-row staging passes with a
// fourth weight stage: 3.4 % slower; and an L1 prefetch of the per-channel constants: no gain, superseded by the shared-memory
// copy below.)
#pragma once
#include "conv_tc.cuh"
#include "sm100_ptx.cuh"

namespace lm {
namespace {

// setmaxnreg budgets: warps 0-3 (producer, issuer, TMEM allocator) give registers to the two epilogue warpgroups
constexpr int kRegsLow = 88, kRegsHigh = 208;

constexpr int BM = 128, BK = kBK, TILE_H = 16, TILE_W = 8;  // BK channels = one 128-byte row (64 fp16)
constexpr int ROW_BYTES = 128;
constexpr int HALO_W = TILE_W + 2, HALO_H = TILE_H + 2;
constexpr int A_PLANE_BYTES_3x3 = HALO_W * HALO_H * ROW_BYTES;  // 180 rows x 128 B = 23040 B per plane
constexpr int A_PLANE_BYTES_1x1 = BM * ROW_BYTES;               // 16 KB per plane
constexpr int F32_ROW_CH = 32;                                  // channels per staged 128-byte row of an fp32 output
constexpr int A_BUF_BYTES = 2 * A_PLANE_BYTES_3x3;           // 46080 B = 45 KB (both planes), 1024-aligned
constexpr int NUM_A_BUFS = 2;
constexpr int STG_WARP_BYTES = 4096;    // output staging per epilogue warp: one 32-pixel plane of 64 channels
constexpr int CONST_WARP_FLOATS = 3 * 64;  // per epilogue warp: bias | BN scale | BN shift of the 64 channels its threads hold
constexpr int NUM_THREADS = 384;
constexpr int EPI_WARP0 = 4;
constexpr int NUM_EPI_THREADS = 256;
constexpr int MAX_CLASSES = 8;

template <int BN>
struct Cfg {
  static constexpr int B_PLANE_BYTES = BN * ROW_BYTES;
  static constexpr int STAGE_BYTES = 2 * B_PLANE_BYTES;      // one weight tile (hi + lo planes) per k-block
  static constexpr int STAGES = (BN == 64) ? 6 : 3;
  static constexpr int ACC_COLS = 2 * BN;          // [0,BN) hi*hi, [BN,2BN) hi*lo + lo*hi
  static constexpr int NBUF = 512 / ACC_COLS;      // accumulator ring: 2 slots (BN=128), 4 slots (BN=64)
  static constexpr int TMEM_COLS = NBUF * ACC_COLS;
  // Epilogue organisation.  BN = 128: the 8 epilogue warps split every tile's columns in two halves (64 per thread).
  // BN = 64: a thread can hold a full row (64 columns), so the warps form TWO GROUPS that take alternate tiles:
  // while one group runs the tile-end epilogue (BN, split, TMA stores - a third of a short 18-k-block tile), the
  // other already drains the next tile's chunks and the tensor pipe never waits for a free accumulator slot.
  static constexpr int HALVES = (BN == 64) ? 1 : 2;
  static constexpr int EGROUPS = (BN == 64) ? 2 : 1;   // (two groups of 128 columns per thread for BN = 128: measured, no gain -
                                                       //  profiles/r02_call7_*: the tile-end latency per tile doubles)
  // Everything lives in dynamic shared memory (declared __align__(1024): the swizzled tiles need it, and no static shared
  // memory means no alignment slack): activation patches | weight ring | output staging | per-channel constants |
  // mbarriers | TMEM base | head
  static constexpr int NUM_BARS = 2 * STAGES + (EGROUPS + 1) * NBUF + 2 * NUM_A_BUFS;
  static constexpr int OFF_B = NUM_A_BUFS * A_BUF_BYTES;
  static constexpr int OFF_STG = OFF_B + STAGES * STAGE_BYTES;
  static constexpr int OFF_CONST = OFF_STG + (NUM_EPI_THREADS / 32) * STG_WARP_BYTES;
  static constexpr int OFF_BARS = OFF_CONST + (NUM_EPI_THREADS / 32) * CONST_WARP_FLOATS * 4;
  static constexpr int OFF_TMEM = OFF_BARS + NUM_BARS * 8;
  static constexpr int OFF_HEAD = OFF_TMEM + 16;                                   // BN = 64 only: head weights + bias
  static constexpr int DYN_SMEM = OFF_HEAD + ((BN == 64) ? (MAX_CLASSES * 64 + MAX_CLASSES) * 4 : 0);
  static_assert(DYN_SMEM <= 232448, "shared-memory budget (227 KB per CTA)");
};

struct TileCoord {
  int n, y0, x0, n0;
};

__device__ __forceinline__ TileCoord decode_tile(int tile, int n_tiles, int tiles_x, int tiles_img, int BN) {
  TileCoord t;
  const int mt = tile / n_tiles;
  t.n0 = (tile - mt * n_tiles) * BN;
  t.n = mt / tiles_img;
  const int r = mt - t.n * tiles_img;
  const int ty = r / tiles_x;
  t.y0 = ty * TILE_H;
  t.x0 = (r - ty * tiles_x) * TILE_W;
  return t;
}

// The epilogue warps (warps EPI_WARP0 .. EPI_WARP0 + 7) of one CTA: tiles first_tile, first_tile + tile_step, ... < total_tiles.
template <int BN>
__device__ __forceinline__ void conv_epilogue_warps(const ConvParams& p, const CUtensorMap* tmOut, const CUtensorMap* tmPool,
                                                    uint32_t tmem_base, uint32_t tfull0, uint32_t tempty0, uint8_t* smem_out,
                                                    float* smem_const, const float* s_head_w, const float* s_head_b, int first_tile,
                                                    int total_tiles, int tile_step, int num_chunks) {
  using C = Cfg<BN>;
  constexpr int NBUF = C::NBUF;
  constexpr int HALVES = C::HALVES, EGROUPS = C::EGROUPS;
  constexpr int NC = BN / HALVES;  // accumulator columns held by one epilogue thread (64)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_x = p.W / TILE_W, tiles_img = tiles_x * (p.H / TILE_H);
  const int n_tiles = p.Cout / BN;
  const int q = warp & 3;
  const int half = (HALVES == 2) ? ((warp - EPI_WARP0) >> 2) : 0;
  const uint32_t egroup = (EGROUPS == 2) ? (uint32_t)((warp - EPI_WARP0) >> 2) : 0u;
  const int row = q * 32 + lane, hl = row >> 3, wl = row & 7;  // 16 x 8 patch, 8 pixels per image row
  const uint32_t lane_base = (uint32_t)(q * 32) << 16;
  const uint32_t tfull_g = tfull0 + 8 * (egroup * NBUF);
  uint32_t buf = 0;          // ring slot of the next chunk (all tiles, both groups, advance it)
  uint32_t phase_bits = 0;   // bit b: parity this group's next wait on slot b expects (its own barrier set)
  uint32_t tseq = 0;
  static_assert(NC == 64, "one epilogue thread holds 64 accumulator columns");
  float* cst = smem_const + (warp - EPI_WARP0) * CONST_WARP_FLOATS;   // this warp's bias | scale | shift (64 floats each)
  int const_n0 = -1;                                                  // channel block they belong to
  for (int tile = first_tile; tile < total_tiles; tile += tile_step, ++tseq) {
    if (EGROUPS == 2 && (tseq & 1u) != egroup) { buf = (buf + (uint32_t)num_chunks) % NBUF; continue; }  // the other group's tile
    const TileCoord t = decode_tile(tile, n_tiles, tiles_x, tiles_img, BN);
    float acc[NC];
#pragma unroll
    for (int i = 0; i < NC; ++i) acc[i] = 0.f;
    if (t.n0 != const_n0) {
      // The tile-end epilogue needs 3 x NC per-channel constants.  Read from global memory there they were its largest
      // stall (long-scoreboard waits on 48 dependent-use LDG.128 per thread with two warps per scheduler to hide them,
      // ncu source view of round 2); the warp copies them into its own 768 bytes of shared memory now - one coalesced
      // LDG per lane, in flight while the tile's chunks are computed - and reads them back as broadcast LDS.128.
      const_n0 = t.n0;
      const int cb0 = t.n0 + half * NC;
      // The stored planes hold y * out_scale with y = relu(..) * scale + shift: the power-of-two factor goes into the copies
      // of scale and shift (scaling by 2^k commutes with every rounding involved).  The head consumes y itself.
      const float cscale = (p.mode == kModeHead) ? 1.f : p.out_scale;
      __syncwarp();                                        // the previous tile's reads are done
      const int arr = lane >> 4, i4 = lane & 15;         // lanes 0-15: bias, 16-31: scale; then lanes 0-15: shift
      const float* src = arr == 0 ? p.bias : p.scale;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (src) v = __ldg(reinterpret_cast<const float4*>(src + cb0) + i4);
      if (arr == 1) { v.x *= cscale; v.y *= cscale; v.z *= cscale; v.w *= cscale; }
      reinterpret_cast<float4*>(cst)[lane] = v;
      if (lane < 16) {
        float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.shift) h = __ldg(reinterpret_cast<const float4*>(p.shift + cb0) + i4);
        h.x *= cscale; h.y *= cscale; h.z *= cscale; h.w *= cscale;
        reinterpret_cast<float4*>(cst)[32 + lane] = h;
      }
      __syncwarp();
    }
    for (int c = 0; c < num_chunks; ++c) {
      { LM_PROF_T0(); mbar_wait<1>(tfull_g + 8 * buf, (phase_bits >> buf) & 1u); if (warp == EPI_WARP0 && lane == 0) LM_PROF_ADD(6); }
      phase_bits ^= 1u << buf;
      tc_fence_after();
      LM_PROF_T0();
      const uint32_t col0 = tmem_base + lane_base + buf * C::ACC_COLS + half * NC;
      const bool last_use = c >= num_chunks - NBUF;  // this slot is not written again in this tile
      auto hand_back = [&]() {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty0 + 8 * buf);
      };
      // all TMEM reads of this slot first, then hand the slot back BEFORE the register adds: the
      // tensor core's next chunk on this slot does not have to wait for the fp32 accumulation
      float v[64];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        if (!(LM_EXP & 2) || last_use) tmem_ld32(col0 + j * 32, v + j * 32);   // hi*hi partial sums of this chunk
      }
      if (last_use) {
        float w[64];
#pragma unroll
        for (int j = 0; j < 2; ++j) tmem_ld32(col0 + BN + j * 32, w + j * 32);  // the slot's corrections, whole tile
        tmem_ld_wait();
        hand_back();
#pragma unroll
        for (int i = 0; i < 64; ++i) acc[i] = (acc[i] + v[i]) + w[i] * kLoUnscale;  // exact power-of-two rescale of hi*lo + lo*hi
      } else {
        tmem_ld_wait();
        hand_back();
#pragma unroll
        for (int i = 0; i < 64; ++i) acc[i] += v[i];
      }
      if (warp == EPI_WARP0 && lane == 0) LM_PROF_ADD(7);
      if (++buf == NBUF) buf = 0;
    }
    LM_PROF_T0();
    // acc * in_unscale undoes the operands' power-of-two scales (1.0 unless the engine rescaled a tensor).  The product is
    // exact, so fma(acc, unscale, bias) below rounds exactly like the separate multiply and add.
    const float unscale = p.in_unscale;
    const int y = t.y0 + hl, x = t.x0 + wl;
    const int cbase = t.n0 + half * NC;
    const float4* bias4 = reinterpret_cast<const float4*>(cst);             // shared memory, all lanes read the same address

    // The tile leaves through shared memory: every thread drops its pixel's 32-channel groups as 128-byte
    // rows (128B-swizzled, conflict-free) into its WARP's 4 KB staging buffer (32 pixels = 4 image rows x 8)
    // and the warp's lane 0 hands the buffer to a TMA store - fully coalesced 128 B bursts instead of 32
    // scattered 16-byte stores per warp instruction (16-23k cycles per tile, profiles/r01_conv_role_stalls_v2.log)
    // - with no cross-warp barrier: each epilogue warp streams its own rows out independently.
    const uint32_t stage = smem_u32(smem_out) + (uint32_t)(warp - EPI_WARP0) * (uint32_t)STG_WARP_BYTES;
    const bool issuer = (lane == 0);
    const int ty0 = t.y0 + 4 * q;  // first image row of this warp's 32 pixels
    auto stage_row = [&](uint32_t r, const uint32_t* v8x4) {  // 32 words (128 B) -> row r, chunk j at (j ^ (r & 7))
      if (LM_EXP & 4) {  // keep the values alive, skip the shared-memory traffic
        uint32_t x = 0;
#pragma unroll
        for (int j = 0; j < 32; ++j) x ^= v8x4[j];
        if (x == 0x12345u) p.labels[0] = 1;
        return;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint32_t addr = stage + r * 128u + (uint32_t)((j ^ (int)(r & 7u)) << 4);
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v8x4[4 * j]), "r"(v8x4[4 * j + 1]),
                     "r"(v8x4[4 * j + 2]), "r"(v8x4[4 * j + 3])
                     : "memory");
      }
    };
    // one 128-byte row of operand-format channels (BK of them) per plane, from fp32 values: both planes in one pass
    auto pack_rows = [&](const float* src, uint32_t* vh, uint32_t* vl) {
#pragma unroll
      for (int i = 0; i < 32; ++i) split_f16x2(src[2 * i], src[2 * i + 1], vh[i], vl[i]);
    };
    auto round_begin = [&]() {
      if (issuer) tma_store_wait_read();  // this warp's previous store has finished reading the buffer
      __syncwarp();
    };
    auto round_end = [&]() {
      fence_proxy_async();
      __syncwarp();
    };

    if (p.mode == kModeLinear) {
#pragma unroll
      for (int g = 0; g < NC / F32_ROW_CH; ++g) {
        uint32_t v[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 b = bias4[g * 8 + i];
          v[4 * i] = __float_as_uint(__fmaf_rn(acc[g * 32 + 4 * i], unscale, b.x)); v[4 * i + 1] = __float_as_uint(__fmaf_rn(acc[g * 32 + 4 * i + 1], unscale, b.y));
          v[4 * i + 2] = __float_as_uint(__fmaf_rn(acc[g * 32 + 4 * i + 2], unscale, b.z)); v[4 * i + 3] = __float_as_uint(__fmaf_rn(acc[g * 32 + 4 * i + 3], unscale, b.w));
        }
        round_begin();
        stage_row((uint32_t)lane, v);
        round_end();
        if (issuer && !(LM_EXP & 4)) { tma_store_4d(tmOut, stage, cbase + g * F32_ROW_CH, t.x0, ty0, t.n); tma_store_commit(); }
      }
    } else {
      const float4* scale4 = bias4 + NC / 4;
      const float4* shift4 = bias4 + 2 * (NC / 4);
      // y = relu(acc + bias) * scale + shift   (Conv -> ReLU -> BatchNorm(eval), resunet.py:93-105)
#pragma unroll
      for (int i = 0; i < NC / 4; ++i) {
        const float4 b = bias4[i], s = scale4[i], h = shift4[i];
        acc[4 * i + 0] = __fadd_rn(__fmul_rn(fmaxf(__fmaf_rn(acc[4 * i + 0], unscale, b.x), 0.f), s.x), h.x);
        acc[4 * i + 1] = __fadd_rn(__fmul_rn(fmaxf(__fmaf_rn(acc[4 * i + 1], unscale, b.y), 0.f), s.y), h.y);
        acc[4 * i + 2] = __fadd_rn(__fmul_rn(fmaxf(__fmaf_rn(acc[4 * i + 2], unscale, b.z), 0.f), s.z), h.z);
        acc[4 * i + 3] = __fadd_rn(__fmul_rn(fmaxf(__fmaf_rn(acc[4 * i + 3], unscale, b.w), 0.f), s.w), h.w);
      }
      if (BN == 64 && p.mode == kModeHead) {   // (the head follows a 64-channel layer: no head code in the BN = 128 kernel)
        // 1x1 head (resunet.py:69): this thread holds all 64 channels of its pixel (BN = 64 rows are not split).
        float lg[MAX_CLASSES];
        float mx = -INFINITY;
#pragma unroll
        for (int k = 0; k < MAX_CLASSES; ++k) {
          float sdot = 0.f;
          if (k < p.K) {
#pragma unroll
            for (int i = 0; i < NC; ++i) sdot = fmaf(s_head_w[k * 64 + (half * NC + i) % 64], acc[i], sdot);
          }
          lg[k] = (k < p.K) ? sdot + s_head_b[k] : -INFINITY;
          mx = fmaxf(mx, lg[k]);
        }
        float se = 0.f;
#pragma unroll
        for (int k = 0; k < MAX_CLASSES; ++k) if (k < p.K) se += expf(lg[k] - mx);
        const float lse = logf(se);
        int best = 0;
        float bestv = -INFINITY;
#pragma unroll
        for (int k = 0; k < MAX_CLASSES; ++k) {
          if (k < p.K) {
            const float sc = (lg[k] - mx) - lse;  // LogSoftmax(dim=1), resunet.py:70
            if (sc > bestv) { bestv = sc; best = k; }  // first index wins ties (mask.py:185)
            if (p.scores) p.scores[(((size_t)t.n * p.K + k) * p.H + y) * p.W + x] = sc;
          }
        }
        p.labels[((size_t)t.n * p.H + y) * p.W + x] = (uint8_t)best;
      } else {
        // (the stored planes hold y * out_scale: the power-of-two factor is already in the scale / shift copies)
        {  // fp16 saturates: report instead of storing inf (the engine lowers out_scale and runs again)
          bool ovf = false;
#pragma unroll
          for (int i = 0; i < NC; ++i) ovf |= !(fabsf(acc[i]) <= kOpMax);
          if (__any_sync(0xffffffffu, ovf) && lane == 0 && p.range_flag) *p.range_flag = 1;
        }
#pragma unroll
        for (int g = 0; g < NC / BK; ++g) {
          uint32_t vh[32], vl[32];
          pack_rows(acc + g * BK, vh, vl);
#pragma unroll
          for (int plane = 0; plane < 2; ++plane) {
            const uint32_t* v = plane ? vl : vh;
            round_begin();
            stage_row((uint32_t)lane, v);
            round_end();
            if (issuer && !(LM_EXP & 4)) { tma_store_5d(tmOut, stage, cbase + g * BK, t.x0, ty0, plane, t.n); tma_store_commit(); }
          }
        }
        if (p.mode == kModeReluBnPool) {
          // 2x2 average (resunet.py:64): partners are lanes ^1 (x) and ^8 (y) of the same warp; the lane with
          // even x and y stages the pooled pixel: 8 per warp (2 pooled rows x 4) = rows 0..7 of the warp's buffer.
          const bool writer = (lane & 9) == 0;
          const uint32_t prow = (uint32_t)((lane >> 4) * (TILE_W / 2) + ((lane & 7) >> 1));
#pragma unroll
          for (int g = 0; g < NC / BK; ++g) {
            float pv[BK];
#pragma unroll
            for (int i = 0; i < BK; ++i) {
              float s = acc[g * BK + i] + __shfl_xor_sync(0xffffffffu, acc[g * BK + i], 1);
              s = s + __shfl_xor_sync(0xffffffffu, s, 8);
              pv[i] = s * 0.25f;
            }
            uint32_t vh[32], vl[32];
            pack_rows(pv, vh, vl);
#pragma unroll
            for (int plane = 0; plane < 2; ++plane) {
              const uint32_t* v = plane ? vl : vh;
              round_begin();
              if (writer) stage_row(prow, v);
              round_end();
              if (issuer && !(LM_EXP & 4)) { tma_store_5d(tmPool, stage, cbase + g * BK, t.x0 >> 1, ty0 >> 1, plane, t.n); tma_store_commit(); }
            }
          }
        }
      }
    }
    if (warp == EPI_WARP0 && lane == 0) LM_PROF_ADD(8);
  }
  if (lane == 0) tma_store_wait_all();  // every epilogue warp's issuer: global writes complete before exit
}

}  // namespace
}  // namespace lm
