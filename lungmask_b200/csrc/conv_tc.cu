// 3x3 / 1x1 convolution as an implicit GEMM on the sm_100a 5th-generation tensor cores.
//
// Replaces, for the U-Net of lungmask/resunet.py, every Conv2d(3x3,pad 1)+ReLU+BatchNorm2d pair
// (resunet.py:93-105), the decoder's 1x1 convolutions (resunet.py:133, evaluated below the upsample),
// the 2x2 average pool (resunet.py:64, fused as an epilogue), the channel concat (resunet.py:147,
// "virtual": the K loop walks two tensor maps) and the head 1x1 + LogSoftmax + argmax
// (resunet.py:69-70, mask.py:184-186, fused into the last convolution's epilogue).
//
// GEMM view: M = 128 output pixels (a 16-row x 8-column patch of one image), N = BN output channels,
// K = taps * Cin walked in k-blocks of BK input channels of one filter tap, BK = one 128-byte row of the operand
// format (conv_tc.cuh: 64 fp16 channels).
//   * A operand: ONE 5-D TMA box per BK-channel block - the patch plus its one-pixel halo,
//     (BK ch, 10 x, 18 y, 2 planes, 1 image) = 180 rows of 128 B per plane - serves all nine taps: the tap
//     (dy,dx) view is the same shared-memory tile entered at row (dy+1)*10 + (dx+1) with an 8-row-group
//     stride of 10 rows.  UMMA shared-memory descriptors allow that: the 128B swizzle is a function of the
//     absolute shared-memory address, so a start address at any 128-byte row and a stride-byte-offset of
//     1280 B address the rows TMA wrote (checked on B200: profiles/r01_umma_rowoffset_probe.log).  This
//     cuts the L2->SM traffic of the activations 6.4x versus one box per tap.  TMA zero-fills outside the
//     image, which IS the convolution's zero padding.
//   * B operand: one 4-D TMA box (BK cin, BN cout, 1 tap, 2 planes) per k-block.
//   * both land 128B-swizzled, K-major, i.e. in the canonical tcgen05 shared-memory layout.
//   * fp32-class accuracy from 11-bit tensor-core operands: every fp32 value is pre-split into a hi and a lo plane
//     (fp16 hi + fp16 lo * 2^-11) and each k-step computes
//     hi*hi, hi*lo and lo*hi - three exact products - with TWO instructions: the B tile's hi and lo planes are
//     adjacent in shared memory, so  A_hi x [B_hi;B_lo]  is one N = 2*BN MMA whose left half of the accumulator is
//     hi*hi and whose right half is hi*lo; A_lo x B_hi (N = BN) then adds lo*hi into that right half.  The
//     tensor-core accumulator rounds toward zero (measured on B200: -6e-5 relative drift over K = 8192,
//     profiles/r01_umma_probe.log), so the dominant hi*hi sum is kept apart from the 2^-11-times-smaller
//     corrections and only `chunk_kb` k-blocks (4 MMA k-steps each) of hi*hi are accumulated in TMEM before the
//     epilogue warps add that partial tile into fp32 registers with round-to-nearest, while the tensor core
//     already works on the next chunk (NBUF TMEM accumulators of 2*BN columns in a ring).  The correction halves
//     are NOT drained per chunk: each ring slot keeps accumulating its corrections for the whole tile (their
//     drift is 2^-11 times smaller still) and is read once, with the slot's last chunk - so the per-chunk drain
//     is BN columns, half of the accumulator.
//   * persistent CTAs (one per SM), warp-specialised: warp 0 TMA producer, warp 1 MMA issuer - one elected lane
//     running mma_issue_loop -, warp 2 TMEM allocator, warps 4-11 epilogue (TMEM lane quarter
//     = warp % 4, two warps share a quarter and split the columns or, for BN = 64, take alternate tiles).
#include <atomic>
#include <stdio.h>
#include "conv_tc.cuh"
#include "sm100_ptx.cuh"

namespace lm {
#ifdef LM_CONV_PROFILE
// Role-level stall accounting for tools/conv_probe: cycles each role spends waiting on each barrier class.
__device__ unsigned long long g_conv_prof[16];
#endif
}  // namespace lm
#ifdef LM_CONV_PROFILE
#define LM_PROF_T0() const long long prof_t0_ = clock64()
#define LM_PROF_ADD(slot) atomicAdd(&g_conv_prof[slot], (unsigned long long)(clock64() - prof_t0_))
#else
#define LM_PROF_T0()
#define LM_PROF_ADD(slot)
#endif
// LM_EXP: bit mask of timing-only ablations for tools/conv_probe (results are wrong with any bit set):
//   1 no correction MMAs, 2 chunk drains skip their TMEM loads, 4 tile epilogue skips staging + TMA stores,
//   16 no wide MMAs (only the N = BN correction MMAs), 32 producer loads no weights after the first ring fill
#ifndef LM_EXP
#define LM_EXP 0
#endif
#include "conv_tc_common.cuh"

namespace lm {
namespace {

struct IssueArgs {
  int first_tile, total_tiles, tile_step, num_cb, chunk_kb;
  uint32_t tmem_base, smem_a, smem_b;
  uint32_t full0, empty0, tfull0, tempty0, afull0, aempty0;  // mbarrier arrays (shared-memory addresses)
};

// The MMA issue loop of the issuer thread.  Chunk g (counted over all tiles of the CTA) lives in accumulator slot
// g % NBUF.
//
// Software pipelining: the tensor pipe's instruction queue is only a few MMAs deep, so the gap between the last MMA
// of one k-block and the first MMA of the next must stay short.  The barrier waits and ring bookkeeping of k-block
// i+1 (weight stage, activation buffer) are therefore executed in the MIDDLE of k-block i's MMA burst and the
// burst's remaining MMAs then follow back to back with k-block i+1's first ones.
template <int BN, int TAPS, bool UNROLL>
__device__ __forceinline__ void mma_issue_loop(const IssueArgs& g) {
  using C = Cfg<BN>;
  constexpr uint32_t STAGES = C::STAGES, NBUF = C::NBUF;
  constexpr int EGROUPS = C::EGROUPS;
  constexpr int PATCH_W = (TAPS == 9) ? HALO_W : TILE_W;  // shared-memory rows per image row of the patch
  constexpr uint32_t A_PLANE = (uint32_t)((TAPS == 9) ? A_PLANE_BYTES_3x3 : A_PLANE_BYTES_1x1) >> 4;
  constexpr uint32_t B_PLANE = (uint32_t)C::B_PLANE_BYTES >> 4;
  constexpr uint32_t idesc_wide = make_idesc_f16(BM, 2 * BN), idesc_corr = make_idesc_f16(BM, BN);
  // shared-memory descriptors as (lo, hi) words: lo = start>>4 | LBO, hi = SBO | version | swizzle.
  // A: K-major SW128 entered at an arbitrary 128-byte row, 8-row group stride = one patch row.
  constexpr uint64_t hi_a = (uint64_t)((uint32_t)((PATCH_W * 128) >> 4) | (1u << 14) | (2u << 29)) << 32;
  constexpr uint64_t hi_b = (uint64_t)((uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29)) << 32;
  const uint32_t a_base_lo = ((g.smem_a & 0x3FFFFu) >> 4) | (1u << 16);
  const uint32_t b_base_lo = ((g.smem_b & 0x3FFFFu) >> 4) | (1u << 16);
  const int num_kb = g.num_cb * TAPS, chunk_kb = g.chunk_kb;
  if (g.first_tile >= g.total_tiles) return;

  // state of the k-block whose barriers have been waited for ("current")
  uint32_t s = 0, ph = 0, ab = 0, aph = 0;  // weight ring / activation ring position and phase
  uint32_t gc = 0;                          // chunks closed by this CTA so far -> slot gc % NBUF
  uint32_t tseq = 0;                        // tiles processed: the epilogue group (BN = 64) of a tile is tseq & 1
  int kc = 0;                               // k-blocks already in the open chunk
  int kb_left = num_kb;                     // k-blocks of the tile still to issue (including the current one)
  uint32_t cit = 0;                         // chunks of this tile already closed
  // waits of the first k-block
  mbar_wait(g.afull0, 0);
  mbar_wait(g.tempty0, 1);
  mbar_wait(g.full0, 0);
#ifdef LM_CONV_PROFILE
  const long long prof_issue_t0 = clock64();
#endif

  for (int tile = g.first_tile; tile < g.total_tiles; tile += g.tile_step) {
    const bool last_tile = tile + g.tile_step >= g.total_tiles;
    for (int cb = 0; cb < g.num_cb; ++cb) {
      const uint32_t a_cb = a_base_lo + ab * (uint32_t)(A_BUF_BYTES >> 4);
      const uint32_t ab_cur = ab;
      const bool last_cb = (cb == g.num_cb - 1);
#pragma unroll(UNROLL ? TAPS : 1)
      for (int tap = 0; tap < TAPS; ++tap) {
        // tap (dy, dx) = the same patch entered (dy * PATCH_W + dx) rows further (16-byte units: 8 per row)
        const uint32_t tap_off = (TAPS == 9) ? (uint32_t)(((tap / 3) * PATCH_W + (tap % 3)) * 8) : 0u;
        const uint32_t buf = gc % NBUF;
        const uint32_t d_tmem = g.tmem_base + buf * (uint32_t)C::ACC_COLS;
        const uint32_t alo = a_cb + tap_off;
        const uint32_t blo = b_base_lo + s * (uint32_t)(C::STAGE_BYTES >> 4);
        const bool first = (kc == 0);
        const uint32_t s_cur = s;
        // ---- first part of the burst
        {
          LM_PROF_T0();
          tc_fence_after();
          if (first) {
            // first k-step of a chunk: hi*hi restarts from zero; the corrections restart only at the slot's first
            // chunk of the tile (cit < NBUF), so the two halves need separate instructions here
            umma_f16_c<false>(d_tmem, hi_a | alo, hi_b | blo, idesc_corr);                              // hi*hi :=
            umma_f16(d_tmem + BN, hi_a | alo, hi_b | (blo + B_PLANE), idesc_corr, cit >= NBUF ? 1u : 0u);  // hi*lo
          } else {
            umma_f16_c<true>(d_tmem, hi_a | alo, hi_b | blo, idesc_wide);                               // [hi*hi | hi*lo] +=
          }
          if (!(LM_EXP & 1)) umma_f16_c<true>(d_tmem + BN, hi_a | (alo + A_PLANE), hi_b | blo, idesc_corr);  // lo*hi
          umma_f16_c<true>(d_tmem, hi_a | (alo + 2u), hi_b | (blo + 2u), idesc_wide);
          if (!(LM_EXP & 1)) umma_f16_c<true>(d_tmem + BN, hi_a | (alo + A_PLANE + 2u), hi_b | (blo + 2u), idesc_corr);
          LM_PROF_ADD(10);   // issuing the first two k-steps of the k-block (the thread blocks here when the MMA queue is full)
        }
        // ---- close the bookkeeping of this k-block, advance to the next one and wait for its barriers
        --kb_left;
        const bool chunk_end = (++kc == chunk_kb) || (kb_left == 0);
        const uint32_t tfull_cur = g.tfull0 + 8 * ((EGROUPS == 2 ? (tseq & 1u) : 0u) * NBUF + buf);
        if (chunk_end) { kc = 0; ++gc; ++cit; }
        if (++s == STAGES) { s = 0; ph ^= 1u; }
        bool has_next = true;
        if (tap == TAPS - 1) {  // the next k-block opens a channel block (possibly of the next tile)
          if (++ab == (uint32_t)NUM_A_BUFS) { ab = 0; aph ^= 1u; }
          if (last_cb) {
            has_next = !last_tile;
            kb_left = num_kb; cit = 0; ++tseq;   // (kc is 0 here: a tile's last k-block closes its chunk)
          }
          if (has_next) { LM_PROF_T0(); mbar_wait(g.afull0 + 8 * ab, aph); LM_PROF_ADD(3); }
        }
        if (has_next) { LM_PROF_T0(); mbar_wait(g.full0 + 8 * s, ph); LM_PROF_ADD(4); }
        // ---- rest of the burst, then the releases
        {
          LM_PROF_T0();
#pragma unroll
          for (int k = 2; k < ROW_BYTES / 32; ++k) {
            const uint32_t ko = (uint32_t)(k * 2);  // one MMA k-step = 32 B along K (16 fp16), >>4
            umma_f16_c<true>(d_tmem, hi_a | (alo + ko), hi_b | (blo + ko), idesc_wide);
            if (!(LM_EXP & 1)) umma_f16_c<true>(d_tmem + BN, hi_a | (alo + A_PLANE + ko), hi_b | (blo + ko), idesc_corr);
          }
          LM_PROF_ADD(11);   // the other two k-steps
          {
            LM_PROF_T0();
            umma_commit(g.empty0 + 8 * s_cur);           // weight stage consumed
            if (chunk_end) umma_commit(tfull_cur);       // chunk complete -> the tile's epilogue group may drain it
            LM_PROF_ADD(12);
          }
        }
        if (tap == TAPS - 1) umma_commit(g.aempty0 + 8 * ab_cur);  // arrives once the MMAs on the buffer have retired
        // the accumulator slot of the next chunk is awaited LAST: with a two-slot ring it is the one hand-shake that
        // regularly blocks (the epilogue drains chunk i-1 while chunk i executes), and blocking in the middle of the
        // burst would leave the tensor pipe with half a k-block queued (measured: 8 % slower on the BN = 128 layers)
        if (has_next && kc == 0) { LM_PROF_T0(); mbar_wait(g.tempty0 + 8 * (gc % NBUF), (((gc / NBUF) & 1u) ^ 1u)); LM_PROF_ADD(2); }
      }
    }
  }
#ifdef LM_CONV_PROFILE
  atomicAdd(&g_conv_prof[5], (unsigned long long)(clock64() - prof_issue_t0));   // the issuer's whole loop (waits included)
#endif
}

template <int BN>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
               const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmOut,
               const __grid_constant__ CUtensorMap tmPool, const ConvParams p) {
  using C = Cfg<BN>;
  constexpr int STAGES = C::STAGES;
  constexpr int NBUF = C::NBUF;
  constexpr int EGROUPS = C::EGROUPS;

  extern __shared__ __align__(1024) uint8_t smem[];   // layout: Cfg<BN> (conv_tc_common.cuh); no static shared memory
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::OFF_BARS);
  uint32_t& tmem_base_s = *reinterpret_cast<uint32_t*>(smem + C::OFF_TMEM);
  float* s_head_w = reinterpret_cast<float*>(smem + C::OFF_HEAD);          // present for BN = 64 only (kModeHead)
  float* s_head_b = s_head_w + MAX_CLASSES * 64;

  const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[STAGES]);
  const uint32_t tfull0 = smem_u32(&bars[2 * STAGES]), tempty0 = smem_u32(&bars[2 * STAGES + EGROUPS * NBUF]);
  const uint32_t afull0 = smem_u32(&bars[2 * STAGES + (EGROUPS + 1) * NBUF]), aempty0 = afull0 + 8 * NUM_A_BUFS;
  uint8_t* smem_b = smem + C::OFF_B;
  uint8_t* smem_out = smem + C::OFF_STG;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int tiles_x = p.W / TILE_W, tiles_img = tiles_x * (p.H / TILE_H);
  const int n_tiles = p.Cout / BN;
  const int total_tiles = p.N * tiles_img * n_tiles;
  const int first_tile = (int)blockIdx.x, tile_step = (int)gridDim.x;   // persistent CTAs walk the tiles round-robin
  const int taps = p.taps;
  const int num_cb = (p.C0 + p.C1) / BK;
  const int num_kb = num_cb * taps;
  const int a_plane_bytes = taps == 9 ? A_PLANE_BYTES_3x3 : A_PLANE_BYTES_1x1;
  const int halo = taps == 9 ? 1 : 0;
  const int chunk_kb = p.chunk_kb;
  const int num_chunks = (num_kb + chunk_kb - 1) / chunk_kb;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
    for (int s = 0; s < NUM_A_BUFS; ++s) { mbar_init(afull0 + 8 * s, 1); mbar_init(aempty0 + 8 * s, 1); }
    for (int b = 0; b < EGROUPS * NBUF; ++b) mbar_init(tfull0 + 8 * b, 1);
    for (int b = 0; b < NBUF; ++b) mbar_init(tempty0 + 8 * b, NUM_EPI_THREADS / 32 / EGROUPS);
    fence_mbar_init();
    tma_prefetch_desc(&tmA0); tma_prefetch_desc(&tmA1); tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmOut); tma_prefetch_desc(&tmPool);
  }
  if (warp == 2) tmem_alloc(smem_u32(&tmem_base_s), C::TMEM_COLS);
  if (BN == 64 && p.mode == kModeHead) {
    for (int i = threadIdx.x; i < p.K * 64; i += NUM_THREADS) s_head_w[i] = p.head_w[i];
    if (threadIdx.x < p.K) s_head_b[threadIdx.x] = p.head_b[threadIdx.x];
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
#ifdef LM_CONV_PROFILE
  const long long prof_kernel_t0 = clock64();
#endif

  // Both single-issuer roles run as warp-uniform loops (all 32 lanes execute the control flow and poll the
  // barriers, one elected lane issues the TMA / MMA / commit): loop state then lives in uniform registers
  // and the issue thread is not throttled by divergent-code bookkeeping.
  // Register reallocation (setmaxnreg): warps 0-3 (producer, issuer, TMEM allocator) give registers to the two epilogue
  // warpgroups, whose chunk drains hold 3 x 64 fp32 values per thread: 128 x kRegsLow + 256 x kRegsHigh <= 384 x 168.
  // Each branch starts with its warpgroups' setmaxnreg and the branches only meet again at the kernel's last barrier.
  if (warp >= EPI_WARP0) {
    setmaxnreg_inc<kRegsHigh>();
    // ------------------------------------------------------------------ epilogue warps
    conv_epilogue_warps<BN>(p, &tmOut, &tmPool, tmem_base, tfull0, tempty0, smem_out, reinterpret_cast<float*>(smem + C::OFF_CONST), s_head_w, s_head_b,
                            first_tile, total_tiles, tile_step, num_chunks);
    tc_fence_before();
    __syncthreads();   // the kernel's last barrier (the other warps arrive at it from their own branch)
    return;
  } else {
    setmaxnreg_dec<kRegsLow>();
  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    uint32_t s = 0, ph = 0, ab = 0, aph = 0;
    const uint32_t a_tx = 2u * (uint32_t)a_plane_bytes;
    for (int tile = first_tile; tile < total_tiles; tile += tile_step) {
      const TileCoord t = decode_tile(tile, n_tiles, tiles_x, tiles_img, BN);
      int c = 0;
      for (int cb = 0; cb < num_cb; ++cb, c += BK) {
        // the activation patch (+ halo) of this channel block, both planes, once for all taps
        { LM_PROF_T0(); mbar_wait(aempty0 + 8 * ab, aph ^ 1); if (lane == 0) LM_PROF_ADD(0); }
        if (elect_one()) {
          mbar_arrive_expect_tx(afull0 + 8 * ab, a_tx);
          const uint32_t dst = smem_u32(smem) + ab * A_BUF_BYTES;
          if (c < p.C0) tma_load_5d(dst, &tmA0, afull0 + 8 * ab, c, t.x0 - halo, t.y0 - halo, 0, t.n);
          else          tma_load_5d(dst, &tmA1, afull0 + 8 * ab, c - p.C0, t.x0 - halo, t.y0 - halo, 0, t.n);
        }
        __syncwarp();
        if (++ab == NUM_A_BUFS) { ab = 0; aph ^= 1; }
        for (int tap = 0; tap < taps; ++tap) {
          { LM_PROF_T0(); mbar_wait(empty0 + 8 * s, ph ^ 1); if (lane == 0) LM_PROF_ADD(1); }
          if (elect_one()) {
            if ((LM_EXP & 32) && (tile != first_tile || cb > 0 || tap >= STAGES)) {
              mbar_arrive(full0 + 8 * s);  // ablation: reuse whatever the stage holds
            } else {
              mbar_arrive_expect_tx(full0 + 8 * s, C::STAGE_BYTES);
              tma_load_4d(smem_u32(smem_b) + s * C::STAGE_BYTES, &tmB, full0 + 8 * s, c, t.n0, tap, 0);
            }
          }
          __syncwarp();
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (one lane)
    // ncu (profiles/r01_ncu_conv_issuer.md) showed the previous warp-uniform issue loops spending ~60 % of their
    // time in per-k-block bookkeeping (~150 scalar instructions at ~8 cycles each for a lone warp), with the tensor
    // pipe idle meanwhile.  The loop therefore runs in ONE lane, the nine taps are unrolled with compile-time
    // descriptor offsets, and the state per k-block is a ring index, a phase bit and a chunk counter.
    if (elect_one()) {  // (elect.sync, not lane == 0: the compiler then knows the region is single-lane and
                        //  feeds the MMA's uniform-register operands without per-lane broadcast loops)
      IssueArgs ia;
      ia.first_tile = first_tile; ia.total_tiles = total_tiles; ia.tile_step = tile_step;
      ia.num_cb = num_cb; ia.chunk_kb = chunk_kb; ia.tmem_base = tmem_base;
      ia.smem_a = smem_u32(smem); ia.smem_b = smem_u32(smem_b);
      ia.full0 = full0; ia.empty0 = empty0; ia.tfull0 = tfull0; ia.tempty0 = tempty0; ia.afull0 = afull0; ia.aempty0 = aempty0;
      // Layers whose tiles are ONE channel block deep (64 input channels: 9 k-blocks per tile) run the nine taps as a real
      // loop instead of unrolled: these are the layers whose epilogue warps are busy most of the time, and the unrolled
      // loop's 16 KB of straight-line code then competes with the epilogue's for instruction fetch - measured -22 % / -16 %
      // on down0.block3 / up3.block3+head, while the 18-k-block up3.block0 is 8 % FASTER unrolled (profiles/r02_call7_*).
      if (taps != 9) mma_issue_loop<BN, 1, true>(ia);
      else if (BN == 64 && num_cb == 1) mma_issue_loop<BN, 9, false>(ia);
      else mma_issue_loop<BN, 9, true>(ia);
    }
    __syncwarp();
  }
  }
  tc_fence_before();
  __syncthreads();
#ifdef LM_CONV_PROFILE
  if (threadIdx.x == 0) atomicAdd(&g_conv_prof[9], (unsigned long long)(clock64() - prof_kernel_t0));
#endif
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qres) != cudaSuccess) return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(f);
  }
  return fn;
}

constexpr CUtensorMapDataType kOpType = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;

int encode(CUtensorMap* m, CUtensorMapDataType dtype, const void* base, int rank, const cuuint64_t* dims,
           const cuuint64_t* strides, const cuuint32_t* box) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return -1;
  cuuint32_t es[5] = {1, 1, 1, 1, 1};
  CUresult r = fn(m, dtype, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box,
                  es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)r;
}

int make_act_map(CUtensorMap* m, const void* base, int n_cap, int H, int W, int Cch, int taps) {
  const cuuint64_t E = kOpBytes;
  cuuint64_t dims[5] = {(cuuint64_t)Cch, (cuuint64_t)W, (cuuint64_t)H, 2, (cuuint64_t)n_cap};
  cuuint64_t strides[4] = {(cuuint64_t)Cch * E, (cuuint64_t)W * Cch * E, (cuuint64_t)H * W * Cch * E,
                           (cuuint64_t)2 * H * W * Cch * E};
  const cuuint32_t halo = taps == 9 ? 2 : 0;
  cuuint32_t box[5] = {BK, TILE_W + halo, TILE_H + halo, 2, 1};
  return encode(m, kOpType, base, 5, dims, strides, box);
}

}  // namespace

int make_conv_maps(ConvMaps* maps, const void* src0, const void* src1, const void* weights,
                   const ConvParams& p, int n_capacity) {
  const cuuint64_t E = kOpBytes;
  if (p.H % TILE_H || p.W % TILE_W || p.C0 % BK || p.C1 % BK || (p.taps != 1 && p.taps != 9)) return -2;
  const int BN = conv_tile_n(p.Cout);
  if (p.Cout % BN) return -3;
  int r = make_act_map(&maps->a0, src0, n_capacity, p.H, p.W, p.C0, p.taps);
  if (r) return r;
  r = (p.C1 > 0) ? make_act_map(&maps->a1, src1, n_capacity, p.H, p.W, p.C1, p.taps)
                 : make_act_map(&maps->a1, src0, n_capacity, p.H, p.W, p.C0, p.taps);
  if (r) return r;
  // TMA-store maps: one epilogue warp's rows per store
  if (p.mode == kModeReluBn || p.mode == kModeReluBnPool) {
    cuuint64_t od[5] = {(cuuint64_t)p.Cout, (cuuint64_t)p.W, (cuuint64_t)p.H, 2, (cuuint64_t)n_capacity};
    cuuint64_t os[4] = {(cuuint64_t)p.Cout * E, (cuuint64_t)p.W * p.Cout * E, (cuuint64_t)p.H * p.W * p.Cout * E,
                        (cuuint64_t)2 * p.H * p.W * p.Cout * E};
    cuuint32_t ob[5] = {BK, TILE_W, 4, 1, 1};  // one epilogue warp: BK channels (128 B) x 8 x 4 pixels of one plane
    r = encode(&maps->out, kOpType, p.out, 5, od, os, ob);
    if (r) return r;
  } else if (p.mode == kModeLinear) {
    cuuint64_t od[4] = {(cuuint64_t)p.Cout, (cuuint64_t)p.W, (cuuint64_t)p.H, (cuuint64_t)n_capacity};
    cuuint64_t os[3] = {(cuuint64_t)p.Cout * 4, (cuuint64_t)p.W * p.Cout * 4, (cuuint64_t)p.H * p.W * p.Cout * 4};
    cuuint32_t ob[4] = {F32_ROW_CH, TILE_W, 4, 1};
    r = encode(&maps->out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, p.out, 4, od, os, ob);
    if (r) return r;
  } else {
    maps->out = maps->a0;
  }
  if (p.mode == kModeReluBnPool) {
    const int Hp = p.H / 2, Wp = p.W / 2;
    cuuint64_t od[5] = {(cuuint64_t)p.Cout, (cuuint64_t)Wp, (cuuint64_t)Hp, 2, (cuuint64_t)n_capacity};
    cuuint64_t os[4] = {(cuuint64_t)p.Cout * E, (cuuint64_t)Wp * p.Cout * E, (cuuint64_t)Hp * Wp * p.Cout * E,
                        (cuuint64_t)2 * Hp * Wp * p.Cout * E};
    cuuint32_t ob[5] = {BK, TILE_W / 2, 2, 1, 1};
    r = encode(&maps->pool, kOpType, p.out_pool, 5, od, os, ob);
    if (r) return r;
  } else {
    maps->pool = maps->a0;
  }
  const int Cin = p.C0 + p.C1;
  cuuint64_t dims[4] = {(cuuint64_t)Cin, (cuuint64_t)p.Cout, (cuuint64_t)p.taps, 2};
  cuuint64_t strides[3] = {(cuuint64_t)Cin * E, (cuuint64_t)p.Cout * Cin * E, (cuuint64_t)p.taps * p.Cout * Cin * E};
  cuuint32_t box[4] = {BK, (cuuint32_t)BN, 1, 2};
  return encode(&maps->b, kOpType, weights, 4, dims, strides, box);
}

template <int BN>
static int launch_impl(const ConvMaps& maps, const ConvParams& p, int num_sms, cudaStream_t stream) {
  // the opt-in to > 48 KB of dynamic shared memory is a per-device function attribute
  static std::atomic<unsigned long long> attr_set_mask{0ull};  // engines of several host threads may launch concurrently
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return -9;
  if (!((attr_set_mask.load(std::memory_order_acquire) >> dev) & 1ull)) {
    cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Cfg<BN>::DYN_SMEM);
    if (e != cudaSuccess) return (int)e;
    attr_set_mask.fetch_or(1ull << dev, std::memory_order_release);
  }
  const int total = p.N * (p.H / TILE_H) * (p.W / TILE_W) * (p.Cout / BN);
  const int grid = total < num_sms ? total : num_sms;
  conv_tc_kernel<BN><<<grid, NUM_THREADS, Cfg<BN>::DYN_SMEM, stream>>>(maps.a0, maps.a1, maps.b, maps.out, maps.pool, p);
  return (int)cudaGetLastError();
}

#ifdef LM_CONV_PROFILE
void conv_prof_reset() { unsigned long long z[16] = {}; cudaMemcpyToSymbol(g_conv_prof, z, sizeof(z)); }
void conv_prof_read(unsigned long long* out) { cudaMemcpyFromSymbol(out, g_conv_prof, 16 * sizeof(unsigned long long)); }
#endif

// Sets the kernels' > 48 KB dynamic shared-memory opt-in on the current device (lm_create calls it, so that no launch -
// in particular none inside a CUDA-graph capture - has to).
int conv_tc_prepare() {
  cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<128>::DYN_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<64>::DYN_SMEM);
  return (int)e;
}

int launch_conv_tc(const ConvMaps& maps, const ConvParams& p, int num_sms, cudaStream_t stream) {
  if (p.mode == kModeHead && (p.Cout != 64 || p.K > MAX_CLASSES)) return -4;
  if (p.chunk_kb < 1) return -5;
  return conv_tile_n(p.Cout) == 128 ? launch_impl<128>(maps, p, num_sms, stream)
                                    : launch_impl<64>(maps, p, num_sms, stream);
}

}  // namespace lm
