// C-ABI engine (include/lungmask_b200.h): owns the device memory, the folded / split weights, the per-layer
// TMA descriptors and the kernel sequence that replaces LMInferer._inference (lungmask/mask.py:141-210).
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>

#include "../../include/lungmask_b200.h"
#include "conv_tc.cuh"
#include "forward_misc.cuh"
#include "postproc.cuh"
#include "preproc.cuh"
#include "shard.cuh"

using namespace lm;

namespace lm_impl {

thread_local std::string g_err;
thread_local unsigned g_fail_serial = 0;   // bumped by every fail(): RC() keeps a callee's own message instead of replacing it
int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  ++g_fail_serial;
  return code ? code : -1;
}
#define CU(x)                                                                                         \
  do {                                                                                                \
    cudaError_t e_ = (x);                                                                             \
    if (e_ != cudaSuccess) return fail((int)e_, "%s failed: %s (%s:%d)", #x, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)
#define RC(x)                                                                            \
  do {                                                                                   \
    const unsigned serial_ = g_fail_serial;                                              \
    int r_ = (x);                                                                        \
    if (r_ && serial_ != g_fail_serial) return r_; /* the callee described the failure */ \
    if (r_) {                                                                            \
      const char* m_ = (r_ > 0 && r_ < 1000) ? cudaGetErrorString((cudaError_t)r_) : ""; \
      return fail(r_, "%s failed with code %d %s (%s:%d)", #x, r_, m_, __FILE__, __LINE__); \
    }                                                                                    \
  } while (0)

constexpr int R = LM_NET_RES;

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  int reserve(size_t want) {
    if (want <= n) return 0;
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
    cudaError_t e = cudaMalloc(&p, want * sizeof(T));
    if (e != cudaSuccess) return (int)e;
    n = want;
    return 0;
  }
  void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
};

// One convolution of the network in execution order.
struct LayerSpec {
  int level;      // spatial level: resolution 256 >> level
  int C0, C1, Cout, taps, mode;
  int src0, src1, dst, dst_pool;  // activation buffer ids (-1 = none)
};

// Activation buffers (ids).  "S" = split planes [N][2][H][W][C], "L" = single fp32 plane [N][H][W][C].
enum Act {
  A0, S0, P0, A1, S1, P1, A2, S2, P2, A3, S3, P3, A4, B4,  // encoder
  L0, U0, C0_, E0, L1, U1, C1_, E1, L2, U2, C2_, E2, L3, U3, C3_,  // decoder
  NUM_ACT
};
struct ActSpec { int level, C, split; };
const ActSpec ACT[NUM_ACT] = {
    {0, 64, 1}, {0, 64, 1}, {1, 64, 1}, {1, 128, 1}, {1, 128, 1}, {2, 128, 1}, {2, 256, 1}, {2, 256, 1}, {3, 256, 1},
    {3, 512, 1}, {3, 512, 1}, {4, 512, 1}, {4, 1024, 1}, {4, 1024, 1},
    {4, 512, 0}, {3, 512, 1}, {3, 512, 1}, {3, 512, 1}, {3, 256, 0}, {2, 256, 1}, {2, 256, 1}, {2, 256, 1},
    {2, 128, 0}, {1, 128, 1}, {1, 128, 1}, {1, 128, 1}, {1, 64, 0}, {0, 64, 1}, {0, 64, 1}};

constexpr int RANGE_STRIDE = NUM_ACT + 1;  // range flags per weight slot: one per activation tensor + one for the weights

// The 21 tensor-core convolutions (the stem 1->64 runs on CUDA cores). Order = execution order = blob order
// for the 3x3 layers (the four 1x1 "up" layers come after them in the blob, see lungmask_b200.h).
const LayerSpec LAYERS[] = {
    {0, 64, 0, 64, 9, kModeReluBnPool, A0, -1, S0, P0},      // down_path.0.block.3
    {1, 64, 0, 128, 9, kModeReluBn, P0, -1, A1, -1},         // down_path.1.block.0
    {1, 128, 0, 128, 9, kModeReluBnPool, A1, -1, S1, P1},    // down_path.1.block.3
    {2, 128, 0, 256, 9, kModeReluBn, P1, -1, A2, -1},        // down_path.2.block.0
    {2, 256, 0, 256, 9, kModeReluBnPool, A2, -1, S2, P2},    // down_path.2.block.3
    {3, 256, 0, 512, 9, kModeReluBn, P2, -1, A3, -1},        // down_path.3.block.0
    {3, 512, 0, 512, 9, kModeReluBnPool, A3, -1, S3, P3},    // down_path.3.block.3
    {4, 512, 0, 1024, 9, kModeReluBn, P3, -1, A4, -1},       // down_path.4.block.0
    {4, 1024, 0, 1024, 9, kModeReluBn, A4, -1, B4, -1},      // down_path.4.block.3
    {4, 1024, 0, 512, 1, kModeLinear, B4, -1, L0, -1},       // up_path.0.up.1 (below the upsample)
    {3, 512, 512, 512, 9, kModeReluBn, U0, S3, C0_, -1},     // up_path.0.conv_block.block.0  cat([up, bridge])
    {3, 512, 0, 512, 9, kModeReluBn, C0_, -1, E0, -1},       // up_path.0.conv_block.block.3
    {3, 512, 0, 256, 1, kModeLinear, E0, -1, L1, -1},        // up_path.1.up.1
    {2, 256, 256, 256, 9, kModeReluBn, U1, S2, C1_, -1},
    {2, 256, 0, 256, 9, kModeReluBn, C1_, -1, E1, -1},
    {2, 256, 0, 128, 1, kModeLinear, E1, -1, L2, -1},        // up_path.2.up.1
    {1, 128, 128, 128, 9, kModeReluBn, U2, S1, C2_, -1},
    {1, 128, 0, 128, 9, kModeReluBn, C2_, -1, E2, -1},
    {1, 128, 0, 64, 1, kModeLinear, E2, -1, L3, -1},         // up_path.3.up.1
    {0, 64, 64, 64, 9, kModeReluBn, U3, S0, C3_, -1},
    {0, 64, 0, 64, 9, kModeHead, C3_, -1, -1, -1},           // up_path.3.conv_block.block.3 + last + LogSoftmax + argmax
};
constexpr int NUM_LAYERS = sizeof(LAYERS) / sizeof(LAYERS[0]);
// upsample steps: after layer index -> (src L buffer, dst U buffer)
struct UpSpec { int after_layer, src, dst; };
const UpSpec UPS[4] = {{9, L0, U0}, {12, L1, U1}, {15, L2, U2}, {18, L3, U3}};

struct LayerWeights {
  float w_scale = 1.f;  // power of two: the planes hold w * w_scale, normalised to max |w * w_scale| in (2^14, 2^15]
  void* w = nullptr;  // op_t [2][taps][Cout][Cin] split
  float* bias = nullptr;
  float* scale = nullptr;
  float* shift = nullptr;
};
struct Slot {
  bool loaded = false;
  int K = 0;
  float *stem_w = nullptr, *stem_bias = nullptr, *stem_scale = nullptr, *stem_shift = nullptr;
  LayerWeights lw[NUM_LAYERS];
  float *head_w = nullptr, *head_b = nullptr;
  ConvMaps maps[NUM_LAYERS];
  ConvParams params[NUM_LAYERS];
  // Power-of-two scale of every split-plane activation tensor (conv_tc.cuh ConvParams::out_scale): all 1 until a value
  // of that tensor left fp16's range in some forward; then range_finish lowers the tensor's scale by 2^-8 (exactly
  // representable, no significand changes) and the forward runs again.  The state sticks to the weights it was found for.
  float act_scale[NUM_ACT];
  Slot() { for (float& s : act_scale) s = 1.f; }
};
// Tensors that feed one convolution together (virtual concat) or leave one epilogue together (block output + its
// pooled copy) share a scale: skip S_i, pooled P_i and the upsampled U_{3-i}.
int scale_group(int a) {
  switch (a) {
    case S0: case P0: case U3: return S0;
    case S1: case P1: case U2: return S1;
    case S2: case P2: case U1: return S2;
    case S3: case P3: case U0: return S3;
    default: return a;
  }
}

}  // namespace lm_impl
using namespace lm_impl;

struct lm_engine {
  int device = 0, B = 0, num_sms = 0;
  cudaStream_t st = nullptr;
  void* act[NUM_ACT] = {};  // split buffers: op_t planes; "L" buffers: fp32
  ShardView shard;             // multi-GPU slice sharding (lm_shard_*): gather blocks of all ranks
  bool shard_connected = false;
  int shard_test_slabs = 0;    // test hook (world == 1): label that many virtual slabs separately and join them
  int shard_slab_ccl = 1;      // 1: every rank labels its own slab, parents travel with the labels, boundaries are joined after
                               // the gather; 0: every rank labels the whole gathered volume
  uint32_t shard_epoch = 0;
  uint32_t* h_shard_err = nullptr;  // pinned copy of the block's error word
  int32_t* d_spare = nullptr;  // device int32[16]: spare label values computed on the device (fusion, mask.py:228)
  int* d_range = nullptr;   // device flags [LM_MAX_SLOTS][NUM_ACT + 1]: a value of activation tensor a (or, last entry, a
                            // weight) of that slot's network left the operand format's range (fp16 build: |x * scale| > 65504)
  int* h_range = nullptr;   // pinned host copy, refreshed at the end of every forward
  int range_slot = -1;      // the slot of the last forward (lm_debug_read_activation unscales with its scales)
  int range_retries = 0;
  Slot slots[LM_MAX_SLOTS];
  DevBuf<int16_t> d_vol, d_resized, d_native;
  DevBuf<uint8_t> d_lps_out, d_native_l, d_native_r;
  DevBuf<int32_t> d_boxes;
  DevBuf<uint8_t> d_labels, d_post, d_out, d_out2, d_fused, d_mask;
  DevBuf<float> d_scores, d_norm;
  DevBuf<uint8_t> d_fvol;   // float volumes (float32 / float64), raw bytes
  DevBuf<uint32_t> d_scratch;
  PostScratch post;
  cudaEvent_t ev[8] = {};
  cudaEvent_t ev_conv[2] = {};
  std::vector<cudaEvent_t> ev_pool;  // per-launch event pairs when conv timing is on
  size_t ev_used = 0;
  bool time_convs = false;
  float last_conv_ms = 0.f;
  int64_t last_conv_launches = 0;
  float last_ms[7] = {};
  int64_t launches = 0;
  // CUDA graphs of whole forwards (all waves of one volume: ~26 launches per wave), keyed by slot / buffers / slice count /
  // input type and valid for one configuration epoch (weights, options and activation scales bump it)
  struct FwdGraph { int slot; const void* in; uint8_t* labels; int S; bool f32; uint64_t epoch; cudaGraphExec_t exec; int64_t launches; };
  std::vector<FwdGraph> graphs;
  uint64_t graph_epoch = 1;
  int use_graphs = 1;     // 0: launch every kernel individually (also whenever per-launch conv timing or score taps are on)
  int64_t graph_launches = 0, graph_hits = 0;
  int chunk_kb = 1;       // k-blocks per TMEM chunk for the 64-channel layers (ring of 4 slots)
  int chunk_kb_wide = 2;  // ... for the layers with Cout >= 128 (ring of 2 slots: chunk 1 leaves the tensor pipe waiting
                          // for the drain; chunk 2 costs < 1e-5 of score accuracy there, tools/debug_gpu.py)
};

namespace {

size_t blob_floats(int K) {
  size_t n = 0;
  // 18 conv3x3 (+BN): stem + the 3x3 entries of LAYERS
  n += 64 * 1 * 9 + 64 * 5;
  for (int i = 0; i < NUM_LAYERS; ++i)
    if (LAYERS[i].taps == 9) n += (size_t)LAYERS[i].Cout * (LAYERS[i].C0 + LAYERS[i].C1) * 9 + (size_t)LAYERS[i].Cout * 5;
  for (int i = 0; i < NUM_LAYERS; ++i)
    if (LAYERS[i].taps == 1) n += (size_t)LAYERS[i].Cout * LAYERS[i].C0 + LAYERS[i].Cout;
  n += (size_t)K * 64 + K;
  return n;
}

// BatchNorm2d(eval) as torch evaluates it on CPU: invstd = 1/sqrt(var+eps); alpha = invstd*gamma; beta = b - mean*alpha
void fold_bn(const float* g, const float* b, const float* mean, const float* var, int C, std::vector<float>& scale,
             std::vector<float>& shift) {
  scale.resize(C);
  shift.resize(C);
  for (int c = 0; c < C; ++c) {
    const float invstd = 1.0f / sqrtf(var[c] + 1e-5f);
    const float alpha = invstd * g[c];
    scale[c] = alpha;
    shift[c] = b[c] - mean[c] * alpha;
  }
}

// Stream-ordered upload: every consumer runs on the engine stream (which does not synchronise with the
// legacy default stream), and a pageable cudaMemcpy may return before its DMA has landed.
int upload(float** dst, const float* src, size_t n, cudaStream_t st) {
  if (*dst == nullptr) {
    cudaError_t e = cudaMalloc(dst, n * sizeof(float));
    if (e != cudaSuccess) return (int)e;
  }
  cudaError_t e = cudaMemcpyAsync(*dst, src, n * sizeof(float), cudaMemcpyHostToDevice, st);
  if (e != cudaSuccess) return (int)e;
  return (int)cudaStreamSynchronize(st);
}

// d_in: the resized slices, int16 HU (in_f32 == false) or the normalised fp32 network input of a float volume
int forward_batch(lm_engine* e, Slot& s, const void* d_in, bool in_f32, int n, uint8_t* d_labels, float* d_scores,
                  bool time_convs) {
  int* const range = e->d_range + (size_t)(&s - e->slots) * RANGE_STRIDE;
  if (in_f32)
    RC(launch_stem_f32(static_cast<const float*>(d_in), e->act[A0], s.stem_w, s.stem_bias, s.stem_scale, s.stem_shift, n, R, R,
                       range + A0, s.act_scale[A0], e->num_sms, e->st));
  else
    RC(launch_stem(static_cast<const int16_t*>(d_in), e->act[A0], s.stem_w, s.stem_bias, s.stem_scale, s.stem_shift, n, R, R,
                   range + A0, s.act_scale[A0], e->num_sms, e->st));
  e->launches++;
  int up = 0;
  for (int i = 0; i < NUM_LAYERS; ++i) {
    ConvParams p = s.params[i];
    p.N = n;
    p.chunk_kb = (p.Cout >= 128) ? e->chunk_kb_wide : e->chunk_kb;
    const LayerSpec& L = LAYERS[i];
    p.range_flag = L.dst >= 0 ? range + L.dst : nullptr;
    p.in_unscale = 1.f / (s.act_scale[L.src0] * s.lw[i].w_scale);   // src1 (virtual concat) shares src0's scale group
    p.out_scale = (L.mode == kModeReluBn || L.mode == kModeReluBnPool) ? s.act_scale[L.dst] : 1.f;
    if (p.mode == kModeHead) { p.labels = d_labels; p.scores = d_scores; }
    if (time_convs) {
      if (e->ev_used + 2 > e->ev_pool.size()) {
        for (int k = 0; k < 64; ++k) { cudaEvent_t ev; CU(cudaEventCreate(&ev)); e->ev_pool.push_back(ev); }
      }
      cudaEventRecord(e->ev_pool[e->ev_used], e->st);
    }
    RC(launch_conv_tc(s.maps[i], p, e->num_sms, e->st));
    if (time_convs) { cudaEventRecord(e->ev_pool[e->ev_used + 1], e->st); e->ev_used += 2; }
    e->launches++;
    if (up < 4 && UPS[up].after_layer == i) {
      const ActSpec& src = ACT[UPS[up].src];
      RC(launch_upsample2x(static_cast<const float*>(e->act[UPS[up].src]), e->act[UPS[up].dst], n, R >> src.level, R >> src.level, src.C,
                           range + UPS[up].dst, s.act_scale[UPS[up].dst], e->num_sms, e->st));
      e->launches++;
      ++up;
    }
  }
  return 0;
}

int drain_conv_events(lm_engine* e) {
  float total = 0.f;
  for (size_t i = 0; i + 1 < e->ev_used; i += 2) {
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e->ev_pool[i], e->ev_pool[i + 1]));
    total += ms;
  }
  e->last_conv_ms = total;
  e->last_conv_launches = (int64_t)(e->ev_used / 2);
  e->ev_used = 0;
  return 0;
}

void drop_graphs(lm_engine* e) {
  for (auto& g : e->graphs) cudaGraphExecDestroy(g.exec);
  e->graphs.clear();
}

// Replays (or first captures) the kernel sequence of one volume's forward - every wave's stem, 21 tensor-core
// convolutions and 4 upsamples - as ONE graph launch on the engine stream.  Returns 0 when the graph was launched,
// 1 when graphs cannot be used (the caller launches the kernels one by one), < 0 on a real error.
int forward_graph(lm_engine* e, int slot, const void* d_in, int S, uint8_t* d_labels, bool in_f32) {
  Slot& s = e->slots[slot];
  for (auto& g : e->graphs) {
    if (g.slot == slot && g.in == d_in && g.labels == d_labels && g.S == S && g.f32 == in_f32 && g.epoch == e->graph_epoch) {
      CU(cudaGraphLaunch(g.exec, e->st));
      e->launches += g.launches;
      e->graph_hits++;
      return 0;
    }
  }
  if (e->graphs.size() >= 24 || (!e->graphs.empty() && e->graphs[0].epoch != e->graph_epoch)) drop_graphs(e);
  if (cudaStreamBeginCapture(e->st, cudaStreamCaptureModeRelaxed) != cudaSuccess) { cudaGetLastError(); e->use_graphs = 0; return 1; }
  const int64_t before = e->launches;
  int rc = 0;
  for (int s0 = 0; s0 < S && rc == 0; s0 += e->B) {
    const int n = S - s0 < e->B ? S - s0 : e->B;
    const void* in_wave = in_f32 ? static_cast<const void*>(static_cast<const float*>(d_in) + (size_t)s0 * R * R)
                                 : static_cast<const void*>(static_cast<const int16_t*>(d_in) + (size_t)s0 * R * R);
    rc = forward_batch(e, s, in_wave, in_f32, n, d_labels + (size_t)s0 * R * R, nullptr, false);
  }
  cudaGraph_t graph = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(e->st, &graph);
  const int64_t captured = e->launches - before;
  e->launches = before;
  if (rc != 0 || ce != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    e->use_graphs = 0;   // stay on plain launches for the rest of this engine's life
    return rc < 0 ? rc : 1;
  }
  cudaGraphExec_t exec = nullptr;
  const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ie != cudaSuccess || !exec) { cudaGetLastError(); e->use_graphs = 0; return 1; }
  e->graphs.push_back({slot, d_in, d_labels, S, in_f32, e->graph_epoch, exec, captured});
  CU(cudaGraphLaunch(exec, e->st));
  e->launches += captured;
  e->graph_launches++;
  return 0;
}

int forward_all(lm_engine* e, int slot, const void* d_in, int S, uint8_t* d_labels, float* h_scores,
                float* conv_ms, bool in_f32 = false) {
  if (slot < 0 || slot >= LM_MAX_SLOTS || !e->slots[slot].loaded) return fail(-30, "weight slot %d not loaded", slot);
  Slot& s = e->slots[slot];
  float* d_scores = nullptr;
  if (h_scores) {
    RC(e->d_scores.reserve((size_t)e->B * s.K * R * R));
    d_scores = e->d_scores.p;
  }
  const bool timing = conv_ms != nullptr || e->time_convs;
  if (e->use_graphs && !timing && !h_scores) {
    int gr = forward_graph(e, slot, d_in, S, d_labels, in_f32);
    if (gr == 0) {
      CU(cudaMemcpyAsync(e->h_range, e->d_range, LM_MAX_SLOTS * RANGE_STRIDE * sizeof(int), cudaMemcpyDeviceToHost, e->st));
      e->range_slot = slot;
      return 0;
    }
    if (gr < 0) return gr;   // gr > 0: graphs are unavailable here (capture failed) - fall through to plain launches
  }
  for (int s0 = 0; s0 < S; s0 += e->B) {
    const int n = S - s0 < e->B ? S - s0 : e->B;
    const void* in_wave = in_f32 ? static_cast<const void*>(static_cast<const float*>(d_in) + (size_t)s0 * R * R)
                                 : static_cast<const void*>(static_cast<const int16_t*>(d_in) + (size_t)s0 * R * R);
    RC(forward_batch(e, s, in_wave, in_f32, n, d_labels + (size_t)s0 * R * R, d_scores, conv_ms != nullptr || e->time_convs));
    if (h_scores) {
      CU(cudaMemcpyAsync(h_scores + (size_t)s0 * s.K * R * R, d_scores, (size_t)n * s.K * R * R * sizeof(float),
                         cudaMemcpyDeviceToHost, e->st));
      CU(cudaStreamSynchronize(e->st));
    }
  }
  CU(cudaMemcpyAsync(e->h_range, e->d_range, LM_MAX_SLOTS * RANGE_STRIDE * sizeof(int), cudaMemcpyDeviceToHost, e->st));  // read by range_finish after the caller's sync
  e->range_slot = slot;
  if (conv_ms) {  // device time of the tensor-core convolution launches alone (CUDA events on the launch stream)
    CU(cudaStreamSynchronize(e->st));
    RC(drain_conv_events(e));
    *conv_ms = e->last_conv_ms;
  }
  return 0;
}

// preprocess -> forward -> postprocess -> reshape, all device-resident. d_out: (S,H,W) uint8.
// vtype: 0 = int16 HU volume, 1 = float32, 2 = float64 (float volumes keep their dtype through the reference's
// pre-processing and normalisation; preproc.cu resize_kernel)
int inference_dev(lm_engine* e, int slot, const void* d_vol, int S, int H, int W, int flags, uint8_t* d_out, int vtype = 0) {
  const size_t nr = (size_t)S * R * R;
  RC(e->d_boxes.reserve((size_t)S * 4));
  if (vtype == 0) RC(e->d_resized.reserve(nr)); else RC(e->d_norm.reserve(nr));
  RC(e->d_labels.reserve(nr));
  RC(e->d_post.reserve(nr));
  CU(cudaEventRecord(e->ev[1], e->st));
  if (vtype == 0) {
    RC(launch_bodymask(static_cast<const int16_t*>(d_vol), S, H, W, e->d_boxes.p, nullptr, e->num_sms, e->st));
    RC(launch_resize(static_cast<const int16_t*>(d_vol), S, H, W, e->d_boxes.p, e->d_resized.p, R, R, 1, e->num_sms, e->st));
  } else {
    RC(launch_bodymask_float(d_vol, vtype == 2, S, H, W, e->d_boxes.p, nullptr, e->num_sms, e->st));
    RC(launch_resize_float(d_vol, vtype == 2, S, H, W, e->d_boxes.p, e->d_norm.p, R, R, e->num_sms, e->st));
  }
  e->launches += 2;
  CU(cudaEventRecord(e->ev[2], e->st));
  if (vtype == 0) RC(forward_all(e, slot, e->d_resized.p, S, e->d_labels.p, nullptr, nullptr));
  else RC(forward_all(e, slot, e->d_norm.p, S, e->d_labels.p, nullptr, nullptr, true));
  CU(cudaEventRecord(e->ev[3], e->st));
  const uint8_t* masks = e->d_labels.p;
  if (!(flags & LM_FLAG_NO_POSTPROCESS)) {
    // labels out of the argmax are < K: the post-processing needs no host round trip to learn which occur
    RC(postprocess_device(e->post, e->d_labels.p, S, R, R, nullptr, 0, nullptr, 0, 3, e->slots[slot].K - 1, e->d_post.p, e->num_sms,
                          e->st, &e->launches));
    masks = e->d_post.p;
  }
  CU(cudaEventRecord(e->ev[4], e->st));
  RC(reshape_device(masks, e->d_boxes.p, S, H, W, R, R, d_out, e->num_sms, e->st));
  e->launches++;
  CU(cudaEventRecord(e->ev[5], e->st));
  return 0;
}

// After a stream synchronisation: did any activation leave the operand format's range during the forward passes?
// Returns 0 (no), 1 (yes: the offending tensors' power-of-two scales were lowered - run the forward again) or an error.
int range_finish(lm_engine* e) {
  bool any = false;
  for (int i = 0; i < LM_MAX_SLOTS * RANGE_STRIDE; ++i) any |= e->h_range[i] != 0;
  if (!any) { e->range_retries = 0; return 0; }
  cudaMemsetAsync(e->d_range, 0, LM_MAX_SLOTS * RANGE_STRIDE * sizeof(int), e->st);
  const bool give_up = ++e->range_retries > 4;
  bool weight_flag = false;
  for (int sl = 0; sl < LM_MAX_SLOTS; ++sl) {
    int* h = e->h_range + sl * RANGE_STRIDE;
    Slot& s = e->slots[sl];
    weight_flag |= h[NUM_ACT] != 0;
    h[NUM_ACT] = 0;
    for (int a = 0; a < NUM_ACT; ++a) {
      if (!h[a]) continue;
      const int g = scale_group(a);
      for (int b = 0; b < NUM_ACT; ++b) {   // one step per group and re-run, whichever members raised their flags
        if (scale_group(b) != g) continue;
        if (!give_up && s.act_scale[b] > 1e-30f) { s.act_scale[b] *= (1.f / 256.f); e->graph_epoch++; }
        h[b] = 0;
      }
    }
  }
  if (weight_flag || give_up) {
    e->range_retries = 0;
    return fail(LM_ERR_RANGE, "an activation exceeded the fp16 operand range even after rescaling by 2^-32 (|x| > 2.8e14): "
                              "the weights are not a usable network");
  }
  return 1;
}

// Enqueue-synchronise-verify: `enqueue` puts a whole call on the engine stream; after the synchronisation the
// post-processing reports whether its region tables were large enough (the region count lives on the device).  If not,
// the tables grow to the reported size and the call is enqueued once more (a label map with more than one region per 32
// voxels; never seen with a trained network).
template <typename F>
int run_checked(lm_engine* e, F&& enqueue) {
  for (int attempt = 0;; ++attempt) {
    RC(enqueue());
    CU(cudaStreamSynchronize(e->st));
    const int rr = range_finish(e);   // 1: a tensor left fp16's range, its scale was lowered -> run again (exact rescale)
    if (rr < 0) return rr;
    const int pf = postprocess_finish(e->post);
    if (!rr && !pf) return 0;
    if (attempt >= 8) return fail(-22, "the call did not settle after %d re-runs (region tables %u regions / operand range)", attempt, e->post.last_regions);
    if (pf) RC(e->post.reserve_regions(e->post.want_regions));
  }
}

void shard_release(lm_engine* e) {
  for (int p = 0; p < e->shard.world; ++p) {
    if (!e->shard.block[p]) continue;
    if (p == e->shard.rank) cudaFree(e->shard.block[p]); else cudaIpcCloseMemHandle(e->shard.block[p]);
    e->shard.block[p] = nullptr;
  }
  if (e->h_shard_err) cudaFreeHost(e->h_shard_err);
  e->h_shard_err = nullptr;
  e->shard = ShardView();
  e->shard_connected = false;
}

void shard_range(int S, int rank, int world, int* lo, int* hi) {
  const int per = (S + world - 1) / world;
  *lo = rank * per < S ? rank * per : S;
  *hi = *lo + per < S ? *lo + per : S;
}

// One volume, slices sharded over the ranks: per-slice stages on this rank's slab, results written straight into the
// rank's gather block, pushed to the peers, post-processing + reshape replicated on the gathered volume (SURVEY 8e).
// d_vol / d_out: WHOLE volume on this rank's device (only the slab of d_vol is read).
int sharded_dev(lm_engine* e, int slot, const int16_t* d_vol, int S, int H, int W, int flags, uint8_t* d_out) {
  const ShardView& v = e->shard;
  if (slot < 0 || slot >= LM_MAX_SLOTS || !e->slots[slot].loaded) return fail(-30, "weight slot %d not loaded", slot);
  int lo, hi;
  shard_range(S, v.rank, v.world, &lo, &hi);
  const size_t plane = (size_t)H * W, rr = (size_t)R * R;
  uint8_t* labels_full = v.block[v.rank] + shard_labels_offset(v.slice_cap);
  int32_t* boxes_full = reinterpret_cast<int32_t*>(v.block[v.rank] + shard_boxes_offset());
  const uint32_t epoch = ++e->shard_epoch;
  const int ns = hi - lo;
  CU(cudaEventRecord(e->ev[1], e->st));
  if (ns > 0) {
    RC(e->d_resized.reserve((size_t)ns * rr));
    RC(launch_bodymask(d_vol + (size_t)lo * plane, ns, H, W, boxes_full + 4 * (size_t)lo, nullptr, e->num_sms, e->st));
    RC(launch_resize(d_vol + (size_t)lo * plane, ns, H, W, boxes_full + 4 * (size_t)lo, e->d_resized.p, R, R, 1, e->num_sms, e->st));
    e->launches += 2;
  }
  CU(cudaEventRecord(e->ev[2], e->st));
  if (ns > 0) RC(forward_all(e, slot, e->d_resized.p, ns, labels_full + (size_t)lo * rr, nullptr, nullptr));
  CU(cudaEventRecord(e->ev[3], e->st));
  // slab-sharded 3-D labelling (SURVEY 8f-1): this rank labels its own slices (26-connected, neighbours outside the slab
  // ignored) and ships the union-find parents with the labels; after the gather every rank only links the slab
  // boundaries and flattens
  const bool want_post = !(flags & LM_FLAG_NO_POSTPROCESS);
  const bool slab_ccl = want_post && e->shard_slab_ccl;
  uint32_t* parents_full = reinterpret_cast<uint32_t*>(v.block[v.rank] + shard_parents_offset(v.slice_cap, rr));
  const int vworld = (v.world == 1 && e->shard_test_slabs > 1) ? e->shard_test_slabs : v.world;   // test hook: virtual slabs on one GPU
  if (slab_ccl) {
    if (vworld == v.world) {
      if (ns > 0) RC(ccl_slab_device(labels_full, parents_full, S, R, R, lo, hi, e->post.ccl_rule, e->num_sms, e->st, &e->launches));
    } else {
      for (int r2 = 0; r2 < vworld; ++r2) {
        int l2, h2;
        shard_range(S, r2, vworld, &l2, &h2);
        RC(ccl_slab_device(labels_full, parents_full, S, R, R, l2, h2, e->post.ccl_rule, e->num_sms, e->st, &e->launches));
      }
    }
  }
  // the collective: wait until the peers have consumed the previous volume, push the slab, wait for theirs
  RC(launch_shard_wait_done(v, epoch, e->st));
  RC(launch_shard_push(v, (size_t)lo, (size_t)hi, rr, slab_ccl, epoch, e->num_sms, e->st));
  RC(launch_shard_wait_ready(v, epoch, e->st));
  e->launches += v.world > 1 ? 3 : 0;
  const uint8_t* masks = labels_full;
  if (want_post) {
    RC(e->d_post.reserve((size_t)S * rr));
    uint32_t* parent_in = nullptr;
    if (slab_ccl) {
      int firsts[kShardMaxWorld], nbounds = 0;
      for (int r2 = 1; r2 < vworld; ++r2) {
        int l2, h2;
        shard_range(S, r2, vworld, &l2, &h2);
        if (h2 > l2) firsts[nbounds++] = l2;
      }
      RC(ccl_join_slabs_device(labels_full, parents_full, S, R, R, firsts, nbounds, e->num_sms, e->st, &e->launches));
      parent_in = parents_full;
    }
    RC(postprocess_device(e->post, labels_full, S, R, R, nullptr, 0, nullptr, 0, 3, e->slots[slot].K - 1, e->d_post.p, e->num_sms, e->st,
                          &e->launches, parent_in));
    masks = e->d_post.p;
  }
  CU(cudaEventRecord(e->ev[4], e->st));
  RC(reshape_device(masks, boxes_full, S, H, W, R, R, d_out, e->num_sms, e->st));
  RC(launch_shard_signal_done(v, epoch, e->st));
  e->launches += v.world > 1 ? 2 : 1;
  CU(cudaEventRecord(e->ev[5], e->st));
  CU(cudaMemcpyAsync(e->h_shard_err, shard_error_word(v), sizeof(uint32_t), cudaMemcpyDeviceToHost, e->st));
  return 0;
}

int shard_check(lm_engine* e) {
  if (e->h_shard_err && *e->h_shard_err) {
    *e->h_shard_err = 0;
    cudaMemsetAsync(shard_error_word(e->shard), 0, sizeof(uint32_t), e->st);
    return fail(-50, "sharded gather: a peer rank did not arrive within the wait limit (rank %d of %d)", e->shard.rank, e->shard.world);
  }
  return 0;
}

void collect_timings(lm_engine* e) {
  if (e->time_convs) drain_conv_events(e);
  for (int i = 0; i < 6; ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, e->ev[i], e->ev[i + 1]) != cudaSuccess) ms = -1.f;
    e->last_ms[i] = ms;
  }
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, e->ev[0], e->ev[6]) != cudaSuccess) ms = -1.f;
  e->last_ms[6] = ms;
}

}  // namespace

extern "C" {

const char* lm_last_error(void) { return g_err.c_str(); }
int lm_device(const lm_engine* e) { return e ? e->device : -1; }
int lm_batch_capacity(const lm_engine* e) { return e ? e->B : 0; }
size_t lm_weight_blob_floats(int n_classes) { return blob_floats(n_classes); }

static int create_resources(lm_engine* e);

int lm_create(int device, int batch_capacity, lm_engine** out) {
  if (!out) return fail(-1, "lm_create: out is NULL");
  *out = nullptr;
  if (batch_capacity < 1 || batch_capacity > 1024) return fail(-1, "lm_create: batch_capacity %d out of range", batch_capacity);
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev == 0)
    return fail(ce ? (int)ce : -2, "lm_create: no CUDA device (%s); this engine has no CPU path", cudaGetErrorString(ce));
  if (device < 0 || device >= ndev) return fail(-1, "lm_create: device %d not in [0,%d)", device, ndev);
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(-3, "lm_create: device %s is sm_%d%d; this build is sm_100a only", prop.name, prop.major, prop.minor);
  lm_engine* e = new lm_engine();
  e->device = device;
  e->B = batch_capacity;
  e->num_sms = prop.multiProcessorCount;
  const int rc = create_resources(e);
  if (rc) {  // nothing of a half-built engine survives a failed create (the message of the failing call is kept)
    const std::string msg = g_err;
    lm_destroy(e);
    cudaGetLastError();
    g_err = msg;
    return rc;
  }
  *out = e;
  return 0;
}

static int create_resources(lm_engine* e) {
  const int batch_capacity = e->B;
  if (const char* c = getenv("LM_CHUNK_KB")) { int v = atoi(c); if (v >= 1) e->chunk_kb = e->chunk_kb_wide = v; }
  if (const char* c = getenv("LM_GRAPHS")) e->use_graphs = atoi(c) != 0;
  if (const char* c = getenv("LM_CCL_RULE")) e->post.ccl_rule = atoi(c) != 0;
  if (const char* c = getenv("LM_MERGE_CTAS")) e->post.merge_ctas = atoi(c) > 0 ? atoi(c) : 0;
  if (const char* c = getenv("LM_CHUNK_KB_WIDE")) { int v = atoi(c); if (v >= 1) e->chunk_kb_wide = v; }
  RC(conv_tc_prepare());
  CU(cudaStreamCreateWithFlags(&e->st, cudaStreamNonBlocking));
  for (int i = 0; i < 8; ++i) CU(cudaEventCreate(&e->ev[i]));
  for (int i = 0; i < 2; ++i) CU(cudaEventCreate(&e->ev_conv[i]));
  for (int a = 0; a < NUM_ACT; ++a) {
    const int hw = R >> ACT[a].level;
    const size_t elems = (size_t)batch_capacity * hw * hw * ACT[a].C;
    CU(cudaMalloc(&e->act[a], ACT[a].split ? elems * 2 * sizeof(op_t) : elems * sizeof(float)));
  }
  CU(cudaMalloc(&e->d_spare, 16 * sizeof(int32_t)));
  CU(cudaMalloc(&e->d_range, LM_MAX_SLOTS * RANGE_STRIDE * sizeof(int)));
  CU(cudaMemset(e->d_range, 0, LM_MAX_SLOTS * RANGE_STRIDE * sizeof(int)));
  CU(cudaMallocHost(&e->h_range, LM_MAX_SLOTS * RANGE_STRIDE * sizeof(int)));
  memset(e->h_range, 0, LM_MAX_SLOTS * RANGE_STRIDE * sizeof(int));
  RC(e->d_scratch.reserve(64));
  return 0;
}

void lm_destroy(lm_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  cudaStreamSynchronize(e->st);
  drop_graphs(e);
  for (int a = 0; a < NUM_ACT; ++a) cudaFree(e->act[a]);
  shard_release(e);
  cudaFree(e->d_range);
  cudaFree(e->d_spare);
  cudaFreeHost(e->h_range);
  for (auto& s : e->slots) {
    cudaFree(s.stem_w); cudaFree(s.stem_bias); cudaFree(s.stem_scale); cudaFree(s.stem_shift); cudaFree(s.head_w); cudaFree(s.head_b);
    for (auto& l : s.lw) { cudaFree(l.w); cudaFree(l.bias); cudaFree(l.scale); cudaFree(l.shift); }
  }
  e->d_norm.release(); e->d_fvol.release();
  e->d_native.release(); e->d_lps_out.release(); e->d_native_l.release(); e->d_native_r.release();
  e->d_vol.release(); e->d_resized.release(); e->d_boxes.release(); e->d_labels.release(); e->d_post.release();
  e->d_out.release(); e->d_out2.release(); e->d_fused.release(); e->d_mask.release(); e->d_scores.release(); e->d_scratch.release();
  e->post.release();
  for (auto& ev : e->ev) cudaEventDestroy(ev);
  for (auto& ev : e->ev_conv) cudaEventDestroy(ev);
  for (auto& ev : e->ev_pool) cudaEventDestroy(ev);
  cudaStreamDestroy(e->st);
  delete e;
}

int lm_load_weights(lm_engine* e, int slot, const float* blob, size_t n_floats, int K) {
  if (!e || !blob) return fail(-1, "lm_load_weights: NULL argument");
  if (slot < 0 || slot >= LM_MAX_SLOTS) return fail(-1, "lm_load_weights: slot %d out of range", slot);
  if (K < 1 || K > 8) return fail(-1, "lm_load_weights: n_classes %d not in [1,8]", K);
  if (n_floats != blob_floats(K)) return fail(-1, "lm_load_weights: blob has %zu floats, expected %zu for %d classes", n_floats, blob_floats(K), K);
  CU(cudaSetDevice(e->device));
  Slot& s = e->slots[slot];
  s.loaded = false;
  s.K = K;
  e->graph_epoch++;
  const float* q = blob;
  std::vector<float> scale, shift;
  struct Tmp {  // staging buffer for one layer's OIHW weights (largest: 1024 x 1024 x 9), freed on every exit path
    float* p = nullptr;
    ~Tmp() { if (p) cudaFree(p); }
  } tmp;
  CU(cudaMalloc(&tmp.p, (size_t)1024 * 1024 * 9 * sizeof(float)));
  float* const d_tmp = tmp.p;
  // stem
  RC(upload(&s.stem_w, q, 64 * 9, e->st)); q += 64 * 9;
  RC(upload(&s.stem_bias, q, 64, e->st)); q += 64;
  fold_bn(q, q + 64, q + 128, q + 192, 64, scale, shift); q += 256;
  RC(upload(&s.stem_scale, scale.data(), 64, e->st));
  RC(upload(&s.stem_shift, shift.data(), 64, e->st));
  auto load_conv = [&](int i, bool has_bn) -> int {
    const LayerSpec& L = LAYERS[i];
    const int Cin = L.C0 + L.C1;
    const size_t nw = (size_t)L.Cout * Cin * L.taps;
    // power-of-two weight scale (undone, exactly, by ConvParams::in_unscale); non-finite weights are refused
    float wmax = 0.f;
    for (size_t k = 0; k < nw; ++k) {
      const float a = fabsf(q[k]);
      if (!(a <= 3.0e38f)) return fail(LM_ERR_RANGE, "lm_load_weights: layer %d holds a non-finite weight", i);
      wmax = a > wmax ? a : wmax;
    }
    // normalise the layer to the top of the operand format's range, max |w| * ws in (2^14, 2^15]: the hi / lo planes then
    // keep their 11 + 11 bits for every weight down to 2^-28 of the largest one, whatever the layer's magnitude
    float ws = 1.f;
    if (wmax > 0.f) {
      while (wmax * ws > 32768.f) ws *= 0.5f;
      while (wmax * ws <= 16384.f && ws < 1.0e30f) ws *= 2.f;
    }
    s.lw[i].w_scale = ws;
    CU(cudaMemcpyAsync(d_tmp, q, nw * sizeof(float), cudaMemcpyHostToDevice, e->st)); q += nw;
    if (!s.lw[i].w) CU(cudaMalloc(&s.lw[i].w, 2 * nw * sizeof(op_t)));
    RC(launch_prep_conv_weights(d_tmp, s.lw[i].w, L.Cout, Cin, L.taps, e->d_range + slot * RANGE_STRIDE + NUM_ACT, ws, e->st));
    CU(cudaStreamSynchronize(e->st));
    RC(upload(&s.lw[i].bias, q, L.Cout, e->st)); q += L.Cout;
    if (has_bn) {
      fold_bn(q, q + L.Cout, q + 2 * L.Cout, q + 3 * L.Cout, L.Cout, scale, shift); q += 4 * L.Cout;
    } else {
      scale.assign(L.Cout, 1.f); shift.assign(L.Cout, 0.f);
    }
    RC(upload(&s.lw[i].scale, scale.data(), L.Cout, e->st));
    RC(upload(&s.lw[i].shift, shift.data(), L.Cout, e->st));
    return 0;
  };
  for (int i = 0; i < NUM_LAYERS; ++i) if (LAYERS[i].taps == 9) RC(load_conv(i, true));
  for (int i = 0; i < NUM_LAYERS; ++i) if (LAYERS[i].taps == 1) RC(load_conv(i, false));
  cudaFree(s.head_w); cudaFree(s.head_b);  // sized by the class count of the previous load
  s.head_w = s.head_b = nullptr;
  RC(upload(&s.head_w, q, (size_t)K * 64, e->st)); q += (size_t)K * 64;
  RC(upload(&s.head_b, q, K, e->st)); q += K;
  if ((size_t)(q - blob) != n_floats) return fail(-1, "lm_load_weights: internal blob walk mismatch");
  int* const h_wflag = e->h_range + slot * RANGE_STRIDE + NUM_ACT;
  CU(cudaMemcpyAsync(h_wflag, e->d_range + slot * RANGE_STRIDE + NUM_ACT, sizeof(int), cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  if (*h_wflag) {
    *h_wflag = 0;
    CU(cudaMemsetAsync(e->d_range + slot * RANGE_STRIDE + NUM_ACT, 0, sizeof(int), e->st));
    return fail(LM_ERR_RANGE, "lm_load_weights: a scaled convolution weight still exceeds the fp16 operand range (internal error)");
  }
  for (float& sc : s.act_scale) sc = 1.f;   // new weights: activation ranges are unknown again
  for (int i = 0; i < NUM_LAYERS; ++i) {
    const LayerSpec& L = LAYERS[i];
    ConvParams p{};
    p.N = e->B; p.H = R >> L.level; p.W = R >> L.level; p.C0 = L.C0; p.C1 = L.C1; p.Cout = L.Cout; p.taps = L.taps;
    p.mode = L.mode; p.chunk_kb = e->chunk_kb;
    p.bias = s.lw[i].bias; p.scale = s.lw[i].scale; p.shift = s.lw[i].shift;
    p.out = L.dst >= 0 ? e->act[L.dst] : nullptr;
    p.out_pool = L.dst_pool >= 0 ? e->act[L.dst_pool] : nullptr;
    p.head_w = s.head_w; p.head_b = s.head_b; p.K = K;
    s.params[i] = p;
    int r = make_conv_maps(&s.maps[i], e->act[L.src0], L.src1 >= 0 ? e->act[L.src1] : nullptr, s.lw[i].w, p, e->B);
    if (r) return fail(r, "make_conv_maps failed for layer %d: %d", i, r);
  }
  s.loaded = true;
  return 0;
}

int lm_apply_volume_dev(lm_engine* e, int slot, const int16_t* d_vol, int S, int H, int W, int flags, uint8_t* d_out) {
  if (!e || !d_vol || !d_out) return fail(-1, "lm_apply_volume_dev: NULL argument");
  if (S < 1 || H < 1 || W < 1) return fail(-1, "lm_apply_volume_dev: empty volume (%d,%d,%d)", S, H, W);
  CU(cudaSetDevice(e->device));
  RC(run_checked(e, [&]() -> int {
    e->launches = 0;
    e->ev_used = 0;
    CU(cudaEventRecord(e->ev[0], e->st));
    RC(inference_dev(e, slot, d_vol, S, H, W, flags, d_out));
    CU(cudaEventRecord(e->ev[6], e->st));
    return 0;
  }));
  collect_timings(e);
  return 0;
}

int lm_apply_volume(lm_engine* e, int slot, const int16_t* vol, int S, int H, int W, int flags, uint8_t* out) {
  if (!e || !vol || !out) return fail(-1, "lm_apply_volume: NULL argument");
  if (S < 1 || H < 1 || W < 1) return fail(-1, "lm_apply_volume: empty volume (%d,%d,%d)", S, H, W);
  CU(cudaSetDevice(e->device));
  const size_t n = (size_t)S * H * W;
  RC(e->d_vol.reserve(n));
  RC(e->d_out.reserve(n));
  RC(run_checked(e, [&]() -> int {
    e->launches = 0;
    e->ev_used = 0;
    CU(cudaEventRecord(e->ev[0], e->st));
    CU(cudaMemcpyAsync(e->d_vol.p, vol, n * sizeof(int16_t), cudaMemcpyHostToDevice, e->st));
    RC(inference_dev(e, slot, e->d_vol.p, S, H, W, flags, e->d_out.p));
    CU(cudaMemcpyAsync(out, e->d_out.p, n, cudaMemcpyDeviceToHost, e->st));
    CU(cudaEventRecord(e->ev[6], e->st));
    return 0;
  }));
  collect_timings(e);
  return 0;
}

// LMInferer.apply with a fill model on a device-resident volume: res_l / res_r in engine buffers, result to d_final
static int fused_enqueue(lm_engine* e, int slot_base, int slot_fill, const void* d_vol, int S, int H, int W, int flags,
                         uint8_t* d_final, int vtype = 0) {
  // both inner inferences honour volume_postprocessing (mask.py:191-194); the fusion post-processing below does not
  const int inner = flags & LM_FLAG_NO_POSTPROCESS;
  const size_t n = (size_t)S * H * W;
  RC(inference_dev(e, slot_base, d_vol, S, H, W, inner, e->d_out.p, vtype));   // res_l (mask.py:225)
  RC(inference_dev(e, slot_fill, d_vol, S, H, W, inner, e->d_out2.p, vtype));  // res_r (mask.py:227)
  RC(fuse_device(e->d_out.p, e->d_out2.p, n, e->d_scratch.p, e->d_spare, e->num_sms, e->st));  // spare stays on the device
  e->launches += 3;
  // labels after the fusion are <= K_base (the spare value is max + 1 <= K_base): mask.py:232
  RC(postprocess_device(e->post, e->d_out.p, S, H, W, nullptr, 0, e->d_spare, 1, 3, e->slots[slot_base].K, d_final, e->num_sms, e->st,
                        &e->launches));
  return 0;
}

int lm_apply_fused(lm_engine* e, int slot_base, int slot_fill, const int16_t* vol, int S, int H, int W, int flags, uint8_t* out) {
  if (!e || !vol || !out) return fail(-1, "lm_apply_fused: NULL argument");
  if (S < 1 || H < 1 || W < 1) return fail(-1, "lm_apply_fused: empty volume");
  if (slot_base < 0 || slot_base >= LM_MAX_SLOTS || !e->slots[slot_base].loaded) return fail(-30, "weight slot %d not loaded", slot_base);
  CU(cudaSetDevice(e->device));
  const size_t n = (size_t)S * H * W;
  RC(e->d_vol.reserve(n));
  RC(e->d_out.reserve(n));
  RC(e->d_out2.reserve(n));
  RC(e->d_fused.reserve(n));
  RC(run_checked(e, [&]() -> int {
    e->launches = 0;
    e->ev_used = 0;
    CU(cudaEventRecord(e->ev[0], e->st));
    CU(cudaMemcpyAsync(e->d_vol.p, vol, n * sizeof(int16_t), cudaMemcpyHostToDevice, e->st));
    RC(fused_enqueue(e, slot_base, slot_fill, e->d_vol.p, S, H, W, flags, e->d_fused.p));
    CU(cudaMemcpyAsync(out, e->d_fused.p, n, cudaMemcpyDeviceToHost, e->st));
    CU(cudaEventRecord(e->ev[6], e->st));
    return 0;
  }));
  collect_timings(e);
  return 0;
}

int lm_apply_fused_dev(lm_engine* e, int slot_base, int slot_fill, const int16_t* d_vol, int S, int H, int W, int flags, uint8_t* d_out) {
  if (!e || !d_vol || !d_out) return fail(-1, "lm_apply_fused_dev: NULL argument");
  if (S < 1 || H < 1 || W < 1) return fail(-1, "lm_apply_fused_dev: empty volume");
  if (slot_base < 0 || slot_base >= LM_MAX_SLOTS || !e->slots[slot_base].loaded) return fail(-30, "weight slot %d not loaded", slot_base);
  CU(cudaSetDevice(e->device));
  const size_t n = (size_t)S * H * W;
  RC(e->d_out.reserve(n));
  RC(e->d_out2.reserve(n));
  RC(run_checked(e, [&]() -> int {
    e->launches = 0;
    e->ev_used = 0;
    CU(cudaEventRecord(e->ev[0], e->st));
    RC(fused_enqueue(e, slot_base, slot_fill, d_vol, S, H, W, flags, d_out));
    CU(cudaEventRecord(e->ev[6], e->st));
    return 0;
  }));
  collect_timings(e);
  return 0;
}

int lm_apply_volume_float(lm_engine* e, int slot, int slot_fill, const void* vol, int is_f64, int S, int H, int W, int flags,
                          uint8_t* out) {
  if (!e || !vol || !out) return fail(-1, "lm_apply_volume_float: NULL argument");
  if (S < 1 || H < 1 || W < 1) return fail(-1, "lm_apply_volume_float: empty volume");
  if (slot < 0 || slot >= LM_MAX_SLOTS || !e->slots[slot].loaded) return fail(-30, "weight slot %d not loaded", slot);
  const bool fused = slot_fill >= 0;
  if (fused && (slot_fill >= LM_MAX_SLOTS || !e->slots[slot_fill].loaded)) return fail(-30, "weight slot %d not loaded", slot_fill);
  CU(cudaSetDevice(e->device));
  const size_t n = (size_t)S * H * W, esz = is_f64 ? 8 : 4;
  RC(e->d_fvol.reserve(n * esz));
  RC(e->d_out.reserve(n));
  if (fused) { RC(e->d_out2.reserve(n)); RC(e->d_fused.reserve(n)); }
  const int vtype = is_f64 ? 2 : 1;
  RC(run_checked(e, [&]() -> int {
    e->launches = 0;
    e->ev_used = 0;
    CU(cudaEventRecord(e->ev[0], e->st));
    CU(cudaMemcpyAsync(e->d_fvol.p, vol, n * esz, cudaMemcpyHostToDevice, e->st));
    const uint8_t* result = e->d_out.p;
    if (fused) { RC(fused_enqueue(e, slot, slot_fill, e->d_fvol.p, S, H, W, flags, e->d_fused.p, vtype)); result = e->d_fused.p; }
    else RC(inference_dev(e, slot, e->d_fvol.p, S, H, W, flags, e->d_out.p, vtype));
    CU(cudaMemcpyAsync(out, result, n, cudaMemcpyDeviceToHost, e->st));
    CU(cudaEventRecord(e->ev[6], e->st));
    return 0;
  }));
  collect_timings(e);
  return 0;
}

int lm_preprocess_float(lm_engine* e, const void* vol, int is_f64, int S, int H, int W, float* normalised, int32_t* boxes) {
  if (!e || !vol || !normalised || !boxes) return fail(-1, "lm_preprocess_float: NULL argument");
  if (S < 1 || H < 1 || W < 1) return fail(-1, "lm_preprocess_float: empty volume");
  CU(cudaSetDevice(e->device));
  const size_t n = (size_t)S * H * W, esz = is_f64 ? 8 : 4, nr = (size_t)S * R * R;
  RC(e->d_fvol.reserve(n * esz));
  RC(e->d_boxes.reserve((size_t)S * 4));
  RC(e->d_norm.reserve(nr));
  CU(cudaMemcpyAsync(e->d_fvol.p, vol, n * esz, cudaMemcpyHostToDevice, e->st));
  RC(launch_bodymask_float(e->d_fvol.p, is_f64, S, H, W, e->d_boxes.p, nullptr, e->num_sms, e->st));
  RC(launch_resize_float(e->d_fvol.p, is_f64, S, H, W, e->d_boxes.p, e->d_norm.p, R, R, e->num_sms, e->st));
  CU(cudaMemcpyAsync(normalised, e->d_norm.p, nr * sizeof(float), cudaMemcpyDeviceToHost, e->st));
  CU(cudaMemcpyAsync(boxes, e->d_boxes.p, (size_t)S * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  return 0;
}

int lm_apply_volume_oriented(lm_engine* e, int slot, int slot_fill, const int16_t* vol, int n0, int n1, int n2, const int* perm,
                             const int* flip, int flags, uint8_t* out) {
  if (!e || !vol || !out || !perm || !flip) return fail(-1, "lm_apply_volume_oriented: NULL argument");
  if (n0 < 1 || n1 < 1 || n2 < 1) return fail(-1, "lm_apply_volume_oriented: empty volume");
  int seen = 0;
  for (int k = 0; k < 3; ++k) { if (perm[k] < 0 || perm[k] > 2) return fail(-1, "lm_apply_volume_oriented: perm is not a permutation"); seen |= 1 << perm[k]; }
  if (seen != 7) return fail(-1, "lm_apply_volume_oriented: perm is not a permutation");
  if (slot < 0 || slot >= LM_MAX_SLOTS || !e->slots[slot].loaded) return fail(-30, "weight slot %d not loaded", slot);
  const bool fused = slot_fill >= 0;
  if (fused && (slot_fill >= LM_MAX_SLOTS || !e->slots[slot_fill].loaded)) return fail(-30, "weight slot %d not loaded", slot_fill);
  CU(cudaSetDevice(e->device));
  const int dn[3] = {n0, n1, n2};
  const int dl[3] = {dn[perm[0]], dn[perm[1]], dn[perm[2]]};   // the LPS array: (slices, rows, columns) of the path
  const int fl[3] = {flip[0] != 0, flip[1] != 0, flip[2] != 0};
  const size_t n = (size_t)n0 * n1 * n2;
  RC(e->d_native.reserve(n));
  RC(e->d_vol.reserve(n));
  RC(e->d_lps_out.reserve(n));
  RC(e->d_native_l.reserve(n));
  if (fused) { RC(e->d_native_r.reserve(n)); RC(e->d_fused.reserve(n)); }
  RC(run_checked(e, [&]() -> int {
    e->launches = 0;
    e->ev_used = 0;
    CU(cudaEventRecord(e->ev[0], e->st));
    CU(cudaMemcpyAsync(e->d_native.p, vol, n * sizeof(int16_t), cudaMemcpyHostToDevice, e->st));
    RC(launch_orient_i16(e->d_native.p, e->d_vol.p, dl, perm, fl, 1, e->num_sms, e->st));            // sitk.DICOMOrient(image, "LPS"), mask.py:163
    const int inner = fused ? (flags & LM_FLAG_NO_POSTPROCESS) : flags;
    RC(inference_dev(e, slot, e->d_vol.p, dl[0], dl[1], dl[2], inner, e->d_lps_out.p));
    RC(launch_orient_u8(e->d_lps_out.p, e->d_native_l.p, dl, perm, fl, 0, e->num_sms, e->st));       // back, mask.py:204-208
    e->launches += 2;
    const uint8_t* result = e->d_native_l.p;
    if (fused) {   // the fusion and its post-processing work on the NATIVE-orientation results (mask.py:225-232)
      RC(inference_dev(e, slot_fill, e->d_vol.p, dl[0], dl[1], dl[2], inner, e->d_lps_out.p));
      RC(launch_orient_u8(e->d_lps_out.p, e->d_native_r.p, dl, perm, fl, 0, e->num_sms, e->st));
      RC(fuse_device(e->d_native_l.p, e->d_native_r.p, n, e->d_scratch.p, e->d_spare, e->num_sms, e->st));
      e->launches += 4;
      RC(postprocess_device(e->post, e->d_native_l.p, n0, n1, n2, nullptr, 0, e->d_spare, 1, 3, e->slots[slot].K, e->d_fused.p,
                            e->num_sms, e->st, &e->launches));
      result = e->d_fused.p;
    }
    CU(cudaMemcpyAsync(out, result, n, cudaMemcpyDeviceToHost, e->st));
    CU(cudaEventRecord(e->ev[6], e->st));
    return 0;
  }));
  collect_timings(e);
  return 0;
}

int lm_shard_init(lm_engine* e, int rank, int world, int max_slices) {
  if (!e) return fail(-1, "lm_shard_init: NULL engine");
  if (world < 1 || world > kShardMaxWorld || rank < 0 || rank >= world) return fail(-1, "lm_shard_init: rank %d / world %d", rank, world);
  if (max_slices < 1) return fail(-1, "lm_shard_init: max_slices < 1");
  CU(cudaSetDevice(e->device));
  CU(cudaStreamSynchronize(e->st));
  shard_release(e);
  e->shard.rank = rank; e->shard.world = world;
  const size_t per = ((size_t)max_slices + world - 1) / world;
  e->shard.slice_cap = per * world;
  e->shard.block_bytes = shard_block_bytes(e->shard.slice_cap, (size_t)R * R);
  void* p = nullptr;
  CU(cudaMalloc(&p, e->shard.block_bytes));
  e->shard.block[rank] = static_cast<uint8_t*>(p);
  CU(cudaMemset(p, 0, e->shard.block_bytes));
  CU(cudaMallocHost(&e->h_shard_err, sizeof(uint32_t)));
  *e->h_shard_err = 0;
  e->shard_epoch = 0;
  e->shard_connected = (world == 1);
  return 0;
}

size_t lm_shard_handle_bytes(void) { return sizeof(cudaIpcMemHandle_t); }

int lm_shard_export(lm_engine* e, void* handle_out) {
  if (!e || !handle_out) return fail(-1, "lm_shard_export: NULL argument");
  if (!e->shard.block[e->shard.rank]) return fail(-51, "lm_shard_export: call lm_shard_init first");
  CU(cudaSetDevice(e->device));
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, e->shard.block[e->shard.rank]));
  memcpy(handle_out, &h, sizeof(h));
  return 0;
}

int lm_shard_connect(lm_engine* e, const void* handles) {
  if (!e || !handles) return fail(-1, "lm_shard_connect: NULL argument");
  if (!e->shard.block[e->shard.rank]) return fail(-51, "lm_shard_connect: call lm_shard_init first");
  CU(cudaSetDevice(e->device));
  const uint8_t* hb = static_cast<const uint8_t*>(handles);
  for (int p = 0; p < e->shard.world; ++p) {
    if (p == e->shard.rank || e->shard.block[p]) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, hb + (size_t)p * sizeof(h), sizeof(h));
    void* ptr = nullptr;
    CU(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    e->shard.block[p] = static_cast<uint8_t*>(ptr);
  }
  e->shard_connected = true;
  return 0;
}

int lm_shard_labels(lm_engine* e, void** d_boxes, void** d_labels, size_t* slice_cap) {
  if (!e) return fail(-1, "lm_shard_labels: NULL engine");
  if (!e->shard.block[e->shard.rank]) return fail(-51, "lm_shard_labels: call lm_shard_init first");
  if (d_boxes) *d_boxes = e->shard.block[e->shard.rank] + shard_boxes_offset();
  if (d_labels) *d_labels = e->shard.block[e->shard.rank] + shard_labels_offset(e->shard.slice_cap);
  if (slice_cap) *slice_cap = e->shard.slice_cap;
  return 0;
}

int lm_apply_volume_sharded_dev(lm_engine* e, int slot, const int16_t* d_vol, int S, int H, int W, int flags, uint8_t* d_out) {
  if (!e || !d_vol || !d_out) return fail(-1, "lm_apply_volume_sharded_dev: NULL argument");
  if (S < 1 || H < 1 || W < 1) return fail(-1, "lm_apply_volume_sharded_dev: empty volume");
  if (!e->shard_connected) return fail(-51, "lm_apply_volume_sharded_dev: call lm_shard_init / lm_shard_connect first");
  if ((size_t)S > e->shard.slice_cap) return fail(-52, "lm_apply_volume_sharded_dev: %d slices exceed the gather capacity %zu", S, e->shard.slice_cap);
  CU(cudaSetDevice(e->device));
  RC(run_checked(e, [&]() -> int {
    e->launches = 0;
    e->ev_used = 0;
    CU(cudaEventRecord(e->ev[0], e->st));
    RC(sharded_dev(e, slot, d_vol, S, H, W, flags, d_out));
    CU(cudaEventRecord(e->ev[6], e->st));
    return 0;
  }));
  collect_timings(e);
  return shard_check(e);
}

int lm_apply_volume_sharded(lm_engine* e, int slot, const int16_t* vol, int S, int H, int W, int flags, uint8_t* out) {
  if (!e || !vol) return fail(-1, "lm_apply_volume_sharded: NULL argument");
  if (S < 1 || H < 1 || W < 1) return fail(-1, "lm_apply_volume_sharded: empty volume");
  if (!e->shard_connected) return fail(-51, "lm_apply_volume_sharded: call lm_shard_init / lm_shard_connect first");
  if ((size_t)S > e->shard.slice_cap) return fail(-52, "lm_apply_volume_sharded: %d slices exceed the gather capacity %zu", S, e->shard.slice_cap);
  CU(cudaSetDevice(e->device));
  const size_t n = (size_t)S * H * W, plane = (size_t)H * W;
  RC(e->d_vol.reserve(n));
  RC(e->d_out.reserve(n));
  int lo, hi;
  shard_range(S, e->shard.rank, e->shard.world, &lo, &hi);
  RC(run_checked(e, [&]() -> int {
    e->launches = 0;
    e->ev_used = 0;
    CU(cudaEventRecord(e->ev[0], e->st));
    if (hi > lo)  // only this rank's slab crosses the PCIe bus
      CU(cudaMemcpyAsync(e->d_vol.p + (size_t)lo * plane, vol + (size_t)lo * plane, (size_t)(hi - lo) * plane * sizeof(int16_t),
                         cudaMemcpyHostToDevice, e->st));
    RC(sharded_dev(e, slot, e->d_vol.p, S, H, W, flags, e->d_out.p));
    if (out) CU(cudaMemcpyAsync(out, e->d_out.p, n, cudaMemcpyDeviceToHost, e->st));
    CU(cudaEventRecord(e->ev[6], e->st));
    return 0;
  }));
  collect_timings(e);
  return shard_check(e);
}

int lm_fuse(lm_engine* e, const uint8_t* res_l, const uint8_t* res_r, int S, int H, int W, uint8_t* fused, int* spare_value) {
  if (!e || !res_l || !res_r || !fused || !spare_value) return fail(-1, "lm_fuse: NULL argument");
  if (S < 1 || H < 1 || W < 1) return fail(-1, "lm_fuse: empty volume");
  CU(cudaSetDevice(e->device));
  const size_t n = (size_t)S * H * W;
  RC(e->d_out.reserve(n));
  RC(e->d_out2.reserve(n));
  CU(cudaMemcpyAsync(e->d_out.p, res_l, n, cudaMemcpyHostToDevice, e->st));
  CU(cudaMemcpyAsync(e->d_out2.p, res_r, n, cudaMemcpyHostToDevice, e->st));
  RC(fuse_device(e->d_out.p, e->d_out2.p, n, e->d_scratch.p, e->d_spare, e->num_sms, e->st));
  CU(cudaMemcpyAsync(fused, e->d_out.p, n, cudaMemcpyDeviceToHost, e->st));
  int32_t spare = 0;
  CU(cudaMemcpyAsync(&spare, e->d_spare, sizeof(int32_t), cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  *spare_value = (int)spare;
  return 0;
}

int lm_preprocess(lm_engine* e, const int16_t* vol, int S, int H, int W, int out_h, int out_w, int clip,
                  int16_t* resized, int32_t* boxes) {
  if (!e || !vol || !resized || !boxes) return fail(-1, "lm_preprocess: NULL argument");
  if (S < 1 || H < 1 || W < 1 || out_h < 1 || out_w < 1) return fail(-1, "lm_preprocess: empty volume");
  CU(cudaSetDevice(e->device));
  const size_t n = (size_t)S * H * W, nr = (size_t)S * out_h * out_w;
  RC(e->d_vol.reserve(n));
  RC(e->d_boxes.reserve((size_t)S * 4));
  RC(e->d_resized.reserve(nr));
  CU(cudaMemcpyAsync(e->d_vol.p, vol, n * sizeof(int16_t), cudaMemcpyHostToDevice, e->st));
  RC(launch_bodymask(e->d_vol.p, S, H, W, e->d_boxes.p, nullptr, e->num_sms, e->st));
  RC(launch_resize(e->d_vol.p, S, H, W, e->d_boxes.p, e->d_resized.p, out_h, out_w, clip, e->num_sms, e->st));
  CU(cudaMemcpyAsync(resized, e->d_resized.p, nr * sizeof(int16_t), cudaMemcpyDeviceToHost, e->st));
  CU(cudaMemcpyAsync(boxes, e->d_boxes.p, (size_t)S * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  return 0;
}

int lm_simple_bodymask(lm_engine* e, const int16_t* slice, int H, int W, uint8_t* mask) {
  if (!e || !slice || !mask) return fail(-1, "lm_simple_bodymask: NULL argument");
  if (H < 1 || W < 1) return fail(-1, "lm_simple_bodymask: empty slice");
  CU(cudaSetDevice(e->device));
  const size_t n = (size_t)H * W;
  RC(e->d_vol.reserve(n));
  RC(e->d_boxes.reserve(4));
  RC(e->d_mask.reserve(n));
  CU(cudaMemcpyAsync(e->d_vol.p, slice, n * sizeof(int16_t), cudaMemcpyHostToDevice, e->st));
  RC(launch_bodymask(e->d_vol.p, 1, H, W, e->d_boxes.p, e->d_mask.p, e->num_sms, e->st));
  CU(cudaMemcpyAsync(mask, e->d_mask.p, n, cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  return 0;
}

int lm_forward(lm_engine* e, int slot, const int16_t* resized, int S, uint8_t* labels, float* scores) {
  if (!e || !resized || !labels) return fail(-1, "lm_forward: NULL argument");
  if (S < 1) return fail(-1, "lm_forward: S < 1");
  CU(cudaSetDevice(e->device));
  const size_t nr = (size_t)S * R * R;
  RC(e->d_resized.reserve(nr));
  RC(e->d_labels.reserve(nr));
  return run_checked(e, [&]() -> int {
    CU(cudaMemcpyAsync(e->d_resized.p, resized, nr * sizeof(int16_t), cudaMemcpyHostToDevice, e->st));
    RC(forward_all(e, slot, e->d_resized.p, S, e->d_labels.p, scores, nullptr));
    CU(cudaMemcpyAsync(labels, e->d_labels.p, nr, cudaMemcpyDeviceToHost, e->st));
    return 0;
  });
}

int lm_forward_dev(lm_engine* e, int slot, const int16_t* d_resized, int S, uint8_t* d_labels, float* conv_ms) {
  if (!e || !d_resized || !d_labels) return fail(-1, "lm_forward_dev: NULL argument");
  CU(cudaSetDevice(e->device));
  return run_checked(e, [&]() -> int {
    e->launches = 0;
    e->ev_used = 0;
    return forward_all(e, slot, d_resized, S, d_labels, nullptr, conv_ms);
  });
}

int lm_postprocess(lm_engine* e, const uint8_t* labels, int S, int H, int W, const int32_t* spare, int n_spare,
                   int skip_below, uint8_t* out) {
  if (!e || !labels || !out) return fail(-1, "lm_postprocess: NULL argument");
  if (S < 1 || H < 1 || W < 1) return fail(-1, "lm_postprocess: empty volume");
  CU(cudaSetDevice(e->device));
  const size_t n = (size_t)S * H * W;
  RC(e->d_out.reserve(n));
  RC(e->d_out2.reserve(n));
  if (n_spare < 0 || n_spare > 16 || (n_spare > 0 && !spare)) return fail(-1, "lm_postprocess: n_spare %d not in [0,16]", n_spare);
  return run_checked(e, [&]() -> int {
    CU(cudaMemcpyAsync(e->d_out.p, labels, n, cudaMemcpyHostToDevice, e->st));
    int64_t launches = 0;
    // arbitrary label values: the post-processing synchronises once to learn which occur (max_label = -1)
    RC(postprocess_device(e->post, e->d_out.p, S, H, W, spare, n_spare, nullptr, 0, skip_below, -1, e->d_out2.p, e->num_sms, e->st,
                          &launches));
    CU(cudaMemcpyAsync(out, e->d_out2.p, n, cudaMemcpyDeviceToHost, e->st));
    return 0;
  });
}

int lm_keep_largest_component(lm_engine* e, const uint8_t* mask, int S, int H, int W, uint8_t* out) {
  if (!e || !mask || !out) return fail(-1, "lm_keep_largest_component: NULL argument");
  if (S < 1 || H < 1 || W < 1) return fail(-1, "lm_keep_largest_component: empty mask");
  CU(cudaSetDevice(e->device));
  const size_t n = (size_t)S * H * W;
  RC(e->d_out.reserve(n));
  RC(e->d_out2.reserve(n));
  CU(cudaMemcpyAsync(e->d_out.p, mask, n, cudaMemcpyHostToDevice, e->st));
  const int r = keep_largest_component_device(e->post, e->d_out.p, S, H, W, e->d_out2.p, e->num_sms, e->st);
  if (r == -21) return fail(-21, "lm_keep_largest_component: the mask has no foreground (the reference raises IndexError here)");
  RC(r);
  CU(cudaMemcpyAsync(out, e->d_out2.p, n, cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  return 0;
}

int lm_reshape_masks(lm_engine* e, const uint8_t* masks, int mask_h, int mask_w, const int32_t* boxes, int S, int H,
                     int W, uint8_t* out) {
  if (!e || !masks || !boxes || !out) return fail(-1, "lm_reshape_masks: NULL argument");
  if (S < 1 || H < 1 || W < 1 || mask_h < 1 || mask_w < 1) return fail(-1, "lm_reshape_masks: empty input");
  CU(cudaSetDevice(e->device));
  const size_t n = (size_t)S * H * W, nr = (size_t)S * mask_h * mask_w;
  RC(e->d_labels.reserve(nr));
  RC(e->d_boxes.reserve((size_t)S * 4));
  RC(e->d_out.reserve(n));
  CU(cudaMemcpyAsync(e->d_labels.p, masks, nr, cudaMemcpyHostToDevice, e->st));
  CU(cudaMemcpyAsync(e->d_boxes.p, boxes, (size_t)S * 4 * sizeof(int32_t), cudaMemcpyHostToDevice, e->st));
  RC(reshape_device(e->d_labels.p, e->d_boxes.p, S, H, W, mask_h, mask_w, e->d_out.p, e->num_sms, e->st));
  CU(cudaMemcpyAsync(out, e->d_out.p, n, cudaMemcpyDeviceToHost, e->st));
  CU(cudaStreamSynchronize(e->st));
  return 0;
}

int lm_debug_activation_info(int act_id, int* level, int* channels, int* split) {
  if (act_id < 0 || act_id >= NUM_ACT) return fail(-1, "activation id %d out of range", act_id);
  if (level) *level = ACT[act_id].level;
  if (channels) *channels = ACT[act_id].C;
  if (split) *split = ACT[act_id].split;
  return 0;
}

int lm_debug_read_activation(lm_engine* e, int act_id, int n, float* out) {
  if (!e || !out) return fail(-1, "lm_debug_read_activation: NULL argument");
  if (act_id < 0 || act_id >= NUM_ACT) return fail(-1, "activation id %d out of range", act_id);
  if (n < 1 || n > e->B) return fail(-1, "n out of range");
  CU(cudaSetDevice(e->device));
  const int hw = R >> ACT[act_id].level;
  const size_t per = (size_t)hw * hw * ACT[act_id].C;
  CU(cudaStreamSynchronize(e->st));
  if (!ACT[act_id].split) {
    CU(cudaMemcpy(out, e->act[act_id], (size_t)n * per * sizeof(float), cudaMemcpyDeviceToHost));
    return 0;
  }
  std::vector<op_t> tmp((size_t)n * 2 * per);
  CU(cudaMemcpy(tmp.data(), e->act[act_id], tmp.size() * sizeof(op_t), cudaMemcpyDeviceToHost));
  const float unscale = (e->range_slot >= 0 && e->range_slot < LM_MAX_SLOTS) ? 1.f / e->slots[e->range_slot].act_scale[act_id] : 1.f;
  for (int i = 0; i < n; ++i)
    for (size_t k = 0; k < per; ++k)
      out[(size_t)i * per + k] = ((float)tmp[((size_t)i * 2) * per + k] + (float)tmp[((size_t)i * 2 + 1) * per + k] * kLoUnscale) * unscale;
  return 0;
}

int lm_set_option(lm_engine* e, const char* key, int value) {
  if (!e || !key) return fail(-1, "lm_set_option: NULL argument");
  e->graph_epoch++;   // captured forwards bake the kernel choices in
  if (!strcmp(key, "graphs")) { e->use_graphs = value != 0; return 0; }
  if (!strcmp(key, "time_convs")) { e->time_convs = value != 0; e->ev_used = 0; return 0; }
  if (!strcmp(key, "post_debug_stage")) { e->post.debug_stage = value; return 0; }
  if (!strcmp(key, "chunk_kb")) { if (value < 1) return fail(-1, "chunk_kb must be >= 1"); e->chunk_kb = e->chunk_kb_wide = value; return 0; }
  if (!strcmp(key, "ccl_rule")) { e->post.ccl_rule = value != 0; return 0; }
  if (!strcmp(key, "shard_slab_ccl")) { e->shard_slab_ccl = value != 0; return 0; }
  if (!strcmp(key, "shard_test_slabs")) { if (value < 0 || value > kShardMaxWorld) return fail(-1, "shard_test_slabs out of range"); e->shard_test_slabs = value; return 0; }
  if (!strcmp(key, "merge_ctas")) { if (value < 0) return fail(-1, "merge_ctas must be >= 0"); e->post.merge_ctas = value; return 0; }
  if (!strcmp(key, "post_region_capacity")) {  // test hook: shrink / grow the region tables (exercises the overflow re-run)
    if (value < 1) return fail(-1, "post_region_capacity must be >= 1");
    CU(cudaSetDevice(e->device));
    CU(cudaStreamSynchronize(e->st));
    e->post.release_regions();
    if (e->post.cap_vox) RC(e->post.reserve_regions((uint32_t)value));
    return 0;
  }
  if (!strcmp(key, "chunk_kb_wide")) { if (value < 1) return fail(-1, "chunk_kb_wide must be >= 1"); e->chunk_kb_wide = value; return 0; }
  return fail(-1, "lm_set_option: unknown key %s", key);
}

int lm_last_conv_timing(const lm_engine* e, float* conv_ms, int64_t* conv_launches) {
  if (!e) return fail(-1, "lm_last_conv_timing: NULL engine");
  if (conv_ms) *conv_ms = e->last_conv_ms;
  if (conv_launches) *conv_launches = e->last_conv_launches;
  return 0;
}

int lm_last_timings(const lm_engine* e, float* ms7, int64_t* kernel_launches) {
  if (!e) return fail(-1, "lm_last_timings: NULL engine");
  if (ms7) memcpy(ms7, e->last_ms, sizeof(e->last_ms));
  if (kernel_launches) *kernel_launches = e->launches;
  return 0;
}

}  // extern "C"
