// Host-visible description of one tensor-core convolution launch (see conv_tc.cu).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

// Operand format of the tensor-core convolutions: fp16 pairs, tcgen05 kind::f16:  x = hi + lo * 2^-11, hi = fp16(x),
// lo = fp16((x - hi) * 2^11).  Both halves carry 11 significant bits (as tf32 does), every product is exact in fp32, and an
// MMA instruction covers K = 16 at the rate kind::tf32 covers K = 8: the 3-product scheme runs at twice the tf32 rate and
// moves half the bytes.  The scaled low half keeps the residuals of small values out of the fp16 subnormal range; the
// hi*lo + lo*hi accumulator is multiplied by 2^-11 when it is read.  fp16 saturates at 65504: the epilogues raise
// ConvParams::range_flag when a value leaves that range; the engine then lowers that tensor's power-of-two scale
// (ConvParams::out_scale) and runs the forward again - exact, and never a wrong mask.

namespace lm {

using op_t = __half;
constexpr float kLoScale = 2048.f, kLoUnscale = 1.f / 2048.f;
constexpr float kOpMax = 65504.f;
constexpr int kOpBytes = (int)sizeof(op_t);
constexpr int kBK = 128 / kOpBytes;  // input channels per k-block: one 128-byte swizzle row (64 fp16)

// Activation tensors feeding / produced by the tensor-core convolutions are "split planes":
//   [N][2][H][W][C] op_t, plane 0 = hi, plane 1 = lo (scaled by kLoScale), so that hi + lo * kLoUnscale
// reproduces the fp32 value to ~2^-22 and both planes are exact tensor-core operands.
// Weights are [2][taps][Cout][Cin] with the same hi / lo split.

enum ConvMode : int {
  kModeReluBn = 0,      // y = bn(relu(acc + bias))              -> split planes
  kModeReluBnPool = 1,  // as 0, plus 2x2 average of y            -> split planes at half resolution
  kModeLinear = 2,      // y = acc + bias                         -> single fp32 plane [N][H][W][C]
  kModeHead = 3,        // y as 0 (not stored); 1x1 head, log-softmax, argmax -> uint8 labels (+ scores)
};

struct ConvParams {
  int N, H, W;        // images, spatial size (input == output, zero padding 1 for 3x3)
  int C0, C1;         // channels taken from src0 / src1 (virtual concat, src0 first); C1 may be 0
  int Cout;
  int taps;           // 9 (3x3, pad 1) or 1 (1x1)
  int mode;           // ConvMode
  int chunk_kb;       // k-blocks (kBK channels x 1 tap) accumulated inside the tensor core before the
                      // partial sum is added, round-to-nearest, into fp32 registers
  const float* bias;  // [Cout]
  const float* scale; // [Cout]  folded BN:  y = relu(.) * scale + shift
  const float* shift; // [Cout]
  void* out;          // mode 0/1: op_t [N][2][H][W][Cout]; mode 2: fp32 [N][H][W][Cout]; mode 3: unused
  void* out_pool;     // mode 1: op_t [N][2][H/2][W/2][Cout]
  int* range_flag;    // set to 1 when an output leaves the operand format's range; may be nullptr
  // Power-of-two range management (exact: a power of two changes no significand).  The operand planes of a tensor hold
  // value * act_scale, weights hold w * w_scale; the epilogue multiplies the accumulator by in_unscale =
  // 1 / (act_scale(in) * w_scale) before the bias and stores y * out_scale.  All 1.0 unless the engine had to move a
  // tensor's range below fp16's 65504 (engine.cu: range_finish); 1.0 multiplications leave every bit as it was.
  float in_unscale, out_scale;
  const float* head_w;  // mode 3: [K][Cout]
  const float* head_b;  // mode 3: [K]
  int K;                // mode 3: classes (<= 8)
  uint8_t* labels;      // mode 3: [N][H][W]
  float* scores;        // mode 3: optional [N][K][H][W] log-softmax scores (nullptr to skip)
};

// Tensor maps for one launch (built once per layer by make_conv_maps).
struct ConvMaps {
  CUtensorMap a0, a1, b;
  CUtensorMap out, pool;  // TMA-store maps of the output tile (mode 0/1/2) and of the pooled tile (mode 1)
};

// Builds the TMA descriptors. src1 may be nullptr when C1 == 0. Returns 0 on success.
int make_conv_maps(ConvMaps* maps, const void* src0, const void* src1, const void* weights,
                   const ConvParams& p, int n_capacity);

// Launches the convolution on `stream`. Returns a cudaError_t value (0 = ok).
int launch_conv_tc(const ConvMaps& maps, const ConvParams& p, int num_sms, cudaStream_t stream);

// Per-device preparation (dynamic shared-memory opt-in of both kernel instantiations); returns a cudaError_t value.
int conv_tc_prepare();

// BN (output-channel tile) chosen for a given Cout.
inline int conv_tile_n(int cout) { return cout >= 128 ? 128 : 64; }

}  // namespace lm
