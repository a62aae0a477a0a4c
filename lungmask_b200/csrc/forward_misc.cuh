// CUDA-core helpers of the U-Net forward (see forward_misc.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "conv_tc.cuh"  // op_t: the operand format of the split planes

namespace lm {
// resized HU slices int16 [N][H][W] -> split planes [N][2][H][W][64]; W must be a multiple of 32 and H of 8
// (range_flag: device int set to 1 when a value leaves the operand format's range; may be nullptr)
int launch_stem(const int16_t* in, void* out, const float* w, const float* bias, const float* scale,
                const float* shift, int N, int H, int W, int* range_flag, float out_scale, int num_sms, cudaStream_t stream);
// the same convolution on an already normalised fp32 input [N][H][W] (float volumes, preproc.cuh launch_resize_float)
int launch_stem_f32(const float* in_norm, void* out, const float* w, const float* bias, const float* scale, const float* shift, int N,
                    int H, int W, int* range_flag, float out_scale, int num_sms, cudaStream_t stream);
// fp32 [N][h][w][C] -> split planes [N][2][2h][2w][C]
// (all planes are stored as value * out_scale, a power of two chosen by the engine: conv_tc.cuh ConvParams)
int launch_upsample2x(const float* in, void* out, int N, int h, int w, int C, int* range_flag, float out_scale, int num_sms,
                      cudaStream_t stream);
// OIHW fp32 -> [2][taps][Cout][Cin] hi/lo operand planes
int launch_prep_conv_weights(const float* oihw, void* out, int Cout, int Cin, int taps, int* range_flag, float w_scale,
                             cudaStream_t stream);
}  // namespace lm
