// CUDA-core kernels around the tensor-core convolutions of the U-Net forward:
//   * stem_kernel      normalise (mask.py:167-168) + Conv2d(1->64, 3x3, pad 1) + ReLU + BatchNorm
//                      (resunet.py:93-97 for down_path.0.block.0/2): K = 9, no tensor-core shape.
//   * upsample2x_kernel  nn.Upsample(mode='bilinear', scale_factor=2) (resunet.py:132), applied AFTER the
//                      1x1 convolution (the two commute: both are linear and the bilinear weights sum
//                      to 1), writing the hi/lo split planes the next convolution consumes.
//   * prep_conv_weights  OIHW fp32 -> [2][tap][Cout][Cin] hi/lo operand planes (one-time, at weight load).
// All are HBM-bound streaming kernels: each thread produces 16 bytes of each plane (CPT = 8 fp16 channels)
// so that every warp store instruction writes fully coalesced 128-byte runs.
#include "forward_misc.cuh"
#include "sm100_ptx.cuh"

namespace lm {
namespace {

constexpr int CPT = 16 / kOpBytes;  // channels per thread

// CPT fp32 values -> 16 bytes of the hi plane and 16 bytes of the lo plane; flags values outside the format's range
__device__ __forceinline__ void split_store(const float* v, op_t* hi_dst, op_t* lo_dst, bool& ovf) {
  uint4 h, l;
  uint32_t* ph = &h.x;
  uint32_t* pl = &l.x;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    split_f16x2(v[2 * e], v[2 * e + 1], ph[e], pl[e]);   // packed conversions: the roundings of split_f16, two values at a time
    ovf |= !(fabsf(v[2 * e]) <= kOpMax) | !(fabsf(v[2 * e + 1]) <= kOpMax);
  }
  *reinterpret_cast<uint4*>(hi_dst) = h;
  *reinterpret_cast<uint4*>(lo_dst) = l;
}

// network input of one sample, from its raw value: int16 HU -> (hu + 1024) / 1624 through the table (mask.py:167-168: float64
// division, then the cast to fp32); float volumes arrive already normalised (preproc.cu resize_kernel<float / double>)
__device__ __forceinline__ float stem_convert(int16_t raw, const float* lut) {
  int hu = raw;
  hu = hu > 600 ? 600 : hu;  // mask.py:167 (no-op after the clip in utils.py:45)
  const int i = hu + 1024;
  // mask.py:168.  Values below -1024 never come out of preprocess; for them (and for every other int16 value) the IEEE fp32
  // quotient of the two exactly representable integers equals the float64 quotient rounded to fp32
  // (tests/test_host_logic.py::test_normalisation_in_fp32_is_exact) - no double-precision division in the hot loop.
  return i >= 0 ? lut[i] : __fdiv_rn((float)i, 1624.f);
}
__device__ __forceinline__ float stem_convert(float raw, const float*) { return raw; }

// stem_kernel.  ncu / SASS of round 2's earlier versions: instruction-bound - every thread normalised its own 3 x 6 input
// window (the 8 channel-group threads of a pixel quad eight times the same one, with a double-precision division in the
// fallback path: 4700 SASS instructions per quad) and reached 1.0 - 1.4 TB/s of the 6.5 TB/s it writes at.
// Here a block owns an 8-row x 32-column tile of one image: the (8+2) x (32+2) normalised samples are built ONCE in shared
// memory (zero padding included), the 64 x 9 weights sit in shared memory too ([channel group][tap][8 channels], read as
// LDS.128 broadcasts: 18 per quad of 4 pixels), and a thread computes 8 channels of a 4-pixel quad from 18 window loads.
// Per output: fmaf over the taps 0..8 from zero, then ReLU, BN, scale.
// ncu's stall breakdown of a version that loaded each tile in front of its barrier is led by long-scoreboard (1.8 stalled warps
// per issue) and barrier (0.9) stalls at two blocks per SM; here every thread fetches its (at most two) raw samples of the NEXT
// tile into registers before it computes the current one, so the loads fly during the 2400 instructions of the compute phase
// and the fill phase is shared-memory work only.
constexpr int S3_TH = 8, S3_TW = 32, S3_PITCH = S3_TW + 2 + 2;   // tile rows / columns, padded row pitch of the input tile
template <typename IT>
__global__ void __launch_bounds__(256) stem_kernel(const IT* __restrict__ in, op_t* __restrict__ out,
                                                   const float* __restrict__ w, const float* __restrict__ bias,
                                                   const float* __restrict__ scale, const float* __restrict__ shift,
                                                   int N, int H, int W, int* __restrict__ range_flag, float out_scale) {
  static_assert(CPT == 8, "stem_kernel is written for 8 channels per thread");
  __shared__ float lut[1625];
  __shared__ __align__(16) float sw[8][9][8];                 // [channel group][tap][channel within the group]
  __shared__ __align__(16) float sc[8][3][8];                 // bias / scale / shift per channel group
  __shared__ float tile[S3_TH + 2][S3_PITCH];
  for (int i = threadIdx.x; i < 1625; i += blockDim.x) lut[i] = __fdiv_rn((float)i, 1624.f);
  for (int i = threadIdx.x; i < 64 * 9; i += blockDim.x) { const int c = i / 9, tap = i % 9; sw[c >> 3][tap][c & 7] = w[i]; }
  if (threadIdx.x < 64) {
    const int c = threadIdx.x;
    sc[c >> 3][0][c & 7] = bias[c]; sc[c >> 3][1][c & 7] = scale[c]; sc[c >> 3][2][c & 7] = shift[c];
  }
  const int tiles_x = W / S3_TW, tiles_y = H / S3_TH;
  const int tiles_img = tiles_x * tiles_y;
  const size_t plane = (size_t)H * W;
  const int cq = threadIdx.x & 7;            // channel group
  const int slot = threadIdx.x >> 3;         // 32 quad slots; the tile has 8 rows x 8 quads = 64 quads: two per slot
  bool ovf = false;
  constexpr int TILE_ELEMS = (S3_TH + 2) * (S3_TW + 2);   // 340 samples incl. the halo: at most two per thread
  static_assert(TILE_ELEMS <= 2 * 256, "two samples per thread");
  IT raw[2] = {IT(0), IT(0)};
  bool ok[2] = {false, false};
  auto fetch = [&](int tid_) {               // raw samples of tile tid_ -> registers (no conversion, nothing waited for)
    const int n_ = tid_ / tiles_img, r_ = tid_ - n_ * tiles_img;
    const int y0_ = (r_ / tiles_x) * S3_TH, x0_ = (r_ % tiles_x) * S3_TW;
    const IT* img_ = in + (size_t)n_ * plane;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int i = threadIdx.x + 256 * k;
      const int ty = i / (S3_TW + 2), tx = i - ty * (S3_TW + 2);
      const int yy = y0_ + ty - 1, xx = x0_ + tx - 1;
      ok[k] = i < TILE_ELEMS && yy >= 0 && yy < H && xx >= 0 && xx < W;
      raw[k] = ok[k] ? img_[(size_t)yy * W + xx] : IT(0);
    }
  };
  if ((int)blockIdx.x < N * tiles_img) fetch(blockIdx.x);
  for (int tile_id = blockIdx.x; tile_id < N * tiles_img; tile_id += gridDim.x) {
    const int n = tile_id / tiles_img, r = tile_id - n * tiles_img;
    const int y0 = (r / tiles_x) * S3_TH, x0 = (r % tiles_x) * S3_TW;
    __syncthreads();                         // the previous tile has been consumed (and, first time, the tables are ready)
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int i = threadIdx.x + 256 * k;
      if (i < TILE_ELEMS) {
        const int ty = i / (S3_TW + 2), tx = i - ty * (S3_TW + 2);
        tile[ty][tx] = ok[k] ? stem_convert(raw[k], lut) : 0.f;   // 0: zero padding of the convolution
      }
    }
    __syncthreads();
    if (tile_id + (int)gridDim.x < N * tiles_img) fetch(tile_id + gridDim.x);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int q = slot + 32 * half;        // quad index in the tile: row q / 8, columns 4 * (q % 8) ..
      const int ty = q >> 3, tx = (q & 7) * 4;
      float win[3][6];
#pragma unroll
      for (int dy = 0; dy < 3; ++dy)
#pragma unroll
        for (int dx = 0; dx < 6; ++dx) win[dy][dx] = tile[ty + dy][tx + dx];
      float acc[4][8];
#pragma unroll
      for (int px = 0; px < 4; ++px)
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[px][e] = 0.f;
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        const float4 w0 = *reinterpret_cast<const float4*>(&sw[cq][tap][0]), w1 = *reinterpret_cast<const float4*>(&sw[cq][tap][4]);
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int px = 0; px < 4; ++px) {
          const float v = win[tap / 3][px + tap % 3];
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[px][e] = fmaf(wv[e], v, acc[px][e]);
        }
      }
      float bv[8], sv[8], hv[8];
      {
        const float4 b0 = *reinterpret_cast<const float4*>(&sc[cq][0][0]), b1 = *reinterpret_cast<const float4*>(&sc[cq][0][4]);
        const float4 s0 = *reinterpret_cast<const float4*>(&sc[cq][1][0]), s1 = *reinterpret_cast<const float4*>(&sc[cq][1][4]);
        const float4 h0 = *reinterpret_cast<const float4*>(&sc[cq][2][0]), h1 = *reinterpret_cast<const float4*>(&sc[cq][2][4]);
        bv[0] = b0.x; bv[1] = b0.y; bv[2] = b0.z; bv[3] = b0.w; bv[4] = b1.x; bv[5] = b1.y; bv[6] = b1.z; bv[7] = b1.w;
        sv[0] = s0.x; sv[1] = s0.y; sv[2] = s0.z; sv[3] = s0.w; sv[4] = s1.x; sv[5] = s1.y; sv[6] = s1.z; sv[7] = s1.w;
        hv[0] = h0.x; hv[1] = h0.y; hv[2] = h0.z; hv[3] = h0.w; hv[4] = h1.x; hv[5] = h1.y; hv[6] = h1.z; hv[7] = h1.w;
      }
#pragma unroll
      for (int px = 0; px < 4; ++px) {
        float yv[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) yv[e] = __fmul_rn(__fadd_rn(__fmul_rn(fmaxf(acc[px][e] + bv[e], 0.f), sv[e]), hv[e]), out_scale);
        const size_t rpix = (size_t)(y0 + ty) * W + x0 + tx + px;
        op_t* o = out + ((size_t)n * 2 * plane + rpix) * 64 + cq * 8;
        split_store(yv, o, o + plane * 64, ovf);
      }
    }
  }
  if (ovf && range_flag) *range_flag = 1;
}

// in: [N][h][w][C] fp32 -> out: [N][2][2h][2w][C] split planes.  PyTorch semantics (align_corners=False), per output
// row / column o: src = max(0.5*(o+0.5)-0.5, 0), i0 = (int)src, i1 = i0 + (i0 < size-1), l1 = src - i0, l0 = 1 - l1 (up_axis).
// Cell-centred work assignment: with scale 2 the output rows 2i+1 and 2i+2 both interpolate between input rows i and i+1
// (weights 0.75/0.25 and 0.25/0.75; the frame rows 0 and 2h-1 take weight 1/0 and a clamped partner), and likewise for
// columns: a thread owns the CELL between input pixels (i, j) and (i+1, j+1), i in [-1, h-1], j in [-1, w-1], loads its four
// corners ONCE (CPT channels each) and writes the (up to) 2 x 2 output pixels - 1 load per output instead of 4, and no 64-bit
// index arithmetic per output.
__device__ __forceinline__ void up_axis(int o, int n_in, int& i0, int& i1, float& l0, float& l1) {
  const float s = fmaxf(0.5f * ((float)o + 0.5f) - 0.5f, 0.f);
  i0 = (int)s;
  i1 = i0 + (i0 < n_in - 1 ? 1 : 0);
  l1 = s - (float)i0;
  l0 = 1.f - l1;
}
// For every output row the pair (i0, i1) that up_axis() names IS the pair of rows (ya, yb) the row's cell loads - frame cells
// included: row 0 names (0, 1), row 2h-1 names (h-1, h-1) - and likewise per column
// (tests/test_host_logic.py::test_upsample_cell_corners_are_the_rows_the_formula_names), so the corners are indexed
// statically.  A run-time selection of the corners put the 32 corner values into local memory (32 LDL + 8 STL per cell in the
// SASS) and hid from the compiler that the two samples of a cell column share the `top` / `bot` terms: 921 -> 712 SASS
// instructions per cell, in an issue-bound kernel.
__global__ void __launch_bounds__(256, 3) upsample2x_kernel(const float* __restrict__ in, op_t* __restrict__ out,
                                                            int N, int h, int w, int C, int* __restrict__ range_flag, float out_scale) {
  const int cq_per_pix = C / CPT;
  const int cw = w + 1, ch = h + 1;
  const int H = 2 * h, W = 2 * w;
  const size_t oplane = (size_t)H * W;
  // (32-bit index arithmetic: N <= 1024 slices x 257 x 257 cells x C / 8 channel groups stays far below 2^32, and the
  //  64-bit divisions were a third of this kernel's instructions)
  const uint32_t total = (uint32_t)N * (uint32_t)ch * (uint32_t)cw * (uint32_t)cq_per_pix;
  bool ovf = false;
  for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
    uint32_t cell = t / (uint32_t)cq_per_pix;
    const int cq = (int)(t - cell * (uint32_t)cq_per_pix);
    uint32_t q2 = cell / (uint32_t)cw;
    const int cj = (int)(cell - q2 * (uint32_t)cw) - 1;
    const uint32_t q3 = q2 / (uint32_t)ch;
    const int ci = (int)(q2 - q3 * (uint32_t)ch) - 1;
    const int n = (int)q3;
    const int ya = ci < 0 ? 0 : ci, yb = ya + 1 < h ? ya + 1 : h - 1;   // the two input rows / columns every sample of the
    const int xa = cj < 0 ? 0 : cj, xb = xa + 1 < w ? xa + 1 : w - 1;   // cell interpolates between (frame cells: clamped)
    const float* base = in + (size_t)n * h * w * C + cq * CPT;
    float p[2][2][CPT];
#pragma unroll
    for (int q = 0; q < CPT / 4; ++q) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(base + ((size_t)ya * w + xa) * C) + q);
      const float4 b = __ldg(reinterpret_cast<const float4*>(base + ((size_t)ya * w + xb) * C) + q);
      const float4 c = __ldg(reinterpret_cast<const float4*>(base + ((size_t)yb * w + xa) * C) + q);
      const float4 e = __ldg(reinterpret_cast<const float4*>(base + ((size_t)yb * w + xb) * C) + q);
      p[0][0][4 * q] = a.x; p[0][0][4 * q + 1] = a.y; p[0][0][4 * q + 2] = a.z; p[0][0][4 * q + 3] = a.w;
      p[0][1][4 * q] = b.x; p[0][1][4 * q + 1] = b.y; p[0][1][4 * q + 2] = b.z; p[0][1][4 * q + 3] = b.w;
      p[1][0][4 * q] = c.x; p[1][0][4 * q + 1] = c.y; p[1][0][4 * q + 2] = c.z; p[1][0][4 * q + 3] = c.w;
      p[1][1][4 * q] = e.x; p[1][1][4 * q + 1] = e.y; p[1][1][4 * q + 2] = e.z; p[1][1][4 * q + 3] = e.w;
    }
    float ly[2][2], lx[2][2];
#pragma unroll
    for (int d = 0; d < 2; ++d) {
      int i0, i1;
      up_axis(2 * ci + 1 + d, h, i0, i1, ly[d][0], ly[d][1]);
      up_axis(2 * cj + 1 + d, w, i0, i1, lx[d][0], lx[d][1]);
    }
    float top[2][CPT], bot[2][CPT];   // the horizontal interpolations per cell column: shared by the column's two samples
#pragma unroll
    for (int e = 0; e < CPT; ++e) {
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        top[dx][e] = __fmaf_rn(lx[dx][1], p[0][1][e], __fmul_rn(lx[dx][0], p[0][0][e]));
        bot[dx][e] = __fmaf_rn(lx[dx][1], p[1][1][e], __fmul_rn(lx[dx][0], p[1][0][e]));
      }
    }
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
      const int y = 2 * ci + 1 + dy;
      if (y < 0 || y >= H) continue;
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const int x = 2 * cj + 1 + dx;
        if (x < 0 || x >= W) continue;
        float vv[CPT];
#pragma unroll
        for (int e = 0; e < CPT; ++e) vv[e] = __fmul_rn(__fmaf_rn(ly[dy][1], bot[dx][e], __fmul_rn(ly[dy][0], top[dx][e])), out_scale);
        const size_t r = (size_t)y * W + x;
        op_t* o = out + ((size_t)n * 2 * oplane + r) * C + cq * CPT;
        split_store(vv, o, o + oplane * C, ovf);
      }
    }
  }
  if (ovf && range_flag) *range_flag = 1;
}

__global__ void prep_conv_weights_kernel(const float* __restrict__ oihw, op_t* __restrict__ out, int Cout, int Cin,
                                         int taps, int* __restrict__ range_flag, float w_scale) {
  const size_t total = (size_t)Cout * Cin * taps;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t tap = i % taps, ci = (i / taps) % Cin, co = i / ((size_t)taps * Cin);
    op_t hi, lo;
    const float wv = __fmul_rn(oihw[i], w_scale);   // power-of-two scale chosen by the engine so that max |w| fits fp16
    split_f16(wv, hi, lo);
    if (!(fabsf(wv) <= kOpMax) && range_flag) *range_flag = 1;
    const size_t o = (tap * Cout + co) * Cin + ci;
    out[o] = hi;
    out[total + o] = lo;
  }
}

inline int grid_for(size_t total, int block, int num_sms) {
  size_t g = (total + block - 1) / block;
  const size_t cap = (size_t)num_sms * 16;
  return (int)(g < cap ? (g ? g : 1) : cap);
}

}  // namespace

// The stem kernel tiles each slice in 8 x 32 blocks (the engine's slices are 256 x 256); other shapes are rejected.
template <typename IT>
static int launch_stem_t(const IT* in, void* out, const float* w, const float* bias, const float* scale, const float* shift, int N,
                         int H, int W, int* range_flag, float out_scale, int num_sms, cudaStream_t stream) {
  if (W % S3_TW || H % S3_TH) return (int)cudaErrorInvalidValue;
  const int tiles = N * (W / S3_TW) * (H / S3_TH);
  const int cap = num_sms * 6;
  stem_kernel<IT><<<tiles < cap ? tiles : cap, 256, 0, stream>>>(in, static_cast<op_t*>(out), w, bias, scale, shift, N, H, W, range_flag,
                                                                 out_scale);
  return (int)cudaGetLastError();
}

int launch_stem(const int16_t* in, void* out, const float* w, const float* bias, const float* scale,
                const float* shift, int N, int H, int W, int* range_flag, float out_scale, int num_sms, cudaStream_t stream) {
  return launch_stem_t<int16_t>(in, out, w, bias, scale, shift, N, H, W, range_flag, out_scale, num_sms, stream);
}
int launch_stem_f32(const float* in_norm, void* out, const float* w, const float* bias, const float* scale, const float* shift, int N,
                    int H, int W, int* range_flag, float out_scale, int num_sms, cudaStream_t stream) {
  return launch_stem_t<float>(in_norm, out, w, bias, scale, shift, N, H, W, range_flag, out_scale, num_sms, stream);
}

int launch_upsample2x(const float* in, void* out, int N, int h, int w, int C, int* range_flag, float out_scale, int num_sms,
                      cudaStream_t stream) {
  const size_t total = (size_t)N * (h + 1) * (w + 1) * (C / CPT);
  upsample2x_kernel<<<grid_for(total, 256, num_sms), 256, 0, stream>>>(in, static_cast<op_t*>(out), N, h, w, C, range_flag, out_scale);
  return (int)cudaGetLastError();
}

int launch_prep_conv_weights(const float* oihw, void* out, int Cout, int Cin, int taps, int* range_flag, float w_scale,
                             cudaStream_t stream) {
  const size_t total = (size_t)Cout * Cin * taps;
  prep_conv_weights_kernel<<<(int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096), 256, 0, stream>>>(
      oihw, static_cast<op_t*>(out), Cout, Cin, taps, range_flag, w_scale);
  return (int)cudaGetLastError();
}

}  // namespace lm
