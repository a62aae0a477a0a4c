// conv_probe: checks conv_tc (lungmask_b200/csrc/conv_tc.cu) against a float64 host convolution on
// procedurally generated data (every element is a hash of its index, so the host can evaluate any
// output pixel without holding the tensors), then times the 22 tensor-core layers of the U-Net at a
// given batch. Test infrastructure only.
//   usage: conv_probe [batch=8] [chunk_kb=4] [timing_only=0] [reps=3]
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <vector>
#include <algorithm>
#include "../lungmask_b200/csrc/conv_tc.cuh"

using namespace lm;
#ifdef LM_CONV_PROFILE
namespace lm { void conv_prof_reset(); void conv_prof_read(unsigned long long*); }
#endif

#define CK(x)                                                                         \
  do {                                                                                \
    cudaError_t e_ = (x);                                                             \
    if (e_ != cudaSuccess) {                                                          \
      printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); \
      exit(2);                                                                        \
    }                                                                                 \
  } while (0)

__host__ __device__ inline uint32_t mix(uint64_t x) {
  x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
  return (uint32_t)x;
}
__host__ __device__ inline float gen(uint32_t seed, uint64_t idx, bool ints) {
  const uint32_t h = mix(idx * 0x9E3779B97F4A7C15ULL + seed);
  if (ints) return (float)((int)(h % 5u) - 2);
  return ((h >> 8) * (1.0f / 16777216.0f) - 0.5f) * 2.0f;
}
// operand-format split (conv_tc.cuh): value = hi + lo * kLoUnscale
struct Split { op_t hi, lo; };
__host__ __device__ inline Split split(float x) {
  Split s;
  s.hi = __float2half_rn(x);
  s.lo = __float2half_rn((x - __half2float(s.hi)) * 2048.f);
  return s;
}
__host__ __device__ inline double joined(const Split& s) { return (double)(float)s.hi + (double)(float)s.lo * (double)kLoUnscale; }

// activation [N][2][H][W][C]; logical value index = ((n*H+y)*W+x)*C+c
__global__ void fill_act(op_t* base, int N, int H, int W, int C, uint32_t seed, bool ints) {
  const size_t total = (size_t)N * H * W * C, plane = (size_t)H * W * C;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t n = i / plane, r = i - n * plane;
    const Split s = split(gen(seed, i, ints));
    base[(n * 2) * plane + r] = s.hi;
    base[(n * 2 + 1) * plane + r] = s.lo;
  }
}
// weights [2][taps][Cout][Cin]; logical OIHW index = ((co*Cin+ci)*taps+tap)
__global__ void fill_w(op_t* base, int Cout, int Cin, int taps, uint32_t seed, float wscale, bool ints) {
  const size_t total = (size_t)Cout * Cin * taps;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t tap = i % taps, ci = (i / taps) % Cin, co = i / ((size_t)taps * Cin);
    const Split s = split(gen(seed, i, ints) * (ints ? 1.f : wscale));
    const size_t o = (tap * Cout + co) * Cin + ci;
    base[o] = s.hi;
    base[total + o] = s.lo;
  }
}

struct Layer {
  const char* name;
  int H, W, C0, C1, Cout, taps, mode, K;
};

static double h_act(uint32_t seed, int H, int W, int C, int n, int y, int x, int c, bool ints) {
  if (y < 0 || y >= H || x < 0 || x >= W) return 0.0;
  const Split s = split(gen(seed, (((uint64_t)n * H + y) * W + x) * C + c, ints));
  return joined(s);
}
static double h_w(uint32_t seed, int Cin, int taps, int co, int ci, int tap, float wscale, bool ints) {
  const Split s = split(gen(seed, ((uint64_t)co * Cin + ci) * taps + tap, ints) * (ints ? 1.f : wscale));
  return joined(s);
}

struct Bufs {
  op_t *src0 = nullptr, *src1 = nullptr, *w = nullptr;
  void *out = nullptr, *pool = nullptr;
  float *bias, *scale, *shift, *hw, *hb, *scores = nullptr;
  int* range_flag = nullptr;
  uint8_t* labels = nullptr;
};

static float h_param(uint32_t seed, int c, int kind, bool ints) {
  if (ints) return kind == 1 ? 1.f : (kind == 0 ? (float)((int)(mix(seed + c) % 3u) - 1) : 0.f);
  const float g = gen(seed + 77u * kind, c, false);
  return kind == 1 ? 1.0f + 0.3f * g : 0.2f * g;
}

static double run_layer(const Layer& L, int N, int chunk_kb, int num_sms, bool check, bool ints, int reps) {
  const int Cin = L.C0 + L.C1;
  const float wscale = 1.0f / sqrtf((float)Cin * L.taps) * 1.7f;
  Bufs b;
  const size_t plane = (size_t)L.H * L.W;
  CK(cudaMalloc(&b.src0, (size_t)N * 2 * plane * L.C0 * sizeof(op_t)));
  if (L.C1) CK(cudaMalloc(&b.src1, (size_t)N * 2 * plane * L.C1 * sizeof(op_t)));
  CK(cudaMalloc(&b.w, (size_t)2 * L.taps * L.Cout * Cin * sizeof(op_t)));
  const size_t out_elems = (size_t)N * plane * L.Cout * (L.mode == kModeLinear ? 1 : 2);
  const size_t out_esize = L.mode == kModeLinear ? 4 : sizeof(op_t);
  CK(cudaMalloc(&b.out, out_elems * out_esize));
  CK(cudaMemset(b.out, 0xFF, out_elems * out_esize));
  if (L.mode == kModeReluBnPool) { CK(cudaMalloc(&b.pool, out_elems / 4 * sizeof(op_t))); CK(cudaMemset(b.pool, 0xFF, out_elems / 4 * sizeof(op_t))); }
  CK(cudaMalloc(&b.range_flag, 4)); CK(cudaMemset(b.range_flag, 0, 4));
  CK(cudaMalloc(&b.bias, L.Cout * 4)); CK(cudaMalloc(&b.scale, L.Cout * 4)); CK(cudaMalloc(&b.shift, L.Cout * 4));
  std::vector<float> hb(L.Cout), hs(L.Cout), hh(L.Cout), hhw(8 * 64), hhb(8);
  for (int c = 0; c < L.Cout; ++c) { hb[c] = h_param(11, c, 0, ints); hs[c] = h_param(11, c, 1, ints); hh[c] = h_param(11, c, 2, ints); }
  for (int i = 0; i < 8 * 64; ++i) hhw[i] = 0.5f * gen(991, i, false);
  for (int i = 0; i < 8; ++i) hhb[i] = 0.1f * gen(992, i, false);
  CK(cudaMemcpy(b.bias, hb.data(), L.Cout * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(b.scale, hs.data(), L.Cout * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(b.shift, hh.data(), L.Cout * 4, cudaMemcpyHostToDevice));
  CK(cudaMalloc(&b.hw, 8 * 64 * 4)); CK(cudaMalloc(&b.hb, 8 * 4));
  CK(cudaMemcpy(b.hw, hhw.data(), 8 * 64 * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(b.hb, hhb.data(), 8 * 4, cudaMemcpyHostToDevice));
  if (L.mode == kModeHead) {
    CK(cudaMalloc(&b.labels, (size_t)N * plane)); CK(cudaMemset(b.labels, 0xEE, (size_t)N * plane));
    CK(cudaMalloc(&b.scores, (size_t)N * L.K * plane * 4));
  }
  fill_act<<<1024, 256>>>(b.src0, N, L.H, L.W, L.C0, 1, ints);
  if (L.C1) fill_act<<<1024, 256>>>(b.src1, N, L.H, L.W, L.C1, 2, ints);
  fill_w<<<1024, 256>>>(b.w, L.Cout, Cin, L.taps, 3, wscale, ints);
  CK(cudaGetLastError());

  ConvParams p{};
  p.N = N; p.H = L.H; p.W = L.W; p.C0 = L.C0; p.C1 = L.C1; p.Cout = L.Cout; p.taps = L.taps; p.mode = L.mode;
  p.chunk_kb = chunk_kb; p.bias = b.bias; p.scale = b.scale; p.shift = b.shift; p.out = b.out; p.out_pool = b.pool;
  p.head_w = b.hw; p.head_b = b.hb; p.K = L.K; p.labels = b.labels; p.scores = b.scores; p.range_flag = b.range_flag;
  p.in_unscale = 1.f; p.out_scale = 1.f;
  ConvMaps maps;
  int r = make_conv_maps(&maps, b.src0, b.src1, b.w, p, N);
  if (r) { printf("make_conv_maps failed %d\n", r); exit(2); }
  cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  auto launch = [&]() { return launch_conv_tc(maps, p, num_sms, 0); };
  r = launch();
  if (r) { printf("launch failed %d\n", r); exit(2); }
  CK(cudaDeviceSynchronize());
  float ms = 0;
#ifdef LM_CONV_PROFILE
  conv_prof_reset();
#endif
  if (reps > 0) {
    CK(cudaEventRecord(e0));
    for (int i = 0; i < reps; ++i) launch();
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    CK(cudaEventElapsedTime(&ms, e0, e1));
    ms /= reps;
  }
  const double flops = 2.0 * N * plane * L.Cout * Cin * L.taps;

  if (check) {
    std::vector<float> ho;       // mode 2: fp32 output
    std::vector<op_t> hs_, hp;   // split-plane outputs
    if (L.mode == kModeLinear) { ho.resize(out_elems); CK(cudaMemcpy(ho.data(), b.out, out_elems * 4, cudaMemcpyDeviceToHost)); }
    else { hs_.resize(out_elems); CK(cudaMemcpy(hs_.data(), b.out, out_elems * sizeof(op_t), cudaMemcpyDeviceToHost)); }
    if (b.pool) { hp.resize(out_elems / 4); CK(cudaMemcpy(hp.data(), b.pool, out_elems / 4 * sizeof(op_t), cudaMemcpyDeviceToHost)); }
    int hflag = 0; CK(cudaMemcpy(&hflag, b.range_flag, 4, cudaMemcpyDeviceToHost));
    if (hflag) printf("range_flag set!\n");
    std::vector<uint8_t> hl; std::vector<float> hsco;
    if (L.mode == kModeHead) {
      hl.resize((size_t)N * plane); CK(cudaMemcpy(hl.data(), b.labels, hl.size(), cudaMemcpyDeviceToHost));
      hsco.resize((size_t)N * L.K * plane); CK(cudaMemcpy(hsco.data(), b.scores, hsco.size() * 4, cudaMemcpyDeviceToHost));
    }
    // choose sample pixels: all for small problems, random subset otherwise
    const size_t npix = (size_t)N * plane;
    const size_t budget = (size_t)(3e8 / ((double)L.Cout * Cin * L.taps)) + 8;  // bounded host work per layer
    const size_t nsamp = std::min<size_t>(npix, ints ? npix : std::min<size_t>(600, budget));
    double max_err = 0, max_ref = 0; size_t bad = 0, label_bad = 0; double max_sc_err = 0, max_pool_err = 0;
    std::vector<double> yv(L.Cout);
    auto eval_pixel = [&](int n, int y, int x, std::vector<double>& out_y) {
      for (int co = 0; co < L.Cout; ++co) {
        double s = 0;
        for (int tap = 0; tap < L.taps; ++tap) {
          const int dy = L.taps == 9 ? tap / 3 - 1 : 0, dx = L.taps == 9 ? tap % 3 - 1 : 0;
          if (y + dy < 0 || y + dy >= L.H || x + dx < 0 || x + dx >= L.W) continue;
          for (int ci = 0; ci < Cin; ++ci) {
            const double a = ci < L.C0 ? h_act(1, L.H, L.W, L.C0, n, y + dy, x + dx, ci, ints)
                                       : h_act(2, L.H, L.W, L.C1, n, y + dy, x + dx, ci - L.C0, ints);
            s += a * h_w(3, Cin, L.taps, co, ci, tap, wscale, ints);
          }
        }
        if (L.mode == kModeLinear) out_y[co] = (double)((float)s + hb[co]);
        else { float v = fmaxf((float)s + hb[co], 0.f); out_y[co] = (double)(v * hs[co] + hh[co]); }
      }
    };
    for (size_t si = 0; si < nsamp; ++si) {
      const size_t pi = nsamp == npix ? si : (size_t)(mix(si * 7919 + 5) % npix);
      const int n = pi / plane, y = (pi % plane) / L.W, x = pi % L.W;
      eval_pixel(n, y, x, yv);
      if (L.mode == kModeHead) {
        double lg[8], mx = -1e300;
        for (int k = 0; k < L.K; ++k) { double s = 0; for (int c = 0; c < 64; ++c) s += (double)hhw[k * 64 + c] * yv[c]; lg[k] = s + hhb[k]; mx = std::max(mx, lg[k]); }
        double se = 0; for (int k = 0; k < L.K; ++k) se += exp(lg[k] - mx);
        int best = 0; double bv = -1e300, second = -1e300;
        for (int k = 0; k < L.K; ++k) {
          const double sc = lg[k] - mx - log(se);
          if (sc > bv) { second = bv; bv = sc; best = k; } else if (sc > second) second = sc;
          max_sc_err = std::max(max_sc_err, fabs(sc - (double)hsco[((size_t)n * L.K + k) * plane + (size_t)y * L.W + x]));
        }
        if (hl[pi] != best && bv - second > 1e-4) ++label_bad;
        continue;
      }
      for (int co = 0; co < L.Cout; ++co) {
        double got;
        if (L.mode == kModeLinear) got = ho[pi * L.Cout + co];
        else {
          const size_t o = ((size_t)n * 2 * plane + (size_t)y * L.W + x) * L.Cout + co;
          got = (double)(float)hs_[o] + (double)(float)hs_[o + plane * L.Cout] * (double)kLoUnscale;
        }
        const double err = fabs(got - yv[co]);
        max_err = std::max(max_err, err); max_ref = std::max(max_ref, fabs(yv[co]));
        if (ints ? err != 0 : err > 2e-5 * std::max(1.0, fabs(yv[co]))) ++bad;
      }
    }
    if (L.mode == kModeReluBnPool) {
      const int Hp = L.H / 2, Wp = L.W / 2;
      std::vector<double> y4[4];
      for (auto& v : y4) v.resize(L.Cout);
      for (int si = 0; si < 40; ++si) {
        const size_t pi = mix(si * 31 + 9) % ((size_t)N * Hp * Wp);
        const int n = pi / (Hp * Wp), yy = (pi % (Hp * Wp)) / Wp, xx = pi % Wp;
        for (int e = 0; e < 4; ++e) eval_pixel(n, 2 * yy + e / 2, 2 * xx + e % 2, y4[e]);
        for (int co = 0; co < L.Cout; ++co) {
          const double ref = 0.25 * (y4[0][co] + y4[1][co] + y4[2][co] + y4[3][co]);
          const size_t o = ((size_t)n * 2 * Hp * Wp + (size_t)yy * Wp + xx) * L.Cout + co;
          const double got = (double)(float)hp[o] + (double)(float)hp[o + (size_t)Hp * Wp * L.Cout] * (double)kLoUnscale;
          max_pool_err = std::max(max_pool_err, fabs(got - ref));
        }
      }
    }
    printf("CHECK %-22s N=%d %3dx%-3d C=%d+%d->%d taps=%d mode=%d: samples=%zu max_abs_err=%.3e (max|ref|=%.2f) bad=%zu",
           L.name, N, L.H, L.W, L.C0, L.C1, L.Cout, L.taps, L.mode, nsamp, max_err, max_ref, bad);
    if (L.mode == kModeReluBnPool) printf(" pool_err=%.3e", max_pool_err);
    if (L.mode == kModeHead) printf(" score_err=%.3e label_mismatch(margin>1e-4)=%zu", max_sc_err, label_bad);
    printf(" %s\n", (bad || label_bad || max_pool_err > 1e-4 || max_sc_err > 1e-4) ? "FAIL" : "ok");
  }
#ifdef LM_CONV_PROFILE
  if (reps > 0) {
    unsigned long long pr[16];
    conv_prof_read(pr);
    const int BNt = conv_tile_n(L.Cout);
    const double tiles = (double)N * (L.H / 16) * (L.W / 8) * (L.Cout / BNt) * reps;
    const double kbs = tiles * (Cin / kBK) * L.taps;
    const double ctas = std::min<double>(num_sms, tiles / reps) * reps;
    printf("PROF  %-18s per k-block cycles: kernel %.0f | producer wait aempty %.0f bempty %.0f | mma wait tempty %.0f afull %.0f bfull %.0f issue %.0f | epi wait tfull %.0f drain %.0f, tile-epilogue per tile %.0f\n",
           L.name, pr[9] / kbs * 1.0 * 1, pr[0] / kbs, pr[1] / kbs, pr[2] / kbs, pr[3] / kbs, pr[4] / kbs, pr[5] / kbs, pr[6] / kbs, pr[7] / kbs, pr[8] / tiles);
    printf("PROF2 %-18s issuer per k-block: first two k-steps %.0f | last two k-steps %.0f | commits %.0f | barrier waits %.0f | everything else %.0f\n",
           L.name, pr[10] / kbs, pr[11] / kbs, pr[12] / kbs, (pr[2] + pr[3] + pr[4]) / kbs,
           (double)pr[5] / kbs - (double)(pr[10] + pr[11] + pr[12] + pr[2] + pr[3] + pr[4]) / kbs);
    (void)ctas;
  }
#endif
  if (reps > 0)
    printf("TIME  %-22s N=%d %3dx%-3d C=%4d+%-4d->%4d taps=%d: %.3f ms  %.1f TFLOP/s(algorithmic)\n", L.name, N, L.H, L.W,
           L.C0, L.C1, L.Cout, L.taps, ms, flops / ms * 1e-9);
  cudaFree(b.src0); cudaFree(b.src1); cudaFree(b.w); cudaFree(b.out); cudaFree(b.pool); cudaFree(b.bias); cudaFree(b.scale);
  cudaFree(b.shift); cudaFree(b.hw); cudaFree(b.hb); cudaFree(b.labels); cudaFree(b.scores); cudaFree(b.range_flag);
  return ms;
}

int main(int argc, char** argv) {
  setvbuf(stdout, nullptr, _IOLBF, 0);
  const int batch = argc > 1 ? atoi(argv[1]) : 8;
  const int chunk = argc > 2 ? atoi(argv[2]) : 4;
  const int timing_only = argc > 3 ? atoi(argv[3]) : 0;
  const int reps = argc > 4 ? atoi(argv[4]) : 3;   // timed repetitions per network layer (0: one untimed launch per layer, for ncu)
  cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, 0));
  const int sms = prop.multiProcessorCount;
  printf("device %s SMs %d; batch %d chunk_kb %d\n", prop.name, sms, batch, chunk);
  if (!timing_only) {
    const Layer small[] = {
        {"ints 1tile", 16, 8, kBK, 0, 64, 9, kModeReluBn, 0},
        {"ints 128->128", 16, 32, 128, 0, 128, 9, kModeReluBn, 0},
        {"ints concat", 16, 16, kBK, kBK, 64, 9, kModeReluBn, 0},
        {"ints 1x1", 16, 8, 64, 0, 128, 1, kModeLinear, 0},
    };
    for (const Layer& L : small) run_layer(L, 2, chunk, sms, true, true, 0);
    const Layer rnd[] = {
        {"rnd 64->64 pool", 32, 32, 64, 0, 64, 9, kModeReluBnPool, 0},
        {"rnd concat 128+128->128", 16, 16, 128, 128, 128, 9, kModeReluBn, 0},
        {"rnd 1x1 256->128", 16, 16, 256, 0, 128, 1, kModeLinear, 0},
        {"rnd head K=3", 16, 32, 64, 0, 64, 9, kModeHead, 3},
        {"rnd head K=6", 16, 32, 64, 0, 64, 9, kModeHead, 6},
        {"rnd 512->256", 16, 16, 512, 0, 256, 9, kModeReluBn, 0},
        {"rnd 1024->1024 pool", 16, 16, 1024, 0, 1024, 9, kModeReluBnPool, 0},
    };
    for (const Layer& L : rnd) run_layer(L, 3, chunk, sms, true, false, 0);
    run_layer(rnd[5], 3, 1, sms, true, false, 0);
    run_layer(rnd[5], 3, 1000, sms, true, false, 0);
  }
  const Layer net[] = {
      {"down0.block3", 256, 256, 64, 0, 64, 9, kModeReluBnPool, 0},
      {"down1.block0", 128, 128, 64, 0, 128, 9, kModeReluBn, 0},
      {"down1.block3", 128, 128, 128, 0, 128, 9, kModeReluBnPool, 0},
      {"down2.block0", 64, 64, 128, 0, 256, 9, kModeReluBn, 0},
      {"down2.block3", 64, 64, 256, 0, 256, 9, kModeReluBnPool, 0},
      {"down3.block0", 32, 32, 256, 0, 512, 9, kModeReluBn, 0},
      {"down3.block3", 32, 32, 512, 0, 512, 9, kModeReluBnPool, 0},
      {"down4.block0", 16, 16, 512, 0, 1024, 9, kModeReluBn, 0},
      {"down4.block3", 16, 16, 1024, 0, 1024, 9, kModeReluBn, 0},
      {"up0.up1x1", 16, 16, 1024, 0, 512, 1, kModeLinear, 0},
      {"up0.block0", 32, 32, 512, 512, 512, 9, kModeReluBn, 0},
      {"up0.block3", 32, 32, 512, 0, 512, 9, kModeReluBn, 0},
      {"up1.up1x1", 32, 32, 512, 0, 256, 1, kModeLinear, 0},
      {"up1.block0", 64, 64, 256, 256, 256, 9, kModeReluBn, 0},
      {"up1.block3", 64, 64, 256, 0, 256, 9, kModeReluBn, 0},
      {"up2.up1x1", 64, 64, 256, 0, 128, 1, kModeLinear, 0},
      {"up2.block0", 128, 128, 128, 128, 128, 9, kModeReluBn, 0},
      {"up2.block3", 128, 128, 128, 0, 128, 9, kModeReluBn, 0},
      {"up3.up1x1", 128, 128, 128, 0, 64, 1, kModeLinear, 0},
      {"up3.block0", 256, 256, 64, 64, 64, 9, kModeReluBn, 0},
      {"up3.block3+head", 256, 256, 64, 0, 64, 9, kModeHead, 3},
  };
  double total_ms = 0;
  for (const Layer& L : net) total_ms += run_layer(L, batch, chunk, sms, false, false, reps);
  printf("TOTAL tensor-core layers: %.3f ms for %d slices -> %.1f slices/s (conv layers only)\n", total_ms, batch,
         batch / total_ms * 1e3);
  printf("conv_probe done\n");
  return 0;
}
