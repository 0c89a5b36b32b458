// lce_b200_builtins.cu -- fp32 TFLite builtins as CUDA kernels (include/
// lce_b200_builtins.h). These are the callers either side of the binary path in the
// QuickNet / Bi-RealNet graphs, kept on the device so activations never leave HBM.
// Semantics follow TFLite's reference kernels (tensorflow/lite/kernels/internal/
// reference/conv.h:27, depthwiseconv_float.h:25, pooling.h:28,196, add.h,
// fully_connected.h:29, softmax.h:31, reduce.h); fp32 accumulate with FMA.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cfloat>
#include <climits>
#include <cstdint>
#include <cstdlib>

#include "lce_b200.h"
#include "lce_b200_builtins.h"

namespace lce_b200_internal {
int fail(const char* fmt, ...);       // lce_b200.cu
int launch_check(const char* what);   // lce_b200.cu
// tcgen05 kind::tf32 pointwise convolution (lce_b200_pw.cuh): 0 launched, -1 not eligible
int pw_tf32_conv(const float* in, const float* filter, const float* bias, float* out, int32_t* packed, long long M, int N,
                 int K, int act, int pairs_ok, void* stream);
// tcgen05 kind::tf32 7x7 / stride 2 / 3 -> 64 convolution (Bi-RealNet's stem): 0 launched, -1 not eligible
int stem7_tf32_conv(const float* in, const float* filter, const float* bias, float* out, int B, int H, int W, int OH, int OW,
                    int ph, int pw, int act, void* stream);
}  // namespace lce_b200_internal
using lce_b200_internal::fail;
using lce_b200_internal::launch_check;

namespace {

__device__ __forceinline__ float apply_act(float x, int act) {
  switch (act) {
    case LCE_ACT_RELU: return fmaxf(x, 0.0f);
    case LCE_ACT_RELU_N1_TO_1: return fminf(fmaxf(x, -1.0f), 1.0f);
    case LCE_ACT_RELU6: return fminf(fmaxf(x, 0.0f), 6.0f);
    default: return x;
  }
}

int out_size(int padding, int image, int filter, int stride, int dil) {
  const int eff = (filter - 1) * dil + 1;
  if (stride == 0) return 0;
  if (padding == LCE_PADDING_SAME) return (image + stride - 1) / stride;
  if (padding == LCE_PADDING_VALID) return (image + stride - eff) / stride;
  return 0;
}
int pad_before(int stride, int dil, int in, int filter, int out) {
  const int eff = (filter - 1) * dil + 1;
  int total = (out - 1) * stride + eff - in;
  if (total < 0) total = 0;
  return total / 2;
}
inline cudaStream_t as_stream(void* s) { return static_cast<cudaStream_t>(s); }
int grid_for(long long n, int per_block, int max_blocks = 148 * 32) {
  long long b = (n + per_block - 1) / per_block;
  if (b < 1) b = 1;
  if (b > max_blocks) b = max_blocks;
  return static_cast<int>(b);
}

struct ConvGeom {
  int B, H, W, Cin, KH, KW, Cout, sh, sw, dh, dw, ph, pw, OH, OW, act;
};

// successful launches per fp32 convolution kernel (lce_b200_f32_conv_path_counts)
enum ConvPath { kPathPwTf32, kPathStem7, kPathDirect16, kPathGemmSmallM, kPathGemm128, kPathIgemm8x8, kPathIgemm8x4,
                kPathGemm, kConvPaths };
std::atomic<uint64_t> g_conv_path[kConvPaths] = {};
void count_path(ConvPath p) { g_conv_path[p].fetch_add(1, std::memory_order_relaxed); }
int launched(ConvPath p, const char* what) {
  const int rc = launch_check(what);
  if (rc == 0) count_path(p);
  return rc;
}

// ---- small-K direct convolution (stem 3x3x3->16, 16->64 pointwise: K <= 32) --------
// One thread = one output pixel x 16 consecutive output channels; consecutive lanes
// take consecutive 16-channel groups of the same pixel, so a warp writes one
// contiguous span (coalesced 128-bit stores) and reads each input value once
// (broadcast). All weights sit in shared memory as [K][group][16 (+4 pad)].
constexpr int kDirectMaxK = 32;
constexpr int kDirectMaxCout = 128;
constexpr int kDirectGroupStride = 20;   // 16 + 4 floats: conflict-free LDS.128 across groups
// KH/KW/CIN > 0: compile-time shape (stem 3x3x3, pointwise 1x1x16) => fully unrolled K loop.
// Each thread computes kPX pixels x 16 channels so every 128-bit weight read from shared
// memory feeds 4*kPX FMAs (with one pixel per thread the kernel was LDS-bound: ncu showed
// short-scoreboard / MIO-throttle stalls dominating).
template <int KH_, int KW_, int CIN_, int kPX, bool kTileLoop = false>
__global__ void __launch_bounds__(128) conv_direct16_kernel(const float* __restrict__ in,
                                                            const float* __restrict__ filter,
                                                            const float* __restrict__ bias,
                                                            float* __restrict__ out, ConvGeom g,
                                                            long long M, int G, int tiles_per_block,
                                                            int32_t* __restrict__ packed) {
  extern __shared__ __align__(16) float w_s[];   // [K][G][20] then bias [G][16]
  const int KH = KH_ ? KH_ : g.KH, KW = KW_ ? KW_ : g.KW, CIN = CIN_ ? CIN_ : g.Cin;
  const int K = KH * KW * CIN;
  float* b_s = w_s + K * G * kDirectGroupStride;
  for (int i = threadIdx.x; i < K * G * 16; i += blockDim.x) {
    const int c = i & 15, gi = (i >> 4) % G, k = (i >> 4) / G;
    const int co = gi * 16 + c;
    w_s[(k * G + gi) * kDirectGroupStride + c] =
        co < g.Cout ? filter[static_cast<size_t>(co) * K + k] : 0.0f;
  }
  for (int i = threadIdx.x; i < G * 16; i += blockDim.x)
    b_s[i] = (bias && i < g.Cout) ? bias[i] : 0.0f;
  __syncthreads();
  // thread -> (pixel quad, channel group); consecutive lanes = consecutive groups, then pixels.
  // Pixel p of a thread is m0 + p * pstride with pstride = blockDim.x / G pixels, so that for
  // every p a warp still writes one contiguous span. 32-bit index math (host checks the range).
  const unsigned px_per_blk = blockDim.x / static_cast<unsigned>(G);
  const unsigned lpx = threadIdx.x / static_cast<unsigned>(G);
  const int gi = static_cast<int>(threadIdx.x - lpx * G);
  if (lpx >= px_per_blk) return;
  const unsigned ohw = g.OH * g.OW;
  // the weights staged above serve `tiles_per_block` consecutive pixel tiles
  const int n_tile = kTileLoop ? tiles_per_block : 1;
  for (int tile = 0; tile < n_tile; ++tile) {
  const unsigned blk_m0 = (blockIdx.x * n_tile + tile) * px_per_blk * kPX;
  if (blk_m0 >= static_cast<unsigned>(M)) break;
  long long ibase[kPX];
  int iy0[kPX], ix0[kPX];
  bool ok[kPX];
#pragma unroll
  for (int p = 0; p < kPX; ++p) {
    const unsigned mu = blk_m0 + p * px_per_blk + lpx;
    ok[p] = mu < static_cast<unsigned>(M);
    const unsigned mm = ok[p] ? mu : 0u;
    const unsigned bu = mm / ohw;
    const unsigned r = mm - bu * ohw;
    const unsigned oy = r / static_cast<unsigned>(g.OW), ox = r - oy * g.OW;
    iy0[p] = static_cast<int>(oy) * g.sh - g.ph;
    ix0[p] = static_cast<int>(ox) * g.sw - g.pw;
    ibase[p] = static_cast<long long>(bu) * g.H * g.W;
  }
  float acc[kPX][16];
#pragma unroll
  for (int p = 0; p < kPX; ++p)
#pragma unroll
    for (int c = 0; c < 16; ++c) acc[p][c] = 0.0f;
  const float* wp = w_s + gi * kDirectGroupStride;
  auto fma16 = [&](const float (&x)[kPX], int k) {
    const float4* w4 = reinterpret_cast<const float4*>(wp + k * G * kDirectGroupStride);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 w = w4[q];
#pragma unroll
      for (int p = 0; p < kPX; ++p) {
        acc[p][4 * q] = fmaf(x[p], w.x, acc[p][4 * q]);
        acc[p][4 * q + 1] = fmaf(x[p], w.y, acc[p][4 * q + 1]);
        acc[p][4 * q + 2] = fmaf(x[p], w.z, acc[p][4 * q + 2]);
        acc[p][4 * q + 3] = fmaf(x[p], w.w, acc[p][4 * q + 3]);
      }
    }
  };
  auto tap = [&](int fy, int fx, int k0, int cin) {
    const float* src[kPX];
    bool inside[kPX];
#pragma unroll
    for (int p = 0; p < kPX; ++p) {
      const int iy = iy0[p] + fy * g.dh, ix = ix0[p] + fx * g.dw;
      inside[p] = ok[p] && static_cast<unsigned>(iy) < static_cast<unsigned>(g.H) &&
                  static_cast<unsigned>(ix) < static_cast<unsigned>(g.W);
      src[p] = in + (ibase[p] + static_cast<long long>(iy) * g.W + ix) * cin;
    }
    if (CIN_ > 0 && CIN_ % 4 == 0) {
#pragma unroll
      for (int c4 = 0; c4 < (CIN_ > 0 ? CIN_ / 4 : 1); ++c4) {
        float4 v[kPX];
#pragma unroll
        for (int p = 0; p < kPX; ++p)
          v[p] = inside[p] ? __ldg(reinterpret_cast<const float4*>(src[p]) + c4)
                           : make_float4(0.f, 0.f, 0.f, 0.f);
        float x[kPX];
#pragma unroll
        for (int p = 0; p < kPX; ++p) x[p] = v[p].x;
        fma16(x, k0 + c4 * 4);
#pragma unroll
        for (int p = 0; p < kPX; ++p) x[p] = v[p].y;
        fma16(x, k0 + c4 * 4 + 1);
#pragma unroll
        for (int p = 0; p < kPX; ++p) x[p] = v[p].z;
        fma16(x, k0 + c4 * 4 + 2);
#pragma unroll
        for (int p = 0; p < kPX; ++p) x[p] = v[p].w;
        fma16(x, k0 + c4 * 4 + 3);
      }
    } else {
      for (int ci = 0; ci < cin; ++ci) {
        float x[kPX];
#pragma unroll
        for (int p = 0; p < kPX; ++p) x[p] = inside[p] ? __ldg(src[p] + ci) : 0.0f;
        fma16(x, k0 + ci);
      }
    }
  };
  if (KH_ > 0) {
#pragma unroll
    for (int fy = 0; fy < (KH_ > 0 ? KH_ : 1); ++fy)
#pragma unroll
      for (int fx = 0; fx < (KW_ > 0 ? KW_ : 1); ++fx) tap(fy, fx, (fy * KW_ + fx) * CIN_, CIN_);
  } else {
    for (int fy = 0; fy < KH; ++fy)
      for (int fx = 0; fx < KW; ++fx) tap(fy, fx, (fy * KW + fx) * CIN, CIN);
  }
  const int c0 = gi * 16;
  const float* bb = b_s + c0;
#pragma unroll
  for (int p = 0; p < kPX; ++p) {
    const long long m = static_cast<long long>(blk_m0) + p * px_per_blk + lpx;
    uint32_t bits = 0;
    if (ok[p]) {
      float* o = out + m * g.Cout + c0;
      if (c0 + 16 <= g.Cout && (g.Cout & 3) == 0) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 v = make_float4(apply_act(acc[p][4 * q] + bb[4 * q], g.act),
                                       apply_act(acc[p][4 * q + 1] + bb[4 * q + 1], g.act),
                                       apply_act(acc[p][4 * q + 2] + bb[4 * q + 2], g.act),
                                       apply_act(acc[p][4 * q + 3] + bb[4 * q + 3], g.act));
          reinterpret_cast<float4*>(o)[q] = v;
          bits |= ((v.x < 0.0f ? 1u : 0u) | (v.y < 0.0f ? 2u : 0u) | (v.z < 0.0f ? 4u : 0u) |
                   (v.w < 0.0f ? 8u : 0u)) << (4 * q);
        }
      } else {
        for (int c = 0; c < 16 && c0 + c < g.Cout; ++c) o[c] = apply_act(acc[p][c] + bb[c], g.act);
      }
    }
    if (packed != nullptr) {
      // fused LceQuantize (host guarantees Cout % 32 == 0 and an even group count): lanes gi and
      // gi ^ 1 are neighbours and hold the two halves of one word; every lane runs the shuffle
      uint32_t v = bits << ((gi & 1) * 16);
      v |= __shfl_xor_sync(0xffffffffu, v, 1);
      if (ok[p] && (gi & 1) == 0) packed[m * (g.Cout >> 5) + (gi >> 1)] = static_cast<int32_t>(v);
    }
  }
  }  // tile
}

// ---- plain-GEMM convolution (1x1, stride 1: A = [M, K] row-major): 128x128x16 tiles, 8x8
// outputs per thread, 128-bit global loads along K, register-prefetch double buffering ----
constexpr int kPM = 128, kPN = 128, kPK = 16;
__global__ void __launch_bounds__(256, 2) conv_gemm128_kernel(const float* __restrict__ A,
                                                           const float* __restrict__ Wt,
                                                           const float* __restrict__ bias,
                                                           float* __restrict__ out, long long M,
                                                           int N, int K, int act,
                                                           int32_t* __restrict__ packed) {
  __shared__ __align__(16) float A_s[2][kPK][kPM + 4];
  __shared__ __align__(16) float B_s[2][kPK][kPN + 4];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const long long m0 = static_cast<long long>(blockIdx.x) * kPM;
  const int n0 = blockIdx.y * kPN;
  // loader mapping: 2 float4 of A and 2 of B per thread per K-chunk
  const int lrow = tid >> 2;          // 0..63 (+64)
  const int lk = (tid & 3) * 4;       // 0,4,8,12
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
  float4 ra[2], rb[2];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const long long m = m0 + lrow + 64 * h;
      const int n = n0 + lrow + 64 * h;
      const int k = k0 + lk;
      ra[h] = (m < M && k < K) ? __ldg(reinterpret_cast<const float4*>(A + m * K + k))
                               : make_float4(0.f, 0.f, 0.f, 0.f);
      rb[h] = (n < N && k < K) ? __ldg(reinterpret_cast<const float4*>(Wt + static_cast<size_t>(n) * K + k))
                               : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto stash = [&](int buf) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int r = lrow + 64 * h;
      A_s[buf][lk][r] = ra[h].x; A_s[buf][lk + 1][r] = ra[h].y;
      A_s[buf][lk + 2][r] = ra[h].z; A_s[buf][lk + 3][r] = ra[h].w;
      B_s[buf][lk][r] = rb[h].x; B_s[buf][lk + 1][r] = rb[h].y;
      B_s[buf][lk + 2][r] = rb[h].z; B_s[buf][lk + 3][r] = rb[h].w;
    }
  };
  fetch(0);
  stash(0);
  __syncthreads();
  const int nk = (K + kPK - 1) / kPK;
  for (int it = 0; it < nk; ++it) {
    const int buf = it & 1;
    if (it + 1 < nk) fetch((it + 1) * kPK);
#pragma unroll
    for (int kk = 0; kk < kPK; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&A_s[buf][kk][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&A_s[buf][kk][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&B_s[buf][kk][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&B_s[buf][kk][64 + tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (it + 1 < nk) {
      stash(buf ^ 1);
      __syncthreads();
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const long long m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    const bool row_ok = m < M;
#pragma unroll
    for (int jh = 0; jh < 2; ++jh) {
      const int n = n0 + jh * 64 + tx * 4;
      float v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q)
        v[q] = apply_act(acc[i][jh * 4 + q] + ((bias && n + q < N) ? bias[n + q] : 0.0f), act);
      if (row_ok) {
        float* o = out + m * N + n;
        if (n + 3 < N && (N & 3) == 0) *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
        else
          for (int q = 0; q < 4 && n + q < N; ++q) o[q] = v[q];
      }
      if (packed != nullptr) {
        // fused LceQuantize (host guarantees N % 32 == 0): the 8 lanes tx & 7 = 0..7 hold one word
        uint32_t w = ((v[0] < 0.0f ? 1u : 0u) | (v[1] < 0.0f ? 2u : 0u) | (v[2] < 0.0f ? 4u : 0u) |
                      (v[3] < 0.0f ? 8u : 0u)) << ((tx & 7) * 4);
        w |= __shfl_xor_sync(0xffffffffu, w, 1);
        w |= __shfl_xor_sync(0xffffffffu, w, 2);
        w |= __shfl_xor_sync(0xffffffffu, w, 4);
        if (row_ok && (tx & 7) == 0 && n < N)
          packed[m * (N >> 5) + ((n0 + jh * 64) >> 5) + (tx >> 3)] = static_cast<int32_t>(w);
      }
    }
  }
}

// ---- plain GEMM for few output rows (FULLY_CONNECTED at batch 256: a 128 x 128 tiling would
// give 16 CTAs to 148 SMs): 32 x 64 tiles, 2 x 4 outputs per thread, K chunks of 32 ----
constexpr int kSM_ = 32, kSN_ = 64, kSK_ = 32;
__global__ void __launch_bounds__(256) gemm_small_m_kernel(const float* __restrict__ A,
                                                           const float* __restrict__ Wt,
                                                           const float* __restrict__ bias,
                                                           float* __restrict__ out, long long M,
                                                           int N, int K, int act) {
  __shared__ __align__(16) float A_s[kSK_][kSM_ + 2];
  __shared__ __align__(16) float B_s[kSK_][kSN_ + 4];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const long long m0 = static_cast<long long>(blockIdx.x) * kSM_;
  const int n0 = blockIdx.y * kSN_;
  const int arow = tid >> 3, akq = (tid & 7) * 4;      // A: 32 rows x 8 float4
  const int bcol = tid >> 2, bkq = (tid & 3) * 8;      // B: 64 cols x 4 x 2 float4
  float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
  for (int k0 = 0; k0 < K; k0 += kSK_) {
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 a = (m0 + arow < M && k0 + akq < K)
                         ? __ldg(reinterpret_cast<const float4*>(A + (m0 + arow) * K + k0 + akq)) : z;
    float4 b[2];
#pragma unroll
    for (int h = 0; h < 2; ++h)
      b[h] = (n0 + bcol < N && k0 + bkq + 4 * h < K)
                 ? __ldg(reinterpret_cast<const float4*>(Wt + static_cast<size_t>(n0 + bcol) * K +
                                                         k0 + bkq + 4 * h)) : z;
    A_s[akq][arow] = a.x; A_s[akq + 1][arow] = a.y; A_s[akq + 2][arow] = a.z; A_s[akq + 3][arow] = a.w;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      B_s[bkq + 4 * h][bcol] = b[h].x; B_s[bkq + 4 * h + 1][bcol] = b[h].y;
      B_s[bkq + 4 * h + 2][bcol] = b[h].z; B_s[bkq + 4 * h + 3][bcol] = b[h].w;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kSK_; ++kk) {
      const float2 av = *reinterpret_cast<const float2*>(&A_s[kk][ty * 2]);
      const float4 bv = *reinterpret_cast<const float4*>(&B_s[kk][tx * 4]);
      acc[0][0] = fmaf(av.x, bv.x, acc[0][0]); acc[0][1] = fmaf(av.x, bv.y, acc[0][1]);
      acc[0][2] = fmaf(av.x, bv.z, acc[0][2]); acc[0][3] = fmaf(av.x, bv.w, acc[0][3]);
      acc[1][0] = fmaf(av.y, bv.x, acc[1][0]); acc[1][1] = fmaf(av.y, bv.y, acc[1][1]);
      acc[1][2] = fmaf(av.y, bv.z, acc[1][2]); acc[1][3] = fmaf(av.y, bv.w, acc[1][3]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const long long m = m0 + ty * 2 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n < N) out[m * N + n] = apply_act(acc[i][j] + (bias ? bias[n] : 0.0f), act);
    }
  }
}

// ---- implicit-GEMM convolution, any filter / stride / dilation: 128 pixels x 64 channels x 16
// tiles, 8 x 4 outputs per thread, register-prefetch double buffering. The k -> (tap, channel)
// decomposition is tabulated once per CTA in shared memory (offset inside the image and the
// (dy, dx) displacement for the bounds test), so the gather costs ~8 instructions per element
// instead of three divisions. Bi-RealNet's 7x7x3 stem (K = 147) runs here.
constexpr int kIM = 128, kIN = 64, kIK = 16, kIKMax = 4096;
__global__ void __launch_bounds__(256, 2) conv_igemm_kernel(const float* __restrict__ in,
                                                            const float* __restrict__ filter,
                                                            const float* __restrict__ bias,
                                                            float* __restrict__ out, ConvGeom g,
                                                            long long M) {
  __shared__ __align__(16) float A_s[2][kIK][kIM + 4];
  __shared__ __align__(16) float B_s[2][kIK][kIN + 4];
  extern __shared__ int ktab[];  // [Kpad] element offset, [Kpad] (dy << 16) | dx
  const int K = g.KH * g.KW * g.Cin;
  const int Kpad = (K + kIK - 1) / kIK * kIK;
  int* koff = ktab;
  int* kdydx = ktab + Kpad;
  const int tid = threadIdx.x;
  for (int k = tid; k < Kpad; k += 256) {
    if (k < K) {
      const int tap = k / g.Cin, ci = k - tap * g.Cin;
      const int fy = tap / g.KW, fx = tap - fy * g.KW;
      koff[k] = (fy * g.dh * g.W + fx * g.dw) * g.Cin + ci;
      kdydx[k] = ((fy * g.dh) << 16) | (fx * g.dw);
    } else {
      koff[k] = 0;
      kdydx[k] = 0x7fff7fff;  // fails every bounds test
    }
  }
  const long long m0 = static_cast<long long>(blockIdx.x) * kIM;
  const int n0 = blockIdx.y * kIN;
  // loader roles: A -- row (tid & 127), 8 consecutive k; B -- channel (tid >> 2), 4 consecutive k
  const int lrow = tid & (kIM - 1);
  const int lkh = (tid >> 7) * 8;
  const int bn = tid >> 2, bkq = (tid & 3) * 4;
  int iy0 = 0, ix0 = 0;
  const float* base = in;
  bool row_ok = m0 + lrow < M;
  if (row_ok) {
    const long long m = m0 + lrow;
    const int ohw = g.OH * g.OW;
    const long long b = m / ohw;
    const int r = static_cast<int>(m - b * ohw);
    const int oy = r / g.OW, ox = r - oy * g.OW;
    iy0 = oy * g.sh - g.ph;
    ix0 = ox * g.sw - g.pw;
    base = in + ((b * g.H + iy0) * g.W + ix0) * g.Cin;  // dereferenced only where in bounds
  }
  const bool bn_ok = n0 + bn < g.Cout;
  const float* wrow = filter + static_cast<size_t>(bn_ok ? n0 + bn : 0) * K;
  __syncthreads();

  float ra[8], rb[4];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = k0 + lkh + e;
      const int d = kdydx[k];
      const int iy = iy0 + (d >> 16), ix = ix0 + (d & 0xffff);
      const bool ok = row_ok && static_cast<unsigned>(iy) < static_cast<unsigned>(g.H) &&
                      static_cast<unsigned>(ix) < static_cast<unsigned>(g.W);
      ra[e] = ok ? __ldg(base + koff[k]) : 0.0f;
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = k0 + bkq + e;
      rb[e] = (bn_ok && k < K) ? __ldg(wrow + k) : 0.0f;
    }
  };
  auto stash = [&](int buf) {
#pragma unroll
    for (int e = 0; e < 8; ++e) A_s[buf][lkh + e][lrow] = ra[e];
#pragma unroll
    for (int e = 0; e < 4; ++e) B_s[buf][bkq + e][bn] = rb[e];
  };
  const int tx = tid & 15, ty = tid >> 4;
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
  fetch(0);
  stash(0);
  __syncthreads();
  const int nk = Kpad / kIK;
  for (int it = 0; it < nk; ++it) {
    const int buf = it & 1;
    if (it + 1 < nk) fetch((it + 1) * kIK);
#pragma unroll
    for (int kk = 0; kk < kIK; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&A_s[buf][kk][ty * 8]);
      const float4 a1 = *reinterpret_cast<const float4*>(&A_s[buf][kk][ty * 8 + 4]);
      const float4 b = *reinterpret_cast<const float4*>(&B_s[buf][kk][tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (it + 1 < nk) {
      stash(buf ^ 1);
      __syncthreads();
    }
  }
  const int n = n0 + tx * 4;
  float bb[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) bb[q] = (bias && n + q < g.Cout) ? bias[n + q] : 0.0f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const long long m = m0 + ty * 8 + i;
    if (m >= M) continue;
    float v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) v[q] = apply_act(acc[i][q] + bb[q], g.act);
    float* o = out + m * g.Cout + n;
    if (n + 3 < g.Cout && (g.Cout & 3) == 0 && !(reinterpret_cast<uintptr_t>(out) & 15))
      *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
    else
      for (int q = 0; q < 4 && n + q < g.Cout; ++q) o[q] = v[q];
  }
}

// Same tiling with 128 threads and 8 x 8 outputs per thread (rows {ty*4.., 64+ty*4..}, channels
// {tx*4.., 32+tx*4..}): half the shared-memory reads per FMA of the 8 x 4 variant, whose ncu
// profile on Bi-RealNet's stem showed the LSU / shared-memory pipe at 61-75 % next to 53 % FMA.
__global__ void __launch_bounds__(128, 4) conv_igemm8x8_kernel(const float* __restrict__ in,
                                                               const float* __restrict__ filter,
                                                               const float* __restrict__ bias,
                                                               float* __restrict__ out, ConvGeom g,
                                                               long long M) {
  __shared__ __align__(16) float A_s[2][kIK][kIM + 4];
  __shared__ __align__(16) float B_s[2][kIK][kIN + 4];
  extern __shared__ int ktab[];
  const int K = g.KH * g.KW * g.Cin;
  const int Kpad = (K + kIK - 1) / kIK * kIK;
  int* koff = ktab;
  int* kdydx = ktab + Kpad;
  const int tid = threadIdx.x;
  for (int k = tid; k < Kpad; k += 128) {
    if (k < K) {
      const int tap = k / g.Cin, ci = k - tap * g.Cin;
      const int fy = tap / g.KW, fx = tap - fy * g.KW;
      koff[k] = (fy * g.dh * g.W + fx * g.dw) * g.Cin + ci;
      kdydx[k] = ((fy * g.dh) << 16) | (fx * g.dw);
    } else {
      koff[k] = 0;
      kdydx[k] = 0x7fff7fff;
    }
  }
  const long long m0 = static_cast<long long>(blockIdx.x) * kIM;
  const int n0 = blockIdx.y * kIN;
  // loader roles: A -- row tid, all 16 k of the chunk; B -- channel tid >> 1, 8 consecutive k
  const int lrow = tid;
  const int bn = tid >> 1, bkq = (tid & 1) * 8;
  int iy0 = 0, ix0 = 0;
  const float* base = in;
  const bool row_ok = m0 + lrow < M;
  if (row_ok) {
    const long long m = m0 + lrow;
    const int ohw = g.OH * g.OW;
    const long long b = m / ohw;
    const int r = static_cast<int>(m - b * ohw);
    const int oy = r / g.OW, ox = r - oy * g.OW;
    iy0 = oy * g.sh - g.ph;
    ix0 = ox * g.sw - g.pw;
    base = in + ((b * g.H + iy0) * g.W + ix0) * g.Cin;
  }
  const bool bn_ok = n0 + bn < g.Cout;
  const float* wrow = filter + static_cast<size_t>(bn_ok ? n0 + bn : 0) * K;
  __syncthreads();

  float ra[16], rb[8];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      const int k = k0 + e;
      const int d = kdydx[k];
      const int iy = iy0 + (d >> 16), ix = ix0 + (d & 0xffff);
      const bool ok = row_ok && static_cast<unsigned>(iy) < static_cast<unsigned>(g.H) &&
                      static_cast<unsigned>(ix) < static_cast<unsigned>(g.W);
      ra[e] = ok ? __ldg(base + koff[k]) : 0.0f;
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = k0 + bkq + e;
      rb[e] = (bn_ok && k < K) ? __ldg(wrow + k) : 0.0f;
    }
  };
  auto stash = [&](int buf) {
#pragma unroll
    for (int e = 0; e < 16; ++e) A_s[buf][e][lrow] = ra[e];
#pragma unroll
    for (int e = 0; e < 8; ++e) B_s[buf][bkq + e][bn] = rb[e];
  };
  const int tx = tid & 7, ty = tid >> 3;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
  fetch(0);
  stash(0);
  __syncthreads();
  const int nk = Kpad / kIK;
  for (int it = 0; it < nk; ++it) {
    const int buf = it & 1;
    if (it + 1 < nk) fetch((it + 1) * kIK);
#pragma unroll
    for (int kk = 0; kk < kIK; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&A_s[buf][kk][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&A_s[buf][kk][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&B_s[buf][kk][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&B_s[buf][kk][32 + tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (it + 1 < nk) {
      stash(buf ^ 1);
      __syncthreads();
    }
  }
  const bool vec = (g.Cout & 3) == 0 && !(reinterpret_cast<uintptr_t>(out) & 15);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const long long m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (m >= M) continue;
#pragma unroll
    for (int jh = 0; jh < 2; ++jh) {
      const int n = n0 + jh * 32 + tx * 4;
      float v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q)
        v[q] = apply_act(acc[i][jh * 4 + q] + ((bias && n + q < g.Cout) ? bias[n + q] : 0.0f), g.act);
      float* o = out + m * g.Cout + n;
      if (vec && n + 3 < g.Cout) *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
      else
        for (int q = 0; q < 4 && n + q < g.Cout; ++q) o[q] = v[q];
    }
  }
}

// ---- general implicit-GEMM convolution: 64x64x16 tiles, 4x4 per thread (fallback for K > 4096) ----------
constexpr int kGM = 64, kGN = 64, kGK = 16;
__global__ void __launch_bounds__(256) conv_gemm_kernel(const float* __restrict__ in,
                                                        const float* __restrict__ filter,
                                                        const float* __restrict__ bias,
                                                        float* __restrict__ out, ConvGeom g,
                                                        long long M) {
  __shared__ __align__(16) float A_s[kGK][kGM + 4];
  __shared__ __align__(16) float B_s[kGK][kGN + 4];
  __shared__ long long pix_base[kGM];  // offset of (b, iy0, ix0) or -1 for rows past M
  __shared__ int pix_iy0[kGM], pix_ix0[kGM];
  const int K = g.KH * g.KW * g.Cin;
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const long long m0 = static_cast<long long>(blockIdx.x) * kGM;
  const int n0 = blockIdx.y * kGN;
  if (tid < kGM) {
    const long long m = m0 + tid;
    if (m < M) {
      const int ohw = g.OH * g.OW;
      const long long b = m / ohw;
      const int r = static_cast<int>(m - b * ohw);
      const int oy = r / g.OW, ox = r - oy * g.OW;
      pix_iy0[tid] = oy * g.sh - g.ph;
      pix_ix0[tid] = ox * g.sw - g.pw;
      pix_base[tid] = b * g.H * g.W;
    } else {
      pix_base[tid] = -1;
      pix_iy0[tid] = pix_ix0[tid] = 0;
    }
  }
  __syncthreads();
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

  const int lk = tid & 15;   // k within the chunk handled by this thread when loading
  const int lr = tid >> 4;   // row group: rows lr, lr+16, lr+32, lr+48
  for (int k0 = 0; k0 < K; k0 += kGK) {
    const int k = k0 + lk;
    int fy = 0, fx = 0, ci = 0;
    const bool k_ok = k < K;
    if (k_ok) {
      const int tap = k / g.Cin;
      ci = k - tap * g.Cin;
      fy = tap / g.KW;
      fx = tap - fy * g.KW;
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int row = lr + 16 * q;
      float v = 0.0f;
      if (k_ok && pix_base[row] >= 0) {
        const int iy = pix_iy0[row] + fy * g.dh, ix = pix_ix0[row] + fx * g.dw;
        if (static_cast<unsigned>(iy) < static_cast<unsigned>(g.H) &&
            static_cast<unsigned>(ix) < static_cast<unsigned>(g.W))
          v = __ldg(in + (pix_base[row] + static_cast<long long>(iy) * g.W + ix) * g.Cin + ci);
      }
      A_s[lk][row] = v;
      const int n = n0 + row;
      B_s[lk][row] = (k_ok && n < g.Cout) ? __ldg(filter + static_cast<size_t>(n) * K + k) : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kGK; ++kk) {
      const float4 a = *reinterpret_cast<const float4*>(&A_s[kk][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&B_s[kk][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n < g.Cout) out[m * g.Cout + n] = apply_act(acc[i][j] + (bias ? bias[n] : 0.0f), g.act);
    }
  }
}

__global__ void __launch_bounds__(256) depthwise_kernel(const float* __restrict__ in,
                                                        const float* __restrict__ filter,
                                                        const float* __restrict__ bias,
                                                        float* __restrict__ out, ConvGeom g,
                                                        long long n) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += stride) {
    const int c = static_cast<int>(i % g.Cout);
    long long r = i / g.Cout;
    const int ox = static_cast<int>(r % g.OW);
    r /= g.OW;
    const int oy = static_cast<int>(r % g.OH);
    const long long b = r / g.OH;
    float acc = 0.0f;
    for (int fy = 0; fy < g.KH; ++fy) {
      const int iy = oy * g.sh - g.ph + fy * g.dh;
      if (static_cast<unsigned>(iy) >= static_cast<unsigned>(g.H)) continue;
      for (int fx = 0; fx < g.KW; ++fx) {
        const int ix = ox * g.sw - g.pw + fx * g.dw;
        if (static_cast<unsigned>(ix) >= static_cast<unsigned>(g.W)) continue;
        acc = fmaf(__ldg(in + ((b * g.H + iy) * g.W + ix) * g.Cin + c),
                   __ldg(filter + (fy * g.KW + fx) * g.Cout + c), acc);
      }
    }
    out[i] = apply_act(acc + (bias ? bias[c] : 0.0f), g.act);
  }
}

// 4 channels per thread (C % 4 == 0): 128-bit loads of inputs, weights and outputs. 3-D grid
// (x: (ox, c4), y: oy, z: batch) -- the flat-index version spent most of its instructions on
// integer div/mod (ncu: issue-bound at ~30 % of DRAM bandwidth).
template <int KHW>   // KHW = 3: 3x3 window fully unrolled (all loads in flight); 0: runtime
__global__ void __launch_bounds__(256) depthwise_v4_kernel(const float4* __restrict__ in,
                                                           const float4* __restrict__ filter,
                                                           const float4* __restrict__ bias,
                                                           float4* __restrict__ out, ConvGeom g) {
  const int C4 = g.Cout >> 2;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= g.OW * C4) return;
  const int ox = i / C4, c = i - ox * C4;
  const int oy = blockIdx.y;
  const long long b = blockIdx.z;
  const int KH = KHW ? KHW : g.KH, KW = KHW ? KHW : g.KW;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  const float4* img = in + b * g.H * g.W * C4 + c;
#pragma unroll
  for (int fy = 0; fy < KH; ++fy) {
    const int iy = oy * g.sh - g.ph + fy * g.dh;
    if (static_cast<unsigned>(iy) >= static_cast<unsigned>(g.H)) continue;
#pragma unroll
    for (int fx = 0; fx < KW; ++fx) {
      const int ix = ox * g.sw - g.pw + fx * g.dw;
      if (static_cast<unsigned>(ix) >= static_cast<unsigned>(g.W)) continue;
      const float4 x = __ldg(img + (static_cast<long long>(iy) * g.W + ix) * C4);
      const float4 w = __ldg(filter + (fy * KW + fx) * C4 + c);
      acc.x = fmaf(x.x, w.x, acc.x); acc.y = fmaf(x.y, w.y, acc.y);
      acc.z = fmaf(x.z, w.z, acc.z); acc.w = fmaf(x.w, w.w, acc.w);
    }
  }
  float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
  if (bias) bb = __ldg(bias + c);
  out[((b * g.OH + oy) * g.OW + ox) * C4 + c] =
      make_float4(apply_act(acc.x + bb.x, g.act), apply_act(acc.y + bb.y, g.act),
                  apply_act(acc.z + bb.z, g.act), apply_act(acc.w + bb.w, g.act));
}

template <bool MAX, int FHW>   // FHW = 2 / 3: window fully unrolled; 0: runtime
__global__ void __launch_bounds__(256) pool_v4_kernel(const float4* __restrict__ in,
                                                      float4* __restrict__ out, int H, int W,
                                                      int C4, int OH, int OW, int fh_, int fw_,
                                                      int sh, int sw, int ph, int pw, int act) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= OW * C4) return;
  const int ox = i / C4, c = i - ox * C4;
  const int oy = blockIdx.y;
  const long long b = blockIdx.z;
  const int fh = FHW ? FHW : fh_, fw = FHW ? FHW : fw_;
  const int y0 = oy * sh - ph, x0 = ox * sw - pw;
  const float4* img = in + b * H * W * C4 + c;
  float4 v = MAX ? make_float4(-FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX)
                 : make_float4(0.f, 0.f, 0.f, 0.f);
  int cnt = 0;
#pragma unroll
  for (int fy = 0; fy < fh; ++fy) {
    const int y = y0 + fy;
    if (static_cast<unsigned>(y) >= static_cast<unsigned>(H)) continue;
#pragma unroll
    for (int fx = 0; fx < fw; ++fx) {
      const int x = x0 + fx;
      if (static_cast<unsigned>(x) >= static_cast<unsigned>(W)) continue;
      const float4 e = __ldg(img + (static_cast<long long>(y) * W + x) * C4);
      ++cnt;
      if (MAX) { v.x = fmaxf(v.x, e.x); v.y = fmaxf(v.y, e.y); v.z = fmaxf(v.z, e.z); v.w = fmaxf(v.w, e.w); }
      else { v.x += e.x; v.y += e.y; v.z += e.z; v.w += e.w; }
    }
  }
  if (!MAX) {
    const float d = static_cast<float>(max(1, cnt));
    v.x = v.x / d; v.y = v.y / d; v.z = v.z / d; v.w = v.w / d;
  }
  out[((b * OH + oy) * OW + ox) * C4 + c] =
      make_float4(apply_act(v.x, act), apply_act(v.y, act), apply_act(v.z, act),
                  apply_act(v.w, act));
}

// max-pool 2x2 / stride 1 / VALID fused into the depthwise 3x3 that consumes it: one thread =
// one output pixel x 4 channels; the 4x4 input window is loaded once (16 x LDG.128), the nine
// pooled values are formed in registers and multiplied in the same (fy, fx) order as
// depthwise_v4_kernel, so the result is bit-identical to the two-kernel sequence.
#ifndef LCE_POOL_MINBLOCKS
#define LCE_POOL_MINBLOCKS 4
#endif
__global__ void __launch_bounds__(256, LCE_POOL_MINBLOCKS) pool2_dw3_v4_kernel(const float4* __restrict__ in,
                                                              const float4* __restrict__ filter,
                                                              const float4* __restrict__ bias,
                                                              float4* __restrict__ out, int H, int W,
                                                              int C4, int PH, int PW, int OH, int OW,
                                                              int sh, int sw, int ph, int pw, int act) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= OW * C4) return;
  const int ox = i / C4, c = i - ox * C4;
  const int oy = blockIdx.y;
  const long long b = blockIdx.z;
  const int y0 = oy * sh - ph, x0 = ox * sw - pw;   // top-left pooled coordinate of the window
  const float4* img = in + b * H * W * C4 + c;
  const float4 lowest = make_float4(-FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX);
  auto vmax = [](const float4& a, const float4& q) {
    return make_float4(fmaxf(a.x, q.x), fmaxf(a.y, q.y), fmaxf(a.z, q.z), fmaxf(a.w, q.w));
  };
  // Interior windows (all 4 x 4 inputs and 3 x 3 pooled values exist; the whole warp agrees): the
  // same arithmetic in the same order with one base pointer and two constant strides. The general
  // path below spends 250 of its 600 instructions on per-load index arithmetic and predicates, and
  // the kernel is issue-bound (ncu: 68 % issue utilisation at half the HBM rate).
  if (__all_sync(__activemask(), y0 >= 0 && x0 >= 0 && y0 + 3 < H && x0 + 3 < W && y0 + 2 < PH && x0 + 2 < PW)) {
    const size_t cs = static_cast<size_t>(C4), rs = static_cast<size_t>(W) * cs;
    const float4* p0 = img + (static_cast<size_t>(y0) * W + x0) * cs;
    const float4* wp = filter + c;
    float4 hp[3];
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int dy = 0; dy < 4; ++dy) {
      const float4* row = p0 + dy * rs;
      const float4 v0 = __ldg(row), v1 = __ldg(row + cs), v2 = __ldg(row + 2 * cs), v3 = __ldg(row + 3 * cs);
      float4 h[3] = {vmax(v0, v1), vmax(v1, v2), vmax(v2, v3)};
      if (dy > 0) {
#pragma unroll
        for (int fx = 0; fx < 3; ++fx) {
          const float4 m = vmax(lowest, vmax(hp[fx], h[fx]));
          const float4 w = __ldg(wp + ((dy - 1) * 3 + fx) * cs);
          acc.x = fmaf(m.x, w.x, acc.x); acc.y = fmaf(m.y, w.y, acc.y);
          acc.z = fmaf(m.z, w.z, acc.z); acc.w = fmaf(m.w, w.w, acc.w);
        }
      }
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) hp[dx] = h[dx];
    }
    float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
    if (bias) bb = __ldg(bias + c);
    out[((b * OH + oy) * OW + ox) * C4 + c] =
        make_float4(apply_act(acc.x + bb.x, act), apply_act(acc.y + bb.y, act),
                    apply_act(acc.z + bb.z, act), apply_act(acc.w + bb.w, act));
    return;
  }
  // Row by row (one input row of 4 pixels live at a time: half the registers of holding the
  // 4 x 4 window, so twice the resident warps): h[x] = max(v[x], v[x+1]) per input row, a pooled
  // row is max(h of two consecutive input rows). max is exact in any order; the final
  // max(lowest, .) reproduces pool_v4_kernel's result for an all-NaN window too.
  bool xin[4];
#pragma unroll
  for (int dx = 0; dx < 4; ++dx) xin[dx] = static_cast<unsigned>(x0 + dx) < static_cast<unsigned>(W);
  float4 hp[3];   // h of the previous input row
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int dy = 0; dy < 4; ++dy) {
    const int y = y0 + dy;
    const bool yin = static_cast<unsigned>(y) < static_cast<unsigned>(H);
    const float4* row = img + (static_cast<long long>(y) * W + x0) * C4;
    float4 v[4];
#pragma unroll
    for (int dx = 0; dx < 4; ++dx) v[dx] = (yin && xin[dx]) ? __ldg(row + dx * C4) : lowest;
    float4 h[3];
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) h[dx] = vmax(v[dx], v[dx + 1]);
    if (dy > 0) {
      const int fy = dy - 1;
      const int py = y0 + fy;
      if (static_cast<unsigned>(py) < static_cast<unsigned>(PH)) {
#pragma unroll
        for (int fx = 0; fx < 3; ++fx) {
          const int px = x0 + fx;
          if (static_cast<unsigned>(px) >= static_cast<unsigned>(PW)) continue;
          const float4 m = vmax(lowest, vmax(hp[fx], h[fx]));
          const float4 w = __ldg(filter + (fy * 3 + fx) * C4 + c);
          acc.x = fmaf(m.x, w.x, acc.x); acc.y = fmaf(m.y, w.y, acc.y);
          acc.z = fmaf(m.z, w.z, acc.z); acc.w = fmaf(m.w, w.w, acc.w);
        }
      }
    }
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) hp[dx] = h[dx];
  }
  float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
  if (bias) bb = __ldg(bias + c);
  out[((b * OH + oy) * OW + ox) * C4 + c] =
      make_float4(apply_act(acc.x + bb.x, act), apply_act(acc.y + bb.y, act),
                  apply_act(acc.z + bb.z, act), apply_act(acc.w + bb.w, act));
}

template <bool MAX>
__global__ void __launch_bounds__(256) pool_kernel(const float* __restrict__ in,
                                                   float* __restrict__ out, int B, int H, int W,
                                                   int C, int OH, int OW, int fh, int fw, int sh,
                                                   int sw, int ph, int pw, int act) {
  const long long n = static_cast<long long>(B) * OH * OW * C;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += stride) {
    const int c = static_cast<int>(i % C);
    long long r = i / C;
    const int ox = static_cast<int>(r % OW);
    r /= OW;
    const int oy = static_cast<int>(r % OH);
    const long long b = r / OH;
    const int y0 = oy * sh - ph, x0 = ox * sw - pw;
    const int ys = max(0, y0), ye = min(H, y0 + fh), xs = max(0, x0), xe = min(W, x0 + fw);
    float v = MAX ? -FLT_MAX : 0.0f;
    for (int y = ys; y < ye; ++y)
      for (int x = xs; x < xe; ++x) {
        const float e = __ldg(in + ((b * H + y) * W + x) * C + c);
        v = MAX ? fmaxf(v, e) : v + e;
      }
    if (!MAX) v = v / static_cast<float>(max(1, (ye - ys) * (xe - xs)));  // pooling.h:60-78
    out[i] = apply_act(v, act);
  }
}

template <int OP>  // 0 add, 1 mul, 2 activation only
__global__ void __launch_bounds__(256) eltwise_kernel(const float* __restrict__ a,
                                                      const float* __restrict__ b,
                                                      float* __restrict__ out, long long n,
                                                      long long b_len, int act, int vec_ok) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  const long long t0 = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (vec_ok) {   // same shape, 16-byte aligned, n % 4 == 0: 128-bit path
    const float4* a4 = reinterpret_cast<const float4*>(a);
    const float4* b4 = reinterpret_cast<const float4*>(b);
    float4* o4 = reinterpret_cast<float4*>(out);
    for (long long i = t0; i < (n >> 2); i += stride) {
      float4 x = a4[i];
      if (OP != 2) {
        const float4 y = b4[i];
        if (OP == 0) { x.x += y.x; x.y += y.y; x.z += y.z; x.w += y.w; }
        else { x.x *= y.x; x.y *= y.y; x.z *= y.z; x.w *= y.w; }
      }
      o4[i] = make_float4(apply_act(x.x, act), apply_act(x.y, act), apply_act(x.z, act),
                          apply_act(x.w, act));
    }
    return;
  }
  for (long long i = t0; i < n; i += stride) {
    float x = a[i];
    if (OP == 0) x += b[i % b_len];
    if (OP == 1) x *= b[i % b_len];
    out[i] = apply_act(x, act);
  }
}

// mean over H*W: one thread per (b, c), c fastest => coalesced rows.
__global__ void __launch_bounds__(256) mean_hw_kernel(const float* __restrict__ in,
                                                      float* __restrict__ out, int B, int HW,
                                                      int C, int pre_act) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * C) return;
  const int b = i / C, c = i - b * C;
  const float* p = in + static_cast<size_t>(b) * HW * C + c;
  float s = 0.0f;
  for (int k = 0; k < HW; ++k) s += apply_act(p[static_cast<size_t>(k) * C], pre_act);
  out[i] = s / static_cast<float>(HW);
}

// softmax: one CTA of 128 threads per row (a warp per row left 256 rows on 32 CTAs); the row
// lives in registers between the three passes (<= 8 elements per thread, else re-read).
__global__ void __launch_bounds__(128) softmax_kernel(const float* __restrict__ in,
                                                      float* __restrict__ out, int cols, float beta) {
  __shared__ float red[4];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* x = in + static_cast<long long>(blockIdx.x) * cols;
  float* y = out + static_cast<long long>(blockIdx.x) * cols;
  constexpr int kR = 8;
  const bool in_regs = cols <= kR * 128;
  float v[kR];
  float mx = -FLT_MAX;
  if (in_regs) {
#pragma unroll
    for (int j = 0; j < kR; ++j) {
      const int c = tid + j * 128;
      v[j] = c < cols ? x[c] : -FLT_MAX;
      mx = fmaxf(mx, v[j]);
    }
  } else {
    for (int c = tid; c < cols; c += 128) mx = fmaxf(mx, x[c]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  mx = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
  __syncthreads();
  float sum = 0.0f;
  if (in_regs) {
#pragma unroll
    for (int j = 0; j < kR; ++j) {
      const int c = tid + j * 128;
      v[j] = c < cols ? expf((v[j] - mx) * beta) : 0.0f;
      sum += v[j];
    }
  } else {
    for (int c = tid; c < cols; c += 128) sum += expf((x[c] - mx) * beta);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  sum = (red[0] + red[1]) + (red[2] + red[3]);
  if (in_regs) {
#pragma unroll
    for (int j = 0; j < kR; ++j) {
      const int c = tid + j * 128;
      if (c < cols) y[c] = v[j] / sum;
    }
  } else {
    for (int c = tid; c < cols; c += 128) y[c] = expf((x[c] - mx) * beta) / sum;
  }
}

// constant pad of a 4-D tensor of 32-bit elements (float32, or bitpacked int32 words).
struct Pad4 { int in[4], out[4], before[4]; };
__global__ void __launch_bounds__(256) pad4d32_kernel(const uint32_t* __restrict__ in,
                                                      uint32_t* __restrict__ out, Pad4 p,
                                                      uint32_t fill, long long total) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i >= total) return;
  long long r = i;
  const int d3 = static_cast<int>(r % p.out[3]); r /= p.out[3];
  const int d2 = static_cast<int>(r % p.out[2]); r /= p.out[2];
  const int d1 = static_cast<int>(r % p.out[1]); r /= p.out[1];
  const int d0 = static_cast<int>(r);
  const int s0 = d0 - p.before[0], s1 = d1 - p.before[1], s2 = d2 - p.before[2],
            s3 = d3 - p.before[3];
  uint32_t v = fill;
  if (static_cast<unsigned>(s0) < static_cast<unsigned>(p.in[0]) &&
      static_cast<unsigned>(s1) < static_cast<unsigned>(p.in[1]) &&
      static_cast<unsigned>(s2) < static_cast<unsigned>(p.in[2]) &&
      static_cast<unsigned>(s3) < static_cast<unsigned>(p.in[3]))
    v = in[((static_cast<long long>(s0) * p.in[1] + s1) * p.in[2] + s2) * p.in[3] + s3];
  out[i] = v;
}

// ---- fused stem: [DEQUANTIZE ->] CONV_2D(3x3, stride 2, 3 -> 16) -> DEPTHWISE_CONV_2D(3x3,
// stride 2) in one pass (QuickNet's stem). Unfused, the dequantised image (154 MB at batch 256) and
// the first conv's map (205 MB) each make a round trip through HBM; fused, a step reads the int8
// image and writes the 51 MB depthwise map.
//   Persistent CTAs (one per SM, 512 threads). A tile = 4 output rows x <= 56 output columns of
// one image. Its 19 x 227 x 3 input patch is fetched as raw bytes (cp.async, double-buffered: the
// next tile's patch arrives while this one computes), padded in the QUANTISED domain (zero point;
// 0.0f for a float image); the 9 x 113 x 16 first-conv strip stays in shared memory. For byte
// images the CTA is two independent groups of 256 threads, each with its own tiles, patch buffers,
// strip and named barrier, so that one group's latency-bound phases (patch wait, depthwise stage,
// barriers) are covered by the other's FMA stage (142 -> 124 us at batch 256).
//   Stage 1: thread = 2 adjacent first-conv pixels x 16 channels. Per patch row it reads 15 input
// values (int8: 4 x LDS.32, then a 256-entry table of float(scale * (q - zero_point)) -- exactly
// DEQUANTIZE's values -- replicated per bank, so a lookup never conflicts) and issues 3 x 3 x 16
// FFMA2: two channels per instruction, the input value broadcast, the weight pair a constant-bank
// operand (the filters travel by value in the parameter bank). A three-register FFMA issues every
// other cycle on sm_100 (B300_MICROARCH.md: fma pipe rt_SMSP = 2); FFMA2 is what reaches the
// fp32 rate, and operands staged in shared memory were bound by the LDS pipe (4 wavefronts per
// LDS.128, broadcast or not) at a fifth of it.
//   Stage 2: thread = (output column, 4 channels, row pair); out-of-range taps are skipped.
// Every output is accumulated in the order of conv_direct16_kernel / depthwise_v4_kernel with the
// same IEEE fma, so the result is bit-identical to the separate kernels.
constexpr int kS2R = 4, kS2TW = 56;
constexpr int kS2R1 = 2 * kS2R + 1;            // 9 first-conv rows per tile
constexpr int kS2C1 = 2 * kS2TW + 1;           // 113 first-conv columns
constexpr int kS2R0 = 2 * kS2R1 + 1;           // 19 input rows
constexpr int kS2C0 = 2 * kS2C1 + 1;           // 227 input columns
constexpr int kS2RawCols = 240;                // fetched per row: 15 x 16 columns
constexpr int kS2Threads = 512;
struct Stem2Geom {
  int B, H, W, OH1, OW1, ph1, pw1, OH2, OW2, ph2, pw2, act1, act2;
  int n_rt, n_ct;        // row / column tiles per image
  int aligned;           // rows can be fetched with 16-byte cp.async
  int in_zero_point;
  double in_scale;
};
struct StemWeights {
  float w1[27][16];   // [tap * 3 + ci][co]
  float b1[16];
  float w2[9][16];    // [tap][c]
  float b2[16];
};
template <typename TIn>
struct Stem2Layout {
  static constexpr int kRawPitch = kS2RawCols * 3 * static_cast<int>(sizeof(TIn));          // 720 / 2880 B
  static constexpr int kLutBytes = sizeof(TIn) == 1 ? 256 * 32 * 4 : 0;
  // byte images: the CTA runs TWO independent groups of 256 threads, each on its own tile with its own
  // patch buffers and strip and its own named barrier -- while one group sits in the latency-bound
  // phases (patch wait, depthwise stage, barriers) the other keeps the FMA pipe busy. Float images
  // need 4x the patch memory: one group of 512 threads.
  static constexpr int kGroups = sizeof(TIn) == 1 ? 2 : 1;
  static constexpr int kC1Bufs = 1;
  static constexpr size_t kGroupRawBytes = 2 * static_cast<size_t>(kS2R0) * kRawPitch + 64;
  static constexpr size_t kSmemBytes = kGroups * (kGroupRawBytes + kC1Bufs * kS2R1 * kS2C1 * 64) + (9 * 16 + 16) * 4 + kLutBytes;
};

template <typename TIn, bool kUnsigned>
__global__ void __launch_bounds__(kS2Threads, 1)
stem_conv_dw_kernel(const TIn* __restrict__ in, float* __restrict__ out, const __grid_constant__ StemWeights Wt,
                    const Stem2Geom s) {
  extern __shared__ __align__(16) unsigned char sm_raw[];
  constexpr int kRawPitch = Stem2Layout<TIn>::kRawPitch;
  constexpr bool kQuant = sizeof(TIn) == 1;
  using Lay = Stem2Layout<TIn>;
  constexpr int kGroups = Lay::kGroups, kG = kS2Threads / kGroups;                // threads per group
  constexpr int kC1Bufs = Lay::kC1Bufs;
  constexpr int kC1Floats = kS2R1 * kS2C1 * 16;
  const int gid = threadIdx.x / kG, tid = threadIdx.x - gid * kG, lane = threadIdx.x & 31;   // tid: inside the group
  unsigned char* raw0 = sm_raw + gid * Lay::kGroupRawBytes;                       // [2][19][kRawPitch] (+ slack)
  float* c1_all = reinterpret_cast<float*>(sm_raw + kGroups * Lay::kGroupRawBytes);
  float* c1_0 = c1_all + gid * kC1Bufs * kC1Floats;                               // [kC1Bufs][9][113][16], swizzled
  float* w2s = c1_all + kGroups * kC1Bufs * kC1Floats;                            // [9][16]
  float* b2s = w2s + 9 * 16;
  float* lut = b2s + 16;                                                          // [256][32]
  auto group_barrier = [&]() {
    if (kGroups == 1) __syncthreads();
    else asm volatile("bar.sync %0, %1;" ::"r"(1 + gid), "r"(kG) : "memory");
  };

  for (int i = threadIdx.x; i < 9 * 16; i += kS2Threads) w2s[i] = Wt.w2[i >> 4][i & 15];
  if (threadIdx.x < 16) b2s[threadIdx.x] = Wt.b2[threadIdx.x];
  if (kQuant) {
    for (int i = threadIdx.x; i < 256 * 32; i += kS2Threads) {
      const int byte = i >> 5;
      const int q = kUnsigned ? byte : (byte < 128 ? byte : byte - 256);
      lut[i] = static_cast<float>(s.in_scale * static_cast<double>(q - s.in_zero_point));
    }
  }
  const TIn pad_value = kQuant ? static_cast<TIn>(s.in_zero_point) : static_cast<TIn>(0);

  const int tiles = s.B * s.n_rt * s.n_ct;
  struct Tile { int b, rt, ct, oy2_0, ox2_0, tw, y1_0, x1_0, y0_0, x0_0; };
  auto place = [&](Tile& T) {
    T.oy2_0 = T.rt * kS2R;
    T.ox2_0 = T.ct * kS2TW;
    T.tw = min(kS2TW, s.OW2 - T.ox2_0);
    T.y1_0 = T.oy2_0 * 2 - s.ph2; T.x1_0 = T.ox2_0 * 2 - s.pw2;
    T.y0_0 = T.y1_0 * 2 - s.ph1;  T.x0_0 = T.x1_0 * 2 - s.pw1;
  };
  // tile index -> (image, row tile, column tile) once; then a step of (groups in the grid) tiles by carries
  const int tile_step = static_cast<int>(gridDim.x) * kGroups;
  const int step_ct = tile_step % s.n_ct, step_r = tile_step / s.n_ct;
  const int step_rt = step_r % s.n_rt, step_b = step_r / s.n_rt;
  auto advance = [&](Tile& T) {
    T.ct += step_ct;
    if (T.ct >= s.n_ct) { T.ct -= s.n_ct; T.rt += 1; }
    T.rt += step_rt;
    if (T.rt >= s.n_rt) { T.rt -= s.n_rt; T.b += 1; }
    T.b += step_b;
    place(T);
  };
  // raw[r][j * 3 + ci] = input(y0_0 + r, x0_0 + j, ci) for j < 227, the pad value outside the image
  auto load_tile = [&](const Tile& T, unsigned char* raw) {
    const TIn* img = in + static_cast<long long>(T.b) * s.H * s.W * 3;
    if (s.aligned && T.x0_0 >= 0 && (T.x0_0 & 15) == 0) {
      const int xr1 = min(s.W, T.x0_0 + kS2RawCols);
      const int row_elems = (xr1 - T.x0_0) * 3;
      const int n16 = (row_elems * static_cast<int>(sizeof(TIn))) >> 4;      // whole chunks: see `aligned`
      for (int i = tid; i < kS2R0 * n16; i += kG) {
        const int r = i / n16, c = i - r * n16;
        const int y = T.y0_0 + r;
        if (static_cast<unsigned>(y) >= static_cast<unsigned>(s.H)) continue;
        const unsigned char* src = reinterpret_cast<const unsigned char*>(img + (static_cast<long long>(y) * s.W + T.x0_0) * 3) + c * 16;
        const uint32_t dst = static_cast<uint32_t>(__cvta_generic_to_shared(raw + r * kRawPitch + c * 16));
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
      }
      // rows above / below the image, and the columns right of it (bytes no chunk writes)
      const int tail = kS2C0 * 3 - row_elems;
      for (int r = 0; r < kS2R0; ++r) {
        TIn* rr = reinterpret_cast<TIn*>(raw + r * kRawPitch);
        if (static_cast<unsigned>(T.y0_0 + r) >= static_cast<unsigned>(s.H)) {
          for (int e = tid; e < kS2C0 * 3; e += kG) rr[e] = pad_value;
        } else if (tid < tail) {
          rr[row_elems + tid] = pad_value;
        }
      }
    } else {
      for (int i = tid; i < kS2R0 * kS2C0; i += kG) {
        const int r = i / kS2C0, j = i - r * kS2C0;
        const int y = T.y0_0 + r, x = T.x0_0 + j;
        TIn* dst = reinterpret_cast<TIn*>(raw + r * kRawPitch) + j * 3;
        if (static_cast<unsigned>(y) < static_cast<unsigned>(s.H) && static_cast<unsigned>(x) < static_cast<unsigned>(s.W)) {
          const TIn* src = img + (static_cast<long long>(y) * s.W + x) * 3;
          dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2];
        } else {
          dst[0] = pad_value; dst[1] = pad_value; dst[2] = pad_value;
        }
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };

  // ---- stage 1: first conv on the strip rows / columns that lie inside its map
  auto stage1 = [&](const Tile& T, const unsigned char* raw, float* c1) {
    const int l1_lo = max(0, -T.y1_0), l1_hi = min(kS2R1, s.OH1 - T.y1_0);
    const int cl_lo = max(0, -T.x1_0) & ~1, cl_hi = min(2 * T.tw + 1, s.OW1 - T.x1_0);
    if (l1_hi <= l1_lo || cl_hi <= cl_lo) return;
    const int tpr = (cl_hi - cl_lo + 1) >> 1;
    const int tasks = (l1_hi - l1_lo) * tpr;
    for (int task = tid; task < tasks; task += kG) {
      const int rr = task / tpr, tt = task - rr * tpr;
      const int l1 = l1_lo + rr, cg = cl_lo + 2 * tt;
      float2 acc[2][8];
#pragma unroll
      for (int p = 0; p < 2; ++p)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[p][c] = make_float2(0.0f, 0.0f);
      const unsigned char* row0 = raw + (2 * l1) * kRawPitch + 6 * cg * static_cast<int>(sizeof(TIn));
      // byte images: all 12 words of the three patch rows are requested before the first lookup
      uint32_t rw[3][4];
      if (kQuant) {
#pragma unroll
        for (int fy = 0; fy < 3; ++fy)
#pragma unroll
          for (int k = 0; k < 4; ++k) rw[fy][k] = reinterpret_cast<const uint32_t*>(row0 + fy * kRawPitch)[k];
      }
#pragma unroll
      for (int fy = 0; fy < 3; ++fy) {
        float xv[16];
        if (kQuant) {
          // 15 bytes from a 4-byte aligned start (cg is even), then table[byte][lane]
          const float* lt = lut + lane;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint32_t w = rw[fy][k];
            xv[4 * k] = lt[__byte_perm(w, 0, 0x4440) << 5];
            xv[4 * k + 1] = lt[__byte_perm(w, 0, 0x4441) << 5];
            xv[4 * k + 2] = lt[__byte_perm(w, 0, 0x4442) << 5];
            if (k < 3) xv[4 * k + 3] = lt[__byte_perm(w, 0, 0x4443) << 5];
          }
        } else {
          const float4* xr = reinterpret_cast<const float4*>(row0 + fy * kRawPitch);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float4 f = xr[k];
            xv[4 * k] = f.x; xv[4 * k + 1] = f.y; xv[4 * k + 2] = f.z; xv[4 * k + 3] = f.w;
          }
        }
#pragma unroll
        for (int fx = 0; fx < 3; ++fx)
#pragma unroll
          for (int ci = 0; ci < 3; ++ci) {
            const int kk = (fy * 3 + fx) * 3 + ci;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const float2 w = make_float2(Wt.w1[kk][2 * c], Wt.w1[kk][2 * c + 1]);
#pragma unroll
              for (int p = 0; p < 2; ++p) {
                const float x = xv[(2 * p + fx) * 3 + ci];
                acc[p][c] = __ffma2_rn(make_float2(x, x), w, acc[p][c]);
              }
            }
          }
      }
#pragma unroll
      for (int p = 0; p < 2; ++p) {
        const int cl = cg + p;
        if (cl >= cl_hi) continue;
        float* dst = c1 + (l1 * kS2C1 + cl) * 16;
        const int sw = (cl >> 1) & 3;   // 16-byte cell swizzle: neighbouring tasks hit different banks
#pragma unroll
        for (int q = 0; q < 4; ++q)
          *reinterpret_cast<float4*>(dst + ((q ^ sw) << 2)) =
              make_float4(apply_act(acc[p][2 * q].x + Wt.b1[4 * q], s.act1), apply_act(acc[p][2 * q].y + Wt.b1[4 * q + 1], s.act1),
                          apply_act(acc[p][2 * q + 1].x + Wt.b1[4 * q + 2], s.act1),
                          apply_act(acc[p][2 * q + 1].y + Wt.b1[4 * q + 3], s.act1));
      }
    }
  };
  // ---- stage 2: depthwise 3x3 stride 2. Thread = (output column, 4 channels, row pair): the
  // column offsets, their validity and the 9 weight vectors are per-thread constants;
  // out-of-range taps are skipped like depthwise_v4_kernel skips them.
  auto stage2 = [&](const Tile& T, const float* c1) {
    const int n2 = T.tw * 4;
    for (int task = tid; task < 2 * n2; task += kG) {
    const int half = task >= n2 ? 1 : 0;
    const int r2 = task - half * n2;
    const int lx = r2 >> 2, q = r2 & 3;
    int off[3];
    bool cok[3];
#pragma unroll
    for (int fx = 0; fx < 3; ++fx) {
      const int cl = 2 * lx + fx;
      cok[fx] = static_cast<unsigned>(T.x1_0 + cl) < static_cast<unsigned>(s.OW1);
      off[fx] = cl * 16 + ((q ^ ((cl >> 1) & 3)) << 2);
    }
    float4 wv[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) wv[k] = *reinterpret_cast<const float4*>(w2s + k * 16 + q * 4);
    const float4 bb = *reinterpret_cast<const float4*>(b2s + q * 4);
    float4* o = reinterpret_cast<float4*>(out) +
                ((static_cast<long long>(T.b) * s.OH2 + T.oy2_0) * s.OW2 + T.ox2_0 + lx) * 4 + q;
    for (int ly = 2 * half; ly < 2 * half + 2 && T.oy2_0 + ly < s.OH2; ++ly) {
      float2 a0 = make_float2(0.f, 0.f), a1 = make_float2(0.f, 0.f);
#pragma unroll
      for (int fy = 0; fy < 3; ++fy) {
        const int l1 = 2 * ly + fy;
        if (static_cast<unsigned>(T.y1_0 + l1) >= static_cast<unsigned>(s.OH1)) continue;
        const float* rowp = c1 + l1 * (kS2C1 * 16);
#pragma unroll
        for (int fx = 0; fx < 3; ++fx) {
          if (!cok[fx]) continue;
          const float4 x = *reinterpret_cast<const float4*>(rowp + off[fx]);
          const float4 w = wv[fy * 3 + fx];
          a0 = __ffma2_rn(make_float2(x.x, x.y), make_float2(w.x, w.y), a0);
          a1 = __ffma2_rn(make_float2(x.z, x.w), make_float2(w.z, w.w), a1);
        }
      }
      o[static_cast<long long>(ly) * s.OW2 * 4] =
          make_float4(apply_act(a0.x + bb.x, s.act2), apply_act(a0.y + bb.y, s.act2),
                      apply_act(a1.x + bb.z, s.act2), apply_act(a1.y + bb.w, s.act2));
    }
    }
  };

  // Pipeline over this group's tiles (one strip):
  //   iteration i:  [barrier: patch i landed, strip free] fetch patch i+1 (async) | stage 1 of tile i |
  //                 [barrier] | stage 2 of tile i
  __syncthreads();                       // the table, depthwise weights (written by all 512 threads)
  int t = blockIdx.x * kGroups + gid;
  if (t >= tiles) return;
  Tile cur;
  cur.ct = t % s.n_ct;
  cur.rt = (t / s.n_ct) % s.n_rt;
  cur.b = t / (s.n_ct * s.n_rt);
  place(cur);
  load_tile(cur, raw0);
  for (int i = 0; t < tiles; t += tile_step, ++i) {
    unsigned char* raw = raw0 + (i & 1) * (kS2R0 * kRawPitch);
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    group_barrier();   // patch i complete for every thread; stage 2 of tile i-1 is done with the strip
    Tile nxt = cur;
    advance(nxt);
    if (t + tile_step < tiles) load_tile(nxt, raw0 + ((i + 1) & 1) * (kS2R0 * kRawPitch));
    stage1(cur, raw, c1_0);
    group_barrier();   // strip complete
    stage2(cur, c1_0);
    cur = nxt;
  }
}

template <typename TIn, bool kUnsigned>
int launch_stem2(const void* in, const StemWeights& wt, float* out, const Stem2Geom& s, void* stream) {
  static bool attr_dev[64] = {};   // the attribute is per device
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  constexpr size_t smem = Stem2Layout<TIn>::kSmemBytes;
  if (!(dev >= 0 && dev < 64 && attr_dev[dev])) {
    if (cudaFuncSetAttribute(stem_conv_dw_kernel<TIn, kUnsigned>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(smem)) != cudaSuccess)
      return fail("stem_conv_dw: cannot raise the shared-memory limit");
    if (dev >= 0 && dev < 64) attr_dev[dev] = true;
  }
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const long long tiles = static_cast<long long>(s.B) * s.n_rt * s.n_ct;
  if (tiles > (1LL << 29)) return fail("stem_conv_dw: too many tiles");
  constexpr int groups = Stem2Layout<TIn>::kGroups;
  const unsigned grid = static_cast<unsigned>(std::min<long long>((tiles + groups - 1) / groups, sms));
  stem_conv_dw_kernel<TIn, kUnsigned><<<grid, kS2Threads, smem, as_stream(stream)>>>(static_cast<const TIn*>(in), out, wt, s);
  return launch_check("stem_conv_dw_kernel");
}

int make_geom(const lce_f32_conv_desc* d, ConvGeom* g) {
  if (d->batch < 0 || d->in_h < 1 || d->in_w < 1 || d->in_c < 1 || d->out_c < 1 ||
      d->filter_h < 1 || d->filter_w < 1 || d->stride_h < 1 || d->stride_w < 1 ||
      d->dilation_h < 1 || d->dilation_w < 1)
    return fail("f32 conv: bad parameters");
  g->B = d->batch; g->H = d->in_h; g->W = d->in_w; g->Cin = d->in_c;
  g->KH = d->filter_h; g->KW = d->filter_w; g->Cout = d->out_c;
  g->sh = d->stride_h; g->sw = d->stride_w; g->dh = d->dilation_h; g->dw = d->dilation_w;
  g->OH = out_size(d->padding, d->in_h, d->filter_h, d->stride_h, d->dilation_h);
  g->OW = out_size(d->padding, d->in_w, d->filter_w, d->stride_w, d->dilation_w);
  g->ph = pad_before(d->stride_h, d->dilation_h, d->in_h, d->filter_h, g->OH);
  g->pw = pad_before(d->stride_w, d->dilation_w, d->in_w, d->filter_w, g->OW);
  g->act = d->activation;
  if (g->OH < 0) g->OH = 0;
  if (g->OW < 0) g->OW = 0;
  return 0;
}

}  // namespace

// DEQUANTIZE (TF/lite/kernels/internal/reference/dequantize.h:32-49): out = float(scale * (q - zp)),
// the product in double as there. 16 quantised values (one 128-bit load) per thread.
template <typename Q>
__global__ void __launch_bounds__(256) dequantize_affine_kernel(const Q* __restrict__ in, float* __restrict__ out,
                                                                long long n, double scale, int zp) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  const long long n16 = n / 16;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n16; i += stride) {
    const uint4 v = __ldcs(reinterpret_cast<const uint4*>(in) + i);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    float4* o = reinterpret_cast<float4*>(out) + i * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float r[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const Q q = static_cast<Q>((w[j] >> (8 * k)) & 0xFFu);
        r[k] = static_cast<float>(scale * static_cast<double>(static_cast<int>(q) - zp));
      }
      o[j] = make_float4(r[0], r[1], r[2], r[3]);
    }
  }
  for (long long i = n16 * 16 + blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n; i += stride)
    out[i] = static_cast<float>(scale * static_cast<double>(static_cast<int>(in[i]) - zp));
}


extern "C" {

int lce_b200_f32_conv_out_shape(const lce_f32_conv_desc* d, int* out_h, int* out_w) {
  ConvGeom g;
  if (make_geom(d, &g)) return 1;
  *out_h = g.OH;
  *out_w = g.OW;
  return 0;
}

// `packed` (optional): LceQuantize of the output. Kernels that can emit it in their epilogue do
// and set *packed_done; the caller packs with the stand-alone kernel otherwise.
static int conv2d_impl(const lce_f32_conv_desc* d, const float* in, const float* filter,
                       const float* bias, float* out, int32_t* packed, bool* packed_done,
                       void* stream) {
  ConvGeom g;
  if (make_geom(d, &g)) return 1;
  const long long M = static_cast<long long>(g.B) * g.OH * g.OW;
  if (M == 0) return 0;
  const int K = g.KH * g.KW * g.Cin;
  // experiments: LCE_B200_DIRECT_MAXK overrides the small-K threshold of the direct kernel
  static const int direct_max_k = [] {
    const char* e = getenv("LCE_B200_DIRECT_MAXK");
    return e ? atoi(e) : kDirectMaxK;
  }();
  // 1x1 stride-1 convolutions are plain GEMMs over the pixels: tensor cores first
  if (g.KH == 1 && g.KW == 1 && g.sh == 1 && g.sw == 1) {
    int32_t* pk = (packed && (g.Cout & 31) == 0) ? packed : nullptr;
    const int rc = lce_b200_internal::pw_tf32_conv(in, filter, bias, out, pk, M, g.Cout, K, g.act,
                                                   ((static_cast<long long>(g.OH) * g.OW) & 1) == 0, stream);
    if (rc >= 0) {
      if (rc == 0) count_path(kPathPwTf32);
      if (rc == 0 && pk) *packed_done = true;
      return rc;
    }
  }
  if (g.KH == 7 && g.KW == 7 && g.Cin == 3 && g.Cout == 64 && g.sh == 2 && g.sw == 2 && g.dh == 1 && g.dw == 1) {
    const int rc = lce_b200_internal::stem7_tf32_conv(in, filter, bias, out, g.B, g.H, g.W, g.OH, g.OW, g.ph, g.pw, g.act,
                                                      stream);
    if (rc == 0) count_path(kPathStem7);
    if (rc >= 0) return rc;
  }
  const int Gd = (g.Cout + 15) / 16;
  const size_t direct_smem =
      (static_cast<size_t>(K) * Gd * kDirectGroupStride + Gd * 16) * sizeof(float);
  if (K <= direct_max_k && g.Cout <= kDirectMaxCout && !((uintptr_t)out & 15) &&
      M * Gd < (1LL << 30) && direct_smem <= 96 * 1024) {
    const int G = Gd;
    const long long threads = M * G;
    const size_t smem = direct_smem;
    if (smem > 48 * 1024) {
      static bool attr[64] = {};   // the attribute is per device
      int dev = 0;
      cudaGetDevice(&dev);
      if (dev < 0 || dev >= 64 || !attr[dev]) {
        cudaFuncSetAttribute(conv_direct16_kernel<0, 0, 0, 4>,
                             cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
        if (dev >= 0 && dev < 64) attr[dev] = true;
      }
    }
    // 128 threads = (128 / G) pixels x G groups, PX pixels each. PX trades shared-memory weight
    // reads per FMA against registers / resident warps: the two compile-time shapes are latency
    // bound at PX = 4 (236 / 130 registers, 12-18 % of the warp slots); measured best: stem PX = 2.
    static const int px_env = [] {
      const char* e = getenv("LCE_B200_DIRECT_PX");
      return e ? atoi(e) : 0;
    }();
    const bool stem = g.KH == 3 && g.KW == 3 && g.Cin == 3;
    const bool pw16 = g.KH == 1 && g.KW == 1 && g.Cin == 16 && !((uintptr_t)in & 15);
    int PX = stem ? 2 : 4;
    if ((stem || pw16) && (px_env == 1 || px_env == 2 || px_env == 4)) PX = px_env;
    const int px_per_blk = 128 / G;
    const long long tiles = (M + px_per_blk * PX - 1) / (px_per_blk * PX);
    // the pointwise 16 -> 64 layer stages 4 KB of weights per block for only 128 pixels: give a
    // block 8 tiles (measured 0.125 -> 0.109 ms); the stem is better off with more, smaller
    // blocks (0.168 -> 0.132 ms at PX = 2, one tile per block)
    const int tpb = (pw16 && PX == 4) ? static_cast<int>(std::max<long long>(
                                            1, std::min<long long>(8, tiles / (148 * 8))))
                                      : 1;
    const unsigned blocks = static_cast<unsigned>((tiles + tpb - 1) / tpb);
    (void)threads;
    cudaStream_t st = as_stream(stream);
    // fused LceQuantize: whole words per pixel, lane pairs hold the two halves of a word
    int32_t* pk = (packed && (g.Cout & 31) == 0 && (G & 1) == 0 && 128 % G == 0) ? packed : nullptr;
    if (pk) *packed_done = true;
#define LCE_DIRECT(KH_, KW_, CIN_, PX_) \
  conv_direct16_kernel<KH_, KW_, CIN_, PX_><<<blocks, 128, smem, st>>>(in, filter, bias, out, g, M, G, tpb, pk)
    if (stem) {
      if (PX == 1) LCE_DIRECT(3, 3, 3, 1);
      else if (PX == 2) LCE_DIRECT(3, 3, 3, 2);
      else LCE_DIRECT(3, 3, 3, 4);
    } else if (pw16) {
      if (PX == 1) LCE_DIRECT(1, 1, 16, 1);
      else if (PX == 2) LCE_DIRECT(1, 1, 16, 2);
      else
        conv_direct16_kernel<1, 1, 16, 4, true><<<blocks, 128, smem, st>>>(in, filter, bias, out, g,
                                                                           M, G, tpb, pk);
    } else {
      LCE_DIRECT(0, 0, 0, 4);
    }
#undef LCE_DIRECT
    return launched(kPathDirect16, "conv_direct16_kernel");
  }
  const bool plain = g.KH == 1 && g.KW == 1 && g.sh == 1 && g.sw == 1 && (K & 3) == 0 &&
                     !((uintptr_t)in & 15) && !((uintptr_t)filter & 15) && !((uintptr_t)out & 15);
  if (plain && ((M + kPM - 1) / kPM) * ((g.Cout + kPN - 1) / kPN) < 74) {
    dim3 sgrid(static_cast<unsigned>((M + kSM_ - 1) / kSM_), (g.Cout + kSN_ - 1) / kSN_);
    gemm_small_m_kernel<<<sgrid, 256, 0, as_stream(stream)>>>(in, filter, bias, out, M, g.Cout, K,
                                                              g.act);
    return launched(kPathGemmSmallM, "gemm_small_m_kernel");
  }
  if (plain) {
    dim3 grid(static_cast<unsigned>((M + kPM - 1) / kPM), (g.Cout + kPN - 1) / kPN);
    int32_t* pk = (packed && (g.Cout & 31) == 0) ? packed : nullptr;
    if (pk) *packed_done = true;
    conv_gemm128_kernel<<<grid, 256, 0, as_stream(stream)>>>(in, filter, bias, out, M, g.Cout, K,
                                                             g.act, pk);
    return launched(kPathGemm128, "conv_gemm128_kernel");
  }
  if (K <= kIKMax && static_cast<long long>(g.H) * g.W * g.Cin < (1LL << 31)) {
    dim3 igrid(static_cast<unsigned>((M + kIM - 1) / kIM), (g.Cout + kIN - 1) / kIN);
    const size_t ksmem = static_cast<size_t>((K + kIK - 1) / kIK * kIK) * 2 * sizeof(int);
    // 25,600 B of static tiles plus a k-table of up to 32 KB: above K = 2944 a block needs more than
    // the default 48 KB, so both kernels opt in to the table's maximum (once per device)
    static bool attr[64] = {};   // the attribute is per device
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !attr[dev]) {
      constexpr int kTabMax = kIKMax * 2 * sizeof(int);
      if (cudaFuncSetAttribute(conv_igemm8x8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTabMax) != cudaSuccess ||
          cudaFuncSetAttribute(conv_igemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTabMax) != cudaSuccess)
        return fail("conv igemm: cannot raise the shared-memory limit");
      if (dev >= 0 && dev < 64) attr[dev] = true;
    }
    static const bool use8x4 = [] {
      const char* e = getenv("LCE_B200_IGEMM_8X4");
      return e && e[0] == '1';
    }();
    if (use8x4) {
      conv_igemm_kernel<<<igrid, 256, ksmem, as_stream(stream)>>>(in, filter, bias, out, g, M);
      return launched(kPathIgemm8x4, "conv_igemm_kernel");
    }
    conv_igemm8x8_kernel<<<igrid, 128, ksmem, as_stream(stream)>>>(in, filter, bias, out, g, M);
    return launched(kPathIgemm8x8, "conv_igemm8x8_kernel");
  }
  dim3 grid(static_cast<unsigned>((M + kGM - 1) / kGM), (g.Cout + kGN - 1) / kGN);
  conv_gemm_kernel<<<grid, 256, 0, as_stream(stream)>>>(in, filter, bias, out, g, M);
  return launched(kPathGemm, "conv_gemm_kernel");
}

void lce_b200_f32_conv_path_counts(uint64_t out[8]) {
  for (int i = 0; i < kConvPaths; ++i) out[i] = g_conv_path[i].load();
}

int lce_b200_f32_conv2d(const lce_f32_conv_desc* d, const float* in, const float* filter,
                        const float* bias, float* out, void* stream) {
  bool done = false;
  return conv2d_impl(d, in, filter, bias, out, nullptr, &done, stream);
}

int lce_b200_f32_conv2d_packed(const lce_f32_conv_desc* d, const float* in, const float* filter,
                               const float* bias, float* out, int32_t* packed_out, void* stream) {
  if (!packed_out) return lce_b200_f32_conv2d(d, in, filter, bias, out, stream);
  bool done = false;
  if (conv2d_impl(d, in, filter, bias, out, packed_out, &done, stream)) return 1;
  if (done) return 0;
  int oh, ow;
  if (lce_b200_f32_conv_out_shape(d, &oh, &ow)) return 1;
  return lce_b200_quantize(LCE_T_FLOAT, out, static_cast<int64_t>(d->batch) * oh * ow, d->out_c, 0,
                           packed_out, stream);
}

int lce_b200_f32_depthwise_conv2d(const lce_f32_conv_desc* d, const float* in,
                                  const float* filter, const float* bias, float* out,
                                  void* stream) {
  ConvGeom g;
  if (make_geom(d, &g)) return 1;
  if (d->out_c != d->in_c) return fail("depthwise conv: depth_multiplier must be 1");
  const long long n = static_cast<long long>(g.B) * g.OH * g.OW * g.Cout;
  if (n == 0) return 0;
  const bool a16 = !((uintptr_t)in & 15) && !((uintptr_t)filter & 15) && !((uintptr_t)out & 15) &&
                   !((uintptr_t)bias & 15);
  if ((g.Cout & 3) == 0 && a16 && g.B <= 65535 && g.OH <= 65535) {
    const int C4 = g.Cout >> 2;
    dim3 grid((g.OW * C4 + 255) / 256, g.OH, g.B);
    if (g.KH == 3 && g.KW == 3)
      depthwise_v4_kernel<3><<<grid, 256, 0, as_stream(stream)>>>(
          reinterpret_cast<const float4*>(in), reinterpret_cast<const float4*>(filter),
          reinterpret_cast<const float4*>(bias), reinterpret_cast<float4*>(out), g);
    else
      depthwise_v4_kernel<0><<<grid, 256, 0, as_stream(stream)>>>(
          reinterpret_cast<const float4*>(in), reinterpret_cast<const float4*>(filter),
          reinterpret_cast<const float4*>(bias), reinterpret_cast<float4*>(out), g);
    return launch_check("depthwise_v4_kernel");
  }
  depthwise_kernel<<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(in, filter, bias, out, g, n);
  return launch_check("depthwise_kernel");
}

int lce_b200_f32_pool_out_shape(const lce_f32_pool_desc* d, int* out_h, int* out_w) {
  if (d->filter_h < 1 || d->filter_w < 1 || d->stride_h < 1 || d->stride_w < 1)
    return fail("pool: bad parameters");
  // VALID with a filter larger than the input has no output (as in make_geom): two negative
  // extents must not multiply into a positive element count
  *out_h = std::max(0, out_size(d->padding, d->in_h, d->filter_h, d->stride_h, 1));
  *out_w = std::max(0, out_size(d->padding, d->in_w, d->filter_w, d->stride_w, 1));
  return 0;
}

static int run_pool(bool is_max, const lce_f32_pool_desc* d, const float* in, float* out,
                    void* stream) {
  int oh, ow;
  if (lce_b200_f32_pool_out_shape(d, &oh, &ow)) return 1;
  const long long n = static_cast<long long>(d->batch) * oh * ow * d->channels;
  if (n <= 0) return 0;
  const int ph = pad_before(d->stride_h, 1, d->in_h, d->filter_h, oh);
  const int pw = pad_before(d->stride_w, 1, d->in_w, d->filter_w, ow);
  if ((d->channels & 3) == 0 && !((uintptr_t)in & 15) && !((uintptr_t)out & 15) &&
      d->batch <= 65535 && oh <= 65535) {
    const int C4 = d->channels >> 2;
    dim3 grid((ow * C4 + 255) / 256, oh, d->batch);
#define LCE_POOL_V4(MAXV, F)                                                                   \
  pool_v4_kernel<MAXV, F><<<grid, 256, 0, as_stream(stream)>>>(                                \
      reinterpret_cast<const float4*>(in), reinterpret_cast<float4*>(out), d->in_h, d->in_w,   \
      C4, oh, ow, d->filter_h, d->filter_w, d->stride_h, d->stride_w, ph, pw, d->activation)
    const int f = (d->filter_h == d->filter_w && (d->filter_h == 2 || d->filter_h == 3))
                      ? d->filter_h : 0;
    if (is_max) {
      if (f == 2) LCE_POOL_V4(true, 2); else if (f == 3) LCE_POOL_V4(true, 3); else LCE_POOL_V4(true, 0);
    } else {
      if (f == 2) LCE_POOL_V4(false, 2); else if (f == 3) LCE_POOL_V4(false, 3); else LCE_POOL_V4(false, 0);
    }
#undef LCE_POOL_V4
    return launch_check("pool_v4_kernel");
  }
  if (is_max)
    pool_kernel<true><<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(
        in, out, d->batch, d->in_h, d->in_w, d->channels, oh, ow, d->filter_h, d->filter_w,
        d->stride_h, d->stride_w, ph, pw, d->activation);
  else
    pool_kernel<false><<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(
        in, out, d->batch, d->in_h, d->in_w, d->channels, oh, ow, d->filter_h, d->filter_w,
        d->stride_h, d->stride_w, ph, pw, d->activation);
  return launch_check("pool_kernel");
}
int lce_b200_f32_max_pool(const lce_f32_pool_desc* d, const float* in, float* out, void* s) {
  return run_pool(true, d, in, out, s);
}
int lce_b200_f32_avg_pool(const lce_f32_pool_desc* d, const float* in, float* out, void* s) {
  return run_pool(false, d, in, out, s);
}

static bool vec4_ok(const void* a, const void* b, const void* o, int64_t n, int64_t b_len) {
  return b_len == n && (n & 3) == 0 && !((uintptr_t)a & 15) && !((uintptr_t)b & 15) &&
         !((uintptr_t)o & 15);
}
int lce_b200_f32_maxpool2x2_depthwise3x3(const lce_f32_pool_desc* pool, const lce_f32_conv_desc* dw,
                                         const float* in, const float* filter, const float* bias,
                                         float* out, void* stream) {
  int ph_, pw_;
  if (lce_b200_f32_pool_out_shape(pool, &ph_, &pw_)) return 1;
  if (pool->filter_h != 2 || pool->filter_w != 2 || pool->stride_h != 1 || pool->stride_w != 1 ||
      pool->padding != LCE_PADDING_VALID || pool->activation != LCE_ACT_NONE)
    return fail("maxpool2x2_depthwise3x3: the pool must be 2x2, stride 1, VALID, no activation");
  ConvGeom g;
  if (make_geom(dw, &g)) return 1;
  if (dw->filter_h != 3 || dw->filter_w != 3 || dw->dilation_h != 1 || dw->dilation_w != 1 ||
      dw->out_c != dw->in_c || (dw->in_c & 3) || dw->in_c != pool->channels ||
      dw->in_h != ph_ || dw->in_w != pw_ || dw->batch != pool->batch)
    return fail("maxpool2x2_depthwise3x3: unsupported depthwise shape");
  if (((uintptr_t)in & 15) || ((uintptr_t)filter & 15) || ((uintptr_t)out & 15) ||
      ((uintptr_t)bias & 15) || g.B > 65535 || g.OH > 65535)
    return fail("maxpool2x2_depthwise3x3: unaligned pointers or too many rows");
  const long long n = static_cast<long long>(g.B) * g.OH * g.OW * g.Cout;
  if (n == 0) return 0;
  const int C4 = g.Cout >> 2;
  dim3 grid((g.OW * C4 + 255) / 256, g.OH, g.B);
  pool2_dw3_v4_kernel<<<grid, 256, 0, as_stream(stream)>>>(
      reinterpret_cast<const float4*>(in), reinterpret_cast<const float4*>(filter),
      reinterpret_cast<const float4*>(bias), reinterpret_cast<float4*>(out), pool->in_h,
      pool->in_w, C4, ph_, pw_, g.OH, g.OW, g.sh, g.sw, g.ph, g.pw, g.act);
  return launch_check("pool2_dw3_v4_kernel");
}

int lce_b200_f32_stem_conv_dw(const lce_f32_conv_desc* conv1, const lce_f32_conv_desc* dw, int in_type, const void* in,
                              double in_scale, int32_t in_zero_point, const float* w1, const float* b1, const float* w2,
                              const float* b2, float* out, void* stream) {
  ConvGeom g1, g2;
  if (make_geom(conv1, &g1) || make_geom(dw, &g2)) return 1;
  const bool ok = g1.KH == 3 && g1.KW == 3 && g1.sh == 2 && g1.sw == 2 && g1.dh == 1 && g1.dw == 1 && g1.Cin == 3 &&
                  g1.Cout == 16 && g2.KH == 3 && g2.KW == 3 && g2.sh == 2 && g2.sw == 2 && g2.dh == 1 && g2.dw == 1 &&
                  g2.Cin == 16 && g2.Cout == 16 && g2.H == g1.OH && g2.W == g1.OW && g2.B == g1.B;
  if (!ok) return fail("stem_conv_dw: unsupported shapes (3x3/s2 3 -> 16, depthwise 3x3/s2)");
  if (in_type != LCE_T_FLOAT && in_type != LCE_T_INT8 && in_type != LCE_T_BOOL) return fail("stem_conv_dw: bad input type");
  if ((uintptr_t)out & 15) return fail("stem_conv_dw: unaligned output");
  if (g1.B == 0 || g2.OH == 0 || g2.OW == 0) return 0;
  Stem2Geom s{};
  s.B = g1.B; s.H = g1.H; s.W = g1.W; s.OH1 = g1.OH; s.OW1 = g1.OW; s.ph1 = g1.ph; s.pw1 = g1.pw;
  s.OH2 = g2.OH; s.OW2 = g2.OW; s.ph2 = g2.ph; s.pw2 = g2.pw; s.act1 = g1.act; s.act2 = g2.act;
  s.n_rt = (g2.OH + kS2R - 1) / kS2R;
  s.n_ct = (g2.OW + kS2TW - 1) / kS2TW;
  s.in_scale = in_scale; s.in_zero_point = in_zero_point;
  const int es = in_type == LCE_T_FLOAT ? 4 : 1;
  // every image row starts 16-byte aligned, so a fetch that starts at a 16-column boundary and ends
  // at the row's end or 240 columns on is a whole number of 16-byte chunks
  s.aligned = (((uintptr_t)in & 15) == 0 && (static_cast<long long>(g1.W) * 3 * es) % 16 == 0) ? 1 : 0;
  if (!w1 || !w2) return fail("stem_conv_dw: the filters must be host pointers");
  StemWeights wt;
  for (int k = 0; k < 27; ++k)
    for (int c = 0; c < 16; ++c) wt.w1[k][c] = w1[c * 27 + k];   // OHWI [16][3][3][3] -> [k][co]
  for (int i = 0; i < 9 * 16; ++i) wt.w2[i / 16][i % 16] = w2[i];
  for (int c = 0; c < 16; ++c) {
    wt.b1[c] = b1 ? b1[c] : 0.0f;
    wt.b2[c] = b2 ? b2[c] : 0.0f;
  }
  if (in_type == LCE_T_FLOAT) return launch_stem2<float, false>(in, wt, out, s, stream);
  if (in_type == LCE_T_INT8) return launch_stem2<int8_t, false>(in, wt, out, s, stream);
  return launch_stem2<uint8_t, true>(in, wt, out, s, stream);
}

int lce_b200_f32_add(const float* a, const float* b, float* out, int64_t n, int64_t b_len,
                     int act, void* stream) {
  if (n <= 0) return 0;
  if (b_len <= 0 || n % b_len) return fail("add: operand shapes do not broadcast");
  eltwise_kernel<0><<<grid_for(n / 4 + 1, 256), 256, 0, as_stream(stream)>>>(
      a, b, out, n, b_len, act, vec4_ok(a, b, out, n, b_len));
  return launch_check("eltwise_kernel<add>");
}
int lce_b200_f32_mul(const float* a, const float* b, float* out, int64_t n, int64_t b_len,
                     int act, void* stream) {
  if (n <= 0) return 0;
  if (b_len <= 0 || n % b_len) return fail("mul: operand shapes do not broadcast");
  eltwise_kernel<1><<<grid_for(n / 4 + 1, 256), 256, 0, as_stream(stream)>>>(
      a, b, out, n, b_len, act, vec4_ok(a, b, out, n, b_len));
  return launch_check("eltwise_kernel<mul>");
}
int lce_b200_f32_activation(const float* in, float* out, int64_t n, int act, void* stream) {
  if (n <= 0) return 0;
  eltwise_kernel<2><<<grid_for(n / 4 + 1, 256), 256, 0, as_stream(stream)>>>(
      in, in, out, n, n, act, vec4_ok(in, in, out, n, n));
  return launch_check("eltwise_kernel<act>");
}

int lce_b200_f32_mean_hw_act(const float* in, float* out, int batch, int h, int w, int c, int pre_activation,
                             void* stream) {
  if (batch <= 0 || c <= 0) return 0;
  if (h * w <= 0) return fail("mean: empty spatial extent");
  mean_hw_kernel<<<(batch * c + 255) / 256, 256, 0, as_stream(stream)>>>(in, out, batch, h * w, c, pre_activation);
  return launch_check("mean_hw_kernel");
}

int lce_b200_f32_mean_hw(const float* in, float* out, int batch, int h, int w, int c,
                         void* stream) {
  return lce_b200_f32_mean_hw_act(in, out, batch, h, w, c, LCE_ACT_NONE, stream);
}

int lce_b200_f32_softmax(const float* in, float* out, int64_t rows, int cols, float beta,
                         void* stream) {
  if (rows <= 0 || cols <= 0) return 0;
  if (rows > 0x7fffffffLL) return fail("softmax: too many rows");
  softmax_kernel<<<static_cast<unsigned>(rows), 128, 0, as_stream(stream)>>>(in, out, cols, beta);
  return launch_check("softmax_kernel");
}

int lce_b200_dequantize_affine(int in_type, const void* in, float* out, int64_t n, double scale,
                               int32_t zero_point, void* stream) {
  if (n <= 0) return 0;
  if ((reinterpret_cast<uintptr_t>(in) & 15u) != 0 || (reinterpret_cast<uintptr_t>(out) & 15u) != 0)
    return fail("dequantize: buffers must be 16-byte aligned");
  const unsigned grid = static_cast<unsigned>(std::min<long long>((n / 16 + 256) / 256, 148 * 16));
  if (in_type == LCE_T_INT8) {
    dequantize_affine_kernel<int8_t><<<grid, 256, 0, as_stream(stream)>>>(static_cast<const int8_t*>(in), out, n, scale,
                                                                          zero_point);
  } else if (in_type == LCE_T_BOOL) {   // the uint8 code of the LCE_T_* enum
    dequantize_affine_kernel<uint8_t><<<grid, 256, 0, as_stream(stream)>>>(static_cast<const uint8_t*>(in), out, n, scale,
                                                                           zero_point);
  } else {
    return fail("dequantize: unsupported quantised type %d", in_type);
  }
  return launch_check("dequantize_affine_kernel");
}

int lce_b200_pad4d_32(const void* in, void* out, const int32_t* in_dims,
                      const int32_t* pad_before, const int32_t* pad_after, uint32_t fill_bits,
                      void* stream) {
  Pad4 p;
  long long total = 1;
  for (int i = 0; i < 4; ++i) {
    if (in_dims[i] < 0 || pad_before[i] < 0 || pad_after[i] < 0)
      return fail("pad: negative dimension or padding");
    p.in[i] = in_dims[i];
    p.before[i] = pad_before[i];
    p.out[i] = in_dims[i] + pad_before[i] + pad_after[i];
    total *= p.out[i];
  }
  if (total == 0) return 0;
  pad4d32_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, as_stream(stream)>>>(
      static_cast<const uint32_t*>(in), static_cast<uint32_t*>(out), p, fill_bits, total);
  return launch_check("pad4d32_kernel");
}

}  // extern "C"
