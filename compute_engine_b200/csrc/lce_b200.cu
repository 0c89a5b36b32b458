// lce_b200.cu -- implementation of the C-ABI CUDA layer declared in
// include/lce_b200.h. Host-side logic restates what the reference's op shell
// does around its kernels (LCE = /root/reference/larq_compute_engine):
//   shape inference          LCE/tflite/kernels/bconv2d.cc:169-248,
//                            tensorflow/lite/kernels/padding.h:32-82
//   output-transform fold    LCE/tflite/kernels/bconv2d.cc:353-389 (in double, on the host)
// and launches the kernels of lce_b200_kernels.cuh. There is no CPU compute path.
#include <algorithm>
#include <atomic>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "lce_b200.h"
#include "lce_b200_kernels.cuh"
#include "lce_b200_imma.cuh"
#include "lce_b200_tc.cuh"
#include "lce_b200_pw.cuh"

namespace {
thread_local std::string g_err;
std::atomic<uint64_t> g_launches{0};
std::atomic<uint64_t> g_path[3] = {};   // inner-product launches: tcgen05 / mma.sync / XOR + POPC
}  // namespace

// shared with lce_b200_builtins.cu
namespace lce_b200_internal {
int fail(const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return 1;
}
int launch_check(const char* what) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail("launch of %s failed: %s", what, cudaGetErrorString(e));
  return 0;
}
}  // namespace lce_b200_internal
using lce_b200_internal::fail;
using lce_b200_internal::launch_check;

namespace {

#define CUDA_OK(expr)                                                            \
  do {                                                                           \
    cudaError_t e__ = (expr);                                                    \
    if (e__ != cudaSuccess)                                                      \
      return fail("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

inline cudaStream_t as_stream(void* s) { return static_cast<cudaStream_t>(s); }
// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute: one flag per (kernel
// instantiation, device), so a process that drives several GPUs raises the limit on each of them.
struct PerDeviceOnce {
  bool done[64] = {};
  bool need() {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return true;
    if (done[dev]) return false;
    done[dev] = true;
    return true;
  }
};
// per-channel vectors (multiplier, bias, thresholds) are padded by one widest channel tile
constexpr int kChanPad = 128;
inline int cdiv(int a, int b) { return (a + b - 1) / b; }

int grid_for(long long work_items, int per_block, int max_blocks = 148 * 16) {
  long long b = (work_items + per_block - 1) / per_block;
  if (b < 1) b = 1;
  if (b > max_blocks) b = max_blocks;
  return static_cast<int>(b);
}

// tensorflow/lite/kernels/padding.h:42-60
int out_size(int padding, int image, int filter, int stride, int dil) {
  const int eff = (filter - 1) * dil + 1;
  if (stride == 0) return 0;
  if (padding == LCE_PADDING_SAME) return (image + stride - 1) / stride;
  if (padding == LCE_PADDING_VALID) return (image + stride - eff) / stride;
  return 0;
}
// tensorflow/lite/kernels/padding.h:32-40
int pad_before(int stride, int dil, int in, int filter, int out) {
  const int eff = (filter - 1) * dil + 1;
  int total = (out - 1) * stride + eff - in;
  if (total < 0) total = 0;
  return total / 2;
}

bool is_device_ptr(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Copy `bytes` from a host-or-device pointer into fresh device memory of
// `alloc_bytes` (zero padded).
int to_device(const void* src, size_t bytes, size_t alloc_bytes, void** dst) {
  CUDA_OK(cudaMalloc(dst, alloc_bytes));
  CUDA_OK(cudaMemset(*dst, 0, alloc_bytes));
  if (bytes)
    CUDA_OK(cudaMemcpy(*dst, src, bytes,
                       is_device_ptr(src) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
  return 0;
}
int to_host(const void* src, size_t bytes, void* dst) {
  CUDA_OK(cudaMemcpy(dst, src, bytes,
                     is_device_ptr(src) ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost));
  return 0;
}

// The part of a plan that the implicit-GEMM kernel needs, shared by LceBconv2d
// and the plain BGEMM.
struct GemmCore {
  int V = 1;            // words per smem vector (largest of 4,2,1 dividing Cw_pg)
  int Cw_pg = 0, taps = 1, Kv = 0, Kc_v = 0, n_chunks = 1;
  int cout = 0, cout_pg = 0, groups = 1, tiles_per_group = 1;
  int out_type = LCE_OUT_FLOAT;
  int clamp_min = 0, clamp_max = 0;
  int32_t* wt = nullptr;        // tiled weights
  float* mul = nullptr;         // folded, padded
  float* bias = nullptr;
  int32_t* thr = nullptr;
  int32_t* tap_popc = nullptr;  // zero-padding correction table
  size_t smem_bytes = 0;
  // int8 tensor-pipe inner product (lce_b200_imma.cuh); absent when LCE_B200_BCONV_IMMA=0 or ineligible
  int32_t* wt_nat = nullptr;    // weights expanded to int8 mma B fragments (8x the packed bytes)
  int32_t* wpop = nullptr;      // popcount of each channel's filter row (padded by BN)
  int imma_Kc_v = 0, imma_chunks = 1;
  size_t imma_smem = 0;
  // tcgen05 inner product (lce_b200_tc.cuh); absent when LCE_B200_BCONV_TC=0 or ineligible
  bool tc_ok = false;
  uint8_t* tc_wt = nullptr;        // [n_tiles][S_t][BN x 128 B] int8 stage images
  int32_t* tc_wpop2 = nullptr;     // 2 * popcount of each filter row, padded
  int32_t* tc_tap_popc_t = nullptr;  // [taps][ldc], zero-padding correction
  float* tc_zpc_cache = nullptr;     // [4][eff_h][eff_w][ldc], the optimised kernels' float corrections
  int tc_BN = 0, tc_n_tiles = 0, tc_CcB = 0, tc_n_chunks = 1, tc_flat = 0, tc_V = 1;
  int tc_S_full = 0, tc_S_last = 0, tc_S_t = 0, tc_ldc = 0;
  // shape-dependent part, cached per input shape
  long long tc_key_M = -1;
  int tc_key_H = 0, tc_key_W = 0, tc_max_px = 0;

  void release() {
    cudaFree(wt); cudaFree(mul); cudaFree(bias); cudaFree(thr); cudaFree(tap_popc);
    cudaFree(wt_nat); cudaFree(wpop);
    cudaFree(tc_wt); cudaFree(tc_wpop2); cudaFree(tc_tap_popc_t); cudaFree(tc_zpc_cache);
    wt = wt_nat = wpop = nullptr; mul = bias = nullptr; thr = tap_popc = nullptr;
    tc_wt = nullptr; tc_wpop2 = tc_tap_popc_t = nullptr; tc_zpc_cache = nullptr; tc_ok = false;
  }
};

// Dynamic shared memory one CTA may use so that kCtasPerSm CTAs stay resident on an SM
// (227 KB per SM, 1 KB reserved per CTA, a little static shared memory).
size_t cta_smem_budget() {
  return (227u * 1024u / lce::kCtasPerSm - 1024u - 256u) & ~size_t{127};
}

template <int V, int OUT>
int launch_conv_vo(const lce::ConvKParams& p, dim3 grid, size_t smem, cudaStream_t s) {
  static PerDeviceOnce once;
  if (once.need())
    CUDA_OK(cudaFuncSetAttribute(lce::bconv_kernel<V, OUT>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(cta_smem_budget())));
  lce::bconv_kernel<V, OUT><<<grid, lce::kThreads, smem, s>>>(p);
  g_path[2].fetch_add(1, std::memory_order_relaxed);
  return launch_check("bconv_kernel");
}
size_t imma_smem_budget(int V) {
  const int ctas = lce::imma_ctas_per_sm(V);
  return (227u * 1024u / ctas - 1024u - 256u) & ~size_t{127};
}

template <int V, int OUT>
int launch_imma_vo(const lce::ConvKParams& p, dim3 grid, size_t smem, cudaStream_t s) {
  static PerDeviceOnce once;
  if (once.need())
    CUDA_OK(cudaFuncSetAttribute(lce::bconv_imma_kernel<V, OUT>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(imma_smem_budget(V))));
  lce::bconv_imma_kernel<V, OUT><<<grid, lce::kIThreads, smem, s>>>(p);
  g_path[1].fetch_add(1, std::memory_order_relaxed);
  return launch_check("bconv_imma_kernel");
}
template <int V>
int launch_imma_v(int out_type, const lce::ConvKParams& p, dim3 grid, size_t smem,
                  cudaStream_t s) {
  if (out_type == LCE_OUT_FLOAT) return launch_imma_vo<V, LCE_OUT_FLOAT>(p, grid, smem, s);
  return launch_imma_vo<V, LCE_OUT_RAW_ACC>(p, grid, smem, s);
}

template <int V>
int launch_conv_v(int out_type, const lce::ConvKParams& p, dim3 grid, size_t smem,
                  cudaStream_t s) {
  switch (out_type) {
    case LCE_OUT_FLOAT: return launch_conv_vo<V, LCE_OUT_FLOAT>(p, grid, smem, s);
    case LCE_OUT_INT8: return launch_conv_vo<V, LCE_OUT_INT8>(p, grid, smem, s);
    case LCE_OUT_BITPACKED: return launch_conv_vo<V, LCE_OUT_BITPACKED>(p, grid, smem, s);
    case LCE_OUT_RAW_ACC: return launch_conv_vo<V, LCE_OUT_RAW_ACC>(p, grid, smem, s);
  }
  return fail("unsupported output type %d", out_type);
}
int tc_launch(GemmCore& c, const lce::ConvKParams& p, cudaStream_t s);

int launch_conv(GemmCore& c, lce::ConvKParams& p, cudaStream_t s) {
  p.fd_ohw = lce::make_fastdiv(static_cast<uint32_t>(p.OH) * p.OW);
  p.fd_ow = lce::make_fastdiv(p.OW);
  p.fd_cwv = lce::make_fastdiv(p.CwV);
  p.fd_kw = lce::make_fastdiv(p.KW);
  p.fd_tpg = lce::make_fastdiv(p.tiles_per_group);
  p.img_words = static_cast<long long>(p.H) * p.W * p.Cw_total;
  if (p.M <= 0) return 0;  // empty batch: nothing to do
  const long long m_tiles = (p.M + lce::kBM - 1) / lce::kBM;
  if (m_tiles > INT_MAX) return fail("too many output pixels");
  if (p.img_words >= (1LL << 31)) return fail("input image too large (>= 2^31 packed words)");
  if (c.tc_ok) {
    // tcgen05 inner product: the same int32 accumulators again, persistent 128 x BN tiles
    const int rc = tc_launch(c, p, s);
    if (rc >= 0) return rc;
  }
  if (c.wt_nat != nullptr && p.vec_store) {
    // int8 tensor-pipe inner product: 128 x 64 tiles, the same int32 accumulators as bconv_kernel
    lce::ConvKParams q = p;
    q.wt = c.wt_nat; q.wpop = c.wpop;
    q.Kc_v = c.imma_Kc_v; q.n_chunks = c.imma_chunks;
    q.res_stage = 0;
    const size_t ismem = c.imma_smem;
    dim3 igrid(static_cast<unsigned>((p.M + lce::kIBM - 1) / lce::kIBM),
               static_cast<unsigned>(c.groups * c.tiles_per_group));
    switch (c.V) {
      case 4: return launch_imma_v<4>(c.out_type, q, igrid, ismem, s);
      case 2: return launch_imma_v<2>(c.out_type, q, igrid, ismem, s);
      default: return launch_imma_v<1>(c.out_type, q, igrid, ismem, s);
    }
  }
  dim3 grid(static_cast<unsigned>(m_tiles), static_cast<unsigned>(c.groups * c.tiles_per_group));
  const size_t smem = c.smem_bytes + (p.res_stage ? lce::kResStageBytes : 0);
  switch (c.V) {
    case 4: return launch_conv_v<4>(c.out_type, p, grid, smem, s);
    case 2: return launch_conv_v<2>(c.out_type, p, grid, smem, s);
    default: return launch_conv_v<1>(c.out_type, p, grid, smem, s);
  }
}


// ------------------------------------------------------------------------- //
// tcgen05 path (lce_b200_tc.cuh): plan-time weight images and the launch.
// ------------------------------------------------------------------------- //
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_map_encoder() {
  static EncodeTiledFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess) {
      cudaGetLastError();
      f = nullptr;
    }
    return reinterpret_cast<EncodeTiledFn>(f);
  }();
  return fn;
}
int num_sms() {
  static int cache[64] = {};
  int dev = 0, v = 148;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && cache[dev]) return cache[dev];
  cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
  if (dev >= 0 && dev < 64) cache[dev] = v;
  return v;
}
constexpr size_t kTcSmemBudget = 226u * 1024u;   // dynamic shared memory of the one CTA per SM

bool tc_enabled() {
  const char* e = getenv("LCE_B200_BCONV_TC");  // read per plan: A/B in one process
  return !(e && e[0] == '0');
}

// Weight stage images, 2 * popc(filter row) and the transposed tap popcounts. Eligibility that
// does not depend on the input shape is decided here; the rest in tc_launch.
int build_tc_weights(GemmCore* c, const int32_t* d_filter, bool want_tap_popc) {
  c->tc_ok = false;
  if (!tc_enabled() || c->groups != 1 || tensor_map_encoder() == nullptr) return 0;
  if ((c->out_type == LCE_OUT_FLOAT || c->out_type == LCE_OUT_RAW_ACC) && (c->cout % 4 != 0 || c->cout < 32))
    return 0;  // TMA store: 16-byte row pitch, 32-column boxes
  if (want_tap_popc && c->taps > 64) return 0;
  const int Cw = c->Cw_pg;
  c->tc_BN = c->cout > 64 ? 128 : (c->cout > 32 ? 64 : 32);
  c->tc_n_tiles = cdiv(c->cout, c->tc_BN);
  if (Cw % 4 == 0) {
    c->tc_flat = 0; c->tc_V = 4;
    c->tc_CcB = std::min(Cw, 32);   // halo stage = pixels x 128 B at most
  } else {
    c->tc_flat = 1; c->tc_V = (Cw % 2 == 0) ? 2 : 1;
    c->tc_CcB = Cw;
    if (Cw > 64) return 0;
  }
  c->tc_n_chunks = cdiv(Cw, c->tc_CcB);
  const int cc_last = Cw - (c->tc_n_chunks - 1) * c->tc_CcB;
  c->tc_S_full = cdiv(c->taps * c->tc_CcB, lce::tc::kWS);
  c->tc_S_last = cdiv(c->taps * cc_last, lce::tc::kWS);
  c->tc_S_t = (c->tc_n_chunks - 1) * c->tc_S_full + c->tc_S_last;
  c->tc_ldc = c->tc_n_tiles * c->tc_BN;
  const long long units = static_cast<long long>(c->tc_n_tiles) * c->taps * Cw * c->tc_BN;
  CUDA_OK(cudaMalloc(&c->tc_wt, static_cast<size_t>(units) * 32));
  lce::tc::expand_weights_tc_kernel<<<grid_for(units, 256, 1 << 22), 256>>>(
      d_filter, c->tc_wt, c->cout, c->taps, Cw, c->tc_CcB, c->tc_BN, units);
  if (launch_check("expand_weights_tc_kernel")) return 1;
  CUDA_OK(cudaMalloc(&c->tc_wpop2, static_cast<size_t>(c->tc_ldc) * 4));
  CUDA_OK(cudaMemset(c->tc_wpop2, 0, static_cast<size_t>(c->tc_ldc) * 4));
  lce::tc::wpop2_kernel<<<cdiv(c->cout, 256), 256>>>(d_filter, c->tc_wpop2, c->cout, c->taps * Cw);
  if (launch_check("wpop2_kernel")) return 1;
  if (want_tap_popc) {
    const size_t n = static_cast<size_t>(c->taps) * c->tc_ldc;
    CUDA_OK(cudaMalloc(&c->tc_tap_popc_t, n * 4));
    CUDA_OK(cudaMemset(c->tc_tap_popc_t, 0, n * 4));
    lce::tc::tap_popc_t_kernel<<<cdiv(c->cout * c->taps, 256), 256>>>(d_filter, c->tc_tap_popc_t, c->cout, c->taps,
                                                                       Cw, c->tc_ldc);
    if (launch_check("tap_popc_t_kernel")) return 1;
  }
  c->tc_ok = true;
  return 0;
}

// Largest halo (input pixels touched by one 128-pixel tile) over all tiles of this shape: the same
// arithmetic as lce::tc::tile_halo, run once per (plan, input shape).
int tc_max_halo_px(const lce::ConvKParams& p) {
  long long best = 1;
  const long long ohw = static_cast<long long>(p.OH) * p.OW;
  const long long total_px = (p.M / ohw) * p.H * p.W;
  auto flat = [&](long long m, int fy, int fx) {
    const long long b = m / ohw, r = m - b * ohw;
    const long long oy = r / p.OW, ox = r - oy * p.OW;
    return (b * p.H + (oy * p.sh - p.ph + fy * p.dh)) * p.W + (ox * p.sw - p.pw + fx * p.dw);
  };
  for (long long m0 = 0; m0 < p.M; m0 += lce::tc::kBM) {
    const long long m1 = std::min<long long>(m0 + lce::tc::kBM, p.M) - 1;
    long long lo = std::max<long long>(flat(m0, 0, 0), 0);
    const long long hi = std::min<long long>(flat(m1, p.KH - 1, p.KW - 1) + 1, total_px);
    if (lo > total_px - 1) lo = total_px - 1;
    best = std::max(best, std::max<long long>(hi - lo, 1));
  }
  return static_cast<int>(std::min<long long>(best, INT_MAX));
}

template <int V, int OUT>
int launch_tc_vo(const CUtensorMap& tm_in, const CUtensorMap& tm_res, const CUtensorMap& tm_out,
                 const lce::tc::TcParams& t, int grid, size_t smem, cudaStream_t s) {
  static PerDeviceOnce once;
  if (once.need())
    CUDA_OK(cudaFuncSetAttribute(lce::tc::bconv_tc_kernel<V, OUT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(kTcSmemBudget)));
  lce::tc::bconv_tc_kernel<V, OUT><<<grid, lce::tc::kThreads, smem, s>>>(tm_in, tm_res, tm_out, t);
  g_path[0].fetch_add(1, std::memory_order_relaxed);
  return launch_check("bconv_tc_kernel");
}
template <int V>
int launch_tc_v(int out_type, const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c,
                const lce::tc::TcParams& t, int grid, size_t smem, cudaStream_t s) {
  switch (out_type) {
    case LCE_OUT_FLOAT: return launch_tc_vo<V, LCE_OUT_FLOAT>(a, b, c, t, grid, smem, s);
    case LCE_OUT_INT8: return launch_tc_vo<V, LCE_OUT_INT8>(a, b, c, t, grid, smem, s);
    case LCE_OUT_BITPACKED: return launch_tc_vo<V, LCE_OUT_BITPACKED>(a, b, c, t, grid, smem, s);
    default: return launch_tc_vo<V, LCE_OUT_RAW_ACC>(a, b, c, t, grid, smem, s);
  }
}

// Returns -1 when this launch is not eligible (the caller falls through to the mma.sync / XOR
// kernels), else the launch status.
int tc_launch(GemmCore& c, const lce::ConvKParams& p, cudaStream_t s) {
  namespace T = lce::tc;
  if (!c.tc_ok || p.M >= (1LL << 31)) return -1;
  const long long ohw = static_cast<long long>(p.OH) * p.OW;
  const long long batch = p.M / ohw;
  const long long total_px = batch * p.H * p.W;
  const long long total_words = total_px * p.Cw_total;
  if (total_words >= (1LL << 31) || total_px < 1) return -1;
  if ((reinterpret_cast<uintptr_t>(p.in) & 15u) != 0) return -1;
  const bool tma_out = c.out_type == LCE_OUT_FLOAT || c.out_type == LCE_OUT_RAW_ACC;
  if (tma_out && (reinterpret_cast<uintptr_t>(p.out) & 15u) != 0) return -1;
  if (p.residual != nullptr && (reinterpret_cast<uintptr_t>(p.residual) & 15u) != 0) return -1;
  if (c.out_type == LCE_OUT_INT8 && (reinterpret_cast<uintptr_t>(p.out) & 15u) != 0) return -1;
  if (c.tc_key_M != p.M || c.tc_key_H != p.H || c.tc_key_W != p.W) {
    c.tc_max_px = tc_max_halo_px(p);
    c.tc_key_M = p.M; c.tc_key_H = p.H; c.tc_key_W = p.W;
  }
  T::TcParams t;
  memset(&t, 0, sizeof(t));
  t.M = p.M; t.total_px = total_px;
  t.H = p.H; t.W = p.W; t.OH = p.OH; t.OW = p.OW; t.KH = p.KH; t.KW = p.KW;
  t.sh = p.sh; t.sw = p.sw; t.dh = p.dh; t.dw = p.dw; t.ph = p.ph; t.pw = p.pw;
  t.taps = p.KH * p.KW;
  t.Cw = c.Cw_pg; t.CcB = c.tc_CcB; t.n_chunks = c.tc_n_chunks; t.mode_flat = c.tc_flat;
  t.cout = c.cout; t.BN = c.tc_BN; t.n_tiles = c.tc_n_tiles;
  t.m_tiles = static_cast<int>((p.M + T::kBM - 1) / T::kBM);
  t.S_full = c.tc_S_full; t.S_last = c.tc_S_last; t.S_t = c.tc_S_t;
  // shared memory: weights | halo stages | epilogue slots | barriers
  size_t raw_stage;
  if (c.tc_flat) raw_stage = static_cast<size_t>(cdiv(c.tc_max_px * c.Cw_pg + 3, 256)) * 1024;
  else raw_stage = static_cast<size_t>(cdiv(c.tc_max_px, 128)) * 128 * c.tc_CcB * 4;
  raw_stage = (raw_stage + 1023) & ~size_t{1023};
  t.raw_stage_bytes = static_cast<int>(raw_stage);
  const size_t stage_bytes = static_cast<size_t>(c.tc_BN) * 32 * T::kWS;     // one ring slot
  const size_t resident_bytes = static_cast<size_t>(c.tc_BN) * 32 * t.taps * c.Cw_pg;  // all K words, dense
  const bool has_res = p.residual != nullptr;
  // Epilogue staging slots (16 KB = 128 rows x 32 channels each; with a shortcut they are also the
  // TMA landing zone of the residual tiles, so their number is the prefetch depth of that stream):
  // as many as fit beside the weights, an even number, at most 8 with and 4 without a shortcut.
  const int ns_max = tma_out ? (has_res ? T::kMaxNS : 4) : 0;
  const int ns_min = tma_out ? 2 : 0;
  const size_t fixed = T::kNR * raw_stage + T::kBarBytes + T::kTabBytes;
  if (fixed + ns_min * T::kSlotBytes > kTcSmemBudget) return -1;
  auto room = [&](int ns) { return kTcSmemBudget - fixed - static_cast<size_t>(ns) * T::kSlotBytes; };
  const bool can_reside = c.tc_n_tiles == 1 && c.tc_S_t <= T::kMaxNB && room(ns_min) >= resident_bytes;
  int nS = ns_min;
  size_t b_bytes;
  if (can_reside) {
    t.b_resident = 1;
    t.nB = c.tc_S_t;
    b_bytes = (resident_bytes + 1023) & ~size_t{1023};
    while (nS + 2 <= ns_max && room(nS + 2) >= b_bytes) nS += 2;
  } else {
    t.b_resident = 0;
    // the weights stream through a ring whose slots are the A stages' (one barrier pair per stage)
    t.nB = T::kNA;
    b_bytes = T::kNA * stage_bytes;
    if (room(ns_min) < b_bytes) return -1;
    while (nS + 2 <= std::min(ns_max, 4) && room(nS + 2) >= b_bytes) nS += 2;
  }
  t.nS = nS;
  t.Kw_total = t.taps * c.Cw_pg;
  t.off_raw = static_cast<int>(b_bytes);
  t.off_slots = t.off_raw + T::kNR * t.raw_stage_bytes;
  t.off_tab = t.off_slots + nS * T::kSlotBytes;
  t.off_bar = t.off_tab + T::kTabBytes;
  const size_t smem = static_cast<size_t>(t.off_bar) + T::kBarBytes;
  t.clamp_min = p.clamp_min; t.clamp_max = p.clamp_max;
  t.has_res = has_res ? 1 : 0; t.residual_act = p.residual_act;
  t.cw_out = p.cw_out; t.zp_half = p.zp_half; t.ldc = c.tc_ldc;
  t.wt = c.tc_wt; t.mul = p.mul; t.bias = p.bias; t.wpop2 = c.tc_wpop2; t.thr = p.thr;
  t.tap_popc_t = p.tap_popc != nullptr ? c.tc_tap_popc_t : nullptr;
  t.zp_float = p.zp_float; t.cin_pg = p.cin_pg;
  t.zpc_cache = c.tc_zpc_cache;
  if (t.zp_float && t.zpc_cache == nullptr) return -1;
  t.out = p.out; t.packed_out = p.packed_out;
  t.fd_ohw = lce::make_fastdiv(static_cast<uint32_t>(ohw));
  t.fd_ow = lce::make_fastdiv(p.OW);
  t.fd_kw = lce::make_fastdiv(p.KW);
  t.fd_cwv_full = lce::make_fastdiv(c.tc_CcB / c.tc_V);
  t.fd_cwv_last = lce::make_fastdiv((c.Cw_pg - (c.tc_n_chunks - 1) * c.tc_CcB) / c.tc_V);
  t.fd_mt = lce::make_fastdiv(t.m_tiles);

  EncodeTiledFn enc = tensor_map_encoder();
  CUtensorMap tm_in, tm_res, tm_out;
  cuuint32_t es[2] = {1, 1};
  if (c.tc_flat) {
    cuuint64_t gd[1] = {static_cast<cuuint64_t>(total_words)};
    cuuint64_t gs[1] = {0};
    cuuint32_t box[1] = {256};
    if (enc(&tm_in, CU_TENSOR_MAP_DATA_TYPE_INT32, 1, const_cast<int32_t*>(p.in), gd, gs, box, es,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return fail("cuTensorMapEncodeTiled (activations, flat) failed");
  } else {
    cuuint64_t gd[2] = {static_cast<cuuint64_t>(p.Cw_total), static_cast<cuuint64_t>(total_px)};
    cuuint64_t gs[1] = {static_cast<cuuint64_t>(p.Cw_total) * 4};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(c.tc_CcB), 128};
    if (enc(&tm_in, CU_TENSOR_MAP_DATA_TYPE_INT32, 2, const_cast<int32_t*>(p.in), gd, gs, box, es,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return fail("cuTensorMapEncodeTiled (activations) failed");
  }
  tm_res = tm_in;
  tm_out = tm_in;
  if (tma_out) {
    cuuint64_t gd[2] = {static_cast<cuuint64_t>(c.cout), static_cast<cuuint64_t>(p.M)};
    cuuint64_t gs[1] = {static_cast<cuuint64_t>(c.cout) * 4};
    cuuint32_t box_st[2] = {32, 32};
    cuuint32_t box_ld[2] = {32, 128};
    const CUtensorMapDataType dt =
        c.out_type == LCE_OUT_FLOAT ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_INT32;
    if (enc(&tm_out, dt, 2, p.out, gd, gs, box_st, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return fail("cuTensorMapEncodeTiled (output) failed");
    if (has_res &&
        enc(&tm_res, dt, 2, const_cast<float*>(p.residual), gd, gs, box_ld, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return fail("cuTensorMapEncodeTiled (shortcut) failed");
  }
  const long long items = static_cast<long long>(t.n_tiles) * t.m_tiles;
  const int grid = static_cast<int>(std::min<long long>(items, num_sms()));
  static long long* d_prof = nullptr;
  static const bool prof_on = [] { const char* e = getenv("LCE_B200_TC_PROF"); return e && e[0] == '1'; }();
  if (prof_on) {
    // development aid: per-role cycle counters of block 0, printed after a synchronising copy
    if (!d_prof) cudaMalloc(&d_prof, 20 * 8 * sizeof(long long));
    cudaMemsetAsync(d_prof, 0, 20 * 8 * sizeof(long long), s);
    t.prof = d_prof;
  }
  struct ProfDump {
    long long* d; cudaStream_t s; const T::TcParams* t; int grid;
    ~ProfDump() {
      if (!d) return;
      long long h[160];
      cudaStreamSynchronize(s);
      cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost);
      fprintf(stderr, "[tc prof] M=%lld BN=%d S_t=%d nB=%d res=%d resident=%d items=%d grid=%d\n", t->M, t->BN, t->S_t,
              t->nB, t->has_res, t->b_resident, t->n_tiles * t->m_tiles, grid);
      const char* names[20] = {"exp0", "exp1", "exp2", "exp3", "exp4", "exp5", "exp6", "exp7", "epi0", "epi1", "epi2", "epi3",
                               "epi4", "epi5", "epi6", "epi7", "act-prod", "res-prod", "w-prod", "mma"};
      for (int w : {16, 19, 18, 17, 0, 4, 8, 12})
        fprintf(stderr, "[tc prof]  %-8s total=%lld  c1=%lld c2=%lld c3=%lld c4=%lld c5=%lld c6=%lld\n", names[w], h[w * 8],
                h[w * 8 + 1], h[w * 8 + 2], h[w * 8 + 3], h[w * 8 + 4], h[w * 8 + 5], h[w * 8 + 6]);
    }
  } prof_dump{prof_on ? d_prof : nullptr, s, &t, grid};
  switch (c.tc_V) {
    case 4: return launch_tc_v<4>(c.out_type, tm_in, tm_res, tm_out, t, grid, smem, s);
    case 2: return launch_tc_v<2>(c.out_type, tm_in, tm_res, tm_out, t, grid, smem, s);
    default: return launch_tc_v<1>(c.out_type, tm_in, tm_res, tm_out, t, grid, smem, s);
  }
}

}  // namespace
// fp32 pointwise convolution on the tensor cores (lce_b200_pw.cuh), called by the CONV_2D builtin
// (lce_b200_builtins.cu). 0 = launched, -1 = shape not eligible (the caller's FMA kernels take
// it), > 0 = error.
namespace lce_b200_internal {
int pw_tf32_conv(const float* in, const float* filter, const float* bias, float* out, int32_t* packed, long long M, int N,
                 int K, int act, int pairs_ok, void* stream) {
  static const bool enabled = [] { const char* e = getenv("LCE_B200_PW_TF32"); return !(e && e[0] == '0'); }();
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enabled || enc == nullptr) return -1;
  if ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(filter) | reinterpret_cast<uintptr_t>(out) |
       reinterpret_cast<uintptr_t>(bias) | reinterpret_cast<uintptr_t>(packed)) & 15)
    return -1;
  // Which kernel runs must not depend on the batch (an image's result must not change with its
  // batch mates): eligibility looks at the layer's shape only; `pairs_ok` = even pixels per image.
  const bool pairs = K == 16 && N == 64 && pairs_ok && (M & 1) == 0;
  // N: whole 128-column tiles, or (no packed output) any multiple of 4 -- TMA zero-fills the filter
  // rows past N and clips the stores (FULLY_CONNECTED's 1000 logits)
  if (!pairs && ((K & 31) != 0 || K > 4096 || (N & 3) != 0 || ((N & 127) != 0 && packed != nullptr))) return -1;
  namespace P = lce::pw;
  P::PwParams p{};
  p.M = pairs ? M / 2 : M;
  p.N = pairs ? 128 : N;
  p.KB = pairs ? 1 : K / 32;
  p.n_tiles = (p.N + 127) / 128;
  const long long m_tiles = (p.M + 127) / 128;
  if (m_tiles > (1 << 22)) return -1;
  p.m_tiles = static_cast<int>(m_tiles);
  p.act = act;
  p.pairs = pairs ? 1 : 0;
  p.w_resident = (p.n_tiles == 1 && p.KB <= P::kPwNS) ? 1 : 0;
  p.bias_mask = pairs ? 63 : 0x7fffffff;
  p.filter = filter;
  p.bias = bias;
  p.packed = packed;
  const int Kp = pairs ? 32 : K;
  CUtensorMap tm_a, tm_w, tm_out;
  cuuint32_t es[2] = {1, 1};
  cuuint32_t box_ld[2] = {32, 128}, box_st[2] = {32, 32};
  {
    cuuint64_t gd[2] = {static_cast<cuuint64_t>(Kp), static_cast<cuuint64_t>(p.M)};
    cuuint64_t gs[1] = {static_cast<cuuint64_t>(Kp) * 4};
    if (enc(&tm_a, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(in), gd, gs, box_ld, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return fail("cuTensorMapEncodeTiled (pointwise input) failed");
  }
  tm_w = tm_a;
  if (!pairs) {
    cuuint64_t gd[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(N)};
    cuuint64_t gs[1] = {static_cast<cuuint64_t>(K) * 4};
    if (enc(&tm_w, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(filter), gd, gs, box_ld, es,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return fail("cuTensorMapEncodeTiled (pointwise filter) failed");
  }
  {
    cuuint64_t gd[2] = {static_cast<cuuint64_t>(p.N), static_cast<cuuint64_t>(p.M)};
    cuuint64_t gs[1] = {static_cast<cuuint64_t>(p.N) * 4};
    if (enc(&tm_out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, out, gd, gs, box_st, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return fail("cuTensorMapEncodeTiled (pointwise output) failed");
  }
  static PerDeviceOnce once;
  if (once.need())
    CUDA_OK(cudaFuncSetAttribute(P::pw_tf32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(P::kPwSmem)));
  const int grid = static_cast<int>(std::min<long long>(m_tiles * p.n_tiles, num_sms()));
  static long long* d_prof = nullptr;
  static const bool prof_on = [] { const char* e = getenv("LCE_B200_TC_PROF"); return e && e[0] == '1'; }();
  if (prof_on) {
    if (!d_prof) cudaMalloc(&d_prof, 22 * 8 * sizeof(long long));
    cudaMemsetAsync(d_prof, 0, 22 * 8 * sizeof(long long), static_cast<cudaStream_t>(stream));
    p.prof = d_prof;
  }
  P::pw_tf32_kernel<<<grid, P::kPwThreads, P::kPwSmem, static_cast<cudaStream_t>(stream)>>>(tm_a, tm_w, tm_out, p);
  if (prof_on) {
    // development aid (LCE_TC_PROF build): per-role cycle counters of block 0
    long long h[22 * 8];
    cudaStreamSynchronize(static_cast<cudaStream_t>(stream));
    cudaMemcpy(h, d_prof, sizeof(h), cudaMemcpyDeviceToHost);
    fprintf(stderr, "[pw prof] M=%lld N=%d KB=%d resident=%d pairs=%d items=%lld grid=%d\n", p.M, p.N, p.KB, p.w_resident, p.pairs,
            m_tiles * p.n_tiles, grid);
    const char* names[22] = {"split0", "split1", "split2", "split3", "epi", "epi", "epi", "epi", "epi", "epi", "epi", "epi", "epi",
                             "epi", "epi", "epi", "epi", "epi", "epi", "epi", "tma", "mma"};
    for (int w : {20, 21, 0, 3, 4, 11, 19})
      fprintf(stderr, "[pw prof]  %-7s w%-2d total=%lld  c1=%lld c2=%lld c3=%lld c4=%lld n=%lld\n", names[w], w, h[w * 8], h[w * 8 + 1],
              h[w * 8 + 2], h[w * 8 + 3], h[w * 8 + 4], h[w * 8 + 5]);
  }
  return launch_check("pw_tf32_kernel");
}
// CONV_2D 7x7 / stride 2 / 3 -> 64 (Bi-RealNet's stem) on tcgen05 kind::tf32 (lce_b200_pw.cuh):
// 0 = launched, -1 = not this shape, > 0 = error.
int stem7_tf32_conv(const float* in, const float* filter, const float* bias, float* out, int B, int H, int W, int OH, int OW,
                    int ph, int pw, int act, void* stream) {
  static const bool enabled = [] { const char* e = getenv("LCE_B200_PW_TF32"); return !(e && e[0] == '0'); }();
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enabled || enc == nullptr) return -1;
  if ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(bias)) & 15) return -1;
  namespace P = lce::pw;
  P::Stem7Params p{};
  p.M = static_cast<long long>(B) * OH * OW;
  const long long m_tiles = (p.M + 127) / 128;
  if (m_tiles > (1 << 23)) return -1;
  p.H = H; p.W = W; p.OH = OH; p.OW = OW; p.ph = ph; p.pw = pw;
  p.m_tiles = static_cast<int>(m_tiles);
  p.act = act;
  p.in = in; p.filter = filter; p.bias = bias;
  CUtensorMap tm_out;
  cuuint32_t es[2] = {1, 1};
  cuuint32_t box_st[2] = {32, 32};
  cuuint64_t gd[2] = {64, static_cast<cuuint64_t>(p.M)};
  cuuint64_t gs[1] = {64 * 4};
  if (enc(&tm_out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, out, gd, gs, box_st, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return fail("cuTensorMapEncodeTiled (7x7 stem output) failed");
  static PerDeviceOnce once;
  if (once.need())
    CUDA_OK(cudaFuncSetAttribute(P::stem7_tf32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(P::kS7Smem)));
  const int grid = static_cast<int>(std::min<long long>(m_tiles, num_sms()));
  P::stem7_tf32_kernel<<<grid, P::kS7Threads, P::kS7Smem, static_cast<cudaStream_t>(stream)>>>(tm_out, p);
  return launch_check("stem7_tf32_kernel");
}
}  // namespace lce_b200_internal
namespace {

// Build the tiled weights (+ optional tap popcounts) from an OHWI-packed filter
// [cout][taps][Cw_pg] that may live on the host or the device.
int build_core_weights(GemmCore* c, const int32_t* filter, bool want_tap_popc) {
  const size_t filter_words = static_cast<size_t>(c->cout) * c->taps * c->Cw_pg;
  int32_t* d_filter = nullptr;
  const bool on_dev = is_device_ptr(filter);
  if (!on_dev) {
    void* tmp = nullptr;
    if (to_device(filter, filter_words * 4, filter_words * 4 + 16, &tmp)) return 1;
    d_filter = static_cast<int32_t*>(tmp);
  } else {
    d_filter = const_cast<int32_t*>(filter);
  }
  c->V = (c->Cw_pg % 4 == 0) ? 4 : (c->Cw_pg % 2 == 0) ? 2 : 1;
  const int CwV = c->Cw_pg / c->V;
  c->Kv = c->taps * CwV;
  const int max_kc_v = lce::kMaxChunkWords / c->V;
  c->n_chunks = cdiv(c->Kv, max_kc_v);
  c->Kc_v = cdiv(c->Kv, c->n_chunks);
  c->smem_bytes = static_cast<size_t>(c->Kc_v) * (lce::kBM + lce::kBN) * c->V * 4;
  c->tiles_per_group = cdiv(c->cout_pg, lce::kBN);
  const long long total = static_cast<long long>(c->groups) * c->tiles_per_group * c->Kv *
                          lce::kBN * c->V;
  CUDA_OK(cudaMalloc(&c->wt, total * 4));
  lce::tile_weights_kernel<<<grid_for(total, 256, 1 << 20), 256>>>(
      d_filter, c->wt, c->cout_pg, c->tiles_per_group, c->taps, c->Cw_pg, c->V, c->Kv, total, 0);
  if (launch_check("tile_weights_kernel")) return 1;
  // int8 tensor-pipe inner product (lce_b200_imma.cuh) where a plan is eligible: full 64-channel
  // tiles, float or raw-accumulator output. LCE_B200_BCONV_IMMA=0 keeps every plan on the
  // XOR + POPC kernel (bench.py reports both).
  const char* imma_env = getenv("LCE_B200_BCONV_IMMA");  // read per plan: A/B in one process
  const bool imma_on = !(imma_env && imma_env[0] == '0');
  if (imma_on && c->cout_pg % lce::kBN == 0 &&
      (c->out_type == LCE_OUT_FLOAT || c->out_type == LCE_OUT_RAW_ACC)) {
    const long long Kw = static_cast<long long>(c->taps) * c->Cw_pg;
    const long long xtotal = static_cast<long long>(c->groups) * c->tiles_per_group * Kw * 256;
    CUDA_OK(cudaMalloc(&c->wt_nat, xtotal * 8));
    lce::expand_weights_imma_kernel<<<grid_for(xtotal, 256, 1 << 22), 256>>>(
        d_filter, reinterpret_cast<uint2*>(c->wt_nat), c->cout_pg, c->tiles_per_group, c->taps,
        c->Cw_pg, xtotal);
    if (launch_check("expand_weights_imma_kernel")) return 1;
    CUDA_OK(cudaMalloc(&c->wpop, static_cast<size_t>(c->cout + lce::kBN) * 4));
    CUDA_OK(cudaMemset(c->wpop, 0, static_cast<size_t>(c->cout + lce::kBN) * 4));
    lce::tap_popc_kernel<<<cdiv(c->cout, 256), 256>>>(d_filter, c->wpop, c->cout, 1,
                                                      c->taps * c->Cw_pg);
    if (launch_check("tap_popc_kernel")) return 1;
    // K staging: everything in one chunk when it fits the CTA's shared-memory share, else a
    // two-deep ring of equal chunks. 3 CTAs per SM for uint4 operands, 4 otherwise (registers).
    const size_t budget = imma_smem_budget(c->V);
    const int single_max = static_cast<int>(budget / lce::kIBytesPerWord) / c->V;      // vectors
    const int ring_max = static_cast<int>(budget / (2 * lce::kIBytesPerWord)) / c->V;
    c->imma_chunks = c->Kv <= single_max ? 1 : cdiv(c->Kv, std::max(ring_max, 1));
    c->imma_Kc_v = cdiv(c->Kv, c->imma_chunks);
    c->imma_smem = static_cast<size_t>(c->imma_Kc_v) * c->V * lce::kIBytesPerWord *
                   (c->imma_chunks > 1 ? 2 : 1);  // two-deep ring
  }
  if (build_tc_weights(c, d_filter, want_tap_popc)) return 1;
  if (want_tap_popc) {
    const size_t n = static_cast<size_t>(c->cout + lce::kBN) * c->taps;
    CUDA_OK(cudaMalloc(&c->tap_popc, n * 4));
    CUDA_OK(cudaMemset(c->tap_popc, 0, n * 4));
    lce::tap_popc_kernel<<<cdiv(c->cout * c->taps, 256), 256>>>(d_filter, c->tap_popc, c->cout,
                                                                c->taps, c->Cw_pg);
    if (launch_check("tap_popc_kernel")) return 1;
  }
  CUDA_OK(cudaDeviceSynchronize());
  if (!on_dev) cudaFree(d_filter);
  return 0;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

// ------------------------------------------------------------------------- //
struct lce_b200_bconv2d {
  lce_bconv2d_desc d;
  int zp_mode = LCE_ZERO_PADDING_REFERENCE;
  int out_h = 0, out_w = 0, pad_h = 0, pad_w = 0;
  GemmCore core;
  int32_t* packed_scratch = nullptr;  // run_f32: packed activations
  size_t packed_scratch_words = 0;
  void* h2d_in = nullptr;             // run_host staging
  void* d2h_out = nullptr;
  size_t h2d_bytes = 0, d2h_bytes = 0;
};

struct lce_b200_bgemm {
  GemmCore core;
  int N = 0, Kw = 0;
};

extern "C" {

int lce_b200_abi_version(void) { return LCE_B200_ABI_VERSION; }
const char* lce_b200_last_error(void) { return g_err.c_str(); }
uint64_t lce_b200_launch_count(void) { return g_launches.load(); }
void lce_b200_path_counts(uint64_t out[3]) {
  for (int i = 0; i < 3; ++i) out[i] = g_path[i].load();
}
int lce_b200_tc_debug(int32_t out[8]) {
  int flag = 0;
  if (cudaMemcpyFromSymbol(&flag, lce::tc::g_tc_abort, sizeof(int)) != cudaSuccess) return 1;
  if (cudaMemcpyFromSymbol(out, lce::tc::g_tc_dbg, 8 * sizeof(int)) != cudaSuccess) return 1;
  out[7] = flag;
  if (flag) {
    const int zero = 0;
    cudaMemcpyToSymbol(lce::tc::g_tc_abort, &zero, sizeof(int));
  }
  return 0;
}

int lce_b200_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

// ------------------------------ LceQuantize ------------------------------ //
int lce_b200_quantize(int in_type, const void* in_dev, int64_t rows, int64_t cols,
                      int32_t zero_point, int32_t* out_dev, void* stream) {
  if (rows < 0 || cols < 0) return fail("quantize: negative shape");
  if (rows == 0 || cols == 0) return 0;
  if (cols > INT_MAX) return fail("quantize: last dimension too large");
  cudaStream_t s = as_stream(stream);
  const int cw = static_cast<int>((cols + 31) / 32);
  const long long n_words = rows * cw;
  switch (in_type) {
    case LCE_T_FLOAT:
      if (cols % 32 == 0 && aligned16(in_dev)) {
        lce::pack_f32_flat_kernel<<<grid_for(n_words * 4, 256), 256, 0, s>>>(
            static_cast<const float4*>(in_dev), out_dev, n_words);
        return launch_check("pack_f32_flat_kernel");
      }
      lce::pack_generic_kernel<float><<<grid_for(n_words * 32, 256), 256, 0, s>>>(
          static_cast<const float*>(in_dev), out_dev, rows, static_cast<int>(cols), cw, 0);
      return launch_check("pack_generic_kernel<float>");
    case LCE_T_INT8:
      lce::pack_generic_kernel<int8_t><<<grid_for(n_words * 32, 256), 256, 0, s>>>(
          static_cast<const int8_t*>(in_dev), out_dev, rows, static_cast<int>(cols), cw,
          zero_point);
      return launch_check("pack_generic_kernel<int8>");
    case LCE_T_BOOL:
      lce::pack_generic_kernel<uint8_t><<<grid_for(n_words * 32, 256), 256, 0, s>>>(
          static_cast<const uint8_t*>(in_dev), out_dev, rows, static_cast<int>(cols), cw, 1);
      return launch_check("pack_generic_kernel<bool>");
  }
  return fail("quantize: unsupported input type %d", in_type);
}

// ----------------------------- LceDequantize ----------------------------- //
int lce_b200_dequantize(int out_type, const int32_t* in_dev, int64_t rows, int64_t cols,
                        float scale, int32_t zero_point, void* out_dev, void* stream) {
  if (rows < 0 || cols < 0) return fail("dequantize: negative shape");
  if (rows == 0 || cols == 0) return 0;
  if (cols > INT_MAX) return fail("dequantize: last dimension too large");
  cudaStream_t s = as_stream(stream);
  const int cw = static_cast<int>((cols + 31) / 32);
  const int grid = grid_for(rows * cols, 256);
  switch (out_type) {
    case LCE_T_FLOAT:
      lce::unpack_kernel<float><<<grid, 256, 0, s>>>(in_dev, static_cast<float*>(out_dev), rows,
                                                     static_cast<int>(cols), cw, 1.0f, -1.0f);
      return launch_check("unpack_kernel<float>");
    case LCE_T_INT8: {
      // quantization.cc:130-138
      const int offset = static_cast<int>(std::round(1.0f / scale));
      const int8_t zero_bit = static_cast<int8_t>(std::min(127, zero_point + offset));
      const int8_t one_bit = static_cast<int8_t>(std::max(-128, zero_point - offset));
      lce::unpack_kernel<int8_t><<<grid, 256, 0, s>>>(in_dev, static_cast<int8_t*>(out_dev), rows,
                                                      static_cast<int>(cols), cw, zero_bit,
                                                      one_bit);
      return launch_check("unpack_kernel<int8>");
    }
    case LCE_T_BOOL:
      lce::unpack_kernel<uint8_t><<<grid, 256, 0, s>>>(in_dev, static_cast<uint8_t*>(out_dev),
                                                       rows, static_cast<int>(cols), cw,
                                                       uint8_t(1), uint8_t(0));
      return launch_check("unpack_kernel<bool>");
  }
  return fail("dequantize: unsupported output type %d", out_type);
}

// ----------------------------- LceBMaxPool2d ----------------------------- //
int lce_b200_bmaxpool_out_shape(const lce_bmaxpool_desc* d, int* out_h, int* out_w) {
  // bmaxpool.cc:51-54
  if (!d->stride_h || !d->stride_w || !d->filter_h || !d->filter_w)
    return fail("bmaxpool: strides and filter sizes must be non-zero");
  if (d->padding != LCE_PADDING_SAME && d->padding != LCE_PADDING_VALID)
    return fail("bmaxpool: unknown padding %d", d->padding);
  *out_h = out_size(d->padding, d->in_h, d->filter_h, d->stride_h, 1);
  *out_w = out_size(d->padding, d->in_w, d->filter_w, d->stride_w, 1);
  return 0;
}

int lce_b200_bmaxpool(const lce_bmaxpool_desc* d, const int32_t* in_dev, int32_t* out_dev,
                      void* stream) {
  int oh, ow;
  if (lce_b200_bmaxpool_out_shape(d, &oh, &ow)) return 1;
  const long long n = static_cast<long long>(d->batch) * oh * ow * d->channels_packed;
  if (n <= 0) return 0;
  const int ph = pad_before(d->stride_h, 1, d->in_h, d->filter_h, oh);
  const int pw = pad_before(d->stride_w, 1, d->in_w, d->filter_w, ow);
  lce::bmaxpool_kernel<<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(
      in_dev, out_dev, d->batch, d->in_h, d->in_w, d->channels_packed, oh, ow, d->filter_h,
      d->filter_w, d->stride_h, d->stride_w, ph, pw);
  return launch_check("bmaxpool_kernel");
}

// ------------------------------- LceBconv2d ------------------------------ //
int lce_b200_bconv2d_out_shape(const lce_bconv2d_desc* d, int* out_h, int* out_w, int* pad_h,
                               int* pad_w) {
  if (d->pad_value != 0 && d->pad_value != 1)
    return fail("Attribute pad_values must be 0 or 1.");  // bconv2d.cc:113-116
  if (d->padding != LCE_PADDING_SAME && d->padding != LCE_PADDING_VALID)
    return fail("bconv2d: unknown padding %d", d->padding);
  if (d->groups < 1 || d->channels_in < 1 || d->channels_out < 1 || d->filter_h < 1 ||
      d->filter_w < 1 || d->stride_h < 1 || d->stride_w < 1 || d->dilation_h < 1 ||
      d->dilation_w < 1)
    return fail("bconv2d: non-positive parameter");
  // bconv2d.cc:169-186
  if (d->channels_in % d->groups != 0)
    return fail("bconv2d: channels_in %d not divisible by groups %d", d->channels_in, d->groups);
  if (d->groups > 1 && (d->channels_in / d->groups) % 32 != 0)
    return fail("bconv2d: grouped convolutions need channels_in/groups %% 32 == 0");
  if (d->channels_out % d->groups != 0)
    return fail("bconv2d: channels_out %d not divisible by groups %d", d->channels_out,
                d->groups);
  *out_h = out_size(d->padding, d->in_h, d->filter_h, d->stride_h, d->dilation_h);
  *out_w = out_size(d->padding, d->in_w, d->filter_w, d->stride_w, d->dilation_w);
  *pad_h = pad_before(d->stride_h, d->dilation_h, d->in_h, d->filter_h, *out_h);
  *pad_w = pad_before(d->stride_w, d->dilation_w, d->in_w, d->filter_w, *out_w);
  if (*out_h < 0) *out_h = 0;
  if (*out_w < 0) *out_w = 0;
  return 0;
}

int lce_b200_bconv2d_create(const lce_bconv2d_desc* d, const int32_t* filter,
                            const float* post_mul, const float* post_bias,
                            const int32_t* thresholds, lce_b200_bconv2d** out_plan) {
  *out_plan = nullptr;
  if (lce_b200_device_count() < 1) return fail("no CUDA device: this library has no CPU path");
  int oh, ow, ph, pw;
  if (lce_b200_bconv2d_out_shape(d, &oh, &ow, &ph, &pw)) return 1;
  if (d->out_type != LCE_OUT_FLOAT && d->out_type != LCE_OUT_INT8 &&
      d->out_type != LCE_OUT_BITPACKED)
    return fail("Supported output types are int8, int32, and float32.");  // bconv2d.cc:158-162
  const bool zero_pad = d->padding == LCE_PADDING_SAME && d->pad_value == 0;
  // bconv2d.cc:188-200: the reference kernel's rule (even channels_in) or the optimised kernels'
  // (float output, no fused activation); the plan starts in the mode whose rule holds
  const bool zp_ref_rule = d->channels_in % 2 == 0;
  const bool zp_opt_rule = d->out_type == LCE_OUT_FLOAT && d->activation == LCE_ACT_NONE;
  if (zero_pad && !zp_ref_rule && !zp_opt_rule)
    return fail("Zero-padding is only supported by the reference kernel with an even number of "
                "input channels, or when using float output with no fused activation function.");
  if (d->out_type == LCE_OUT_BITPACKED) {
    if (!thresholds) return fail("bconv2d: bitpacked output needs the thresholds input");
  } else if (!post_mul || !post_bias) {
    return fail("bconv2d: float/int8 output needs post_activation_multiplier and bias");
  }
  if (!filter) return fail("bconv2d: filter is null");

  auto* plan = new lce_b200_bconv2d();
  plan->d = *d;
  plan->zp_mode = (zero_pad && !zp_ref_rule) ? LCE_ZERO_PADDING_CORRECTION : LCE_ZERO_PADDING_REFERENCE;
  plan->out_h = oh; plan->out_w = ow; plan->pad_h = ph; plan->pad_w = pw;
  GemmCore& c = plan->core;
  c.groups = d->groups;
  c.cout = d->channels_out;
  c.cout_pg = d->channels_out / d->groups;
  c.Cw_pg = cdiv(d->channels_in / d->groups, 32);
  c.taps = d->filter_h * d->filter_w;
  c.out_type = d->out_type;
  int rc = build_core_weights(&c, filter, zero_pad);

  const size_t padded = static_cast<size_t>(c.cout) + kChanPad;
  if (!rc && d->out_type != LCE_OUT_BITPACKED) {
    // OneTimeSetup (bconv2d.cc:353-389): fold in double on the host.
    std::vector<float> pm(c.cout), pb(c.cout), fm(padded, 0.f), fb(padded, 0.f);
    rc = to_host(post_mul, c.cout * sizeof(float), pm.data()) ||
         to_host(post_bias, c.cout * sizeof(float), pb.data());
    const int32_t backtransform_add = d->filter_h * d->filter_w * (d->channels_in / d->groups);
    const double scale = d->out_type == LCE_OUT_INT8 ? static_cast<double>(d->out_scale) : 1.0;
    const double zp = d->out_type == LCE_OUT_INT8 ? static_cast<double>(d->out_zero_point) : 0.0;
    for (int i = 0; i < c.cout; ++i) {
      const double m = pm[i], b = pb[i];
      fm[i] = static_cast<float>(-1 * m / scale);
      fb[i] = static_cast<float>((b + static_cast<double>(backtransform_add) * m) / scale + zp);
    }
    int32_t nmin, nmax;  // CalculateActivationRange<int32>, kernel_util.h:285-300
    switch (d->activation) {
      case LCE_ACT_RELU: nmin = 0; nmax = INT32_MAX; break;
      case LCE_ACT_RELU6: nmin = 0; nmax = 6; break;
      case LCE_ACT_RELU_N1_TO_1: nmin = -1; nmax = 1; break;
      default: nmin = INT32_MIN; nmax = INT32_MAX; break;
    }
    nmin = std::max(nmin, -backtransform_add);
    nmax = std::min(nmax, backtransform_add);
    c.clamp_min = -nmax + backtransform_add;
    c.clamp_max = -nmin + backtransform_add;
    void *dm = nullptr, *db = nullptr;
    rc = rc || to_device(fm.data(), padded * 4, padded * 4, &dm) ||
         to_device(fb.data(), padded * 4, padded * 4, &db);
    c.mul = static_cast<float*>(dm);
    c.bias = static_cast<float*>(db);
    if (!rc && zero_pad && zp_opt_rule && c.tc_ok && c.tc_tap_popc_t != nullptr) {
      // the optimised kernels' correction cache (zero_padding_correction.h:39-176), once per plan
      const int eff_h = (d->filter_h - 1) * d->dilation_h + 1, eff_w = (d->filter_w - 1) * d->dilation_w + 1;
      const size_t n = static_cast<size_t>(4) * eff_h * eff_w * c.tc_ldc;
      if (cudaMalloc(&c.tc_zpc_cache, n * 4) != cudaSuccess || cudaMemset(c.tc_zpc_cache, 0, n * 4) != cudaSuccess) {
        rc = fail("bconv2d: cannot allocate the zero-padding correction cache");
      } else {
        const int total = 4 * eff_h * eff_w * c.cout;
        lce::tc::zpc_cache_kernel<<<cdiv(total, 256), 256>>>(c.tc_tap_popc_t, c.mul, c.tc_zpc_cache, c.cout, c.tc_ldc,
                                                           d->filter_h, d->filter_w, d->dilation_h, d->dilation_w,
                                                           d->channels_in / d->groups);
        rc = launch_check("zpc_cache_kernel");
        if (!rc && cudaDeviceSynchronize() != cudaSuccess) rc = fail("zpc_cache_kernel failed");
      }
    }
  } else if (!rc) {
    void* dt = nullptr;
    rc = to_device(thresholds, c.cout * 4, padded * 4, &dt);
    c.thr = static_cast<int32_t*>(dt);
  }
  if (rc) {
    c.release();
    delete plan;
    return 1;
  }
  *out_plan = plan;
  return 0;
}

int lce_b200_bconv2d_set_input_shape(lce_b200_bconv2d* plan, int batch, int in_h, int in_w) {
  lce_bconv2d_desc d = plan->d;
  d.batch = batch; d.in_h = in_h; d.in_w = in_w;
  if (batch < 0 || in_h < 1 || in_w < 1) return fail("bconv2d: bad input shape");
  int oh, ow, ph, pw;
  if (lce_b200_bconv2d_out_shape(&d, &oh, &ow, &ph, &pw)) return 1;
  plan->d = d;
  plan->out_h = oh; plan->out_w = ow; plan->pad_h = ph; plan->pad_w = pw;
  return 0;
}

int lce_b200_bconv2d_set_zero_padding_mode(lce_b200_bconv2d* plan, int mode) {
  const lce_bconv2d_desc& d = plan->d;
  if (mode == LCE_ZERO_PADDING_CORRECTION) {
    if (d.padding == LCE_PADDING_SAME && d.pad_value == 0 &&
        !(d.out_type == LCE_OUT_FLOAT && d.activation == LCE_ACT_NONE))
      return fail("Zero-padding is only supported by the reference kernel with an even number of "
                  "input channels, or when using float output with no fused activation function.");
  } else if (mode == LCE_ZERO_PADDING_REFERENCE) {
    if (d.padding == LCE_PADDING_SAME && d.pad_value == 0 && d.channels_in % 2 != 0)
      return fail("Zero-padding is only supported by the reference kernel with an even number of "
                  "input channels, or when using float output with no fused activation function.");
  } else {
    return fail("bconv2d: unknown zero-padding mode %d", mode);
  }
  plan->zp_mode = mode;
  return 0;
}

int lce_b200_bconv2d_get_desc(const lce_b200_bconv2d* plan, lce_bconv2d_desc* d, int* out_h,
                              int* out_w) {
  *d = plan->d;
  *out_h = plan->out_h;
  *out_w = plan->out_w;
  return 0;
}

static size_t bconv_out_bytes(const lce_b200_bconv2d* plan) {
  const size_t px = static_cast<size_t>(plan->d.batch) * plan->out_h * plan->out_w;
  switch (plan->d.out_type) {
    case LCE_OUT_BITPACKED: return px * cdiv(plan->d.channels_out, 32) * 4;
    case LCE_OUT_INT8: return px * plan->d.channels_out;
    default: return px * plan->d.channels_out * 4;
  }
}

static int bconv_run_impl(lce_b200_bconv2d* plan, const int32_t* in_dev, void* out_dev,
                          const float* residual, int residual_act, int32_t* packed_out,
                          void* stream) {
  const lce_bconv2d_desc& d = plan->d;
  GemmCore& c = plan->core;
  cudaStream_t s = as_stream(stream);
  lce::ConvKParams p;
  memset(&p, 0, sizeof(p));
  p.in = in_dev; p.wt = c.wt; p.out = out_dev;
  p.mul = c.mul; p.bias = c.bias; p.thr = c.thr; p.tap_popc = c.tap_popc;
  p.residual = residual; p.packed_out = packed_out; p.residual_act = residual_act;
  p.M = static_cast<long long>(d.batch) * plan->out_h * plan->out_w;
  p.H = d.in_h; p.W = d.in_w;
  p.Cw_total = cdiv(d.channels_in, 32);
  p.Cw_pg = c.Cw_pg; p.CwV = c.Cw_pg / c.V;
  p.KH = d.filter_h; p.KW = d.filter_w;
  p.sh = d.stride_h; p.sw = d.stride_w; p.dh = d.dilation_h; p.dw = d.dilation_w;
  p.ph = plan->pad_h; p.pw = plan->pad_w; p.OH = plan->out_h; p.OW = plan->out_w;
  p.cout = c.cout; p.cout_pg = c.cout_pg; p.tiles_per_group = c.tiles_per_group;
  p.Kv = c.Kv; p.Kc_v = c.Kc_v; p.n_chunks = c.n_chunks;
  p.clamp_min = c.clamp_min; p.clamp_max = c.clamp_max;
  p.cw_out = cdiv(c.cout, 32);
  p.zp_half = (d.channels_in / d.groups) / 2;
  if (d.out_type == LCE_OUT_INT8)
    p.vec_store = (c.cout % 8 == 0 && c.cout_pg % 8 == 0 &&
                   (reinterpret_cast<uintptr_t>(out_dev) & 7u) == 0);
  else
    p.vec_store = (c.cout % 4 == 0 && c.cout_pg % 4 == 0 && aligned16(out_dev));
  p.bp_fast = (c.groups == 1 || c.cout_pg % 32 == 0);
  // Stage the shortcut rows through shared memory when every tile is full (so each thread
  // owns 8 valid, 16-byte aligned channels) and the extra 16 KB keep the CTAs/SM resident.
  static const bool res_stage_on = [] {
    const char* e = getenv("LCE_B200_RES_STAGE");
    return !(e && e[0] == '0');
  }();
  p.res_stage = res_stage_on && residual != nullptr && d.out_type == LCE_OUT_FLOAT &&
                p.vec_store && c.cout_pg % lce::kBN == 0 &&
                c.smem_bytes + lce::kResStageBytes <= cta_smem_budget();
  if (p.M == 0) return 0;
  // The 4V-byte cp.async gathers need 4V-byte aligned pixels.
  if ((reinterpret_cast<uintptr_t>(in_dev) & (4u * c.V - 1)) != 0)
    return fail("bconv2d: input pointer must be %d-byte aligned", 4 * c.V);
  if (d.out_type == LCE_OUT_BITPACKED && !p.bp_fast)
    CUDA_OK(cudaMemsetAsync(out_dev, 0, bconv_out_bytes(plan), s));
  const bool zp_float = c.tap_popc != nullptr && plan->zp_mode == LCE_ZERO_PADDING_CORRECTION;
  if (!zp_float) return launch_conv(c, p, s);
  // the optimised kernels' zero padding: one-padding accumulators + a float correction. The
  // tcgen05 kernel does it in its epilogue; the others run unfused and a tail pass finishes.
  p.zp_float = 1;
  p.cin_pg = d.channels_in / d.groups;
  if (c.tc_ok) {
    const int rc = tc_launch(c, p, s);
    if (rc >= 0) return rc;
  }
  lce::ConvKParams q = p;
  q.tap_popc = nullptr; q.residual = nullptr; q.packed_out = nullptr; q.res_stage = 0; q.zp_float = 0;
  const bool tc_was = c.tc_ok;
  c.tc_ok = false;
  const int rc = launch_conv(c, q, s);
  c.tc_ok = tc_was;
  if (rc) return rc;
  lce::ZpcTailParams z;
  z.out = static_cast<float*>(out_dev); z.mul = c.mul; z.tap_popc = c.tap_popc;
  z.residual = residual; z.packed_out = packed_out; z.M = p.M;
  z.H = p.H; z.W = p.W; z.OH = p.OH; z.OW = p.OW; z.KH = p.KH; z.KW = p.KW;
  z.sh = p.sh; z.sw = p.sw; z.dh = p.dh; z.dw = p.dw;
  z.cout = c.cout; z.cin_pg = p.cin_pg; z.cw_out = p.cw_out; z.residual_act = residual_act;
  lce::zpc_tail_kernel<<<grid_for(p.M * cdiv(c.cout, 32) * 32, 256), 256, 0, s>>>(z);
  return launch_check("zpc_tail_kernel");
}

int lce_b200_bconv2d_run(lce_b200_bconv2d* plan, const int32_t* in_dev, void* out_dev,
                         void* stream) {
  return bconv_run_impl(plan, in_dev, out_dev, nullptr, LCE_ACT_NONE, nullptr, stream);
}

int lce_b200_bconv2d_run_fused(lce_b200_bconv2d* plan, const int32_t* in_dev,
                               const float* residual_dev, int add_activation, float* out_dev,
                               int32_t* packed_out_dev, void* stream) {
  if (plan->d.out_type != LCE_OUT_FLOAT)
    return fail("bconv2d_run_fused: only float-output plans can take a residual");
  if (packed_out_dev && plan->d.groups != 1)
    return fail("bconv2d_run_fused: packed output needs groups == 1");
  if (residual_dev && (reinterpret_cast<uintptr_t>(residual_dev) & 15u) != 0)
    return fail("bconv2d_run_fused: residual must be 16-byte aligned");
  return bconv_run_impl(plan, in_dev, out_dev, residual_dev, add_activation, packed_out_dev,
                        stream);
}

int lce_b200_bconv2d_run_f32(lce_b200_bconv2d* plan, const float* in_dev, void* out_dev,
                             void* stream) {
  const lce_bconv2d_desc& d = plan->d;
  const int cw = cdiv(d.channels_in, 32);
  const size_t rows = static_cast<size_t>(d.batch) * d.in_h * d.in_w;
  const size_t words = rows * cw;
  if (words > plan->packed_scratch_words) {
    cudaFree(plan->packed_scratch);
    plan->packed_scratch = nullptr;
    plan->packed_scratch_words = 0;
    CUDA_OK(cudaMalloc(&plan->packed_scratch, words * 4 + 16));
    plan->packed_scratch_words = words;
  }
  if (lce_b200_quantize(LCE_T_FLOAT, in_dev, static_cast<int64_t>(rows), d.channels_in, 0,
                        plan->packed_scratch, stream))
    return 1;
  return lce_b200_bconv2d_run(plan, plan->packed_scratch, out_dev, stream);
}

int lce_b200_bconv2d_run_host(lce_b200_bconv2d* plan, const int32_t* in_host, void* out_host) {
  const lce_bconv2d_desc& d = plan->d;
  const size_t in_bytes =
      static_cast<size_t>(d.batch) * d.in_h * d.in_w * cdiv(d.channels_in, 32) * 4;
  const size_t out_bytes = bconv_out_bytes(plan);
  if (in_bytes > plan->h2d_bytes) {
    cudaFree(plan->h2d_in);
    plan->h2d_in = nullptr; plan->h2d_bytes = 0;
    CUDA_OK(cudaMalloc(&plan->h2d_in, in_bytes + 16));
    plan->h2d_bytes = in_bytes;
  }
  if (out_bytes > plan->d2h_bytes) {
    cudaFree(plan->d2h_out);
    plan->d2h_out = nullptr; plan->d2h_bytes = 0;
    CUDA_OK(cudaMalloc(&plan->d2h_out, out_bytes + 16));
    plan->d2h_bytes = out_bytes;
  }
  if (in_bytes) CUDA_OK(cudaMemcpyAsync(plan->h2d_in, in_host, in_bytes, cudaMemcpyHostToDevice, 0));
  if (lce_b200_bconv2d_run(plan, static_cast<const int32_t*>(plan->h2d_in), plan->d2h_out,
                           nullptr))
    return 1;
  if (out_bytes)
    CUDA_OK(cudaMemcpyAsync(out_host, plan->d2h_out, out_bytes, cudaMemcpyDeviceToHost, 0));
  CUDA_OK(cudaStreamSynchronize(0));
  return 0;
}

void lce_b200_bconv2d_destroy(lce_b200_bconv2d* plan) {
  if (!plan) return;
  plan->core.release();
  cudaFree(plan->packed_scratch);
  cudaFree(plan->h2d_in);
  cudaFree(plan->d2h_out);
  delete plan;
}

// --------------------------------- BGEMM --------------------------------- //
int lce_b200_bgemm_create(int N, int Kw, const int32_t* W, const lce_bgemm_epilogue* ep,
                          lce_b200_bgemm** out_plan) {
  *out_plan = nullptr;
  if (lce_b200_device_count() < 1) return fail("no CUDA device: this library has no CPU path");
  if (N < 1 || Kw < 1 || !W || !ep) return fail("bgemm: bad arguments");
  if (ep->out_type < LCE_OUT_FLOAT || ep->out_type > LCE_OUT_RAW_ACC)
    return fail("bgemm: unsupported output type %d", ep->out_type);
  auto* plan = new lce_b200_bgemm();
  plan->N = N; plan->Kw = Kw;
  GemmCore& c = plan->core;
  c.groups = 1; c.cout = N; c.cout_pg = N; c.Cw_pg = Kw; c.taps = 1;
  c.out_type = ep->out_type;
  c.clamp_min = ep->clamp_min; c.clamp_max = ep->clamp_max;
  int rc = build_core_weights(&c, W, false);
  const size_t padded = static_cast<size_t>(N) + kChanPad;
  if (!rc && (ep->out_type == LCE_OUT_FLOAT || ep->out_type == LCE_OUT_INT8)) {
    if (!ep->multiplier || !ep->bias) rc = fail("bgemm: multiplier/bias missing");
    void *dm = nullptr, *db = nullptr;
    rc = rc || to_device(ep->multiplier, N * 4, padded * 4, &dm) ||
         to_device(ep->bias, N * 4, padded * 4, &db);
    c.mul = static_cast<float*>(dm);
    c.bias = static_cast<float*>(db);
  } else if (!rc && ep->out_type == LCE_OUT_BITPACKED) {
    if (!ep->thresholds) rc = fail("bgemm: thresholds missing");
    void* dt = nullptr;
    rc = rc || to_device(ep->thresholds, N * 4, padded * 4, &dt);
    c.thr = static_cast<int32_t*>(dt);
  }
  if (rc) {
    c.release();
    delete plan;
    return 1;
  }
  *out_plan = plan;
  return 0;
}

int lce_b200_bgemm_run(lce_b200_bgemm* plan, int64_t M, const int32_t* A_dev, void* out_dev,
                       void* stream) {
  GemmCore& c = plan->core;
  if (M < 0) return fail("bgemm: negative M");
  if (M == 0) return 0;
  if (M > INT_MAX) return fail("bgemm: M too large");
  lce::ConvKParams p;
  memset(&p, 0, sizeof(p));
  p.in = A_dev; p.wt = c.wt; p.out = out_dev;
  p.mul = c.mul; p.bias = c.bias; p.thr = c.thr; p.tap_popc = nullptr;
  p.M = M;
  p.H = 1; p.W = 1;  // every row of A is its own 1 x 1 "image": offsets stay 32-bit
  p.Cw_total = plan->Kw; p.Cw_pg = plan->Kw; p.CwV = plan->Kw / c.V;
  p.KH = p.KW = 1; p.sh = p.sw = p.dh = p.dw = 1; p.ph = p.pw = 0;
  p.OH = 1; p.OW = 1;
  p.cout = c.cout; p.cout_pg = c.cout_pg; p.tiles_per_group = c.tiles_per_group;
  p.Kv = c.Kv; p.Kc_v = c.Kc_v; p.n_chunks = c.n_chunks;
  p.clamp_min = c.clamp_min; p.clamp_max = c.clamp_max;
  p.cw_out = cdiv(c.cout, 32);
  if (c.out_type == LCE_OUT_INT8)
    p.vec_store = (c.cout % 8 == 0 && (reinterpret_cast<uintptr_t>(out_dev) & 7u) == 0);
  else
    p.vec_store = (c.cout % 4 == 0 && aligned16(out_dev));
  p.bp_fast = 1;
  if ((reinterpret_cast<uintptr_t>(A_dev) & (4u * c.V - 1)) != 0)
    return fail("bgemm: A must be %d-byte aligned", 4 * c.V);
  return launch_conv(c, p, as_stream(stream));
}

void lce_b200_bgemm_destroy(lce_b200_bgemm* plan) {
  if (!plan) return;
  plan->core.release();
  delete plan;
}

}  // extern "C"
