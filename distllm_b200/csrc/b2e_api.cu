// libb2e.so -- C ABI (include/b2e.h) over the sm_100a kernels.  Host runtime only: handle,
// lazily grown workspace, TMA descriptors and launches.  No CPU fallback: without an sm_100 device
// every compute entry point fails with B2E_ERR_NO_DEVICE.
#include "../../include/b2e.h"
#include "../../include/b2e_debug.h"

#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "attention3.cuh"
#include "attention4.cuh"
#include "attention5.cuh"
#include "binsearch.cuh"
#include "common.cuh"
#include "gemm.cuh"
#include "gemm2.cuh"
#include "mistral_ops.cuh"
#include "pack.cuh"
#include "rowops.cuh"
#include "topk.cuh"
#include "topk_tc.cuh"

using namespace b2e;

// the 16-bit storage type of this build (common.cuh): tensor-map element type and its ABI dtype code
#ifdef B2E_STORAGE_BF16
#define B2E_TMAP_DTYPE CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
constexpr int kStorageDtype = B2E_DTYPE_BF16;
#else
#define B2E_TMAP_DTYPE CU_TENSOR_MAP_DATA_TYPE_FLOAT16
constexpr int kStorageDtype = B2E_DTYPE_F16;
#endif

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                    \
  do {                                                                                    \
    cudaError_t e_ = (expr);                                                              \
    if (e_ != cudaSuccess)                                                                \
      return fail(B2E_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_),   \
                  __FILE__, __LINE__);                                                    \
  } while (0)

// ---- driver entry point for tensor-map encoding (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// 2-D half row-major [rows, cols] tensor, box = 64 columns (128 B, swizzle-128B) x box_rows.
int make_tmap_h16(CUtensorMap* tm, const void* base, uint64_t rows, uint64_t cols,
                   uint32_t box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return fail(B2E_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, B2E_TMAP_DTYPE, 2, const_cast<void*>(base), dims, strides,
                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(B2E_ERR_CUDA, "cuTensorMapEncodeTiled(rows=%llu, cols=%llu, box_rows=%u) -> %d",
                (unsigned long long)rows, (unsigned long long)cols, box_rows, (int)r);
  return B2E_OK;
}

// 2-D float32 row-major tensor, box = 32 columns (128 bytes) x box_rows, 128-byte swizzle; rows beyond the
// tensor read as zeros
int make_tmap_f32(CUtensorMap* tm, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return fail(B2E_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * 4};
  cuuint32_t box[2] = {32, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(B2E_ERR_CUDA, "cuTensorMapEncodeTiled f32(rows=%llu, cols=%llu, box_rows=%u) -> %d",
                (unsigned long long)rows, (unsigned long long)cols, box_rows, (int)r);
  return B2E_OK;
}

struct DeviceInfo {
  int sms = 0;
  int cc_major = 0;
  bool ok = false;
};

int device_info(int device, DeviceInfo* info) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    cudaGetLastError();
    return fail(B2E_ERR_NO_DEVICE, "no CUDA device visible; libb2e has no CPU fallback");
  }
  if (device < 0 || device >= n) return fail(B2E_ERR_INVALID, "device %d out of range", device);
  cudaDeviceProp p;
  CUDA_TRY(cudaGetDeviceProperties(&p, device));
  if (p.major != 10)
    return fail(B2E_ERR_NO_DEVICE, "device %d is sm_%d%d; libb2e is built for sm_100a only", device,
                p.major, p.minor);
  info->sms = p.multiProcessorCount;
  info->cc_major = p.major;
  info->ok = true;
  return B2E_OK;
}

int current_device_info(DeviceInfo* info) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();
    return fail(B2E_ERR_NO_DEVICE, "no CUDA device visible; libb2e has no CPU fallback");
  }
  static DeviceInfo cache[64];
  if (dev < 64 && cache[dev].ok) {
    *info = cache[dev];
    return B2E_OK;
  }
  int rc = device_info(dev, info);
  if (rc == B2E_OK && dev < 64) cache[dev] = *info;
  return rc;
}

// Opt a kernel in to `bytes` of dynamic shared memory, once per (kernel, device): the attribute belongs
// to the device's context, and a process may drive more than one device over its lifetime.
template <typename Kern>
int ensure_smem_attr(Kern kern, int bytes) {
  // keyed by the kernel's ADDRESS (kernels with equal signatures share one C++ type) and the device
  static std::vector<std::pair<const void*, int>> done;
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  const void* key = reinterpret_cast<const void*>(kern);
  for (const auto& d : done)
    if (d.first == key && d.second == dev) return B2E_OK;
  CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  done.emplace_back(key, dev);
  return B2E_OK;
}

// ---------------------------------------------------------------- launches
template <int BN, int STAGES, int EPI>
int launch_gemm_cfg(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tout,
                    const float* bias, const h16* resid, int M, int N, int K, int sms,
                    cudaStream_t st, const int* m_dev = nullptr) {
  using Cfg = GemmCfg<BN, STAGES>;
  auto kern = gemm_h16_tcgen05_kernel<BN, STAGES, EPI>;
  {
    const int arc = ensure_smem_attr(kern, Cfg::SMEM_BYTES);
    if (arc) return arc;
  }
  const int tiles = ((M + GEMM_BM - 1) / GEMM_BM) * (N / BN);
  const int grid = tiles < sms ? tiles : sms;
  static int cluster_probe = -1;  // B2E_GEMM=v1cluster: same kernel, launched as clusters of 2 (experiment)
  if (cluster_probe < 0) {
    const char* e = getenv("B2E_GEMM");
    cluster_probe = (e && strcmp(e, "v1cluster") == 0) ? 1 : 0;
  }
  if (cluster_probe) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid & ~1);
    cfg.blockDim = dim3(GEMM_THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, ta, tb, tout, bias, resid, M, N, K, m_dev));
    return B2E_OK;
  }
  kern<<<grid, GEMM_THREADS, Cfg::SMEM_BYTES, st>>>(ta, tb, tout, bias, resid, M, N, K, m_dev);
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

template <int BN, int STAGES>
int launch_gemm_bn(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tout,
                   const float* bias, const h16* resid, int M, int N, int K, int epi, int sms,
                   cudaStream_t st, const int* m_dev = nullptr) {
  switch (epi) {
    case B2E_EPI_BIAS:
      return launch_gemm_cfg<BN, STAGES, EPI_BIAS>(ta, tb, tout, bias, resid, M, N, K, sms, st, m_dev);
    case B2E_EPI_BIAS_GELU:
      return launch_gemm_cfg<BN, STAGES, EPI_BIAS_GELU>(ta, tb, tout, bias, resid, M, N, K, sms, st, m_dev);
    case B2E_EPI_BIAS_RESID:   // m_dev used to be dropped here: with N % 256 == 128 every row tile up to M was written
      return launch_gemm_cfg<BN, STAGES, EPI_BIAS_RESID>(ta, tb, tout, bias, resid, M, N, K, sms, st, m_dev);
    case B2E_EPI_SWIGLU:
      if constexpr (BN == 256)
        return launch_gemm_cfg<256, STAGES, EPI_SWIGLU>(ta, tb, tout, bias, resid, M, N, K, sms, st, m_dev);
      else
        return fail(B2E_ERR_INVALID, "SwiGLU epilogue needs N %% 256 == 0");
    case B2E_EPI_GEGLU:
      if constexpr (BN == 256)
        return launch_gemm_cfg<256, STAGES, EPI_GEGLU>(ta, tb, tout, bias, resid, M, N, K, sms, st, m_dev);
      else
        return fail(B2E_ERR_INVALID, "GeGLU epilogue needs N %% 256 == 0");
  }
  return fail(B2E_ERR_INVALID, "unknown epilogue %d", epi);
}

// The CTA-pair kernel (gemm2.cuh, 256 x 256 tiles over two SMs) is the default whenever N is a multiple
// of 256; B2E_GEMM=single forces the single-CTA kernel (gemm.cuh), which also serves N % 256 == 128.
inline bool gemm_use_pair() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B2E_GEMM");
    v = (e && strcmp(e, "single") == 0) ? 0 : 1;
  }
  return v == 1;
}
// rows of the W tile one TMA box covers: the pair kernel stages half of the 256-row tile per CTA
inline int gemm_bn_for(int N) { return (N % 256 == 0 && !gemm_use_pair()) ? 256 : 128; }

int check_gemm_shape(int M, int N, int K) {
  if (M <= 0 || N <= 0 || K <= 0) return fail(B2E_ERR_INVALID, "gemm: empty shape %dx%dx%d", M, N, K);
  if (N % 128 != 0) return fail(B2E_ERR_INVALID, "gemm: N=%d must be a multiple of 128", N);
  if (K % 64 != 0) return fail(B2E_ERR_INVALID, "gemm: K=%d must be a multiple of 64", K);
  return B2E_OK;
}

bool g_gemm2_profiling = false;   // b2e_debug_set_clock_buffer / b2e_debug_set_pair_flags: use the instrumented GEMM

template <int STAGES, int EPI>
int launch_gemm2_cfg(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tout,
                     const float* bias, const h16* resid, int M, int N, int K, int sms,
                     cudaStream_t st, const int* m_dev = nullptr) {
  using Cfg = Gemm2Cfg<STAGES>;
  const int tiles = ((M + 255) / 256) * (N / G2_BN);
  int grid = 2 * tiles;
  if (grid > (sms & ~1)) grid = sms & ~1;
  if constexpr (EPI == EPI_BIAS) {
    if (g_gemm2_profiling) {   // a clock buffer or an experiment flag is set: the instrumented instantiation
      auto kern_tl = gemm2_h16_pair_kernel<STAGES, EPI, true>;
      const int arc = ensure_smem_attr(kern_tl, Cfg::SMEM_BYTES);
      if (arc) return arc;
      kern_tl<<<grid, G2_THREADS, Cfg::SMEM_BYTES, st>>>(ta, tb, tout, bias, resid, M, N, K, m_dev);
      CUDA_TRY(cudaGetLastError());
      return B2E_OK;
    }
  }
  auto kern = gemm2_h16_pair_kernel<STAGES, EPI>;
  {
    const int arc = ensure_smem_attr(kern, Cfg::SMEM_BYTES);
    if (arc) return arc;
  }
  kern<<<grid, G2_THREADS, Cfg::SMEM_BYTES, st>>>(ta, tb, tout, bias, resid, M, N, K, m_dev);
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

// A map: [M,K] box 128 rows; W map: [N,K] box gemm_bn_for(N) rows.
// m_dev (nullable): device-resident row count <= M (packed token layout); M sizes the grid and the tensor maps.
int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, void* out, const float* bias,
                const void* resid, int M, int N, int K, int epi, int sms, cudaStream_t st,
                const int* m_dev = nullptr) {
  const h16* r = static_cast<const h16*>(resid);
  // output tiles leave through TMA stores: [M,N] row-major, box = 64 columns x 32 rows
  CUtensorMap tout;
  int rc;
  const bool glu = epi == B2E_EPI_SWIGLU || epi == B2E_EPI_GEGLU;
  const int n_out = glu ? N / 2 : N;   // the gated epilogues write act(first) * second: [M, N/2]
  if ((rc = make_tmap_h16(&tout, out, M, n_out, GEMM_OUT_BOX_ROWS))) return rc;
  if (N % 256 == 0 && gemm_use_pair()) {
    constexpr int PS = 5;   // 5 x 32 KiB stages + two staging tiles per epilogue warp
    switch (epi) {
      case B2E_EPI_BIAS: return launch_gemm2_cfg<PS, EPI_BIAS>(ta, tb, tout, bias, r, M, N, K, sms, st, m_dev);
      case B2E_EPI_BIAS_GELU: return launch_gemm2_cfg<PS, EPI_BIAS_GELU>(ta, tb, tout, bias, r, M, N, K, sms, st, m_dev);
      case B2E_EPI_BIAS_RESID: return launch_gemm2_cfg<PS, EPI_BIAS_RESID>(ta, tb, tout, bias, r, M, N, K, sms, st, m_dev);
      case B2E_EPI_SWIGLU: return launch_gemm2_cfg<PS, EPI_SWIGLU>(ta, tb, tout, bias, r, M, N, K, sms, st, m_dev);
      case B2E_EPI_GEGLU: return launch_gemm2_cfg<PS, EPI_GEGLU>(ta, tb, tout, bias, r, M, N, K, sms, st, m_dev);
    }
    return fail(B2E_ERR_INVALID, "unknown epilogue %d", epi);
  }
  if (N % 256 == 0) return launch_gemm_bn<256, 4>(ta, tb, tout, bias, r, M, N, K, epi, sms, st, m_dev);
  return launch_gemm_bn<128, 6>(ta, tb, tout, bias, r, M, N, K, epi, sms, st, m_dev);
}

// Per-forward attention inputs derived from the mask (attention3.cuh): additive key bias rows and
// the number of 64-key chunks that hold an attended key.
struct AttnScratch {
  float* bias = nullptr;   // [B, S_pad]
  int* kv_chunks = nullptr;  // [B]
  int* plain_chunks = nullptr;  // [B]  leading fully-attended chunks
  size_t cap_bias = 0, cap_b = 0;
  uint64_t gen = 0;   // bumped on every reallocation
  int device = -1;    // the buffers live on this device; a call from another one starts over
  int ensure(int B, int S_pad) {
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev != device) {
      release();
      device = dev;
      ++gen;
    }
    if ((size_t)B * S_pad > cap_bias || (size_t)B > cap_b) ++gen;
    // pointer nulled and capacity zeroed BEFORE the new allocation: a failed cudaMalloc must not leave
    // a dangling pointer behind a non-zero capacity
    if ((size_t)B * S_pad > cap_bias) {
      cudaFree(bias);
      bias = nullptr;
      cap_bias = 0;
      CUDA_TRY(cudaMalloc(&bias, sizeof(float) * (size_t)B * S_pad));
      cap_bias = (size_t)B * S_pad;
    }
    if ((size_t)B > cap_b) {
      cudaFree(kv_chunks); cudaFree(plain_chunks);
      kv_chunks = plain_chunks = nullptr;
      cap_b = 0;
      CUDA_TRY(cudaMalloc(&kv_chunks, sizeof(int) * B));
      CUDA_TRY(cudaMalloc(&plain_chunks, sizeof(int) * B));
      cap_b = B;
    }
    return B2E_OK;
  }
  void release() {
    cudaFree(bias); cudaFree(kv_chunks); cudaFree(plain_chunks);
    bias = nullptr; kv_chunks = plain_chunks = nullptr; cap_bias = cap_b = 0;
  }
};

inline int attn_s_pad(int S) { return (S + AT3_KC - 1) / AT3_KC * AT3_KC; }

int attention_prepare(AttnScratch& sc, const int64_t* mask, int B, int S, cudaStream_t st) {
  int rc;
  const int S_pad = attn_s_pad(S);
  if ((rc = sc.ensure(B, S_pad))) return rc;
  attn_prep_kernel<<<(B + 7) / 8, 256, 0, st>>>(mask, sc.bias, sc.kv_chunks, sc.plain_chunks, B, S, S_pad);
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

// Softmax variant of the head_dim-64 attention kernel (template parameter V of attention3_d64_kernel);
// B2E_ATT3=<n> or b2e_debug_set_att3_variant picks one of the instantiated ones for A/B measurements.
// 65 = four softmax warpgroups (attention5.cuh), fully attended chunks known from attn_prep: same-box A/B of the whole
// step against 5 (two warpgroups + one exponential in four on the FMA pipe): C2 49.58 vs 49.81 ms, C5 100.6 vs 102.5 ms
// (profiles/r02_step_ab_att5.log); both kernels pass the same tests.
constexpr int AT3_DEFAULT_VARIANT = 65;
int g_att3_variant = -1;
inline int att3_variant() {
  if (g_att3_variant < 0) {
    const char* e = getenv("B2E_ATT3");
    g_att3_variant = e ? atoi(e) : AT3_DEFAULT_VARIANT;
  }
  return g_att3_variant;
}

// Token layout of a forward pass (pack.cuh): null pointers = the padded [B, S] layout.
struct SeqLayout {
  const int* cu = nullptr;       // [B + 1]
  const int* len = nullptr;      // [B]
  const int* t_real = nullptr;   // [2]: rows in use, packed flag
  const int* tok_src = nullptr;  // [B * S]
};

template <int V>
int launch_attention_v(const CUtensorMap& tq, const CUtensorMap& tkv, const AttnScratch& sc,
                       const CUtensorMap& tctx, void* ctx, const SeqLayout& lay, int B, int S, int heads,
                       int grid, float scale_log2e, cudaStream_t st, int window = 0) {
  if constexpr ((V & 64) != 0) {   // four softmax warpgroups, chunks split by key columns (attention5.cuh)
    auto kern5 = attention5_d64_kernel<(V & ~64)>;
    constexpr bool epi = (V & 128) != 0;   // + the epilogue warpgroup
    constexpr int smem5 = At5Smem<epi>::BYTES;
    const int arc5 = ensure_smem_attr(kern5, smem5);
    if (arc5) return arc5;
    kern5<<<grid, epi ? AT5_THREADS_EPI : AT5_THREADS, smem5, st>>>(tq, tkv, sc.bias, sc.kv_chunks, sc.plain_chunks, tctx, B, S,
                                                     attn_s_pad(S), heads, scale_log2e, window, lay.cu, lay.len,
                                                     static_cast<h16*>(ctx));
    CUDA_TRY(cudaGetLastError());
    return B2E_OK;
  }
  auto kern = attention3_d64_kernel<V>;
  const int arc = ensure_smem_attr(kern, AT3_SMEM_BYTES);
  if (arc) return arc;
  kern<<<grid, AT3_THREADS, AT3_SMEM_BYTES, st>>>(tq, tkv, sc.bias, sc.kv_chunks, sc.plain_chunks, tctx, B, S,
                                                  attn_s_pad(S), heads, scale_log2e, window, lay.cu, lay.len,
                                                  static_cast<h16*>(ctx));
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

// tq: [T,3H] box 64x128, tkv: [T,3H] box 64x64.  `sc` must have been prepared for this batch's mask.
// window > 0: bidirectional sliding window |q - k| <= window (ModernBERT's local layers), else full attention.
int launch_attention(const CUtensorMap& tq, const CUtensorMap& tkv, const AttnScratch& sc, void* ctx,
                     int B, int S, int heads, int sms, cudaStream_t st, int window = 0,
                     const SeqLayout& lay = SeqLayout()) {
  const float scale_log2e = 0.125f * 1.4426950408889634f;  // 1/sqrt(64) * log2(e)
  const int nq = (S + 127) / 128;
  const long long items = (long long)B * heads * ((nq + 1) / 2);
  const int grid = items < sms ? (int)items : sms;
  CUtensorMap tctx;  // [B*S, H]: full 128-row tiles leave through TMA, a sequence's partial last tile row by row
  int rc;
  if ((rc = make_tmap_h16(&tctx, ctx, (uint64_t)B * S, (uint64_t)heads * AT3_D, 128))) return rc;
  if (window > 0) {
    if ((att3_variant() & 192) == 192)
      return launch_attention_v<192 + 17>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st, window);
    if (att3_variant() & 64)
      return launch_attention_v<64 + 17>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st, window);
    return launch_attention_v<17>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st, window);
  }
  switch (att3_variant()) {
    case 0: return launch_attention_v<0>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 1: return launch_attention_v<1>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 2: return launch_attention_v<2>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 3: return launch_attention_v<3>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 7: return launch_attention_v<7>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 11: return launch_attention_v<11>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 5: return launch_attention_v<5>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 33: return launch_attention_v<33>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 37: return launch_attention_v<37>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 41: return launch_attention_v<41>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 45: return launch_attention_v<45>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 64: return launch_attention_v<64>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 65: return launch_attention_v<65>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 69: return launch_attention_v<69>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 73: return launch_attention_v<73>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 193: return launch_attention_v<193>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
    case 261: return launch_attention_v<261>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);   // 5 + timeline stamps
    case 321: return launch_attention_v<321>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);   // 65 + timeline stamps
    case 197: return launch_attention_v<197>(tq, tkv, sc, tctx, ctx, lay, B, S, heads, grid, scale_log2e, st);
  }
  return fail(B2E_ERR_INVALID, "attention variant %d is not instantiated (0,1,2,3,5,7,11,33,37,41,45,64,65,69,73,193,197,261,321)",
              att3_variant());
}

// Causal grouped-query attention, head_dim 128 (attention4.cuh).  qkv is [B*S, (heads + 2 kv_heads)*128]
// with columns  q heads | k heads | v heads;  sc must have been prepared for (mask, B, S).
int launch_attention_causal_d128(const void* qkv, AttnScratch& sc, void* ctx, int B, int S, int heads,
                                 int kv_heads, int window, int sms, cudaStream_t st,
                                 const SeqLayout& lay = SeqLayout()) {
  {
    const int arc = ensure_smem_attr(attention4_d128_causal_kernel, AT4_SMEM_BYTES);
    if (arc) return arc;
  }
  const uint64_t ld = (uint64_t)(heads + 2 * kv_heads) * AT4_D;
  CUtensorMap tq, tkv, tctx;
  int rc;
  if ((rc = make_tmap_h16(&tq, qkv, (uint64_t)B * S, ld, 128))) return rc;
  if ((rc = make_tmap_h16(&tkv, qkv, (uint64_t)B * S, ld, AT4_KC))) return rc;
  // [B*S, heads*128]: full 128-row tiles leave through TMA, a sequence's partial last tile row by row
  if ((rc = make_tmap_h16(&tctx, ctx, (uint64_t)B * S, (uint64_t)heads * AT4_D, 128))) return rc;
  const int nq = (S + 127) / 128;
  const long long items = (long long)B * heads * ((nq + 1) / 2);
  const int grid = items < sms ? (int)items : sms;
  const float scale_log2e = 0.08838834764831845f * 1.4426950408889634f;  // 128^-0.5 * log2(e)
  attention4_d128_causal_kernel<<<grid, AT4_THREADS, AT4_SMEM_BYTES, st>>>(
      tq, tkv, sc.bias, sc.kv_chunks, sc.plain_chunks, tctx, B, S, attn_s_pad(S), heads, kv_heads, window,
      scale_log2e, lay.cu, lay.len, static_cast<h16*>(ctx));
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

#define DISPATCH_NV(H, CALL)                                        \
  switch ((H) / 256) {                                              \
    case 1: { constexpr int NV = 1; CALL; break; }                  \
    case 2: { constexpr int NV = 2; CALL; break; }                  \
    case 3: { constexpr int NV = 3; CALL; break; }                  \
    case 4: { constexpr int NV = 4; CALL; break; }                  \
    case 5: { constexpr int NV = 5; CALL; break; }                  \
    case 8: { constexpr int NV = 8; CALL; break; }                  \
    case 10: { constexpr int NV = 10; CALL; break; }                \
    case 16: { constexpr int NV = 16; CALL; break; }                \
    default: return fail(B2E_ERR_INVALID, "hidden size %d not supported (need 256*{1,2,3,4,5,8,10,16})", (H)); \
  }

inline int row_blocks(int rows) { return (rows + ROW_WARPS - 1) / ROW_WARPS; }

// The row kernels are instantiated per H/256 (DISPATCH_NV): reject every other width up front, i.e.
// at b2e_encoder_create, before any weight is touched, not at the first forward pass.
int check_h(int H) {
  if (H % 256 != 0) return fail(B2E_ERR_INVALID, "hidden size %d must be a multiple of 256", H);
  switch (H / 256) {
    case 1: case 2: case 3: case 4: case 5: case 8: case 10: case 16: return B2E_OK;
  }
  return fail(B2E_ERR_UNSUPPORTED, "hidden size %d not supported (built: 256 x {1,2,3,4,5,8,10,16})", H);
}

// Pool-weight scratch shared by the fused and the standalone poolers.
struct PoolScratch {
  int* seq_len = nullptr;  // [B]
  int* kill = nullptr;     // [S]
  int* idx = nullptr;      // [B]
  float* w = nullptr;      // [B,S]
  float* count = nullptr;  // [B]
  float* part = nullptr;   // [B,nsplit,H]
  size_t cap_b = 0, cap_s = 0, cap_bs = 0, cap_part = 0;
  int device = -1;
  uint64_t gen = 0;   // bumped on every reallocation (captured CUDA graphs hold these pointers)

  int ensure(int B, int S, size_t part_elems) {
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev != device) {   // buffers of another device: start over on this one
      release();
      device = dev;
      ++gen;
    }
    if ((size_t)B > cap_b || (size_t)S > cap_s || (size_t)B * S > cap_bs || part_elems > cap_part) ++gen;
    // every branch: free, null the pointers and zero the capacity, THEN allocate (a failed cudaMalloc
    // leaves "nothing allocated", never a dangling pointer that a smaller later call would reuse)
    if ((size_t)B > cap_b) {
      cudaFree(seq_len); cudaFree(idx); cudaFree(count);
      seq_len = idx = nullptr;
      count = nullptr;
      cap_b = 0;
      CUDA_TRY(cudaMalloc(&seq_len, sizeof(int) * B));
      CUDA_TRY(cudaMalloc(&idx, sizeof(int) * B));
      CUDA_TRY(cudaMalloc(&count, sizeof(float) * B));
      cap_b = B;
    }
    if ((size_t)S > cap_s) {
      cudaFree(kill);
      kill = nullptr;
      cap_s = 0;
      CUDA_TRY(cudaMalloc(&kill, sizeof(int) * S));
      cap_s = S;
    }
    if ((size_t)B * S > cap_bs) {
      cudaFree(w);
      w = nullptr;
      cap_bs = 0;
      CUDA_TRY(cudaMalloc(&w, sizeof(float) * (size_t)B * S));
      cap_bs = (size_t)B * S;
    }
    if (part_elems > cap_part) {
      cudaFree(part);
      part = nullptr;
      cap_part = 0;
      CUDA_TRY(cudaMalloc(&part, sizeof(float) * part_elems));
      cap_part = part_elems;
    }
    return B2E_OK;
  }
  void release() {
    cudaFree(seq_len); cudaFree(kill); cudaFree(idx); cudaFree(w); cudaFree(count); cudaFree(part);
    seq_len = kill = idx = nullptr; w = count = part = nullptr;
    cap_b = cap_s = cap_bs = cap_part = 0;
  }
};

inline int pool_nsplit(int S) {
  int n = (S + 63) / 64;  // ~64 rows per block keeps every SM busy at B >= 32
  return n < 1 ? 1 : (n > 16 ? 16 : n);
}

int launch_pool_weights(PoolScratch& ps, int64_t* mask, int B, int S, int pool_kind, int mutate,
                        cudaStream_t st) {
  seq_len_kernel<<<(B + 7) / 8, 256, 0, st>>>(mask, ps.seq_len, B, S);
  CUDA_TRY(cudaMemsetAsync(ps.kill, 0, sizeof(int) * S, st));
  kill_columns_kernel<<<(B + 255) / 256, 256, 0, st>>>(ps.seq_len, ps.kill, B, S);
  pool_weights_kernel<<<(B + 7) / 8, 256, 0, st>>>(mask, ps.seq_len, ps.kill, ps.w, ps.count, B, S,
                                                    pool_kind == B2E_POOL_MEAN_REF ? 1 : 0, mutate);
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

int launch_finalize(PoolScratch& ps, float* out, int B, int H, int nsplit, int l2, int round_mode,
                    cudaStream_t st) {
  pool_finalize_kernel<<<B, 256, (H + 32) * sizeof(float), st>>>(ps.part, ps.count, out, H, nsplit,
                                                                 l2, round_mode);
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

// Restores the caller's current device on scope exit: create / destroy / embed_host switch to the
// encoder's device and must not leave torch's notion of the current device changed behind its back.
struct DeviceGuard {
  int prev = -1;
  DeviceGuard() {
    if (cudaGetDevice(&prev) != cudaSuccess) {
      cudaGetLastError();
      prev = -1;
    }
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

thread_local PoolScratch g_pool_scratch;  // for the handle-less standalone poolers
thread_local AttnScratch g_attn_scratch;  // for the standalone attention op

}  // namespace

// ================================================================== encoder handle
struct B2EEncoder {
  B2EModelDesc desc;
  int full_layers = 0;   // desc.num_layers as created (b2e_debug_set_layers may lower desc.num_layers)
  std::vector<const void*> w;
  int device = 0;
  int sms = 0;
  // activations (h16)
  size_t cap_tokens = 0;
  h16 *hidden = nullptr, *qkv = nullptr, *ctx = nullptr, *tmp = nullptr, *ffn = nullptr;
  PoolScratch pool;
  AttnScratch attn;
  // padding-free token layout of the pooled forward pass (pack.cuh)
  int *pk_len_raw = nullptr, *pk_ok = nullptr, *pk_len = nullptr, *pk_cu = nullptr, *pk_treal = nullptr,
      *pk_src = nullptr;
  size_t pk_cap_b = 0, pk_cap_t = 0;
  // weight tensor maps, one per layer
  std::vector<CUtensorMap> tm_wqkv, tm_wo, tm_w1, tm_w2;
  // host-loop staging
  int64_t* stage_in = nullptr;
  size_t stage_cap = 0;
  float* stage_out = nullptr;
  size_t stage_out_cap = 0;
  cudaStream_t own_stream = nullptr;

  // BERT weight slots
  const float* word() const { return (const float*)w[0]; }
  const float* pos() const { return (const float*)w[1]; }
  const float* type() const { return (const float*)w[2]; }
  const float* emb_g() const { return (const float*)w[3]; }
  const float* emb_b() const { return (const float*)w[4]; }
  const void* L(int l, int k) const { return w[5 + 12 * l + k]; }

  // ESM-2: fp32 residual stream, token-dropout scales, rotary tables; weight slots (weights.py):
  //   0 word emb, 1/2 final LayerNorm; per layer (3 + 12 l): ln1 g/b, Wqkv, bqkv, Wo, bo, ln2 g/b,
  //   W1, b1, W2, b2
  float* xres = nullptr;
  float* tok_scale = nullptr;
  size_t cap_scale = 0;
  float *rope_cos = nullptr, *rope_sin = nullptr;
  const void* E(int l, int k) const { return w[3 + 12 * l + k]; }

  // Mistral family: fp32 residual stream and rotary tables as above; weight slots (weights.py):
  //   0 embed_tokens, 1 final norm; per layer (2 + 6 l): input norm, Wqkv, Wo, post-attention norm,
  //   Wgu (gate/up interleaved), Wd
  const void* Mi(int l, int k) const { return w[2 + 6 * l + k]; }
  // ModernBERT: weight slots (weights.py): 0 tok_embeddings, 1/2 embeddings.norm g/b, 3/4 final_norm g/b; per
  // layer (5 + 8 l): attn_norm g/b, Wqkv, Wo, mlp_norm g/b, Wi (input/gate interleaved), mlp.Wo.  rope_cos/sin =
  // full-attention layers' table, rope_cos2/sin2 = sliding-attention layers'
  const void* Mb(int l, int k) const { return w[5 + 8 * l + k]; }
  float *rope_cos2 = nullptr, *rope_sin2 = nullptr;
  // b2e_embed_host replays one CUDA graph per (batch shape, pooling, staging slot) instead of ~90
  // launches per batch; every graph is dropped when a buffer it points into is reallocated
  struct StepGraph {
    int B, S, pool_kind, l2, has_types, slot;
    cudaGraphExec_t exec;
  };
  std::vector<StepGraph> graphs;
  uint64_t ws_gen = 0;        // bumped when the workspace or a staging buffer is reallocated
  uint64_t graphs_stamp = 0;  // buffer_stamp() at the time the cached graphs were captured
  uint64_t buffer_stamp() const { return ws_gen + pool.gen + attn.gen; }
  void drop_graphs() {
    for (auto& g : graphs) cudaGraphExecDestroy(g.exec);
    graphs.clear();
  }

  int qkv_cols() const {
    return desc.arch == B2E_ARCH_MISTRAL ? (desc.heads + 2 * desc.kv_heads) * desc.head_dim
                                         : 3 * desc.hidden;
  }
  int ctx_cols() const {
    return desc.arch == B2E_ARCH_MISTRAL ? desc.heads * desc.head_dim : desc.hidden;
  }
  bool has_xres() const { return desc.arch != B2E_ARCH_BERT; }
};

namespace {

size_t tokens_bytes(const B2EModelDesc& d, size_t tokens) {
  if (d.arch == B2E_ARCH_MISTRAL)
    return tokens * (size_t)(2 * d.hidden + (2 * d.heads + 2 * d.kv_heads) * d.head_dim + d.intermediate) * 2;
  return tokens * (size_t)(6 * d.hidden + d.intermediate) * 2;
}

int ensure_workspace(B2EEncoder* e, int B, int S) {
  const size_t tokens = (size_t)B * S;
  if (tokens > e->cap_tokens) {
    ++e->ws_gen;
    cudaFree(e->hidden); cudaFree(e->qkv); cudaFree(e->ctx); cudaFree(e->tmp); cudaFree(e->ffn);
    e->hidden = e->qkv = e->ctx = e->tmp = e->ffn = nullptr;
    e->cap_tokens = 0;
    const size_t H = e->desc.hidden, I = e->desc.intermediate;
    CUDA_TRY(cudaMalloc(&e->hidden, tokens * H * 2));
    CUDA_TRY(cudaMalloc(&e->qkv, tokens * (size_t)e->qkv_cols() * 2));
    CUDA_TRY(cudaMalloc(&e->ctx, tokens * (size_t)e->ctx_cols() * 2));
    CUDA_TRY(cudaMalloc(&e->tmp, tokens * H * 2));
    CUDA_TRY(cudaMalloc(&e->ffn, tokens * I * 2));
    // zeroed once: with the packed token layout rows behind the last attended token are never written by a
    // forward pass but ARE read (partial GEMM tiles, the last key chunk of the last sequence) -- they must
    // hold finite values, never whatever the allocator left there
    CUDA_TRY(cudaMemset(e->hidden, 0, tokens * H * 2));
    CUDA_TRY(cudaMemset(e->qkv, 0, tokens * (size_t)e->qkv_cols() * 2));
    CUDA_TRY(cudaMemset(e->ctx, 0, tokens * (size_t)e->ctx_cols() * 2));
    CUDA_TRY(cudaMemset(e->tmp, 0, tokens * H * 2));
    CUDA_TRY(cudaMemset(e->ffn, 0, tokens * I * 2));
    if (e->has_xres()) {
      cudaFree(e->xres);
      e->xres = nullptr;
      CUDA_TRY(cudaMalloc(&e->xres, tokens * H * 4));
      CUDA_TRY(cudaMemset(e->xres, 0, tokens * H * 4));
    }
    e->cap_tokens = tokens;
  }
  if (e->desc.arch == B2E_ARCH_ESM2 && (size_t)B > e->cap_scale) {
    ++e->ws_gen;
    cudaFree(e->tok_scale);
    e->tok_scale = nullptr;
    e->cap_scale = 0;
    CUDA_TRY(cudaMalloc(&e->tok_scale, sizeof(float) * B));
    e->cap_scale = B;
  }
  if ((size_t)B > e->pk_cap_b) {
    ++e->ws_gen;
    cudaFree(e->pk_len_raw); cudaFree(e->pk_ok); cudaFree(e->pk_len); cudaFree(e->pk_cu); cudaFree(e->pk_treal);
    e->pk_len_raw = e->pk_ok = e->pk_len = e->pk_cu = e->pk_treal = nullptr;
    e->pk_cap_b = 0;
    CUDA_TRY(cudaMalloc(&e->pk_len_raw, sizeof(int) * B));
    CUDA_TRY(cudaMalloc(&e->pk_ok, sizeof(int) * B));
    CUDA_TRY(cudaMalloc(&e->pk_len, sizeof(int) * B));
    CUDA_TRY(cudaMalloc(&e->pk_cu, sizeof(int) * (B + 1)));
    CUDA_TRY(cudaMalloc(&e->pk_treal, sizeof(int) * 2));
    e->pk_cap_b = B;
  }
  if (tokens > e->pk_cap_t) {
    ++e->ws_gen;
    cudaFree(e->pk_src);
    e->pk_src = nullptr;
    e->pk_cap_t = 0;
    CUDA_TRY(cudaMalloc(&e->pk_src, sizeof(int) * tokens));
    e->pk_cap_t = tokens;
  }
  return e->pool.ensure(B, S, (size_t)B * pool_nsplit(S) * e->desc.hidden);
}

// B2E_PACKED=0 keeps the padded [B, S] layout on every path (A/B measurements, debugging)
int g_packing = -1;   // -1: not decided yet (B2E_PACKED), 0 / 1: b2e_debug_set_packing or the environment
inline bool packing_enabled() {
  if (g_packing < 0) {
    const char* e = getenv("B2E_PACKED");
    g_packing = (e && e[0] == '0') ? 0 : 1;
  }
  return g_packing == 1;
}

// Token layout of this forward pass (pack.cuh), decided and built ON DEVICE from the mask: attended tokens
// back to back when every mask row is a non-empty prefix and `enable`, else the identity ([B, S]) layout
// expressed through the same descriptors.
int pack_prepare(B2EEncoder* e, const int64_t* mask, int B, int S, bool enable, cudaStream_t st, SeqLayout* lay) {
  pack_lengths_kernel<<<(B + 7) / 8, 256, 0, st>>>(mask, e->pk_len_raw, e->pk_ok, B, S);
  pack_scan_kernel<<<1, 256, 0, st>>>(e->pk_len_raw, e->pk_ok, e->pk_len, e->pk_cu, e->pk_treal, B, S,
                                      enable ? 1 : 0);
  pack_fill_kernel<<<dim3((S + 255) / 256, B), 256, 0, st>>>(e->pk_len, e->pk_cu, e->pk_src, B, S);
  CUDA_TRY(cudaGetLastError());
  lay->cu = e->pk_cu;
  lay->len = e->pk_len;
  lay->t_real = e->pk_treal;
  lay->tok_src = e->pk_src;
  return B2E_OK;
}

int validate_batch(const B2EEncoder* e, int B, int S) {
  if (!e) return fail(B2E_ERR_INVALID, "null encoder handle");
  if (B <= 0 || S <= 0) return fail(B2E_ERR_INVALID, "empty batch B=%d S=%d", B, S);
  int cur = -1;
  if (cudaGetDevice(&cur) == cudaSuccess && cur != e->device)
    return fail(B2E_ERR_INVALID, "encoder lives on device %d but device %d is current", e->device, cur);
  if (S > e->desc.max_pos)
    return fail(B2E_ERR_INVALID, "S=%d exceeds max_position_embeddings=%d", S, e->desc.max_pos);
  return B2E_OK;
}

// Layers 0..L-1 up to (and including) the last FFN-down GEMM: leaves the pre-LayerNorm residual sum
// of the final layer split as e->tmp (FFN-down output + bias) and e->hidden (the residual it still has
// to be added to); every earlier LayerNorm output lives in e->hidden.
int run_bert_trunk(B2EEncoder* e, const int64_t* ids, const int64_t* mask, const int64_t* types,
                   int B, int S, cudaStream_t st,
                   const SeqLayout& lay = SeqLayout()) {
  const B2EModelDesc& d = e->desc;
  const int M = B * S, H = d.hidden, I = d.intermediate;
  int rc;
  DISPATCH_NV(H, (embed_layernorm_kernel<NV><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                     ids, types, e->word(), e->pos(), e->type(), e->emb_g(), e->emb_b(), e->hidden,
                     M, S, d.eps, lay.t_real, lay.tok_src)));
  CUDA_TRY(cudaGetLastError());

  if ((rc = attention_prepare(e->attn, mask, B, S, st))) return rc;
  CUtensorMap tm_hidden, tm_ctx, tm_ffn, tm_qkv, tm_kv64;
  if ((rc = make_tmap_h16(&tm_kv64, e->qkv, M, 3 * H, AT3_KC))) return rc;
  if ((rc = make_tmap_h16(&tm_hidden, e->hidden, M, H, 128))) return rc;
  if ((rc = make_tmap_h16(&tm_ctx, e->ctx, M, H, 128))) return rc;
  if ((rc = make_tmap_h16(&tm_ffn, e->ffn, M, I, 128))) return rc;
  if ((rc = make_tmap_h16(&tm_qkv, e->qkv, M, 3 * H, 128))) return rc;

  for (int l = 0; l < d.num_layers; ++l) {
    if ((rc = launch_gemm(tm_hidden, e->tm_wqkv[l], e->qkv, (const float*)e->L(l, 1), nullptr, M,
                          3 * H, H, B2E_EPI_BIAS, e->sms, st, lay.t_real)))
      return rc;
    if ((rc = launch_attention(tm_qkv, tm_kv64, e->attn, e->ctx, B, S, d.heads, e->sms, st, 0, lay)))
      return rc;
    // the residual add rides on the LayerNorm's coalesced reads, not on the GEMM epilogue
    if ((rc = launch_gemm(tm_ctx, e->tm_wo[l], e->tmp, (const float*)e->L(l, 3), nullptr, M, H, H,
                          B2E_EPI_BIAS, e->sms, st, lay.t_real)))
      return rc;
    DISPATCH_NV(H, (layernorm_kernel<NV, h16><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                       e->tmp, e->hidden, (const float*)e->L(l, 4), (const float*)e->L(l, 5),
                       e->hidden, M, d.eps, lay.t_real)));
    if ((rc = launch_gemm(tm_hidden, e->tm_w1[l], e->ffn, (const float*)e->L(l, 7), nullptr, M, I,
                          H, B2E_EPI_BIAS_GELU, e->sms, st, lay.t_real)))
      return rc;
    if ((rc = launch_gemm(tm_ffn, e->tm_w2[l], e->tmp, (const float*)e->L(l, 9), nullptr, M, H, I,
                          B2E_EPI_BIAS, e->sms, st, lay.t_real)))
      return rc;
    if (l + 1 < d.num_layers) {
      DISPATCH_NV(H, (layernorm_kernel<NV, h16><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                         e->tmp, e->hidden, (const float*)e->L(l, 10), (const float*)e->L(l, 11),
                         e->hidden, M, d.eps, lay.t_real)));
    }
  }
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

// ESM-2 (pre-LayerNorm, rotary): transformers/models/esm/modeling_esm.py:189-234 (embeddings with
// token dropout), :318-362 (attention, rotary on q/k), :386-404 / :446-483 (pre-LN blocks).  The
// residual stream e->xres stays fp32; each add_layernorm call folds the previous GEMM output into it
// and emits the next GEMM's h16 input.  Leaves xres (before the last FFN output is added) and e->tmp
// (that FFN-down output): the caller applies emb_layer_norm_after to xres + tmp.
int run_esm_trunk(B2EEncoder* e, const int64_t* ids, const int64_t* mask, int B, int S,
                  cudaStream_t st, const SeqLayout& lay = SeqLayout()) {
  const B2EModelDesc& d = e->desc;
  const int M = B * S, H = d.hidden, I = d.intermediate, L = d.num_layers;
  const int mask_token = d.reserved - 1;  // reserved = mask_token_id + 1, 0 = token dropout off
  int rc;
  esm_token_scale_kernel<<<(B + 7) / 8, 256, 0, st>>>(ids, mask, e->tok_scale, B, S, mask_token);
  DISPATCH_NV(H, (esm_embed_kernel<NV><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                     ids, mask, (const float*)e->w[0], e->tok_scale, e->xres, M, S, mask_token, lay.t_real,
                     lay.tok_src)));
  CUDA_TRY(cudaGetLastError());
  if ((rc = attention_prepare(e->attn, mask, B, S, st))) return rc;
  CUtensorMap tm_hidden, tm_ctx, tm_ffn, tm_qkv, tm_kv64;
  if ((rc = make_tmap_h16(&tm_hidden, e->hidden, M, H, 128))) return rc;
  if ((rc = make_tmap_h16(&tm_ctx, e->ctx, M, H, 128))) return rc;
  if ((rc = make_tmap_h16(&tm_ffn, e->ffn, M, I, 128))) return rc;
  if ((rc = make_tmap_h16(&tm_qkv, e->qkv, M, 3 * H, 128))) return rc;
  if ((rc = make_tmap_h16(&tm_kv64, e->qkv, M, 3 * H, AT3_KC))) return rc;

  DISPATCH_NV(H, (add_layernorm_kernel<NV, h16><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                     e->xres, nullptr, (const float*)e->E(0, 0), (const float*)e->E(0, 1), e->hidden,
                     M, d.eps, lay.t_real)));
  const long long rope_work = (long long)M * d.heads * 2;
  for (int l = 0; l < L; ++l) {
    if ((rc = launch_gemm(tm_hidden, e->tm_wqkv[l], e->qkv, (const float*)e->E(l, 3), nullptr, M,
                          3 * H, H, B2E_EPI_BIAS, e->sms, st, lay.t_real)))
      return rc;
    rope_halves_kernel<32><<<(unsigned)((rope_work * 4 + 255) / 256), 256, 0, st>>>(
        e->qkv, e->rope_cos, e->rope_sin, M, S, 2 * d.heads, 3 * H, lay.t_real, lay.tok_src);
    if ((rc = launch_attention(tm_qkv, tm_kv64, e->attn, e->ctx, B, S, d.heads, e->sms, st, 0, lay)))
      return rc;
    if ((rc = launch_gemm(tm_ctx, e->tm_wo[l], e->tmp, (const float*)e->E(l, 5), nullptr, M, H, H,
                          B2E_EPI_BIAS, e->sms, st, lay.t_real)))
      return rc;
    DISPATCH_NV(H, (add_layernorm_kernel<NV, h16><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                       e->xres, e->tmp, (const float*)e->E(l, 6), (const float*)e->E(l, 7), e->hidden,
                       M, d.eps, lay.t_real)));
    if ((rc = launch_gemm(tm_hidden, e->tm_w1[l], e->ffn, (const float*)e->E(l, 9), nullptr, M, I, H,
                          B2E_EPI_BIAS_GELU, e->sms, st, lay.t_real)))
      return rc;
    if ((rc = launch_gemm(tm_ffn, e->tm_w2[l], e->tmp, (const float*)e->E(l, 11), nullptr, M, H, I,
                          B2E_EPI_BIAS, e->sms, st, lay.t_real)))
      return rc;
    if (l + 1 < L) {
      DISPATCH_NV(H, (add_layernorm_kernel<NV, h16><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                         e->xres, e->tmp, (const float*)e->E(l + 1, 0), (const float*)e->E(l + 1, 1),
                         e->hidden, M, d.eps, lay.t_real)));
    }
  }
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

// Mistral family (pre-RMSNorm decoder blocks, rotary, grouped-query causal attention, SwiGLU):
// transformers/models/mistral/modeling_mistral.py:328-400 (model), :202-242 (block), :122-180
// (attention), :35-48 (MLP).  Like the ESM-2 trunk it leaves xres (before the last MLP output is
// added) and e->tmp (that down_proj output); the caller applies the final norm to xres + tmp.
int run_mistral_trunk(B2EEncoder* e, const int64_t* ids, const int64_t* mask, int B, int S,
                      cudaStream_t st, const SeqLayout& lay = SeqLayout()) {
  const B2EModelDesc& d = e->desc;
  const int M = B * S, H = d.hidden, I = d.intermediate, L = d.num_layers;
  const int QC = e->qkv_cols(), CC = e->ctx_cols();
  int rc;
  DISPATCH_NV(H, (mistral_embed_kernel<NV><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                     ids, (const float*)e->w[0], e->xres, M, lay.t_real, lay.tok_src)));
  CUDA_TRY(cudaGetLastError());
  if ((rc = attention_prepare(e->attn, mask, B, S, st))) return rc;
  CUtensorMap tm_hidden, tm_ctx, tm_ffn;
  if ((rc = make_tmap_h16(&tm_hidden, e->hidden, M, H, 128))) return rc;
  if ((rc = make_tmap_h16(&tm_ctx, e->ctx, M, CC, 128))) return rc;
  if ((rc = make_tmap_h16(&tm_ffn, e->ffn, M, I, 128))) return rc;

  DISPATCH_NV(H, (add_rmsnorm_kernel<NV, h16><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                     e->xres, nullptr, (const float*)e->Mi(0, 0), e->hidden, M, d.eps, lay.t_real)));
  const int n_rot = d.heads + d.kv_heads;   // q heads and k heads are adjacent columns of qkv
  const long long rope_work = (long long)M * n_rot;
  for (int l = 0; l < L; ++l) {
    if ((rc = launch_gemm(tm_hidden, e->tm_wqkv[l], e->qkv, nullptr, nullptr, M, QC, H, B2E_EPI_BIAS,
                          e->sms, st, lay.t_real)))
      return rc;
    rope_halves_kernel<64><<<(unsigned)((rope_work * 8 + 255) / 256), 256, 0, st>>>(
        e->qkv, e->rope_cos, e->rope_sin, M, S, n_rot, QC, lay.t_real, lay.tok_src);
    if ((rc = launch_attention_causal_d128(e->qkv, e->attn, e->ctx, B, S, d.heads, d.kv_heads,
                                           d.sliding_window, e->sms, st, lay)))
      return rc;
    if ((rc = launch_gemm(tm_ctx, e->tm_wo[l], e->tmp, nullptr, nullptr, M, H, CC, B2E_EPI_BIAS,
                          e->sms, st, lay.t_real)))
      return rc;
    DISPATCH_NV(H, (add_rmsnorm_kernel<NV, h16><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                       e->xres, e->tmp, (const float*)e->Mi(l, 3), e->hidden, M, d.eps, lay.t_real)));
    // gate and up in one GEMM (interleaved rows), silu(gate) * up in its epilogue: [M, I]
    if ((rc = launch_gemm(tm_hidden, e->tm_w1[l], e->ffn, nullptr, nullptr, M, 2 * I, H,
                          B2E_EPI_SWIGLU, e->sms, st, lay.t_real)))
      return rc;
    if ((rc = launch_gemm(tm_ffn, e->tm_w2[l], e->tmp, nullptr, nullptr, M, H, I, B2E_EPI_BIAS,
                          e->sms, st, lay.t_real)))
      return rc;
    if (l + 1 < L) {
      DISPATCH_NV(H, (add_rmsnorm_kernel<NV, h16><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                         e->xres, e->tmp, (const float*)e->Mi(l + 1, 0), e->hidden, M, d.eps, lay.t_real)));
    }
  }
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

// ModernBERT (pre-LayerNorm blocks, rotary with one base per layer type, alternating full / sliding-window
// bidirectional attention, GeGLU MLP, no Linear biases): transformers/models/modernbert/modeling_modernbert.py
// :52-71 (embeddings), :232-310 (attention), :74-91 (MLP), :313-343 (block; layer 0 has no attn_norm),
// :424-490 (model).  Leaves xres (before the last MLP output is added) and e->tmp (that output): the caller
// applies final_norm to xres + tmp.
int run_modernbert_trunk(B2EEncoder* e, const int64_t* ids, const int64_t* mask, int B, int S,
                         cudaStream_t st, const SeqLayout& lay = SeqLayout()) {
  const B2EModelDesc& d = e->desc;
  const int M = B * S, H = d.hidden, I = d.intermediate, L = d.num_layers;
  int rc;
  DISPATCH_NV(H, (modernbert_embed_kernel<NV><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                     ids, (const float*)e->w[0], (const float*)e->w[1], (const float*)e->w[2], e->xres,
                     e->hidden, M, d.eps, lay.t_real, lay.tok_src)));
  CUDA_TRY(cudaGetLastError());
  if ((rc = attention_prepare(e->attn, mask, B, S, st))) return rc;
  CUtensorMap tm_hidden, tm_ctx, tm_ffn, tm_qkv, tm_kv64;
  if ((rc = make_tmap_h16(&tm_hidden, e->hidden, M, H, 128))) return rc;
  if ((rc = make_tmap_h16(&tm_ctx, e->ctx, M, H, 128))) return rc;
  if ((rc = make_tmap_h16(&tm_ffn, e->ffn, M, I, 128))) return rc;
  if ((rc = make_tmap_h16(&tm_qkv, e->qkv, M, 3 * H, 128))) return rc;
  if ((rc = make_tmap_h16(&tm_kv64, e->qkv, M, 3 * H, AT3_KC))) return rc;
  const long long rope_work = (long long)M * d.heads * 2;
  for (int l = 0; l < L; ++l) {
    const bool global = (l % d.global_every) == 0;
    if (l > 0) {
      DISPATCH_NV(H, (add_layernorm_kernel<NV, h16><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                         e->xres, e->tmp, (const float*)e->Mb(l, 0), (const float*)e->Mb(l, 1), e->hidden, M,
                         d.eps, lay.t_real)));
    }
    if ((rc = launch_gemm(tm_hidden, e->tm_wqkv[l], e->qkv, nullptr, nullptr, M, 3 * H, H, B2E_EPI_BIAS,
                          e->sms, st, lay.t_real)))
      return rc;
    rope_halves_kernel<32><<<(unsigned)((rope_work * 4 + 255) / 256), 256, 0, st>>>(
        e->qkv, global ? e->rope_cos : e->rope_cos2, global ? e->rope_sin : e->rope_sin2, M, S, 2 * d.heads,
        3 * H, lay.t_real, lay.tok_src);
    if ((rc = launch_attention(tm_qkv, tm_kv64, e->attn, e->ctx, B, S, d.heads, e->sms, st,
                               global ? 0 : d.sliding_window, lay)))
      return rc;
    if ((rc = launch_gemm(tm_ctx, e->tm_wo[l], e->tmp, nullptr, nullptr, M, H, H, B2E_EPI_BIAS, e->sms, st, lay.t_real)))
      return rc;
    DISPATCH_NV(H, (add_layernorm_kernel<NV, h16><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                       e->xres, e->tmp, (const float*)e->Mb(l, 4), (const float*)e->Mb(l, 5), e->hidden, M,
                       d.eps, lay.t_real)));
    // Wi with its input / gate halves interleaved: gelu(input) * gate in the epilogue -> [M, I]
    if ((rc = launch_gemm(tm_hidden, e->tm_w1[l], e->ffn, nullptr, nullptr, M, 2 * I, H, B2E_EPI_GEGLU,
                          e->sms, st, lay.t_real)))
      return rc;
    if ((rc = launch_gemm(tm_ffn, e->tm_w2[l], e->tmp, nullptr, nullptr, M, H, I, B2E_EPI_BIAS, e->sms, st, lay.t_real)))
      return rc;
  }
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

}  // namespace

// ================================================================== C ABI
extern "C" {

int b2e_version(void) { return B2E_ABI_VERSION; }
int b2e_storage_dtype(void) { return kStorageDtype; }

// Profiling hooks (include/b2e_debug.h, not part of the reference-facing ABI): device buffer of
// 4 x 256 int64 that CTAs 0 and 1 of the CTA-pair GEMM fill with clock64() stamps ([cta*2 + role][n],
// role 0 = producer, 1 = MMA).  Same idea for the streaming attention kernel: 3 roles x (256 clocks +
// 256 event codes) int64.
int b2e_debug_set_att3_clock(void* device_buffer) {
  long long* p = static_cast<long long*>(device_buffer);
  CUDA_TRY(cudaMemcpyToSymbol(g_att3_clock, &p, sizeof(p)));
  return B2E_OK;
}

int b2e_debug_set_att3_flags(int flags) {
  CUDA_TRY(cudaMemcpyToSymbol(g_att3_flags, &flags, sizeof(flags)));
  return B2E_OK;
}

// 0: every forward pass keeps the padded [B, S] token layout; 1: pooled passes pack attended tokens (default)
int b2e_debug_set_packing(int on) {
  g_packing = on ? 1 : 0;
  return B2E_OK;
}

int b2e_debug_set_att3_variant(int variant) {
  g_att3_variant = variant;
  return B2E_OK;
}

// Experiment knob for the CTA-pair GEMM: bit 0 = skip the epilogue's math and stores.
int b2e_debug_set_pair_flags(int flags) {
  g_gemm2_profiling = flags != 0;
  CUDA_TRY(cudaMemcpyToSymbol(g_gemm2_flags, &flags, sizeof(flags)));
  return B2E_OK;
}

int b2e_debug_set_clock_buffer(void* device_buffer) {
  long long* p = static_cast<long long*>(device_buffer);
  g_gemm2_profiling = p != nullptr;
  CUDA_TRY(cudaMemcpyToSymbol(g_gemm2_clock, &p, sizeof(p)));
  return B2E_OK;
}
// Run only the first n layers from now on (1 <= n <= the model's depth; 0 restores the full depth).  The
// output is what a checkpoint truncated to n layers would give: BERT's hidden_states[n]; for the pre-norm
// families the final norm applied to the residual stream after n layers.  Used by tools/drift_report.py.
int b2e_debug_set_layers(B2EEncoder* e, int n) {
  if (!e) return fail(B2E_ERR_INVALID, "null encoder handle");
  if (n == 0) n = e->full_layers;
  if (n < 1 || n > e->full_layers)
    return fail(B2E_ERR_INVALID, "layer count %d outside [1, %d]", n, e->full_layers);
  if (n != e->desc.num_layers) e->drop_graphs();
  e->desc.num_layers = n;
  return B2E_OK;
}
const char* b2e_last_error(void) { return g_err.c_str(); }

int b2e_num_weights(const B2EModelDesc* desc) {
  if (!desc) return -1;
  if (desc->arch == B2E_ARCH_BERT) return 5 + 12 * desc->num_layers;
  if (desc->arch == B2E_ARCH_ESM2) return 3 + 12 * desc->num_layers;
  if (desc->arch == B2E_ARCH_MISTRAL) return 2 + 6 * desc->num_layers;
  if (desc->arch == B2E_ARCH_MODERNBERT) return 5 + 8 * desc->num_layers;
  return -1;
}

// Everything b2e_encoder_create would reject about the SHAPE of a model, without touching a device or
// a weight: callers run it before they upload gigabytes of parameters.
int b2e_check_model(const B2EModelDesc* desc) {
  if (!desc) return fail(B2E_ERR_INVALID, "null model description");
  if (desc->num_layers <= 0 || desc->hidden <= 0 || desc->heads <= 0 || desc->intermediate <= 0)
    return fail(B2E_ERR_INVALID, "model description has a non-positive size");
  int rc;
  if (desc->arch == B2E_ARCH_MISTRAL) {
    if (desc->head_dim != 128 || desc->kv_heads <= 0 || desc->heads % desc->kv_heads != 0)
      return fail(B2E_ERR_UNSUPPORTED, "need head_dim 128 and heads %% kv_heads == 0 (got %d/%d x %d)",
                  desc->heads, desc->kv_heads, desc->head_dim);
    if (desc->intermediate % 128 != 0)
      return fail(B2E_ERR_UNSUPPORTED, "intermediate size %d must be a multiple of 128", desc->intermediate);
    if (desc->sliding_window < 0) return fail(B2E_ERR_INVALID, "negative sliding_window");
    const int H = desc->hidden, I = desc->intermediate;
    const int QC = (desc->heads + 2 * desc->kv_heads) * 128, CC = desc->heads * 128;
    if ((rc = check_h(H))) return rc;
    if ((rc = check_gemm_shape(128, QC, H))) return rc;
    if ((rc = check_gemm_shape(128, H, CC))) return rc;
    if ((rc = check_gemm_shape(128, 2 * I, H))) return rc;
    return check_gemm_shape(128, H, I);
  }
  if (desc->arch != B2E_ARCH_BERT && desc->arch != B2E_ARCH_ESM2 && desc->arch != B2E_ARCH_MODERNBERT)
    return fail(B2E_ERR_UNSUPPORTED, "arch %d: unknown architecture", desc->arch);
  if (desc->arch == B2E_ARCH_MODERNBERT) {
    if (desc->global_every <= 0) return fail(B2E_ERR_INVALID, "ModernBERT: global_every must be positive");
    if (desc->sliding_window <= 0) return fail(B2E_ERR_INVALID, "ModernBERT: sliding_window must be positive");
    if ((2 * desc->intermediate) % 256 != 0)
      return fail(B2E_ERR_UNSUPPORTED, "ModernBERT: 2 * intermediate_size = %d must be a multiple of 256 (the gated "
                  "epilogue pairs 128 input with 128 gate columns)", 2 * desc->intermediate);
  }
  if (desc->head_dim != 64 || desc->heads * desc->head_dim != desc->hidden)
    return fail(B2E_ERR_UNSUPPORTED,
                "need head_dim 64 and heads*64 == hidden (got %d heads x %d, H=%d); of the ESM-2 family that "
                "is esm2_t33_650M (H=1280) and esm2_t36_3B (H=2560)",
                desc->heads, desc->head_dim, desc->hidden);
  if ((rc = check_h(desc->hidden))) return rc;
  if ((rc = check_gemm_shape(128, 3 * desc->hidden, desc->hidden))) return rc;
  if ((rc = check_gemm_shape(128, desc->intermediate, desc->hidden))) return rc;
  return check_gemm_shape(128, desc->hidden, desc->intermediate);
}

namespace {
// Mistral family: head_dim 128, grouped-query heads, SwiGLU MLP, no biases.
int create_mistral(const B2EModelDesc* desc, const void* const* weights, int n_weights, int device,
                   B2EEncoder** out) {
  const int L = desc->num_layers, H = desc->hidden, I = desc->intermediate;
  const int QC = (desc->heads + 2 * desc->kv_heads) * 128, CC = desc->heads * 128;
  int rc;
  if ((rc = b2e_check_model(desc))) return rc;
  if (n_weights != b2e_num_weights(desc))
    return fail(B2E_ERR_INVALID, "expected %d weight pointers, got %d", b2e_num_weights(desc), n_weights);
  for (int i = 0; i < n_weights; ++i)
    if (!weights[i]) return fail(B2E_ERR_INVALID, "weight pointer %d is null", i);
  DeviceInfo info;
  if ((rc = device_info(device, &info))) return rc;
  DeviceGuard guard;
  CUDA_TRY(cudaSetDevice(device));
  B2EEncoder* e = new B2EEncoder();
  e->desc = *desc;
  e->full_layers = desc->num_layers;
  e->w.assign(weights, weights + n_weights);
  e->device = device;
  e->sms = info.sms;
  e->tm_wqkv.resize(L); e->tm_wo.resize(L); e->tm_w1.resize(L); e->tm_w2.resize(L);
  for (int l = 0; l < L; ++l) {
    if ((rc = make_tmap_h16(&e->tm_wqkv[l], e->Mi(l, 1), QC, H, gemm_bn_for(QC))) ||
        (rc = make_tmap_h16(&e->tm_wo[l], e->Mi(l, 2), H, CC, gemm_bn_for(H))) ||
        (rc = make_tmap_h16(&e->tm_w1[l], e->Mi(l, 4), 2 * I, H, gemm_bn_for(2 * I))) ||
        (rc = make_tmap_h16(&e->tm_w2[l], e->Mi(l, 5), H, I, gemm_bn_for(H)))) {
      delete e;
      return rc;
    }
  }
  const size_t n = (size_t)desc->max_pos * 64;
  if (cudaMalloc(&e->rope_cos, n * sizeof(float)) != cudaSuccess ||
      cudaMalloc(&e->rope_sin, n * sizeof(float)) != cudaSuccess) {
    b2e_encoder_destroy(e);
    return fail(B2E_ERR_CUDA, "cudaMalloc of the rotary tables failed");
  }
  rope_table_theta_kernel<<<(unsigned)((n + 255) / 256), 256>>>(e->rope_cos, e->rope_sin, desc->max_pos,
                                                                64, desc->rope_theta);
  if (cudaDeviceSynchronize() != cudaSuccess) {
    b2e_encoder_destroy(e);
    return fail(B2E_ERR_CUDA, "rotary table kernel failed: %s", cudaGetErrorString(cudaGetLastError()));
  }
  *out = e;
  return B2E_OK;
}
}  // namespace

int b2e_encoder_create(const B2EModelDesc* desc, const void* const* weights, int n_weights,
                       int device, B2EEncoder** out) {
  if (!desc || !weights || !out) return fail(B2E_ERR_INVALID, "null argument");
  *out = nullptr;
  if (desc->arch == B2E_ARCH_MISTRAL) return create_mistral(desc, weights, n_weights, device, out);
  int rc;
  if ((rc = b2e_check_model(desc))) return rc;
  if (n_weights != b2e_num_weights(desc))
    return fail(B2E_ERR_INVALID, "expected %d weight pointers, got %d", b2e_num_weights(desc),
                n_weights);
  for (int i = 0; i < n_weights; ++i)
    if (!weights[i]) return fail(B2E_ERR_INVALID, "weight pointer %d is null", i);
  DeviceInfo info;
  if ((rc = device_info(device, &info))) return rc;
  DeviceGuard guard;
  CUDA_TRY(cudaSetDevice(device));

  B2EEncoder* e = new B2EEncoder();
  e->desc = *desc;
  e->full_layers = desc->num_layers;
  e->w.assign(weights, weights + n_weights);
  e->device = device;
  e->sms = info.sms;
  const int L = desc->num_layers, H = desc->hidden, I = desc->intermediate;
  e->tm_wqkv.resize(L); e->tm_wo.resize(L); e->tm_w1.resize(L); e->tm_w2.resize(L);
  const bool esm = desc->arch == B2E_ARCH_ESM2;
  const bool mbert = desc->arch == B2E_ARCH_MODERNBERT;
  const int n1 = mbert ? 2 * I : I;   // ModernBERT's Wi holds input and gate rows
  for (int l = 0; l < L; ++l) {
    const void* wqkv = mbert ? e->Mb(l, 2) : esm ? e->E(l, 2) : e->L(l, 0);
    const void* wo = mbert ? e->Mb(l, 3) : esm ? e->E(l, 4) : e->L(l, 2);
    const void* w1 = mbert ? e->Mb(l, 6) : esm ? e->E(l, 8) : e->L(l, 6);
    const void* w2 = mbert ? e->Mb(l, 7) : esm ? e->E(l, 10) : e->L(l, 8);
    if ((rc = make_tmap_h16(&e->tm_wqkv[l], wqkv, 3 * H, H, gemm_bn_for(3 * H))) ||
        (rc = make_tmap_h16(&e->tm_wo[l], wo, H, H, gemm_bn_for(H))) ||
        (rc = make_tmap_h16(&e->tm_w1[l], w1, n1, H, gemm_bn_for(n1))) ||
        (rc = make_tmap_h16(&e->tm_w2[l], w2, H, I, gemm_bn_for(H)))) {
      delete e;
      return rc;
    }
  }
  if (mbert) {
    const size_t n = (size_t)desc->max_pos * 32;
    if (cudaMalloc(&e->rope_cos, n * sizeof(float)) != cudaSuccess ||
        cudaMalloc(&e->rope_sin, n * sizeof(float)) != cudaSuccess ||
        cudaMalloc(&e->rope_cos2, n * sizeof(float)) != cudaSuccess ||
        cudaMalloc(&e->rope_sin2, n * sizeof(float)) != cudaSuccess) {
      b2e_encoder_destroy(e);
      return fail(B2E_ERR_CUDA, "cudaMalloc of the rotary tables failed");
    }
    rope_table_theta_kernel<<<(unsigned)((n + 255) / 256), 256>>>(e->rope_cos, e->rope_sin, desc->max_pos, 32,
                                                                  desc->rope_theta);
    rope_table_theta_kernel<<<(unsigned)((n + 255) / 256), 256>>>(e->rope_cos2, e->rope_sin2, desc->max_pos, 32,
                                                                  desc->rope_theta_local);
    if (cudaDeviceSynchronize() != cudaSuccess) {
      b2e_encoder_destroy(e);
      return fail(B2E_ERR_CUDA, "rotary table kernel failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
  }
  if (esm) {
    const size_t n = (size_t)desc->max_pos * 32;
    if (cudaMalloc(&e->rope_cos, n * sizeof(float)) != cudaSuccess ||
        cudaMalloc(&e->rope_sin, n * sizeof(float)) != cudaSuccess) {
      b2e_encoder_destroy(e);
      return fail(B2E_ERR_CUDA, "cudaMalloc of the rotary tables failed");
    }
    rope_table_kernel<<<(unsigned)((n + 255) / 256), 256>>>(e->rope_cos, e->rope_sin, desc->max_pos);
    if (cudaDeviceSynchronize() != cudaSuccess) {
      b2e_encoder_destroy(e);
      return fail(B2E_ERR_CUDA, "rotary table kernel failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
  }
  *out = e;
  return B2E_OK;
}

void b2e_encoder_destroy(B2EEncoder* e) {
  if (!e) return;
  DeviceGuard guard;
  cudaSetDevice(e->device);
  cudaFree(e->hidden); cudaFree(e->qkv); cudaFree(e->ctx); cudaFree(e->tmp); cudaFree(e->ffn);
  cudaFree(e->stage_in); cudaFree(e->stage_out);
  cudaFree(e->xres); cudaFree(e->tok_scale); cudaFree(e->rope_cos); cudaFree(e->rope_sin);
  cudaFree(e->rope_cos2); cudaFree(e->rope_sin2);
  cudaFree(e->pk_len_raw); cudaFree(e->pk_ok); cudaFree(e->pk_len); cudaFree(e->pk_cu); cudaFree(e->pk_treal);
  cudaFree(e->pk_src);
  e->drop_graphs();
  e->pool.release();
  e->attn.release();
  if (e->own_stream) cudaStreamDestroy(e->own_stream);
  delete e;
}

int64_t b2e_workspace_bytes(const B2EEncoder* e, int B, int S) {
  if (!e || B <= 0 || S <= 0) return -1;
  const size_t tokens = (size_t)B * S;
  size_t bytes = tokens_bytes(e->desc, tokens);
  if (e->has_xres()) bytes += tokens * e->desc.hidden * 4 + (size_t)B * sizeof(float);
  bytes += tokens * sizeof(float) + (size_t)S * sizeof(int) + (size_t)B * (2 * sizeof(int) + sizeof(float));
  bytes += (size_t)B * pool_nsplit(S) * e->desc.hidden * sizeof(float);
  return (int64_t)bytes;
}

int b2e_encode(B2EEncoder* e, const int64_t* ids, const int64_t* mask, const int64_t* types, int B,
               int S, void* out_hidden, int out_dtype, void* stream) {
  int rc;
  if ((rc = validate_batch(e, B, S))) return rc;
  if (!ids || !mask || !out_hidden) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (out_dtype != B2E_DTYPE_F32 && out_dtype != kStorageDtype)
    return fail(B2E_ERR_INVALID, "encode: out_dtype must be F32 or this build's storage type (%d)", kStorageDtype);
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = ensure_workspace(e, B, S))) return rc;
  const B2EModelDesc& d = e->desc;
  const int M = B * S, H = d.hidden, l = d.num_layers - 1;
  if (d.arch == B2E_ARCH_MISTRAL) {
    if ((rc = run_mistral_trunk(e, ids, mask, B, S, st))) return rc;
    // final RMSNorm over (residual stream + last down_proj output)
    if (out_dtype == B2E_DTYPE_F32) {
      DISPATCH_NV(H, (add_rmsnorm_kernel<NV, float><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                         e->xres, e->tmp, (const float*)e->w[1], (float*)out_hidden, M, d.eps)));
    } else {
      DISPATCH_NV(H, (add_rmsnorm_kernel<NV, h16><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                         e->xres, e->tmp, (const float*)e->w[1], (h16*)out_hidden, M, d.eps)));
    }
    CUDA_TRY(cudaGetLastError());
    return B2E_OK;
  }
  if (d.arch == B2E_ARCH_ESM2 || d.arch == B2E_ARCH_MODERNBERT) {
    const bool mb = d.arch == B2E_ARCH_MODERNBERT;
    if ((rc = mb ? run_modernbert_trunk(e, ids, mask, B, S, st) : run_esm_trunk(e, ids, mask, B, S, st))) return rc;
    // emb_layer_norm_after / final_norm over (residual stream + last FFN output)
    const float* fg = (const float*)e->w[mb ? 3 : 1];
    const float* fb = (const float*)e->w[mb ? 4 : 2];
    if (out_dtype == B2E_DTYPE_F32) {
      DISPATCH_NV(H, (add_layernorm_kernel<NV, float><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                         e->xres, e->tmp, fg, fb, (float*)out_hidden, M, d.eps)));
    } else {
      DISPATCH_NV(H, (add_layernorm_kernel<NV, h16><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                         e->xres, e->tmp, fg, fb, (h16*)out_hidden, M, d.eps)));
    }
    CUDA_TRY(cudaGetLastError());
    return B2E_OK;
  }
  if ((rc = run_bert_trunk(e, ids, mask, types, B, S, st))) return rc;
  if (out_dtype == B2E_DTYPE_F32) {
    DISPATCH_NV(H, (layernorm_kernel<NV, float><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                       e->tmp, e->hidden, (const float*)e->L(l, 10), (const float*)e->L(l, 11),
                       (float*)out_hidden, M, d.eps)));
  } else {
    DISPATCH_NV(H, (layernorm_kernel<NV, h16><<<row_blocks(M), ROW_THREADS, 0, st>>>(
                       e->tmp, e->hidden, (const float*)e->L(l, 10), (const float*)e->L(l, 11),
                       (h16*)out_hidden, M, d.eps)));
  }
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

int b2e_encode_pooled(B2EEncoder* e, const int64_t* ids, const int64_t* mask, const int64_t* types,
                      int B, int S, int pool_kind, int l2, float* out, void* stream) {
  int rc;
  if ((rc = validate_batch(e, B, S))) return rc;
  if (!ids || !mask || !out) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (pool_kind < B2E_POOL_MEAN_REF || pool_kind > B2E_POOL_LAST_TOKEN)
    return fail(B2E_ERR_INVALID, "unknown pool_kind %d", pool_kind);
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = ensure_workspace(e, B, S))) return rc;
  const B2EModelDesc& d = e->desc;
  const int H = d.hidden, l = d.num_layers - 1;
  PoolScratch& ps = e->pool;
  // Pooled paths run on the padding-free token layout (pack.cuh): only attended tokens go through the GEMMs, norms
  // and attention query tiles; nothing here can observe a padded position.
  SeqLayout lay;
  if ((rc = pack_prepare(e, mask, B, S, packing_enabled(), st, &lay))) return rc;
  if (d.arch == B2E_ARCH_MISTRAL) {
    if ((rc = run_mistral_trunk(e, ids, mask, B, S, st, lay))) return rc;
    if (pool_kind == B2E_POOL_LAST_TOKEN) {
      // only the B selected rows go through the final norm (fp32 end to end)
      seq_len_kernel<<<(B + 7) / 8, 256, 0, st>>>(mask, ps.seq_len, B, S);
      last_token_index_kernel<<<1, 256, 0, st>>>(mask, ps.seq_len, ps.idx, B, S);
      DISPATCH_NV(H, (rmsnorm_gather_kernel<NV><<<row_blocks(B), ROW_THREADS, 0, st>>>(
                         e->xres, e->tmp, (const float*)e->w[1], ps.idx, out, B, S, d.eps, lay.cu)));
      if (l2) l2_normalize_kernel<<<(B + 7) / 8, 256, 0, st>>>(out, B, H);
      CUDA_TRY(cudaGetLastError());
      return B2E_OK;
    }
    // mean poolers: final RMSNorm fused with the masked sum, fp32 end to end, [B,S,H] never written
    if ((rc = launch_pool_weights(ps, const_cast<int64_t*>(mask), B, S, pool_kind, 0, st))) return rc;
    const int nsplit = pool_nsplit(S);
    const int rows_per = (S + nsplit - 1) / nsplit;
    dim3 grid(B, nsplit);
    DISPATCH_NV(H, (addnorm_pool_kernel<NV, true><<<grid, ROW_THREADS, 0, st>>>(
                       e->xres, e->tmp, (const float*)e->w[1], nullptr, ps.w, ps.part, S, rows_per, d.eps, lay.cu)));
    CUDA_TRY(cudaGetLastError());
    return launch_finalize(ps, out, B, H, nsplit, l2, /*round_mode=*/0, st);
  }
  if (d.arch == B2E_ARCH_ESM2 || d.arch == B2E_ARCH_MODERNBERT) {
    const bool mb = d.arch == B2E_ARCH_MODERNBERT;
    if ((rc = mb ? run_modernbert_trunk(e, ids, mask, B, S, st, lay) : run_esm_trunk(e, ids, mask, B, S, st, lay)))
      return rc;
    const float* fg = (const float*)e->w[mb ? 3 : 1];
    const float* fb = (const float*)e->w[mb ? 4 : 2];
    if (pool_kind == B2E_POOL_LAST_TOKEN) {
      // only the B selected rows go through emb_layer_norm_after (fp32 end to end)
      seq_len_kernel<<<(B + 7) / 8, 256, 0, st>>>(mask, ps.seq_len, B, S);
      last_token_index_kernel<<<1, 256, 0, st>>>(mask, ps.seq_len, ps.idx, B, S);
      DISPATCH_NV(H, (addnorm_gather_kernel<NV><<<row_blocks(B), ROW_THREADS, 0, st>>>(
                         e->xres, e->tmp, fg, fb, ps.idx, out, B, S, d.eps, lay.cu)));
      if (l2) l2_normalize_kernel<<<(B + 7) / 8, 256, 0, st>>>(out, B, H);
      CUDA_TRY(cudaGetLastError());
      return B2E_OK;
    }
    // mean poolers: final LayerNorm fused with the masked sum, fp32 end to end, [B,S,H] never written
    if ((rc = launch_pool_weights(ps, const_cast<int64_t*>(mask), B, S, pool_kind, 0, st))) return rc;
    const int nsplit = pool_nsplit(S);
    const int rows_per = (S + nsplit - 1) / nsplit;
    dim3 grid(B, nsplit);
    DISPATCH_NV(H, (addnorm_pool_kernel<NV, false><<<grid, ROW_THREADS, 0, st>>>(
                       e->xres, e->tmp, fg, fb, ps.w, ps.part, S, rows_per, d.eps, lay.cu)));
    CUDA_TRY(cudaGetLastError());
    return launch_finalize(ps, out, B, H, nsplit, l2, /*round_mode=*/0, st);
  }
  if ((rc = run_bert_trunk(e, ids, mask, types, B, S, st, lay))) return rc;
  const float* g = (const float*)e->L(l, 10);
  const float* bt = (const float*)e->L(l, 11);
  if (pool_kind == B2E_POOL_LAST_TOKEN) {
    seq_len_kernel<<<(B + 7) / 8, 256, 0, st>>>(mask, ps.seq_len, B, S);
    last_token_index_kernel<<<1, 256, 0, st>>>(mask, ps.seq_len, ps.idx, B, S);
    DISPATCH_NV(H, (layernorm_gather_kernel<NV><<<row_blocks(B), ROW_THREADS, 0, st>>>(
                       e->tmp, e->hidden, ps.idx, g, bt, out, B, S, d.eps, lay.cu)));
    if (l2) l2_normalize_kernel<<<(B + 7) / 8, 256, 0, st>>>(out, B, H);
    CUDA_TRY(cudaGetLastError());
    return B2E_OK;
  }
  // the fused path never edits the caller's mask: weights are built from a read-only view
  if ((rc = launch_pool_weights(ps, const_cast<int64_t*>(mask), B, S, pool_kind, /*mutate=*/0, st)))
    return rc;
  const int nsplit = pool_nsplit(S);
  const int rows_per = (S + nsplit - 1) / nsplit;
  dim3 grid(B, nsplit);
  DISPATCH_NV(H, (layernorm_pool_kernel<NV><<<grid, ROW_THREADS, 0, st>>>(
                     e->tmp, e->hidden, g, bt, ps.w, ps.part, S, rows_per, d.eps, lay.cu)));
  CUDA_TRY(cudaGetLastError());
  return launch_finalize(ps, out, B, H, nsplit, l2, /*round_mode=*/0, st);
}

int b2e_embed_host(B2EEncoder* e, const int64_t* ids, const int64_t* mask, const int64_t* types,
                   int64_t n_rows, int S, int batch, int pool_kind, int l2, float* out_host) {
  if (!e) return fail(B2E_ERR_INVALID, "null encoder handle");
  if (n_rows < 0 || batch <= 0) return fail(B2E_ERR_INVALID, "bad n_rows/batch");
  if (n_rows == 0) return B2E_OK;
  if (!ids || !mask || !out_host) return fail(B2E_ERR_INVALID, "null host pointer");
  int rc;
  DeviceGuard guard;
  CUDA_TRY(cudaSetDevice(e->device));   // host entry point: it owns its device context and stream
  if ((rc = validate_batch(e, batch, S))) return rc;
  if (!e->own_stream) CUDA_TRY(cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking));
  cudaStream_t st = e->own_stream;
  const int H = e->desc.hidden;
  // two input slots (ids | mask | types) so batch i+1 uploads while batch i computes
  const size_t slot = (size_t)batch * S * 3;
  if (2 * slot > e->stage_cap) {
    ++e->ws_gen;
    cudaFree(e->stage_in);
    e->stage_in = nullptr;
    e->stage_cap = 0;
    CUDA_TRY(cudaMalloc(&e->stage_in, 2 * slot * sizeof(int64_t)));
    e->stage_cap = 2 * slot;
  }
  const size_t out_elems = (size_t)batch * H * 2;
  if (out_elems > e->stage_out_cap) {
    ++e->ws_gen;
    cudaFree(e->stage_out);
    e->stage_out = nullptr;
    e->stage_out_cap = 0;
    CUDA_TRY(cudaMalloc(&e->stage_out, out_elems * sizeof(float)));
    e->stage_out_cap = out_elems;
  }
  static const bool use_graphs = [] {
    const char* v = getenv("B2E_GRAPHS");   // B2E_GRAPHS=0: every batch launches its kernels one by one
    return !(v && v[0] == '0');
  }();
  int which = 0;
  for (int64_t r0 = 0; r0 < n_rows; r0 += batch, which ^= 1) {
    const int B = (int)((n_rows - r0 < batch) ? (n_rows - r0) : batch);
    const size_t n = (size_t)B * S;
    int64_t* d_ids = e->stage_in + which * slot;
    int64_t* d_mask = d_ids + (size_t)batch * S;
    int64_t* d_types = d_mask + (size_t)batch * S;
    float* d_out = e->stage_out + (size_t)which * batch * H;
    CUDA_TRY(cudaMemcpyAsync(d_ids, ids + r0 * S, n * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_mask, mask + r0 * S, n * 8, cudaMemcpyHostToDevice, st));
    if (types) CUDA_TRY(cudaMemcpyAsync(d_types, types + r0 * S, n * 8, cudaMemcpyHostToDevice, st));
    // The first batch runs eagerly (it sizes every buffer and sets the kernels' attributes); later
    // FULL batches replay a graph captured once per (shape, pooling, staging slot): one launch
    // instead of ~90, which is what a small `batch_size` (the reference's default is 8) is bound by.
    const bool eager = !use_graphs || r0 == 0 || B != batch;
    if (eager) {
      if ((rc = b2e_encode_pooled(e, d_ids, d_mask, types ? d_types : nullptr, B, S, pool_kind, l2,
                                  d_out, st)))
        return rc;
    } else {
      if (e->graphs_stamp != e->buffer_stamp()) {
        e->drop_graphs();
        e->graphs_stamp = e->buffer_stamp();
      }
      cudaGraphExec_t exec = nullptr;
      for (const auto& g : e->graphs)
        if (g.B == B && g.S == S && g.pool_kind == pool_kind && g.l2 == l2 &&
            g.has_types == (types != nullptr) && g.slot == which)
          exec = g.exec;
      if (!exec) {
        cudaGraph_t graph = nullptr;
        CUDA_TRY(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        rc = b2e_encode_pooled(e, d_ids, d_mask, types ? d_types : nullptr, B, S, pool_kind, l2, d_out, st);
        const cudaError_t ce = cudaStreamEndCapture(st, &graph);
        if (rc) {
          if (graph) cudaGraphDestroy(graph);
          return rc;
        }
        if (ce != cudaSuccess) return fail(B2E_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(ce));
        if (e->graphs_stamp != e->buffer_stamp()) {   // a buffer moved during capture: do not keep it
          cudaGraphDestroy(graph);
          return fail(B2E_ERR_CUDA, "workspace reallocated while capturing a step graph");
        }
        const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) return fail(B2E_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(ie));
        e->graphs.push_back({B, S, pool_kind, l2, types != nullptr, which, exec});
      }
      CUDA_TRY(cudaGraphLaunch(exec, st));
    }
    CUDA_TRY(cudaMemcpyAsync(out_host + r0 * H, d_out, (size_t)B * H * sizeof(float),
                             cudaMemcpyDeviceToHost, st));
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  return B2E_OK;
}

int b2e_pool_mean(const void* hidden, int dtype, int64_t* mask, int B, int S, int H, int pool_kind,
                  int quirk_mutate, float* out, void* stream) {
  if (!hidden || !mask || !out) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (B <= 0 || S <= 0) return fail(B2E_ERR_INVALID, "empty batch B=%d S=%d", B, S);
  if (pool_kind != B2E_POOL_MEAN_REF && pool_kind != B2E_POOL_MEAN_PER_ROW)
    return fail(B2E_ERR_INVALID, "pool_mean: pool_kind %d", pool_kind);
  int rc;
  if ((rc = check_h(H))) return rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  PoolScratch& ps = g_pool_scratch;
  const int nsplit = pool_nsplit(S);
  const int rows_per = (S + nsplit - 1) / nsplit;
  if ((rc = ps.ensure(B, S, (size_t)B * nsplit * H))) return rc;
  if ((rc = launch_pool_weights(ps, mask, B, S, pool_kind, quirk_mutate, st))) return rc;
  dim3 grid(B, nsplit);
  int round_mode = 0;
  switch (dtype) {
    case B2E_DTYPE_F32:
      DISPATCH_NV(H, (pool_sum_kernel<NV, float><<<grid, ROW_THREADS, 0, st>>>(
                         (const float*)hidden, ps.w, ps.part, S, rows_per)));
      break;
    case B2E_DTYPE_BF16:
      round_mode = 1;
      DISPATCH_NV(H, (pool_sum_kernel<NV, bf16><<<grid, ROW_THREADS, 0, st>>>(
                         (const bf16*)hidden, ps.w, ps.part, S, rows_per)));
      break;
    case B2E_DTYPE_F16:
      round_mode = 2;
      DISPATCH_NV(H, (pool_sum_kernel<NV, __half><<<grid, ROW_THREADS, 0, st>>>(
                         (const __half*)hidden, ps.w, ps.part, S, rows_per)));
      break;
    default:
      return fail(B2E_ERR_INVALID, "pool_mean: dtype %d", dtype);
  }
  CUDA_TRY(cudaGetLastError());
  return launch_finalize(ps, out, B, H, nsplit, 0, round_mode, st);
}

int b2e_pool_last_token(const void* hidden, int dtype, const int64_t* mask, int B, int S, int H,
                        float* out, void* stream) {
  if (!hidden || !mask || !out) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (B <= 0 || S <= 0) return fail(B2E_ERR_INVALID, "empty batch B=%d S=%d", B, S);
  if (H % 8 != 0) return fail(B2E_ERR_INVALID, "H=%d must be a multiple of 8", H);
  int rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  PoolScratch& ps = g_pool_scratch;
  if ((rc = ps.ensure(B, S, 0))) return rc;
  seq_len_kernel<<<(B + 7) / 8, 256, 0, st>>>(mask, ps.seq_len, B, S);
  last_token_index_kernel<<<1, 256, 0, st>>>(mask, ps.seq_len, ps.idx, B, S);
  switch (dtype) {
    case B2E_DTYPE_F32:
      gather_rows_kernel<float><<<B, 128, 0, st>>>((const float*)hidden, ps.idx, out, B, S, H);
      break;
    case B2E_DTYPE_BF16:
      gather_rows_kernel<bf16><<<B, 128, 0, st>>>((const bf16*)hidden, ps.idx, out, B, S, H);
      break;
    case B2E_DTYPE_F16:
      gather_rows_kernel<__half><<<B, 128, 0, st>>>((const __half*)hidden, ps.idx, out, B, S, H);
      break;
    default:
      return fail(B2E_ERR_INVALID, "pool_last_token: dtype %d", dtype);
  }
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

int b2e_l2_normalize(float* x, int64_t n_rows, int H, void* stream) {
  if (!x) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (n_rows <= 0) return B2E_OK;
  if (H % 4 != 0) return fail(B2E_ERR_INVALID, "H=%d must be a multiple of 4", H);
  int rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  l2_normalize_kernel<<<(unsigned)((n_rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(x, (int)n_rows,
                                                                                   H);
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

int b2e_adjacent_cosine_dist(const void* emb, int dtype, int64_t n_rows, int H,
                             const int32_t* doc_id, float* out, void* stream) {
  if (n_rows <= 1) return B2E_OK;  // no adjacent pair: nothing to write (semantic_chunk.py:80-81)
  if (!emb || !out) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (H % 8 != 0) return fail(B2E_ERR_INVALID, "H=%d must be a multiple of 8", H);
  int rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned blocks = (unsigned)((n_rows - 1 + 7) / 8);
  switch (dtype) {
    case B2E_DTYPE_F32:
      adjacent_cosine_kernel<float><<<blocks, 256, 0, st>>>((const float*)emb, doc_id, out,
                                                            (int)n_rows, H);
      break;
    case B2E_DTYPE_BF16:
      adjacent_cosine_kernel<bf16><<<blocks, 256, 0, st>>>((const bf16*)emb, doc_id, out,
                                                           (int)n_rows, H);
      break;
    case B2E_DTYPE_F16:
      adjacent_cosine_kernel<__half><<<blocks, 256, 0, st>>>((const __half*)emb, doc_id, out,
                                                             (int)n_rows, H);
      break;
    default:
      return fail(B2E_ERR_INVALID, "adjacent_cosine_dist: dtype %d", dtype);
  }
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

// b2e_gemm_h16 and b2e_debug_gemm_rows: m_dev (nullable) = device-resident row count <= M, as in the trunks
static int gemm_h16_checked(const void* A, const void* W, const float* bias, const void* resid, void* out,
                            int M, int N, int K, int epi, const int* m_dev, void* stream) {
  if (!A || !W || !out) return fail(B2E_ERR_INVALID, "null tensor pointer");  // bias may be null
  if (epi == B2E_EPI_BIAS_RESID && !resid) return fail(B2E_ERR_INVALID, "resid epilogue needs resid");
  int rc;
  if ((rc = check_gemm_shape(M, N, K))) return rc;
  if ((epi == B2E_EPI_SWIGLU || epi == B2E_EPI_GEGLU) && N % 256 != 0)
    return fail(B2E_ERR_INVALID, "gemm: the gated epilogues need N %% 256 == 0 (got %d)", N);
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  CUtensorMap ta, tb;
  if ((rc = make_tmap_h16(&ta, A, M, K, 128))) return rc;
  if ((rc = make_tmap_h16(&tb, W, N, K, gemm_bn_for(N)))) return rc;
  return launch_gemm(ta, tb, out, bias, resid, M, N, K, epi, info.sms, (cudaStream_t)stream, m_dev);
}

int b2e_gemm_h16(const void* A, const void* W, const float* bias, const void* resid, void* out,
                  int M, int N, int K, int epi, void* stream) {
  return gemm_h16_checked(A, W, bias, resid, out, M, N, K, epi, nullptr, stream);
}

// Test hook (b2e_debug.h): b2e_gemm_h16 with the row count read on the device, as the packed trunks run it.
int b2e_debug_gemm_rows(const void* A, const void* W, const float* bias, const void* resid, void* out,
                        int M, int N, int K, int epi, const int* m_dev, void* stream) {
  if (!m_dev) return fail(B2E_ERR_INVALID, "gemm_rows: null device row count");
  return gemm_h16_checked(A, W, bias, resid, out, M, N, K, epi, m_dev, stream);
}

int b2e_attention_d64(const void* qkv, const int64_t* mask, void* ctx, int B, int S, int heads,
                      float* dbg, void* stream) {
  if (!qkv || !mask || !ctx) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (B <= 0 || S <= 0 || heads <= 0) return fail(B2E_ERR_INVALID, "empty attention problem");
  if (dbg) return fail(B2E_ERR_UNSUPPORTED, "the score dump of the first attention kernel is gone: pass NULL");
  int rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  CUtensorMap tq, tkv;
  if ((rc = make_tmap_h16(&tq, qkv, (uint64_t)B * S, (uint64_t)3 * heads * AT3_D, 128))) return rc;
  if ((rc = make_tmap_h16(&tkv, qkv, (uint64_t)B * S, (uint64_t)3 * heads * AT3_D, AT3_KC))) return rc;
  if ((rc = attention_prepare(g_attn_scratch, mask, B, S, st))) return rc;
  return launch_attention(tq, tkv, g_attn_scratch, ctx, B, S, heads, info.sms, st);
}

int b2e_attention_d64_window(const void* qkv, const int64_t* mask, void* ctx, int B, int S, int heads,
                             int window, void* stream) {
  if (!qkv || !mask || !ctx) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (B <= 0 || S <= 0 || heads <= 0 || window < 0) return fail(B2E_ERR_INVALID, "bad windowed attention problem");
  int rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  CUtensorMap tq, tkv;
  if ((rc = make_tmap_h16(&tq, qkv, (uint64_t)B * S, (uint64_t)3 * heads * AT3_D, 128))) return rc;
  if ((rc = make_tmap_h16(&tkv, qkv, (uint64_t)B * S, (uint64_t)3 * heads * AT3_D, AT3_KC))) return rc;
  if ((rc = attention_prepare(g_attn_scratch, mask, B, S, st))) return rc;
  return launch_attention(tq, tkv, g_attn_scratch, ctx, B, S, heads, info.sms, st, window);
}

int b2e_attention_causal_d128(const void* qkv, const int64_t* mask, void* ctx, int B, int S, int heads,
                              int kv_heads, int window, void* stream) {
  if (!qkv || !mask || !ctx) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (B <= 0 || S <= 0 || heads <= 0 || kv_heads <= 0 || heads % kv_heads != 0 || window < 0)
    return fail(B2E_ERR_INVALID, "bad causal attention problem B=%d S=%d heads=%d/%d window=%d", B, S,
                heads, kv_heads, window);
  int rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = attention_prepare(g_attn_scratch, mask, B, S, st))) return rc;
  return launch_attention_causal_d128(qkv, g_attn_scratch, ctx, B, S, heads, kv_heads, window,
                                      info.sms, st);
}

// Test hooks (b2e_debug.h) for the padding-free token layout (pack.cuh): the layout kernels of pack_prepare, and the
// attention kernels on rows cu[b] .. cu[b] + len[b] - 1 of [B*S]-row buffers, exactly as the encoder runs them.
int b2e_debug_pack_layout(const int64_t* mask, int B, int S, int enable, int* cu, int* len, int* t_real,
                          int* tok_src, void* stream) {
  if (!mask || !cu || !len || !t_real || !tok_src) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (B <= 0 || S <= 0) return fail(B2E_ERR_INVALID, "empty batch B=%d S=%d", B, S);
  int rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  int* scratch = nullptr;   // len_raw | ok, released in stream order
  CUDA_TRY(cudaMallocAsync(&scratch, sizeof(int) * 2 * (size_t)B, st));
  pack_lengths_kernel<<<(B + 7) / 8, 256, 0, st>>>(mask, scratch, scratch + B, B, S);
  pack_scan_kernel<<<1, 256, 0, st>>>(scratch, scratch + B, len, cu, t_real, B, S, enable ? 1 : 0);
  pack_fill_kernel<<<dim3((S + 255) / 256, B), 256, 0, st>>>(len, cu, tok_src, B, S);
  const cudaError_t le = cudaGetLastError();
  CUDA_TRY(cudaFreeAsync(scratch, st));
  CUDA_TRY(le);
  return B2E_OK;
}

int b2e_debug_attention_packed(const void* qkv, const int64_t* mask, const int* cu, const int* len, void* ctx,
                               int B, int S, int heads, int kv_heads, int head_dim, int window, void* stream) {
  if (!qkv || !mask || !cu || !len || !ctx) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (B <= 0 || S <= 0 || heads <= 0 || window < 0) return fail(B2E_ERR_INVALID, "bad attention problem");
  if (head_dim == 64 && kv_heads != heads)
    return fail(B2E_ERR_INVALID, "head_dim 64 attention has no grouped-query form (kv_heads %d != heads %d)",
                kv_heads, heads);
  if (head_dim == 128 && (kv_heads <= 0 || heads % kv_heads != 0))
    return fail(B2E_ERR_INVALID, "heads %d not a multiple of kv_heads %d", heads, kv_heads);
  if (head_dim != 64 && head_dim != 128) return fail(B2E_ERR_INVALID, "head_dim %d (need 64 or 128)", head_dim);
  int rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  SeqLayout lay;
  lay.cu = cu;
  lay.len = len;
  if ((rc = attention_prepare(g_attn_scratch, mask, B, S, st))) return rc;
  if (head_dim == 128)
    return launch_attention_causal_d128(qkv, g_attn_scratch, ctx, B, S, heads, kv_heads, window, info.sms, st, lay);
  CUtensorMap tq, tkv;
  if ((rc = make_tmap_h16(&tq, qkv, (uint64_t)B * S, (uint64_t)3 * heads * AT3_D, 128))) return rc;
  if ((rc = make_tmap_h16(&tkv, qkv, (uint64_t)B * S, (uint64_t)3 * heads * AT3_D, AT3_KC))) return rc;
  return launch_attention(tq, tkv, g_attn_scratch, ctx, B, S, heads, info.sms, st, window, lay);
}

// ---- exact inner-product top-k (retrieval query path)
extern "C++" {
namespace {
struct TopkScratch {
  float* score = nullptr;
  int64_t* index = nullptr;
  size_t cap = 0;
  int device = -1;
  int ensure(size_t elems) {
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev != device) {
      cudaFree(score); cudaFree(index);
      score = nullptr; index = nullptr; cap = 0;
      device = dev;
    }
    if (elems > cap) {
      cudaFree(score); cudaFree(index);
      score = nullptr; index = nullptr; cap = 0;
      CUDA_TRY(cudaMalloc(&score, elems * sizeof(float)));
      CUDA_TRY(cudaMalloc(&index, elems * sizeof(int64_t)));
      cap = elems;
    }
    return B2E_OK;
  }
};
thread_local TopkScratch g_topk_scratch;

template <typename T, int QT, int ROWS, int VMAX>
int launch_topk_cfg(const float* queries, int Q, const T* corpus, int64_t N, int H, int k, float* out_score,
                    int64_t* out_index, int sms, cudaStream_t st, const int* run_flag = nullptr) {
  // queries per pass: bounded by QT and by ~160 KiB of shared memory for the query tile
  int qt = QT;
  while (qt > 1 && (size_t)qt * H * 4 > 160 * 1024) qt >>= 1;
  const long long rows_per_cta = (TOPK_THREADS / 32) * ROWS;
  const long long want = (N + rows_per_cta - 1) / rows_per_cta;
  const int grid = (int)(want < (long long)2 * sms ? (want > 0 ? want : 1) : (long long)2 * sms);
  int rc;
  if ((rc = g_topk_scratch.ensure((size_t)grid * qt * k))) return rc;
  auto kern = topk_scan_kernel<T, QT, ROWS, VMAX>;
  const size_t smem_max = (size_t)qt * H * 4 + (size_t)qt * k * 12 + 8 + (size_t)qt * 12;
  // (k varies between calls: always set the attribute to this call's worst case)
  CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
  for (int q0 = 0; q0 < Q; q0 += qt) {
    const int nq = (Q - q0 < qt) ? (Q - q0) : qt;
    const size_t smem = (size_t)nq * H * 4 + (size_t)nq * k * 12 + 8 + (size_t)nq * 12;
    kern<<<grid, TOPK_THREADS, smem, st>>>(queries + (size_t)q0 * H, corpus, nq, (long long)N, H, k,
                                           g_topk_scratch.score, g_topk_scratch.index, run_flag);
    topk_merge_kernel<<<nq, TOPK_THREADS, 0, st>>>(g_topk_scratch.score, g_topk_scratch.index, grid, nq,
                                                   k, out_score + (size_t)q0 * k,
                                                   out_index + (size_t)q0 * k, k, run_flag);
  }
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

// one to four queries: the narrow, deeper scan; more: 16 queries per pass
template <typename T, int VWIDE, int VNARROW>
int launch_topk(const float* queries, int Q, const T* corpus, int64_t N, int H, int k, float* out_score,
                int64_t* out_index, int sms, cudaStream_t st, const int* run_flag = nullptr) {
  if (Q <= 4)
    return launch_topk_cfg<T, 4, 8, VNARROW>(queries, Q, corpus, N, H, k, out_score, out_index, sms, st, run_flag);
  return launch_topk_cfg<T, TOPK_QT, 4, VWIDE>(queries, Q, corpus, N, H, k, out_score, out_index, sms, st,
                                               run_flag);
}

// ---- tensor-core fast path (topk_tc.cuh)
struct TcScratch {
  float* scores = nullptr;      // [tiles * 128, 16]
  float* qpad = nullptr;        // [16, H]
  TcQuery* meta = nullptr;      // [16]
  unsigned* hist = nullptr;     // [16, TC_BINS]
  unsigned* cand = nullptr;     // [16, TC_MAX_CAND]
  unsigned* n_cand = nullptr;   // [16]
  int* flag = nullptr;          // [2]: fallback requested; passes that requested it (debug)
  float* norm2 = nullptr;       // [1]
  size_t cap_rows = 0, cap_h = 0;
  int device = -1;
  void release() {
    cudaFree(scores); cudaFree(qpad); cudaFree(meta); cudaFree(hist); cudaFree(cand); cudaFree(n_cand);
    cudaFree(flag); cudaFree(norm2);
    scores = qpad = norm2 = nullptr; meta = nullptr; hist = cand = n_cand = nullptr; flag = nullptr;
    cap_rows = cap_h = 0;
  }
  int ensure(size_t rows, size_t h) {
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev != device) {
      release();
      device = dev;
    }
    if (rows <= cap_rows && h <= cap_h && flag != nullptr) return B2E_OK;
    const size_t r = rows > cap_rows ? rows : cap_rows, hh = h > cap_h ? h : cap_h;
    release();
    CUDA_TRY(cudaMalloc(&scores, r * TC_NQ * sizeof(float)));
    CUDA_TRY(cudaMalloc(&qpad, (size_t)TC_NQ * hh * sizeof(float)));
    CUDA_TRY(cudaMalloc(&meta, TC_NQ * sizeof(TcQuery)));
    CUDA_TRY(cudaMalloc(&hist, (size_t)TC_NQ * TC_BINS * sizeof(unsigned)));
    CUDA_TRY(cudaMalloc(&cand, (size_t)TC_NQ * TC_MAX_CAND * sizeof(unsigned)));
    CUDA_TRY(cudaMalloc(&n_cand, TC_NQ * sizeof(unsigned)));
    CUDA_TRY(cudaMalloc(&flag, 2 * sizeof(int)));
    CUDA_TRY(cudaMalloc(&norm2, sizeof(float)));
    CUDA_TRY(cudaMemset(flag, 0, 2 * sizeof(int)));
    cap_rows = r;
    cap_h = hh;
    return B2E_OK;
  }
};
thread_local TcScratch g_tc_scratch;
}  // namespace
}  // extern "C++"

int b2e_topk_ip(const float* queries, int Q, const void* corpus, int corpus_dtype, int64_t N, int H,
                int k, float* out_scores, int64_t* out_indices, void* stream) {
  if (!queries || !corpus || !out_scores || !out_indices) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (Q <= 0 || N <= 0) return fail(B2E_ERR_INVALID, "topk: empty problem Q=%d N=%lld", Q, (long long)N);
  if (k <= 0 || k > TOPK_MAX_K) return fail(B2E_ERR_INVALID, "topk: k=%d must be in [1, %d]", k, TOPK_MAX_K);
  const int hq = (corpus_dtype == B2E_DTYPE_BF16) ? 256 : 128;   // one 16-byte vector per lane
  if (H % hq != 0 || H > 8192)
    return fail(B2E_ERR_INVALID, "topk: H=%d must be a multiple of %d (<= 8192)", H, hq);
  int rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  switch (corpus_dtype) {
    case B2E_DTYPE_F32:
      return launch_topk<float, 6, 3>(queries, Q, (const float*)corpus, N, H, k, out_scores, out_indices, info.sms, st);
    case B2E_DTYPE_BF16:
      return launch_topk<bf16, 3, 2>(queries, Q, (const bf16*)corpus, N, H, k, out_scores, out_indices, info.sms, st);
  }
  return fail(B2E_ERR_INVALID, "topk: corpus dtype %d (F32 or BF16)", corpus_dtype);
}

// largest Euclidean row norm of a float32 matrix (synchronises the stream: an index-build step, not a query step)
int b2e_max_row_norm(const float* x, int64_t N, int H, float* out_host, void* stream) {
  if (!x || !out_host) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (N <= 0 || H <= 0 || H % 4 != 0) return fail(B2E_ERR_INVALID, "max_row_norm: N=%lld H=%d", (long long)N, H);
  int rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  TcScratch& sc = g_tc_scratch;
  if ((rc = sc.ensure(TC_ROWS, 128))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_TRY(cudaMemsetAsync(sc.norm2, 0, sizeof(float), st));
  max_row_norm2_kernel<<<info.sms * 4, 256, 0, st>>>(x, (long long)N, H, sc.norm2);
  float n2 = 0.0f;
  CUDA_TRY(cudaMemcpyAsync(&n2, sc.norm2, sizeof(float), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  *out_host = sqrtf(n2);
  return B2E_OK;
}

// Exact inner-product top-k with the scan on the tensor cores (topk_tc.cuh).  corpus_max_norm bounds the Euclidean
// norm of every corpus row (b2e_max_row_norm; 1 for normalised embeddings): it sizes the TF32 error margin.
// Same results as b2e_topk_ip; small problems and anything the fast path cannot take go there directly.
int b2e_topk_ip_tc(const float* queries, int Q, const float* corpus, int64_t N, int H, int k,
                   float corpus_max_norm, float* out_scores, int64_t* out_indices, void* stream) {
  if (!queries || !corpus || !out_scores || !out_indices) return fail(B2E_ERR_INVALID, "null tensor pointer");
  const bool fast = N >= 32768 && N < ((int64_t)1 << 31) - TC_ROWS && H % 128 == 0 && H <= 8192 && k > 0 && k <= TOPK_MAX_K &&
                    corpus_max_norm > 0.0f && corpus_max_norm < 1e30f && Q > 0;
  if (!fast) return b2e_topk_ip(queries, Q, corpus, B2E_DTYPE_F32, N, H, k, out_scores, out_indices, stream);
  int rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const long long tiles = (N + TC_ROWS - 1) / TC_ROWS;
  TcScratch& sc = g_tc_scratch;
  if ((rc = sc.ensure((size_t)tiles * TC_ROWS, (size_t)H))) return rc;
  CUtensorMap tm_c, tm_q;
  if ((rc = make_tmap_f32(&tm_c, corpus, (uint64_t)N, (uint64_t)H, TC_ROWS))) return rc;
  if ((rc = make_tmap_f32(&tm_q, sc.qpad, TC_NQ, (uint64_t)H, TC_NQ))) return rc;
  if ((rc = ensure_smem_attr(tf32_scan_kernel, TC_SMEM_BYTES))) return rc;
  if ((rc = ensure_smem_attr(score_hist_kernel, TC_NQ * TC_BINS * 4))) return rc;
  if ((rc = ensure_smem_attr(exact_rescore_kernel, TC_MAX_CAND * 8 + 8192 * 4))) return rc;
  CUDA_TRY(cudaMemsetAsync(sc.flag, 0, 2 * sizeof(int), st));
  const int grid_scan = tiles < info.sms ? (int)tiles : info.sms;
  const int grid_rows = info.sms * 2;
  for (int q0 = 0; q0 < Q; q0 += TC_NQ) {
    const int nq = Q - q0 < TC_NQ ? Q - q0 : TC_NQ;
    tc_prepare_queries_kernel<<<TC_NQ, 256, 0, st>>>(queries + (size_t)q0 * H, nq, H, corpus_max_norm, sc.qpad,
                                                     sc.meta);
    CUDA_TRY(cudaMemsetAsync(sc.hist, 0, (size_t)TC_NQ * TC_BINS * sizeof(unsigned), st));
    CUDA_TRY(cudaMemsetAsync(sc.n_cand, 0, TC_NQ * sizeof(unsigned), st));
    tf32_scan_kernel<<<grid_scan, TC_THREADS, TC_SMEM_BYTES, st>>>(tm_c, tm_q, sc.scores, tiles, H);
    score_hist_kernel<<<grid_rows, 512, (size_t)nq * TC_BINS * 4, st>>>(sc.scores, (long long)N, nq, sc.meta,
                                                                        sc.hist);
    score_threshold_kernel<<<1, 32 * TC_NQ, 0, st>>>(sc.hist, nq, (long long)N, k, sc.meta);
    score_select_kernel<<<grid_rows, 512, 0, st>>>(sc.scores, (long long)N, nq, sc.meta, sc.cand, sc.n_cand);
    exact_rescore_kernel<<<nq, 512, (size_t)TC_MAX_CAND * 8 + (size_t)H * 4, st>>>(
        sc.cand, sc.n_cand, sc.meta, queries + (size_t)q0 * H, corpus, H, k, out_scores + (size_t)q0 * k,
        out_indices + (size_t)q0 * k, sc.flag);
  }
  CUDA_TRY(cudaGetLastError());
  // the exact scan redoes the call when a candidate list overflowed; otherwise its kernels return at once
  return launch_topk<float, 6, 3>(queries, Q, corpus, N, H, k, out_scores, out_indices, info.sms, st, sc.flag);
}

// 1 when the last b2e_topk_ip_tc call of this thread had to fall back to the exact scan (synchronises the device)
int b2e_debug_topk_tc_fell_back(int* out) {
  if (!out) return fail(B2E_ERR_INVALID, "null pointer");
  *out = 0;
  if (g_tc_scratch.flag == nullptr) return B2E_OK;
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpy(out, g_tc_scratch.flag, sizeof(int), cudaMemcpyDeviceToHost));
  return B2E_OK;
}

// ---- ubinary retrieval: packed bits, Hamming top-K, float rescoring (binsearch.cuh)
extern "C++" {
namespace {
struct BinScratch {
  uint32_t* qbits = nullptr;            // [Q, W]
  unsigned* hist = nullptr;             // [Q, H+1]
  int* thr = nullptr;                   // [Q, 2]
  unsigned long long* cand = nullptr;   // [Q, BIN_MAX_CAND]
  unsigned* n_cand = nullptr;           // [Q]
  size_t cap_q = 0, cap_h = 0;
  int device = -1;
  void release() {
    cudaFree(qbits); cudaFree(hist); cudaFree(thr); cudaFree(cand); cudaFree(n_cand);
    qbits = nullptr; hist = nullptr; thr = nullptr; cand = nullptr; n_cand = nullptr;
    cap_q = cap_h = 0;
  }
  int ensure(int Q, int H) {
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev != device) {
      release();
      device = dev;
    }
    if ((size_t)Q <= cap_q && (size_t)H <= cap_h) return B2E_OK;
    release();
    const size_t q = (size_t)Q > 8 ? Q : 8, h = (size_t)H > 1024 ? H : 1024;
    CUDA_TRY(cudaMalloc(&qbits, q * (h / 32) * sizeof(uint32_t)));
    CUDA_TRY(cudaMalloc(&hist, q * (h + 1) * sizeof(unsigned)));
    CUDA_TRY(cudaMalloc(&thr, q * 2 * sizeof(int)));
    CUDA_TRY(cudaMalloc(&cand, q * BIN_MAX_CAND * sizeof(unsigned long long)));
    CUDA_TRY(cudaMalloc(&n_cand, q * sizeof(unsigned)));
    cap_q = q;
    cap_h = h;
    return B2E_OK;
  }
};
thread_local BinScratch g_bin_scratch;

template <int Q>
int launch_bin_pass(const uint32_t* corpus, const uint32_t* qbits, int64_t N, int W, int H, long long K,
                    BinScratch& sc, int q0, int grid, cudaStream_t st) {
  const size_t smem_hist = (size_t)Q * W * 4 + (size_t)Q * (H + 1) * 4;
  const size_t smem_sel = (size_t)Q * W * 4;
  auto hist_k = hamming_hist_kernel<Q>;
  auto sel_k = hamming_select_kernel<Q>;
  int rc;
  // the attribute is set ONCE per kernel and device: to the largest size any call may ask for (Q <= 8 queries of
  // H <= 8192 stay under 160 KiB by the choice of qp in the caller), not to this call's size
  if ((rc = ensure_smem_attr(hist_k, 164 * 1024))) return rc;
  hist_k<<<grid, BIN_THREADS, smem_hist, st>>>(corpus, qbits + (size_t)q0 * W, N, W, H,
                                               sc.hist + (size_t)q0 * (H + 1));
  hamming_threshold_kernel<<<1, 32, 0, st>>>(sc.hist + (size_t)q0 * (H + 1), H, K, Q, sc.thr + 2 * q0);
  sel_k<<<grid, BIN_THREADS, smem_sel, st>>>(corpus, qbits + (size_t)q0 * W, N, W, sc.thr + 2 * q0,
                                             sc.cand + (size_t)q0 * BIN_MAX_CAND, sc.n_cand + q0, BIN_MAX_CAND);
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}
}  // namespace
}  // extern "C++"

int b2e_pack_ubinary(const float* emb, int64_t n_rows, int H, uint8_t* out, void* stream) {
  if (n_rows <= 0) return B2E_OK;
  if (!emb || !out) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (H <= 0 || H % 8 != 0) return fail(B2E_ERR_INVALID, "pack_ubinary: H=%d must be a positive multiple of 8", H);
  int rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  const long long total = (long long)n_rows * (H / 8);
  long long blocks = (total + 255) / 256;
  if (blocks > (long long)info.sms * 16) blocks = (long long)info.sms * 16;
  pack_ubinary_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(emb, out, n_rows, H);
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

int b2e_search_ubinary(const float* queries, int Q, const uint8_t* corpus_bits, int64_t N, int H, int k,
                       int rescore_multiplier, float* out_scores, int64_t* out_indices, void* stream) {
  if (!queries || !corpus_bits || !out_scores || !out_indices) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (Q <= 0 || N <= 0) return fail(B2E_ERR_INVALID, "search_ubinary: empty problem Q=%d N=%lld", Q, (long long)N);
  if (H <= 0 || H % 32 != 0 || H / 32 > BIN_MAX_WORDS)
    return fail(B2E_ERR_INVALID, "search_ubinary: H=%d must be a multiple of 32 (<= %d)", H, 32 * BIN_MAX_WORDS);
  if (N >= (1ll << 40)) return fail(B2E_ERR_INVALID, "search_ubinary: N=%lld too large", (long long)N);
  if (k <= 0 || rescore_multiplier <= 0) return fail(B2E_ERR_INVALID, "search_ubinary: k and rescore_multiplier must be positive");
  const long long K = (long long)k * rescore_multiplier;
  if (2 * K > BIN_MAX_CAND)
    return fail(B2E_ERR_INVALID, "search_ubinary: k * rescore_multiplier = %lld exceeds %d", K, BIN_MAX_CAND / 2);
  if ((reinterpret_cast<uintptr_t>(corpus_bits) & 15u) != 0)
    return fail(B2E_ERR_INVALID, "search_ubinary: corpus_bits must be 16-byte aligned");
  int rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  BinScratch& sc = g_bin_scratch;
  if ((rc = sc.ensure(Q, H))) return rc;
  const int W = H / 32;
  const uint32_t* corpus = reinterpret_cast<const uint32_t*>(corpus_bits);
  if ((rc = b2e_pack_ubinary(queries, Q, H, reinterpret_cast<uint8_t*>(sc.qbits), stream))) return rc;
  CUDA_TRY(cudaMemsetAsync(sc.hist, 0, (size_t)Q * (H + 1) * sizeof(unsigned), st));
  CUDA_TRY(cudaMemsetAsync(sc.n_cand, 0, (size_t)Q * sizeof(unsigned), st));
  long long want = (N + BIN_THREADS - 1) / BIN_THREADS;
  const int grid = (int)(want < (long long)info.sms * 8 ? want : (long long)info.sms * 8);
  // queries per pass over the corpus: as many as the shared-memory histogram allows (<= 8)
  int qp = 8;
  while (qp > 1 && (size_t)qp * (W + H + 1) * 4 > 160 * 1024) qp >>= 1;
  for (int q0 = 0; q0 < Q;) {
    int n = Q - q0 < qp ? Q - q0 : qp;
    if (n >= 8) { n = 8; rc = launch_bin_pass<8>(corpus, sc.qbits, N, W, H, K, sc, q0, grid, st); }
    else if (n >= 4) { n = 4; rc = launch_bin_pass<4>(corpus, sc.qbits, N, W, H, K, sc, q0, grid, st); }
    else if (n >= 2) { n = 2; rc = launch_bin_pass<2>(corpus, sc.qbits, N, W, H, K, sc, q0, grid, st); }
    else { n = 1; rc = launch_bin_pass<1>(corpus, sc.qbits, N, W, H, K, sc, q0, grid, st); }
    if (rc) return rc;
    q0 += n;
  }
  // candidates: the K nearest plus every row tied with the K-th; sort width = next power of two >= 2K
  int n_pow2 = 2;
  while (n_pow2 < 2 * K || n_pow2 < 64) n_pow2 <<= 1;
  if (n_pow2 < BIN_MAX_CAND) n_pow2 = BIN_MAX_CAND;   // ties beyond 2K still fit up to the buffer size
  const size_t smem = (size_t)n_pow2 * 8 + (size_t)H * 4;
  if ((rc = ensure_smem_attr(binary_rescore_kernel, BIN_MAX_CAND * 8 + 32 * BIN_MAX_WORDS * 4))) return rc;
  binary_rescore_kernel<<<Q, BIN_THREADS, smem, st>>>(sc.cand, sc.n_cand, BIN_MAX_CAND, n_pow2, corpus, W, H,
                                                      queries, K, k, out_scores,
                                                      reinterpret_cast<long long*>(out_indices));
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

int b2e_layernorm(const void* in, const float* gamma, const float* beta, void* out, int rows, int H,
                  float eps, int out_dtype, void* stream) {
  if (!in || !gamma || !beta || !out) return fail(B2E_ERR_INVALID, "null tensor pointer");
  if (rows <= 0) return B2E_OK;
  int rc;
  if ((rc = check_h(H))) return rc;
  DeviceInfo info;
  if ((rc = current_device_info(&info))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (out_dtype == B2E_DTYPE_F32) {
    DISPATCH_NV(H, (layernorm_kernel<NV, float><<<row_blocks(rows), ROW_THREADS, 0, st>>>(
                       (const h16*)in, nullptr, gamma, beta, (float*)out, rows, eps)));
  } else if (out_dtype == kStorageDtype) {
    DISPATCH_NV(H, (layernorm_kernel<NV, h16><<<row_blocks(rows), ROW_THREADS, 0, st>>>(
                       (const h16*)in, nullptr, gamma, beta, (h16*)out, rows, eps)));
  } else {
    return fail(B2E_ERR_INVALID, "layernorm: out_dtype must be F32 or the storage type");
  }
  CUDA_TRY(cudaGetLastError());
  return B2E_OK;
}

}  // extern "C"
