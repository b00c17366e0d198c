// extern "C" surface shared by all kernels: error state, device checks, GEMM entry points.
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "common.cuh"
#include "tmap.cuh"

namespace merv {

static thread_local char g_error[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
  return code;
}

static int g_dev_ok[64];    // 0 unknown, 1 ok, -1 wrong arch
static int g_dev_sms[64];

int require_sm100() {
  int dev = -1;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return fail(MERV_E_CUDA, "cudaGetDevice failed: %s (no CUDA device? this library has no CPU path)", cudaGetErrorString(e));
  if (dev < 0 || dev >= 64) return fail(MERV_E_CUDA, "device index %d out of range", dev);
  if (g_dev_ok[dev] == 0) {
    int major = 0, sms = 0;
    e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return fail(MERV_E_CUDA, "cudaDeviceGetAttribute failed: %s", cudaGetErrorString(e));
    g_dev_sms[dev] = sms;
    g_dev_ok[dev] = (major == 10) ? 1 : -1;
  }
  if (g_dev_ok[dev] < 0) return fail(MERV_E_ARCH, "device %d is not compute capability 10.x; libmerv_fusion is built for sm_100a only", dev);
  return MERV_OK;
}

bool pdl_enabled() {
  const char* e = getenv("MERV_PDL");
  return !(e != nullptr && e[0] == '0');
}

int sm_count() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (g_dev_sms[dev] == 0) {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) return 148;
    g_dev_sms[dev] = sms;
  }
  return g_dev_sms[dev];
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  });
  return fn;
}

constexpr int kTmapCacheSize = 128;
static TmapKey g_tmap_keys[kTmapCacheSize];
static CUtensorMap g_tmap_vals[kTmapCacheSize];
static int g_tmap_used = 0, g_tmap_next = 0;
static std::mutex g_tmap_mutex;

int encode_tmap_cached(CUtensorMap* out, int dtype, int rank, const void* base, const unsigned long long* dims,
                       const unsigned long long* strides_bytes, const unsigned* box, int swizzle) {
  TmapKey key;
  memset(&key, 0, sizeof(key));  // padding participates in the memcmp
  key.base = base; key.dtype = dtype; key.rank = rank; key.swizzle = swizzle;
  for (int i = 0; i < rank; ++i) { key.dims[i] = dims[i]; key.box[i] = box[i]; }
  for (int i = 0; i + 1 < rank; ++i) key.strides[i] = strides_bytes[i];
  {
    std::lock_guard<std::mutex> lock(g_tmap_mutex);
    for (int i = 0; i < g_tmap_used; ++i)
      if (g_tmap_keys[i] == key) {
        *out = g_tmap_vals[i];
        return MERV_OK;
      }
  }
  EncodeTiledFn enc = encode_tiled_fn();
  if (enc == nullptr) return fail(MERV_E_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  // cuTensorMapEncodeTiled is a DRIVER call: it needs a context current on the calling thread, and a thread whose first CUDA work is this
  // call (autograd's worker thread entering a backward that starts with a GEMM) has none yet -> CUDA_ERROR_INVALID_CONTEXT.  One
  // runtime call binds the device's primary context to the thread.
  static thread_local bool ctx_bound = false;
  if (!ctx_bound) {
    cudaFree(nullptr);
    ctx_bound = true;
  }
  cuuint64_t d[5], st[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { d[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) st[i] = strides_bytes[i];
  const CUresult r = enc(out, static_cast<CUtensorMapDataType>(dtype), rank, const_cast<void*>(base), d, st, bx, es,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, static_cast<CUtensorMapSwizzle>(swizzle), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(MERV_E_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d (rank %d, dims %llu x %llu, box %u x %u)", int(r), rank, dims[0],
                rank > 1 ? dims[1] : 1ull, box[0], rank > 1 ? box[1] : 1u);
  std::lock_guard<std::mutex> lock(g_tmap_mutex);
  const int slot = g_tmap_used < kTmapCacheSize ? g_tmap_used++ : (g_tmap_next++ % kTmapCacheSize);
  g_tmap_keys[slot] = key;
  g_tmap_vals[slot] = *out;
  return MERV_OK;
}

}  // namespace merv

using namespace merv;

extern "C" int merv_abi_version(void) { return MERV_ABI_VERSION; }
extern "C" const char* merv_last_error(void) { return g_error; }
extern "C" int merv_device_check(void) { return require_sm100(); }
extern "C" int merv_num_sms(void) { return sm_count(); }

// impl: 0 = default for the dtype (bf16 -> tcgen05, fp32 -> SIMT); MERV_GEMM_IMPL=simt forces the SIMT kernel for
// bf16 too (used by the tests to cross-check the tensor-core kernel on the GPU; never a CPU path).
static bool force_simt() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MERV_GEMM_IMPL");
    v = (e != nullptr && strcmp(e, "simt") == 0) ? 1 : 0;
  }
  return v == 1;
}

extern "C" int merv_linear_bias_act(const void* A, int64_t lda, const void* W, int64_t ldw, const void* bias, void* Y,
                                    int64_t ldy, int M, int N, int K, int act, int dtype, const float* rowdot_vec,
                                    float* rowdot_out, void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_linear_bias_act: unknown dtype %d", dtype);
  MERV_REQUIRE(act == MERV_ACT_NONE || act == MERV_ACT_GELU_ERF, MERV_E_DTYPE, "merv_linear_bias_act: unknown activation %d", act);
  MERV_REQUIRE(A && W && Y, MERV_E_ARG, "merv_linear_bias_act: NULL operand");
  MERV_REQUIRE(M >= 0 && N > 0 && K > 0, MERV_E_SHAPE, "merv_linear_bias_act: M=%d N=%d K=%d", M, N, K);
  MERV_REQUIRE(lda >= K && ldw >= K && ldy >= N, MERV_E_SHAPE, "merv_linear_bias_act: leading dimensions lda=%lld ldw=%lld ldy=%lld too small",
               (long long)lda, (long long)ldw, (long long)ldy);
  if (int rc = require_sm100()) return rc;
  if (M == 0) return MERV_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dtype == MERV_BF16 && !force_simt()) {
    GemmSegment seg = {A, lda, W, ldw, K};
    return launch_gemm_tcgen05(&seg, 1, nullptr, nullptr, M, bias, act, rowdot_vec, rowdot_out, Y, ldy, 0, M, N, 0, s);
  }
  MERV_REQUIRE(rowdot_vec == nullptr && rowdot_out == nullptr, MERV_E_DTYPE,
               "merv_linear_bias_act: the row-dot epilogue exists only on the bf16 tensor-core path");
  return launch_gemm_simt(A, lda, W, ldw, bias, Y, ldy, M, N, K, act, dtype, s);
}

extern "C" int merv_gemm_ex(const void* A, int64_t lda, int a_mn, const void* W, int64_t ldw, int w_mn, const void* bias, void* Y, int64_t ldy,
                            int M, int N, int K, int act, void* stream) {
  MERV_REQUIRE(act == MERV_ACT_NONE || act == MERV_ACT_GELU_ERF, MERV_E_DTYPE, "merv_gemm_ex: unknown activation %d", act);
  MERV_REQUIRE(A && W && Y, MERV_E_ARG, "merv_gemm_ex: NULL operand");
  MERV_REQUIRE(M >= 0 && N > 0 && K > 0 && ldy >= N, MERV_E_SHAPE, "merv_gemm_ex: M=%d N=%d K=%d ldy=%lld", M, N, K, (long long)ldy);
  if (int rc = require_sm100()) return rc;
  if (M == 0) return MERV_OK;
  GemmSegment seg = {A, lda, W, ldw, K, a_mn ? 1 : 0, w_mn ? 1 : 0};
  return launch_gemm_tcgen05(&seg, 1, nullptr, nullptr, M, bias, act, nullptr, nullptr, Y, ldy, 0, M, N, 0, static_cast<cudaStream_t>(stream));
}

extern "C" int merv_fused_linear_mix_gather(const void* const* A, const int64_t* lda, const void* const* W, const int64_t* ldw,
                                            const int32_t* K, int nseg, const float* scale, const float* bias_mix, void* out,
                                            int64_t ldo, int64_t out_batch_stride, int M, int N, int rows_per_video, int max_ctas,
                                            void* const* peer_out, int num_peers, void* stream) {
  MERV_REQUIRE(A && lda && W && ldw && K && scale && out, MERV_E_ARG, "merv_fused_linear_mix: NULL pointer");
  MERV_REQUIRE(nseg >= 1 && nseg <= MERV_MAX_SEGMENTS, MERV_E_ARG, "merv_fused_linear_mix: nseg=%d not in [1,%d]", nseg, MERV_MAX_SEGMENTS);
  MERV_REQUIRE(M >= 0 && N > 0 && rows_per_video > 0, MERV_E_SHAPE, "merv_fused_linear_mix: M=%d N=%d rows_per_video=%d", M, N, rows_per_video);
  MERV_REQUIRE(M % rows_per_video == 0, MERV_E_SHAPE, "merv_fused_linear_mix: M=%d is not a multiple of rows_per_video=%d", M, rows_per_video);
  if (int rc = require_sm100()) return rc;
  if (M == 0) return MERV_OK;
  GemmSegment seg[MERV_MAX_SEGMENTS];
  for (int s = 0; s < nseg; ++s) seg[s] = GemmSegment{A[s], lda[s], W[s], ldw[s], K[s]};
  return launch_gemm_tcgen05(seg, nseg, scale, bias_mix, rows_per_video, nullptr, MERV_ACT_NONE, nullptr, nullptr, out, ldo, out_batch_stride,
                             M, N, max_ctas, static_cast<cudaStream_t>(stream), peer_out, num_peers);
}

extern "C" int merv_fused_linear_mix_multicast(const void* const* A, const int64_t* lda, const void* const* W, const int64_t* ldw,
                                               const int32_t* K, int nseg, const float* scale, const float* bias_mix, void* out,
                                               int64_t ldo, int M, int N, int rows_per_video, int max_ctas, void* mc_out, void* stream) {
  MERV_REQUIRE(A && lda && W && ldw && K && scale && out && mc_out, MERV_E_ARG, "merv_fused_linear_mix_multicast: NULL pointer");
  MERV_REQUIRE(nseg >= 1 && nseg <= MERV_MAX_SEGMENTS, MERV_E_ARG, "merv_fused_linear_mix_multicast: nseg=%d not in [1,%d]", nseg, MERV_MAX_SEGMENTS);
  MERV_REQUIRE(M >= 0 && N > 0 && rows_per_video > 0 && M % rows_per_video == 0, MERV_E_SHAPE,
               "merv_fused_linear_mix_multicast: M=%d N=%d rows_per_video=%d", M, N, rows_per_video);
  if (int rc = require_sm100()) return rc;
  if (M == 0) return MERV_OK;
  GemmSegment seg[MERV_MAX_SEGMENTS];
  for (int s = 0; s < nseg; ++s) seg[s] = GemmSegment{A[s], lda[s], W[s], ldw[s], K[s]};
  return launch_gemm_tcgen05(seg, nseg, scale, bias_mix, rows_per_video, nullptr, MERV_ACT_NONE, nullptr, nullptr, out, ldo, 0, M, N, max_ctas,
                             static_cast<cudaStream_t>(stream), nullptr, 0, false, mc_out);
}

extern "C" int merv_fused_linear_mix(const void* const* A, const int64_t* lda, const void* const* W, const int64_t* ldw,
                                     const int32_t* K, int nseg, const float* scale, const float* bias_mix, void* out,
                                     int64_t ldo, int64_t out_batch_stride, int M, int N, int rows_per_video, int max_ctas, void* stream) {
  return merv_fused_linear_mix_gather(A, lda, W, ldw, K, nseg, scale, bias_mix, out, ldo, out_batch_stride, M, N, rows_per_video, max_ctas,
                                      nullptr, 0, stream);
}

extern "C" int merv_concat_linear(const void* const* A, const int64_t* lda, const void* W, int64_t ldw, const int32_t* K, int nseg,
                                  const void* bias, void* out, int64_t ldo, int M, int N, void* stream) {
  MERV_REQUIRE(A && lda && W && K && out, MERV_E_ARG, "merv_concat_linear: NULL pointer");
  MERV_REQUIRE(nseg >= 1 && nseg <= MERV_MAX_SEGMENTS, MERV_E_ARG, "merv_concat_linear: nseg=%d not in [1,%d]", nseg, MERV_MAX_SEGMENTS);
  MERV_REQUIRE(M >= 0 && N > 0, MERV_E_SHAPE, "merv_concat_linear: M=%d N=%d", M, N);
  if (int rc = require_sm100()) return rc;
  if (M == 0) return MERV_OK;
  GemmSegment seg[MERV_MAX_SEGMENTS];
  long long k0 = 0;
  for (int s = 0; s < nseg; ++s) {
    MERV_REQUIRE(K[s] > 0 && K[s] % 8 == 0, MERV_E_ALIGN, "merv_concat_linear: K[%d]=%d must be a positive multiple of 8", s, K[s]);
    seg[s] = GemmSegment{A[s], lda[s], static_cast<const char*>(W) + k0 * 2, ldw, K[s]};  // column block k0 .. k0 + K_s of W
    k0 += K[s];
  }
  MERV_REQUIRE(ldw >= k0, MERV_E_SHAPE, "merv_concat_linear: ldw=%lld < sum K = %lld", (long long)ldw, k0);
  return launch_gemm_tcgen05(seg, nseg, nullptr, nullptr, M, bias, MERV_ACT_NONE, nullptr, nullptr, out, ldo, 0, M, N, 0,
                             static_cast<cudaStream_t>(stream));
}

// callers built against ABI v5 lay the descriptor out this way (LP64)
static_assert(sizeof(merv_fused_desc) == 744 && offsetof(merv_fused_desc, reserved_ptr_) == 728 && offsetof(merv_fused_desc, reserved_) == 736,
              "merv_fused_desc must keep its ABI v5 layout");

extern "C" int merv_fused_forward(const merv_fused_desc* d, void* stream) {
  MERV_REQUIRE(d != nullptr, MERV_E_ARG, "merv_fused_forward: desc is NULL");
  const int E = d->num_encoders;
  MERV_REQUIRE(E >= 1 && E <= MERV_MAX_SEGMENTS, MERV_E_ARG, "merv_fused_forward: num_encoders=%d not in [1,%d]", E, MERV_MAX_SEGMENTS);
  MERV_REQUIRE(d->B >= 0 && d->N > 0 && d->rows_per_video > 0, MERV_E_SHAPE, "merv_fused_forward: B=%d N=%d rows_per_video=%d", d->B, d->N,
               d->rows_per_video);
  MERV_REQUIRE(d->scores && d->weights && d->bias_mix && d->out, MERV_E_ARG, "merv_fused_forward: NULL workspace or output");
  if (d->B == 0) return MERV_OK;
  const void* A[MERV_MAX_SEGMENTS];
  int64_t lda[MERV_MAX_SEGMENTS];
  int32_t K[MERV_MAX_SEGMENTS];
  const float* partial[MERV_MAX_SEGMENTS];
  for (int e = 0; e < E; ++e) {
    const merv_pool_desc& p = d->pool[e];
    MERV_REQUIRE(p.T * p.S * p.S == d->rows_per_video, MERV_E_SHAPE, "merv_fused_forward: encoder %d emits %d tokens, expected %d", e,
                 p.T * p.S * p.S, d->rows_per_video);
    MERV_REQUIRE(p.score_vec && p.score_partial && d->parts[e] > 0, MERV_E_ARG, "merv_fused_forward: encoder %d needs score_vec / score_partial / parts", e);
    A[e] = p.y; lda[e] = p.y_row_stride; K[e] = p.C; partial[e] = p.score_partial;
  }
  // Three launches chained by programmatic dependent launch: the pool kernel releases its dependents at once, so the tiny
  // scores kernel is resident (blocked in griddepcontrol.wait) when the pool's last CTA retires, and the GEMM's CTAs run their
  // prologue (barriers, TMEM allocation, tensor-map prefetch) on every SM the pool has left — no launch gap between the stages.
  const bool pdl = pdl_enabled();
  if (int rc = merv_pool3d(d->pool, E, d->B, MERV_BF16, 0, stream)) return rc;
  if (int rc = launch_scores_softmax_weights(partial, d->parts, d->c, d->bias, d->scores, d->weights, d->weights_bf16, d->bias_mix, d->B, E,
                                             d->rows_per_video, d->N, static_cast<cudaStream_t>(stream), pdl))
    return rc;
  MERV_REQUIRE(d->B * (long long)d->rows_per_video <= 0x7fffffffLL, MERV_E_SHAPE, "merv_fused_forward: B * rows_per_video overflows");
  GemmSegment seg[MERV_MAX_SEGMENTS];
  for (int e = 0; e < E; ++e) seg[e] = GemmSegment{A[e], lda[e], d->W[e], d->ldw[e], K[e]};
  return launch_gemm_tcgen05(seg, E, d->weights, d->bias_mix, d->rows_per_video, nullptr, MERV_ACT_NONE, nullptr, nullptr, d->out, d->ldo,
                             d->out_batch_stride, d->B * d->rows_per_video, d->N, 0, static_cast<cudaStream_t>(stream), nullptr, 0, pdl);
}
