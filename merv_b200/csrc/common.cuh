// Shared helpers for libmerv_fusion.so (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdarg>
#include <cstdio>

#include "merv_fusion.h"

namespace merv {

// ---- host-side error plumbing -----------------------------------------------------------------------------
int fail(int code, const char* fmt, ...);

#define MERV_CUDA_OK(expr)                                                                            \
  do {                                                                                                \
    cudaError_t _e = (expr);                                                                          \
    if (_e != cudaSuccess) return ::merv::fail(MERV_E_CUDA, "%s failed: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

#define MERV_REQUIRE(cond, code, ...) \
  do {                                \
    if (!(cond)) return ::merv::fail(code, __VA_ARGS__); \
  } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
int require_sm100();   // MERV_OK or MERV_E_ARCH for the current device (cached per device)
int sm_count();        // SM count of the current device

struct AssistArgs;  // pool_assist.cuh
// Weight gradient over per-video segments (gemm_tcgen05.cu, kVid): the single (A, W) segment handed to launch_gemm_tcgen05 covers all
// `videos` x kblocks_per_video k-blocks; the kernel drains the accumulator once per video.
struct WgradVideoArgs {
  int videos, kblocks_per_video;
  const float* scale;      // scale[b * scale_stride] multiplies video b's contribution to the sum (NULL: 1)
  long long scale_stride;
  const void* W;           // [M, N] bf16, row stride ldw: <W, per-video product> is emitted per (video, tile, epilogue warp)
  long long ldw;
  float* dot_out;          // [videos, wgrad_video_parts(M, N)]
  int split;               // work items per tile: the videos in `split` contiguous ranges (1: no split, the result goes straight to Y)
  float* partial;          // [split, M, N] fp32 when split > 1
};
int wgrad_video_parts(int M, int N);
int wgrad_video_split(int M, int N, int videos);  // the split that fills the SMs best (1 if nothing is gained)
// one (A_s, W_s, K_s) product of the tcgen05 GEMM (see gemm_tcgen05.cu)
struct GemmSegment {
  const void* A;
  long long lda;
  const void* W;
  long long ldw;
  int K;
  // Operand majorness.  0 (default): K-major — A is [M, K] and W is [N, K] row-major, the contraction dimension contiguous.
  // 1: MN-major — the operand is given TRANSPOSED in memory, A as [K, M] / W as [K, N] row-major (ld = its row stride), i.e. the
  // M / N dimension contiguous.  tcgen05 reads either form straight from shared memory, so a weight gradient dW = dY^T X or an
  // input gradient dX = dY W needs no transposed copy of dY, X or W.
  int a_mn = 0, b_mn = 0;
};
// pdl: launch with programmatic stream serialization — the kernel's prologue (barrier init, TMEM allocation, tensor-map
// prefetch) may overlap the tail of the preceding kernel in the stream; it executes griddepcontrol.wait before touching global memory.
int launch_gemm_tcgen05(const GemmSegment* seg, int nseg, const float* seg_scale, const float* bias_rows, int rows_per_video,
                        const void* bias, int act, const float* rowdot_vec, float* rowdot_out, void* Y, long long ldy, long long y_batch_stride,
                        int M, int N, int max_ctas, cudaStream_t stream, void* const* extra_out = nullptr, int num_extra = 0, bool pdl = false,
                        void* mc_out = nullptr, const struct AssistArgs* assist = nullptr, const WgradVideoArgs* vid = nullptr);
int launch_scores_softmax_weights(const float* const* partial, const int32_t* count, const float* const* c, const void* const* bias,
                                  float* scores, float* weights, void* weights_bf16, float* bias_mix, int B, int E, int T, int N,
                                  cudaStream_t stream, bool pdl, int* sync_ws = nullptr, int sync_ints = 0);
// tcgen05 cross attention (attention_tcgen05.cu): bf16, at most 128 queries and 256 keys per frame, head_dim % 32 == 0 and <= 128
bool attention_tcgen05_supported(int n_q, int n_kv, int heads, int hd, long long ldq, long long q_batch_stride, long long ldkv, long long ldo);
int launch_attention_tcgen05(const void* q, long long ldq, long long q_batch_stride, const void* kv, long long ldkv, void* out, long long ldo,
                             int batches, int n_q, int n_kv, int heads, int hd, float scale, cudaStream_t stream);
// the tcgen05 backward's tile: bf16, n_q <= 64, n_kv <= 256, head_dim % 32 == 0 and <= 128 (false under MERV_ATTN_IMPL=simt).  Row
// alignment is not part of it: both backward kernels require 16-byte aligned rows.
bool attention_bwd_tcgen05_supported(int n_q, int n_kv, int hd);
int launch_attention_bwd_tcgen05(const void* q, long long ldq, long long q_batch_stride, const void* kv, long long ldkv, const void* dout, long long lddo,
                                 void* dq, long long lddq, void* dkv, long long lddkv, int batches, int n_q, int n_kv, int heads, int hd, float scale,
                                 cudaStream_t stream);
// MERV_PDL=0 disables programmatic dependent launch inside merv_fused_forward (A/B measurements); read per call
bool pdl_enabled();
int launch_gemm_simt(const void* A, long long lda, const void* W, long long ldw, const void* bias, void* Y, long long ldy,
                     int M, int N, int K, int act, int dtype, cudaStream_t s);

// ---- device helpers ---------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL).  pdl_launch_dependents(): the next kernel in the stream, if it was launched with
// programmatic stream serialization, may start being scheduled now (it still cannot read this grid's results before its own
// pdl_wait()).  pdl_wait(): blocks until every prerequisite grid has completed and its writes are visible; a no-op for a
// kernel launched without the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename T> struct VecTraits;
template <> struct VecTraits<__nv_bfloat16> { static constexpr int kVec = 8; };  // 16 bytes
template <> struct VecTraits<float> { static constexpr int kVec = 4; };          // 16 bytes

__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
// cached variant (lets L1 absorb the window overlap re-reads of the pool kernel)
__device__ __forceinline__ uint4 ldg_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_na_v4(void* p, const uint4& v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ float bf16_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}

// 16-byte vector <-> fp32 lanes
template <typename T> struct Vec16;
template <> struct Vec16<__nv_bfloat16> {
  static constexpr int kN = 8;
  __device__ static __forceinline__ void unpack(const uint4& r, float (&f)[8]) {
    f[0] = bf16_lo(r.x); f[1] = bf16_hi(r.x); f[2] = bf16_lo(r.y); f[3] = bf16_hi(r.y);
    f[4] = bf16_lo(r.z); f[5] = bf16_hi(r.z); f[6] = bf16_lo(r.w); f[7] = bf16_hi(r.w);
  }
  __device__ static __forceinline__ uint4 pack(const float (&f)[8]) {
    return make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
  }
};
template <> struct Vec16<float> {
  static constexpr int kN = 4;
  __device__ static __forceinline__ void unpack(const uint4& r, float (&f)[4]) {
    f[0] = __uint_as_float(r.x); f[1] = __uint_as_float(r.y); f[2] = __uint_as_float(r.z); f[3] = __uint_as_float(r.w);
  }
  __device__ static __forceinline__ uint4 pack(const float (&f)[4]) {
    return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3]));
  }
};

__device__ __forceinline__ float to_float(float v) { return v; }
__device__ __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// nn.GELU() default (approximate='none'): 0.5 x (1 + erf(x / sqrt 2))   [merv/util/nn_utils.py:48]
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }


// erf-GELU for the bf16 tensor-core epilogue: erf by Abramowitz & Stegun 7.1.26 (|error| <= 1.5e-7, far below one
// bf16 ulp of the output), branch-free, ~16 instructions instead of erff's two-branch polynomial.
__device__ __forceinline__ float gelu_erf_fast(float x) {
  const float z = x * 0.70710678118654752440f;
  const float az = fabsf(z);
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, az, 1.0f)));  // MUFU.RCP, ~1 ulp
  float poly = fmaf(1.061405429f, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  poly *= t;
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(az * az * -1.4426950408889634f));  // exp(-z^2), MUFU.EX2
  const float erf_abs = fmaf(-poly, e, 1.0f);
  return 0.5f * x * (1.0f + copysignf(erf_abs, z));
}

// Two erf-GELUs at once on Blackwell's packed fp32 pipe (FFMA2): the same A&S 7.1.26 evaluation as gelu_erf_fast with
// the 12 multiply-add steps done as f32x2 instructions; only |z|, the two MUFU ops and copysign stay scalar.  The tensor
// -core GEMM's activated epilogue is issue-bound, so instruction count is what matters here.
__device__ __forceinline__ unsigned long long f32x2_pack(float a, float b) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void f32x2_unpack(unsigned long long v, float& a, float& b) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ unsigned long long f32x2_fma(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ unsigned long long f32x2_mul(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
// 16-byte vector <-> packed fp32 pairs.  The streaming kernels (LayerNorm, pooling) turned out instruction-ISSUE bound before they
// were HBM-bound, so their arithmetic runs on Blackwell's packed fp32 pipe (fma.rn.f32x2: one instruction per two elements).
template <typename T> struct Pairs;
template <> struct Pairs<__nv_bfloat16> {
  static constexpr int kP = 4;
  __device__ static __forceinline__ void unpack(const uint4& r, unsigned long long (&x)[4]) {
    x[0] = f32x2_pack(bf16_lo(r.x), bf16_hi(r.x));
    x[1] = f32x2_pack(bf16_lo(r.y), bf16_hi(r.y));
    x[2] = f32x2_pack(bf16_lo(r.z), bf16_hi(r.z));
    x[3] = f32x2_pack(bf16_lo(r.w), bf16_hi(r.w));
  }
  __device__ static __forceinline__ uint4 pack(const unsigned long long (&x)[4]) {
    float a[4], b[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) f32x2_unpack(x[q], a[q], b[q]);
    return make_uint4(pack_bf16x2(a[0], b[0]), pack_bf16x2(a[1], b[1]), pack_bf16x2(a[2], b[2]), pack_bf16x2(a[3], b[3]));
  }
};
template <> struct Pairs<float> {
  static constexpr int kP = 2;
  __device__ static __forceinline__ void unpack(const uint4& r, unsigned long long (&x)[2]) {
    x[0] = f32x2_pack(__uint_as_float(r.x), __uint_as_float(r.y));
    x[1] = f32x2_pack(__uint_as_float(r.z), __uint_as_float(r.w));
  }
  __device__ static __forceinline__ uint4 pack(const unsigned long long (&x)[2]) {
    float a[2], b[2];
    f32x2_unpack(x[0], a[0], b[0]);
    f32x2_unpack(x[1], a[1], b[1]);
    return make_uint4(__float_as_uint(a[0]), __float_as_uint(b[0]), __float_as_uint(a[1]), __float_as_uint(b[1]));
  }
};
__device__ __forceinline__ void gelu_erf_fast2(float& x0, float& x1) {
#define MERV_C2(v) f32x2_pack(v, v)
  const unsigned long long x = f32x2_pack(x0, x1);
  const unsigned long long z = f32x2_mul(x, MERV_C2(0.70710678118654752440f));
  float z0, z1;
  f32x2_unpack(z, z0, z1);
  const unsigned long long den = f32x2_fma(MERV_C2(0.3275911f), f32x2_pack(fabsf(z0), fabsf(z1)), MERV_C2(1.0f));
  float d0, d1, t0, t1;
  f32x2_unpack(den, d0, d1);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t0) : "f"(d0));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t1) : "f"(d1));
  const unsigned long long t = f32x2_pack(t0, t1);
  // -poly(t): the coefficients carry the sign so that erf = 1 + (-poly) * exp(-z^2) is one FFMA2
  unsigned long long np = f32x2_fma(MERV_C2(-1.061405429f), t, MERV_C2(1.453152027f));
  np = f32x2_fma(np, t, MERV_C2(-1.421413741f));
  np = f32x2_fma(np, t, MERV_C2(0.284496736f));
  np = f32x2_fma(np, t, MERV_C2(-0.254829592f));
  np = f32x2_mul(np, t);
  const unsigned long long arg = f32x2_mul(f32x2_mul(z, MERV_C2(-1.4426950408889634f)), z);  // -z^2 log2(e)
  float a0, a1, e0, e1;
  f32x2_unpack(arg, a0, a1);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(a0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(a1));
  const unsigned long long erf_abs = f32x2_fma(np, f32x2_pack(e0, e1), MERV_C2(1.0f));
  float r0, r1;
  f32x2_unpack(erf_abs, r0, r1);
  const unsigned long long hx = f32x2_mul(x, MERV_C2(0.5f));
  const unsigned long long out = f32x2_fma(hx, f32x2_pack(copysignf(r0, z0), copysignf(r1, z1)), hx);
  f32x2_unpack(out, x0, x1);
#undef MERV_C2
}

}  // namespace merv
