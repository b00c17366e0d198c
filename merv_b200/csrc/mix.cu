// Encoder scores, softmax over encoders and the weighted mix of CrossAttentionAdapterLearnableQuery.forward
// (reference merv/util/nn_utils.py:487-521), restated through the identity of SURVEY.md §3.3:
//     weights[b,:] = softmax_e(u . mean_t V[b,e,t,:]),   u = Wk^T (Wq Q^T + b_q) / sqrt(embed)
// (b_k adds a per-row constant that cancels in the softmax; Wv, b_v and out_proj never reach an output).
// All reductions use a fixed order (no float atomics) so results are bit-reproducible per video, independent
// of batch size and of how the batch is sharded across GPUs.
#include "common.cuh"

namespace merv {

// block-wide sum with a fixed reduction tree; result valid in every thread
template <int kThreads>
__device__ __forceinline__ float block_sum(float v, float* smem /* >= 32 floats */) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  float r = (lane < kThreads / 32) ? smem[lane] : 0.f;
  r = warp_sum(r);
  return r;
}

// ---- u = Wk^T (Wq Q^T + b_q) / sqrt(embed) --------------------------------------------------------------
// q[d] = sum_j Wq[d,j] Q[j] + b_q[d] : one warp per row, coalesced along j
template <typename T>
__global__ void __launch_bounds__(256) qproj_kernel(const T* __restrict__ Wq, const T* __restrict__ Q,
                                                    const T* __restrict__ bias, float* __restrict__ q, int embed) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= embed) return;
  const int lane = threadIdx.x & 31;
  const T* w = Wq + (long long)row * embed;
  float acc = 0.f;
  for (int j = lane; j < embed; j += 32) acc += to_float(w[j]) * to_float(Q[j]);
  acc = warp_sum(acc);
  if (lane == 0) q[row] = acc + (bias ? to_float(bias[row]) : 0.f);
}

// out[k] = scale * sum_d W[d,k] * x[d]  (W row-major [D, K], leading dimension ldw): 32 columns x 8 row-lanes
template <typename T>
__global__ void __launch_bounds__(256) gemv_t_kernel(const T* __restrict__ W, long long ldw, const float* __restrict__ x,
                                                     float* __restrict__ out, int D, int K, float scale) {
  __shared__ float part[8][33];
  const int kx = threadIdx.x & 31, dy = threadIdx.x >> 5;
  const int k = blockIdx.x * 32 + kx;
  float acc = 0.f;
  if (k < K)
    for (int d = dy; d < D; d += 8) acc += to_float(W[(long long)d * ldw + k]) * x[d];
  part[dy][kx] = acc;
  __syncthreads();
  if (dy == 0 && k < K) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += part[i][kx];
    out[k] = s * scale;
  }
}

// Two-stage form for narrow outputs (K / 32 CTAs of the kernel above cannot fill the GPU: W_e^T u has K = C_e = 768..1024):
// stage 1: CTA = (256-byte column block, block of rows), 16-byte loads, 8 row lanes reduced in fixed order -> partial[row block, k]
// stage 2: out[k] = scale * sum over the row blocks (fixed order).  Deterministic like the single-stage kernel.
constexpr int kGemvTRows = 64;  // rows per CTA
template <typename T>
__global__ void __launch_bounds__(256) gemv_t_partial_kernel(const T* __restrict__ W, long long ldw, const float* __restrict__ x,
                                                             float* __restrict__ partial, int D, int K) {
  constexpr int VEC = Vec16<T>::kN;
  __shared__ float part[8][32 * VEC + 1];
  const int cv = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int k0 = (blockIdx.x * 32 + cv) * VEC;
  const int d0 = blockIdx.y * kGemvTRows, d1 = min(D, d0 + kGemvTRows);
  float acc[VEC];
#pragma unroll
  for (int c = 0; c < VEC; ++c) acc[c] = 0.f;
  if (k0 < K) {
    for (int d = d0 + rl; d < d1; d += 8) {
      float w[VEC];
      Vec16<T>::unpack(ldg_nc_v4(W + (long long)d * ldw + k0), w);
      const float xd = x[d];
#pragma unroll
      for (int c = 0; c < VEC; ++c) acc[c] = fmaf(w[c], xd, acc[c]);
    }
  }
#pragma unroll
  for (int c = 0; c < VEC; ++c) part[rl][cv * VEC + c] = acc[c];
  __syncthreads();
  for (int i = threadIdx.x; i < 32 * VEC; i += 256) {
    const int k = blockIdx.x * 32 * VEC + i;
    if (k < K) {
      float sum = 0.f;
#pragma unroll
      for (int g = 0; g < 8; ++g) sum += part[g][i];
      partial[(long long)blockIdx.y * K + k] = sum;
    }
  }
}
__global__ void __launch_bounds__(256) gemv_t_final_kernel(const float* __restrict__ partial, float* __restrict__ out, int K, int nblocks, float scale) {
  const int k = blockIdx.x * 256 + threadIdx.x;
  if (k >= K) return;
  float sum = 0.f;
  for (int b = 0; b < nblocks; ++b) sum += partial[(long long)b * K + k];
  out[k] = sum * scale;
}

// floats of workspace the two-stage form needs for a [D, K] matrix; 0 = the single-stage kernel already fills the GPU (wide K)
static size_t gemv_t_workspace(int D, int K) {
  if (D <= 0 || K <= 0 || (K + 31) / 32 >= 4 * sm_count()) return 0;
  return (size_t)((D + kGemvTRows - 1) / kGemvTRows) * (size_t)K;
}

template <typename T>
static void launch_gemv_t(const T* W, long long ldw, const float* x, float* out, int D, int K, float scale, float* workspace, size_t workspace_floats,
                          cudaStream_t s) {
  constexpr int VEC = Vec16<T>::kN;
  const size_t need = gemv_t_workspace(D, K);
  if (need > 0 && workspace != nullptr && workspace_floats >= need && K % VEC == 0 && ldw % VEC == 0 && aligned16(W)) {
    const int nblocks = (D + kGemvTRows - 1) / kGemvTRows;
    gemv_t_partial_kernel<T><<<dim3((K / VEC + 31) / 32, nblocks), 256, 0, s>>>(W, ldw, x, workspace, D, K);
    gemv_t_final_kernel<<<(K + 255) / 256, 256, 0, s>>>(workspace, out, K, nblocks, scale);
  } else {
    gemv_t_kernel<T><<<(K + 31) / 32, 256, 0, s>>>(W, ldw, x, out, D, K, scale);
  }
}

// c = sum_n u[n] * bias[n]
template <typename T>
__global__ void __launch_bounds__(256) dot_kernel(const T* __restrict__ bias, const float* __restrict__ u, float* __restrict__ c, int N) {
  __shared__ float red[32];
  float acc = 0.f;
  if (bias != nullptr)
    for (int n = threadIdx.x; n < N; n += 256) acc += u[n] * to_float(bias[n]);
  acc = block_sum<256>(acc, red);
  if (threadIdx.x == 0) *c = acc;
}

// ---- scores from the projected tokens themselves ----------------------------------------------------------
struct TokenScoreParams {
  const void* V[MERV_MAX_ENCODERS];
  int tokens[MERV_MAX_ENCODERS];
};

// partial[(b*E+e)*chunks + chunk] = sum_{t in chunk} sum_k u[t * u_stride + k] * V_e[b,t,k]
//   u_stride == 0, full == 0 : the averagetoken=True branch (nn_utils.py:507-512) — one u for every token, T_e in {T, 1} tokens summed
//   u_stride == K, full == 1 : the averagetoken=False branch (nn_utils.py:514-518) — key = the flattened [T*K] tokens, so u has one
//                              row per token and a single-token encoder is read T times (its repeat at nn_utils.py:502)
template <typename T>
__global__ void __launch_bounds__(256) token_score_kernel(const __grid_constant__ TokenScoreParams p, const float* __restrict__ u,
                                                          float* __restrict__ partial, int E, int K, int chunks, int Ttok,
                                                          long long u_stride, int full) {
  constexpr int VEC = Vec16<T>::kN;
  __shared__ float red[32];
  const int chunk = blockIdx.x, e = blockIdx.y, b = blockIdx.z;
  const int Te = p.tokens[e];
  const int Tl = full ? Ttok : Te;
  const int per = (Tl + chunks - 1) / chunks;
  const int t0 = chunk * per, t1 = min(Tl, t0 + per);
  const T* base = static_cast<const T*>(p.V[e]) + (long long)b * Te * K;
  const int nvec = K / VEC;
  float acc = 0.f;
  for (int t = t0; t < t1; ++t) {
    const T* row = base + (long long)(Te == 1 ? 0 : t) * K;
    const float* ut = u + (long long)t * u_stride;
    for (int v = threadIdx.x; v < nvec; v += 256) {
      float x[VEC];
      Vec16<T>::unpack(ldg_nc_v4(row + v * VEC), x);
      const float4* uu = reinterpret_cast<const float4*>(ut + v * VEC);
#pragma unroll
      for (int c = 0; c < VEC; c += 4) {
        const float4 w = uu[c / 4];
        acc += x[c] * w.x + x[c + 1] * w.y + x[c + 2] * w.z + x[c + 3] * w.w;
      }
    }
  }
  acc = block_sum<256>(acc, red);
  if (threadIdx.x == 0) partial[((long long)b * E + e) * chunks + chunk] = acc;
}

// scores[b,e] = (sum of n contiguous partials) * inv[e] (+ c[e])  — one warp per (b,e), fixed order
struct ScaleParams {
  float inv[MERV_MAX_ENCODERS];
};
__global__ void __launch_bounds__(32) reduce_scale_kernel(const float* __restrict__ partial, float* __restrict__ scores,
                                                          const __grid_constant__ ScaleParams sp, const float* __restrict__ c, int n, int E) {
  const long long id = blockIdx.x;
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += 32) acc += partial[id * n + i];
  acc = warp_sum(acc);
  if (threadIdx.x == 0) {
    const float r = acc * sp.inv[id % E];
    scores[id] = c != nullptr ? r + c[id % E] : r;
  }
}

// c_out[e] = u . pe[e,:] (+ *c_in[e]) : the additive score constants of positional_embedding=True (nn_utils.py:510-511)
struct ConstParams {
  const float* c_in[MERV_MAX_ENCODERS];
};
template <typename T>
__global__ void __launch_bounds__(256) score_const_kernel(const T* __restrict__ pe, long long ldpe, const float* __restrict__ u,
                                                          const __grid_constant__ ConstParams cp, float* __restrict__ c_out, int K) {
  __shared__ float red[32];
  const int e = blockIdx.x;
  const T* row = pe + (long long)e * ldpe;
  float acc = 0.f;
  for (int k = threadIdx.x; k < K; k += 256) acc += u[k] * to_float(row[k]);
  acc = block_sum<256>(acc, red);
  if (threadIdx.x == 0) c_out[e] = acc + (cp.c_in[e] != nullptr ? *cp.c_in[e] : 0.f);
}

// ---- scores from partial dot products (pool kernel's score_partial / GEMM epilogue's rowdot_out) ----------
struct PartialParams {
  const float* p[MERV_MAX_ENCODERS];
  const float* c[MERV_MAX_ENCODERS];
  int count[MERV_MAX_ENCODERS];
};

// scores[b,e] = (1/T) * sum_{i<count[e]} partial_e[b*count[e] + i] + c_e   (fixed order -> deterministic)
__global__ void __launch_bounds__(256) partial_score_kernel(const __grid_constant__ PartialParams p, float* __restrict__ scores, int E, int T) {
  __shared__ float red[32];
  const int e = blockIdx.x, b = blockIdx.y;
  const int n = p.count[e];
  const float* src = p.p[e] + (long long)b * n;
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) acc += src[i];
  acc = block_sum<256>(acc, red);
  if (threadIdx.x == 0) scores[(long long)b * E + e] = acc / float(T) + (p.c[e] ? *p.c[e] : 0.f);
}

// ---- softmax over the E encoders with warp shuffles ----
// lane e (< E) passes its score; every lane gets the weight of lane e back in the same lane
__device__ __forceinline__ float warp_softmax_over_encoders(float score, int lane, int E) {
  const float s = lane < E ? score : -INFINITY;
  const float m = warp_max(s);
  const float ex = lane < E ? expf(s - m) : 0.f;
  const float den = warp_sum(ex);
  return ex / den;
}

struct BiasParams {
  const void* bias[MERV_MAX_ENCODERS];
};

// weights[b,:] = softmax(scores[b,:]);  bias_mix[b,n] = sum_e weights[b,e] * bias_e[n]
template <typename T>
__global__ void __launch_bounds__(256) softmax_weights_kernel(const float* __restrict__ scores, float* __restrict__ weights,
                                                              __nv_bfloat16* __restrict__ weights_bf16,
                                                              const __grid_constant__ BiasParams bp, float* __restrict__ bias_mix,
                                                              int E, int N) {
  const int b = blockIdx.y, lane = threadIdx.x & 31;
  const float w = warp_softmax_over_encoders(lane < E ? scores[(long long)b * E + lane] : 0.f, lane, E);
  if (blockIdx.x == 0 && threadIdx.x < E) {
    weights[(long long)b * E + threadIdx.x] = w;
    if (weights_bf16 != nullptr) weights_bf16[(long long)b * E + threadIdx.x] = __float2bfloat16_rn(w);
  }
  if (bias_mix == nullptr) return;
  const int n = blockIdx.x * 256 + threadIdx.x;
  float acc = 0.f;
  for (int e = 0; e < E; ++e) {
    const float we = __shfl_sync(0xffffffffu, w, e);
    const T* be = static_cast<const T*>(bp.bias[e]);
    if (be != nullptr && n < N) acc += we * to_float(be[n]);
  }
  if (n < N) bias_mix[(long long)b * N + n] = acc;
}

// scores -> softmax -> weights (+ bf16 copy) -> bias_mix in ONE launch (small-batch latency: merv_fused_forward).  The
// score reduction repeats partial_score_kernel's exact summation order in every block, so the results are bit-identical
// to the two-kernel sequence.
template <typename T>
__global__ void __launch_bounds__(256) scores_softmax_kernel(const __grid_constant__ PartialParams pp, const __grid_constant__ BiasParams bp,
                                                             float* __restrict__ scores, float* __restrict__ weights,
                                                             __nv_bfloat16* __restrict__ weights_bf16, float* __restrict__ bias_mix, int E,
                                                             int Ttok, int N) {
  __shared__ float red[32];
  __shared__ float sc[MERV_MAX_ENCODERS];
  const int b = blockIdx.y, lane = threadIdx.x & 31;
  pdl_launch_dependents();  // the GEMM behind this kernel may start its prologue now
  pdl_wait();               // the pool kernel's score partials are complete and visible
  for (int e = 0; e < E; ++e) {
    const int n = pp.count[e];
    const float* src = pp.p[e] + (long long)b * n;
    float acc = 0.f;
    for (int i = threadIdx.x; i < n; i += 256) acc += src[i];
    acc = block_sum<256>(acc, red);
    if (threadIdx.x == 0) sc[e] = acc / float(Ttok) + (pp.c[e] ? *pp.c[e] : 0.f);
  }
  __syncthreads();
  const float w = warp_softmax_over_encoders(lane < E ? sc[lane] : 0.f, lane, E);
  if (blockIdx.x == 0 && threadIdx.x < E) {
    scores[(long long)b * E + threadIdx.x] = sc[threadIdx.x];
    weights[(long long)b * E + threadIdx.x] = w;
    if (weights_bf16 != nullptr) weights_bf16[(long long)b * E + threadIdx.x] = __float2bfloat16_rn(w);
  }
  const int nn = blockIdx.x * 256 + threadIdx.x;
  float acc = 0.f;
  for (int e = 0; e < E; ++e) {
    const float we = __shfl_sync(0xffffffffu, w, e);
    const T* be = static_cast<const T*>(bp.bias[e]);
    if (be != nullptr && nn < N) acc += we * to_float(be[nn]);
  }
  if (nn < N) bias_mix[(long long)b * N + nn] = acc;
}

// ---- out[b,t,:] = sum_e w[b,e] * V_e[b,t,:]  (HBM-bound: E reads + 1 write per element, each exactly once) --
struct MixParams {
  const void* V[MERV_MAX_ENCODERS];
  int tokens[MERV_MAX_ENCODERS];  // T or 1 (broadcast, nn_utils.py:502)
};

template <typename T, int E>
__global__ void __launch_bounds__(256) softmax_mix_kernel(const __grid_constant__ MixParams p, const float* __restrict__ scores,
                                                          float* __restrict__ weights, T* __restrict__ out, long long ldo, long long obs, int Ttok,
                                                          int K) {
  constexpr int VEC = Vec16<T>::kN;
  const int b = blockIdx.y, lane = threadIdx.x & 31;
  float wl;
  if (scores != nullptr) {
    wl = warp_softmax_over_encoders(lane < E ? scores[(long long)b * E + lane] : 0.f, lane, E);
    if (blockIdx.x == 0 && threadIdx.x < E) weights[(long long)b * E + threadIdx.x] = wl;
  } else {
    wl = lane < E ? weights[(long long)b * E + lane] : 0.f;
  }
  float w[E];
  const T* src[E];
  long long tstride[E];
#pragma unroll
  for (int e = 0; e < E; ++e) {
    w[e] = __shfl_sync(0xffffffffu, wl, e);
    const int Te = p.tokens[e];
    src[e] = static_cast<const T*>(p.V[e]) + (long long)b * Te * K;
    tstride[e] = Te == 1 ? 0 : K;
  }
  const int kvec = K / VEC;
  const long long nvec = (long long)Ttok * kvec;
  T* ob = out + (long long)b * obs;
  const long long stride = (long long)gridDim.x * 256;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < nvec; i += 2 * stride) {
    const long long i2 = i + stride;
    const bool has2 = i2 < nvec;
    const long long t1 = i / kvec, t2 = has2 ? i2 / kvec : 0;
    const int c1 = int(i - t1 * kvec) * VEC, c2 = has2 ? int(i2 - t2 * kvec) * VEC : 0;
    uint4 r1[E], r2[E];
#pragma unroll
    for (int e = 0; e < E; ++e) r1[e] = ldg_nc_v4(src[e] + t1 * tstride[e] + c1);
    if (has2) {
#pragma unroll
      for (int e = 0; e < E; ++e) r2[e] = ldg_nc_v4(src[e] + t2 * tstride[e] + c2);
    }
    float acc[VEC];
#pragma unroll
    for (int c = 0; c < VEC; ++c) acc[c] = 0.f;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      float x[VEC];
      Vec16<T>::unpack(r1[e], x);
#pragma unroll
      for (int c = 0; c < VEC; ++c) acc[c] = fmaf(w[e], x[c], acc[c]);
    }
    stg_na_v4(ob + t1 * ldo + c1, Vec16<T>::pack(acc));
    if (has2) {
#pragma unroll
      for (int c = 0; c < VEC; ++c) acc[c] = 0.f;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        float x[VEC];
        Vec16<T>::unpack(r2[e], x);
#pragma unroll
        for (int c = 0; c < VEC; ++c) acc[c] = fmaf(w[e], x[c], acc[c]);
      }
      stg_na_v4(ob + t2 * ldo + c2, Vec16<T>::pack(acc));
    }
  }
}

template <typename T>
static int launch_mix(const MixParams& p, const float* scores, float* weights, void* out, long long ldo, long long obs, int B, int E, int Ttok,
                      int K, cudaStream_t s) {
  constexpr int VEC = Vec16<T>::kN;
  const long long nvec = (long long)Ttok * (K / VEC);
  // ~8 waves of 256-thread CTAs in total across the batch, at least 1 and at most what the video needs
  long long per_video = (nvec + 511) / 512;
  long long want = (long long)sm_count() * 8 * 8 / (B > 0 ? B : 1);
  if (want < 1) want = 1;
  const int gx = int(per_video < want ? per_video : want);
  dim3 grid(gx, B);
  T* o = static_cast<T*>(out);
  switch (E) {
#define MERV_MIX_CASE(n) \
  case n: softmax_mix_kernel<T, n><<<grid, 256, 0, s>>>(p, scores, weights, o, ldo, obs, Ttok, K); break;
    MERV_MIX_CASE(1) MERV_MIX_CASE(2) MERV_MIX_CASE(3) MERV_MIX_CASE(4) MERV_MIX_CASE(5) MERV_MIX_CASE(6) MERV_MIX_CASE(7) MERV_MIX_CASE(8)
#undef MERV_MIX_CASE
    default: return fail(MERV_E_ARG, "merv_softmax_mix: E=%d not in [1,%d]", E, MERV_MAX_ENCODERS);
  }
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

}  // namespace merv

using namespace merv;

#define MERV_DTYPE_OK(fn) MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, fn ": unknown dtype %d", dtype)

extern "C" size_t merv_gemv_t_workspace(int D, int K) { return gemv_t_workspace(D, K); }

extern "C" int merv_fusion_query_vec(const void* Q, const void* Wq, const void* Wk, const void* in_proj_bias, float* u,
                                     float* workspace, size_t workspace_floats, int embed, int llm_dim, int dtype, void* stream) {
  MERV_DTYPE_OK("merv_fusion_query_vec");
  MERV_REQUIRE(Q && Wq && Wk && u && workspace, MERV_E_ARG, "merv_fusion_query_vec: NULL pointer");
  MERV_REQUIRE(embed > 0 && llm_dim > 0, MERV_E_SHAPE, "merv_fusion_query_vec: embed=%d llm_dim=%d", embed, llm_dim);
  MERV_REQUIRE(workspace_floats >= (size_t)embed, MERV_E_ARG, "merv_fusion_query_vec: workspace holds %zu floats, need >= %d", workspace_floats, embed);
  if (int rc = require_sm100()) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const float scale = 1.0f / sqrtf(float(embed));
  // q in the first `embed` floats (rounded up to a 16-byte boundary), the rest is the two-stage workspace of Wk^T q
  const size_t qpad = ((size_t)embed + 3) & ~(size_t)3;
  float* rest = workspace_floats > qpad ? workspace + qpad : nullptr;
  const size_t rest_floats = workspace_floats > qpad ? workspace_floats - qpad : 0;
  if (dtype == MERV_BF16) {
    using T = __nv_bfloat16;
    qproj_kernel<T><<<(embed + 7) / 8, 256, 0, s>>>((const T*)Wq, (const T*)Q, (const T*)in_proj_bias, workspace, embed);
    launch_gemv_t<T>((const T*)Wk, llm_dim, workspace, u, embed, llm_dim, scale, rest, rest_floats, s);
  } else {
    using T = float;
    qproj_kernel<T><<<(embed + 7) / 8, 256, 0, s>>>((const T*)Wq, (const T*)Q, (const T*)in_proj_bias, workspace, embed);
    launch_gemv_t<T>((const T*)Wk, llm_dim, workspace, u, embed, llm_dim, scale, rest, rest_floats, s);
  }
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

extern "C" int merv_affine_score_vec(const void* W, int64_t ldw, const void* bias, const float* u, float* v, float* c, float* workspace,
                                     size_t workspace_floats, int N, int K, int dtype, void* stream) {
  MERV_DTYPE_OK("merv_affine_score_vec");
  MERV_REQUIRE(W && u && v && c, MERV_E_ARG, "merv_affine_score_vec: NULL pointer");
  MERV_REQUIRE(N > 0 && K > 0 && ldw >= K, MERV_E_SHAPE, "merv_affine_score_vec: N=%d K=%d ldw=%lld", N, K, (long long)ldw);
  if (int rc = require_sm100()) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dtype == MERV_BF16) {
    using T = __nv_bfloat16;
    launch_gemv_t<T>((const T*)W, ldw, u, v, N, K, 1.0f, workspace, workspace_floats, s);
    dot_kernel<T><<<1, 256, 0, s>>>((const T*)bias, u, c, N);
  } else {
    using T = float;
    launch_gemv_t<T>((const T*)W, ldw, u, v, N, K, 1.0f, workspace, workspace_floats, s);
    dot_kernel<T><<<1, 256, 0, s>>>((const T*)bias, u, c, N);
  }
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

static int token_score_chunks(int T) { return T < 32 ? T : 32; }

extern "C" size_t merv_scores_from_tokens_workspace(int B, int E, int T, int K) {
  (void)K;
  if (B <= 0 || E <= 0 || T <= 0) return 0;
  return (size_t)B * E * token_score_chunks(T);
}

extern "C" int merv_scores_from_tokens_ex(const void* const* V, const int32_t* tokens, const float* u, int64_t u_token_stride,
                                          const float* c, int mean, float* scores, float* workspace, size_t workspace_floats, int B,
                                          int E, int T, int K, int dtype, void* stream) {
  MERV_DTYPE_OK("merv_scores_from_tokens");
  MERV_REQUIRE(V && tokens && u && scores && workspace, MERV_E_ARG, "merv_scores_from_tokens: NULL pointer");
  MERV_REQUIRE(E >= 1 && E <= MERV_MAX_ENCODERS, MERV_E_ARG, "merv_scores_from_tokens: E=%d", E);
  MERV_REQUIRE(B >= 0 && T > 0 && K > 0, MERV_E_SHAPE, "merv_scores_from_tokens: B=%d T=%d K=%d", B, T, K);
  const int vec = dtype == MERV_BF16 ? 8 : 4;
  MERV_REQUIRE(K % vec == 0, MERV_E_SHAPE, "merv_scores_from_tokens: K=%d must be a multiple of %d", K, vec);
  MERV_REQUIRE(u_token_stride == 0 || u_token_stride >= K, MERV_E_SHAPE, "merv_scores_from_tokens: u_token_stride=%lld (0 or >= K)",
               (long long)u_token_stride);
  MERV_REQUIRE(aligned16(u) && u_token_stride % 4 == 0, MERV_E_ALIGN, "merv_scores_from_tokens: u rows must be 16-byte aligned");
  MERV_REQUIRE(workspace_floats >= merv_scores_from_tokens_workspace(B, E, T, K), MERV_E_ARG,
               "merv_scores_from_tokens: workspace too small");
  if (int rc = require_sm100()) return rc;
  if (B == 0) return MERV_OK;
  const int full = u_token_stride != 0;  // one u row per token: every encoder contributes T terms (single-token ones repeated)
  TokenScoreParams p;
  ScaleParams sp;
  for (int e = 0; e < E; ++e) {
    MERV_REQUIRE(V[e] && aligned16(V[e]), MERV_E_ALIGN, "merv_scores_from_tokens: V[%d] NULL or not 16-byte aligned", e);
    // reference assert (nn_utils.py:494-495): every encoder has token_length tokens, or exactly 1
    MERV_REQUIRE(tokens[e] == T || tokens[e] == 1, MERV_E_SHAPE, "merv_scores_from_tokens: encoder %d has %d tokens, expected %d or 1",
                 e, tokens[e], T);
    p.V[e] = V[e];
    p.tokens[e] = tokens[e];
    sp.inv[e] = mean ? 1.0f / float(full ? T : tokens[e]) : 1.0f;
  }
  const int chunks = token_score_chunks(T);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  dim3 grid(chunks, E, B);
  if (dtype == MERV_BF16)
    token_score_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(p, u, workspace, E, K, chunks, T, u_token_stride, full);
  else
    token_score_kernel<float><<<grid, 256, 0, s>>>(p, u, workspace, E, K, chunks, T, u_token_stride, full);
  reduce_scale_kernel<<<B * E, 32, 0, s>>>(workspace, scores, sp, c, chunks, E);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

extern "C" int merv_scores_from_tokens(const void* const* V, const int32_t* tokens, const float* u, float* scores,
                                       float* workspace, size_t workspace_floats, int B, int E, int T, int K, int dtype,
                                       void* stream) {
  return merv_scores_from_tokens_ex(V, tokens, u, 0, nullptr, 1, scores, workspace, workspace_floats, B, E, T, K, dtype, stream);
}

extern "C" int merv_score_consts(const void* pe, int64_t ldpe, const float* u, const float* const* c_in, float* c_out, int E, int K,
                                 int dtype, void* stream) {
  MERV_DTYPE_OK("merv_score_consts");
  MERV_REQUIRE(pe && u && c_out, MERV_E_ARG, "merv_score_consts: NULL pointer");
  MERV_REQUIRE(E >= 1 && E <= MERV_MAX_ENCODERS, MERV_E_ARG, "merv_score_consts: E=%d", E);
  MERV_REQUIRE(K > 0 && ldpe >= K, MERV_E_SHAPE, "merv_score_consts: K=%d ldpe=%lld", K, (long long)ldpe);
  if (int rc = require_sm100()) return rc;
  ConstParams cp = {};
  for (int e = 0; e < E; ++e) cp.c_in[e] = c_in ? c_in[e] : nullptr;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dtype == MERV_BF16)
    score_const_kernel<__nv_bfloat16><<<E, 256, 0, s>>>((const __nv_bfloat16*)pe, ldpe, u, cp, c_out, K);
  else
    score_const_kernel<float><<<E, 256, 0, s>>>((const float*)pe, ldpe, u, cp, c_out, K);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

extern "C" int merv_scores_from_partials(const float* const* partial, const int32_t* count, const float* const* c, float* scores,
                                         int B, int E, int T, void* stream) {
  MERV_REQUIRE(partial && count && scores, MERV_E_ARG, "merv_scores_from_partials: NULL pointer");
  MERV_REQUIRE(E >= 1 && E <= MERV_MAX_ENCODERS, MERV_E_ARG, "merv_scores_from_partials: E=%d", E);
  MERV_REQUIRE(B >= 0 && T > 0, MERV_E_SHAPE, "merv_scores_from_partials: B=%d T=%d", B, T);
  if (int rc = require_sm100()) return rc;
  if (B == 0) return MERV_OK;
  PartialParams p = {};
  for (int e = 0; e < E; ++e) {
    MERV_REQUIRE(partial[e] && count[e] > 0, MERV_E_ARG, "merv_scores_from_partials: encoder %d: NULL partials or count=%d", e, count[e]);
    p.p[e] = partial[e];
    p.c[e] = c ? c[e] : nullptr;
    p.count[e] = count[e];
  }
  partial_score_kernel<<<dim3(E, B), 256, 0, static_cast<cudaStream_t>(stream)>>>(p, scores, E, T);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

extern "C" int merv_softmax_weights_ex(const float* scores, float* weights, void* weights_bf16, const void* const* bias,
                                       float* bias_mix, int B, int E, int N, int dtype, void* stream);
extern "C" int merv_softmax_weights(const float* scores, float* weights, const void* const* bias, float* bias_mix, int B,
                                    int E, int N, int dtype, void* stream) {
  return merv_softmax_weights_ex(scores, weights, nullptr, bias, bias_mix, B, E, N, dtype, stream);
}

extern "C" int merv_softmax_weights_ex(const float* scores, float* weights, void* weights_bf16, const void* const* bias,
                                       float* bias_mix, int B, int E, int N, int dtype, void* stream) {
  MERV_DTYPE_OK("merv_softmax_weights");
  MERV_REQUIRE(scores && weights, MERV_E_ARG, "merv_softmax_weights: NULL pointer");
  MERV_REQUIRE(E >= 1 && E <= MERV_MAX_ENCODERS, MERV_E_ARG, "merv_softmax_weights: E=%d", E);
  MERV_REQUIRE(B >= 0 && (bias_mix == nullptr || N > 0), MERV_E_SHAPE, "merv_softmax_weights: B=%d N=%d", B, N);
  if (int rc = require_sm100()) return rc;
  if (B == 0) return MERV_OK;
  BiasParams bp = {};
  if (bias_mix != nullptr) {
    MERV_REQUIRE(bias != nullptr, MERV_E_ARG, "merv_softmax_weights: bias_mix requested but bias is NULL");
    for (int e = 0; e < E; ++e) bp.bias[e] = bias[e];
  }
  const int gx = bias_mix ? (N + 255) / 256 : 1;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dtype == MERV_BF16)
    softmax_weights_kernel<__nv_bfloat16><<<dim3(gx, B), 256, 0, s>>>(scores, weights, static_cast<__nv_bfloat16*>(weights_bf16), bp, bias_mix, E, N);
  else
    softmax_weights_kernel<float><<<dim3(gx, B), 256, 0, s>>>(scores, weights, static_cast<__nv_bfloat16*>(weights_bf16), bp, bias_mix, E, N);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

// out video b's rows start at out + b * out_batch_stride, rows ldo apart: the fused tokens go straight into the prefix slot of the
// [B, L + T, K] multimodal embedding buffer.  Nothing outside the [B, T, K] block is written.  ldo == K, out_batch_stride == T * K is
// merv_softmax_mix (the same kernel, bit-identical).
extern "C" int merv_softmax_mix_ex(const void* const* V, const int32_t* tokens, const float* scores, float* weights, void* out, int64_t ldo,
                                   int64_t out_batch_stride, int B, int E, int T, int K, int dtype, void* stream) {
  MERV_DTYPE_OK("merv_softmax_mix");
  MERV_REQUIRE(V && tokens && weights && out, MERV_E_ARG, "merv_softmax_mix: NULL pointer");
  MERV_REQUIRE(E >= 1 && E <= MERV_MAX_ENCODERS, MERV_E_ARG, "merv_softmax_mix: E=%d not in [1,%d]", E, MERV_MAX_ENCODERS);
  MERV_REQUIRE(B >= 0 && T > 0 && K > 0, MERV_E_SHAPE, "merv_softmax_mix: B=%d T=%d K=%d", B, T, K);
  const int vec = dtype == MERV_BF16 ? 8 : 4;
  MERV_REQUIRE(K % vec == 0, MERV_E_SHAPE, "merv_softmax_mix: K=%d must be a multiple of %d", K, vec);
  MERV_REQUIRE(aligned16(out), MERV_E_ALIGN, "merv_softmax_mix: out not 16-byte aligned");
  MERV_REQUIRE(ldo % vec == 0 && out_batch_stride % vec == 0, MERV_E_ALIGN,
               "merv_softmax_mix_ex: ldo=%lld / out_batch_stride=%lld must be whole 16-byte vectors", (long long)ldo, (long long)out_batch_stride);
  MERV_REQUIRE(ldo >= K && out_batch_stride >= (int64_t)T * ldo, MERV_E_SHAPE,
               "merv_softmax_mix_ex: ldo=%lld < K or out_batch_stride=%lld < T * ldo (rows or videos would overlap)", (long long)ldo,
               (long long)out_batch_stride);
  if (int rc = require_sm100()) return rc;
  if (B == 0) return MERV_OK;
  MixParams p;
  for (int e = 0; e < E; ++e) {
    MERV_REQUIRE(V[e] && aligned16(V[e]), MERV_E_ALIGN, "merv_softmax_mix: V[%d] NULL or not 16-byte aligned", e);
    MERV_REQUIRE(tokens[e] == T || tokens[e] == 1, MERV_E_SHAPE, "merv_softmax_mix: encoder %d has %d tokens, expected %d or 1", e,
                 tokens[e], T);
    p.V[e] = V[e];
    p.tokens[e] = tokens[e];
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dtype == MERV_BF16) return launch_mix<__nv_bfloat16>(p, scores, weights, out, ldo, out_batch_stride, B, E, T, K, s);
  return launch_mix<float>(p, scores, weights, out, ldo, out_batch_stride, B, E, T, K, s);
}

extern "C" int merv_softmax_mix(const void* const* V, const int32_t* tokens, const float* scores, float* weights, void* out,
                                int B, int E, int T, int K, int dtype, void* stream) {
  return merv_softmax_mix_ex(V, tokens, scores, weights, out, K, (int64_t)T * K, B, E, T, K, dtype, stream);
}

// merv_scores_from_partials + merv_softmax_weights_ex in one launch (bf16 biases); used by merv_fused_forward
namespace merv {
int launch_scores_softmax_weights(const float* const* partial, const int32_t* count, const float* const* c, const void* const* bias,
                                  float* scores, float* weights, void* weights_bf16, float* bias_mix, int B, int E, int T, int N,
                                  cudaStream_t stream, bool pdl) {
  MERV_REQUIRE(partial && count && bias && scores && weights && bias_mix, MERV_E_ARG, "merv_scores_softmax_weights: NULL pointer");
  MERV_REQUIRE(E >= 1 && E <= MERV_MAX_ENCODERS, MERV_E_ARG, "merv_scores_softmax_weights: E=%d", E);
  MERV_REQUIRE(B >= 0 && T > 0 && N > 0, MERV_E_SHAPE, "merv_scores_softmax_weights: B=%d T=%d N=%d", B, T, N);
  if (int rc = require_sm100()) return rc;
  if (B == 0) return MERV_OK;
  PartialParams pp = {};
  BiasParams bp = {};
  for (int e = 0; e < E; ++e) {
    MERV_REQUIRE(partial[e] && count[e] > 0, MERV_E_ARG, "merv_scores_softmax_weights: encoder %d: NULL partials or count=%d", e, count[e]);
    pp.p[e] = partial[e];
    pp.c[e] = c ? c[e] : nullptr;
    pp.count[e] = count[e];
    bp.bias[e] = bias[e];
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((N + 255) / 256, B);
  cfg.blockDim = dim3(256);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  MERV_CUDA_OK(cudaLaunchKernelEx(&cfg, scores_softmax_kernel<__nv_bfloat16>, pp, bp, scores, weights, static_cast<__nv_bfloat16*>(weights_bf16),
                                  bias_mix, E, T, N));
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}
}  // namespace merv

extern "C" int merv_scores_softmax_weights(const float* const* partial, const int32_t* count, const float* const* c, const void* const* bias,
                                           float* scores, float* weights, void* weights_bf16, float* bias_mix, int B, int E, int T, int N,
                                           void* stream) {
  return merv::launch_scores_softmax_weights(partial, count, c, bias, scores, weights, weights_bf16, bias_mix, B, E, T, N,
                                             static_cast<cudaStream_t>(stream), false);
}
