// Backward of the module-by-module path (SURVEY.md §8 f-1): the gradients MERV's training step needs through the
// projectors and the fusion adapter (both trainable in every stage, merv/models/vidlms/merv.py:318-320,342-343,363-365).
// The backbones are frozen (merv.py:316,339,361), so no gradient flows into the patch features.
//
//   LinearProjector      y = P W^T + b           dW = dY^T P (tcgen05 GEMM on transposed copies), db = colsum(dY)
//   adapter (nn_utils.py:487-521, restated as  w = softmax_e(u . mean_t V_e),  out = sum_e w_e V_e):
//        dw_e   = <dOut, V_e>                     ds = softmax'(w) dw
//        dV_e   = w_e dOut + (ds_e / T) u         du = sum_{b,e} ds_e mean_t V_e
//        u = Wk^T q / sqrt(E), q = Wq Q^T + b_q:  dq = Wk du / sqrt(E), dWk = q du^T / sqrt(E), dWq = dq Q, db_q = dq, dQ = Wq^T dq
//   the other configurations of the adapter (merv_mix_backward_ex), same ds:
//     positional_embedding  w = softmax_e(u . (mean_t V_e + pe_e)):  dV_e as above,  du = sum_{b,e} ds_e (mean_t V_e + pe_e),
//                           dpe_e = (sum_b ds_e) u                                        (du_pe_kernel; no extra pass over V)
//     averagetoken=False    w = softmax_e(sum_t u_t . V_e[t]), u [T*K]:  dV_e[t] = w_e dOut[t] + ds_e u_t,
//                           du_t = sum_{b,e} ds_e V_e[b,t]  (length T*K, in the dV pass: mix_bwd_dv_flat_kernel)
//     single-token encoder  (repeated to T tokens) dV_e[b,0] = sum_t of the rows above = w_e gsum[b] + ds_e ubar,
//                           gsum[b] = sum_t dOut[b,t], ubar = u or sum_t u_t;  dw_e = <gsum[b], V_e[b,0]>, mean_t V_e = V_e[b,0]
//   v_proj_weight / out_proj / b_k / b_v receive no (zero) gradient, exactly as in the reference where the attention
//   output is discarded and b_k cancels in the softmax.
//   ScalarAdapter (nn_utils.py:524-537, w = softmax(scalar) for every video, out = sum_e w_e V_e):
//        dV_e = w_e dOut,  g_e = sum_b <dOut[b], V_e[b]> + dweights_out[e],  dscalar = w (.) (g - <w, g>)   (merv_scalar_mix_backward;
//        in front of linked linear projectors merv_scalar_fused_backward finishes the fused step)
// All reductions are fixed-order (deterministic, no atomics).
#include "common.cuh"

namespace merv {

template <int kThreads>
__device__ __forceinline__ float bwd_block_sum(float v, float* smem) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  float r = (lane < kThreads / 32) ? smem[lane] : 0.f;
  return warp_sum(r);
}

template <typename T> __device__ __forceinline__ T from_float(float v);
template <> __device__ __forceinline__ float from_float<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_float<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// ---- y[c, r] = x[r, c] : 32 x 32 tiles through shared memory, coalesced both ways ------------------------
template <typename T>
__global__ void __launch_bounds__(256) transpose_kernel(const T* __restrict__ x, T* __restrict__ y, int R, int C, long long ldx, long long ldy) {
  __shared__ T tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    const int r = r0 + ty + i, c = c0 + tx;
    if (r < R && c < C) tile[ty + i][tx] = x[(long long)r * ldx + c];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    const int c = c0 + ty + i, r = r0 + tx;
    if (r < R && c < C) y[(long long)c * ldy + r] = tile[tx][ty + i];
  }
}

// ---- out[n] = sum_m x[m, n]  (bias gradient): two fixed-order stages ---------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) colsum_partial_kernel(const T* __restrict__ x, float* __restrict__ partial, int M, int N, long long ld, int rows_per_block) {
  const int n = blockIdx.x * 256 + threadIdx.x;
  const int m0 = blockIdx.y * rows_per_block, m1 = min(M, m0 + rows_per_block);
  if (n >= N) return;
  float acc = 0.f;
  for (int m = m0; m < m1; ++m) acc += to_float(x[(long long)m * ld + n]);
  partial[(long long)blockIdx.y * N + n] = acc;
}
template <typename T>
__global__ void __launch_bounds__(256) colsum_final_kernel(const float* __restrict__ partial, T* __restrict__ out, int N, int nblocks) {
  const int n = blockIdx.x * 256 + threadIdx.x;
  if (n >= N) return;
  float acc = 0.f;
  for (int i = 0; i < nblocks; ++i) acc += partial[(long long)i * N + n];
  out[n] = from_float<T>(acc);
}

// ---- adapter backward, stage 1: dw[b,e] = <dOut[b], V_e[b]> and vbar[b,e,:] = mean_t V_e[b,t,:] ------------
struct BwdPtrs {
  const void* V[MERV_MAX_ENCODERS];
  void* dV[MERV_MAX_ENCODERS];
  int tokens[MERV_MAX_ENCODERS];  // T or 1 (a single-token encoder, repeated to T tokens in the forward)
};

// grid (column blocks of 8 vectors = 128 bytes, E, B), 256 threads = 8 vectors x 32 token groups; a thread walks every 32nd token with four
// independent pairs of 16-byte loads in flight, the 32 groups are then reduced through shared memory in a fixed order.  (The first version
// gave one thread a whole column of T tokens: 256 CTAs x 2 loads in flight = 1.4 TB/s, 0.49 ms of the 2.2 ms training step at 16 videos.)
// A single-token encoder reads dOut only: its column sums gsum[b,:] = sum_t dOut[b,t,:] (same fixed order) give dw = <gsum, V_e[b,0]>,
// vbar = V_e[b,0], and are kept for its dV (written by the CTAs of encoder gsum_e, the first single-token one).
constexpr int kMixRedCols = 8;  // 16-byte vectors per CTA
template <typename T>
__global__ void __launch_bounds__(256) mix_bwd_reduce_kernel(const __grid_constant__ BwdPtrs p, const T* __restrict__ dOut, float* __restrict__ dw_partial,
                                                             float* __restrict__ vbar, float* __restrict__ gsum, int gsum_e, int E, int Ttok, int K) {
  constexpr int VEC = Vec16<T>::kN;
  __shared__ float part[32][kMixRedCols * VEC + 1];
  __shared__ float red[32];
  const int kb = blockIdx.x, e = blockIdx.y, b = blockIdx.z;
  const int cv = threadIdx.x & (kMixRedCols - 1), rg = threadIdx.x / kMixRedCols;
  const int k0 = (kb * kMixRedCols + cv) * VEC;
  if (p.tokens[e] != Ttok) {
    float gs[VEC];
#pragma unroll
    for (int c = 0; c < VEC; ++c) gs[c] = 0.f;
    if (k0 < K) {
      const T* g = dOut + (long long)b * Ttok * K + k0;
      int t = rg;
      for (; t + 96 < Ttok; t += 128) {
        uint4 rd[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) rd[i] = ldg_nc_v4(g + (long long)(t + 32 * i) * K);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float d[VEC];
          Vec16<T>::unpack(rd[i], d);
#pragma unroll
          for (int c = 0; c < VEC; ++c) gs[c] += d[c];
        }
      }
      for (; t < Ttok; t += 32) {
        float d[VEC];
        Vec16<T>::unpack(ldg_nc_v4(g + (long long)t * K), d);
#pragma unroll
        for (int c = 0; c < VEC; ++c) gs[c] += d[c];
      }
    }
#pragma unroll
    for (int c = 0; c < VEC; ++c) part[rg][cv * VEC + c] = gs[c];
    __syncthreads();
    float sdot = 0.f;
    if (threadIdx.x < kMixRedCols * VEC) {
      const int k = kb * kMixRedCols * VEC + threadIdx.x;
      if (k < K) {
        float sum = 0.f;
#pragma unroll
        for (int gidx = 0; gidx < 32; ++gidx) sum += part[gidx][threadIdx.x];
        const float v = to_float(static_cast<const T*>(p.V[e])[(long long)b * K + k]);
        vbar[((long long)b * E + e) * K + k] = v;
        if (e == gsum_e) gsum[(long long)b * K + k] = sum;
        sdot = sum * v;
      }
    }
    sdot = bwd_block_sum<256>(sdot, red);
    if (threadIdx.x == 0) dw_partial[((long long)b * E + e) * gridDim.x + kb] = sdot;
    return;
  }
  float vs[VEC], dot = 0.f;
#pragma unroll
  for (int c = 0; c < VEC; ++c) vs[c] = 0.f;
  if (k0 < K) {
    const T* v = static_cast<const T*>(p.V[e]) + (long long)b * Ttok * K + k0;
    const T* g = dOut + (long long)b * Ttok * K + k0;
    int t = rg;
    for (; t + 96 < Ttok; t += 128) {
      uint4 ra[4], rd[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        ra[i] = ldg_nc_v4(v + (long long)(t + 32 * i) * K);
        rd[i] = ldg_nc_v4(g + (long long)(t + 32 * i) * K);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float a[VEC], d[VEC];
        Vec16<T>::unpack(ra[i], a);
        Vec16<T>::unpack(rd[i], d);
#pragma unroll
        for (int c = 0; c < VEC; ++c) {
          vs[c] += a[c];
          dot = fmaf(a[c], d[c], dot);
        }
      }
    }
    for (; t < Ttok; t += 32) {
      float a[VEC], d[VEC];
      Vec16<T>::unpack(ldg_nc_v4(v + (long long)t * K), a);
      Vec16<T>::unpack(ldg_nc_v4(g + (long long)t * K), d);
#pragma unroll
      for (int c = 0; c < VEC; ++c) {
        vs[c] += a[c];
        dot = fmaf(a[c], d[c], dot);
      }
    }
  }
#pragma unroll
  for (int c = 0; c < VEC; ++c) part[rg][cv * VEC + c] = vs[c];
  __syncthreads();
  if (threadIdx.x < kMixRedCols * VEC) {
    const int k = kb * kMixRedCols * VEC + threadIdx.x;
    if (k < K) {
      float sum = 0.f;
#pragma unroll
      for (int gidx = 0; gidx < 32; ++gidx) sum += part[gidx][threadIdx.x];
      vbar[((long long)b * E + e) * K + k] = sum / float(Ttok);
    }
  }
  dot = bwd_block_sum<256>(dot, red);
  if (threadIdx.x == 0) dw_partial[((long long)b * E + e) * gridDim.x + kb] = dot;
}

// ---- stage 2 (one warp per video): ds = softmax backward ------------------------------------------------------
__global__ void __launch_bounds__(32) mix_bwd_scores_kernel(const float* __restrict__ dw_partial, const float* __restrict__ weights,
                                                            const float* __restrict__ dweights_out, float* __restrict__ ds, int E, int kblocks) {
  const int b = blockIdx.x, lane = threadIdx.x;
  float dw = 0.f, w = 0.f;
  if (lane < E) {
    for (int i = 0; i < kblocks; ++i) dw += dw_partial[((long long)b * E + lane) * kblocks + i];
    if (dweights_out != nullptr) dw += dweights_out[(long long)b * E + lane];
    w = weights[(long long)b * E + lane];
  }
  const float inner = warp_sum(w * dw);
  if (lane < E) ds[(long long)b * E + lane] = w * (dw - inner);
}

// ---- stage 3: dV_e[b,t,:] = w[b,e] dOut[b,t,:] + (ds[b,e] / T) u  for the encoders in full_mask (the T-token ones) --------------
template <typename T, int E>
__global__ void __launch_bounds__(256) mix_bwd_dv_kernel(const __grid_constant__ BwdPtrs p, const T* __restrict__ dOut, const float* __restrict__ weights,
                                                         const float* __restrict__ ds, const float* __restrict__ u, int Ttok, int K, unsigned full_mask) {
  constexpr int VEC = Vec16<T>::kN;
  const int b = blockIdx.y;
  float w[E], s[E];
#pragma unroll
  for (int e = 0; e < E; ++e) {
    w[e] = weights[(long long)b * E + e];
    s[e] = ds[(long long)b * E + e] / float(Ttok);
  }
  const int kvec = K / VEC;
  const long long nvec = (long long)Ttok * kvec;
  const T* g = dOut + (long long)b * Ttok * K;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < nvec; i += (long long)gridDim.x * 256) {
    const int kc = int(i % kvec) * VEC;
    float d[VEC], uu[VEC];
    Vec16<T>::unpack(ldg_nc_v4(g + i * VEC), d);
#pragma unroll
    for (int c = 0; c < VEC; c += 4) {
      const float4 u4 = __ldg(reinterpret_cast<const float4*>(u + kc + c));
      uu[c] = u4.x; uu[c + 1] = u4.y; uu[c + 2] = u4.z; uu[c + 3] = u4.w;
    }
#pragma unroll
    for (int e = 0; e < E; ++e) {
      if (!((full_mask >> e) & 1u)) continue;
      float o[VEC];
#pragma unroll
      for (int c = 0; c < VEC; ++c) o[c] = fmaf(w[e], d[c], s[e] * uu[c]);
      stg_na_v4(static_cast<T*>(p.dV[e]) + (long long)b * Ttok * K + i * VEC, Vec16<T>::pack(o));
    }
  }
}

// ---- stage 3, averagetoken=False (u [T, K], one row per token, no token mean in the score), with du in the same pass ------------
//   dV_e[b,t,:] = w[b,e] dOut[b,t,:] + ds[b,e] u[t,:]   (T-token encoders, full_mask)
//   du[t,:]     = sum_b sum_e ds[b,e] V_e[b,t,:]         (a single-token encoder contributes its one row V_e[b,0,:] to every t)
// du needs ds, hence the second read of V; a thread owns one 16-byte column vector of one token for ALL videos, so du is summed in a fixed
// order (videos, then encoders) in registers and written once: no atomics, no [B, T*K] partials.
template <typename T, int E>
__global__ void __launch_bounds__(256) mix_bwd_dv_flat_kernel(const __grid_constant__ BwdPtrs p, const T* __restrict__ dOut, const float* __restrict__ weights,
                                                              const float* __restrict__ ds, const float* __restrict__ u, float* __restrict__ du, int B,
                                                              int Ttok, int K, unsigned full_mask) {
  constexpr int VEC = Vec16<T>::kN;
  const int kvec = K / VEC;
  const long long nvec = (long long)Ttok * kvec;
  const long long vstride = (long long)Ttok * K;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < nvec; i += (long long)gridDim.x * 256) {
    const int kc = int(i % kvec) * VEC;
    float uu[VEC], acc[VEC];
#pragma unroll
    for (int c = 0; c < VEC; c += 4) {
      const float4 u4 = __ldg(reinterpret_cast<const float4*>(u + i * VEC + c));
      uu[c] = u4.x; uu[c + 1] = u4.y; uu[c + 2] = u4.z; uu[c + 3] = u4.w;
    }
#pragma unroll
    for (int c = 0; c < VEC; ++c) acc[c] = 0.f;
    for (int b = 0; b < B; ++b) {
      float d[VEC];
      Vec16<T>::unpack(ldg_nc_v4(dOut + b * vstride + i * VEC), d);
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const float w = __ldg(weights + (long long)b * E + e), s = __ldg(ds + (long long)b * E + e);
        const bool full = (full_mask >> e) & 1u;
        const T* v = static_cast<const T*>(p.V[e]) + (full ? b * vstride + i * VEC : (long long)b * K + kc);
        float a[VEC];
        Vec16<T>::unpack(full ? ldg_nc_v4(v) : ldg_v4(v), a);
#pragma unroll
        for (int c = 0; c < VEC; ++c) acc[c] = fmaf(s, a[c], acc[c]);
        if (full) {
          float o[VEC];
#pragma unroll
          for (int c = 0; c < VEC; ++c) o[c] = fmaf(w, d[c], s * uu[c]);
          stg_na_v4(static_cast<T*>(p.dV[e]) + b * vstride + i * VEC, Vec16<T>::pack(o));
        }
      }
    }
#pragma unroll
    for (int c = 0; c < VEC; ++c) du[i * VEC + c] = acc[c];  // du sits at a workspace offset that need not be 16-byte aligned
  }
}

// ---- stage 3 of a single-token encoder: dV_e[b,0,:] = sum_t (row t of the T-token gradient) = w[b,e] gsum[b,:] + ds[b,e] ubar,
//      ubar = u (averagetoken: T rows of (ds / T) u) or sum_t u[t,:] (averagetoken=False, u_rows = T).  grid (ceil(K / 256), B) --------
template <typename T>
__global__ void __launch_bounds__(256) mix_bwd_dv_single_kernel(const __grid_constant__ BwdPtrs p, const float* __restrict__ weights, const float* __restrict__ ds,
                                                                const float* __restrict__ u, int u_rows, const float* __restrict__ gsum, int E, int K,
                                                                unsigned full_mask) {
  const int k = blockIdx.x * 256 + threadIdx.x, b = blockIdx.y;
  if (k >= K) return;
  float ub = 0.f;
  for (int r = 0; r < u_rows; ++r) ub += u[(long long)r * K + k];
  const float g = gsum[(long long)b * K + k];
  for (int e = 0; e < E; ++e) {
    if ((full_mask >> e) & 1u) continue;
    const float w = weights[(long long)b * E + e], s = ds[(long long)b * E + e];
    static_cast<T*>(p.dV[e])[(long long)b * K + k] = from_float<T>(fmaf(w, g, s * ub));
  }
}

// ---- query-vector backward ----------------------------------------------------------------------------------------
// du[k] = sum_{b,e} ds[b,e] vbar[b,e,k]
__global__ void __launch_bounds__(256) du_kernel(const float* __restrict__ ds, const float* __restrict__ vbar, float* __restrict__ du, int BE, int K) {
  const int k = blockIdx.x * 256 + threadIdx.x;
  if (k >= K) return;
  float acc = 0.f;
  for (int i = 0; i < BE; ++i) acc = fmaf(ds[i], vbar[(long long)i * K + k], acc);
  du[k] = acc;
}
// positional_embedding=True: the key is mean_t V_e + pe[e], so  du[k] = sum_{b,e} ds[b,e] (vbar[b,e,k] + pe[e,k])  and
// dpe[e,k] = (sum_b ds[b,e]) u[k]; the column sums sig_e are recomputed per thread (B * E floats from L1, fixed order)
template <typename T>
__global__ void __launch_bounds__(256) du_pe_kernel(const float* __restrict__ ds, const float* __restrict__ vbar, const T* __restrict__ pe, long long ldpe,
                                                    const float* __restrict__ u, float* __restrict__ du, T* __restrict__ dpe, int B, int E, int K) {
  const int k = blockIdx.x * 256 + threadIdx.x;
  if (k >= K) return;
  float acc = 0.f;
  for (int i = 0; i < B * E; ++i) acc = fmaf(ds[i], vbar[(long long)i * K + k], acc);
  const float uk = u[k];
  for (int e = 0; e < E; ++e) {
    float sig = 0.f;
    for (int b = 0; b < B; ++b) sig += ds[(long long)b * E + e];
    acc = fmaf(sig, to_float(pe[(long long)e * ldpe + k]), acc);
    dpe[(long long)e * K + k] = from_float<T>(sig * uk);
  }
  du[k] = acc;
}
// out[d] = scale * sum_k W[d,k] x[k] (+ bias[d]) : one warp per row
template <typename T, typename X>
__global__ void __launch_bounds__(256) gemv_n_kernel(const T* __restrict__ W, const X* __restrict__ x, const T* __restrict__ bias, float* __restrict__ out,
                                                     int D, int K, float scale) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= D) return;
  const int lane = threadIdx.x & 31;
  const T* w = W + (long long)row * K;
  float acc = 0.f;
  for (int k = lane; k < K; k += 32) acc += to_float(w[k]) * to_float(x[k]);
  acc = warp_sum(acc);
  if (lane == 0) out[row] = acc * scale + (bias ? to_float(bias[row]) : 0.f);
}
// the same with 16-byte loads of W (K % VEC == 0, rows 16-byte aligned)
template <typename T> __device__ __forceinline__ void load_vec_as_float(const T* p, float (&f)[Vec16<T>::kN]) { Vec16<T>::unpack(ldg_v4(p), f); }
template <typename T>
__device__ __forceinline__ void load_x_vec(const float* x, float (&f)[Vec16<T>::kN]) {
#pragma unroll
  for (int c = 0; c < Vec16<T>::kN; c += 4) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(x + c));
    f[c] = v.x; f[c + 1] = v.y; f[c + 2] = v.z; f[c + 3] = v.w;
  }
}
template <typename T>
__device__ __forceinline__ void load_x_vec(const __nv_bfloat16* x, float (&f)[Vec16<T>::kN]) {
  static_assert(Vec16<T>::kN == 8, "bf16 x goes with bf16 W");
  Vec16<__nv_bfloat16>::unpack(ldg_v4(x), f);
}
template <typename T, typename X>
__global__ void __launch_bounds__(256) gemv_n_vec_kernel(const T* __restrict__ W, const X* __restrict__ x, const T* __restrict__ bias, float* __restrict__ out,
                                                         int D, int K, float scale) {
  constexpr int VEC = Vec16<T>::kN;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= D) return;
  const int lane = threadIdx.x & 31;
  const T* w = W + (long long)row * K;
  float acc = 0.f;
  for (int k = lane * VEC; k < K; k += 32 * VEC) {
    float a[VEC], b[VEC];
    Vec16<T>::unpack(ldg_nc_v4(w + k), a);
    load_x_vec<T>(x + k, b);
#pragma unroll
    for (int c = 0; c < VEC; ++c) acc = fmaf(a[c], b[c], acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) out[row] = acc * scale + (bias ? to_float(bias[row]) : 0.f);
}
template <typename T, typename X>
static void launch_gemv_n(const T* W, const X* x, const T* bias, float* out, int D, int K, float scale, cudaStream_t s) {
  constexpr int VEC = Vec16<T>::kN;
  const bool vec_ok = K % VEC == 0 && aligned16(W) && aligned16(x) && (sizeof(X) == 4 || sizeof(T) == 2);
  if (vec_ok)
    gemv_n_vec_kernel<T, X><<<(D + 7) / 8, 256, 0, s>>>(W, x, bias, out, D, K, scale);
  else
    gemv_n_kernel<T, X><<<(D + 7) / 8, 256, 0, s>>>(W, x, bias, out, D, K, scale);
}

// out[j] = sum_d W[d,j] x[d]  (W [D, J] row-major), fp32 x
template <typename T>
__global__ void __launch_bounds__(256) gemv_tf_kernel(const T* __restrict__ W, const float* __restrict__ x, T* __restrict__ out, int D, int J) {
  __shared__ float part[8][33];
  const int jx = threadIdx.x & 31, dy = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + jx;
  float acc = 0.f;
  if (j < J)
    for (int d = dy; d < D; d += 8) acc += to_float(W[(long long)d * J + j]) * x[d];
  part[dy][jx] = acc;
  __syncthreads();
  if (dy == 0 && j < J) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += part[i][jx];
    out[j] = from_float<T>(s);
  }
}
// out[i, j] = scale * a[i] * b[j]
template <typename T, typename Bv>
__global__ void __launch_bounds__(256) outer_kernel(const float* __restrict__ a, const Bv* __restrict__ b, T* __restrict__ out, int I, int J, float scale) {
  const long long idx = (long long)blockIdx.x * 256 + threadIdx.x;
  if (idx >= (long long)I * J) return;
  const int i = int(idx / J), j = int(idx % J);
  out[idx] = from_float<T>(scale * a[i] * to_float(b[j]));
}
template <typename T>
__global__ void __launch_bounds__(256) bias_grad_kernel(const float* __restrict__ dq, T* __restrict__ dbias, int embed) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < 3 * embed) dbias[i] = from_float<T>(i < embed ? dq[i] : 0.f);  // b_k cancels in the softmax, b_v is dead
}

// ---- elementwise erf-GELU forward / backward for the MLP projectors' training path (nn.GELU(), nn_utils.py:48) --------
// y = gelu(z);  dz = dy * gelu'(z),  gelu'(z) = 0.5 (1 + erf(z / sqrt 2)) + z exp(-z^2 / 2) / sqrt(2 pi)
template <typename T, bool kBackward>
__global__ void __launch_bounds__(256) gelu_kernel(const T* __restrict__ z, const T* __restrict__ dy, T* __restrict__ out, long long nvec) {
  constexpr int VEC = Vec16<T>::kN;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < nvec; i += (long long)gridDim.x * 256) {
    float a[VEC], g[VEC], o[VEC];
    Vec16<T>::unpack(ldg_nc_v4(z + i * VEC), a);
    if (kBackward) Vec16<T>::unpack(ldg_nc_v4(dy + i * VEC), g);
#pragma unroll
    for (int c = 0; c < VEC; ++c) {
      const float cdf = 0.5f * (1.0f + erff(a[c] * 0.70710678118654752440f));
      if (kBackward)
        o[c] = g[c] * (cdf + a[c] * 0.3989422804014327f * expf(-0.5f * a[c] * a[c]));
      else
        o[c] = a[c] * cdf;
    }
    stg_na_v4(out + i * VEC, Vec16<T>::pack(o));
  }
}

template <typename T>
static int launch_mix_dv(const BwdPtrs& p, const void* dOut, const float* weights, const float* ds, const float* u, int B, int E, int Ttok, int K,
                         unsigned full_mask, cudaStream_t s) {
  constexpr int VEC = Vec16<T>::kN;
  const long long nvec = (long long)Ttok * (K / VEC);
  long long gx = (nvec + 255) / 256;
  const long long cap = (long long)sm_count() * 16 / (B > 0 ? B : 1) + 1;
  if (gx > cap) gx = cap;
  dim3 grid((unsigned)gx, B);
  const T* g = static_cast<const T*>(dOut);
  switch (E) {
#define MERV_DV_CASE(n) case n: mix_bwd_dv_kernel<T, n><<<grid, 256, 0, s>>>(p, g, weights, ds, u, Ttok, K, full_mask); break;
    MERV_DV_CASE(1) MERV_DV_CASE(2) MERV_DV_CASE(3) MERV_DV_CASE(4) MERV_DV_CASE(5) MERV_DV_CASE(6) MERV_DV_CASE(7) MERV_DV_CASE(8)
#undef MERV_DV_CASE
    default: return fail(MERV_E_ARG, "merv_mix_backward: E=%d", E);
  }
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

template <typename T>
static int launch_mix_dv_flat(const BwdPtrs& p, const void* dOut, const float* weights, const float* ds, const float* u, float* du, int B, int E,
                              int Ttok, int K, unsigned full_mask, cudaStream_t s) {
  constexpr int VEC = Vec16<T>::kN;
  const long long nvec = (long long)Ttok * (K / VEC);
  long long gx = (nvec + 255) / 256;
  const long long cap = (long long)sm_count() * 16;  // every thread walks all B videos
  if (gx > cap) gx = cap;
  const T* g = static_cast<const T*>(dOut);
  switch (E) {
#define MERV_DV_CASE(n) case n: mix_bwd_dv_flat_kernel<T, n><<<(unsigned)gx, 256, 0, s>>>(p, g, weights, ds, u, du, B, Ttok, K, full_mask); break;
    MERV_DV_CASE(1) MERV_DV_CASE(2) MERV_DV_CASE(3) MERV_DV_CASE(4) MERV_DV_CASE(5) MERV_DV_CASE(6) MERV_DV_CASE(7) MERV_DV_CASE(8)
#undef MERV_DV_CASE
    default: return fail(MERV_E_ARG, "merv_mix_backward_ex: E=%d", E);
  }
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

// ============================================================================================================
// ScalarAdapter (feature_fusion == "scalar", nn_utils.py:524-537):  w = softmax(scalar) [E], the same for every video,
// out = sum_e w_e V_e, returned weights w[None].  With dweights_out [E] the gradient of the returned weights:
//     dV_e    = w_e dOut                                   (independent of the scalar gradient: one pass suffices)
//     g_e     = sum_b <dOut[b], V_e[b]> + dweights_out[e]
//     dscalar = w (.) (g - <w, g>)
// ============================================================================================================

// ---- one pass: grid (column blocks of 8 vectors = 128 bytes, B), 256 threads = 8 vectors x 32 token groups as in mix_bwd_reduce_kernel,
//      but a CTA owns its column block for ALL encoders: every dOut vector is read once (not once per encoder), every V_e vector once and
//      every dV_e vector written once, (1 + 2E) B T K elements in all.  Two tokens per iteration keep 2 (1 + E) independent 16-byte loads
//      in flight per thread.  The dots are reduced in a fixed order (warp butterfly, then the 8 warps in order) into partial[b, e, kb].
template <typename T, int E>
__global__ void __launch_bounds__(256) scalar_mix_bwd_kernel(const __grid_constant__ BwdPtrs p, const T* __restrict__ dOut, const float* __restrict__ weights,
                                                             float* __restrict__ partial, int Ttok, int K) {
  constexpr int VEC = Vec16<T>::kN;
  __shared__ float red[E][8];
  const int kb = blockIdx.x, b = blockIdx.y;
  const int cv = threadIdx.x & (kMixRedCols - 1), rg = threadIdx.x / kMixRedCols;
  const int k0 = (kb * kMixRedCols + cv) * VEC;
  float w[E], dot[E];
#pragma unroll
  for (int e = 0; e < E; ++e) {
    w[e] = weights[e];
    dot[e] = 0.f;
  }
  if (k0 < K) {
    const long long base = (long long)b * Ttok * K + k0;
    const T* g = dOut + base;
    const T* vb[E];
    T* db[E];
#pragma unroll
    for (int e = 0; e < E; ++e) {
      vb[e] = static_cast<const T*>(p.V[e]) + base;
      db[e] = static_cast<T*>(p.dV[e]) + base;
    }
    int t = rg;
    for (; t + 32 < Ttok; t += 64) {
      uint4 rd[2], rv[2][E];
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const long long off = (long long)(t + 32 * i) * K;
        rd[i] = ldg_nc_v4(g + off);
#pragma unroll
        for (int e = 0; e < E; ++e) rv[i][e] = ldg_nc_v4(vb[e] + off);
      }
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const long long off = (long long)(t + 32 * i) * K;
        float d[VEC];
        Vec16<T>::unpack(rd[i], d);
#pragma unroll
        for (int e = 0; e < E; ++e) {
          float a[VEC], o[VEC];
          Vec16<T>::unpack(rv[i][e], a);
#pragma unroll
          for (int c = 0; c < VEC; ++c) {
            dot[e] = fmaf(a[c], d[c], dot[e]);
            o[c] = w[e] * d[c];
          }
          stg_na_v4(db[e] + off, Vec16<T>::pack(o));
        }
      }
    }
#pragma unroll 1
    for (; t < Ttok; t += 32) {
      const long long off = (long long)t * K;
      float d[VEC];
      Vec16<T>::unpack(ldg_nc_v4(g + off), d);
#pragma unroll
      for (int e = 0; e < E; ++e) {
        float a[VEC], o[VEC];
        Vec16<T>::unpack(ldg_nc_v4(vb[e] + off), a);
#pragma unroll
        for (int c = 0; c < VEC; ++c) {
          dot[e] = fmaf(a[c], d[c], dot[e]);
          o[c] = w[e] * d[c];
        }
        stg_na_v4(db[e] + off, Vec16<T>::pack(o));
      }
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const float v = warp_sum(dot[e]);
    if (lane == 0) red[e][warp] = v;
  }
  __syncthreads();
  if (threadIdx.x < E) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[threadIdx.x][i];
    partial[((long long)b * E + threadIdx.x) * gridDim.x + kb] = s;
  }
}

// ---- the end of both scalar backward paths (256 threads, all of them call it): per-thread sums acc[e] -> block sums (warp butterfly, then
//      the 8 warps in order) -> g_e = block sum + dweights_out[e] -> dscalar = w (.) (g - <w, g>) ------------------------------------------
__device__ __forceinline__ void scalar_grad_from_block(const float (&acc)[MERV_MAX_ENCODERS], const float* __restrict__ weights,
                                                       const float* __restrict__ dweights_out, float* __restrict__ dscalar, int E) {
  __shared__ float red[MERV_MAX_ENCODERS][8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int e = 0; e < MERV_MAX_ENCODERS; ++e) {
    if (e >= E) break;
    const float v = warp_sum(acc[e]);
    if (lane == 0) red[e][warp] = v;
  }
  __syncthreads();
  if (warp == 0) {
    float g = 0.f, w = 0.f;
    if (lane < E) {
#pragma unroll
      for (int i = 0; i < 8; ++i) g += red[lane][i];
      if (dweights_out != nullptr) g += dweights_out[lane];
      w = weights[lane];
    }
    const float inner = warp_sum(w * g);
    if (lane < E) dscalar[lane] = w * (g - inner);
  }
}

// ---- fold of the one-pass partials, one CTA: thread i sums the (video, column block) pairs i, i + 256, ... (videos outer) of every encoder.
//      (A single warp would wait on B * kblocks / 32 dependent loads per encoder, 128 at 64 videos of merv-full.) --------------------------
__global__ void __launch_bounds__(256) scalar_mix_fold_kernel(const float* __restrict__ partial, const float* __restrict__ weights,
                                                              const float* __restrict__ dweights_out, float* __restrict__ dscalar, int B, int E,
                                                              int kblocks) {
  float acc[MERV_MAX_ENCODERS];
#pragma unroll
  for (int e = 0; e < MERV_MAX_ENCODERS; ++e) acc[e] = 0.f;
  const long long n = (long long)B * kblocks;
  for (long long i = threadIdx.x; i < n; i += 256) {
    const long long b = i / kblocks, kb = i - b * kblocks;
#pragma unroll
    for (int e = 0; e < MERV_MAX_ENCODERS; ++e)
      if (e < E) acc[e] += partial[(b * E + e) * kblocks + kb];
  }
  scalar_grad_from_block(acc, weights, dweights_out, dscalar, E);
}

template <typename T>
static int launch_scalar_mix_bwd(const BwdPtrs& p, const void* dOut, const float* weights, float* partial, int B, int E, int Ttok, int K,
                                 int kblocks, cudaStream_t s) {
  dim3 grid(kblocks, B);
  const T* g = static_cast<const T*>(dOut);
  switch (E) {
#define MERV_SCALAR_CASE(n) case n: scalar_mix_bwd_kernel<T, n><<<grid, 256, 0, s>>>(p, g, weights, partial, Ttok, K); break;
    MERV_SCALAR_CASE(1) MERV_SCALAR_CASE(2) MERV_SCALAR_CASE(3) MERV_SCALAR_CASE(4) MERV_SCALAR_CASE(5) MERV_SCALAR_CASE(6) MERV_SCALAR_CASE(7)
    MERV_SCALAR_CASE(8)
#undef MERV_SCALAR_CASE
    default: return fail(MERV_E_ARG, "merv_scalar_mix_backward: E=%d", E);
  }
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}


// ============================================================================================================
// Backward of the FUSED path (linear projectors linked to the adapter; merv_fused_linear_mix forward).
//   forward :  s_e = u . mean_t(P_e W_e^T + b_e),  w = softmax_e(s),  out = sum_e w_e (P_e W_e^T + b_e)      (P_e = pooled tokens)
//   backward:  neither the per-encoder projections Y_e nor their gradients dV_e are ever materialised (2 x 33.5 MB per video):
//        dw_e = <dOut, Y_e> = <dOut W_e, P_e> + b_e . colsum_t(dOut)         Z_e = dOut W_e: dgrad-shaped tcgen05 GEMM, [M, C_e] only
//        ds   = softmax backward of (dw + dweights_out)
//        dW_e = dV_e^T P_e = dOut^T (w_e (.) P_e) + u (x) g_e,   g_e = sum_b ds_e[b] mean_t P_e[b]      (w_e scales the rows of P_e per video)
//        db_e = sum_b w_e[b] colsum_t(dOut[b]) + u sum_b ds_e[b]
//        du   = sum_e (W_e g_e + b_e sum_b ds_e[b])        then dq, dWk, dWq, db_q, dQ as in merv_mix_backward
// The kernels below are the HBM-bound / tiny pieces; the two GEMMs per encoder run on the tcgen05 kernel.
// ============================================================================================================

// ---- out[b, k] = scale * sum_t x[b, t, k] (fp32): CTA = (8 vectors = 128-byte column block, video), 32 row groups, fixed-order
//      reduction; narrow column blocks keep enough CTAs in flight at the small per-device batches of the training step ----
template <typename T>
__global__ void __launch_bounds__(256) video_colsum_kernel(const T* __restrict__ x, float* __restrict__ out, int Ttok, int K, long long ld,
                                                           long long batch_stride, float scale) {
  constexpr int VEC = Vec16<T>::kN;
  __shared__ float part[32][8 * VEC + 1];
  const int cv = threadIdx.x & 7, rg = threadIdx.x >> 3;
  const int k0 = (blockIdx.x * 8 + cv) * VEC;
  const int b = blockIdx.y;
  float acc[VEC];
#pragma unroll
  for (int c = 0; c < VEC; ++c) acc[c] = 0.f;
  if (k0 < K) {
    const T* base = x + (long long)b * batch_stride + k0;
    int t = rg;
    for (; t + 96 < Ttok; t += 128) {  // four independent 16-byte loads in flight per thread
      uint4 r[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) r[i] = ldg_nc_v4(base + (long long)(t + 32 * i) * ld);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float f[VEC];
        Vec16<T>::unpack(r[i], f);
#pragma unroll
        for (int c = 0; c < VEC; ++c) acc[c] += f[c];
      }
    }
    for (; t < Ttok; t += 32) {
      float f[VEC];
      Vec16<T>::unpack(ldg_nc_v4(base + (long long)t * ld), f);
#pragma unroll
      for (int c = 0; c < VEC; ++c) acc[c] += f[c];
    }
  }
#pragma unroll
  for (int c = 0; c < VEC; ++c) part[rg][cv * VEC + c] = acc[c];
  __syncthreads();
  if (threadIdx.x < 8 * VEC) {
    const int k = blockIdx.x * 8 * VEC + threadIdx.x;
    if (k < K) {
      float sum = 0.f;
#pragma unroll
      for (int g = 0; g < 32; ++g) sum += part[g][threadIdx.x];
      out[(long long)b * K + k] = sum * scale;
    }
  }
}

// ---- partial[b, chunk] = sum over the chunk of x[b, i] * y[b, i]  (both [B, n] contiguous) --------------------------------
constexpr int kPairDotChunks = 32;
// Optionally also writes ys[b, i] = scale[b * scale_stride] * y[b, i] in the same pass (the per-video mixing weight applied to the pooled
// tokens: the MN-major W-operand of dW_e = dOut^T (w_e (.) P_e)), so P_e is read once for both.
template <typename T>
__global__ void __launch_bounds__(256) pair_dot_kernel(const T* __restrict__ x, const T* __restrict__ y, float* __restrict__ partial, long long nvec,
                                                       const float* __restrict__ scale = nullptr, long long scale_stride = 0, T* __restrict__ ys = nullptr) {
  constexpr int VEC = Vec16<T>::kN;
  __shared__ float red[32];
  const int chunk = blockIdx.x, b = blockIdx.y;
  const float sc = scale != nullptr ? scale[(long long)b * scale_stride] : 1.0f;
  T* ysb = ys != nullptr ? ys + (long long)b * nvec * VEC : nullptr;
  const long long per = (nvec + kPairDotChunks - 1) / kPairDotChunks;
  const long long v0 = chunk * per, v1 = v0 + per < nvec ? v0 + per : nvec;
  const T* xb = x + (long long)b * nvec * VEC;
  const T* yb = y + (long long)b * nvec * VEC;
  float acc = 0.f;
  for (long long v = v0 + threadIdx.x; v < v1; v += 512) {
    const long long v2 = v + 256;
    const bool has2 = v2 < v1;
    const uint4 a1 = ldg_nc_v4(xb + v * VEC), b1 = ldg_nc_v4(yb + v * VEC);
    uint4 a2 = make_uint4(0u, 0u, 0u, 0u), b2 = a2;
    if (has2) {
      a2 = ldg_nc_v4(xb + v2 * VEC);
      b2 = ldg_nc_v4(yb + v2 * VEC);
    }
    float fa[VEC], fb[VEC];
    Vec16<T>::unpack(a1, fa);
    Vec16<T>::unpack(b1, fb);
#pragma unroll
    for (int c = 0; c < VEC; ++c) acc = fmaf(fa[c], fb[c], acc);
    if (ysb != nullptr) {
#pragma unroll
      for (int c = 0; c < VEC; ++c) fb[c] *= sc;
      stg_na_v4(ysb + v * VEC, Vec16<T>::pack(fb));
    }
    Vec16<T>::unpack(a2, fa);
    Vec16<T>::unpack(b2, fb);
#pragma unroll
    for (int c = 0; c < VEC; ++c) acc = fmaf(fa[c], fb[c], acc);
    if (ysb != nullptr && has2) {
#pragma unroll
      for (int c = 0; c < VEC; ++c) fb[c] *= sc;
      stg_na_v4(ysb + v2 * VEC, Vec16<T>::pack(fb));
    }
  }
  acc = bwd_block_sum<256>(acc, red);
  if (threadIdx.x == 0) partial[(long long)b * kPairDotChunks + chunk] = acc;
}

// ---- y[c, r] = scale(r) * x[r, c] for r < R, 0 for R <= r < R_pad : 64 x 64 tiles, 4-byte accesses both ways (bf16) --------------
// scale(r) = scale[(r / rows_per_scale) * scale_stride] (fp32) or 1: the per-video mixing weight applied to the pooled tokens.
template <typename T>
__global__ void __launch_bounds__(256) transpose_rowscale_kernel(const T* __restrict__ x, T* __restrict__ y, int R, int R_pad, int C, long long ldx,
                                                                 long long ldy, const float* __restrict__ scale, long long scale_stride,
                                                                 int rows_per_scale) {
  __shared__ float tile[64][65];
  const int c0 = blockIdx.x * 64, r0 = blockIdx.y * 64;
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;  // 64 x 4
  for (int i = ty; i < 64; i += 4) {
    const int r = r0 + i, c = c0 + tx;
    float v = 0.f;
    if (r < R && c < C) {
      v = to_float(x[(long long)r * ldx + c]);
      if (scale != nullptr) v *= scale[(long long)(r / rows_per_scale) * scale_stride];
    }
    tile[i][tx] = v;
  }
  __syncthreads();
  for (int i = ty; i < 64; i += 4) {
    const int c = c0 + i, r = r0 + tx;
    if (r < R_pad && c < C) y[(long long)c * ldy + r] = from_float<T>(tile[tx][i]);
  }
}

// ---- the same for bf16 with 16-byte global accesses both ways (C % 8 == 0, R_pad % 8 == 0, 16-byte aligned rows) ----------------
// 64 x 64 tile as 32-bit words (bf16 pairs) with a 33-word pitch.  Load: one 16-byte vector = 4 words per thread and row, written
// conflict-free (bank = row + 4 * vec + k).  Store: a thread owns a column PAIR and 8 consecutive rows: 8 word reads give it two
// 16-byte output vectors (rows c and c + 1 of y); the 8 lanes of a column pair write 128 contiguous bytes.
__global__ void __launch_bounds__(256) transpose_bf16_vec_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, int R, int R_pad, int C,
                                                                 long long ldx, long long ldy, const float* __restrict__ scale, long long scale_stride,
                                                                 int rows_per_scale) {
  __shared__ uint32_t tile[64][33];
  const int c0 = blockIdx.x * 64, r0 = blockIdx.y * 64;
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int id = threadIdx.x + it * 256;
    const int row = id >> 3, v = id & 7;
    const int r = r0 + row, c = c0 + v * 8;
    uint4 q = make_uint4(0u, 0u, 0u, 0u);
    if (r < R && c < C) {
      q = ldg_nc_v4(x + (long long)r * ldx + c);
      if (scale != nullptr) {
        const float sc = scale[(long long)(r / rows_per_scale) * scale_stride];
        float f[8];
        Vec16<__nv_bfloat16>::unpack(q, f);
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] *= sc;
        q = Vec16<__nv_bfloat16>::pack(f);
      }
    }
    tile[row][v * 4 + 0] = q.x;
    tile[row][v * 4 + 1] = q.y;
    tile[row][v * 4 + 2] = q.z;
    tile[row][v * 4 + 3] = q.w;
  }
  __syncthreads();
  const int rb = threadIdx.x & 7, cp = threadIdx.x >> 3;  // 8 row blocks x 32 column pairs
  uint32_t w[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) w[i] = tile[rb * 8 + i][cp];
  const int r = r0 + rb * 8, c = c0 + cp * 2;
  if (r < R_pad && c < C) {
    // low halves -> row c of y, high halves -> row c + 1 (C is even)
    const uint4 lo = make_uint4(__byte_perm(w[0], w[1], 0x5410), __byte_perm(w[2], w[3], 0x5410), __byte_perm(w[4], w[5], 0x5410),
                                __byte_perm(w[6], w[7], 0x5410));
    const uint4 hi = make_uint4(__byte_perm(w[0], w[1], 0x7632), __byte_perm(w[2], w[3], 0x7632), __byte_perm(w[4], w[5], 0x7632),
                                __byte_perm(w[6], w[7], 0x7632));
    *reinterpret_cast<uint4*>(y + (long long)c * ldy + r) = lo;
    *reinterpret_cast<uint4*>(y + (long long)(c + 1) * ldy + r) = hi;
  }
}

// ---- tiny kernels of the fused backward ------------------------------------------------------------------------------------------
struct FusedBwdPtrs {
  const float* dw_partial[MERV_MAX_ENCODERS];  // [B, kPairDotChunks]
  const float* pbar[MERV_MAX_ENCODERS];        // [B, C_e] per-video column means of the pooled tokens
  const void* W[MERV_MAX_ENCODERS];            // [K, C_e]
  const void* bias[MERV_MAX_ENCODERS];         // [K] or NULL
  void* dW[MERV_MAX_ENCODERS];                 // [K, C_e] in/out
  void* db[MERV_MAX_ENCODERS];                 // [K] or NULL
  long long ldw[MERV_MAX_ENCODERS], lddw[MERV_MAX_ENCODERS];
  int C[MERV_MAX_ENCODERS];
  int goff[MERV_MAX_ENCODERS];                 // offset of g_e in the workspace
};

// one warp per video: dw_e = sum of the pair-dot partials + b_e . gsum[b] (+ dweights_out), ds = softmax backward
template <typename T>
__global__ void __launch_bounds__(32) fused_bwd_scores_kernel(const __grid_constant__ FusedBwdPtrs p, const float* __restrict__ gsum,
                                                              const float* __restrict__ weights, const float* __restrict__ dweights_out,
                                                              float* __restrict__ ds, int E, int K) {
  const int b = blockIdx.x, lane = threadIdx.x;
  float mine = 0.f;
  for (int e = 0; e < E; ++e) {
    float acc = 0.f;
    if (lane < kPairDotChunks) acc = p.dw_partial[e][(long long)b * kPairDotChunks + lane];
    if (p.bias[e] != nullptr) {
      const T* be = static_cast<const T*>(p.bias[e]);
      for (int k = lane; k < K; k += 32) acc = fmaf(to_float(be[k]), gsum[(long long)b * K + k], acc);
    }
    acc = warp_sum(acc);
    if (lane == e) mine = acc;
  }
  float w = 0.f;
  if (lane < E) {
    if (dweights_out != nullptr) mine += dweights_out[(long long)b * E + lane];
    w = weights[(long long)b * E + lane];
  }
  const float inner = warp_sum(lane < E ? w * mine : 0.f);
  if (lane < E) ds[(long long)b * E + lane] = w * (mine - inner);
}

// g_e[c] = sum_b ds[b, e] * pbar_e[b, c]   grid (ceil(C_max / 256), E)
__global__ void __launch_bounds__(256) fused_bwd_g_kernel(const __grid_constant__ FusedBwdPtrs p, const float* __restrict__ ds, float* __restrict__ g,
                                                          int B, int E) {
  const int e = blockIdx.y, c = blockIdx.x * 256 + threadIdx.x;
  if (c >= p.C[e]) return;
  float acc = 0.f;
  for (int b = 0; b < B; ++b) acc = fmaf(ds[(long long)b * E + e], p.pbar[e][(long long)b * p.C[e] + c], acc);
  g[p.goff[e] + c] = acc;
}

// db_e[n] = sum_b w[b, e] gsum[b, n] + u[n] sum_b ds[b, e]   grid (ceil(K / 256), E)
template <typename T>
__global__ void __launch_bounds__(256) fused_bwd_db_kernel(const __grid_constant__ FusedBwdPtrs p, const float* __restrict__ gsum,
                                                           const float* __restrict__ weights, const float* __restrict__ ds, const float* __restrict__ u,
                                                           int B, int E, int K) {
  const int e = blockIdx.y, n = blockIdx.x * 256 + threadIdx.x;
  if (n >= K || p.db[e] == nullptr) return;
  float acc = 0.f, sig = 0.f;
  for (int b = 0; b < B; ++b) {
    acc = fmaf(weights[(long long)b * E + e], gsum[(long long)b * K + n], acc);
    sig += ds[(long long)b * E + e];
  }
  static_cast<T*>(p.db[e])[n] = from_float<T>(fmaf(u[n], sig, acc));
}

// dW_e[n, c] += u[n] * g_e[c]   grid (blocks, E): block-stride loop over the K x C_e elements of encoder blockIdx.y, 16 bytes per
// thread when the rows allow it (kVecOK: C_e % VEC == 0, 16-byte aligned rows — always true for buffers the GEMM wrote)
template <typename T, bool kVecOK>
__global__ void __launch_bounds__(256) fused_bwd_rank1_kernel(const __grid_constant__ FusedBwdPtrs p, const float* __restrict__ u, const float* __restrict__ g,
                                                              int K) {
  constexpr int VEC = kVecOK ? Vec16<T>::kN : 1;
  const int e = blockIdx.y, C = p.C[e], cv = C / VEC;
  T* dW = static_cast<T*>(p.dW[e]);
  const long long ld = p.lddw[e];
  const float* ge = g + p.goff[e];
  const long long total = (long long)K * cv;
  for (long long idx = (long long)blockIdx.x * 256 + threadIdx.x; idx < total; idx += (long long)gridDim.x * 256) {
    const int n = int(idx / cv), c = int(idx - (long long)n * cv) * VEC;
    T* d = dW + (long long)n * ld + c;
    const float un = u[n];
    if constexpr (kVecOK) {
      float f[Vec16<T>::kN], gg[Vec16<T>::kN];
      Vec16<T>::unpack(*reinterpret_cast<const uint4*>(d), f);
      load_x_vec<T>(ge + c, gg);
#pragma unroll
      for (int i = 0; i < Vec16<T>::kN; ++i) f[i] = fmaf(un, gg[i], f[i]);
      *reinterpret_cast<uint4*>(d) = Vec16<T>::pack(f);
    } else {
      *d = from_float<T>(fmaf(un, ge[c], to_float(*d)));
    }
  }
}

// du[n] = sum_e (sum_c W_e[n, c] g_e[c] + sig_e b_e[n]) : one warp per row, encoders in order (fixed summation order)
template <typename T, bool kVecOK>
__global__ void __launch_bounds__(256) fused_bwd_du_kernel(const __grid_constant__ FusedBwdPtrs p, const float* __restrict__ g, const float* __restrict__ ds,
                                                           float* __restrict__ du, int K, int B, int E) {
  constexpr int VEC = kVecOK ? Vec16<T>::kN : 1;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= K) return;
  const int lane = threadIdx.x & 31;
  float total = 0.f;
  for (int e = 0; e < E; ++e) {
    const T* w = static_cast<const T*>(p.W[e]) + (long long)row * p.ldw[e];
    const float* ge = g + p.goff[e];
    float acc = 0.f;
    for (int c = lane * VEC; c < p.C[e]; c += 32 * VEC) {
      if constexpr (kVecOK) {
        float a[Vec16<T>::kN], b[Vec16<T>::kN];
        Vec16<T>::unpack(ldg_nc_v4(w + c), a);
        load_x_vec<T>(ge + c, b);
#pragma unroll
        for (int i = 0; i < Vec16<T>::kN; ++i) acc = fmaf(a[i], b[i], acc);
      } else {
        acc = fmaf(to_float(w[c]), ge[c], acc);
      }
    }
    if (p.bias[e] != nullptr) {  // sig_e = sum_b ds[b, e], spread over the lanes
      float sig = 0.f;
      for (int b = lane; b < B; b += 32) sig += ds[(long long)b * E + e];
      acc = fmaf(sig, to_float(static_cast<const T*>(p.bias[e])[row]), acc);
    }
    total += warp_sum(acc);
  }
  if (lane == 0) du[row] = total;
}

// two outer products in one launch: blockIdx.y == 0: dWk[i, j] = rs * q[i] * du[j];  == 1: dWq[i, j] = dq[i] * Q[j]
template <typename T, bool kVecOK>
__global__ void __launch_bounds__(256) fused_bwd_outer_kernel(const float* __restrict__ q, const float* __restrict__ du, const float* __restrict__ dq,
                                                              const T* __restrict__ Q, T* __restrict__ dWk, T* __restrict__ dWq, int embed, int K, float rs) {
  constexpr int VEC = kVecOK ? Vec16<T>::kN : 1;
  const bool first = blockIdx.y == 0;
  const int J = first ? K : embed, jv = J / VEC;
  const long long total = (long long)embed * jv;
  for (long long idx = (long long)blockIdx.x * 256 + threadIdx.x; idx < total; idx += (long long)gridDim.x * 256) {
    const int i = int(idx / jv), j = int(idx - (long long)i * jv) * VEC;
    const float a = first ? rs * q[i] : dq[i];
    T* dst = (first ? dWk : dWq) + (long long)i * J + j;
    if constexpr (kVecOK) {
      float b[Vec16<T>::kN];
      if (first) load_x_vec<T>(du + j, b);
      else Vec16<T>::unpack(ldg_v4(Q + j), b);
#pragma unroll
      for (int c = 0; c < Vec16<T>::kN; ++c) b[c] *= a;
      stg_na_v4(dst, Vec16<T>::pack(b));
    } else {
      *dst = from_float<T>(a * (first ? du[j] : to_float(Q[j])));
    }
  }
}

// dQ[j] = sum_d Wq[d, j] dq[d], stage 1: partial[s, j] over the rows d = s, s + S, ... (grid (ceil(J / 32), S), 8 row groups per CTA)
template <typename T>
__global__ void __launch_bounds__(256) gemv_tf_partial_kernel(const T* __restrict__ W, const float* __restrict__ x, float* __restrict__ partial, int D, int J) {
  __shared__ float part[8][33];
  const int jx = threadIdx.x & 31, dy = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + jx;
  float acc = 0.f;
  if (j < J)
    for (int d = blockIdx.y * 8 + dy; d < D; d += 8 * gridDim.y) acc += to_float(W[(long long)d * J + j]) * x[d];
  part[dy][jx] = acc;
  __syncthreads();
  if (dy == 0 && j < J) {
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) sum += part[i][jx];
    partial[(long long)blockIdx.y * J + j] = sum;
  }
}
// stage 2 merged with the in_proj_bias gradient: dQ[j] = sum_s partial[s, j];  dbias = [dq, 0, 0]
template <typename T>
__global__ void __launch_bounds__(256) fused_bwd_final_kernel(const float* __restrict__ partial, int S, const float* __restrict__ dq, T* __restrict__ dQ,
                                                              T* __restrict__ dbias, int embed) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < embed) {
    float sum = 0.f;
    for (int k = 0; k < S; ++k) sum += partial[(long long)k * embed + i];
    dQ[i] = from_float<T>(sum);
  }
  if (i < 3 * embed) dbias[i] = from_float<T>(i < embed ? dq[i] : 0.f);  // b_k cancels in the softmax, b_v is dead
}

// ---- fused scalar step (linear projectors linked to the ScalarAdapter; forward = merv_fused_linear_mix with the same w for every video).
//      merv_wgrad_video with scale_stride 0 gives dW_e = w_e dOut^T P_e and the partials of <W_e, dOut[b]^T P_e[b]> = <dOut[b], Y_e[b] - b_e>;
//      with gs = sum_b gsum[b] (the column sums of dOut over every token):
//          db_e = w_e gs,   g_e = sum of those partials + b_e . gs + dweights_out[e],   dscalar = w (.) (g - <w, g>)
struct ScalarFusedPtrs {
  const float* dw_partial[MERV_MAX_ENCODERS];  // [B, kPairDotChunks]
  const void* bias[MERV_MAX_ENCODERS];         // [K] or NULL
  void* db[MERV_MAX_ENCODERS];                 // [K] or NULL
};

// stage 1, grid ceil(K / 256): gs for 256 columns (videos in order), db_e, and the per-CTA sums of b_e . gs -> bpart[e, block]
template <typename T>
__global__ void __launch_bounds__(256) scalar_fused_bias_kernel(const __grid_constant__ ScalarFusedPtrs p, const float* __restrict__ gsum,
                                                                const float* __restrict__ weights, float* __restrict__ bpart, int B, int E, int K) {
  __shared__ float red[32];
  const int k = blockIdx.x * 256 + threadIdx.x;
  float gs = 0.f;
  if (k < K)
    for (int b = 0; b < B; ++b) gs += gsum[(long long)b * K + k];
  for (int e = 0; e < E; ++e) {
    float v = 0.f;
    if (k < K) {
      if (p.db[e] != nullptr) static_cast<T*>(p.db[e])[k] = from_float<T>(weights[e] * gs);
      if (p.bias[e] != nullptr) v = to_float(static_cast<const T*>(p.bias[e])[k]) * gs;
    }
    v = bwd_block_sum<256>(v, red);
    if (threadIdx.x == 0) bpart[(long long)e * gridDim.x + blockIdx.x] = v;
  }
}

// stage 2, one CTA: g_e = the wgrad_video partials of encoder e (videos in order) + its bpart row + dweights_out[e], then dscalar
__global__ void __launch_bounds__(256) scalar_fused_final_kernel(const __grid_constant__ ScalarFusedPtrs p, const float* __restrict__ bpart, int nbpart,
                                                                 const float* __restrict__ weights, const float* __restrict__ dweights_out,
                                                                 float* __restrict__ dscalar, int B, int E) {
  float acc[MERV_MAX_ENCODERS];
  const int n = B * kPairDotChunks;
#pragma unroll
  for (int e = 0; e < MERV_MAX_ENCODERS; ++e) {
    acc[e] = 0.f;
    if (e >= E) continue;
    for (int i = threadIdx.x; i < n; i += 256) acc[e] += p.dw_partial[e][i];
    for (int i = threadIdx.x; i < nbpart; i += 256) acc[e] += bpart[(long long)e * nbpart + i];
  }
  scalar_grad_from_block(acc, weights, dweights_out, dscalar, E);
}

}  // namespace merv

using namespace merv;

extern "C" int merv_transpose_rowscale(const void* x, void* y, int R, int R_pad, int C, int64_t ldx, int64_t ldy, const float* scale,
                                       int64_t scale_stride, int rows_per_scale, int dtype, void* stream);

extern "C" int merv_transpose(const void* x, void* y, int R, int C, int64_t ldx, int64_t ldy, int dtype, void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_transpose: unknown dtype %d", dtype);
  MERV_REQUIRE(x && y, MERV_E_ARG, "merv_transpose: NULL pointer");
  MERV_REQUIRE(R >= 0 && C >= 0 && ldx >= C && ldy >= R, MERV_E_SHAPE, "merv_transpose: R=%d C=%d ldx=%lld ldy=%lld", R, C, (long long)ldx, (long long)ldy);
  if (int rc = require_sm100()) return rc;
  if (R == 0 || C == 0) return MERV_OK;
  if (dtype == MERV_BF16 && C % 8 == 0 && R % 8 == 0 && ldx % 8 == 0 && ldy % 8 == 0 && aligned16(x) && aligned16(y))
    return merv_transpose_rowscale(x, y, R, R, C, ldx, ldy, nullptr, 0, 1, dtype, stream);
  dim3 grid((C + 31) / 32, (R + 31) / 32);
  MERV_REQUIRE(grid.y <= 65535, MERV_E_SHAPE, "merv_transpose: R=%d too large", R);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dtype == MERV_BF16)
    transpose_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)y, R, C, ldx, ldy);
  else
    transpose_kernel<float><<<grid, 256, 0, s>>>((const float*)x, (float*)y, R, C, ldx, ldy);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

extern "C" size_t merv_colsum_workspace(int M, int N) { return (size_t)((M + 255) / 256) * (size_t)(N > 0 ? N : 0); }

extern "C" int merv_colsum(const void* x, void* out, float* workspace, int M, int N, int64_t ld, int dtype, void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_colsum: unknown dtype %d", dtype);
  MERV_REQUIRE(x && out && workspace, MERV_E_ARG, "merv_colsum: NULL pointer");
  MERV_REQUIRE(M > 0 && N > 0 && ld >= N, MERV_E_SHAPE, "merv_colsum: M=%d N=%d ld=%lld", M, N, (long long)ld);
  if (int rc = require_sm100()) return rc;
  const int nblocks = (M + 255) / 256;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  dim3 grid((N + 255) / 256, nblocks);
  const int vec = dtype == MERV_BF16 ? 8 : 4;
  if (N % vec == 0 && ld % vec == 0 && aligned16(x)) {
    // vectorised first stage: video_colsum_kernel over blocks of 256 rows (16-byte loads, 4 in flight per thread, 32 row groups per
    // CTA) — the scalar kernel below reads 2 bytes per thread and load (3.2-3.5 TB/s on the 0.5 GB bias-gradient inputs); a tail of
    // fewer than 256 rows is a second launch.  Same partial layout [block, N] and the same fixed-order second stage.
    const int full = M / 256, tail = M - full * 256;
    const dim3 g1((N / vec + 7) / 8, full > 0 ? full : 1);
    if (dtype == MERV_BF16) {
      if (full > 0) video_colsum_kernel<__nv_bfloat16><<<g1, 256, 0, s>>>((const __nv_bfloat16*)x, workspace, 256, N, ld, 256 * ld, 1.0f);
      if (tail > 0)
        video_colsum_kernel<__nv_bfloat16><<<dim3(g1.x, 1), 256, 0, s>>>((const __nv_bfloat16*)x + (long long)full * 256 * ld, workspace + (size_t)full * N, tail, N,
                                                                          ld, 0, 1.0f);
      colsum_final_kernel<__nv_bfloat16><<<(N + 255) / 256, 256, 0, s>>>(workspace, (__nv_bfloat16*)out, N, nblocks);
    } else {
      if (full > 0) video_colsum_kernel<float><<<g1, 256, 0, s>>>((const float*)x, workspace, 256, N, ld, 256 * ld, 1.0f);
      if (tail > 0)
        video_colsum_kernel<float><<<dim3(g1.x, 1), 256, 0, s>>>((const float*)x + (long long)full * 256 * ld, workspace + (size_t)full * N, tail, N, ld, 0, 1.0f);
      colsum_final_kernel<float><<<(N + 255) / 256, 256, 0, s>>>(workspace, (float*)out, N, nblocks);
    }
    MERV_CUDA_OK(cudaGetLastError());
    return MERV_OK;
  }
  if (dtype == MERV_BF16) {
    colsum_partial_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, workspace, M, N, ld, 256);
    colsum_final_kernel<__nv_bfloat16><<<(N + 255) / 256, 256, 0, s>>>(workspace, (__nv_bfloat16*)out, N, nblocks);
  } else {
    colsum_partial_kernel<float><<<grid, 256, 0, s>>>((const float*)x, workspace, M, N, ld, 256);
    colsum_final_kernel<float><<<(N + 255) / 256, 256, 0, s>>>(workspace, (float*)out, N, nblocks);
  }
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

constexpr int kMixDqSplit = 16;  // row splits of the two-stage dQ = Wq^T dq (3072 x 3072: 96 CTAs in one stage could not fill the GPU)
// floats of the workspace without the single-token column sums: dw partials | vbar | ds | du (ku floats) | q | dq | dq partials
static size_t mix_bwd_base_floats(int B, int E, int K, size_t ku, int embed) {
  const size_t kblocks = (size_t)(K + kMixRedCols * 4 - 1) / (kMixRedCols * 4);  // upper bound (fp32 vectors are the narrower ones)
  return (size_t)B * E * kblocks + (size_t)B * E * K + (size_t)B * E + ku + 2 * (size_t)embed + (size_t)kMixDqSplit * embed;
}

extern "C" size_t merv_mix_backward_workspace(int B, int E, int T, int K, int embed) {
  (void)T;
  if (B <= 0 || E <= 0 || K <= 0) return 0;
  return mix_bwd_base_floats(B, E, K, (size_t)K, embed);
}

extern "C" size_t merv_mix_backward_ex_workspace(int B, int E, int T, int K, int embed, int64_t u_token_stride) {
  if (B <= 0 || E <= 0 || T <= 0 || K <= 0) return 0;
  const size_t ku = u_token_stride != 0 ? (size_t)T * K : (size_t)K;
  return mix_bwd_base_floats(B, E, K, ku, embed) + (size_t)B * K;  // + gsum [B, K] of the single-token encoders
}

// Every case of CrossAttentionAdapterLearnableQuery.forward (nn_utils.py:487-521).  V_e [B, T_e, K] with T_e = tokens[e] in {T, 1},
// dOut [B, T, K], weights fp32 [B, E] (forward output), dweights_out (optional) fp32 [B, E]: gradient w.r.t. the returned weights.
//   u_token_stride == 0 : averagetoken=True,  u fp32 [K],    s_e = u . (mean_t V_e + pe[e])     (pe [E, K] (ldpe) or NULL)
//   u_token_stride == K : averagetoken=False, u fp32 [T*K],  s_e = sum_t u[t,:] . V_e[b,t,:]    (pe must be NULL; Wk is [embed, T*K])
// Outputs: dV_e [B, T_e, K], dQ [embed], dWq [embed, embed], dWk [embed, T*K or K], dbias [3 * embed] and, with pe, dpe [E, K] (all `dtype`).
// The T-token-only, stride-0, pe-less call is merv_mix_backward: the same kernels, bit-identical gradients.
extern "C" int merv_mix_backward_ex(const void* const* V, const int32_t* tokens, const void* dOut, const float* weights, const float* dweights_out,
                                    const float* u, int64_t u_token_stride, const void* pe, int64_t ldpe, const void* Q, const void* Wq, const void* Wk,
                                    const void* in_proj_bias, void* const* dV, void* dQ, void* dWq, void* dWk, void* dbias, void* dpe, float* workspace,
                                    size_t workspace_floats, int B, int E, int T, int K, int embed, int dtype, void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_mix_backward_ex: unknown dtype %d", dtype);
  MERV_REQUIRE(V && tokens && dOut && weights && u && Q && Wq && Wk && dV && dQ && dWq && dWk && dbias && workspace, MERV_E_ARG,
               "merv_mix_backward_ex: NULL pointer");
  MERV_REQUIRE(E >= 1 && E <= MERV_MAX_ENCODERS, MERV_E_ARG, "merv_mix_backward_ex: E=%d", E);
  MERV_REQUIRE(B > 0 && T > 0 && K > 0 && embed > 0, MERV_E_SHAPE, "merv_mix_backward_ex: B=%d T=%d K=%d embed=%d", B, T, K, embed);
  const int vec = dtype == MERV_BF16 ? 8 : 4;
  MERV_REQUIRE(K % vec == 0, MERV_E_SHAPE, "merv_mix_backward_ex: K=%d must be a multiple of %d", K, vec);
  const bool flat = u_token_stride != 0;
  MERV_REQUIRE(!flat || u_token_stride == K, MERV_E_SHAPE, "merv_mix_backward_ex: u_token_stride=%lld (0 or K=%d)", (long long)u_token_stride, K);
  MERV_REQUIRE(!flat || (long long)T * K <= 0x7fffffffLL, MERV_E_SHAPE, "merv_mix_backward_ex: T*K overflows");
  MERV_REQUIRE(!(flat && pe), MERV_E_ARG, "merv_mix_backward_ex: pe is only read with averagetoken=True (u_token_stride == 0)");
  MERV_REQUIRE((pe == nullptr) == (dpe == nullptr), MERV_E_ARG, "merv_mix_backward_ex: pe and dpe go together");
  MERV_REQUIRE(pe == nullptr || ldpe >= K, MERV_E_SHAPE, "merv_mix_backward_ex: ldpe=%lld < K=%d", (long long)ldpe, K);
  MERV_REQUIRE(aligned16(u), MERV_E_ALIGN, "merv_mix_backward_ex: u must be 16-byte aligned");
  if (int rc = require_sm100()) return rc;
  BwdPtrs p = {};
  unsigned full_mask = 0;
  int gsum_e = -1;
  for (int e = 0; e < E; ++e) {
    MERV_REQUIRE(tokens[e] == T || tokens[e] == 1, MERV_E_SHAPE, "merv_mix_backward_ex: encoder %d has %d tokens, expected %d or 1", e, tokens[e], T);
    MERV_REQUIRE(V[e] && dV[e] && aligned16(V[e]) && aligned16(dV[e]), MERV_E_ALIGN, "merv_mix_backward_ex: encoder %d: NULL or misaligned tensor", e);
    p.V[e] = V[e];
    p.dV[e] = dV[e];
    p.tokens[e] = tokens[e];
    if (tokens[e] == T) full_mask |= 1u << e;
    else if (gsum_e < 0) gsum_e = e;
  }
  const int Ku = flat ? T * K : K;  // length of u, du and the rows of Wk / dWk
  const size_t base = mix_bwd_base_floats(B, E, K, (size_t)Ku, embed);
  MERV_REQUIRE(workspace_floats >= base + (gsum_e >= 0 ? (size_t)B * K : 0), MERV_E_ARG, "merv_mix_backward_ex: workspace too small");
  const int kblocks = (K / vec + kMixRedCols - 1) / kMixRedCols;
  float* dw_partial = workspace;
  float* vbar = dw_partial + (size_t)B * E * ((K + kMixRedCols * 4 - 1) / (kMixRedCols * 4));
  float* ds = vbar + (size_t)B * E * K;
  float* du = ds + (size_t)B * E;
  float* q = du + Ku;
  float* dq = q + embed;
  float* dq_partial = dq + embed;  // [kMixDqSplit, embed]
  float* gsum = workspace + base;  // [B, K], single-token encoders only
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const float rs = 1.0f / sqrtf(float(embed));
  const long long nWk = (long long)embed * Ku, nWq = (long long)embed * embed;
#define MERV_MIX_BWD_BODY(T_)                                                                                                                      \
  mix_bwd_reduce_kernel<T_><<<dim3(kblocks, E, B), 256, 0, s>>>(p, (const T_*)dOut, dw_partial, vbar, gsum, gsum_e, E, T, K);                     \
  mix_bwd_scores_kernel<<<B, 32, 0, s>>>(dw_partial, weights, dweights_out, ds, E, kblocks);                                                       \
  if (flat) {                                                                                                                                      \
    if (int rc = launch_mix_dv_flat<T_>(p, dOut, weights, ds, u, du, B, E, T, K, full_mask, s)) return rc;                                         \
  } else {                                                                                                                                         \
    if (full_mask != 0) {                                                                                                                          \
      if (int rc = launch_mix_dv<T_>(p, dOut, weights, ds, u, B, E, T, K, full_mask, s)) return rc;                                                \
    }                                                                                                                                              \
    if (pe != nullptr)                                                                                                                             \
      du_pe_kernel<T_><<<(K + 255) / 256, 256, 0, s>>>(ds, vbar, (const T_*)pe, ldpe, u, du, (T_*)dpe, B, E, K);                                   \
    else                                                                                                                                           \
      du_kernel<<<(K + 255) / 256, 256, 0, s>>>(ds, vbar, du, B * E, K);                                                                           \
  }                                                                                                                                                \
  if (gsum_e >= 0)                                                                                                                                 \
    mix_bwd_dv_single_kernel<T_><<<dim3((K + 255) / 256, B), 256, 0, s>>>(p, weights, ds, u, flat ? T : 1, gsum, E, K, full_mask);                 \
  launch_gemv_n<T_, T_>((const T_*)Wq, (const T_*)Q, (const T_*)in_proj_bias, q, embed, embed, 1.0f, s);                                          \
  launch_gemv_n<T_, float>((const T_*)Wk, du, nullptr, dq, embed, Ku, rs, s);                                                                      \
  outer_kernel<T_, float><<<(unsigned)((nWk + 255) / 256), 256, 0, s>>>(q, du, (T_*)dWk, embed, Ku, rs);                                          \
  outer_kernel<T_, T_><<<(unsigned)((nWq + 255) / 256), 256, 0, s>>>(dq, (const T_*)Q, (T_*)dWq, embed, embed, 1.0f);                             \
  gemv_tf_partial_kernel<T_><<<dim3((embed + 31) / 32, kMixDqSplit), 256, 0, s>>>((const T_*)Wq, dq, dq_partial, embed, embed);                    \
  fused_bwd_final_kernel<T_><<<(3 * embed + 255) / 256, 256, 0, s>>>(dq_partial, kMixDqSplit, dq, (T_*)dQ, (T_*)dbias, embed);
  if (dtype == MERV_BF16) {
    MERV_MIX_BWD_BODY(__nv_bfloat16)
  } else {
    MERV_MIX_BWD_BODY(float)
  }
#undef MERV_MIX_BWD_BODY
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

// V_e [B, T, K] (all encoders must have T tokens), dOut [B, T, K], weights fp32 [B, E] (forward output), u fp32 [K];
// dweights_out (optional) fp32 [B, E]: gradient w.r.t. the returned weights.  Outputs: dV_e [B, T, K] (dtype) and the parameter
// gradients dQ [embed], dWq [embed, embed], dWk [embed, K], dbias [3 * embed] in `dtype`.
extern "C" int merv_mix_backward(const void* const* V, const void* dOut, const float* weights, const float* dweights_out, const float* u,
                                 const void* Q, const void* Wq, const void* Wk, const void* in_proj_bias, void* const* dV, void* dQ, void* dWq,
                                 void* dWk, void* dbias, float* workspace, size_t workspace_floats, int B, int E, int T, int K, int embed,
                                 int dtype, void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_mix_backward: unknown dtype %d", dtype);
  MERV_REQUIRE(V && dOut && weights && u && Q && Wq && Wk && dV && dQ && dWq && dWk && dbias && workspace, MERV_E_ARG, "merv_mix_backward: NULL pointer");
  MERV_REQUIRE(E >= 1 && E <= MERV_MAX_ENCODERS, MERV_E_ARG, "merv_mix_backward: E=%d", E);
  MERV_REQUIRE(B > 0 && T > 0 && K > 0 && embed > 0, MERV_E_SHAPE, "merv_mix_backward: B=%d T=%d K=%d embed=%d", B, T, K, embed);
  const int vec = dtype == MERV_BF16 ? 8 : 4;
  MERV_REQUIRE(K % vec == 0, MERV_E_SHAPE, "merv_mix_backward: K=%d must be a multiple of %d", K, vec);
  MERV_REQUIRE(workspace_floats >= merv_mix_backward_workspace(B, E, T, K, embed), MERV_E_ARG, "merv_mix_backward: workspace too small");
  int32_t tokens[MERV_MAX_ENCODERS];
  for (int e = 0; e < E; ++e) tokens[e] = T;
  return merv_mix_backward_ex(V, tokens, dOut, weights, dweights_out, u, 0, nullptr, 0, Q, Wq, Wk, in_proj_bias, dV, dQ, dWq, dWk, dbias, nullptr,
                              workspace, workspace_floats, B, E, T, K, embed, dtype, stream);
}

// ---- ScalarAdapter backward (see the block comment above scalar_mix_bwd_kernel) -------------------------------------------------------
// floats of the [B, E, kblocks] partials; kblocks is bounded with the narrower fp32 vectors, as in mix_bwd_base_floats
extern "C" size_t merv_scalar_mix_backward_workspace(int B, int E, int K) {
  if (B <= 0 || E <= 0 || K <= 0) return 0;
  return (size_t)B * E * ((K + kMixRedCols * 4 - 1) / (kMixRedCols * 4));
}

// V_e, dOut, dV_e [B, T, K] contiguous (`dtype`), weights = softmax(scalar) fp32 [E], dweights_out fp32 [E] or NULL, dscalar fp32 [E].
// B == 0 (a rank without videos) reads no tensor and gives dscalar from dweights_out alone.
extern "C" int merv_scalar_mix_backward(const void* const* V, const void* dOut, const float* weights, const float* dweights_out, void* const* dV,
                                        float* dscalar, float* workspace, size_t workspace_floats, int B, int E, int T, int K, int dtype,
                                        void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_scalar_mix_backward: unknown dtype %d", dtype);
  MERV_REQUIRE(V && dV && weights && dscalar, MERV_E_ARG, "merv_scalar_mix_backward: NULL pointer");
  MERV_REQUIRE(E >= 1 && E <= MERV_MAX_ENCODERS, MERV_E_ARG, "merv_scalar_mix_backward: E=%d not in [1,%d]", E, MERV_MAX_ENCODERS);
  MERV_REQUIRE(B >= 0 && T > 0 && K > 0, MERV_E_SHAPE, "merv_scalar_mix_backward: B=%d T=%d K=%d", B, T, K);
  const int vec = dtype == MERV_BF16 ? 8 : 4;
  MERV_REQUIRE(K % vec == 0, MERV_E_SHAPE, "merv_scalar_mix_backward: K=%d must be a multiple of %d", K, vec);
  BwdPtrs p = {};
  if (B > 0) {
    MERV_REQUIRE(dOut && workspace, MERV_E_ARG, "merv_scalar_mix_backward: NULL pointer");
    MERV_REQUIRE(aligned16(dOut), MERV_E_ALIGN, "merv_scalar_mix_backward: dOut must be 16-byte aligned");
    for (int e = 0; e < E; ++e) {
      MERV_REQUIRE(V[e] && dV[e], MERV_E_ARG, "merv_scalar_mix_backward: encoder %d: NULL pointer", e);
      MERV_REQUIRE(aligned16(V[e]) && aligned16(dV[e]), MERV_E_ALIGN, "merv_scalar_mix_backward: encoder %d: tensor not 16-byte aligned", e);
      p.V[e] = V[e];
      p.dV[e] = dV[e];
      p.tokens[e] = T;
    }
    MERV_REQUIRE(workspace_floats >= merv_scalar_mix_backward_workspace(B, E, K), MERV_E_ARG, "merv_scalar_mix_backward: workspace too small");
  }
  MERV_REQUIRE(B <= 65535, MERV_E_SHAPE, "merv_scalar_mix_backward: B=%d too large", B);
  if (int rc = require_sm100()) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int kblocks = (K / vec + kMixRedCols - 1) / kMixRedCols;
  if (B > 0) {
    const int rc = dtype == MERV_BF16 ? launch_scalar_mix_bwd<__nv_bfloat16>(p, dOut, weights, workspace, B, E, T, K, kblocks, s)
                                      : launch_scalar_mix_bwd<float>(p, dOut, weights, workspace, B, E, T, K, kblocks, s);
    if (rc) return rc;
  }
  scalar_mix_fold_kernel<<<1, 256, 0, s>>>(workspace, weights, dweights_out, dscalar, B, E, kblocks);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

extern "C" size_t merv_scalar_fused_backward_workspace(int E, int K) {
  if (E <= 0 || K <= 0) return 0;
  return (size_t)E * ((K + 255) / 256);
}

// The fused scalar step after its merv_wgrad_video / merv_video_colsum calls: weights = softmax(scalar) fp32 [E], dweights_out fp32 [E] or
// NULL, gsum fp32 [B, K] (merv_video_colsum(dOut)), dw_partial[e] fp32 [B, merv_pair_dot_chunks()] (merv_wgrad_video of encoder e with
// scale_stride 0), bias[e] / db[e] [K] (`dtype`) or NULL, dscalar fp32 [E].
extern "C" int merv_scalar_fused_backward(const float* weights, const float* dweights_out, const float* gsum, const float* const* dw_partial,
                                          const void* const* bias, void* const* db, float* dscalar, float* workspace, size_t workspace_floats, int B,
                                          int E, int K, int dtype, void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_scalar_fused_backward: unknown dtype %d", dtype);
  MERV_REQUIRE(weights && dw_partial && bias && db && dscalar && workspace, MERV_E_ARG, "merv_scalar_fused_backward: NULL pointer");
  MERV_REQUIRE(E >= 1 && E <= MERV_MAX_ENCODERS, MERV_E_ARG, "merv_scalar_fused_backward: E=%d not in [1,%d]", E, MERV_MAX_ENCODERS);
  MERV_REQUIRE(B >= 0 && K > 0 && (long long)B * kPairDotChunks <= 0x7fffffffLL, MERV_E_SHAPE, "merv_scalar_fused_backward: B=%d K=%d", B, K);
  MERV_REQUIRE(B == 0 || gsum, MERV_E_ARG, "merv_scalar_fused_backward: NULL gsum");
  MERV_REQUIRE(workspace_floats >= merv_scalar_fused_backward_workspace(E, K), MERV_E_ARG, "merv_scalar_fused_backward: workspace too small");
  ScalarFusedPtrs p = {};
  for (int e = 0; e < E; ++e) {
    MERV_REQUIRE(B == 0 || dw_partial[e], MERV_E_ARG, "merv_scalar_fused_backward: encoder %d: NULL dw_partial", e);
    p.dw_partial[e] = dw_partial[e];
    p.bias[e] = bias[e];
    p.db[e] = db[e];
  }
  if (int rc = require_sm100()) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int nb = (K + 255) / 256;
  if (dtype == MERV_BF16)
    scalar_fused_bias_kernel<__nv_bfloat16><<<nb, 256, 0, s>>>(p, gsum, weights, workspace, B, E, K);
  else
    scalar_fused_bias_kernel<float><<<nb, 256, 0, s>>>(p, gsum, weights, workspace, B, E, K);
  scalar_fused_final_kernel<<<1, 256, 0, s>>>(p, workspace, nb, weights, dweights_out, dscalar, B, E);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

// out = gelu(z) (dy == NULL) or out = dy * gelu'(z); n elements, contiguous, n % (16 / sizeof) == 0
extern "C" int merv_gelu(const void* z, const void* dy, void* out, int64_t n, int dtype, void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_gelu: unknown dtype %d", dtype);
  MERV_REQUIRE(z && out, MERV_E_ARG, "merv_gelu: NULL pointer");
  const int vec = dtype == MERV_BF16 ? 8 : 4;
  MERV_REQUIRE(n >= 0 && n % vec == 0, MERV_E_SHAPE, "merv_gelu: n=%lld must be a multiple of %d", (long long)n, vec);
  MERV_REQUIRE(aligned16(z) && aligned16(out) && (dy == nullptr || aligned16(dy)), MERV_E_ALIGN, "merv_gelu: pointers must be 16-byte aligned");
  if (int rc = require_sm100()) return rc;
  if (n == 0) return MERV_OK;
  const long long nvec = n / vec;
  long long blocks = (nvec + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dtype == MERV_BF16) {
    using T_ = __nv_bfloat16;
    if (dy) gelu_kernel<T_, true><<<(unsigned)blocks, 256, 0, s>>>((const T_*)z, (const T_*)dy, (T_*)out, nvec);
    else gelu_kernel<T_, false><<<(unsigned)blocks, 256, 0, s>>>((const T_*)z, nullptr, (T_*)out, nvec);
  } else {
    if (dy) gelu_kernel<float, true><<<(unsigned)blocks, 256, 0, s>>>((const float*)z, (const float*)dy, (float*)out, nvec);
    else gelu_kernel<float, false><<<(unsigned)blocks, 256, 0, s>>>((const float*)z, nullptr, (float*)out, nvec);
  }
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

// ---- fused-path backward entry points (see the block comment above the kernels) ---------------------------------------------------
extern "C" int merv_video_colsum(const void* x, float* out, int B, int T, int K, int64_t ld, int64_t batch_stride, float scale, int dtype,
                                 void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_video_colsum: unknown dtype %d", dtype);
  MERV_REQUIRE(x && out, MERV_E_ARG, "merv_video_colsum: NULL pointer");
  const int vec = dtype == MERV_BF16 ? 8 : 4;
  MERV_REQUIRE(B >= 0 && T > 0 && K > 0 && K % vec == 0 && ld >= K && ld % vec == 0 && batch_stride % vec == 0, MERV_E_SHAPE,
               "merv_video_colsum: B=%d T=%d K=%d ld=%lld batch_stride=%lld", B, T, K, (long long)ld, (long long)batch_stride);
  MERV_REQUIRE(aligned16(x), MERV_E_ALIGN, "merv_video_colsum: x must be 16-byte aligned");
  if (int rc = require_sm100()) return rc;
  if (B == 0) return MERV_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  dim3 grid((K / vec + 7) / 8, B);
  if (dtype == MERV_BF16)
    video_colsum_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, out, T, K, ld, batch_stride, scale);
  else
    video_colsum_kernel<float><<<grid, 256, 0, s>>>((const float*)x, out, T, K, ld, batch_stride, scale);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

extern "C" int merv_pair_dot_chunks(void) { return kPairDotChunks; }

// out[b, c] = sum_{i = c, c + chunks, ...} in[b, i] (ascending i: fixed order): folds the per-(tile, warp) dots of merv_wgrad_video into the
// [B, merv_pair_dot_chunks()] layout merv_fused_backward reads
__global__ void __launch_bounds__(32) fold_partials_kernel(const float* __restrict__ in, float* __restrict__ out, int parts) {
  const int b = blockIdx.x, c = threadIdx.x;
  float acc = 0.f;
  for (int i = c; i < parts; i += kPairDotChunks) acc += in[(long long)b * parts + i];
  if (c < kPairDotChunks) out[(long long)b * kPairDotChunks + c] = acc;
}

// dW[m, n] = bf16(sum_q partial[q, m, n]) (ascending q: fixed order) — the fold of a weight gradient that was split over the videos
__global__ void __launch_bounds__(256) fold_wgrad_parts_kernel(const float* __restrict__ partial, __nv_bfloat16* __restrict__ dW, long long lddw, int M, int N,
                                                               int parts) {
  const long long v = (long long)blockIdx.x * 256 + threadIdx.x;  // one 4-column vector per thread
  const int nv = N / 4;
  if (v >= (long long)M * nv) return;
  const long long m = v / nv, n = (v % nv) * 4;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int q = 0; q < parts; ++q) {
    const float4 x = __ldcs(reinterpret_cast<const float4*>(partial + ((long long)q * M + m) * N + n));
    acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
  }
  uint2 o = make_uint2(pack_bf16x2(acc.x, acc.y), pack_bf16x2(acc.z, acc.w));
  *reinterpret_cast<uint2*>(dW + m * lddw + n) = o;
}

extern "C" int merv_wgrad_video_parts(int N_out, int C) { return wgrad_video_parts(N_out, C); }
/* floats of workspace merv_wgrad_video needs: the per-(video, tile, warp) dots + the fp32 partial tiles of a split over the videos */
extern "C" size_t merv_wgrad_video_workspace(int videos, int N_out, int C) {
  if (videos <= 0 || N_out <= 0 || C <= 0) return 0;
  const int split = wgrad_video_split(N_out, C, videos);
  size_t dots = (size_t)videos * wgrad_video_parts(N_out, C);
  dots = (dots + 3) / 4 * 4;  // keeps the partial tiles 16-byte aligned
  return dots + (split > 1 ? (size_t)split * N_out * C : 0);
}

extern "C" int merv_wgrad_video(const void* dY, int64_t lddy, const void* X, int64_t ldx, const float* scale, int64_t scale_stride, const void* W,
                                int64_t ldw, void* dW, int64_t lddw, float* dot_partial, float* workspace, int videos, int tokens_per_video,
                                int N_out, int C, void* stream) {
  MERV_REQUIRE(dY && X && W && dW && dot_partial && workspace, MERV_E_ARG, "merv_wgrad_video: NULL pointer");
  MERV_REQUIRE(videos >= 0 && tokens_per_video > 0 && N_out > 0 && C > 0, MERV_E_SHAPE, "merv_wgrad_video: videos=%d tokens=%d N_out=%d C=%d", videos,
               tokens_per_video, N_out, C);
  MERV_REQUIRE(tokens_per_video % 64 == 0, MERV_E_SHAPE, "merv_wgrad_video: tokens_per_video=%d must be a multiple of 64 (one k-block never spans two videos)",
               tokens_per_video);
  MERV_REQUIRE((long long)videos * tokens_per_video <= 0x7fffffffLL, MERV_E_SHAPE, "merv_wgrad_video: videos * tokens overflows");
  MERV_REQUIRE(lddy >= N_out && ldx >= C && ldw >= C && lddw >= C, MERV_E_SHAPE, "merv_wgrad_video: leading dimensions too small");
  static_assert(kPairDotChunks == 32, "fold_partials_kernel: one lane per chunk");
  if (int rc = require_sm100()) return rc;
  if (videos == 0) return MERV_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // dW [N_out, C] = dY^T X: A-operand = dY [tokens, N_out] read as [K, M], W-operand = X [tokens, C] read as [K, N] (both MN-major, in place)
  GemmSegment seg = {dY, lddy, X, ldx, videos * tokens_per_video, 1, 1};
  const int split = (C % 4 == 0 && lddw % 4 == 0) ? wgrad_video_split(N_out, C, videos) : 1;
  size_t dots = (size_t)videos * wgrad_video_parts(N_out, C);
  dots = (dots + 3) / 4 * 4;
  float* partial = split > 1 ? workspace + dots : nullptr;
  MERV_REQUIRE(aligned16(workspace), MERV_E_ALIGN, "merv_wgrad_video: workspace must be 16-byte aligned");
  WgradVideoArgs vid = {videos, tokens_per_video / 64, scale, scale_stride, W, ldw, workspace, split, partial};
  if (int rc = launch_gemm_tcgen05(&seg, 1, nullptr, nullptr, N_out, nullptr, MERV_ACT_NONE, nullptr, nullptr, dW, lddw, 0, N_out, C, 0, s, nullptr, 0,
                                   false, nullptr, nullptr, &vid))
    return rc;
  if (split > 1) {
    const long long vecs = (long long)N_out * (C / 4);
    fold_wgrad_parts_kernel<<<(unsigned)((vecs + 255) / 256), 256, 0, s>>>(partial, static_cast<__nv_bfloat16*>(dW), lddw, N_out, C, split);
    MERV_CUDA_OK(cudaGetLastError());
  }
  fold_partials_kernel<<<videos, 32, 0, s>>>(workspace, dot_partial, wgrad_video_parts(N_out, C));
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

extern "C" int merv_pair_dot_scale(const void* x, const void* y, float* partial, const float* scale, int64_t scale_stride, void* y_scaled, int B,
                                   int64_t n, int dtype, void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_pair_dot: unknown dtype %d", dtype);
  MERV_REQUIRE(x && y && partial, MERV_E_ARG, "merv_pair_dot: NULL pointer");
  MERV_REQUIRE((scale == nullptr) == (y_scaled == nullptr), MERV_E_ARG, "merv_pair_dot_scale: scale and y_scaled go together");
  const int vec = dtype == MERV_BF16 ? 8 : 4;
  MERV_REQUIRE(B >= 0 && n > 0 && n % vec == 0, MERV_E_SHAPE, "merv_pair_dot: B=%d n=%lld", B, (long long)n);
  MERV_REQUIRE(aligned16(x) && aligned16(y) && (y_scaled == nullptr || aligned16(y_scaled)), MERV_E_ALIGN, "merv_pair_dot: operands must be 16-byte aligned");
  if (int rc = require_sm100()) return rc;
  if (B == 0) return MERV_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  dim3 grid(kPairDotChunks, B);
  if (dtype == MERV_BF16)
    pair_dot_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, (const __nv_bfloat16*)y, partial, n / vec, scale, scale_stride,
                                                        (__nv_bfloat16*)y_scaled);
  else
    pair_dot_kernel<float><<<grid, 256, 0, s>>>((const float*)x, (const float*)y, partial, n / vec, scale, scale_stride, (float*)y_scaled);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

extern "C" int merv_pair_dot(const void* x, const void* y, float* partial, int B, int64_t n, int dtype, void* stream) {
  return merv_pair_dot_scale(x, y, partial, nullptr, 0, nullptr, B, n, dtype, stream);
}

extern "C" int merv_transpose_rowscale(const void* x, void* y, int R, int R_pad, int C, int64_t ldx, int64_t ldy, const float* scale,
                                       int64_t scale_stride, int rows_per_scale, int dtype, void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_transpose_rowscale: unknown dtype %d", dtype);
  MERV_REQUIRE(x && y, MERV_E_ARG, "merv_transpose_rowscale: NULL pointer");
  MERV_REQUIRE(R >= 0 && C >= 0 && R_pad >= R && ldx >= C && ldy >= R_pad && (scale == nullptr || rows_per_scale > 0), MERV_E_SHAPE,
               "merv_transpose_rowscale: R=%d R_pad=%d C=%d ldx=%lld ldy=%lld rows_per_scale=%d", R, R_pad, C, (long long)ldx, (long long)ldy,
               rows_per_scale);
  if (int rc = require_sm100()) return rc;
  if (R_pad == 0 || C == 0) return MERV_OK;
  dim3 grid((C + 63) / 64, (R_pad + 63) / 64);
  MERV_REQUIRE(grid.y <= 65535, MERV_E_SHAPE, "merv_transpose_rowscale: R=%d too large", R);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool vec_ok = dtype == MERV_BF16 && C % 8 == 0 && R_pad % 8 == 0 && ldx % 8 == 0 && ldy % 8 == 0 && aligned16(x) && aligned16(y);
  if (vec_ok)
    transpose_bf16_vec_kernel<<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)y, R, R_pad, C, ldx, ldy, scale, scale_stride, rows_per_scale);
  else if (dtype == MERV_BF16)
    transpose_rowscale_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)y, R, R_pad, C, ldx, ldy, scale, scale_stride,
                                                                 rows_per_scale);
  else
    transpose_rowscale_kernel<float><<<grid, 256, 0, s>>>((const float*)x, (float*)y, R, R_pad, C, ldx, ldy, scale, scale_stride, rows_per_scale);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

constexpr int kDqSplits = 8;
extern "C" size_t merv_fused_backward_workspace(const merv_fused_bwd_desc* d) {
  if (d == nullptr || d->E <= 0) return 0;
  size_t g = 0;
  for (int e = 0; e < d->E && e < MERV_MAX_ENCODERS; ++e) g += (size_t)d->C[e];
  return g + (size_t)d->K + (2 + kDqSplits) * (size_t)d->embed;
}

extern "C" int merv_fused_backward(const merv_fused_bwd_desc* d, int dtype, void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_fused_backward: unknown dtype %d", dtype);
  MERV_REQUIRE(d != nullptr, MERV_E_ARG, "merv_fused_backward: NULL descriptor");
  const int B = d->B, E = d->E, K = d->K, embed = d->embed;
  MERV_REQUIRE(E >= 1 && E <= MERV_MAX_ENCODERS, MERV_E_ARG, "merv_fused_backward: E=%d", E);
  MERV_REQUIRE(B > 0 && K > 0 && embed > 0, MERV_E_SHAPE, "merv_fused_backward: B=%d K=%d embed=%d", B, K, embed);
  MERV_REQUIRE(d->weights && d->u && d->gsum && d->ds && d->Q && d->Wq && d->Wk && d->dQ && d->dWq && d->dWk && d->dbias && d->workspace, MERV_E_ARG,
               "merv_fused_backward: NULL pointer");
  MERV_REQUIRE(d->workspace_floats >= merv_fused_backward_workspace(d), MERV_E_ARG, "merv_fused_backward: workspace too small");
  if (int rc = require_sm100()) return rc;
  FusedBwdPtrs p = {};
  int goff = 0, cmax = 0;
  for (int e = 0; e < E; ++e) {
    MERV_REQUIRE(d->dw_partial[e] && d->pbar[e] && d->W[e] && d->dW[e] && d->C[e] > 0 && d->ldw[e] >= d->C[e] && d->lddw[e] >= d->C[e], MERV_E_ARG,
                 "merv_fused_backward: encoder %d: NULL pointer or bad leading dimension", e);
    p.dw_partial[e] = d->dw_partial[e];
    p.pbar[e] = d->pbar[e];
    p.W[e] = d->W[e];
    p.bias[e] = d->bias[e];
    p.dW[e] = d->dW[e];
    p.db[e] = d->db[e];
    p.ldw[e] = d->ldw[e];
    p.lddw[e] = d->lddw[e];
    p.C[e] = d->C[e];
    p.goff[e] = goff;
    goff += d->C[e];
    cmax = d->C[e] > cmax ? d->C[e] : cmax;
  }
  float* g = d->workspace;
  float* du = g + goff;
  float* q = du + K;
  float* dq = q + embed;
  float* dqp = dq + embed;
  const int vec = dtype == MERV_BF16 ? 8 : 4;
  bool vec_rows = goff % 4 == 0;  // g_e offsets stay 16-byte aligned
  for (int e = 0; e < E; ++e)
    vec_rows = vec_rows && p.C[e] % vec == 0 && p.ldw[e] % vec == 0 && p.lddw[e] % vec == 0 && aligned16(p.W[e]) && aligned16(p.dW[e]) && p.goff[e] % 4 == 0;
  const bool vec_outer = K % vec == 0 && embed % vec == 0 && goff % 4 == 0 && aligned16(d->workspace) && aligned16(d->Q) && aligned16(d->dWk) && aligned16(d->dWq);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const float rs = 1.0f / sqrtf(float(embed));
#define MERV_FUSED_BWD_BODY(T_)                                                                                                                   \
  fused_bwd_scores_kernel<T_><<<B, 32, 0, s>>>(p, d->gsum, d->weights, d->dweights_out, d->ds, E, K);                                             \
  fused_bwd_g_kernel<<<dim3((cmax + 255) / 256, E), 256, 0, s>>>(p, d->ds, g, B, E);                                                              \
  fused_bwd_db_kernel<T_><<<dim3((K + 255) / 256, E), 256, 0, s>>>(p, d->gsum, d->weights, d->ds, d->u, B, E, K);                                 \
  if (vec_rows) {                                                                                                                                 \
    fused_bwd_rank1_kernel<T_, true><<<dim3(sm_count() * 4, E), 256, 0, s>>>(p, d->u, g, K);                                                      \
    fused_bwd_du_kernel<T_, true><<<(K + 7) / 8, 256, 0, s>>>(p, g, d->ds, du, K, B, E);                                                          \
  } else {                                                                                                                                        \
    fused_bwd_rank1_kernel<T_, false><<<dim3(sm_count() * 4, E), 256, 0, s>>>(p, d->u, g, K);                                                     \
    fused_bwd_du_kernel<T_, false><<<(K + 7) / 8, 256, 0, s>>>(p, g, d->ds, du, K, B, E);                                                         \
  }                                                                                                                                               \
  launch_gemv_n<T_, T_>((const T_*)d->Wq, (const T_*)d->Q, (const T_*)d->in_proj_bias, q, embed, embed, 1.0f, s);                                \
  launch_gemv_n<T_, float>((const T_*)d->Wk, du, nullptr, dq, embed, K, rs, s);                                                                  \
  if (vec_outer)                                                                                                                                  \
    fused_bwd_outer_kernel<T_, true><<<dim3(sm_count() * 4, 2), 256, 0, s>>>(q, du, dq, (const T_*)d->Q, (T_*)d->dWk, (T_*)d->dWq, embed, K, rs); \
  else                                                                                                                                            \
    fused_bwd_outer_kernel<T_, false><<<dim3(sm_count() * 4, 2), 256, 0, s>>>(q, du, dq, (const T_*)d->Q, (T_*)d->dWk, (T_*)d->dWq, embed, K, rs);\
  gemv_tf_partial_kernel<T_><<<dim3((embed + 31) / 32, kDqSplits), 256, 0, s>>>((const T_*)d->Wq, dq, dqp, embed, embed);                         \
  fused_bwd_final_kernel<T_><<<(3 * embed + 255) / 256, 256, 0, s>>>(dqp, kDqSplits, dq, (T_*)d->dQ, (T_*)d->dbias, embed);
  if (dtype == MERV_BF16) {
    MERV_FUSED_BWD_BODY(__nv_bfloat16)
  } else {
    MERV_FUSED_BWD_BODY(float)
  }
#undef MERV_FUSED_BWD_BODY
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}
