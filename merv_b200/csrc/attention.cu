// Cross attention of the attentive pooler ("attntv" resampler): a few learned queries attend to the patch tokens of one frame.
//   CrossAttention.forward, merv/util/nn_utils.py:393-412 (called from CrossAttentionBlock.forward :447-451 inside
//   AttentivePooler.forward :229-238):  out[b, q, h*hd:(h+1)*hd] = softmax_k(scale * Q[q, h] . K[b, k, h]) V[b, k, h]
// with K, V the two halves of the `kv` Linear's output row ([K(C) | V(C)], heads contiguous inside each half, :398-399) and the
// same projected queries for every batch entry (the query tokens are parameters, :196,232).
//
// First version: fp32 SIMT flash-style kernel for both storage dtypes (exact softmax in fp32: it is also what the fp32 parity path
// needs).  CTA = (head, batch entry), 8 warps; a warp owns 8 queries at a time, keys are staged in shared memory 64 at a time, online
// softmax across the chunks, probabilities go through a per-warp shared tile to the P.V phase.  K/V are read from HBM/L2 once per 64
// queries.  The two contractions are 2 * n_q * n_kv * C FLOP per frame on the CUDA cores; bf16 frames that fit its tile run the
// tcgen05 kernel instead (attention_tcgen05.cu, DESIGN.md §5.6).  The backward of every shape this kernel runs is below.
#include "common.cuh"

namespace merv {

constexpr int kAttWarps = 8;
constexpr int kAttQB = 8;     // queries per warp and pass: 64 queries per CTA pass
constexpr int kAttKeys = 64;  // keys staged per chunk

// Shared memory per CTA: K chunk in the storage dtype (padded rows), V chunk and the queries as fp32, one probability tile per warp.
// The kernel is issue- and shared-memory-bound, not FMA-bound (profiles/r1g_prof_cross_attention.txt), hence: 8 queries x 2 keys of
// register blocking per lane (one K load feeds 8 queries, one Q load 2 keys), K read 8 dims per 16-byte load when it is bf16, and both
// contractions on the packed fp32 pipe (fma.rn.f32x2): pairs of head dims in Q K^T, pairs of queries in P V.
template <typename T>
__host__ __device__ constexpr size_t att_smem_bytes(int hd) {
  constexpr int VEC = 16 / (int)sizeof(T);
  return (size_t)kAttKeys * (hd + VEC) * sizeof(T) +
         ((size_t)kAttKeys * hd + (size_t)kAttWarps * kAttQB * hd + (size_t)kAttWarps * kAttQB * kAttKeys) * sizeof(float);
}

template <typename T>
__device__ __forceinline__ void att_stage(float* dst, const uint4& r) {
  constexpr int VEC = Vec16<T>::kN;
  float f[VEC];
  Vec16<T>::unpack(r, f);
#pragma unroll
  for (int c = 0; c < VEC; c += 4) *reinterpret_cast<float4*>(dst + c) = make_float4(f[c], f[c + 1], f[c + 2], f[c + 3]);
}

template <typename T, int DPL>
__global__ void __launch_bounds__(kAttWarps * 32) cross_attention_kernel(const T* __restrict__ q, long long ldq, long long q_batch_stride,
                                                                        const T* __restrict__ kv, long long ldkv, T* __restrict__ out, long long ldo,
                                                                        int n_q, int n_kv, int hd, int C, float scale) {
  constexpr int VEC = Vec16<T>::kN;
  constexpr int P = Pairs<T>::kP;  // fp32 pairs per 16-byte vector of T
  constexpr int KC = kAttKeys;
  constexpr int KPL = KC / 32;  // keys per lane in the score phase
  constexpr int QB = kAttQB;
  typedef unsigned long long u64;
  extern __shared__ uint4 att_smem[];
  const int kpitch = hd + VEC;  // padded K rows: lanes read different rows with 16-byte loads, conflict-free
  T* Ks = reinterpret_cast<T*>(att_smem);
  float* Vs = reinterpret_cast<float*>(Ks + KC * kpitch);
  float* Qs = Vs + KC * hd;
  float* Ps = Qs + kAttWarps * QB * hd;
  const int h = blockIdx.x, b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const T* kb = kv + (long long)b * n_kv * ldkv + (long long)h * hd;  // K head slice of row 0; V is C columns further
  const T* qb = q + (long long)b * q_batch_stride + (long long)h * hd;
  float* Qw = Qs + warp * QB * hd;
  float* Pw = Ps + warp * QB * KC;  // [key][query]: the 8 queries of one key are adjacent (pairs of queries in the P V phase)
  const int hv = hd / VEC;

  for (int q0 = 0; q0 < n_q; q0 += kAttWarps * QB) {
    const int qbase = q0 + warp * QB;
    // this warp's queries -> shared as fp32 (zeros past n_q)
    for (int i = lane; i < QB * hv; i += 32) {
      const int j = i / hv, v = i - j * hv;
      uint4 r = make_uint4(0u, 0u, 0u, 0u);
      if (qbase + j < n_q) r = ldg_v4(qb + (long long)(qbase + j) * ldq + v * VEC);
      att_stage<T>(Qw + j * hd + v * VEC, r);
    }
    float m[QB], l[QB];
    u64 o2[QB / 2][DPL];  // (query 2 jp, query 2 jp + 1) x head dim i * 32 + lane
#pragma unroll
    for (int j = 0; j < QB; ++j) {
      m[j] = -INFINITY;
      l[j] = 0.f;
    }
#pragma unroll
    for (int jp = 0; jp < QB / 2; ++jp)
#pragma unroll
      for (int i = 0; i < DPL; ++i) o2[jp][i] = f32x2_pack(0.f, 0.f);
    for (int c0 = 0; c0 < n_kv; c0 += KC) {
      __syncthreads();  // everyone is done with the previous chunk (and the Q tile is written)
      for (int i = threadIdx.x; i < KC * hv; i += kAttWarps * 32) {
        const int r = i / hv, v = i - r * hv;
        uint4 kk = make_uint4(0u, 0u, 0u, 0u), vv = kk;
        if (c0 + r < n_kv) {
          const T* row = kb + (long long)(c0 + r) * ldkv + v * VEC;
          kk = ldg_nc_v4(row);
          vv = ldg_nc_v4(row + C);
        }
        *reinterpret_cast<uint4*>(Ks + r * kpitch + v * VEC) = kk;
        att_stage<T>(Vs + r * hd + v * VEC, vv);
      }
      __syncthreads();
      // ---- scores of this warp's 8 queries against the chunk: lane owns keys lane and lane + 32; pairs of head dims ----
      u64 s2[QB][KPL];
#pragma unroll
      for (int j = 0; j < QB; ++j)
#pragma unroll
        for (int t = 0; t < KPL; ++t) s2[j][t] = f32x2_pack(0.f, 0.f);
      for (int v = 0; v < hv; ++v) {
        u64 kf[KPL][P];
#pragma unroll
        for (int t = 0; t < KPL; ++t) Pairs<T>::unpack(*reinterpret_cast<const uint4*>(Ks + (t * 32 + lane) * kpitch + v * VEC), kf[t]);
#pragma unroll
        for (int j = 0; j < QB; ++j) {
#pragma unroll
          for (int h2 = 0; h2 < P / 2; ++h2) {
            const ulonglong2 qq = *reinterpret_cast<const ulonglong2*>(Qw + j * hd + v * VEC + h2 * 4);  // broadcast: two pairs
#pragma unroll
            for (int t = 0; t < KPL; ++t) {
              s2[j][t] = f32x2_fma(qq.x, kf[t][2 * h2], s2[j][t]);
              s2[j][t] = f32x2_fma(qq.y, kf[t][2 * h2 + 1], s2[j][t]);
            }
          }
        }
      }
      // ---- online softmax update, probabilities to the warp's shared tile ----
#pragma unroll
      for (int j = 0; j < QB; ++j) {
        float sv[KPL];
        float mx = -INFINITY;
#pragma unroll
        for (int t = 0; t < KPL; ++t) {
          float a0, a1;
          f32x2_unpack(s2[j][t], a0, a1);
          sv[t] = (c0 + t * 32 + lane < n_kv) ? (a0 + a1) * scale : -INFINITY;
          mx = fmaxf(mx, sv[t]);
        }
        mx = warp_max(mx);
        const float m_new = fmaxf(m[j], mx);  // finite: every chunk holds at least one key
        const float alpha = expf(m[j] - m_new);
        float rs = 0.f;
#pragma unroll
        for (int t = 0; t < KPL; ++t) {
          const float p = expf(sv[t] - m_new);
          Pw[(t * 32 + lane) * QB + j] = p;
          rs += p;
        }
        rs = warp_sum(rs);
        l[j] = l[j] * alpha + rs;
        m[j] = m_new;
        // rescale this query's half of its accumulator pairs
        const u64 a2 = (j & 1) ? f32x2_pack(1.0f, alpha) : f32x2_pack(alpha, 1.0f);
#pragma unroll
        for (int i = 0; i < DPL; ++i) o2[j / 2][i] = f32x2_mul(o2[j / 2][i], a2);
      }
      __syncwarp();
      // ---- o += P V: lane owns head dims lane, lane + 32, ...; pairs of queries ----
#pragma unroll 2
      for (int k = 0; k < KC; ++k) {
        const ulonglong2 pa = *reinterpret_cast<const ulonglong2*>(Pw + k * QB);      // broadcast: queries 0..3 of key k
        const ulonglong2 pb = *reinterpret_cast<const ulonglong2*>(Pw + k * QB + 4);  // queries 4..7
#pragma unroll
        for (int i = 0; i < DPL; ++i) {
          const int d = i * 32 + lane;
          const float vv = d < hd ? Vs[k * hd + d] : 0.f;
          const u64 v2 = f32x2_pack(vv, vv);
          o2[0][i] = f32x2_fma(pa.x, v2, o2[0][i]);
          o2[1][i] = f32x2_fma(pa.y, v2, o2[1][i]);
          o2[2][i] = f32x2_fma(pb.x, v2, o2[2][i]);
          o2[3][i] = f32x2_fma(pb.y, v2, o2[3][i]);
        }
      }
      __syncwarp();
    }
    // ---- normalise and store (heads concatenated along the channel dimension, nn_utils.py:409) ----
#pragma unroll
    for (int jp = 0; jp < QB / 2; ++jp) {
#pragma unroll
      for (int i = 0; i < DPL; ++i) {
        const int d = i * 32 + lane;
        float oa, ob;
        f32x2_unpack(o2[jp][i], oa, ob);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int j = 2 * jp + half;
          if (qbase + j < n_q && d < hd) {
            const float val = (half ? ob : oa) / l[j];
            T* dst = out + ((long long)b * n_q + qbase + j) * ldo + (long long)h * hd + d;
            if constexpr (sizeof(T) == 2) *dst = __float2bfloat16_rn(val);
            else *dst = val;
          }
        }
      }
    }
  }
}

// ---- backward on the CUDA cores: every shape the SIMT forward runs, fp32 and bf16 ----------------------------------------------
// CTA = (head, frame), 8 warps, a query block = 64 queries (8 per warp), a key chunk = 64 keys.  No softmax statistics come from the
// forward, so the kernel makes two sweeps:
//   1. per query block, over all key chunks: online row max m and sum l of exp(S - m), and D = sum_j P_ij dP_ij with dP = dO V^T
//      (rescaled alongside l), written to the CTA's stats slice of the workspace;
//   2. keys outer: per key chunk, over all query blocks, S and dP again, P = exp(S - m) / l, dS = scale P (.) (dP - D) into shared
//      tiles; dV = P^T dO and dK = dS^T Q of the chunk's keys stay in registers until the last query block and are written once;
//      dQ = dS K of the block is added to the CTA's fp32 dQ slice (the last chunk writes dq instead).
// Every sum runs in a fixed order with no atomics (a CTA owns its outputs and workspace slices), so results are bit-reproducible and a
// frame does not depend on the others in the batch.  P stays fp32; everything is accumulated in fp32 and rounded once on store.
constexpr int kAbQBlock = kAttWarps * kAttQB;  // 64 queries per block

__host__ __device__ constexpr int att_bwd_kpitch(int hd) { return hd % 8 ? hd : hd + 4; }  // odd multiple of 4: conflict-free row reads
__host__ __device__ constexpr size_t att_bwd_smem_bytes(int hd) {
  // K and V chunks (padded rows), Q and dO of the query block, the P and dS tiles [query][key]; all fp32
  return ((size_t)2 * kAttKeys * att_bwd_kpitch(hd) + (size_t)2 * kAbQBlock * hd + (size_t)2 * kAbQBlock * kAttKeys) * sizeof(float);
}
constexpr size_t kAbSmemMax = att_bwd_smem_bytes(128);

// rows r0 .. r0 + 63 of a [rows, hd] slice (rows `ld` apart, zeros past n) -> shared fp32 rows `pitch` apart
template <typename T>
__device__ __forceinline__ void att_bwd_stage(float* dst, int pitch, const T* src, long long ld, int r0, int n, int hd) {
  constexpr int VEC = Vec16<T>::kN;
  const int hv = hd / VEC;
  for (int i = threadIdx.x; i < 64 * hv; i += kAttWarps * 32) {
    const int r = i / hv, v = i - r * hv;
    uint4 x = make_uint4(0u, 0u, 0u, 0u);
    if (r0 + r < n) x = ldg_v4(src + (long long)(r0 + r) * ld + v * VEC);
    att_stage<T>(dst + r * pitch + v * VEC, x);
  }
}

// s2[j][t] = pairs of partial dot products of row j of A (this warp's 8 rows, `hd` apart) with row t * 32 + lane of B (`kp` apart):
// the score is the sum of the two halves
__device__ __forceinline__ void att_bwd_dots(const float* A, const float* Bm, int hd, int kp, int lane, unsigned long long (&s2)[kAttQB][2]) {
#pragma unroll
  for (int j = 0; j < kAttQB; ++j) s2[j][0] = s2[j][1] = f32x2_pack(0.f, 0.f);
  for (int v = 0; v < hd; v += 4) {
    ulonglong2 bf[2];
#pragma unroll
    for (int t = 0; t < 2; ++t) bf[t] = *reinterpret_cast<const ulonglong2*>(Bm + (t * 32 + lane) * kp + v);
#pragma unroll
    for (int j = 0; j < kAttQB; ++j) {
      const ulonglong2 a = *reinterpret_cast<const ulonglong2*>(A + j * hd + v);  // broadcast
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        s2[j][t] = f32x2_fma(a.x, bf[t].x, s2[j][t]);
        s2[j][t] = f32x2_fma(a.y, bf[t].y, s2[j][t]);
      }
    }
  }
}

__device__ __forceinline__ float att_bwd_sum2(unsigned long long x) {
  float a, b;
  f32x2_unpack(x, a, b);
  return a + b;
}

template <typename T>
__device__ __forceinline__ void att_bwd_store(T* dst, float v) {
  if constexpr (sizeof(T) == 2) *dst = __float2bfloat16_rn(v);
  else *dst = v;
}

template <typename T, int DPL>
__global__ void __launch_bounds__(kAttWarps * 32) cross_attention_bwd_kernel(const T* __restrict__ q, long long ldq, long long q_batch_stride,
                                                                            const T* __restrict__ kv, long long ldkv, const T* __restrict__ dout,
                                                                            long long lddo, T* __restrict__ dq, long long lddq, T* __restrict__ dkv,
                                                                            long long lddkv, float* __restrict__ ws, int n_q, int n_kv, int hd,
                                                                            int C, float scale) {
  constexpr int KC = kAttKeys, QB = kAttQB, QBLK = kAbQBlock;
  typedef unsigned long long u64;
  extern __shared__ float4 ab_smem[];
  const int kp = att_bwd_kpitch(hd);
  float* Ks = reinterpret_cast<float*>(ab_smem);
  float* Vs = Ks + KC * kp;
  float* Qs = Vs + KC * kp;
  float* Gs = Qs + QBLK * hd;  // dO
  float* Ps = Gs + QBLK * hd;  // [query][key]
  float* Ss = Ps + QBLK * KC;  // dS, [query][key]
  const int h = blockIdx.x, b = blockIdx.y, heads = gridDim.x, batches = gridDim.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const T* kb = kv + (long long)b * n_kv * ldkv + (long long)h * hd;  // K head slice of row 0; V is C columns further
  const T* qb = q + (long long)b * q_batch_stride + (long long)h * hd;
  const T* gb = dout + (long long)b * n_q * lddo + (long long)h * hd;
  const long long cta = (long long)b * heads + h;
  float* stats = ws + cta * n_q * 3;                                            // (m, l, D) per query
  float* dqw = ws + (long long)batches * heads * n_q * 3 + cta * n_q * hd;     // fp32 dQ over the key chunks done so far

  // ---- sweep 1: softmax statistics and D ----
  for (int q0 = 0; q0 < n_q; q0 += QBLK) {
    __syncthreads();
    att_bwd_stage<T>(Qs, hd, qb, ldq, q0, n_q, hd);
    att_bwd_stage<T>(Gs, hd, gb, lddo, q0, n_q, hd);
    float m[QB], l[QB], dd[QB];
#pragma unroll
    for (int j = 0; j < QB; ++j) {
      m[j] = -INFINITY;
      l[j] = dd[j] = 0.f;
    }
    for (int c0 = 0; c0 < n_kv; c0 += KC) {
      __syncthreads();
      att_bwd_stage<T>(Ks, kp, kb, ldkv, c0, n_kv, hd);
      att_bwd_stage<T>(Vs, kp, kb + C, ldkv, c0, n_kv, hd);
      __syncthreads();
      u64 s2[QB][2], p2[QB][2];
      att_bwd_dots(Qs + warp * QB * hd, Ks, hd, kp, lane, s2);
      att_bwd_dots(Gs + warp * QB * hd, Vs, hd, kp, lane, p2);
#pragma unroll
      for (int j = 0; j < QB; ++j) {
        float sv[2], mx = -INFINITY;
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          sv[t] = c0 + t * 32 + lane < n_kv ? att_bwd_sum2(s2[j][t]) * scale : -INFINITY;
          mx = fmaxf(mx, sv[t]);
        }
        mx = warp_max(mx);
        const float m_new = fmaxf(m[j], mx);  // finite: every chunk holds at least one key
        const float alpha = expf(m[j] - m_new);
        float rs = 0.f, rd = 0.f;
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          const float p = expf(sv[t] - m_new);
          rs += p;
          rd = fmaf(p, att_bwd_sum2(p2[j][t]), rd);
        }
        rs = warp_sum(rs);
        rd = warp_sum(rd);
        l[j] = l[j] * alpha + rs;
        dd[j] = dd[j] * alpha + rd;
        m[j] = m_new;
      }
    }
    if (lane == 0) {
#pragma unroll
      for (int j = 0; j < QB; ++j) {
        const int i = q0 + warp * QB + j;
        if (i < n_q) {
          stats[3 * i] = m[j];
          stats[3 * i + 1] = l[j];
          stats[3 * i + 2] = dd[j] / l[j];
        }
      }
    }
  }

  // ---- sweep 2: keys outer ----
  for (int c0 = 0; c0 < n_kv; c0 += KC) {
    const bool last_chunk = c0 + KC >= n_kv;
    __syncthreads();
    att_bwd_stage<T>(Ks, kp, kb, ldkv, c0, n_kv, hd);
    att_bwd_stage<T>(Vs, kp, kb + C, ldkv, c0, n_kv, hd);
    u64 dk2[QB / 2][DPL], dv2[QB / 2][DPL];  // keys c0 + warp * 8 + (2 kk, 2 kk + 1) x head dim i * 32 + lane
#pragma unroll
    for (int kk = 0; kk < QB / 2; ++kk)
#pragma unroll
      for (int i = 0; i < DPL; ++i) dk2[kk][i] = dv2[kk][i] = f32x2_pack(0.f, 0.f);
    for (int q0 = 0; q0 < n_q; q0 += QBLK) {
      __syncthreads();  // the chunk is staged / the previous block's tiles are consumed
      att_bwd_stage<T>(Qs, hd, qb, ldq, q0, n_q, hd);
      att_bwd_stage<T>(Gs, hd, gb, lddo, q0, n_q, hd);
      __syncthreads();
      const int qw = q0 + warp * QB;
      {
        u64 s2[QB][2], p2[QB][2];
        att_bwd_dots(Qs + warp * QB * hd, Ks, hd, kp, lane, s2);
        att_bwd_dots(Gs + warp * QB * hd, Vs, hd, kp, lane, p2);
#pragma unroll
        for (int j = 0; j < QB; ++j) {
          const bool qok = qw + j < n_q;
          const float mj = qok ? stats[3 * (qw + j)] : 0.f, lj = qok ? stats[3 * (qw + j) + 1] : 1.f, dj = qok ? stats[3 * (qw + j) + 2] : 0.f;
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            const int k = t * 32 + lane;
            float p = 0.f, ds = 0.f;
            if (qok && c0 + k < n_kv) {
              p = expf(att_bwd_sum2(s2[j][t]) * scale - mj) / lj;
              ds = scale * p * (att_bwd_sum2(p2[j][t]) - dj);
            }
            Ps[(warp * QB + j) * KC + k] = p;
            Ss[(warp * QB + j) * KC + k] = ds;
          }
        }
      }
      __syncthreads();
      // dQ of this warp's queries: lane owns head dims lane, lane + 32, ...
      {
        float acc[QB][DPL];
#pragma unroll
        for (int j = 0; j < QB; ++j)
#pragma unroll
          for (int i = 0; i < DPL; ++i) acc[j][i] = 0.f;
        const int kn = min(KC, n_kv - c0);
        for (int k = 0; k < kn; k += 4) {  // rows past n_kv are zeros in Ks and Ss
          float4 s4[QB];
#pragma unroll
          for (int j = 0; j < QB; ++j) s4[j] = *reinterpret_cast<const float4*>(Ss + (warp * QB + j) * KC + k);  // broadcast
#pragma unroll
          for (int i = 0; i < DPL; ++i) {
            const int d = i * 32 + lane;
            float kx[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) kx[u] = d < hd ? Ks[(k + u) * kp + d] : 0.f;
#pragma unroll
            for (int j = 0; j < QB; ++j) {
              acc[j][i] = fmaf(s4[j].x, kx[0], acc[j][i]);
              acc[j][i] = fmaf(s4[j].y, kx[1], acc[j][i]);
              acc[j][i] = fmaf(s4[j].z, kx[2], acc[j][i]);
              acc[j][i] = fmaf(s4[j].w, kx[3], acc[j][i]);
            }
          }
        }
#pragma unroll
        for (int j = 0; j < QB; ++j) {
          if (qw + j >= n_q) continue;
#pragma unroll
          for (int i = 0; i < DPL; ++i) {
            const int d = i * 32 + lane;
            if (d >= hd) continue;
            float* w = dqw + (long long)(qw + j) * hd + d;
            const float tot = c0 == 0 ? acc[j][i] : *w + acc[j][i];
            if (last_chunk) att_bwd_store(dq + ((long long)b * n_q + qw + j) * lddq + (long long)h * hd + d, tot);
            else *w = tot;
          }
        }
      }
      // dV += P^T dO and dK += dS^T Q for this warp's 8 keys: pairs of keys, lane owns head dims
      const int qn = min(QBLK, n_q - q0);
      for (int r = 0; r < qn; ++r) {
        const ulonglong2 pa = *reinterpret_cast<const ulonglong2*>(Ps + r * KC + warp * QB);  // broadcast: keys 0..3
        const ulonglong2 pb = *reinterpret_cast<const ulonglong2*>(Ps + r * KC + warp * QB + 4);
        const ulonglong2 sa = *reinterpret_cast<const ulonglong2*>(Ss + r * KC + warp * QB);
        const ulonglong2 sb = *reinterpret_cast<const ulonglong2*>(Ss + r * KC + warp * QB + 4);
#pragma unroll
        for (int i = 0; i < DPL; ++i) {
          const int d = i * 32 + lane;
          const float gv = d < hd ? Gs[r * hd + d] : 0.f, qv = d < hd ? Qs[r * hd + d] : 0.f;
          const u64 g2 = f32x2_pack(gv, gv), q2 = f32x2_pack(qv, qv);
          dv2[0][i] = f32x2_fma(pa.x, g2, dv2[0][i]);
          dv2[1][i] = f32x2_fma(pa.y, g2, dv2[1][i]);
          dv2[2][i] = f32x2_fma(pb.x, g2, dv2[2][i]);
          dv2[3][i] = f32x2_fma(pb.y, g2, dv2[3][i]);
          dk2[0][i] = f32x2_fma(sa.x, q2, dk2[0][i]);
          dk2[1][i] = f32x2_fma(sa.y, q2, dk2[1][i]);
          dk2[2][i] = f32x2_fma(sb.x, q2, dk2[2][i]);
          dk2[3][i] = f32x2_fma(sb.y, q2, dk2[3][i]);
        }
      }
    }
    // [dK | dV] of the chunk's keys, in the layout of kv
#pragma unroll
    for (int kk = 0; kk < QB / 2; ++kk) {
#pragma unroll
      for (int i = 0; i < DPL; ++i) {
        const int d = i * 32 + lane;
        float k0, k1, v0, v1;
        f32x2_unpack(dk2[kk][i], k0, k1);
        f32x2_unpack(dv2[kk][i], v0, v1);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int key = c0 + warp * QB + 2 * kk + half;
          if (key < n_kv && d < hd) {
            T* row = dkv + ((long long)b * n_kv + key) * lddkv + (long long)h * hd + d;
            att_bwd_store(row, half ? k1 : k0);
            att_bwd_store(row + C, half ? v1 : v0);
          }
        }
      }
    }
  }
}

// out[m, :] = a[m, :] + b[m % period, :]   (the two residual adds of CrossAttentionBlock.forward, nn_utils.py:449-450; period = number
// of query tokens when b holds the learned queries that every frame starts from, period = M for a plain tensor sum)
template <typename T>
__global__ void __launch_bounds__(256) add_rows_kernel(const T* __restrict__ a, long long lda, const T* __restrict__ b, long long ldb, T* __restrict__ out,
                                                       long long ldo, long long M, int cv, int period) {
  constexpr int VEC = Vec16<T>::kN;
  const long long total = M * cv;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const long long m = i / cv;
    const int c = int(i - m * cv) * VEC;
    float x[VEC], y[VEC];
    Vec16<T>::unpack(ldg_nc_v4(a + m * lda + c), x);
    Vec16<T>::unpack(ldg_v4(b + (m % period) * ldb + c), y);
#pragma unroll
    for (int k = 0; k < VEC; ++k) x[k] += y[k];
    stg_na_v4(out + m * ldo + c, Vec16<T>::pack(x));
  }
}

template <typename T>
static int launch_attention(const void* q, long long ldq, long long q_batch_stride, const void* kv, long long ldkv, void* out, long long ldo,
                            int batches, int n_q, int n_kv, int heads, int hd, float scale, cudaStream_t s) {
  const int C = heads * hd;
  const size_t smem = att_smem_bytes<T>(hd);
  MERV_REQUIRE(smem <= 160 * 1024, MERV_E_SHAPE, "merv_cross_attention: head_dim %d needs %zu bytes of shared memory", hd, smem);
  const int dpl = (hd + 31) / 32;
  dim3 grid(heads, batches);
#define MERV_ATT_CASE(n)                                                                                                              \
  case n: {                                                                                                                           \
    static bool opted[64] = {};                                                                                                       \
    int dev = 0;                                                                                                                      \
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;                                                          \
    if (!opted[dev]) {                                                                                                                \
      cudaFuncSetAttribute(cross_attention_kernel<T, n>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);                    \
      opted[dev] = true;                                                                                                              \
    }                                                                                                                                 \
    cross_attention_kernel<T, n><<<grid, kAttWarps * 32, smem, s>>>((const T*)q, ldq, q_batch_stride, (const T*)kv, ldkv, (T*)out, ldo, n_q, n_kv, \
                                                                   hd, C, scale);                                                     \
  } break;
  switch (dpl) {
    MERV_ATT_CASE(1) MERV_ATT_CASE(2) MERV_ATT_CASE(3) MERV_ATT_CASE(4)
    default: return fail(MERV_E_SHAPE, "merv_cross_attention: head_dim %d > 128", hd);
  }
#undef MERV_ATT_CASE
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

static size_t attention_bwd_simt_workspace(int batches, int n_q, int heads, int hd) {
  return (size_t)batches * heads * n_q * (hd + 3);  // (m, l, D) and the fp32 dQ of every (frame, head, query)
}

template <typename T>
static int launch_attention_bwd(const void* q, long long ldq, long long q_batch_stride, const void* kv, long long ldkv, const void* dout,
                                long long lddo, void* dq, long long lddq, void* dkv, long long lddkv, float* ws, int batches, int n_q, int n_kv,
                                int heads, int hd, float scale, cudaStream_t s) {
  const int C = heads * hd;
  const size_t smem = att_bwd_smem_bytes(hd);
  dim3 grid(heads, batches);
#define MERV_ATT_BWD_CASE(n)                                                                                                          \
  case n: {                                                                                                                           \
    static bool opted[64] = {};                                                                                                       \
    int dev = 0;                                                                                                                      \
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;                                                          \
    if (!opted[dev]) {                                                                                                                \
      MERV_CUDA_OK(cudaFuncSetAttribute(cross_attention_bwd_kernel<T, n>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kAbSmemMax)); \
      opted[dev] = true;                                                                                                              \
    }                                                                                                                                 \
    cross_attention_bwd_kernel<T, n><<<grid, kAttWarps * 32, smem, s>>>((const T*)q, ldq, q_batch_stride, (const T*)kv, ldkv, (const T*)dout, \
                                                                       lddo, (T*)dq, lddq, (T*)dkv, lddkv, ws, n_q, n_kv, hd, C, scale); \
  } break;
  switch ((hd + 31) / 32) {
    MERV_ATT_BWD_CASE(1) MERV_ATT_BWD_CASE(2) MERV_ATT_BWD_CASE(3) MERV_ATT_BWD_CASE(4)
    default: return fail(MERV_E_SHAPE, "merv_cross_attention_backward_ex: head_dim %d > 128", hd);
  }
#undef MERV_ATT_BWD_CASE
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

}  // namespace merv

using namespace merv;

extern "C" int merv_cross_attention(const void* q, int64_t ldq, int64_t q_batch_stride, const void* kv, int64_t ldkv, void* out, int64_t ldo,
                                    int batches, int n_q, int n_kv, int heads, int head_dim, float scale, int dtype, void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_cross_attention: unknown dtype %d", dtype);
  MERV_REQUIRE(q && kv && out, MERV_E_ARG, "merv_cross_attention: NULL pointer");
  const int vec = dtype == MERV_BF16 ? 8 : 4;
  const long long C = (long long)heads * head_dim;
  MERV_REQUIRE(batches >= 0 && n_q > 0 && n_kv > 0 && heads > 0 && heads <= 65535 && head_dim > 0 && head_dim % vec == 0, MERV_E_SHAPE,
               "merv_cross_attention: batches=%d n_q=%d n_kv=%d heads=%d head_dim=%d (head_dim must be a multiple of %d)", batches, n_q, n_kv, heads,
               head_dim, vec);
  MERV_REQUIRE(batches <= 65535, MERV_E_SHAPE, "merv_cross_attention: %d batch entries exceed the grid limit; split the call", batches);
  MERV_REQUIRE(ldq >= C && ldkv >= 2 * C && ldo >= C && ldq % vec == 0 && ldkv % vec == 0 && q_batch_stride % vec == 0 && aligned16(q) && aligned16(kv),
               MERV_E_ALIGN, "merv_cross_attention: rows must be 16-byte aligned with ldq >= C, ldkv >= 2C, ldo >= C");
  if (int rc = require_sm100()) return rc;
  if (batches == 0) return MERV_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // bf16: both contractions on the tensor cores whenever the frame fits the tcgen05 kernel's tile (MERV_ATTN_IMPL=simt forces this
  // file's CUDA-core kernel, which stays the fp32 parity path and the fallback for other shapes)
  if (dtype == MERV_BF16 && attention_tcgen05_supported(n_q, n_kv, heads, head_dim, ldq, q_batch_stride, ldkv, ldo))
    return launch_attention_tcgen05(q, ldq, q_batch_stride, kv, ldkv, out, ldo, batches, n_q, n_kv, heads, head_dim, scale, s);
  if (dtype == MERV_BF16)
    return launch_attention<__nv_bfloat16>(q, ldq, q_batch_stride, kv, ldkv, out, ldo, batches, n_q, n_kv, heads, head_dim, scale, s);
  return launch_attention<float>(q, ldq, q_batch_stride, kv, ldkv, out, ldo, batches, n_q, n_kv, heads, head_dim, scale, s);
}

extern "C" size_t merv_cross_attention_backward_ex_workspace(int batches, int n_q, int n_kv, int heads, int head_dim, int dtype) {
  if (batches <= 0 || n_q <= 0 || n_kv <= 0 || heads <= 0 || head_dim <= 0) return 0;
  if (dtype == MERV_BF16 && attention_bwd_tcgen05_supported(n_q, n_kv, head_dim)) return 0;
  return attention_bwd_simt_workspace(batches, n_q, heads, head_dim);
}

extern "C" int merv_cross_attention_backward_ex(const void* q, int64_t ldq, int64_t q_batch_stride, const void* kv, int64_t ldkv, const void* dout,
                                                int64_t lddo, void* dq, int64_t lddq, void* dkv, int64_t lddkv, int batches, int n_q, int n_kv,
                                                int heads, int head_dim, float scale, int dtype, float* workspace, size_t workspace_floats,
                                                void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_cross_attention_backward_ex: unknown dtype %d", dtype);
  MERV_REQUIRE(q && kv && dout && dq && dkv, MERV_E_ARG, "merv_cross_attention_backward: NULL pointer");
  MERV_REQUIRE(batches >= 0 && n_q > 0 && n_kv > 0 && heads > 0 && head_dim > 0, MERV_E_SHAPE,
               "merv_cross_attention_backward: batches=%d n_q=%d n_kv=%d heads=%d head_dim=%d", batches, n_q, n_kv, heads, head_dim);
  const long long C = (long long)heads * head_dim;
  MERV_REQUIRE(ldq >= C && ldkv >= 2 * C && lddo >= C && lddq >= C && lddkv >= 2 * C, MERV_E_SHAPE, "merv_cross_attention_backward: leading dimensions too small");
  // bf16 inside the tcgen05 tile runs the tensor-core kernel; without a workspace only that kernel can run, so other shapes are rejected
  // by its own checks (merv_cross_attention_backward's domain)
  const bool tc = dtype == MERV_BF16 && (workspace == nullptr || attention_bwd_tcgen05_supported(n_q, n_kv, head_dim));
  if (!tc) {
    const int vec = dtype == MERV_BF16 ? 8 : 4;
    MERV_REQUIRE(head_dim <= 128 && head_dim % vec == 0 && heads <= 65535 && batches <= 65535, MERV_E_SHAPE,
                 "merv_cross_attention_backward_ex: head_dim=%d (at most 128, a multiple of %d), heads=%d, batches=%d (at most 65535 each)", head_dim,
                 vec, heads, batches);
    MERV_REQUIRE(ldq % vec == 0 && ldkv % vec == 0 && lddo % vec == 0 && lddq % vec == 0 && lddkv % vec == 0 && q_batch_stride % vec == 0 &&
                     aligned16(q) && aligned16(kv) && aligned16(dout) && aligned16(dq) && aligned16(dkv),
                 MERV_E_ALIGN, "merv_cross_attention_backward_ex: rows must be 16-byte aligned");
    const size_t need = attention_bwd_simt_workspace(batches, n_q, heads, head_dim);
    MERV_REQUIRE(workspace_floats >= need && (need == 0 || workspace != nullptr), MERV_E_ARG,
                 "merv_cross_attention_backward_ex: workspace of %zu floats given, %zu needed", workspace_floats, need);
  }
  if (int rc = require_sm100()) return rc;
  if (batches == 0) return MERV_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (tc)
    return launch_attention_bwd_tcgen05(q, ldq, q_batch_stride, kv, ldkv, dout, lddo, dq, lddq, dkv, lddkv, batches, n_q, n_kv, heads, head_dim, scale, s);
  if (dtype == MERV_BF16)
    return launch_attention_bwd<__nv_bfloat16>(q, ldq, q_batch_stride, kv, ldkv, dout, lddo, dq, lddq, dkv, lddkv, workspace, batches, n_q, n_kv, heads,
                                               head_dim, scale, s);
  return launch_attention_bwd<float>(q, ldq, q_batch_stride, kv, ldkv, dout, lddo, dq, lddq, dkv, lddkv, workspace, batches, n_q, n_kv, heads,
                                     head_dim, scale, s);
}

extern "C" int merv_cross_attention_backward(const void* q, int64_t ldq, int64_t q_batch_stride, const void* kv, int64_t ldkv, const void* dout,
                                             int64_t lddo, void* dq, int64_t lddq, void* dkv, int64_t lddkv, int batches, int n_q, int n_kv, int heads,
                                             int head_dim, float scale, void* stream) {
  return merv_cross_attention_backward_ex(q, ldq, q_batch_stride, kv, ldkv, dout, lddo, dq, lddq, dkv, lddkv, batches, n_q, n_kv, heads, head_dim,
                                          scale, MERV_BF16, nullptr, 0, stream);
}

extern "C" int merv_add_rows(const void* a, int64_t lda, const void* b, int64_t ldb, void* out, int64_t ldo, int64_t M, int C, int period, int dtype,
                             void* stream) {
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_add_rows: unknown dtype %d", dtype);
  MERV_REQUIRE(a && b && out, MERV_E_ARG, "merv_add_rows: NULL pointer");
  const int vec = dtype == MERV_BF16 ? 8 : 4;
  MERV_REQUIRE(M >= 0 && C > 0 && C % vec == 0 && period > 0 && lda >= C && ldb >= C && ldo >= C && lda % vec == 0 && ldb % vec == 0 && ldo % vec == 0,
               MERV_E_SHAPE, "merv_add_rows: M=%lld C=%d period=%d lda=%lld ldb=%lld ldo=%lld", (long long)M, C, period, (long long)lda, (long long)ldb,
               (long long)ldo);
  MERV_REQUIRE(aligned16(a) && aligned16(b) && aligned16(out), MERV_E_ALIGN, "merv_add_rows: operands must be 16-byte aligned");
  if (int rc = require_sm100()) return rc;
  if (M == 0) return MERV_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int cv = C / vec;
  long long blocks = (M * cv + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  if (dtype == MERV_BF16)
    add_rows_kernel<__nv_bfloat16><<<(unsigned)blocks, 256, 0, s>>>((const __nv_bfloat16*)a, lda, (const __nv_bfloat16*)b, ldb, (__nv_bfloat16*)out, ldo, M, cv,
                                                                   period);
  else
    add_rows_kernel<float><<<(unsigned)blocks, 256, 0, s>>>((const float*)a, lda, (const float*)b, ldb, (float*)out, ldo, M, cv, period);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}
