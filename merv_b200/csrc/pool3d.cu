// Adaptive spatio-temporal average pooling, channel-last in -> channel-last out, all encoders in one launch.
//
// Replaces the rearrange -> AdaptiveAvgPool3d -> rearrange of AveragePooling3DProjector.forward
// (reference merv/util/nn_utils.py:320-329).  The reference permutes to channel-major, pools with ATen's
// generic kernel and permutes back through a transposed view; here the channel dimension stays the
// contiguous one end to end and the [B, T*S*S, C] result is directly the K-major A operand of the projector
// GEMM.  HBM-bound: compulsory traffic = input + pooled output (33.75 MB/video at merv-full).
//
// Main kernel (pool3d_tma_kernel): persistent, one CTA per SM, warp-specialised.
//   warp 12 (producer): one lane streams slabs [frames of the temporal window x H x W x 128-byte channel chunk]
//                      into a 6-stage shared-memory ring with 5-D TMA (cp.async.bulk.tensor): up to ~190 KB in
//                      flight per SM, independent of register pressure, which is what saturates HBM3e;
//   warps 0-11 (consumers): 3 groups of 4 warps; group g owns every 3rd slab (and ring stages g, g+3), so three
//                      slabs are reduced concurrently and no warp ever waits on another group.  A thread owns (output token,
//                      16-byte channel vector) units: up to 9 window taps are fetched with back-to-back 128-bit
//                      shared loads (conflict-free: 8 lanes cover one 128-byte row), accumulated in fp32,
//                      scaled and written with one 128-bit store.
// Window overlap (14 -> 8 uses 2/3-wide overlapping windows) costs shared-memory reads only: every input byte
// is fetched from HBM exactly once and every output byte written exactly once.
//
// Optional side output: deterministic partial dot products sum_{tokens, channels} score_vec[c] * P[token, c]
// per work item, from which the affine fast path derives the encoder scores without re-reading anything.
//
// Fallback kernel (pool3d_direct_kernel): plain vectorised loads, for shapes the TMA path does not cover
// (slab of more than 2048 patch tokens, more than 256 output tokens per frame).
#include <cuda.h>

#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "tcgen05_util.cuh"
#include "tmap.cuh"

namespace merv {

// L2 prefetch of the producer's next batch of slabs: measured SLOWER on B200 (3.9 vs 4.4 TB/s on 16 videos), kept as a
// compile-time experiment only.
#ifndef MERV_POOL_L2_PREFETCH
#define MERV_POOL_L2_PREFETCH 0
#endif
// build-time switch for A/B measurements: 1 = always the general consumer loop
#ifndef MERV_POOL_GENERIC_ONLY
#define MERV_POOL_GENERIC_ONLY 0
#endif

__device__ __forceinline__ void window(int k, int n_in, int n_out, int& lo, int& hi) {
  lo = (k * n_in) / n_out;                    // floor(k * n_in / n_out)
  hi = ((k + 1) * n_in + n_out - 1) / n_out;  // ceil((k+1) * n_in / n_out)
}

// fixed-tree block reduction over `nwarps` warps (deterministic); result valid in thread 0 of the group
__device__ __forceinline__ float group_sum(float v, float* red, int warp, int lane, int nwarps, int bar_id, int bar_threads) {
  v = warp_sum(v);
  if (lane == 0) red[warp] = v;
  asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(bar_threads) : "memory");
  float r = 0.f;
  if (warp == 0) {
    r = lane < nwarps ? red[lane] : 0.f;
    r = warp_sum(r);
  }
  asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(bar_threads) : "memory");
  return r;
}

// ============================================================================================================
// TMA-staged persistent kernel
// ============================================================================================================
constexpr int PT_STAGES = 6;
constexpr int PT_STAGE_BYTES = 32768;
constexpr int PT_CONSUMERS = 384;      // 12 consumer warps
constexpr int PT_CWARPS = PT_CONSUMERS / 32;
constexpr int PT_BATCH = 16;           // items whose coordinates the producer warp computes (and L2-prefetches) at once
constexpr int PT_GROUPS = 3;           // consumer groups working on different slabs concurrently
// Each stage must belong to exactly ONE group (slab n -> group n % PT_GROUPS, stage n % PT_STAGES): a group then visits
// its stages in order, one mbarrier phase at a time.  If a group skipped phases of a stage, a parity wait could be
// satisfied by a stale phase (mbarrier waits only distinguish the current phase from the previous one).
static_assert(PT_STAGES % PT_GROUPS == 0, "every ring stage must be owned by one consumer group");
constexpr int PT_GROUP_THREADS = PT_CONSUMERS / PT_GROUPS;
constexpr int PT_GROUP_WARPS = PT_GROUP_THREADS / 32;
constexpr int PT_THREADS = PT_CONSUMERS + 32;
constexpr int PT_MAX_TOKENS = 256;     // S * S output tokens per frame covered by the shared window table
constexpr int PT_TABLE_BYTES = MERV_MAX_ENCODERS * PT_MAX_TOKENS * 12;
constexpr int PT_SMEM = 1024 + PT_STAGES * PT_STAGE_BYTES + 256 + PT_TABLE_BYTES;

struct PoolTmaEnc {
  void* y;
  const float* score_vec;
  float* score_partial;
  const int* batch_index;
  int F, H, W, C, T, S;
  int cb;        // channels per slab (elements); cb * sizeof(T) <= 128 bytes
  int vpr;       // 16-byte vectors per slab row (1, 2, 4 or 8)
  int vshift;    // log2(vpr)
  int nchunks;   // ceil(C / cb)
  int units;     // S * S * vpr
  int nf_max;    // frames per slab (longest temporal window)
  int item_begin, items;  // range in the global item list; items = B * T * nchunks
  int slab_bytes;
  int sf, sh, sw;         // displacement of the windows (a convolution tap); out-of-grid positions are zero-filled by the TMA unit
  long long ybs, yrs;
};
struct PoolTmaParams {
  PoolTmaEnc enc[MERV_MAX_ENCODERS];
  int n_enc;
  int total_items;
};
struct PoolTmaMaps {
  CUtensorMap m[MERV_MAX_ENCODERS];
};

__device__ __forceinline__ uint32_t pt_smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void pt_mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void pt_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void pt_mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool pt_mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void pt_mbar_wait(uint32_t bar, uint32_t parity) {
  if (pt_mbar_try_wait(bar, parity)) return;
  unsigned long long t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  while (!mbar_try_wait_parked(bar, parity, MERV_WAIT_HINT_NS)) {  // parked in hardware until the phase completes (tcgen05_util.cuh)
    unsigned long long t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (t1 - t0 > 4000000000ull) {  // a protocol bug must trap, never hang the GPU
      printf("merv pool3d: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_5d(const CUtensorMap* map, uint32_t bar, uint32_t dst, int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}
// L2 prefetch of a future slab (experiment, see MERV_POOL_L2_PREFETCH).
__device__ __forceinline__ void tma_prefetch_5d(const CUtensorMap* map, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.async.bulk.prefetch.tensor.5d.L2.global [%0, {%1, %2, %3, %4, %5}];"
               ::"l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}
__device__ __forceinline__ int pt_find_encoder(const PoolTmaParams& p, int item) {
  int e = 0;
#pragma unroll 1
  while (e + 1 < p.n_enc && item >= p.enc[e + 1].item_begin) ++e;
  return e;
}

template <int N_IN, int N_OUT>
struct PoolWin {  // adaptive pooling window k of an axis N_IN -> N_OUT: [floor(k N_IN / N_OUT), ceil((k + 1) N_IN / N_OUT))
  __host__ __device__ static constexpr int lo(int i) { return (i * N_IN) / N_OUT; }
  __host__ __device__ static constexpr int hi(int i) { return ((i + 1) * N_IN + N_OUT - 1) / N_OUT; }
};

__device__ __forceinline__ uint4 lds_v4(uint32_t addr) {
  uint4 r;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
  return r;
}
// predicated 128-bit shared load: zeros when !ok, no branch
__device__ __forceinline__ uint4 lds_v4_if(uint32_t addr, bool ok) {
  uint4 r;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.u32 p, %5, 0;\n\t"
      "mov.u32 %0, 0;\n\tmov.u32 %1, 0;\n\tmov.u32 %2, 0;\n\tmov.u32 %3, 0;\n\t"
      "@p ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];\n\t}"
      : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr), "r"(uint32_t(ok)));
  return r;
}

// ---- specialised consumer for the square grids of the shipped encoders (16 x 16 and 14 x 14 patches -> 8 x 8), 128-byte rows ----
// The general loop below issues a predicated 3 x 3 tap block per output vector and spends ~185 instructions on it whatever
// the window; with 12 consumer warps that made the kernel instruction-ISSUE bound (both encoder shapes ran at the same
// ~3.9 G warp-instructions/s per SM: 6.2 TB/s for 16 x 16, 4.9 TB/s for 14 x 14).  Here the pooling is done separably
// with compile-time row windows: a thread owns one (output column, 16-byte channel vector) and half of the output rows; for
// every input row of its half it sums the 2-3 taps of its column window ONCE (packed fp32 adds) and adds that row sum to
// the 1-2 output rows whose window holds the row.  ~2x fewer instructions per output, same shared-memory traffic pattern
// (8 lanes cover one 128-byte row: conflict-free).
template <typename T, int H, int S, int HF>
__device__ __forceinline__ void pool_square_half(uint32_t slab, int nf, int v, int wo, T* __restrict__ yb, long long yrs, bool c_ok,
                                                 const float* sv, float inv_nf, float& dot) {
  constexpr int P = Pairs<T>::kP;
  constexpr int HALF = S / 2;
  constexpr int O0 = HF * HALF;
  constexpr int R_LO = PoolWin<H, S>::lo(O0), R_HI = PoolWin<H, S>::hi(O0 + HALF - 1);
  constexpr bool kThird = (H % S) != 0;  // windows are H / S wide when S divides H, else up to H / S + 2 (= 3 taps for 14 -> 8)
  static_assert(H / S + (kThird ? 2 : 0) <= 3 && H / S >= 1, "column windows of up to three taps");
  typedef unsigned long long u64;
  const int w0 = (wo * H) / S;
  const int wn = ((wo + 1) * H + S - 1) / S - w0;
  const u64 one2 = f32x2_pack(1.0f, 1.0f);
  u64 sv2[P], dot2 = f32x2_pack(0.f, 0.f);
#pragma unroll
  for (int q = 0; q < P; ++q) sv2[q] = f32x2_pack(sv[2 * q], sv[2 * q + 1]);
  u64 acc[HALF][P];
#pragma unroll
  for (int o = 0; o < HALF; ++o)
#pragma unroll
    for (int q = 0; q < P; ++q) acc[o][q] = f32x2_pack(0.f, 0.f);
  const uint32_t col = slab + uint32_t(w0) * 128u + uint32_t(v) * 16u;
  for (int f = 0; f < nf; ++f) {
    const uint32_t fb = col + uint32_t(f) * uint32_t(H * H * 128);
#pragma unroll
    for (int r = R_LO; r < R_HI; ++r) {
      const uint32_t a = fb + uint32_t(r * H * 128);
      u64 rs[P], t[P];
      Pairs<T>::unpack(lds_v4(a), rs);
      if constexpr (H / S >= 2 || kThird) {
        Pairs<T>::unpack(lds_v4_if(a + 128u, wn >= 2), t);
#pragma unroll
        for (int q = 0; q < P; ++q) rs[q] = f32x2_fma(t[q], one2, rs[q]);
      }
      if constexpr (H / S + (kThird ? 2 : 0) >= 3) {
        Pairs<T>::unpack(lds_v4_if(a + 256u, wn >= 3), t);
#pragma unroll
        for (int q = 0; q < P; ++q) rs[q] = f32x2_fma(t[q], one2, rs[q]);
      }
#pragma unroll
      for (int o = 0; o < HALF; ++o) {
        if (r >= PoolWin<H, S>::lo(O0 + o) && r < PoolWin<H, S>::hi(O0 + o)) {  // compile-time after unrolling
#pragma unroll
          for (int q = 0; q < P; ++q) acc[o][q] = f32x2_fma(rs[q], one2, acc[o][q]);
        }
      }
    }
  }
#pragma unroll
  for (int o = 0; o < HALF; ++o) {
    const int hn = PoolWin<H, S>::hi(O0 + o) - PoolWin<H, S>::lo(O0 + o);
    const float inv = (1.0f / float(hn * wn)) * inv_nf;
    const u64 inv2 = f32x2_pack(inv, inv);
    u64 out[P];
#pragma unroll
    for (int q = 0; q < P; ++q) out[q] = f32x2_mul(acc[o][q], inv2);
    const uint4 packed = Pairs<T>::pack(out);
    const int tok = (O0 + o) * S + wo;
    if (c_ok) *reinterpret_cast<uint4*>(yb + (long long)tok * yrs) = packed;
    u64 rr[P];
    Pairs<T>::unpack(packed, rr);  // dot with the values as stored (what the GEMM will consume)
#pragma unroll
    for (int q = 0; q < P; ++q) dot2 = f32x2_fma(sv2[q], rr[q], dot2);
  }
  float d0, d1;
  f32x2_unpack(dot2, d0, d1);
  dot += d0 + d1;
}

// one slab of a square H x H grid pooled to S x S by one consumer group of S * S * 2 = 128 threads (vpr == 8)
template <typename T, int H, int S>
__device__ __forceinline__ void pool_square(uint32_t slab, int nf, int gtid, T* __restrict__ yb, long long yrs, bool c_ok,
                                            const float* sv, float inv_nf, float& dot) {
  static_assert(S == 8 && PT_GROUP_THREADS == 2 * S * 8, "thread map: 8 vectors x 8 output columns x 2 row halves");
  const int v = gtid & 7, wo = (gtid >> 3) & 7;
  if ((gtid >> 6) == 0)  // warp-uniform: a half is two warps
    pool_square_half<T, H, S, 0>(slab, nf, v, wo, yb, yrs, c_ok, sv, inv_nf, dot);
  else
    pool_square_half<T, H, S, 1>(slab, nf, v, wo, yb, yrs, c_ok, sv, inv_nf, dot);
}

template <typename T>
__global__ void __launch_bounds__(PT_THREADS, 1)
pool3d_tma_kernel(const __grid_constant__ PoolTmaMaps maps, const __grid_constant__ PoolTmaParams p) {
  constexpr int VEC = Vec16<T>::kN;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = pt_smem_u32(smem_raw);
  const uint32_t slab_addr = (raw_addr + 1023u) & ~1023u;
  uint8_t* slabs = smem_raw + (slab_addr - raw_addr);
  uint64_t* bars = reinterpret_cast<uint64_t*>(slabs + PT_STAGES * PT_STAGE_BYTES);
  const uint32_t full_bar = pt_smem_u32(bars), empty_bar = full_bar + 8 * PT_STAGES;
  // per-stage item descriptor written by the producer: (encoder | frames-in-window << 8, channel chunk, b, t)
  int4* smeta = reinterpret_cast<int4*>(bars + 2 * PT_STAGES);  // PT_STAGES x 16 bytes (barriers use 96 of the 256 bytes)
  // per-encoder window tables: tok -> (h0 | w0 << 16, hn | wn << 16) and 1 / (hn * wn); hoist all integer division
  uint2* wtab = reinterpret_cast<uint2*>(slabs + PT_STAGES * PT_STAGE_BYTES + 256);
  float* itab = reinterpret_cast<float*>(wtab + MERV_MAX_ENCODERS * PT_MAX_TOKENS);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // PDL: a dependent kernel launched with programmatic stream serialization (the scores kernel of merv_fused_forward) may be
  // made resident already; it blocks in griddepcontrol.wait until this grid has completed.  No-op otherwise.
  pdl_launch_dependents();
  if (threadIdx.x == 0) {
    for (int i = 0; i < PT_STAGES; ++i) {
      pt_mbar_init(full_bar + 8 * i, 1);
      pt_mbar_init(empty_bar + 8 * i, PT_GROUP_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  for (int idx = threadIdx.x; idx < p.n_enc * PT_MAX_TOKENS; idx += PT_THREADS) {
    const PoolTmaEnc& e = p.enc[idx / PT_MAX_TOKENS];
    const int tok = idx % PT_MAX_TOKENS;
    uint2 w2 = make_uint2(0, 0);
    float inv = 0.f;
    if (tok < e.S * e.S) {
      int h0, h1, w0, w1;
      window(tok / e.S, e.H, e.S, h0, h1);
      window(tok % e.S, e.W, e.S, w0, w1);
      w2 = make_uint2(uint32_t(h0) | (uint32_t(w0) << 16), uint32_t(h1 - h0) | (uint32_t(w1 - w0) << 16));
      inv = 1.0f / float((h1 - h0) * (w1 - w0));
    }
    wtab[idx] = w2;
    itab[idx] = inv;
  }
  __syncthreads();

  if (warp == PT_CWARPS) {
    // ===== producer warp: all per-item index arithmetic lives here, consumers read it from smeta.  The integer
    //       divisions (~1.5k cycles per item when done serially) are computed for 32 items at once, one per lane;
    //       the lanes then take turns, in ring order, to wait for a free stage and issue their TMA. =====
    if (lane == 0)
      for (int e = 0; e < p.n_enc; ++e) asm volatile("prefetch.tensormap [%0];" ::"l"(&maps.m[e]) : "memory");
    uint32_t it = 0;
    const int stride = int(gridDim.x);
    for (int base_item = blockIdx.x; base_item < p.total_items; base_item += PT_BATCH * stride) {
      const int item = base_item + lane * stride;
      int ei = 0, chunk = 0, b = 0, t = 0, f0 = 0, f1 = 1;
      const bool mine = lane < PT_BATCH && item < p.total_items;
      if (mine) {
        ei = pt_find_encoder(p, item);
        const PoolTmaEnc& e = p.enc[ei];
        const int local = item - e.item_begin;
        chunk = local % e.nchunks;
        const int bt = local / e.nchunks;
        t = bt % e.T;
        b = bt / e.T;
        window(t, e.F, e.T, f0, f1);
        if (MERV_POOL_L2_PREFETCH) tma_prefetch_5d(&maps.m[ei], chunk * e.cb, e.sw, e.sh, f0 + e.sf, b);  // the whole batch, up front
      }
      __syncwarp();
      const int remaining = (p.total_items - base_item + stride - 1) / stride;
      const int count = remaining < PT_BATCH ? remaining : PT_BATCH;
      for (int j = 0; j < count; ++j) {
        if (lane == j) {
          const uint32_t n = it + uint32_t(j);
          const uint32_t stage = n % PT_STAGES, ph = (n / PT_STAGES) & 1u;
          const PoolTmaEnc& e = p.enc[ei];
          pt_mbar_wait(empty_bar + 8 * stage, ph ^ 1u);
          smeta[stage] = make_int4(ei | ((f1 - f0) << 8), chunk, b, t);  // ordered before the consumers' acquire by the arrive below
          pt_mbar_expect_tx(full_bar + 8 * stage, e.slab_bytes);
          // the box always spans nf_max frames starting at f0; frames past the window (or past F: zero-filled) are ignored
          tma_load_5d(&maps.m[ei], full_bar + 8 * stage, slab_addr + stage * PT_STAGE_BYTES, chunk * e.cb, e.sw, e.sh, f0 + e.sf,
                      e.batch_index ? __ldg(e.batch_index + b) : b);
        }
        __syncwarp();
      }
      it += uint32_t(count);
    }
  } else if (blockIdx.x < p.total_items) {
    // ===== consumers: group g reduces the CTA's slabs g, g + 3, g + 6, ... =====
    const int group = warp / PT_GROUP_WARPS;
    const int gtid = threadIdx.x - group * PT_GROUP_THREADS;
    const int gwarp = warp - group * PT_GROUP_WARPS;
    const int n_items = (p.total_items - int(blockIdx.x) + int(gridDim.x) - 1) / int(gridDim.x);
    for (int n = group; n < n_items; n += PT_GROUPS) {
      const uint32_t stage = uint32_t(n) % PT_STAGES, ph = (uint32_t(n) / PT_STAGES) & 1u;
      pt_mbar_wait(full_bar + 8 * stage, ph);
      const int4 m = smeta[stage];
      const int ei = m.x & 0xff, nf = m.x >> 8;
      const PoolTmaEnc& e = p.enc[ei];
      const int vshift = e.vshift;
      const int v = gtid & ((1 << vshift) - 1);  // PT_GROUP_THREADS % vpr == 0: one vector column per thread
      const int c_base = m.y * e.cb + v * VEC;
      const bool c_ok = c_base < e.C;  // the last chunk may hang over C (TMA zero-fills it)
      float sv[VEC];
#pragma unroll
      for (int c = 0; c < VEC; ++c) sv[c] = 0.f;
      if (e.score_vec != nullptr && c_ok) {  // issued before the slab is touched: off the critical path
#pragma unroll
        for (int c = 0; c < VEC; c += 4) {
          const float4 s4 = __ldg(reinterpret_cast<const float4*>(e.score_vec + c_base + c));
          sv[c] = s4.x; sv[c + 1] = s4.y; sv[c + 2] = s4.z; sv[c + 3] = s4.w;
        }
      }
      const uint32_t row_bytes = 16u << vshift;
      const uint32_t h_pitch = uint32_t(e.W) * row_bytes;
      const uint32_t f_pitch = uint32_t(e.H) * h_pitch;
      const uint2* tab = wtab + ei * PT_MAX_TOKENS;
      const float* inv_tab = itab + ei * PT_MAX_TOKENS;
      const float inv_nf = 1.0f / float(nf);
      const int units = e.units;
      const uint32_t base = slab_addr + stage * PT_STAGE_BYTES + uint32_t(v) * 16u;
      T* yb = static_cast<T*>(e.y) + (long long)m.z * e.ybs + (long long)m.w * e.S * e.S * e.yrs + c_base;
      const long long yrs = e.yrs;
      float dot = 0.f;

      const bool square8 = vshift == 3 && e.S == 8 && e.H == e.W && !MERV_POOL_GENERIC_ONLY;
      if (square8 && e.H == 16) {
        pool_square<T, 16, 8>(slab_addr + stage * PT_STAGE_BYTES, nf, gtid, yb, yrs, c_ok, sv, inv_nf, dot);
      } else if (square8 && e.H == 14) {
        pool_square<T, 14, 8>(slab_addr + stage * PT_STAGE_BYTES, nf, gtid, yb, yrs, c_ok, sv, inv_nf, dot);
      } else
      for (int u = gtid; u < units; u += PT_GROUP_THREADS) {
        const int tok = u >> vshift;
        const uint2 tw = tab[tok];
        const uint32_t hn = tw.y & 0xffffu, wn = tw.y >> 16;
        const uint32_t origin = base + (tw.x & 0xffffu) * h_pitch + (tw.x >> 16) * row_bytes;
        float acc[VEC];
#pragma unroll
        for (int c = 0; c < VEC; ++c) acc[c] = 0.f;
        for (int f = 0; f < nf; ++f) {
          for (uint32_t hb = 0; hb < hn; hb += 3) {
            for (uint32_t wb = 0; wb < wn; wb += 3) {
              // up to 3 x 3 taps in flight at once (predicated, branch-free): one shared-memory latency per block
              uint4 r[9];
#pragma unroll
              for (int dh = 0; dh < 3; ++dh)
#pragma unroll
                for (int dw = 0; dw < 3; ++dw)
                  r[dh * 3 + dw] = lds_v4_if(origin + uint32_t(f) * f_pitch + (hb + dh) * h_pitch + (wb + dw) * row_bytes,
                                             hb + dh < hn && wb + dw < wn);
#pragma unroll
              for (int i = 0; i < 9; ++i) {
                float val[VEC];
                Vec16<T>::unpack(r[i], val);
#pragma unroll
                for (int c = 0; c < VEC; ++c) acc[c] += val[c];
              }
            }
          }
        }
        const float inv = inv_tab[tok] * inv_nf;
#pragma unroll
        for (int c = 0; c < VEC; ++c) acc[c] *= inv;
        const uint4 packed = Vec16<T>::pack(acc);
        if (c_ok) *reinterpret_cast<uint4*>(yb + (long long)tok * yrs) = packed;
        float rr[VEC];
        Vec16<T>::unpack(packed, rr);  // dot with the values as stored (what the GEMM will consume)
#pragma unroll
        for (int c = 0; c < VEC; ++c) dot = fmaf(sv[c], rr[c], dot);
      }
      __syncwarp();
      if (lane == 0) pt_mbar_arrive(empty_bar + 8 * stage);  // this warp is done with the slab (and with smeta[stage])
      if (e.score_partial != nullptr) {  // one partial per (item, warp of the group): no CTA-wide barrier on the hot path
        dot = warp_sum(dot);
        if (lane == 0) e.score_partial[(((long long)m.z * e.T + m.w) * e.nchunks + m.y) * PT_GROUP_WARPS + gwarp] = dot;
      }
    }
  }
}

// ============================================================================================================
// direct (non-TMA) fallback kernel
// ============================================================================================================
struct PoolEnc {
  const void* x;
  void* y;
  const float* score_vec;
  float* score_partial;
  const int* batch_index;
  int F, H, W, C, T, S;
  int src_batch;              // videos in x (bound of the batch_index gather)
  int sf, sh, sw;             // displacement of the windows (a convolution tap); out-of-grid positions contribute zero
  int rows_per_item, groups;  // output rows handled by one CTA; groups = ceil(S / rows_per_item)
  int items;                  // B * T * groups
  long long xbs, xfs, xts, ybs, yrs;
};
struct PoolParams {
  PoolEnc enc[MERV_MAX_ENCODERS];
};

template <typename T>
__global__ void __launch_bounds__(256) pool3d_direct_kernel(const __grid_constant__ PoolParams p) {
  constexpr int VEC = Vec16<T>::kN;
  __shared__ float red[8];
  const PoolEnc& e = p.enc[blockIdx.y];
  const int item = blockIdx.x;
  if (item >= e.items) return;
  const int g = item % e.groups;
  const int t = (item / e.groups) % e.T;
  const int b = item / (e.groups * e.T);
  int f0, f1;
  window(t, e.F, e.T, f0, f1);
  const int i_begin = g * e.rows_per_item;
  const int i_end = min(e.S, i_begin + e.rows_per_item);
  const int nvec = e.C / VEC;
  // an out-of-range gather index must never read outside x: clamp it (the TMA kernel's loads are bounds-checked by the tensor map)
  int src = e.batch_index ? e.batch_index[b] : b;
  src = src < 0 ? 0 : (src >= e.src_batch ? e.src_batch - 1 : src);
  const T* __restrict__ xb = static_cast<const T*>(e.x) + (long long)src * e.xbs;
  T* __restrict__ yb = static_cast<T*>(e.y) + (long long)b * e.ybs;
  float dot = 0.f;

  for (int v = threadIdx.x; v < nvec; v += blockDim.x) {
    float sv[VEC];
#pragma unroll
    for (int c = 0; c < VEC; ++c) sv[c] = e.score_vec ? e.score_vec[v * VEC + c] : 0.f;
    for (int i = i_begin; i < i_end; ++i) {
      int h0, h1;
      window(i, e.H, e.S, h0, h1);
      for (int j = 0; j < e.S; ++j) {
        int w0, w1;
        window(j, e.W, e.S, w0, w1);
        float acc[VEC];
#pragma unroll
        for (int c = 0; c < VEC; ++c) acc[c] = 0.f;
        for (int f = f0; f < f1; ++f) {
          const int fs = f + e.sf;
          if (fs < 0 || fs >= e.F) continue;
          for (int h = h0; h < h1; ++h) {
            const int hs = h + e.sh;
            if (hs < 0 || hs >= e.H) continue;
            const T* row = xb + (long long)fs * e.xfs + (long long)(hs * e.W) * e.xts + (long long)v * VEC;
#pragma unroll 3
            for (int w = w0; w < w1; ++w) {
              const int ws = w + e.sw;
              if (ws < 0 || ws >= e.W) continue;
              float val[VEC];
              Vec16<T>::unpack(ldg_v4(row + (long long)ws * e.xts), val);
#pragma unroll
              for (int c = 0; c < VEC; ++c) acc[c] += val[c];
            }
          }
        }
        const float cnt = float((f1 - f0) * (h1 - h0) * (w1 - w0));
#pragma unroll
        for (int c = 0; c < VEC; ++c) acc[c] = acc[c] / cnt;
        const uint4 packed = Vec16<T>::pack(acc);
        const long long tok = (long long)(t * e.S + i) * e.S + j;
        *reinterpret_cast<uint4*>(yb + tok * e.yrs + (long long)v * VEC) = packed;
        float rounded[VEC];
        Vec16<T>::unpack(packed, rounded);
#pragma unroll
        for (int c = 0; c < VEC; ++c) dot = fmaf(sv[c], rounded[c], dot);
      }
    }
  }
  if (e.score_partial != nullptr) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float s = group_sum(dot, red, warp, lane, blockDim.x >> 5, 0, blockDim.x);
    if (threadIdx.x == 0) e.score_partial[(long long)b * (e.T * e.groups) + t * e.groups + g] = s;
  }
}

// ============================================================================================================
// host side
// ============================================================================================================
static int direct_rows_per_item(int S) {
  // Up to 4 row-groups per output frame.  Deliberately independent of the batch size so the fp32 summation
  // order of the score partials — hence every mixing weight — is bit-identical whether a video is processed
  // alone, in a batch of 64, or on another rank.
  const int groups = S < 4 ? S : 4;
  return (S + groups - 1) / groups;
}

struct TmaPlan {
  bool ok;
  int cb, vpr, nchunks, units, slab_bytes, nf_max;
};

// The plan depends only on the encoder's shape (never on B): see direct_rows_per_item.
static TmaPlan plan_tma(const merv_pool_desc& d, int dtype) {
  TmaPlan pl = {};
  const int es = dtype == MERV_BF16 ? 2 : 4;
  const int vec = 16 / es;
  if (d.H > 256 || d.W > 256 || d.S * d.S > PT_MAX_TOKENS || d.C % vec != 0) return pl;
  int nf_max = 1;
  for (int t = 0; t < d.T; ++t) {
    const int lo = (t * d.F) / d.T, hi = ((t + 1) * d.F + d.T - 1) / d.T;
    nf_max = hi - lo > nf_max ? hi - lo : nf_max;
  }
  if (nf_max > 255) return pl;
  for (int row_bytes = 128; row_bytes >= 16; row_bytes >>= 1) {
    const long long slab = (long long)nf_max * d.H * d.W * row_bytes;
    if (slab > PT_STAGE_BYTES) continue;
    pl.cb = row_bytes / es;
    pl.vpr = row_bytes / 16;
    pl.nchunks = (d.C + pl.cb - 1) / pl.cb;
    pl.units = d.S * d.S * pl.vpr;
    pl.slab_bytes = int(slab);
    pl.nf_max = nf_max;
    pl.ok = true;
    return pl;
  }
  return pl;
}

static bool use_tma(const merv_pool_desc* enc, int n, int dtype) {
  // MERV_POOL_IMPL=direct forces the plain-load kernel (read per call so the tests can exercise both kernels)
  const char* env = getenv("MERV_POOL_IMPL");
  const bool force_direct = env != nullptr && strcmp(env, "direct") == 0;
  if (force_direct) return false;
  for (int i = 0; i < n; ++i)
    if (!plan_tma(enc[i], dtype).ok) return false;
  return true;
}

static int validate(const merv_pool_desc* enc, int num_encoders, int B, int dtype) {
  MERV_REQUIRE(enc != nullptr, MERV_E_ARG, "merv_pool3d: enc is NULL");
  MERV_REQUIRE(num_encoders >= 1 && num_encoders <= MERV_MAX_ENCODERS, MERV_E_ARG,
               "merv_pool3d: num_encoders=%d not in [1,%d]", num_encoders, MERV_MAX_ENCODERS);
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_pool3d: unknown dtype %d", dtype);
  MERV_REQUIRE(B >= 0, MERV_E_SHAPE, "merv_pool3d: B=%d", B);
  const int vec = dtype == MERV_BF16 ? 8 : 4;
  for (int i = 0; i < num_encoders; ++i) {
    const merv_pool_desc& d = enc[i];
    MERV_REQUIRE(d.x && d.y, MERV_E_ARG, "merv_pool3d: encoder %d has a NULL tensor", i);
    MERV_REQUIRE(d.F > 0 && d.H > 0 && d.W > 0 && d.C > 0 && d.T > 0 && d.S > 0, MERV_E_SHAPE,
                 "merv_pool3d: encoder %d has a non-positive dimension (F=%d H=%d W=%d C=%d T=%d S=%d)", i, d.F,
                 d.H, d.W, d.C, d.T, d.S);
    MERV_REQUIRE(d.C % vec == 0, MERV_E_SHAPE, "merv_pool3d: encoder %d: C=%d must be a multiple of %d", i, d.C, vec);
    MERV_REQUIRE(aligned16(d.x) && aligned16(d.y) && (d.score_vec == nullptr || aligned16(d.score_vec)), MERV_E_ALIGN,
                 "merv_pool3d: encoder %d: base pointers must be 16-byte aligned", i);
    MERV_REQUIRE(d.x_batch_stride % vec == 0 && d.x_frame_stride % vec == 0 && d.x_token_stride % vec == 0 &&
                     d.y_batch_stride % vec == 0 && d.y_row_stride % vec == 0 && d.x_token_stride >= d.C &&
                     d.y_row_stride >= d.C,
                 MERV_E_ALIGN, "merv_pool3d: encoder %d: strides must be multiples of %d elements and >= C", i, vec);
    MERV_REQUIRE(d.batch_index == nullptr || d.src_batch > 0, MERV_E_ARG, "merv_pool3d: encoder %d: batch_index needs src_batch > 0", i);
    MERV_REQUIRE((d.score_vec == nullptr) == (d.score_partial == nullptr), MERV_E_ARG,
                 "merv_pool3d: encoder %d: score_vec and score_partial go together", i);
  }
  return MERV_OK;
}

template <typename T>
static int launch_tma(const merv_pool_desc* enc, int n, int B, int dtype, int max_ctas, cudaStream_t s) {
  const int es = sizeof(T);
  PoolTmaMaps maps;
  PoolTmaParams p = {};
  p.n_enc = n;
  int begin = 0;
  for (int i = 0; i < n; ++i) {
    const merv_pool_desc& d = enc[i];
    const TmaPlan pl = plan_tma(d, dtype);
    PoolTmaEnc& e = p.enc[i];
    e.y = d.y; e.score_vec = d.score_vec; e.score_partial = d.score_partial; e.batch_index = d.batch_index;
    e.F = d.F; e.H = d.H; e.W = d.W; e.C = d.C; e.T = d.T; e.S = d.S;
    e.nf_max = pl.nf_max; e.cb = pl.cb; e.vpr = pl.vpr; e.vshift = pl.vpr == 8 ? 3 : pl.vpr == 4 ? 2 : pl.vpr == 2 ? 1 : 0; e.nchunks = pl.nchunks; e.units = pl.units; e.slab_bytes = pl.slab_bytes;
    e.item_begin = begin; e.items = B * d.T * pl.nchunks;
    e.sf = d.shift_f; e.sh = d.shift_h; e.sw = d.shift_w;
    begin += e.items;
    e.ybs = d.y_batch_stride; e.yrs = d.y_row_stride;
    // x as a 5-D tensor (C, W, H, F, B), channel innermost; one box = the [nf_max, H, W, cb] slab of one output frame
    const unsigned long long dims[5] = {(unsigned long long)d.C, (unsigned long long)d.W, (unsigned long long)d.H, (unsigned long long)d.F,
                                        (unsigned long long)(d.batch_index && d.src_batch > 0 ? d.src_batch : B)};
    const unsigned long long strides[4] = {(unsigned long long)d.x_token_stride * es, (unsigned long long)d.x_token_stride * d.W * es,
                                           (unsigned long long)d.x_frame_stride * es, (unsigned long long)d.x_batch_stride * es};
    const unsigned box[5] = {(unsigned)pl.cb, (unsigned)d.W, (unsigned)d.H, (unsigned)pl.nf_max, 1};
    if (int rc = encode_tmap_cached(&maps.m[i], es == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, d.x, dims, strides,
                                    box, CU_TENSOR_MAP_SWIZZLE_NONE))
      return rc;
  }
  for (int i = n; i < MERV_MAX_ENCODERS; ++i) maps.m[i] = maps.m[0];
  p.total_items = begin;
  MERV_CUDA_OK(cudaFuncSetAttribute(pool3d_tma_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, PT_SMEM));
  int sms = sm_count();
  if (max_ctas > 0 && max_ctas < sms) sms = max_ctas;
  const int grid = begin < sms ? begin : sms;
  pool3d_tma_kernel<T><<<grid, PT_THREADS, PT_SMEM, s>>>(maps, p);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

static int launch_direct(const merv_pool_desc* enc, int n, int B, int dtype, cudaStream_t s) {
  const int vec = dtype == MERV_BF16 ? 8 : 4;
  PoolParams p;
  int max_items = 0, max_vec = 0;
  for (int i = 0; i < n; ++i) {
    const merv_pool_desc& d = enc[i];
    PoolEnc& e = p.enc[i];
    e.x = d.x; e.y = d.y; e.score_vec = d.score_vec; e.score_partial = d.score_partial; e.batch_index = d.batch_index;
    e.F = d.F; e.H = d.H; e.W = d.W; e.C = d.C; e.T = d.T; e.S = d.S;
    e.src_batch = d.batch_index && d.src_batch > 0 ? d.src_batch : B;
    e.sf = d.shift_f; e.sh = d.shift_h; e.sw = d.shift_w;
    e.rows_per_item = direct_rows_per_item(d.S);
    e.groups = (d.S + e.rows_per_item - 1) / e.rows_per_item;
    e.items = B * d.T * e.groups;
    e.xbs = d.x_batch_stride; e.xfs = d.x_frame_stride; e.xts = d.x_token_stride;
    e.ybs = d.y_batch_stride; e.yrs = d.y_row_stride;
    max_items = e.items > max_items ? e.items : max_items;
    max_vec = d.C / vec > max_vec ? d.C / vec : max_vec;
  }
  int threads = ((max_vec + 31) / 32) * 32;
  if (threads > 256) threads = 256;
  dim3 grid(max_items, n);
  if (dtype == MERV_BF16)
    pool3d_direct_kernel<__nv_bfloat16><<<grid, threads, 0, s>>>(p);
  else
    pool3d_direct_kernel<float><<<grid, threads, 0, s>>>(p);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

}  // namespace merv

using namespace merv;

extern "C" int merv_pool3d_score_parts(const merv_pool_desc* enc, int num_encoders, int dtype, int32_t* parts) {
  MERV_REQUIRE(enc && parts, MERV_E_ARG, "merv_pool3d_score_parts: NULL pointer");
  MERV_REQUIRE(num_encoders >= 1 && num_encoders <= MERV_MAX_ENCODERS, MERV_E_ARG, "merv_pool3d_score_parts: num_encoders=%d", num_encoders);
  MERV_REQUIRE(dtype == MERV_F32 || dtype == MERV_BF16, MERV_E_DTYPE, "merv_pool3d_score_parts: unknown dtype %d", dtype);
  const bool tma = use_tma(enc, num_encoders, dtype);
  for (int i = 0; i < num_encoders; ++i) {
    const merv_pool_desc& d = enc[i];
    MERV_REQUIRE(d.T > 0 && d.S > 0 && d.C > 0 && d.H > 0 && d.W > 0, MERV_E_SHAPE, "merv_pool3d_score_parts: encoder %d has a non-positive dimension", i);
    if (tma) {
      parts[i] = d.T * plan_tma(d, dtype).nchunks * PT_GROUP_WARPS;
    } else {
      const int rpi = direct_rows_per_item(d.S);
      parts[i] = d.T * ((d.S + rpi - 1) / rpi);
    }
  }
  return MERV_OK;
}

extern "C" int merv_pool3d(const merv_pool_desc* enc, int num_encoders, int B, int dtype, int max_ctas, void* stream) {
  if (int rc = validate(enc, num_encoders, B, dtype)) return rc;
  if (int rc = require_sm100()) return rc;
  if (B == 0) return MERV_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (use_tma(enc, num_encoders, dtype))
    return dtype == MERV_BF16 ? launch_tma<__nv_bfloat16>(enc, num_encoders, B, dtype, max_ctas, s) : launch_tma<float>(enc, num_encoders, B, dtype, max_ctas, s);
  return launch_direct(enc, num_encoders, B, dtype, s);
}
