// Cross attention of the attentive pooler ("attntv" resampler) on the 5th-gen tensor cores.
//   CrossAttention.forward, merv/util/nn_utils.py:393-412 (inside AttentivePooler.forward :229-238):
//       out[b, q, h*hd:(h+1)*hd] = softmax_k(scale * Q[q, h] . K[b, k, h]) V[b, k, h]
// K and V are the two halves of the `kv` Linear's output row ([K(C) | V(C)], heads contiguous inside each half, :398-399); the learned
// queries are the same for every batch entry (frame).  Both contractions are GEMM-shaped (2 * 2 * n_q * n_kv * C FLOP per frame) and run
// as tcgen05.mma with the accumulators in TMEM; the fp32 SIMT kernel of attention.cu remains the 1e-5 parity path (fp32 storage) and
// the fallback for shapes outside this kernel's tile (more than 128 queries or 256 keys per frame, head_dim not a multiple of 32).
//
// Work item = (frame b, head h); persistent CTAs, 6 warps:
//   warp 4  producer : TMA loads of Q_h [n_q x hd], K_h [n_kv x hd], V_h [n_kv x hd] through 4-D tensor maps (hd, head, row, frame): rows
//                      past n_q / n_kv and head dims past hd are zero-filled, so padding never needs masking on the operand side
//   warp 5  MMA      : S = Q_h K_h^T   (UMMA 128 x n_kv x 16, A and B K-major)            -> TMEM columns [0, 256)
//                      O = P V_h       (UMMA 128 x hd x 16, A = P K-major from shared memory, B = V_h read MN-major IN PLACE:
//                                       the same [keys x hd] image the TMA wrote, no transposed copy)  -> TMEM columns [256, 256 + hd)
//   warps 0-3 softmax: thread = query row: two passes over its S row in TMEM (tcgen05.ld): max, then exp2 / sum / bf16 P into shared
//                      memory in the 128-byte-swizzled K-major layout the second MMA reads; later O * (1 / sum) -> bf16 -> global.
// K is released as soon as the S MMAs have read it and V as soon as the PV MMAs have, so the loads of the next item overlap the
// softmax and the second MMA of the current one.
#include <cuda.h>

#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "tcgen05_util.cuh"
#include "tmap.cuh"

namespace merv {

constexpr int AT_M = 128;                  // UMMA M: query rows (zero-padded)
constexpr int AT_KEYS = 256;               // keys per frame covered by the S tile
constexpr int AT_MAX_HD = 128;
constexpr int AT_Q_CHUNK = AT_M * 128;     // [128 rows x 64 head dims] bf16, 128-byte swizzle
constexpr int AT_KV_CHUNK = AT_KEYS * 128; // [256 keys x 64 head dims]
constexpr int AT_P_CHUNK = AT_M * 128;     // [128 rows x 64 keys]
constexpr int AT_HD_CHUNKS = AT_MAX_HD / 64;
constexpr int AT_Q_OFF = 0;
constexpr int AT_K_OFF = AT_Q_OFF + AT_HD_CHUNKS * AT_Q_CHUNK;
constexpr int AT_V_OFF = AT_K_OFF + AT_HD_CHUNKS * AT_KV_CHUNK;
constexpr int AT_P_OFF = AT_V_OFF + AT_HD_CHUNKS * AT_KV_CHUNK;
constexpr int AT_BAR_OFF = AT_P_OFF + (AT_KEYS / 64) * AT_P_CHUNK;
constexpr int AT_SMEM = 1024 + AT_BAR_OFF + 128;
static_assert(AT_SMEM <= 232448, "227 KB of shared memory per CTA");
constexpr int AT_THREADS = 192;
constexpr int AT_TMEM_COLS = 512;          // S: columns [0, 256), O: [256, 256 + hd)

struct AttnParams {
  __nv_bfloat16* out;
  long long ldo;
  int batches, heads, n_q, n_kv, hd;
  int q_per_batch;   // 1: every frame has its own queries (4th coordinate of the Q map = frame), 0: shared learned queries
  float scale_log2e; // softmax scale * log2(e)
};
struct AttnMaps {
  CUtensorMap q, kv;
};

__device__ __forceinline__ void tma_load_4d(const CUtensorMap* map, uint32_t bar, uint32_t dst, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
               ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
// MN-major operand with an explicit distance between its 64-element chunks (see umma_desc_mn_sw128)
__device__ __forceinline__ uint64_t umma_desc_mn_sw128_lbo(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(lbo_bytes >> 4) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

__global__ void __launch_bounds__(AT_THREADS, 1) cross_attention_tcgen05_kernel(const __grid_constant__ AttnMaps maps, const __grid_constant__ AttnParams p) {
  extern __shared__ uint8_t at_smem_raw[];
  const uint32_t raw = smem_u32(at_smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* aligned = at_smem_raw + (base - raw);
  uint64_t* bars = reinterpret_cast<uint64_t*>(aligned + AT_BAR_OFF);
  const uint32_t bar0 = smem_u32(bars);
  const uint32_t k_full = bar0, k_empty = bar0 + 8, v_full = bar0 + 16, v_empty = bar0 + 24, s_full = bar0 + 32, s_empty = bar0 + 40,
                 p_full = bar0 + 48, o_full = bar0 + 56, o_empty = bar0 + 64;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 10);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int items = p.batches * p.heads;
  const int hd_chunks = (p.hd + 63) / 64;

  if (warp == 4 && lane == 0) {
    prefetch_tmap(&maps.q);
    prefetch_tmap(&maps.kv);
    mbar_init(k_full, 1); mbar_init(k_empty, 1); mbar_init(v_full, 1); mbar_init(v_empty, 1);
    mbar_init(s_full, 1); mbar_init(s_empty, 4); mbar_init(p_full, 4); mbar_init(o_full, 1); mbar_init(o_empty, 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 5) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "n"(AT_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const uint32_t tmem_S = tmem_base, tmem_O = tmem_base + AT_KEYS;

  if (warp == 4) {
    {
      // ===== producer (warp-uniform loop, one lane issues under elect.sync: tcgen05_util.cuh) =====
      uint32_t it = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
        const int b = item / p.heads, h = item - b * p.heads;
        const uint32_t ph = it & 1u;
        mbar_wait(k_empty, ph ^ 1u);
        if (elect_one()) {
          mbar_expect_tx(k_full, uint32_t(hd_chunks) * (AT_Q_CHUNK + AT_KV_CHUNK));
          for (int c = 0; c < hd_chunks; ++c) {
            tma_load_4d(&maps.q, k_full, base + AT_Q_OFF + c * AT_Q_CHUNK, c * 64, h, 0, p.q_per_batch ? b : 0);
            tma_load_4d(&maps.kv, k_full, base + AT_K_OFF + c * AT_KV_CHUNK, c * 64, h, 0, b);
          }
        }
        __syncwarp();
        mbar_wait(v_empty, ph ^ 1u);
        if (elect_one()) {
          mbar_expect_tx(v_full, uint32_t(hd_chunks) * AT_KV_CHUNK);
          for (int c = 0; c < hd_chunks; ++c) tma_load_4d(&maps.kv, v_full, base + AT_V_OFF + c * AT_KV_CHUNK, c * 64, p.heads + h, 0, b);
        }
        __syncwarp();
      }
    }
  } else if (warp == 5) {
    {
      // ===== MMA issuer (warp-uniform loop, one lane issues under elect.sync) =====
      const int n_keys16 = (p.n_kv + 15) & ~15;  // UMMA N of S and the k extent of P V
      const uint32_t idesc_s = umma_idesc_bf16(AT_M, n_keys16, 0, 0);
      const uint32_t idesc_o = umma_idesc_bf16(AT_M, p.hd, 0, 1);  // B = V_h MN-major
      uint32_t it = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
        const uint32_t ph = it & 1u;
        mbar_wait(k_full, ph);
        mbar_wait(s_empty, ph ^ 1u);
        tc_fence_after();
        if (elect_one()) {
          for (int ks = 0; ks < p.hd / UMMA_K; ++ks) {
            const uint64_t a = umma_desc_sw128(base + AT_Q_OFF + (ks >> 2) * AT_Q_CHUNK) + 2 * (ks & 3);
            const uint64_t bd = umma_desc_sw128(base + AT_K_OFF + (ks >> 2) * AT_KV_CHUNK) + 2 * (ks & 3);
            umma_bf16(tmem_S, a, bd, idesc_s, ks != 0 ? 1u : 0u);
          }
          umma_commit(s_full);
          umma_commit(k_empty);  // Q_h / K_h may be overwritten by the next item's loads
        }
        __syncwarp();
        mbar_wait(p_full, ph);
        mbar_wait(v_full, ph);
        mbar_wait(o_empty, ph ^ 1u);
        tc_fence_after();
        if (elect_one()) {
          for (int ks = 0; ks < n_keys16 / UMMA_K; ++ks) {
            const uint64_t a = umma_desc_sw128(base + AT_P_OFF + (ks >> 2) * AT_P_CHUNK) + 2 * (ks & 3);
            const uint64_t bd = umma_desc_mn_sw128_lbo(base + AT_V_OFF, AT_KV_CHUNK) + uint64_t(ks) * (2048u >> 4);
            umma_bf16(tmem_O, a, bd, idesc_o, ks != 0 ? 1u : 0u);
          }
          umma_commit(o_full);
          umma_commit(v_empty);
        }
        __syncwarp();
      }
    }
  } else {
    // ===== softmax + output (warp w owns TMEM lanes 32 w .. 32 w + 31 = query rows) =====
    const int row = warp * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(warp * 32) << 16;
    const uint32_t p_row = base + AT_P_OFF + uint32_t(row) * 128u;
    const uint32_t sw = uint32_t(row) & 7u;
    uint32_t it = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
      const int b = item / p.heads, h = item - b * p.heads;
      const uint32_t ph = it & 1u;
      mbar_wait(s_full, ph);
      tc_fence_after();
      float m = -INFINITY;
#pragma unroll 1
      for (int c = 0; c < AT_KEYS / 32; ++c) {
        if (c * 32 >= p.n_kv) break;  // warp-uniform
        uint32_t v[32];
        tmem_ld32(tmem_S + lane_addr + c * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (c * 32 + i < p.n_kv) m = fmaxf(m, __uint_as_float(v[i]));
      }
      const float mo = m * p.scale_log2e;
      float sum = 0.f;
#pragma unroll 1
      for (int c = 0; c < AT_KEYS / 32; ++c) {
        if (c * 32 >= ((p.n_kv + 15) & ~15)) break;  // the second MMA reads P up to the next multiple of 16 keys only
        uint32_t v[32];
        const bool live = c * 32 < p.n_kv;  // warp-uniform
        if (live) {
          tmem_ld32(tmem_S + lane_addr + c * 32, v);
          tmem_ld_wait();
        }
        uint32_t packed[16];
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          float e0 = 0.f, e1 = 0.f;
          if (live && c * 32 + i < p.n_kv) e0 = exp2f(fmaf(__uint_as_float(v[i]), p.scale_log2e, -mo));
          if (live && c * 32 + i + 1 < p.n_kv) e1 = exp2f(fmaf(__uint_as_float(v[i + 1]), p.scale_log2e, -mo));
          sum += e0 + e1;
          packed[i >> 1] = pack_bf16x2(e0, e1);
        }
        // 32 keys = 64 bytes = four 16-byte chunks of this row inside the [128 x 64-key] P chunk c / 2
        const uint32_t chunk_base = p_row + uint32_t(c >> 1) * AT_P_CHUNK;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint32_t c16 = uint32_t((c & 1) * 4 + j);
          sts_v4(chunk_base + ((c16 ^ sw) << 4), make_uint4(packed[4 * j], packed[4 * j + 1], packed[4 * j + 2], packed[4 * j + 3]));
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes of P -> visible to the tensor core's shared-memory reads
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(p_full);
        mbar_arrive(s_empty);  // this warp is done with its rows of S
      }
      const float inv = 1.0f / sum;
      mbar_wait(o_full, ph);
      tc_fence_after();
      __nv_bfloat16* orow = p.out + ((long long)b * p.n_q + row) * p.ldo + (long long)h * p.hd;
#pragma unroll 1
      for (int c = 0; c < p.hd / 32; ++c) {
        uint32_t v[32];
        tmem_ld32(tmem_O + lane_addr + c * 32, v);
        tmem_ld_wait();
        if (row < p.n_q) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float o[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = __uint_as_float(v[8 * j + i]) * inv;
            *reinterpret_cast<uint4*>(orow + c * 32 + 8 * j) = Vec16<__nv_bfloat16>::pack(o);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_empty);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(AT_TMEM_COLS) : "memory");
  }
}

// ============================================================================================================
// Backward of the cross attention (training the "attntv" resampler): all five contractions on the tensor cores.
//   S  = Q K^T, P = softmax(scale S)                       (recomputed, not stored by the forward)
//   dP = dO V^T;   D_i = sum_j P_ij dP_ij;   dS = scale P (.) (dP - D)
//   dV = P^T dO;   dK = dS^T Q;   dQ = dS K                (dQ per frame; the caller sums the frames when the queries are shared)
// One shared-memory image per operand serves BOTH of its roles, because a [rows x 128 B] swizzled tile is K-major with respect to its
// rows and MN-major with respect to its columns: Q is the K-major A of S and the MN-major B of dK, dO the K-major A of dP and the MN-major
// B of dV, K the K-major B of S and the MN-major B of dQ, V the K-major B of dP; P and dS (written by the softmax warps) are the
// MN-major A of dV / dK (M = keys) and dS also the K-major A of dQ.  n_q <= 64 (the resampler's queries per frame), n_kv <= 256.
// TMEM: S -> [0, 256), dP -> [256, 512); once both are consumed, dV_half -> [0, hd), dK_half -> [128, 128 + hd) for the two halves of the
// keys in turn and dQ -> [256, 256 + hd).
// ============================================================================================================
constexpr int AB_ROWS = 64;                 // query rows held in shared memory (the UMMAs still run M = 128: rows past 64 read the next buffer)
constexpr int AB_CH = AB_ROWS * 128;        // [64 rows x 64 elements] chunk, 8 KB
constexpr int AB_Q_OFF = 0;                                         // 2 chunks (head dims 0-63, 64-127)
constexpr int AB_DO_OFF = AB_Q_OFF + AT_HD_CHUNKS * AB_CH;
constexpr int AB_K_OFF = AB_DO_OFF + AT_HD_CHUNKS * AB_CH;
constexpr int AB_V_OFF = AB_K_OFF + AT_HD_CHUNKS * AT_KV_CHUNK;
constexpr int AB_DS_OFF = AB_V_OFF + AT_HD_CHUNKS * AT_KV_CHUNK;    // 4 chunks (keys 0-63, ...); its M = 128 reads run over into P: finite data
constexpr int AB_P_OFF = AB_DS_OFF + (AT_KEYS / 64) * AB_CH;
constexpr int AB_BAR_OFF = AB_P_OFF + (AT_KEYS / 64) * AB_CH;  // P is only read MN-major (k = query rows < 64): nothing runs over its end
constexpr int AB_SMEM = 1024 + AB_BAR_OFF + 128;
static_assert(AB_SMEM <= 232448, "227 KB of shared memory per CTA");

struct AttnBwdParams {
  __nv_bfloat16* dkv;  // [batches * n_kv, 2 C] = [dK | dV]
  long long lddkv;
  __nv_bfloat16* dq;   // [batches, n_q, C]: dQ of every frame
  long long lddq;
  int batches, heads, n_q, n_kv, hd;
  int q_per_batch;
  float scale, scale_log2e;
};
struct AttnBwdMaps {
  CUtensorMap q, kv, dout;
};

__global__ void __launch_bounds__(AT_THREADS, 1) cross_attention_bwd_tcgen05_kernel(const __grid_constant__ AttnBwdMaps maps,
                                                                                    const __grid_constant__ AttnBwdParams p) {
  extern __shared__ uint8_t at_smem_raw[];
  const uint32_t raw = smem_u32(at_smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* aligned = at_smem_raw + (base - raw);
  uint64_t* bars = reinterpret_cast<uint64_t*>(aligned + AB_BAR_OFF);
  const uint32_t bar0 = smem_u32(bars);
  const uint32_t ld_full = bar0, ld_empty = bar0 + 8, sdp_full = bar0 + 16, pds_full = bar0 + 24, dvk_full0 = bar0 + 32, dvk_full1 = bar0 + 40,
                 dvk_empty0 = bar0 + 48, dvk_empty1 = bar0 + 56, dq_full = bar0 + 64, dq_empty = bar0 + 72;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 11);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int items = p.batches * p.heads;
  const int hd_chunks = (p.hd + 63) / 64;
  constexpr int ROW_WARPS = AB_ROWS / 32;  // softmax warps that own query rows

  if (warp == 4 && lane == 0) {
    prefetch_tmap(&maps.q);
    prefetch_tmap(&maps.kv);
    prefetch_tmap(&maps.dout);
    mbar_init(ld_full, 1); mbar_init(ld_empty, 1); mbar_init(sdp_full, 1); mbar_init(pds_full, ROW_WARPS);
    mbar_init(dvk_full0, 1); mbar_init(dvk_full1, 1); mbar_init(dvk_empty0, 4); mbar_init(dvk_empty1, 4);
    mbar_init(dq_full, 1); mbar_init(dq_empty, ROW_WARPS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 5) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "n"(AT_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // the run-over reads of the M = 128 UMMAs must see finite data from the first item on
  for (int i = threadIdx.x; i < (AB_BAR_OFF - AB_DS_OFF) / 16; i += AT_THREADS)
    reinterpret_cast<uint4*>(aligned + AB_DS_OFF)[i] = make_uint4(0u, 0u, 0u, 0u);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const int n_keys16 = (p.n_kv + 15) & ~15;
  const int n_q16 = (p.n_q + 15) & ~15;

  if (warp == 4) {
    {
      // ===== producer: Q_h, dO_h, K_h, V_h of one (frame, head); warp-uniform loop, one lane issues under elect.sync =====
      uint32_t it = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
        const int b = item / p.heads, h = item - b * p.heads;
        mbar_wait(ld_empty, (it & 1u) ^ 1u);
        if (elect_one()) {
          mbar_expect_tx(ld_full, uint32_t(hd_chunks) * (2 * AB_CH + 2 * AT_KV_CHUNK));
          for (int c = 0; c < hd_chunks; ++c) {
            tma_load_4d(&maps.q, ld_full, base + AB_Q_OFF + c * AB_CH, c * 64, h, 0, p.q_per_batch ? b : 0);
            tma_load_4d(&maps.dout, ld_full, base + AB_DO_OFF + c * AB_CH, c * 64, h, 0, b);
            tma_load_4d(&maps.kv, ld_full, base + AB_K_OFF + c * AT_KV_CHUNK, c * 64, h, 0, b);
            tma_load_4d(&maps.kv, ld_full, base + AB_V_OFF + c * AT_KV_CHUNK, c * 64, p.heads + h, 0, b);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 5) {
    {
      // ===== MMA issuer (warp-uniform loop, one lane issues under elect.sync) =====
      const uint32_t idesc_s = umma_idesc_bf16(AT_M, n_keys16, 0, 0);   // S, dP: [128 x keys], K-major operands
      const uint32_t idesc_t = umma_idesc_bf16(AT_M, p.hd, 1, 1);       // dV, dK: [128 keys x hd], both operands MN-major
      const uint32_t idesc_q = umma_idesc_bf16(AT_M, p.hd, 0, 1);       // dQ: [128 x hd], A = dS K-major, B = K_h MN-major
      uint32_t it = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
        const uint32_t ph = it & 1u;
        mbar_wait(ld_full, ph);
        mbar_wait(dvk_empty1, ph ^ 1u);  // the previous item's accumulators have been drained
        mbar_wait(dq_empty, ph ^ 1u);
        tc_fence_after();
        if (elect_one()) {
        for (int ks = 0; ks < p.hd / UMMA_K; ++ks) {  // S = Q K^T and dP = dO V^T
          const uint32_t off = uint32_t(ks >> 2), k2 = 2u * uint32_t(ks & 3);
          umma_bf16(tmem_base, umma_desc_sw128(base + AB_Q_OFF + off * AB_CH) + k2, umma_desc_sw128(base + AB_K_OFF + off * AT_KV_CHUNK) + k2, idesc_s,
                    ks != 0 ? 1u : 0u);
        }
        for (int ks = 0; ks < p.hd / UMMA_K; ++ks) {
          const uint32_t off = uint32_t(ks >> 2), k2 = 2u * uint32_t(ks & 3);
          umma_bf16(tmem_base + AT_KEYS, umma_desc_sw128(base + AB_DO_OFF + off * AB_CH) + k2, umma_desc_sw128(base + AB_V_OFF + off * AT_KV_CHUNK) + k2,
                    idesc_s, ks != 0 ? 1u : 0u);
        }
        umma_commit(sdp_full);
        }
        __syncwarp();
        mbar_wait(pds_full, ph);
        tc_fence_after();
        auto dvk = [&](int half) {  // dV_half = P[:, half]^T dO -> columns [0, hd); dK_half = dS[:, half]^T Q -> columns [128, 128 + hd)
          for (int ks = 0; ks < n_q16 / UMMA_K; ++ks) {
            const uint64_t kstep = uint64_t(ks) * (2048u >> 4);
            umma_bf16(tmem_base, umma_desc_mn_sw128_lbo(base + AB_P_OFF + half * 2 * AB_CH, AB_CH) + kstep,
                      umma_desc_mn_sw128_lbo(base + AB_DO_OFF, AB_CH) + kstep, idesc_t, ks != 0 ? 1u : 0u);
          }
          for (int ks = 0; ks < n_q16 / UMMA_K; ++ks) {
            const uint64_t kstep = uint64_t(ks) * (2048u >> 4);
            umma_bf16(tmem_base + 128, umma_desc_mn_sw128_lbo(base + AB_DS_OFF + half * 2 * AB_CH, AB_CH) + kstep,
                      umma_desc_mn_sw128_lbo(base + AB_Q_OFF, AB_CH) + kstep, idesc_t, ks != 0 ? 1u : 0u);
          }
        };
        if (elect_one()) {
        dvk(0);
        umma_commit(dvk_full0);
        for (int ks = 0; ks < n_keys16 / UMMA_K; ++ks) {  // dQ = dS K -> columns [256, 256 + hd)
          const uint64_t a = umma_desc_sw128(base + AB_DS_OFF + (ks >> 2) * AB_CH) + 2 * (ks & 3);
          const uint64_t bd = umma_desc_mn_sw128_lbo(base + AB_K_OFF, AT_KV_CHUNK) + uint64_t(ks) * (2048u >> 4);
          umma_bf16(tmem_base + AT_KEYS, a, bd, idesc_q, ks != 0 ? 1u : 0u);
        }
        umma_commit(dq_full);
        }
        __syncwarp();
        mbar_wait(dvk_empty0, ph);
        tc_fence_after();
        if (elect_one()) {
          dvk(1);
          umma_commit(dvk_full1);
          umma_commit(ld_empty);  // every operand of this item has been read
        }
        __syncwarp();
      }
    }
  } else {
    // ===== softmax / dS (warps 0 .. ROW_WARPS-1: thread = query row) and accumulator drains (all four warps: thread = key or query row) =====
    const int row = warp * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(warp * 32) << 16;
    const uint32_t sw = uint32_t(row) & 7u;
    uint32_t it = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
      const int b = item / p.heads, h = item - b * p.heads;
      const uint32_t ph = it & 1u;
      if (warp < ROW_WARPS) {
        mbar_wait(sdp_full, ph);
        tc_fence_after();
        const int nc = (n_keys16 + 31) / 32;
        float m = -INFINITY;
#pragma unroll 1
        for (int c = 0; c < nc; ++c) {
          uint32_t v[32];
          tmem_ld32(tmem_base + lane_addr + c * 32, v);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (c * 32 + i < p.n_kv) m = fmaxf(m, __uint_as_float(v[i]));
        }
        const float mo = m * p.scale_log2e;
        float sum = 0.f, dn = 0.f;
#pragma unroll 1
        for (int c = 0; c < nc; ++c) {
          uint32_t v[32], g[32];
          tmem_ld32(tmem_base + lane_addr + c * 32, v);
          tmem_ld32(tmem_base + AT_KEYS + lane_addr + c * 32, g);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            if (c * 32 + i < p.n_kv) {
              const float e = exp2f(fmaf(__uint_as_float(v[i]), p.scale_log2e, -mo));
              sum += e;
              dn = fmaf(e, __uint_as_float(g[i]), dn);
            }
          }
        }
        const float inv = 1.0f / sum;
        const float D = dn * inv;
#pragma unroll 1
        for (int c = 0; c < nc; ++c) {
          uint32_t v[32], g[32];
          tmem_ld32(tmem_base + lane_addr + c * 32, v);
          tmem_ld32(tmem_base + AT_KEYS + lane_addr + c * 32, g);
          tmem_ld_wait();
          uint32_t pp[16], ds[16];
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            float p0 = 0.f, p1 = 0.f;
            if (c * 32 + i < p.n_kv) p0 = exp2f(fmaf(__uint_as_float(v[i]), p.scale_log2e, -mo)) * inv;
            if (c * 32 + i + 1 < p.n_kv) p1 = exp2f(fmaf(__uint_as_float(v[i + 1]), p.scale_log2e, -mo)) * inv;
            pp[i >> 1] = pack_bf16x2(p0, p1);
            ds[i >> 1] = pack_bf16x2(p.scale * p0 * (__uint_as_float(g[i]) - D), p.scale * p1 * (__uint_as_float(g[i + 1]) - D));
          }
          const uint32_t chunk = uint32_t(c >> 1) * AB_CH + uint32_t(row) * 128u;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t c16 = ((uint32_t((c & 1) * 4 + j)) ^ sw) << 4;
            sts_v4(base + AB_P_OFF + chunk + c16, make_uint4(pp[4 * j], pp[4 * j + 1], pp[4 * j + 2], pp[4 * j + 3]));
            sts_v4(base + AB_DS_OFF + chunk + c16, make_uint4(ds[4 * j], ds[4 * j + 1], ds[4 * j + 2], ds[4 * j + 3]));
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(pds_full);
      }
      auto drain_dvk = [&](int half, uint32_t full_bar, uint32_t empty_bar) {
        mbar_wait(full_bar, ph);
        tc_fence_after();
        const int key = half * 128 + row;
        __nv_bfloat16* dst = p.dkv + ((long long)b * p.n_kv + key) * p.lddkv + (long long)h * p.hd;
        const long long v_off = (long long)p.heads * p.hd;  // the dV half of the row
#pragma unroll 1
        for (int c = 0; c < p.hd / 32; ++c) {
          uint32_t dv[32], dk[32];
          tmem_ld32(tmem_base + lane_addr + c * 32, dv);
          tmem_ld32(tmem_base + 128 + lane_addr + c * 32, dk);
          tmem_ld_wait();
          if (key < p.n_kv) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              float a[8], bb[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                a[i] = __uint_as_float(dk[8 * j + i]);
                bb[i] = __uint_as_float(dv[8 * j + i]);
              }
              *reinterpret_cast<uint4*>(dst + c * 32 + 8 * j) = Vec16<__nv_bfloat16>::pack(a);
              *reinterpret_cast<uint4*>(dst + v_off + c * 32 + 8 * j) = Vec16<__nv_bfloat16>::pack(bb);
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(empty_bar);
      };
      drain_dvk(0, dvk_full0, dvk_empty0);
      if (warp < ROW_WARPS) {
        mbar_wait(dq_full, ph);
        tc_fence_after();
        __nv_bfloat16* dst = p.dq + ((long long)b * p.n_q + row) * p.lddq + (long long)h * p.hd;
#pragma unroll 1
        for (int c = 0; c < p.hd / 32; ++c) {
          uint32_t v[32];
          tmem_ld32(tmem_base + AT_KEYS + lane_addr + c * 32, v);
          tmem_ld_wait();
          if (row < p.n_q) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              float a[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) a[i] = __uint_as_float(v[8 * j + i]);
              *reinterpret_cast<uint4*>(dst + c * 32 + 8 * j) = Vec16<__nv_bfloat16>::pack(a);
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(dq_empty);
      }
      drain_dvk(1, dvk_full1, dvk_empty1);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(AT_TMEM_COLS) : "memory");
  }
}

static int make_attn_map(CUtensorMap* map, const void* ptr, int hd, int heads_dim, int rows, long long ld, long long batch_stride, int batches, int box_rows) {
  const unsigned long long dims[4] = {(unsigned long long)hd, (unsigned long long)heads_dim, (unsigned long long)rows, (unsigned long long)batches};
  const unsigned long long strides[3] = {(unsigned long long)hd * 2, (unsigned long long)ld * 2, (unsigned long long)batch_stride * 2};
  const unsigned box[4] = {64, 1, (unsigned)box_rows, 1};
  return encode_tmap_cached(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, ptr, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

int launch_attention_bwd_tcgen05(const void* q, long long ldq, long long q_batch_stride, const void* kv, long long ldkv, const void* dout, long long lddo,
                                 void* dq, long long lddq, void* dkv, long long lddkv, int batches, int n_q, int n_kv, int heads, int hd, float scale,
                                 cudaStream_t stream) {
  MERV_REQUIRE(n_q <= AB_ROWS && n_kv <= AT_KEYS && hd % 32 == 0 && hd <= AT_MAX_HD, MERV_E_SHAPE,
               "cross attention backward: at most %d queries and %d keys per frame, head_dim a multiple of 32 up to %d (got n_q=%d n_kv=%d head_dim=%d)",
               AB_ROWS, AT_KEYS, AT_MAX_HD, n_q, n_kv, hd);
  MERV_REQUIRE(ldq % 8 == 0 && ldkv % 8 == 0 && lddo % 8 == 0 && lddq % 8 == 0 && lddkv % 8 == 0 && q_batch_stride % 8 == 0 && aligned16(q) && aligned16(kv) &&
                   aligned16(dout) && aligned16(dq) && aligned16(dkv),
               MERV_E_ALIGN, "cross attention backward: rows must be 16-byte aligned");
  AttnBwdMaps maps;
  AttnBwdParams p = {};
  p.dkv = static_cast<__nv_bfloat16*>(dkv); p.lddkv = lddkv; p.dq = static_cast<__nv_bfloat16*>(dq); p.lddq = lddq;
  p.batches = batches; p.heads = heads; p.n_q = n_q; p.n_kv = n_kv; p.hd = hd;
  p.q_per_batch = q_batch_stride != 0 ? 1 : 0;
  p.scale = scale; p.scale_log2e = scale * 1.4426950408889634f;
  if (int rc = make_attn_map(&maps.q, q, hd, heads, n_q, ldq, p.q_per_batch ? q_batch_stride : (long long)n_q * ldq, p.q_per_batch ? batches : 1, AB_ROWS)) return rc;
  if (int rc = make_attn_map(&maps.dout, dout, hd, heads, n_q, lddo, (long long)n_q * lddo, batches, AB_ROWS)) return rc;
  if (int rc = make_attn_map(&maps.kv, kv, hd, 2 * heads, n_kv, ldkv, (long long)n_kv * ldkv, batches, AT_KEYS)) return rc;
  static const cudaError_t attr_rc =
      cudaFuncSetAttribute(cross_attention_bwd_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AB_SMEM);
  MERV_REQUIRE(attr_rc == cudaSuccess, MERV_E_CUDA, "cudaFuncSetAttribute(max dynamic smem=%d) failed: %s", AB_SMEM, cudaGetErrorString(attr_rc));
  const long long items = (long long)batches * heads;
  const int sms = sm_count();
  const unsigned grid = unsigned(items < sms ? items : sms);
  cross_attention_bwd_tcgen05_kernel<<<grid, AT_THREADS, AB_SMEM, stream>>>(maps, p);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

static bool attention_simt_forced() {
  const char* e = getenv("MERV_ATTN_IMPL");
  return e != nullptr && strcmp(e, "simt") == 0;
}

bool attention_bwd_tcgen05_supported(int n_q, int n_kv, int hd) {
  return !attention_simt_forced() && n_q <= AB_ROWS && n_kv <= AT_KEYS && hd % 32 == 0 && hd <= AT_MAX_HD;
}

bool attention_tcgen05_supported(int n_q, int n_kv, int heads, int hd, long long ldq, long long q_batch_stride, long long ldkv, long long ldo) {
  if (attention_simt_forced()) return false;
  (void)heads;
  return n_q <= AT_M && n_kv <= AT_KEYS && hd % 32 == 0 && hd <= AT_MAX_HD && ldq % 8 == 0 && ldkv % 8 == 0 && ldo % 8 == 0 && q_batch_stride % 8 == 0;
}

int launch_attention_tcgen05(const void* q, long long ldq, long long q_batch_stride, const void* kv, long long ldkv, void* out, long long ldo,
                             int batches, int n_q, int n_kv, int heads, int hd, float scale, cudaStream_t stream) {
  MERV_REQUIRE(aligned16(q) && aligned16(kv) && aligned16(out), MERV_E_ALIGN, "cross attention: operands must be 16-byte aligned");
  AttnMaps maps;
  AttnParams p = {};
  p.out = static_cast<__nv_bfloat16*>(out); p.ldo = ldo;
  p.batches = batches; p.heads = heads; p.n_q = n_q; p.n_kv = n_kv; p.hd = hd;
  p.q_per_batch = q_batch_stride != 0 ? 1 : 0;
  p.scale_log2e = scale * 1.4426950408889634f;
  {
    // Q as (head dim, head, query row, frame); rows past n_q and head dims past hd are zero-filled by TMA
    const unsigned long long dims[4] = {(unsigned long long)hd, (unsigned long long)heads, (unsigned long long)n_q,
                                        (unsigned long long)(p.q_per_batch ? batches : 1)};
    const unsigned long long strides[3] = {(unsigned long long)hd * 2, (unsigned long long)ldq * 2,
                                           (unsigned long long)(p.q_per_batch ? q_batch_stride : (long long)n_q * ldq) * 2};
    const unsigned box[4] = {64, 1, AT_M, 1};
    if (int rc = encode_tmap_cached(&maps.q, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, q, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  }
  {
    // kv rows [K(C) | V(C)] as (head dim, 2 x heads, key, frame): head h of K is "head" h, of V "head" heads + h
    const unsigned long long dims[4] = {(unsigned long long)hd, (unsigned long long)(2 * heads), (unsigned long long)n_kv, (unsigned long long)batches};
    const unsigned long long strides[3] = {(unsigned long long)hd * 2, (unsigned long long)ldkv * 2, (unsigned long long)n_kv * ldkv * 2};
    const unsigned box[4] = {64, 1, AT_KEYS, 1};
    if (int rc = encode_tmap_cached(&maps.kv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, kv, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  }
  static const cudaError_t attr_rc =
      cudaFuncSetAttribute(cross_attention_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AT_SMEM);
  MERV_REQUIRE(attr_rc == cudaSuccess, MERV_E_CUDA, "cudaFuncSetAttribute(max dynamic smem=%d) failed: %s", AT_SMEM, cudaGetErrorString(attr_rc));
  const long long items = (long long)batches * heads;
  const int sms = sm_count();
  const unsigned grid = unsigned(items < sms ? items : sms);
  cross_attention_tcgen05_kernel<<<grid, AT_THREADS, AT_SMEM, stream>>>(maps, p);
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

}  // namespace merv
