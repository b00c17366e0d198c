// bf16 projector GEMM on the 5th-gen tensor cores (tcgen05.mma, accumulators in TMEM, operands by TMA).
//
// One persistent, warp-specialised kernel body (gemm_body) serves every dense contraction of the path:
//
//   merv_linear_bias_act   Y = act(A W^T + bias)                  (nn.Linear [+ nn.GELU], merv/util/nn_utils.py:31-32,46-55)
//   merv_fused_linear_mix  out = sum_s w[video,s] * (A_s W_s^T) + bias_mix[video]
//                          (E LinearProjectors + the stack/bmm of CrossAttentionAdapterLearnableQuery.forward,
//                           nn_utils.py:31-32,503,521, without ever writing the per-encoder projections to HBM)
//   merv_gemm_ex           the same with either operand stored transposed (MN-major: the backward's dX = dY W, dW = dY^T X)
//   merv_wgrad_video       dW = sum_b w[b] dY[b]^T X[b] and <W, dY[b]^T X[b]> per video: the accumulator is drained once per video
//
// Tile 128 x 256 x 64 per CTA, as a CTA pair (cluster 2 x 1, cta_group::2, UMMA 256x256x16: each CTA loads its 128 rows of A and HALF of
// the W tile, 6-stage ring of 32 KB) or as a single CTA (UMMA 128x256x16, 4 stages of 48 KB); TMA -> shared memory with 128-byte swizzle;
// two 256-column TMEM accumulators.  A "segment" is one (A_s, W_s, K_s) product; the MMA warp alternates accumulators per segment, the 16
// epilogue warps drain each finished accumulator into fp32 registers scaled by the segment's mixing weight while the next segment (or
// next tile) is being multiplied, and after the last segment apply bias / erf-GELU / optional row-dot, stage the bf16 rows in shared
// memory and write them with TMA stores — each output element is written exactly once.
//
//   warp 0      TMA producer   \  warp-uniform loops; one lane issues under elect.sync (lane-0 guards made the compiler wrap every
//   warp 1      tcgen05.mma issuer /  UTMALDG / UTCHMMA in an ELECT / R2UR waterfall loop: tensor pipe 84 % -> 95 % of elapsed without them)
//   warp 2      TMEM allocator
//   warp 3      idle
//   warps 4-19  epilogue: warp w owns TMEM lanes 32*(w%4)..+31 and columns 64*((w-4)/4)..+63 of the tile
// Template parameters: kCtas (1 | 2), kWide (128-byte-row output boxes: NVLink peer stores, short contractions), kGelu, kMaj (operand
// majorness, compile-time), kVid, kDy3.  Measured: fused forward 1614 TFLOP/s in the bench = 0.98 of the burst cuBLAS peak (DESIGN.md 5.2).
#include <cuda.h>

#include <cstdlib>

#include "common.cuh"
#include "tcgen05_util.cuh"
#include "tmap.cuh"

namespace merv {

constexpr int BM = 128, BN = 256, BK = 64;  // BM = rows per CTA; a CTA pair (cta_group::2) computes 256 x 256
constexpr int A_BYTES = BM * BK * 2;
// per-CTA stage: its 128 rows of A and, for a CTA pair, its half (128 rows) of the W tile
constexpr int EPI_WARPS = 16;                          // 4 per scheduler: the epilogue (erf-GELU, bias, row-dot) is issue/latency bound
constexpr int OUT_GROUPS = EPI_WARPS / 4;              // 4 groups of 4 warps, one staging box each
// kWide (the fused all-gather variant): output boxes of 128-byte rows instead of 64-byte rows — NVLink peer writes are
// packetised per box row, and 64-byte payloads only reach ~380 GB/s of egress — paid for with one ring stage.
template <int kCtas, bool kWide> struct Cfg {
  static constexpr int STAGES = (kCtas == 1 ? 4 : 6) - (kWide ? 1 : 0);
  static constexpr int B_ROWS = BN / kCtas;
  static constexpr int B_BYTES = B_ROWS * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int RING_BYTES = STAGES * STAGE_BYTES;  // 192 KB (144 / 160 KB when wide)
  static constexpr int OUT_BOX_COLS = kWide ? 64 : 32;      // one staged output box: 128 rows x 32 (64) bf16, 64B (128B) swizzle
  static constexpr int OUT_BOX_BYTES = BM * OUT_BOX_COLS * 2;
  static constexpr int SMEM_BYTES = 1024 /*align slack*/ + RING_BYTES + OUT_GROUPS * OUT_BOX_BYTES + 256 /*barriers*/;
  static_assert(RING_BYTES % 1024 == 0 && OUT_BOX_BYTES % 1024 == 0, "swizzle atoms need 1024-byte aligned boxes");
  static_assert(SMEM_BYTES <= 232448, "227 KB of shared memory per CTA");
};
constexpr int GEMM_THREADS = 128 + EPI_WARPS * 32;    // 640
constexpr int EPI_COLS = BN / (EPI_WARPS / 4);         // 64 accumulator columns per epilogue warp
static_assert(MERV_ROWDOT_BLOCK == EPI_COLS, "one row-dot partial per epilogue warp slice");
constexpr int TMEM_COLS = 512;
constexpr int KERNEL_REGS = 96, PRODUCER_REGS = 64, EPILOGUE_REGS = 104;  // see setmaxnreg below
static_assert(GEMM_THREADS * KERNEL_REGS <= 65536, "register file");
static_assert(128 * PRODUCER_REGS + EPI_WARPS * 32 * EPILOGUE_REGS <= GEMM_THREADS * KERNEL_REGS, "setmaxnreg.inc must fit in what setmaxnreg.dec released");

// MERV_GEMM_WARP_UNIFORM (build-time, A/B): the TMA producer and the MMA issuer run their loops as WHOLE warps and issue under elect.sync.
// With `lane == 0` guards the compiler cannot prove the operands of UTMALDG / UTCHMMA warp-uniform and wraps every issue in an
// ELECT / R2UR "waterfall" loop: ~80 (producer) and ~115 (MMA issuer) instructions per k-block for threads that get an issue slot every
// ~4 cycles, against ~512 cycles of tensor work per k-block.
#ifndef MERV_GEMM_WARP_UNIFORM
#define MERV_GEMM_WARP_UNIFORM 1
#endif
struct GemmParams {
  int M, N;
  int nseg;
  int kblocks[MERV_MAX_SEGMENTS];
  int a_mn_mask, b_mn_mask;  // bit s: segment s has an MN-major A / W operand (see GemmSegment)
  const float* seg_scale;  // [videos, nseg] or NULL (=1)
  const float* bias_rows;  // [videos, N] fp32 or NULL
  int rows_per_video;
  int num_videos;
  const __nv_bfloat16* bias;  // [N] or NULL
  int act;
  const float* rowdot_vec;  // [N] or NULL
  float* rowdot_out;        // [M, rowdot_nblk]
  int rowdot_nblk;
  __nv_bfloat16* Y;
  long long ldy;
  int m_blocks, n_blocks;
  // fused all-gather through the NVSwitch multicast mapping: when set, every output box is written ONCE with multimem.st to this
  // address (replicated by the switch into every rank's buffer, the local one included) and no TMA store is issued
  __nv_bfloat16* mc_out;
  // kVid (weight gradient over per-video segments, launch_gemm_tcgen05's `vid` argument): p.nseg videos share maps a[0] / b[0]; segment s
  // covers k-blocks [s * vid_kblocks, (s + 1) * vid_kblocks), is scaled by seg_scale[s * seg_scale_stride] when it is added to the
  // running sum, and its accumulator is ALSO dotted with dot_w [M, N]: dot_out[(s * tiles + tile) * EPI_WARPS + epilogue warp]
  int vid_kblocks;
  long long seg_scale_stride;
  const __nv_bfloat16* dot_w;
  long long dot_ldw;
  float* dot_out;
  // kVid split over the videos: a tile's videos are divided into vid_parts contiguous ranges, each range a separate work item whose
  // running sum goes to vid_partial [vid_parts, M, N] (fp32) instead of Y; folded afterwards in fixed order (fold_wgrad_parts_kernel).
  // 96 - 128 tiles leave 14 - 35 % of the 148 SMs idle for the whole launch; 288 - 1024 items of a third / an eighth of the work do not.
  int vid_parts;
  float* vid_partial;
  int num_out;   // destinations of every output tile: 1 (local) + peers' buffers over NVLink (fused all-gather)
  int out_flat;  // 1: Y is one contiguous [M, N] matrix (output map = [1, M, N]); 0: [videos, rows_per_video, N] with a batch stride
};

struct TensorMaps {
  CUtensorMap a[MERV_MAX_SEGMENTS];
  CUtensorMap b[MERV_MAX_SEGMENTS];
  // Y as [videos, rows_per_video, N] (batch stride may exceed rows_per_video * ldy), boxes of 128 x 32; out[0] is the local
  // destination, out[1..] the same rows of the peers' symmetric buffers (peer-mapped addresses)
  CUtensorMap out[MERV_MAX_ENCODERS];
};

// ---- the kernel -------------------------------------------------------------------------------------------
// kCtas == 1: one CTA per 128 x 256 tile.  kCtas == 2: a CTA pair (cluster 2x1, cta_group::2) per 256 x 256 tile — each CTA
// holds its 128 rows of A and HALF of the W tile, the leader's single thread issues UMMA 256x256x16 for both SMs, each
// CTA's TMEM receives its own 128 accumulator rows: per-SM shared-memory and L2->SM operand traffic drop by a third.
// kMn: the variant that honours MN-major operand flags (backward GEMMs).  It is a separate instantiation because the single producer /
// MMA threads run on 40 registers: the per-segment majorness selects cost the forward kernels 14 % when they were runtime branches.
// kMaj: operand majorness as a COMPILE-TIME value — bit 0: A is MN-major, bit 1: W is MN-major, the same for every segment.  As runtime
// flags the selects and the predicated second set of TMA issues made the producer's per-k-block instruction stream ~170 instructions
// long; a lone thread sustains roughly one instruction per 4 cycles, a k-block lasts ~560, and the CTA PAIR (whose two producers feed
// one MMA stream) ran 35 % SLOWER than the single CTA on MN-major operands — on K-major ones too when sent through that code
// (scripts/gpu_mn_pair_lab.py).
// kDy3 (kVid only): the A operand (dY, MN-major) is a 3-D map (N_out columns, token in video, video), so video b's rows may start at any
// 16-byte aligned batch stride — the gradient of a prefix slot inside the [B, L + T, N] multimodal embedding buffer, read in place.
template <int kCtas, bool kWide, bool kGelu, int kMaj, bool kVid = false, bool kDy3 = false>
__device__ __forceinline__ void gemm_body(const TensorMaps& maps, const GemmParams& p) {
  using C = Cfg<kCtas, kWide>;
  constexpr int STAGES = C::STAGES, STAGE_BYTES = C::STAGE_BYTES, RING_BYTES = C::RING_BYTES;
  constexpr int OUT_BOX_COLS = C::OUT_BOX_COLS, OUT_BOX_BYTES = C::OUT_BOX_BYTES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t tiles_addr = (raw_addr + 1023u) & ~1023u;  // SWIZZLE_128B atoms need 1024-byte alignment
  uint8_t* tiles = smem_raw + (tiles_addr - raw_addr);
  const uint32_t stage_out_addr = tiles_addr + RING_BYTES;  // 4 x 8 KB, 1024-byte aligned
  uint64_t* bars = reinterpret_cast<uint64_t*>(tiles + RING_BYTES + OUT_GROUPS * OUT_BOX_BYTES);
  const uint32_t full_bar = smem_u32(bars);                  // [STAGES]
  const uint32_t empty_bar = full_bar + 8 * STAGES;          // [STAGES]
  const uint32_t tfull_bar = empty_bar + 8 * STAGES;         // [2]
  const uint32_t tempty_bar = tfull_bar + 16;                // [2]
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = kCtas == 2 ? cluster_ctarank() : 0u;  // 0 = leader of the pair
  const int unit = kCtas == 2 ? int(blockIdx.x >> 1) : int(blockIdx.x);  // tile-processing unit: a CTA or a CTA pair
  const int num_units = int(gridDim.x) / kCtas;
  const int total_tiles = p.m_blocks * p.n_blocks;  // m_blocks counts (128 * kCtas)-row blocks
  const int total_items = kVid ? total_tiles * p.vid_parts : total_tiles;  // kVid: (tile, range of videos) work items
  // first segment of part q: all segments when the launch is not split; otherwise the videos in vid_parts near-equal contiguous ranges
  auto seg_first = [&](int q) { return kVid ? int(((long long)q * p.nseg) / p.vid_parts) : (q == 0 ? 0 : p.nseg); };

  if (warp == 0 && lane == 0) {
    // kVid: p.nseg counts videos, but every video reads the one map pair a[0] / b[0] (a and b hold only MERV_MAX_SEGMENTS maps)
    for (int s = 0; s < (kVid ? 1 : p.nseg); ++s) {
      prefetch_tmap(&maps.a[s]);
      prefetch_tmap(&maps.b[s]);
    }
    for (int d = 0; d < p.num_out; ++d) prefetch_tmap(&maps.out[d]);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(full_bar + 8 * i, 1);
      mbar_init(empty_bar + 8 * i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(tfull_bar + 8 * i, 1);
      mbar_init(tempty_bar + 8 * i, EPI_WARPS * kCtas);  // in a pair, both CTAs' epilogue warps arrive on the leader's barrier
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 2) {
    if constexpr (kCtas == 1) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "n"(TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    } else {  // the same warp of both CTAs, same destination offset
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "n"(TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  if constexpr (kCtas == 2) cluster_sync_all();  // the peer's barriers are initialised before anything remote touches them
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  // PDL: everything above touched only shared memory / TMEM and may have run while the previous kernel of the stream was
  // still finishing; from here on operands and per-video scales are read from global memory.
  pdl_wait();

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");  // 128 x 64 + 512 x 104 = 61440 = the whole launch-time allocation
    if (warp == 0 && (MERV_GEMM_WARP_UNIFORM || lane == 0)) {
      // ===== TMA producer (one elected lane issues; the loop itself is warp-uniform) =====
      uint32_t it = 0;
      const uint32_t leader_full = kCtas == 2 ? mapa_rank(full_bar, 0) : full_bar;
      for (int item = unit; item < total_items; item += num_units) {
        const int tile = kVid ? item % total_tiles : item, part = kVid ? item / total_tiles : 0;
        const int m_blk = tile / p.n_blocks, n_blk = tile % p.n_blocks;
        for (int s0 = seg_first(part); s0 < seg_first(part + 1); ++s0) {
          const int s = kVid ? 0 : s0;                       // kVid: every video reads the same pair of tensors ...
          const int nkb = kVid ? p.vid_kblocks : p.kblocks[s];
          const int kb_end = kVid ? (s0 + 1) * nkb : nkb;    // ... at its own k-blocks
          for (int kb = kVid ? s0 * nkb : 0; kb < kb_end; ++kb, ++it) {
            const uint32_t stage = it % STAGES, ph = (it / STAGES) & 1u;
            mbar_wait(empty_bar + 8 * stage, ph ^ 1u);  // own barrier: the pair's MMA commit is multicast to both CTAs
            const uint32_t sa = tiles_addr + stage * STAGE_BYTES;
            constexpr bool a_mn = (kMaj & 1) != 0, b_mn = (kMaj & 2) != 0;
            const int m0 = (m_blk * kCtas + int(rank)) * BM, n0 = n_blk * BN + int(rank) * C::B_ROWS;
            const uint32_t bar = (kCtas == 2 ? leader_full : full_bar) + 8 * stage;
            if (MERV_GEMM_WARP_UNIFORM && !elect_one()) continue;  // (the next wait re-converges the warp: elect.sync takes the full mask)
            // the leader's barrier counts the bytes of BOTH CTAs' loads; only the leader arrives on it
            if (kCtas == 1 || rank == 0) mbar_expect_tx(full_bar + 8 * stage, kCtas * STAGE_BYTES);
            auto load = [&](const CUtensorMap* map, uint32_t dst, int x, int y, uint64_t policy) {
              if constexpr (kCtas == 2) tma_load_2d_pair(map, bar, dst, x, y, policy);
              else tma_load_2d(map, bar, dst, x, y, policy);
            };
            // activations stream through once per wave of tiles; the weights are re-read by every M block, so they
            // are kept in L2 preferentially (for the 4096 x 16384 second MLP layer they barely fit: 134 of 126 MB)
            if (!a_mn) {
              load(&maps.a[s], sa, kb * BK, m0, L2_EVICT_NORMAL);
            } else if constexpr (kDy3) {  // video s0's k-block (a k-block never spans two videos) at its own batch stride
              const int t0 = (kb - s0 * nkb) * BK;
#pragma unroll
              for (int j = 0; j < BM / 64; ++j) {
                if constexpr (kCtas == 2) tma_load_3d_pair(&maps.a[s], bar, sa + j * MN_CHUNK_BYTES, m0 + 64 * j, t0, s0, L2_EVICT_NORMAL);
                else tma_load_3d(&maps.a[s], bar, sa + j * MN_CHUNK_BYTES, m0 + 64 * j, t0, s0, L2_EVICT_NORMAL);
              }
            } else {  // A given as [K, M]: one [64 m x BK k] box per 64 rows of the tile
#pragma unroll
              for (int j = 0; j < BM / 64; ++j) load(&maps.a[s], sa + j * MN_CHUNK_BYTES, m0 + 64 * j, kb * BK, L2_EVICT_NORMAL);
            }
            if (!b_mn) {
              load(&maps.b[s], sa + A_BYTES, kb * BK, n0, L2_EVICT_LAST);
            } else {
#pragma unroll
              for (int j = 0; j < C::B_ROWS / 64; ++j) load(&maps.b[s], sa + A_BYTES + j * MN_CHUNK_BYTES, n0 + 64 * j, kb * BK, L2_EVICT_LAST);
            }
          }
        }
      }
    } else if (warp == 1 && (MERV_GEMM_WARP_UNIFORM || lane == 0) && rank == 0) {
      // ===== MMA issuer (the leader CTA's elected lane drives both SMs of a pair; the loop is warp-uniform) =====
      uint32_t it = 0, acc_it = 0;
      for (int item = unit; item < total_items; item += num_units) {
        const int part = kVid ? item / total_tiles : 0;
        for (int s0 = seg_first(part); s0 < seg_first(part + 1); ++s0, ++acc_it) {
          const int s = kVid ? 0 : s0;
          constexpr bool a_mn = (kMaj & 1) != 0, b_mn = (kMaj & 2) != 0;
          const uint32_t idesc = umma_idesc_bf16(BM * kCtas, BN, a_mn, b_mn);
          // per UMMA (16 k): +32 bytes inside the swizzle atom for a K-major operand, +2 atoms of 8 k-rows for an MN-major one
          const uint32_t a_step = a_mn ? (2048u >> 4) : 2u, b_step = b_mn ? (2048u >> 4) : 2u;
          const uint32_t buf = acc_it & 1u, aph = (acc_it >> 1) & 1u;
          mbar_wait(tempty_bar + 8 * buf, aph ^ 1u);  // epilogue has drained this accumulator
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + buf * BN;
          const int nkb = kVid ? p.vid_kblocks : p.kblocks[s];
          for (int kb = 0; kb < nkb; ++kb, ++it) {
            const uint32_t stage = it % STAGES, ph = (it / STAGES) & 1u;
            mbar_wait(full_bar + 8 * stage, ph);
            tc_fence_after();
            const uint32_t sa = tiles_addr + stage * STAGE_BYTES;
            const uint64_t a_desc = a_mn ? umma_desc_mn_sw128(sa) : umma_desc_sw128(sa);
            const uint64_t b_desc = b_mn ? umma_desc_mn_sw128(sa + A_BYTES) : umma_desc_sw128(sa + A_BYTES);
            if (!MERV_GEMM_WARP_UNIFORM || elect_one()) {
#pragma unroll
              for (int k = 0; k < BK / UMMA_K; ++k) {
                if constexpr (kCtas == 2) umma_bf16_pair(d_tmem, a_desc + a_step * k, b_desc + b_step * k, idesc, (kb | k) != 0 ? 1u : 0u);
                else umma_bf16(d_tmem, a_desc + a_step * k, b_desc + b_step * k, idesc, (kb | k) != 0 ? 1u : 0u);
              }
              // frees the smem stage (in both CTAs of a pair) once these MMAs have read it
              if constexpr (kCtas == 2) umma_commit_pair(empty_bar + 8 * stage);
              else umma_commit(empty_bar + 8 * stage);
              // accumulator complete -> epilogue (of both CTAs): committed by the same lane, right behind the segment's last MMAs
              if (kb == nkb - 1) {
                if constexpr (kCtas == 2) umma_commit_pair(tfull_bar + 8 * buf);
                else umma_commit(tfull_bar + 8 * buf);
              }
            }
            if (MERV_GEMM_WARP_UNIFORM) __syncwarp();
          }
        }
      }
    }
  } else {
    // Register redistribution happens INSIDE the CTA's launch-time allocation (640 threads x 96 = 61440): warps 0-3 give
    // back 128 x (96 - 40) = 7168, so the 512 epilogue threads can grow by at most 14 each -> 104 (a larger request
    // would block forever in setmaxnreg.inc).
    asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
    // ===== epilogue =====
    const int q = warp & 3;          // TMEM lane quarter this warp may access
    const int h = (warp - 4) >> 2;   // column group of the tile: columns 64 h .. 64 h + 63
    uint32_t acc_it = 0;
    const uint32_t leader_tempty = kCtas == 2 ? mapa_rank(tempty_bar, 0) : tempty_bar;
    for (int item = unit; item < total_items; item += num_units) {
      const int tile = kVid ? item % total_tiles : item, part = kVid ? item / total_tiles : 0;
      const int m_blk = tile / p.n_blocks, n_blk = tile % p.n_blocks;
      const int m_base = (m_blk * kCtas + int(rank)) * BM;  // first output row of THIS CTA's half of the tile
      const int row = m_base + q * 32 + lane;
      int video = row / p.rows_per_video;
      if (video >= p.num_videos) video = p.num_videos - 1;
      // ---- finalize of one staged box: bias, activation, optional row-dot, bf16 pack; rows staged in shared memory
      //      (swizzled) and written with TMA stores: fully coalesced, asynchronous, M/N tails clipped by the tensor map ----
      const int col0 = n_blk * BN + h * EPI_COLS;
      const bool row_ok = row < p.M;
      float rd[8];  // 8 independent partial sums: no serial dependency chain through the 128 columns (zeroed right before the first pass)
      const uint32_t my_box = stage_out_addr + h * OUT_BOX_BYTES;
      const uint32_t my_row = my_box + uint32_t(q * 32 + lane) * uint32_t(OUT_BOX_COLS * 2);
      // 16-byte chunk index XOR address bits [7,..): SWIZZLE_64B (64-byte rows) -> (row >> 1) & 3; SWIZZLE_128B -> row & 7
      const uint32_t sw = kWide ? (uint32_t(lane) & 7u) : (uint32_t(lane >> 1) & 3u);
      constexpr int PASSES = EPI_COLS / OUT_BOX_COLS, CHUNKS = OUT_BOX_COLS / 8;
      const bool issuer = (warp == 4 + 4 * h) && lane == 0;
      auto emit_pass = [&](const int pass, const float* val) {  // val: this row's OUT_BOX_COLS accumulator values of the pass
        if (issuer) tma_store_wait_read();  // the previous store has finished reading this staging box
        named_bar_sync(1 + h, 128);
#pragma unroll
        for (int c8 = 0; c8 < CHUNKS; ++c8) {
          const int n = col0 + (pass * CHUNKS + c8) * 8;
          uint4 packed = make_uint4(0, 0, 0, 0);
          if (n < p.N) {  // N % 8 == 0 is enforced on the host
            float b[8];
            if (p.bias != nullptr) {
              Vec16<__nv_bfloat16>::unpack(__ldg(reinterpret_cast<const uint4*>(p.bias + n)), b);
            } else if (p.bias_rows != nullptr) {
              const float4* br = reinterpret_cast<const float4*>(p.bias_rows + (long long)video * p.N + n);
              const float4 b0 = __ldg(br), b1 = __ldg(br + 1);
              b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w; b[4] = b1.x; b[5] = b1.y; b[6] = b1.z; b[7] = b1.w;
            } else {
#pragma unroll
              for (int i = 0; i < 8; ++i) b[i] = 0.f;
            }
            float o[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = val[c8 * 8 + i] + b[i];
            if constexpr (kGelu) {  // compile-time: the un-activated kernels carry none of this (registers, code size)
#pragma unroll
              for (int i = 0; i < 8; i += 2) gelu_erf_fast2(o[i], o[i + 1]);
            }
            packed = Vec16<__nv_bfloat16>::pack(o);
            if (p.rowdot_vec != nullptr) {
              float r[8];
              Vec16<__nv_bfloat16>::unpack(packed, r);  // dot with the values as stored
              const float4* rv = reinterpret_cast<const float4*>(p.rowdot_vec + n);
              const float4 r0 = __ldg(rv), r1 = __ldg(rv + 1);
              rd[0] = fmaf(r[0], r0.x, rd[0]); rd[1] = fmaf(r[1], r0.y, rd[1]); rd[2] = fmaf(r[2], r0.z, rd[2]); rd[3] = fmaf(r[3], r0.w, rd[3]);
              rd[4] = fmaf(r[4], r1.x, rd[4]); rd[5] = fmaf(r[5], r1.y, rd[5]); rd[6] = fmaf(r[6], r1.z, rd[6]); rd[7] = fmaf(r[7], r1.w, rd[7]);
            }
          }
          sts_v4(my_row + ((uint32_t(c8) ^ sw) << 4), packed);
        }
        if (p.mc_out != nullptr) {
          // multicast all-gather: the group's 128 threads copy the staged box to the multicast address, 16 bytes each, a quarter
          // warp per 128-byte (64-byte) row: coalesced rows, conflict-free shared reads, ONE NVLink egress write per byte
          named_bar_sync(1 + h, 128);
          const int tg = (q * 32 + lane);
          const int colbase = col0 + pass * OUT_BOX_COLS;
#pragma unroll
          for (int i = 0; i < CHUNKS; ++i) {
            const int idx = i * 128 + tg;
            const int r = idx / CHUNKS, c = idx % CHUNKS;
            const uint32_t rsw = kWide ? (uint32_t(r) & 7u) : (uint32_t(r >> 1) & 3u);
            const uint4 v = lds_v4_g(my_box + uint32_t(r) * uint32_t(OUT_BOX_COLS * 2) + ((uint32_t(c) ^ rsw) << 4));
            if (m_base + r < p.M && colbase + c * 8 < p.N)
              multimem_st_v4(p.mc_out + (long long)(m_base + r) * p.ldy + colbase + c * 8, v);
          }
          return;  // the next pass's first barrier orders these shared reads before the box is overwritten
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the TMA engine
        named_bar_sync(1 + h, 128);
        if (issuer && col0 + pass * OUT_BOX_COLS < p.N) {
          const int m0 = m_base;
          const int v0 = p.out_flat ? 0 : m0 / p.rows_per_video;
          for (int d = 0; d < p.num_out; ++d)  // fused all-gather: the same box goes to every rank's buffer
            tma_store_3d(&maps.out[d], my_box, col0 + pass * OUT_BOX_COLS, m0 - v0 * p.rows_per_video, v0);
          tma_store_commit();
        }
      };
      auto release_accumulator = [&](const uint32_t buf) {  // the MMA issuer (in the leader CTA) may overwrite this TMEM buffer
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (kCtas == 2) mbar_arrive_cluster(leader_tempty + 8 * buf);
          else mbar_arrive(tempty_bar + 8 * buf);
        }
      };

      if constexpr (kGelu) {
        // activated GEMM (always one segment, no per-video scale): finalize straight out of TMEM, 32 columns at a time,
        // so only 32 accumulator values are live next to the packed-math constants of the GELU
        static_assert(!kGelu || (OUT_BOX_COLS == 32 && PASSES == 2), "one tcgen05.ld.x32 per staged box");
        const uint32_t buf = acc_it & 1u, aph = (acc_it >> 1) & 1u;
        ++acc_it;
        mbar_wait(tfull_bar + 8 * buf, aph);
        tc_fence_after();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + buf * BN + h * EPI_COLS;
#pragma unroll
        for (int i = 0; i < 8; ++i) rd[i] = 0.f;
#pragma unroll
        for (int pass = 0; pass < PASSES; ++pass) {
          uint32_t v[32];
          tmem_ld32(taddr + pass * 32, v);
          tmem_ld_wait();
          if (pass == PASSES - 1) release_accumulator(buf);
          float val[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) val[i] = __uint_as_float(v[i]);
          emit_pass(pass, val);
        }
      } else {
        float sum[EPI_COLS];
#pragma unroll
        for (int i = 0; i < EPI_COLS; ++i) sum[i] = 0.f;
        for (int s = seg_first(part); s < seg_first(part + 1); ++s, ++acc_it) {
          const uint32_t buf = acc_it & 1u, aph = (acc_it >> 1) & 1u;
          float scale = 1.0f;
          if constexpr (kVid) scale = p.seg_scale ? __ldg(p.seg_scale + (long long)s * p.seg_scale_stride) : 1.0f;
          else scale = p.seg_scale ? __ldg(p.seg_scale + (long long)video * p.nseg + s) : 1.0f;
          mbar_wait(tfull_bar + 8 * buf, aph);
          tc_fence_after();
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + buf * BN + h * EPI_COLS;
          if constexpr (kVid) {
            // per-video segment of a weight gradient: G = dY[video]^T X[video] sits in the accumulator.  It joins the running sum scaled by
            // the video's weight, and <W, G> — the gradient w.r.t. that weight — is taken from the same registers, 16 columns at a time
            const __nv_bfloat16* wrow = p.dot_w + (long long)(row_ok ? row : 0) * p.dot_ldw + col0;
            float dot = 0.f;
#pragma unroll
            for (int c = 0; c < EPI_COLS / 16; ++c) {
              uint4 w0 = make_uint4(0, 0, 0, 0), w1 = w0;
              if (row_ok && col0 + c * 16 < p.N) w0 = __ldg(reinterpret_cast<const uint4*>(wrow + c * 16));
              if (row_ok && col0 + c * 16 + 8 < p.N) w1 = __ldg(reinterpret_cast<const uint4*>(wrow + c * 16 + 8));
              uint32_t v[16];
              tmem_ld16(taddr + c * 16, v);
              tmem_ld_wait();
              float wf[16];
              Vec16<__nv_bfloat16>::unpack(w0, *reinterpret_cast<float(*)[8]>(wf));
              Vec16<__nv_bfloat16>::unpack(w1, *reinterpret_cast<float(*)[8]>(wf + 8));
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float a = __uint_as_float(v[i]);
                dot = fmaf(a, wf[i], dot);
                sum[c * 16 + i] = fmaf(scale, a, sum[c * 16 + i]);
              }
            }
            release_accumulator(buf);
            dot = warp_sum(dot);
            if (lane == 0) p.dot_out[(((long long)s * total_tiles + tile) * kCtas + int(rank)) * EPI_WARPS + (warp - 4)] = dot;
          } else {
#pragma unroll
          for (int c = 0; c < EPI_COLS / 32; ++c) {
            uint32_t v[32];
            tmem_ld32(taddr + c * 32, v);
            tmem_ld_wait();
            if (p.nseg == 1 && p.seg_scale == nullptr) {  // plain GEMM: the accumulator IS the result
#pragma unroll
              for (int i = 0; i < 32; ++i) sum[c * 32 + i] = __uint_as_float(v[i]);
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i) sum[c * 32 + i] = fmaf(scale, __uint_as_float(v[i]), sum[c * 32 + i]);
            }
          }
          release_accumulator(buf);
          }
        }
        if (kVid && p.vid_parts > 1) {
          // this item covered only `part` of the videos: fp32 partial tile, 64 contiguous columns per thread
          if (row_ok) {
            float* dst = p.vid_partial + ((long long)part * p.M + row) * p.N + col0;
#pragma unroll
            for (int c = 0; c < EPI_COLS; c += 4)
              if (col0 + c < p.N) *reinterpret_cast<float4*>(dst + c) = make_float4(sum[c], sum[c + 1], sum[c + 2], sum[c + 3]);
          }
          continue;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) rd[i] = 0.f;
#pragma unroll
        for (int pass = 0; pass < PASSES; ++pass) emit_pass(pass, sum + pass * OUT_BOX_COLS);
      }
      if (p.rowdot_vec != nullptr && row_ok && col0 < p.N)
        p.rowdot_out[(long long)row * p.rowdot_nblk + (col0 / MERV_ROWDOT_BLOCK)] = ((rd[0] + rd[1]) + (rd[2] + rd[3])) + ((rd[4] + rd[5]) + (rd[6] + rd[7]));
    }
    if (((warp - 4) & 3) == 0 && lane == 0) tma_store_wait_all();  // outstanding stores complete before the CTA retires
  }

  tc_fence_before();
  if constexpr (kCtas == 2) cluster_sync_all();  // the peer may still read this CTA's operands / arrive on its barriers
  else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if constexpr (kCtas == 1)
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
  }
}

template <int kCtas, bool kWide, bool kGelu, int kMaj = 0>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_tcgen05_kernel(const __grid_constant__ TensorMaps maps, const __grid_constant__ GemmParams p) {
  gemm_body<kCtas, kWide, kGelu, kMaj>(maps, p);
}

// weight gradient over per-video segments (single CTA, MN-major operands): dW = sum_b scale[b] dY[b]^T X[b] and <W, dY[b]^T X[b]> per video
template <int kCtas>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_wgrad_video_tcgen05_kernel(const __grid_constant__ TensorMaps maps, const __grid_constant__ GemmParams p) {
  gemm_body<kCtas, false, false, 3, true>(maps, p);
}

// the same with dY read through the 3-D (batch-strided) map: a separate kernel, so the contiguous one above keeps its code
template <int kCtas>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_wgrad_video_strided_tcgen05_kernel(const __grid_constant__ TensorMaps maps, const __grid_constant__ GemmParams p) {
  gemm_body<kCtas, false, false, 3, true, true>(maps, p);
}

// ---- host side ---------------------------------------------------------------------------------------------
// Which variant runs.  Round-2 measurements on B200 (65536 x 4096 bf16, 24 back-to-back calls from an idle GPU,
// scripts/gpu_gemm_lab.py -> profiles/r2_gemm_lab.json): the CTA pair wins everywhere — fused 4-segment K = 3584: 1.315 ms (1464 TFLOP/s)
// vs 1.377 (1398) for the single CTA; plain K = 1024: 0.424 (1297) vs 0.454 (1210); + GELU 0.452 vs 0.463; M = 262144, K = 768: 1.372 vs
// 1.378.  (Round 1 had the fused GEMM 2 % slower on the pair; that was measured inside long power-capped loops.)  cuBLAS on the same
// shapes: 1.225 / 0.402 / - / 1.265 ms.  MERV_GEMM_CTA_GROUP=1|2 overrides (read per call so the tests can run both).
// K-major operands: the pair wins at every shape measured with more than one row block (65536 x 1024 x 4096: 0.372 vs 0.410 ms; 65536 x
// 768 x 4096: 0.293 vs 0.338; the shapes above).  MN-major operands (the backward's dX = dY W and dW = dY^T X), with the majorness compiled
// in (kMaj; scripts/gpu_mn_pair_lab.py, profiles/r2b_mn_pair_lab.json): an MN-major W only (dX) — pair 0.384 vs single 0.410 ms; an
// MN-major A (dW, contraction over 65536 tokens) — single 0.398 vs pair 0.418; the per-video weight gradient — single 0.458 vs pair 0.461.
// (With RUNTIME majorness flags the pair took 0.50-0.54 ms on all of them: the producer's instruction stream was too long for one thread.)
static int gemm_cta_group(int M, bool a_mn_major) {
  const char* e = getenv("MERV_GEMM_CTA_GROUP");
  if (e != nullptr && e[0] == '1') return 1;
  if (e != nullptr && e[0] == '2') return 2;
  if (M <= BM) return 1;  // a pair computes 256 rows: with at most 128 rows its second CTA would only multiply padding
  return a_mn_major ? 1 : 2;
}

// 2-D bf16 row-major [rows, cols] (leading dimension ld elements) -> box [box_rows, box_cols] with 128-byte swizzle
static int make_tmap(CUtensorMap* map, const void* base, long long rows, long long cols, long long ld, int box_rows, int box_cols = BK) {
  const unsigned long long dims[2] = {(unsigned long long)cols, (unsigned long long)rows};
  const unsigned long long strides[1] = {(unsigned long long)ld * 2};
  const unsigned box[2] = {(unsigned)box_cols, (unsigned)box_rows};
  return encode_tmap_cached(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

template <auto kKernel, int kSmem>
static int launch_kernel(cudaLaunchConfig_t& cfg, const TensorMaps& maps, const GemmParams& p) {
  static const cudaError_t attr_rc =  // once per kernel (thread-safe static init)
      cudaFuncSetAttribute(kKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
  MERV_REQUIRE(attr_rc == cudaSuccess, MERV_E_CUDA, "cudaFuncSetAttribute(max dynamic smem=%d) failed: %s", kSmem, cudaGetErrorString(attr_rc));
  cfg.dynamicSmemBytes = kSmem;
  MERV_CUDA_OK(cudaLaunchKernelEx(&cfg, kKernel, maps, p));
  MERV_CUDA_OK(cudaGetLastError());
  return MERV_OK;
}

template <int kCtas, bool kWide, bool kGelu, int kMaj = 0>
static int launch_variant(cudaLaunchConfig_t& cfg, const TensorMaps& maps, const GemmParams& p) {
  return launch_kernel<gemm_bf16_tcgen05_kernel<kCtas, kWide, kGelu, kMaj>, Cfg<kCtas, kWide>::SMEM_BYTES>(cfg, maps, p);
}

static int wgrad_video_ctas(int M) { return gemm_cta_group(M, true); }
// partial dots per video: one per (tile, CTA of the tile's unit, epilogue warp)
int wgrad_video_parts(int M, int N) {
  const int ctas = wgrad_video_ctas(M);
  return ((M + BM * ctas - 1) / (BM * ctas)) * ctas * ((N + BN - 1) / BN) * EPI_WARPS;
}

// Split of a per-video weight gradient over the videos: with `tiles` tiles on `units` persistent CTAs (pairs), s work items per tile take
// ceil(tiles s / units) / s tile-times.  Measured (scripts/gpu_mn_pair_lab.py, profiles/r2b_mn_pair_lab.json): the fp32 round trip of the
// partial tiles and the extra pipeline ramps eat most of it — C = 768 (96 tiles, 64 videos) 0.465 -> 0.415 ms with 3 ranges (predicted
// 0.667x), C = 1024 (128 tiles) 0.443 -> 0.580 with 8 (predicted 0.875x), everything slower at 16 videos.  So: split only when the
// prediction is at least 30 % and there are at least 32 videos; the smallest s within 2 % of the best of {1..8} wins.
int wgrad_video_split(int M, int N, int videos) {
  if (const char* e = getenv("MERV_WGRAD_SPLIT")) {
    const int s = atoi(e);
    if (s >= 1) return s < videos ? s : (videos > 0 ? videos : 1);
  }
  const int ctas = wgrad_video_ctas(M);
  const long long tiles = (long long)((M + BM * ctas - 1) / (BM * ctas)) * ((N + BN - 1) / BN);
  const long long units = sm_count() / ctas;
  double best = 1e30;
  double cost[9];
  for (int s = 1; s <= 8; ++s) {
    cost[s] = s <= videos ? double((tiles * s + units - 1) / units) / s : 1e30;
    if (cost[s] < best) best = cost[s];
  }
  if (best > 0.70 * cost[1] || videos < 32) return 1;
  for (int s = 1; s <= 8; ++s)
    if (cost[s] <= 1.02 * best) return s;
  return 1;
}

int launch_gemm_tcgen05(const GemmSegment* seg, int nseg, const float* seg_scale, const float* bias_rows, int rows_per_video,
                        const void* bias, int act, const float* rowdot_vec, float* rowdot_out, void* Y, long long ldy, long long y_batch_stride,
                        int M, int N, int max_ctas, cudaStream_t stream, void* const* extra_out, int num_extra, bool pdl, void* mc_out,
                        const WgradVideoArgs* vid) {
  MERV_REQUIRE(nseg >= 1 && nseg <= MERV_MAX_SEGMENTS, MERV_E_ARG, "gemm: nseg=%d not in [1,%d]", nseg, MERV_MAX_SEGMENTS);
  MERV_REQUIRE(M > 0 && N > 0, MERV_E_SHAPE, "gemm: M=%d N=%d", M, N);
  MERV_REQUIRE(N % 8 == 0 && ldy % 8 == 0 && ldy >= N, MERV_E_ALIGN, "gemm: N=%d and ldy=%lld must be multiples of 8 (16-byte rows)", N, ldy);
  MERV_REQUIRE(aligned16(Y) && (bias == nullptr || aligned16(bias)) && (bias_rows == nullptr || aligned16(bias_rows)) &&
                   (rowdot_vec == nullptr || aligned16(rowdot_vec)),
               MERV_E_ALIGN, "gemm: Y / bias / rowdot_vec must be 16-byte aligned");
  MERV_REQUIRE(rows_per_video > 0, MERV_E_SHAPE, "gemm: rows_per_video=%d", rows_per_video);
  MERV_REQUIRE((rowdot_vec == nullptr) == (rowdot_out == nullptr), MERV_E_ARG, "gemm: rowdot_vec and rowdot_out go together");
  long long total_k = 0;
  for (int i = 0; i < nseg; ++i) total_k += seg[i].K;
  bool any_mn = false, a_mn_any = false;
  for (int i = 0; i < nseg; ++i) {
    any_mn = any_mn || seg[i].a_mn || seg[i].b_mn;
    a_mn_any = a_mn_any || seg[i].a_mn;
  }
  const int ctas = vid != nullptr ? wgrad_video_ctas(M) : gemm_cta_group(M, a_mn_any);
  // majorness is compiled into the kernel (kMaj): one choice per launch
  for (int i = 1; i < nseg; ++i)
    MERV_REQUIRE(seg[i].a_mn == seg[0].a_mn && seg[i].b_mn == seg[0].b_mn, MERV_E_ARG, "gemm: all segments of a launch share the operand majorness");
  if (vid != nullptr) {
    MERV_REQUIRE(nseg == 1 && seg[0].a_mn && seg[0].b_mn && act == MERV_ACT_NONE && num_extra == 0 && mc_out == nullptr &&
                     bias == nullptr && bias_rows == nullptr && rowdot_vec == nullptr && seg_scale == nullptr,
                 MERV_E_ARG, "gemm: the per-video weight gradient takes one MN-major segment and no epilogue options");
    MERV_REQUIRE(vid->videos >= 1 && vid->kblocks_per_video >= 1 && (long long)vid->videos * vid->kblocks_per_video * BK == seg[0].K, MERV_E_SHAPE,
                 "gemm: %d videos x %d k-blocks of %d do not cover K=%d", vid->videos, vid->kblocks_per_video, BK, seg[0].K);
    MERV_REQUIRE(vid->W && vid->dot_out && vid->ldw >= N && vid->ldw % 8 == 0 && aligned16(vid->W), MERV_E_ARG, "gemm: per-video weight gradient: W / dot_out");
  }
  // wide output boxes only pay when the kernel is NVLink-bound: with one peer (2 GPUs) it still is tensor-bound and the
  // ring stage given up for the staging costs more (2.05 vs 1.95 ms); from 2 peers on the link decides (3.15 vs 4.36 ms
  // at 4 GPUs).  MERV_GEMM_WIDE_OUT=0|1 overrides, for the tests.
  // multimem.st is packetised per contiguous run like the peer stores: measured at 2 GPUs, 64 videos each, the multicast gather takes
  // 2.15 ms with 128-byte rows and 2.75 ms with 64-byte rows (compute alone 1.71 ms) — so the multicast variant uses the wide boxes too
  bool wide = num_extra >= 2 || mc_out != nullptr;
  // ... and when the epilogue is the bottleneck: with a short contraction a tile's MMAs take less time than two staged passes through
  // the single staging box (the second pass waits for the first pass's TMA store to have read it).  One 128-byte-row pass per tile
  // instead: M = 262144, K = 768 (SigLIP single) on the pair 1199 -> 1283 TFLOP/s; at K = 1024 the ring stage given up costs more
  // (1374 -> 1350), at K = 3584 too (profiles/r2b_gemm_lab_wide.json)
  if (ctas == 2 && total_k <= 832 && !any_mn && vid == nullptr) wide = true;
  if (const char* e = getenv("MERV_GEMM_WIDE_OUT")) wide = e[0] == '1';
  MERV_REQUIRE(act == MERV_ACT_NONE || act == MERV_ACT_GELU_ERF, MERV_E_ARG, "gemm: unknown activation %d", act);
  if (act != MERV_ACT_NONE) {
    MERV_REQUIRE(nseg == 1 && seg_scale == nullptr, MERV_E_ARG, "gemm: an activation needs a single segment without per-video scales");
    MERV_REQUIRE(num_extra == 0 && mc_out == nullptr, MERV_E_ARG, "gemm: extra / multicast output destinations are only supported without an activation");
    wide = false;
  }
  const int out_box_cols = wide ? Cfg<1, true>::OUT_BOX_COLS : Cfg<1, false>::OUT_BOX_COLS;

  TensorMaps maps;
  GemmParams p = {};
  p.M = M; p.N = N; p.nseg = nseg;
  for (int s = 0; s < nseg; ++s) {
    const GemmSegment& g = seg[s];
    MERV_REQUIRE(g.A && g.W, MERV_E_ARG, "gemm: segment %d has a NULL operand", s);
    MERV_REQUIRE(g.K > 0 && g.lda % 8 == 0 && g.ldw % 8 == 0 && (g.K % 8 == 0 || (g.a_mn && g.b_mn)), MERV_E_ALIGN,
                 "gemm: segment %d: K=%d lda=%lld ldw=%lld: leading dimensions must be multiples of 8, and so must K unless both operands are MN-major",
                 s, g.K, g.lda, g.ldw);
    MERV_REQUIRE(aligned16(g.A) && aligned16(g.W), MERV_E_ALIGN, "gemm: segment %d: operands must be 16-byte aligned", s);
    // K-major: tensor [rows = M (N), cols = K], box [BM (BN / ctas) x BK].  MN-major: tensor [rows = K, cols = M (N)], box [BK x 64]
    if (g.a_mn) {
      MERV_REQUIRE(g.lda >= M, MERV_E_ALIGN, "gemm: segment %d: an MN-major A ([K, M]) needs lda >= M", s);
      if (int rc = make_tmap(&maps.a[s], g.A, g.K, M, g.lda, BK, 64)) return rc;
      p.a_mn_mask |= 1 << s;
    } else {
      MERV_REQUIRE(g.lda >= g.K, MERV_E_ALIGN, "gemm: segment %d: lda=%lld < K=%d", s, g.lda, g.K);
      if (int rc = make_tmap(&maps.a[s], g.A, M, g.K, g.lda, BM)) return rc;
    }
    if (g.b_mn) {
      MERV_REQUIRE(g.ldw >= N, MERV_E_ALIGN, "gemm: segment %d: an MN-major W ([K, N]) needs ldw >= N", s);
      if (int rc = make_tmap(&maps.b[s], g.W, g.K, N, g.ldw, BK, 64)) return rc;
      p.b_mn_mask |= 1 << s;
    } else {
      MERV_REQUIRE(g.ldw >= g.K, MERV_E_ALIGN, "gemm: segment %d: ldw=%lld < K=%d", s, g.ldw, g.K);
      if (int rc = make_tmap(&maps.b[s], g.W, N, g.K, g.ldw, BN / ctas)) return rc;  // a CTA of a pair loads half of the W tile
    }
    p.kblocks[s] = (g.K + BK - 1) / BK;  // the K tail is zero-filled by TMA
  }
  for (int s = nseg; s < MERV_MAX_SEGMENTS; ++s) { maps.a[s] = maps.a[0]; maps.b[s] = maps.b[0]; }
  {
    // output as a 3-D tensor (N, rows, videos): flat when the videos are back to back, otherwise one "video" per
    // batch-stride step (e.g. the prefix slot of a [B, 1 + T + L_text, N] multimodal embedding buffer, merv.py:633-640)
    const bool flat = y_batch_stride == 0 || y_batch_stride == (long long)rows_per_video * ldy;
    MERV_REQUIRE(flat || (rows_per_video % BM == 0 && y_batch_stride % 8 == 0 && y_batch_stride >= (long long)rows_per_video * ldy), MERV_E_SHAPE,
                 "gemm: a batch-strided output needs rows_per_video %% %d == 0 and a 16-byte aligned batch stride >= rows_per_video * ldo", BM);
    p.out_flat = flat ? 1 : 0;
    MERV_REQUIRE(mc_out == nullptr || (flat && num_extra == 0 && aligned16(mc_out)), MERV_E_ARG,
                 "gemm: the multicast output needs a flat [M, N] destination, no unicast peers and a 16-byte aligned address");
    p.mc_out = static_cast<__nv_bfloat16*>(mc_out);
    const unsigned long long dims[3] = {(unsigned long long)N, (unsigned long long)(flat ? M : rows_per_video), (unsigned long long)(flat ? 1 : (M / rows_per_video))};
    const unsigned long long strides[2] = {(unsigned long long)ldy * 2, (unsigned long long)(flat ? (long long)M * ldy : y_batch_stride) * 2};
    const unsigned box[3] = {(unsigned)out_box_cols, BM, 1};
    MERV_REQUIRE(num_extra >= 0 && num_extra < MERV_MAX_ENCODERS && (num_extra == 0 || extra_out != nullptr), MERV_E_ARG,
                 "gemm: %d extra output destinations (at most %d)", num_extra, MERV_MAX_ENCODERS - 1);
    p.num_out = 1 + num_extra;
    for (int d = 0; d < p.num_out; ++d) {
      void* base = d == 0 ? Y : extra_out[d - 1];
      MERV_REQUIRE(base != nullptr && aligned16(base), MERV_E_ALIGN, "gemm: output destination %d is NULL or not 16-byte aligned", d);
      if (int rc = encode_tmap_cached(&maps.out[d], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, strides, box,
                                      wide ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B))
        return rc;
    }
    for (int d = p.num_out; d < MERV_MAX_ENCODERS; ++d) maps.out[d] = maps.out[0];
  }
  p.seg_scale = seg_scale; p.bias_rows = bias_rows; p.rows_per_video = rows_per_video;
  p.num_videos = (M + rows_per_video - 1) / rows_per_video;
  p.bias = static_cast<const __nv_bfloat16*>(bias); p.act = act;
  p.rowdot_vec = rowdot_vec; p.rowdot_out = rowdot_out; p.rowdot_nblk = (N + MERV_ROWDOT_BLOCK - 1) / MERV_ROWDOT_BLOCK;
  p.Y = static_cast<__nv_bfloat16*>(Y); p.ldy = ldy;
  p.m_blocks = (M + BM * ctas - 1) / (BM * ctas); p.n_blocks = (N + BN - 1) / BN;
  if (vid != nullptr) {
    p.nseg = vid->videos; p.vid_kblocks = vid->kblocks_per_video;
    p.seg_scale = vid->scale; p.seg_scale_stride = vid->scale_stride;
    p.dot_w = static_cast<const __nv_bfloat16*>(vid->W); p.dot_ldw = vid->ldw; p.dot_out = vid->dot_out;
    MERV_REQUIRE(vid->split >= 1 && vid->split <= vid->videos && (vid->split == 1 || (vid->partial != nullptr && aligned16(vid->partial) && N % 4 == 0)), MERV_E_ARG,
                 "gemm: per-video weight gradient: split=%d of %d videos needs a 16-byte aligned partial buffer", vid->split, vid->videos);
    p.vid_parts = vid->split; p.vid_partial = vid->partial;
    if (vid->dy_batch_stride != 0) {  // dY as (N_out columns, token in video, video); same [64 x BK] boxes and swizzle as the 2-D map
      const long long tpv = (long long)vid->kblocks_per_video * BK;
      MERV_REQUIRE(vid->dy_batch_stride % 8 == 0 && vid->dy_batch_stride >= tpv * seg[0].lda, MERV_E_SHAPE,
                   "gemm: per-video weight gradient: dY batch stride %lld must be a multiple of 8 and >= %lld", vid->dy_batch_stride, tpv * seg[0].lda);
      const unsigned long long dims[3] = {(unsigned long long)M, (unsigned long long)tpv, (unsigned long long)vid->videos};
      const unsigned long long strides[2] = {(unsigned long long)seg[0].lda * 2, (unsigned long long)vid->dy_batch_stride * 2};
      const unsigned box[3] = {64u, (unsigned)BK, 1u};
      if (int rc = encode_tmap_cached(&maps.a[0], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, seg[0].A, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
      for (int s = 1; s < MERV_MAX_SEGMENTS; ++s) maps.a[s] = maps.a[0];
    }
  }
  const long long total = (long long)p.m_blocks * p.n_blocks * (vid != nullptr ? vid->split : 1);
  int sms = sm_count();
  if (max_ctas > 0 && max_ctas < sms) sms = max_ctas;
  long long units = sms / ctas;  // persistent: one CTA (or CTA pair) per SM (pair)
  if (units > total) units = total;
  if (units < 1) units = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(unsigned(units * ctas));
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = unsigned(ctas);
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 2 : 1;
  if (vid != nullptr) {
    constexpr int smem1 = Cfg<1, false>::SMEM_BYTES, smem2 = Cfg<2, false>::SMEM_BYTES;
    if (vid->dy_batch_stride != 0)
      return ctas == 2 ? launch_kernel<gemm_wgrad_video_strided_tcgen05_kernel<2>, smem2>(cfg, maps, p)
                       : launch_kernel<gemm_wgrad_video_strided_tcgen05_kernel<1>, smem1>(cfg, maps, p);
    return ctas == 2 ? launch_kernel<gemm_wgrad_video_tcgen05_kernel<2>, smem2>(cfg, maps, p)
                     : launch_kernel<gemm_wgrad_video_tcgen05_kernel<1>, smem1>(cfg, maps, p);
  }
  if (p.a_mn_mask | p.b_mn_mask) {
    MERV_REQUIRE(act == MERV_ACT_NONE && !wide, MERV_E_ARG, "gemm: MN-major operands are supported without an activation and without extra output destinations");
    const int maj = (p.a_mn_mask ? 1 : 0) | (p.b_mn_mask ? 2 : 0);
    if (ctas == 2)
      return maj == 3 ? launch_variant<2, false, false, 3>(cfg, maps, p) : maj == 2 ? launch_variant<2, false, false, 2>(cfg, maps, p)
                                                                                     : launch_variant<2, false, false, 1>(cfg, maps, p);
    return maj == 3 ? launch_variant<1, false, false, 3>(cfg, maps, p) : maj == 2 ? launch_variant<1, false, false, 2>(cfg, maps, p)
                                                                                   : launch_variant<1, false, false, 1>(cfg, maps, p);
  }
  if (act == MERV_ACT_GELU_ERF) return ctas == 2 ? launch_variant<2, false, true>(cfg, maps, p) : launch_variant<1, false, true>(cfg, maps, p);
  if (ctas == 2) return wide ? launch_variant<2, true, false>(cfg, maps, p) : launch_variant<2, false, false>(cfg, maps, p);
  return wide ? launch_variant<1, true, false>(cfg, maps, p) : launch_variant<1, false, false>(cfg, maps, p);
}

}  // namespace merv
