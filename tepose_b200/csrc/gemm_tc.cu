// K1 -- GRU input projection on the 5th-gen tensor cores:  out = A . W^T + bias
// (replaces the input GEMM inside cuDNN's GRU / the x.W_ih^T half of torch.nn.GRU,
// reference lib/models/tepose.py:53-64,73,76).
//
//   * operands bf16, K-major, moved by TMA (cp.async.bulk.tensor, 128-byte swizzle) into a
//     5/6-stage shared-memory ring guarded by mbarriers;
//   * one elected thread issues tcgen05.mma (cta_group::1, M=128, N=BN, K=16) with the fp32
//     accumulator in TMEM;
//   * PERSISTENT CTAs (one per SM) walk the tile list with a stride of gridDim.x, and the accumulator is DOUBLE-BUFFERED in
//     TMEM (2 x BN columns): while the four epilogue warps read tile i back with tcgen05.ld, add the bias and store it, the
//     producer and the MMA thread are already deep in tile i+1.  The one-tile-per-CTA version of this kernel had its tensor
//     pipe busy 43 % of the time: TMEM allocation, the first TMA round trip and the whole epilogue were exposed once per tile.
// Tiles that share a W tile are adjacent in the tile order, so the W tile is fetched from HBM once and re-served from L2.
#include "common.cuh"
#include "umma.cuh"
#include <cuda.h>

namespace tp {

// Tile 128 x BN, BN = 192 or 128 (chosen per launch): every k-step a CTA pulls (128 + BN) x 64 bf16 through the L2 -> SM path
// (the kernel's bound, see the note at k_gemm_bf16_tc2), so a wider tile raises the MACs per byte; BN = 192 also turns the 2.92 waves of the B=32,T=16 input projection (432 tiles
// of 128 x 128) into 1.95 (288 tiles).  Skinny launches (one wave or less of 128-wide tiles, e.g. the B = 1 live window)
// stay at BN = 128: they stream weights and want more CTAs.
constexpr int TC_BM = 128, TC_BK = 64;
template <int BN> struct TcCfg {
  static_assert(BN % 32 == 0 && BN >= 32 && BN <= 256, "UMMA N / epilogue chunking");
  static constexpr int A_BYTES = TC_BM * TC_BK * 2;                   // the A block of a k-step: 16 KB
  static constexpr int STAGE_BYTES = A_BYTES + BN * TC_BK * 2;        // 40 KB at 192, 32 KB at 128
  static constexpr int STAGES = (200 * 1024) / STAGE_BYTES;           // 5 / 6
  static constexpr int TMEM_COLS = 2 * BN <= 256 ? 256 : 512;         // two accumulators
  static constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
};
constexpr int TC_MAX_SEGS = 8;
constexpr int TC_THREADS = 192;       // warp 0: TMA producer, warp 1: MMA issuer, warps 2..5: epilogue (TMEM lane groups 2, 3, 0, 1)

struct TcParams {
  tp_gemm_seg seg[TC_MAX_SEGS];
  int tile_begin[TC_MAX_SEGS + 1];
  int nseg, kblocks;
};

struct TcTile { tp_gemm_seg sg; int m0, n0; };
template <int BN>
__device__ __forceinline__ TcTile tc_decode(const TcParams& p, int tile) {
  int s = 0;
#pragma unroll
  for (int q = 1; q < TC_MAX_SEGS; ++q)
    if (q < p.nseg && tile >= p.tile_begin[q]) s = q;
  // static-index select: a dynamic index into the kernel parameters costs a constant-cache miss per field
  TcTile t;
  t.sg = p.seg[0];
  int tile0 = p.tile_begin[0];
#pragma unroll
  for (int q = 1; q < TC_MAX_SEGS; ++q)
    if (q == s) { t.sg = p.seg[q]; tile0 = p.tile_begin[q]; }
  const int local = tile - tile0;
  const int m_tiles = (t.sg.m_rows + TC_BM - 1) / TC_BM;
  const int n_tile = local / m_tiles, m_tile = local - n_tile * m_tiles;
  t.m0 = m_tile * TC_BM; t.n0 = n_tile * BN;            // segment-local
  return t;
}

template <int BN>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_gemm_bf16_tc(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w, const TcParams p) {
  using Cfg = TcCfg<BN>;
  constexpr int TC_STAGES = Cfg::STAGES, TC_STAGE_BYTES = Cfg::STAGE_BYTES;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // carve: [stages][A 16KB | W] (1024-aligned), then barriers
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + TC_STAGES * TC_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + TC_STAGES;
  uint64_t* tmem_full_bar = empty_bar + TC_STAGES;      // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;         // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
  __shared__ float s_bias[2][BN];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total = p.tile_begin[TC_MAX_SEGS];

  if (threadIdx.x == 0) {
    for (int i = 0; i < TC_STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full_bar[i], 1); mbar_init(&tmem_empty_bar[i], 4); }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(reinterpret_cast<uint64_t>(&map_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(reinterpret_cast<uint64_t>(&map_w)) : "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)Cfg::TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::);
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  // PDL: barriers, TMEM and the tensor maps were set up while the producer of A (the pack kernel) was still running
  pdl_wait();
  pdl_launch_dependents();

  if (warp == 0) {
    if (elect_one()) {  // ===== TMA producer: runs ahead of the MMAs by the ring depth, across tile boundaries =====
      int it = 0;
      for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const TcTile t = tc_decode<BN>(p, tile);
        for (int kb = 0; kb < p.kblocks; ++kb, ++it) {
          const int st = it % TC_STAGES;
          const uint32_t ph = (it / TC_STAGES) & 1;
          mbar_wait(&empty_bar[st], ph ^ 1);
          unsigned char* a_dst = smem + st * TC_STAGE_BYTES;
          mbar_expect_tx(&full_bar[st], (uint32_t)TC_STAGE_BYTES);
          tma_load_2d(a_dst, &map_a, &full_bar[st], kb * TC_BK, t.sg.m_start + t.m0);
          tma_load_2d(a_dst + Cfg::A_BYTES, &map_w, &full_bar[st], kb * TC_BK, t.sg.n_start + t.n0);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (elect_one()) {  // ===== MMA issuer =====
      int it = 0, i = 0;
      for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++i) {
        const int acc = i & 1;
        mbar_wait(&tmem_empty_bar[acc], ((i >> 1) & 1) ^ 1);     // the epilogue has drained this accumulator (two tiles ago)
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        for (int kb = 0; kb < p.kblocks; ++kb, ++it) {
          const int st = it % TC_STAGES;
          const uint32_t ph = (it / TC_STAGES) & 1;
          mbar_wait(&full_bar[st], ph);
          asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
          const uint32_t a_addr = smem_u32(smem + st * TC_STAGE_BYTES);
          const uint64_t da = umma_desc_sw128(a_addr), db = umma_desc_sw128(a_addr + Cfg::A_BYTES);
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k)    // advance 16 elements (32 B) along K inside the 128-byte swizzle row: +2 in 16-byte units
            umma_f16(tmem_base + (uint32_t)(acc * BN), da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), Cfg::IDESC, (kb | k) != 0 ? 1u : 0u);
          umma_commit(&empty_bar[st]);            // slot reusable once these MMAs have read it
        }
        umma_commit(&tmem_full_bar[acc]);         // accumulator complete
      }
    }
    __syncwarp();
  } else {
    // ===== epilogue: warps 2..5; a warp may only touch the TMEM lanes 32 (warp % 4) .. +31 =====
    const int lg = warp & 3, et = threadIdx.x - 64;     // lane group, index among the 128 epilogue threads
    int i = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++i) {
      const TcTile t = tc_decode<BN>(p, tile);
      const int acc = i & 1;
      // bias of this tile's columns -> shared memory (two buffers: the previous tile's readers may still be in flight)
      for (int c = et; c < BN; c += 128) s_bias[acc][c] = (t.sg.bias && t.n0 + c < t.sg.n_cols) ? t.sg.bias[t.n0 + c] : 0.0f;
      asm volatile("bar.sync 1, 128;\n" ::: "memory");
      mbar_wait(&tmem_full_bar[acc], (i >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
      const int row = t.m0 + lg * 32 + lane;             // segment-local output row of this thread (= its TMEM lane)
      const bool row_ok = row < t.sg.m_rows;
      const bool relu = (t.sg.flags & TP_GEMM_RELU) != 0, out_lp = (t.sg.flags & TP_GEMM_OUT_BF16) != 0;
      const bool vec_ok = ((t.sg.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(t.sg.out) & 15) == 0);
      float* orow = t.sg.out + (int64_t)row * t.sg.ldc + t.n0;
      __nv_bfloat16* orow_lp = reinterpret_cast<__nv_bfloat16*>(t.sg.out) + (int64_t)row * t.sg.ldc + t.n0;
      const __nv_bfloat16* rrow = t.sg.residual ? reinterpret_cast<const __nv_bfloat16*>(t.sg.residual) + (int64_t)row * t.sg.ldr + t.n0 : nullptr;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(acc * BN + c0), v);
        asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
        if (row_ok) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {                   // 8 columns at a time
            const int n = t.n0 + c0 + q * 8;
            if (n >= t.sg.n_cols) break;
            float o[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) o[u] = __uint_as_float(v[q * 8 + u]) + s_bias[acc][c0 + q * 8 + u];
            const bool full = n + 7 < t.sg.n_cols;
            if (rrow && full) {
              const uint4 rv = *reinterpret_cast<const uint4*>(rrow + c0 + q * 8);
              const __nv_bfloat162* rh = reinterpret_cast<const __nv_bfloat162*>(&rv);
#pragma unroll
              for (int u = 0; u < 4; ++u) { const float2 f = __bfloat1622float2(rh[u]); o[2 * u] += f.x; o[2 * u + 1] += f.y; }
            } else if (rrow) {
              for (int u = 0; u < 8; ++u)
                if (n + u < t.sg.n_cols) o[u] += __bfloat162float(rrow[c0 + q * 8 + u]);
            }
            if (relu) {
#pragma unroll
              for (int u = 0; u < 8; ++u) o[u] = fmaxf(o[u], 0.0f);
            }
            if (out_lp) {
              if (full) {
                __nv_bfloat162 h[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) h[u] = __floats2bfloat162_rn(o[2 * u], o[2 * u + 1]);
                *reinterpret_cast<uint4*>(orow_lp + c0 + q * 8) = *reinterpret_cast<const uint4*>(h);
              } else {
                for (int u = 0; u < 8; ++u)
                  if (n + u < t.sg.n_cols) orow_lp[c0 + q * 8 + u] = __float2bfloat16_rn(o[u]);
              }
            } else if (full && vec_ok) {
              *reinterpret_cast<float4*>(orow + c0 + q * 8) = make_float4(o[0], o[1], o[2], o[3]);      // a thread writes 128 contiguous bytes of its row per chunk
              *reinterpret_cast<float4*>(orow + c0 + q * 8 + 4) = make_float4(o[4], o[5], o[6], o[7]);
            } else {
              for (int u = 0; u < 8; ++u)
                if (n + u < t.sg.n_cols) orow[c0 + q * 8 + u] = o[u];
            }
          }
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(&tmem_empty_bar[acc])) : "memory");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS));
  }
}

// ---------------------------------------------------------------------------------------------------------------------------
// CTA-PAIR variant (tcgen05.mma.cta_group::2, M = 256) -- OPT-IN (TP_TC_2CTA=1): measured 47 us against the 43 us of the
// one-CTA kernel above on the B=32,T=16 input projection.
// What bounds the one-CTA kernel (ncu, profiles/): tensor pipe 49 % active, DRAM 29 %, and 5.4 TB/s leaving the L2 towards the
// SMs averaged over the whole kernel (200 MB: the L2 merges concurrent requests for the same line, the CTAs ask for 392 MB) --
// the L2 -> SM side runs at the ~6.9 TB/s scripts/micro/l2bw.cu measures as its ceiling while the mainloop is active.  Neither
// multicasting the shared operand inside a cluster of 2 (no change: the merging already did that) nor a contiguous, pre-swizzled
// copy of W fetched with plain bulk copies (no change: HBM is not the limit) moved it.  A CTA pair computes a 256 x 256 tile with
// each CTA holding its own 128 rows of A and only HALF of the W tile -- the tensor core reads the other half out of the peer's
// shared memory -- 0.60x the operand bytes per MAC; the pair's cross-CTA barrier hops and the 120 pair tiles on 74 pairs (1.62
// waves, the 32-row segment wasting half of its pair tiles) cost more than that saves at this size.
//   * both CTAs run a TMA producer (own A rows, own half of W); every load completes the LEADER's full barrier
//     (cp.async.bulk.tensor ... cta_group::2), and only the leader issues the MMAs;
//   * tcgen05.commit multicasts to both CTAs' empty barriers (a slot is free in BOTH rings once the pair's MMAs have read
//     it) and to both CTAs' accumulator-full barriers; the epilogue warps of both CTAs drain their own 128 TMEM lanes and
//     arrive on the leader's accumulator-empty barrier (8 arrivals);
//   * persistent pairs, double-buffered accumulator (2 x 256 TMEM columns), as above.
constexpr int TC2_BN = 256, TC2_STAGE_BYTES = TC_BM * TC_BK * 2 + (TC2_BN / 2) * TC_BK * 2, TC2_STAGES = 6;
constexpr uint32_t TC2_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TC2_BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);

struct Tc2Params {
  tp_gemm_seg seg[TC_MAX_SEGS];
  int tile_begin[TC_MAX_SEGS + 1];     // in pair tiles (256 x 256)
  int nseg, kblocks;
};

__device__ __forceinline__ TcTile tc2_decode(const Tc2Params& p, int tile) {
  int s = 0;
#pragma unroll
  for (int q = 1; q < TC_MAX_SEGS; ++q)
    if (q < p.nseg && tile >= p.tile_begin[q]) s = q;
  TcTile t;
  t.sg = p.seg[0];
  int tile0 = p.tile_begin[0];
#pragma unroll
  for (int q = 1; q < TC_MAX_SEGS; ++q)
    if (q == s) { t.sg = p.seg[q]; tile0 = p.tile_begin[q]; }
  const int local = tile - tile0;
  const int m_pairs = (t.sg.m_rows + 2 * TC_BM - 1) / (2 * TC_BM);
  const int n_tile = local / m_pairs, m_pair = local - n_tile * m_pairs;
  t.m0 = m_pair * 2 * TC_BM; t.n0 = n_tile * TC2_BN;
  return t;
}

__device__ __forceinline__ uint32_t tc2_map(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void tc2_tma_load(void* smem_dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::
          "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc2_umma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc2_commit(uint64_t* bar) {      // arrives on the barrier at this offset in BOTH CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n" ::
                   "r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}

__global__ void __launch_bounds__(TC_THREADS, 1)
k_gemm_bf16_tc2(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w, const Tc2Params p) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + TC2_STAGES * TC2_STAGE_BYTES);     // used in the leader
  uint64_t* empty_bar = full_bar + TC2_STAGES;                                              // per CTA
  uint64_t* tmem_full_bar = empty_bar + TC2_STAGES;      // [2], per CTA
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;          // [2], used in the leader: 8 arrivals (4 epilogue warps x 2 CTAs)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
  __shared__ float s_bias[2][TC2_BN];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t rank;
  asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(rank));
  const int total = p.tile_begin[TC_MAX_SEGS];
  const int pair_id = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  constexpr int A_BYTES = TC_BM * TC_BK * 2;

  if (threadIdx.x == 0) {
    for (int i = 0; i < TC2_STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full_bar[i], 1); mbar_init(&tmem_empty_bar[i], 8); }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(reinterpret_cast<uint64_t>(&map_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(reinterpret_cast<uint64_t>(&map_w)) : "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n" ::);
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  pdl_launch_dependents();

  if (warp == 0) {
    if (elect_one()) {  // ===== TMA producer (both CTAs): own 128 rows of A, own half of the W tile; completion on the LEADER's barrier =====
      int it = 0;
      for (int tile = pair_id; tile < total; tile += n_pairs) {
        const TcTile t = tc2_decode(p, tile);
        for (int kb = 0; kb < p.kblocks; ++kb, ++it) {
          const int st = it % TC2_STAGES;
          const uint32_t ph = (it / TC2_STAGES) & 1;
          mbar_wait(&empty_bar[st], ph ^ 1);
          unsigned char* a_dst = smem + st * TC2_STAGE_BYTES;
          if (rank == 0) mbar_expect_tx(&full_bar[st], (uint32_t)(2 * TC2_STAGE_BYTES));
          const uint32_t lead_bar = tc2_map(smem_u32(&full_bar[st]), 0);
          tc2_tma_load(a_dst, &map_a, lead_bar, kb * TC_BK, t.sg.m_start + t.m0 + (int)rank * TC_BM);
          tc2_tma_load(a_dst + A_BYTES, &map_w, lead_bar, kb * TC_BK, t.sg.n_start + t.n0 + (int)rank * (TC2_BN / 2));
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (rank == 0 && elect_one()) {  // ===== MMA issuer: the leader CTA only =====
      int it = 0, i = 0;
      for (int tile = pair_id; tile < total; tile += n_pairs, ++i) {
        const int acc = i & 1;
        mbar_wait(&tmem_empty_bar[acc], ((i >> 1) & 1) ^ 1);     // both CTAs' epilogues have drained this accumulator
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        for (int kb = 0; kb < p.kblocks; ++kb, ++it) {
          const int st = it % TC2_STAGES;
          const uint32_t ph = (it / TC2_STAGES) & 1;
          mbar_wait(&full_bar[st], ph);
          asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
          const uint32_t a_addr = smem_u32(smem + st * TC2_STAGE_BYTES);
          const uint64_t da = umma_desc_sw128(a_addr), db = umma_desc_sw128(a_addr + A_BYTES);
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k)
            tc2_umma(tmem_base + (uint32_t)(acc * TC2_BN), da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), TC2_IDESC, (kb | k) != 0 ? 1u : 0u);
          tc2_commit(&empty_bar[st]);
        }
        tc2_commit(&tmem_full_bar[acc]);
      }
    }
    __syncwarp();
  } else {
    // ===== epilogue (both CTAs): warps 2..5, TMEM lane group = warp % 4; this CTA's rows are m0 + 128 rank + lane group * 32 + lane =====
    const int lg = warp & 3, et = threadIdx.x - 64;
    const uint32_t lead_empty0 = tc2_map(smem_u32(&tmem_empty_bar[0]), 0);
    int i = 0;
    for (int tile = pair_id; tile < total; tile += n_pairs, ++i) {
      const TcTile t = tc2_decode(p, tile);
      const int acc = i & 1;
      for (int c = et; c < TC2_BN; c += 128) s_bias[acc][c] = (t.sg.bias && t.n0 + c < t.sg.n_cols) ? t.sg.bias[t.n0 + c] : 0.0f;
      asm volatile("bar.sync 1, 128;\n" ::: "memory");
      mbar_wait(&tmem_full_bar[acc], (i >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
      const int row = t.m0 + (int)rank * TC_BM + lg * 32 + lane;
      const bool row_ok = row < t.sg.m_rows;
      const bool relu = (t.sg.flags & TP_GEMM_RELU) != 0, out_lp = (t.sg.flags & TP_GEMM_OUT_BF16) != 0;
      const bool vec_ok = ((t.sg.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(t.sg.out) & 15) == 0);
      float* orow = t.sg.out + (int64_t)row * t.sg.ldc + t.n0;
      __nv_bfloat16* orow_lp = reinterpret_cast<__nv_bfloat16*>(t.sg.out) + (int64_t)row * t.sg.ldc + t.n0;
      const __nv_bfloat16* rrow = t.sg.residual ? reinterpret_cast<const __nv_bfloat16*>(t.sg.residual) + (int64_t)row * t.sg.ldr + t.n0 : nullptr;
#pragma unroll 1
      for (int c0 = 0; c0 < TC2_BN; c0 += 32) {
        if (t.n0 + c0 >= t.sg.n_cols) break;             // (warp-uniform) nothing left in this tile's ragged tail
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(acc * TC2_BN + c0), v);
        asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
        if (row_ok) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int n = t.n0 + c0 + q * 8;
            if (n >= t.sg.n_cols) break;
            float o[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) o[u] = __uint_as_float(v[q * 8 + u]) + s_bias[acc][c0 + q * 8 + u];
            const bool full = n + 7 < t.sg.n_cols;
            if (rrow) {
              for (int u = 0; u < 8; ++u)
                if (n + u < t.sg.n_cols) o[u] += __bfloat162float(rrow[c0 + q * 8 + u]);
            }
            if (relu) {
#pragma unroll
              for (int u = 0; u < 8; ++u) o[u] = fmaxf(o[u], 0.0f);
            }
            if (out_lp) {
              for (int u = 0; u < 8; ++u)
                if (n + u < t.sg.n_cols) orow_lp[c0 + q * 8 + u] = __float2bfloat16_rn(o[u]);
            } else if (full && vec_ok) {
              *reinterpret_cast<float4*>(orow + c0 + q * 8) = make_float4(o[0], o[1], o[2], o[3]);
              *reinterpret_cast<float4*>(orow + c0 + q * 8 + 4) = make_float4(o[4], o[5], o[6], o[7]);
            } else {
              for (int u = 0; u < 8; ++u)
                if (n + u < t.sg.n_cols) orow[c0 + q * 8 + u] = o[u];
            }
          }
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];\n" ::"r"(lead_empty0 + 8u * acc) : "memory");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(512u));
  }
}

// ---- host side: tensor maps through the driver entry point (no libcuda link dependency)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  }
  return fn;
}

static int make_map(CUtensorMap* map, const void* base, int rows, int kp, int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail(TP_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)kp, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)kp * 2};
  cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(TP_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return TP_OK;
}

}  // namespace tp

using namespace tp;

extern "C" int tp_gemm_bf16_tc(const void* A, int a_rows, const void* W, int w_rows, int kp,
                               const tp_gemm_seg* segs, int nseg, void* stream) {
  TP_CHECK_ARG(A && W && segs, "tp_gemm_bf16_tc: null pointer");
  TP_CHECK_ARG(nseg >= 1 && nseg <= TC_MAX_SEGS, "tp_gemm_bf16_tc: nseg=%d out of range", nseg);
  TP_CHECK_ARG(kp > 0 && kp % TC_BK == 0, "tp_gemm_bf16_tc: kp=%d must be a positive multiple of %d", kp, TC_BK);
  TP_CHECK_ARG(a_rows > 0 && w_rows > 0, "tp_gemm_bf16_tc: empty operand");
  TP_CHECK_ARG(aligned16(A) && aligned16(W), "tp_gemm_bf16_tc: operands must be 16-byte aligned");
  int dev = 0, major = 0;
  TP_CUDA(cudaGetDevice(&dev));
  TP_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) return fail(TP_ERR_UNSUPPORTED, "tp_gemm_bf16_tc needs an sm_100 device (found sm_%d)", major);
  TcParams p;
  memset(&p, 0, sizeof(p));
  p.nseg = nseg;
  p.kblocks = kp / TC_BK;
  // tile width: once the launch has more than one wave of 128 x 128 tiles, tiles get wider (192: more MACs per operand byte, and
  // 1.95 instead of 2.92 waves at the B=32,T=16 input projection); skinny launches stay at 128 x 128: they stream weights and want CTAs.
  int tiles128 = 0;
  for (int i = 0; i < nseg; ++i) tiles128 += (int)(ceil_div(segs[i].m_rows, TC_BM) * ceil_div(segs[i].n_cols, 128));
  static const int bn_env = getenv("TP_TC_BN") ? atoi(getenv("TP_TC_BN")) : 0;
  const int bn = bn_env == 128 || bn_env == 192 ? bn_env : (tiles128 > sm_count() ? 192 : 128);
  int tiles = 0;
  for (int i = 0; i < nseg; ++i) {
    const tp_gemm_seg& sg = segs[i];
    TP_CHECK_ARG(sg.out && sg.m_rows > 0 && sg.n_cols > 0, "tp_gemm_bf16_tc: segment %d is empty / has no output", i);
    TP_CHECK_ARG(sg.m_start >= 0 && sg.m_start + sg.m_rows <= a_rows, "tp_gemm_bf16_tc: segment %d rows out of range", i);
    TP_CHECK_ARG(sg.n_start >= 0 && sg.n_start + sg.n_cols <= w_rows, "tp_gemm_bf16_tc: segment %d cols out of range", i);
    TP_CHECK_ARG(sg.n_cols % 16 == 0, "tp_gemm_bf16_tc: segment %d: n_cols=%d must be a multiple of 16", i, sg.n_cols);
    TP_CHECK_ARG(!(sg.flags & TP_GEMM_OUT_BF16) || (sg.ldc % 8 == 0 && aligned16(sg.out)), "tp_gemm_bf16_tc: segment %d: bf16 output needs ldc %% 8 == 0 and 16-byte alignment", i);
    TP_CHECK_ARG(!sg.residual || (sg.ldr % 8 == 0 && aligned16(sg.residual)), "tp_gemm_bf16_tc: segment %d: residual needs ldr %% 8 == 0 and 16-byte alignment", i);
    p.seg[i] = sg;
    p.tile_begin[i] = tiles;
    tiles += (int)(ceil_div(sg.m_rows, TC_BM) * ceil_div(sg.n_cols, bn));
  }
  for (int i = nseg; i <= TC_MAX_SEGS; ++i) p.tile_begin[i] = tiles;
  CUtensorMap map_a, map_w;
  int rc = make_map(&map_a, A, a_rows, kp, TC_BM);
  if (rc != TP_OK) return rc;
  rc = make_map(&map_w, W, w_rows, kp, bn);
  if (rc != TP_OK) return rc;
  static const bool use_2cta = getenv("TP_TC_2CTA") != nullptr;
  if (use_2cta && tiles128 > sm_count() && kp % TC_BK == 0) {
    // CTA pairs on 256 x 256 tiles (k_gemm_bf16_tc2): measured 47 us against 43 us on the B=32,T=16 input projection -- opt-in
    Tc2Params q;
    memset(&q, 0, sizeof(q));
    q.nseg = nseg; q.kblocks = kp / TC_BK;
    int ptiles = 0;
    for (int i = 0; i < nseg; ++i) {
      q.seg[i] = segs[i];
      q.tile_begin[i] = ptiles;
      ptiles += (int)(ceil_div(segs[i].m_rows, 2 * TC_BM) * ceil_div(segs[i].n_cols, TC2_BN));
    }
    for (int i = nseg; i <= TC_MAX_SEGS; ++i) q.tile_begin[i] = ptiles;
    CUtensorMap map_w2;
    rc = make_map(&map_w2, W, w_rows, kp, TC2_BN / 2);
    if (rc != TP_OK) return rc;
    const size_t smem = (size_t)TC2_STAGES * TC2_STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
    TP_CUDA(cudaFuncSetAttribute(k_gemm_bf16_tc2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int pairs = ptiles < sm_count() / 2 ? ptiles : sm_count() / 2;
    PdlConfig lc(dim3((unsigned)(2 * pairs)), dim3(TC_THREADS), smem, (cudaStream_t)stream);
    cudaLaunchAttribute at[2];
    at[0] = lc.attr[0];
    at[1].id = cudaLaunchAttributeClusterDimension;
    at[1].val.clusterDim.x = 2; at[1].val.clusterDim.y = 1; at[1].val.clusterDim.z = 1;
    lc.cfg.attrs = at; lc.cfg.numAttrs = 2;
    TP_CUDA(cudaLaunchKernelEx(&lc.cfg, k_gemm_bf16_tc2, map_a, map_w2, q));
    TP_LAUNCH_CHECK();
    return TP_OK;
  }
  const int grid = tiles < sm_count() ? tiles : sm_count();      // persistent: CTA c takes tiles c, c + grid, ...
  if (bn == 192) {
    using Cfg = TcCfg<192>;
    const size_t smem = (size_t)Cfg::STAGES * Cfg::STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
    TP_CUDA(cudaFuncSetAttribute(k_gemm_bf16_tc<192>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    PdlConfig lc(dim3((unsigned)grid), dim3(TC_THREADS), smem, (cudaStream_t)stream);
    TP_CUDA(cudaLaunchKernelEx(&lc.cfg, k_gemm_bf16_tc<192>, map_a, map_w, p));
  } else {
    using Cfg = TcCfg<128>;
    const size_t smem = (size_t)Cfg::STAGES * Cfg::STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
    TP_CUDA(cudaFuncSetAttribute(k_gemm_bf16_tc<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    PdlConfig lc(dim3((unsigned)grid), dim3(TC_THREADS), smem, (cudaStream_t)stream);
    TP_CUDA(cudaLaunchKernelEx(&lc.cfg, k_gemm_bf16_tc<128>, map_a, map_w, p));
  }
  TP_LAUNCH_CHECK();
  return TP_OK;
}
