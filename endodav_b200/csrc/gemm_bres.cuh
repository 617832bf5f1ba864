// B-RESIDENT tcgen05 GEMM for the short-K linears of the ViT-S encoder (qkv, fc1: K = D = 384) and the motion modules:
//
//   C[M,N] = A[M,K] * W[N,K]^T (+ bias, GELU | ReLU), 16-bit output         K <= 384, K % 64 == 0, N % BN == 0
//
// Why: with K = 384 the streaming kernel (gemm_tc.cuh) re-fetches BOTH operands from L2 for every 128 x BN output
// tile -- 40-48 KB per 64-wide k-block for 384-512 cycles of tensor work, i.e. 70-100 B/cycle/SM, ~20 TB/s over the
// chip.  Its in-kernel timeline (tools/gemm_timeline.py) shows k-blocks arriving every ~590 cycles against 384
// cycles of MMA: the mainloop waits for the L2 -> shared-memory traffic, not for the tensor core.  The weights are
// the small operand (BN x K x 2 B = 144 KB for BN = 192), so here a CTA keeps ITS n-tile of W in shared memory for
// the whole kernel and streams only A: 16 KB per k-block (42 B/cycle/SM at full MMA rate), 2.5x less L2 traffic.
//
//   CTA c  ->  n-tile  c % n_tiles;  m-tiles  c / n_tiles, + group size, ...   (persistent, one CTA per SM)
//   warp 0       TMA producer: the n-tile of W once (K/64 boxes), then the A k-blocks of its m-tiles through a ring
//   warp 1       TMEM allocator + MMA issuer (warp-uniform loop, elected lane; two accumulator buffers)
//   warps 4..19  four epilogue warpgroups, ALL of them on every tile (columns [wg * BN/4, +BN/4)): thread = row,
//                16-column steps: tcgen05.ld -> bias / GELU / ReLU -> 16-bit -> swizzled shared-memory sub-tile -> TMA
//                store: gemm_tc's TMA-store epilogue (gt_epilogue_tma) with ONE 4 KB staging sub-tile per warpgroup, as
//                shared memory is full -- 144 KB W + 64 KB A ring + 16 KB staging
#pragma once
#include "gemm_tc.cuh"

namespace tc {

constexpr int GB_THREADS = 640;
constexpr int GB_A_STAGE = GT_BM * 128;   // one 128 x 64 16-bit k-block of A
constexpr int GB_PF_TILES = 2;            // A tiles prefetched into L2 ahead of the ring

template <int BN> constexpr uint32_t gb_tmem_cols() { return 2 * BN <= 256 ? 256 : 512; }

template <typename T, int BN>
__global__ void __launch_bounds__(GB_THREADS, 1) gemm_bres_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                  const __grid_constant__ CUtensorMap tmB,
                                                                  const __grid_constant__ CUtensorMap tmC, Epi e, int M, int K,
                                                                  int stages, int n_tiles, int m_tiles) {
  pdl_launch();   // PDL: the next kernel of the stream may start its prologue (common.cuh)
  constexpr uint32_t B_KB_BYTES = BN * 128;                 // one 64-wide k-block of the resident W tile
  constexpr uint32_t TMEM_COLS = gb_tmem_cols<BN>();
  constexpr int CW = BN / 4;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int kblocks = K / 64;
  unsigned char* sB = smem;                                              // kblocks x BN x 128 B
  unsigned char* sA = sB + (size_t)kblocks * B_KB_BYTES;                 // stages x 16 KB
  unsigned char* stg = sA + (size_t)stages * GB_A_STAGE;                 // 4 warpgroups x 4 KB
  float* bias_base = reinterpret_cast<float*>(stg + 4 * GT_OUT_SUB_BYTES);   // 4 warpgroups x 64 floats
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(bias_base + 4 * 64);
  uint64_t* empty_bar = full_bar + stages;
  uint64_t* b_full = empty_bar + stages;      // 1: the resident W tile has landed
  uint64_t* tfull_bar = b_full + 1;           // 2
  uint64_t* tempty_bar = tfull_bar + 2;       // 2
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  // Warp roles by VIRTUAL warp id: the SM's issue arbiter favours the highest warp ids of a sub-partition, so the two
  // latency-critical single-lane roles (TMA producer, MMA issuer) take physical warps 16 / 17 and the sixteen epilogue
  // warps physical warps 0..15 (with the roles on warps 0 / 1 the issuer starved behind four busy epilogue warps of
  // its sub-partition: k-blocks were issued every 575-800 cycles against 384 cycles of tensor work).  The TMEM lane
  // quarter of an epilogue warp is warp % 4 either way.
  const int pwarp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int warp = pwarp >= 16 ? pwarp - 16 : pwarp + 4;
  // optional in-kernel timeline, same slot table as gemm_tc_kernel (tools/gemm_timeline.py)
  long long* tm_ = (e.tim && blockIdx.x < 4) ? e.tim + blockIdx.x * 256 : nullptr;
  if (tm_ && threadIdx.x == 0) tm_[0] = clock64();
  // this CTA's n-tile and its share of the m-tiles
  const int tile_n = blockIdx.x % n_tiles;
  const int grp = blockIdx.x / n_tiles;
  const int grp_size = ((int)gridDim.x - tile_n + n_tiles - 1) / n_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmC);
    for (int s = 0; s < stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(b_full, 1);
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], 512);
    }
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  // PDL: everything above ran under the previous kernel's tail; its results are visible after pdl_wait().  The producer
  // first issues the loads of its resident W tile -- weights are never written inside a forward -- so that up to 144 KB
  // of L2 -> shared-memory traffic also travels under the previous kernel's tail.
  if (warp != 0) pdl_wait();
  if (tm_ && threadIdx.x == 0) tm_[1] = clock64();

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(b_full, (uint32_t)kblocks * B_KB_BYTES);
      for (int kb = 0; kb < kblocks; ++kb) tma_load_2d(sB + (size_t)kb * B_KB_BYTES, &tmB, b_full, kb * 64, tile_n * BN);
    }
    pdl_wait();
    if (lane == 0) {
      uint32_t kc = 0;
      int ti = 0;
      // L2 prefetch distance: GB_PF_TILES m-tiles of A ahead of the shared-memory ring (tc_common.cuh tma_prefetch_2d)
      for (int p = 0; p < GB_PF_TILES; ++p) {
        const int tp = grp + p * grp_size;
        if (tp < m_tiles)
          for (int kb = 0; kb < kblocks; ++kb) tma_prefetch_2d(&tmA, kb * 64, tp * GT_BM);
      }
      for (int tm = grp; tm < m_tiles; tm += grp_size, ++ti) {
        const int tp = tm + GB_PF_TILES * grp_size;
        if (tp < m_tiles)
          for (int kb = 0; kb < kblocks; ++kb) tma_prefetch_2d(&tmA, kb * 64, tp * GT_BM);
        for (int kb = 0; kb < kblocks; ++kb, ++kc) {
          const int s = kc % stages;
          mbar_wait(&empty_bar[s], ((kc / stages) & 1) ^ 1);
          mbar_expect_tx(&full_bar[s], GB_A_STAGE);
          tma_load_2d(sA + (size_t)s * GB_A_STAGE, &tmA, &full_bar[s], kb * 64, tm * GT_BM);
        }
        if (tm_ && ti < 20) tm_[100 + ti] = clock64();
      }
    }
  } else if (warp == 1) {
    const uint32_t leader = elect_one_sync();
    const uint32_t sa_addr = smem_u32(sA), sb_addr = smem_u32(sB);
    const auto ab = [&](int s, int kb) { return make_uint2(sa_addr + s * GB_A_STAGE, sb_addr + kb * B_KB_BYTES); };
    mbar_wait(b_full, 0);
    fence_after_sync();
    uint32_t kc = 0, it = 0;
    for (int tm = grp; tm < m_tiles; tm += grp_size, ++it) {
      const uint32_t b = it & 1;
      mma_tile<T, BN, 64>(leader, tmem_base + b * BN, &tempty_bar[b], &tfull_bar[b], full_bar, empty_bar, stages, kblocks, kc, it, ab, tm_);
    }
  } else if (warp >= 4) {
    const int wg = (warp - 4) >> 2;
    const int q = warp & 3;
    const int r = q * 32 + lane;
    unsigned char* stg_wg = stg + wg * GT_OUT_SUB_BYTES;
    float* bias_s = bias_base + wg * 64;
    const int kind = e.kind & ~EF_TMA_OUT;
    if ((kind & EF_BIAS) && q == 0) {
      // the n-tile is fixed: this warpgroup's bias slice is staged once
      for (int i = lane; i < CW; i += 32) bias_s[i] = __ldg(e.bias + tile_n * BN + wg * CW + i);
    }
    wg_bar_sync(1 + wg);
    uint32_t it = 0;
    for (int tm = grp; tm < m_tiles; tm += grp_size, ++it) {
      const uint32_t b = it & 1;
      mbar_wait(&tfull_bar[b], (it >> 1) & 1);
      fence_after_sync();
      const bool stamp = tm_ && wg == 0 && q == 0 && lane == 0 && it < 20;
      if (stamp) tm_[10 + 4 * it] = clock64();
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + b * BN + wg * CW;
      const int row0 = tm * GT_BM, col0 = tile_n * BN + wg * CW;
      switch (kind) {
#define EDV_TMA_CASE(F_) case F_: gt_epilogue_tma<T, BN, F_, 1>(&tmC, trow, row0, col0, r, wg, stg_wg, bias_s, &tempty_bar[b], nullptr); break;
        EDV_EPI_TMA_KINDS(EDV_TMA_CASE)
#undef EDV_TMA_CASE
        default: __builtin_unreachable();   // EF_TMA_OUT is set for these kinds only (gemm_tma_out_ok)
      }
      if (stamp) tm_[11 + 4 * it] = clock64();
    }
    if (q == 0) {
      if (elect_one_sync()) tma_store_wait_all();   // shared memory stays valid until the last store has read it
      __syncwarp();
    }
  }
  __syncthreads();
  if (warp == 1) {
    fence_after_sync();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

}  // namespace tc
