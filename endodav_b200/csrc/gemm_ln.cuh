// Row-owning tcgen05 GEMM with fused residual add and LayerNorm for the ViT-S encoder (D = 384):
//
//   x[m, :]  += A[m, :] W^T + bias                (fp32 residual stream, in place;  LayerScale is folded into W / bias)
//   xn[m, :]  = LayerNorm(x[m, :]; gamma, beta)   (16-bit operand of the NEXT GEMM: norm2 -> fc1, or the next block's norm1 -> qkv)
//
// Replaces `x = x + ls(attn.proj(...))` / `x = x + ls(mlp.fc2(...))` followed by the next `norm` (layers/block.py:110-116,
// 143-145): the separate LayerNorm kernel (24 launches per ViT-S forward) re-read the fp32 stream that had just been
// written.  Both ops are HBM-bound (proj: 590 KB per 128-row tile against ~6 000 cycles of tensor work).
//
// A CLUSTER OF TWO CTAs owns a 128-row tile: CTA `rank` computes columns [192 rank, +192) (one N = 192 accumulator, so
// TWO accumulator buffers fit in TMEM and the epilogue of tile i runs under the mainloop of tile i+1 -- a single CTA
// with the whole 384-column row in TMEM has to alternate mainloop and epilogue, and with all CTAs in lockstep HBM
// idles during the mainloops: measured 108 us for fc2 + norm against 101 us unfused).  The LayerNorm statistics of
// a row are combined across the pair through distributed shared memory:
//   pass 1  acc + bias + residual -> x (fp32; residual sub-tiles by TMA load, result back through the same staging
//           buffer + TMA store), x kept in TMEM (tcgen05.st), half-row sum        -> half-row mean
//   pass 2  centred sum of squares of the half row (from TMEM)
//   exchange (sum, M2) of the half row -> peer CTA (st.shared::cluster + remote mbarrier arrive); Chan's
//           combination gives the full-row mean / variance with two-pass accuracy
//   pass 3  (x - mean) * rstd * gamma + beta -> 16 bit -> TMA store of xn
// thread = row, warpgroup wg = columns [48 wg, +48) of the half, 16-column steps; pass 3 stages and stores each step
// with the steps of gemm_tc.cuh's TMA-store epilogue (pack16, stage_store16).
//
//   warp 16 (virtual 0)   TMA producer: A k-block (128 x 64) + this CTA's 192 rows of the W k-block, 3-stage ring,
//                         A L2-prefetched a few k-blocks ahead
//   warp 17 (virtual 1)   TMEM allocator + MMA issuer (warp-uniform loop, elected lane)
//   warps 0..15           four epilogue warpgroups
#pragma once
#include "gemm_tc.cuh"

namespace tc {

constexpr int GL_N = 384;
constexpr int GL_HN = 192;                             // columns per CTA of the pair
constexpr int GL_THREADS = 640;
constexpr int GL_STAGES = 3;
constexpr uint32_t GL_A_BYTES = GT_BM * 128;           // 128 x 64 16-bit
constexpr uint32_t GL_B_BYTES = GL_HN * 128;           // 192 x 64 16-bit
constexpr uint32_t GL_STAGE_BYTES = GL_A_BYTES + GL_B_BYTES;   // 40 KB
constexpr int GL_CW = GL_HN / 4;                       // 48 columns per warpgroup
constexpr int GL_NSUB = GL_CW / 16;                    // 3
constexpr uint32_t GL_RES_BYTES = GT_BM * 16 * 4;      // fp32 residual sub-tile: 128 rows x 64 B (SWIZZLE_64B)
constexpr size_t GL_SMEM = 1024 + (size_t)GL_STAGES * GL_STAGE_BYTES + 4 * 2 * GL_RES_BYTES + 4 * GT_OUT_SUB_BYTES + 4 * GT_BM * 8 +
                           2 * GT_BM * 8 + 3 * GL_HN * 4 + 256;

__device__ __forceinline__ void tmem_st16_f(uint32_t taddr, const float* v) {
  uint32_t r[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) r[i] = __float_as_uint(v[i]);
  tmem_st16(taddr, r);
}
__device__ __forceinline__ void epi_bar_sync_all() { asm volatile("bar.sync 5, 512;" ::: "memory"); }
// address of the same shared-memory location in the cluster's CTA `rank`
__device__ __forceinline__ uint32_t map_to_cta(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_cluster_f2(uint32_t addr, float a, float b) {
  asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0, polls = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (++polls > (1u << 28)) __trap();
  }
}

template <typename T>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GL_THREADS, 1)
    gemm_ln_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmXn, const float* __restrict__ bias,
                   const float* __restrict__ gamma, const float* __restrict__ beta, float eps, int M, int K, int m_tiles, int do_ln,
                   long long* __restrict__ tim) {
  pdl_launch();   // PDL: the next kernel of the stream may start its prologue (common.cuh)
  // tim: optional timeline of cluster 0's even CTA: per tile i < 8, slots [8i..8i+7] = residual loads issued, accumulator
  // complete, pass 1 done, mean known, pass 2 done, peer statistics in, pass 3 done (clock64)
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* ring = smem;
  unsigned char* res = ring + (size_t)GL_STAGES * GL_STAGE_BYTES;        // [wg][2] x 8 KB
  unsigned char* xns = res + 4 * 2 * GL_RES_BYTES;                       // [wg] x 4 KB
  float2* part = reinterpret_cast<float2*>(xns + 4 * GT_OUT_SUB_BYTES);  // [wg][128] partial statistics of the half row
  float2* mail = part + 4 * GT_BM;                                       // [2][128] the PEER's half-row (sum, M2), by tile parity
  float* sbias = reinterpret_cast<float*>(mail + 2 * GT_BM);             // 192 each: this CTA's columns
  float* sgamma = sbias + GL_HN;
  float* sbeta = sgamma + GL_HN;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sbeta + GL_HN);
  uint64_t* empty_bar = full_bar + GL_STAGES;
  uint64_t* tfull_bar = empty_bar + GL_STAGES;    // 2
  uint64_t* tempty_bar = tfull_bar + 2;           // 2 (512 arrivals)
  uint64_t* res_full = tempty_bar + 2;            // [wg][2]
  uint64_t* mail_bar = res_full + 8;              // 2 (128 remote arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mail_bar + 2);

  const int pwarp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int warp = pwarp >= 16 ? pwarp - 16 : pwarp + 4;    // virtual warp id: roles as in gemm_bres.cuh
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int col_half = (int)rank * GL_HN;
  const int kblocks = K / 64;

  for (int i = threadIdx.x; i < GL_HN; i += GL_THREADS) {
    sbias[i] = bias ? bias[col_half + i] : 0.f;
    sgamma[i] = do_ln ? gamma[col_half + i] : 1.f;
    sbeta[i] = do_ln ? beta[col_half + i] : 0.f;
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmXn);
    for (int s = 0; s < GL_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], 512);
      mbar_init(&mail_bar[b], GT_BM);
    }
    for (int i = 0; i < 8; ++i) mbar_init(&res_full[i], 1);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  fence_before_sync();
  cluster_sync_all();                       // both CTAs' barriers exist before any remote arrive
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();     // PDL: everything above ran under the previous kernel's tail; its results are visible from here

  if (warp == 0) {
    if (lane == 0) {
      uint32_t kc = 0;
      for (int tile = pair; tile < m_tiles; tile += npairs) {
        for (int kb = 0; kb < kblocks; ++kb, ++kc) {
          const int s = kc % GL_STAGES;
          // L2 prefetch of the A k-block a few steps ahead (this tile or the head of the next one); the even CTA
          // prefetches for the pair
          if (rank == 0) {
            int pk = kb + 6, pt = tile;
            if (pk >= kblocks) { pk -= kblocks; pt += npairs; }
            if (pk < kblocks && pt < m_tiles) tma_prefetch_2d(&tmA, pk * 64, pt * GT_BM);
          }
          mbar_wait(&empty_bar[s], ((kc / GL_STAGES) & 1) ^ 1);
          unsigned char* st = ring + (size_t)s * GL_STAGE_BYTES;
          mbar_expect_tx(&full_bar[s], GL_STAGE_BYTES);
          tma_load_2d(st, &tmA, &full_bar[s], kb * 64, tile * GT_BM);
          tma_load_2d(st + GL_A_BYTES, &tmB, &full_bar[s], kb * 64, col_half);
        }
      }
    }
  } else if (warp == 1) {
    const uint32_t leader = elect_one_sync();
    const uint32_t ring_addr = smem_u32(ring);
    const auto ab = [&](int s, int) {
      const uint32_t sa = ring_addr + s * GL_STAGE_BYTES;
      return make_uint2(sa, sa + GL_A_BYTES);
    };
    uint32_t kc = 0, it = 0;
    for (int tile = pair; tile < m_tiles; tile += npairs, ++it) {
      const uint32_t b = it & 1;
      mma_tile<T, GL_HN, 64>(leader, tmem_base + b * GL_HN, &tempty_bar[b], &tfull_bar[b], full_bar, empty_bar, GL_STAGES, kblocks, kc, it, ab,
                             nullptr);
    }
  } else if (warp >= 4) {
    // Epilogue, thread = row.  (Direct 128-bit global loads / stores in this row-owner pattern -- 64 contiguous bytes
    // per thread and step -- were tried and are 2x SLOWER than staging through shared memory + TMA: every warp-level
    // instruction touches 32 different sectors half-used, which the L2 / LSU path handles badly.)
    const int wg = (warp - 4) >> 2;
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const bool w0 = (q == 0);                                   // warp 0 of the warpgroup issues its TMA traffic
    unsigned char* res_wg = res + wg * (2 * GL_RES_BYTES);
    unsigned char* xn_wg = xns + wg * GT_OUT_SUB_BYTES;
    uint64_t* rfull = res_full + wg * 2;
    const int sw64 = (r >> 1) & 3;                              // SWIZZLE_64B (fp32 sub-tiles, 64-byte rows)
    const int col_wg = wg * GL_CW;                              // within this CTA's half
    const int gcol_wg = col_half + col_wg;                      // global column
    const uint32_t peer_mail = map_to_cta(mail, rank ^ 1);
    const uint32_t peer_bar = map_to_cta(mail_bar, rank ^ 1);
    uint32_t nuse0 = 0, nuse1 = 0;                              // uses of each residual buffer so far (barrier phases)
    uint32_t it = 0;
    long long* tm_ = (tim && blockIdx.x == 0 && wg == 0 && r == 0) ? tim : nullptr;
    for (int tile = pair; tile < m_tiles; tile += npairs, ++it) {
      const uint32_t b = it & 1;
      const int row0 = tile * GT_BM;
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + b * GL_HN + col_wg;
      // Residual sub-tiles: the first two of a tile are loaded right after pass 1 of the PREVIOUS tile (below), i.e.
      // they travel while passes 2 / 3 and the next mainloop run; only the very first tile loads them here.  All three
      // sub-tiles of the next tile are L2-prefetched now, so the third (loaded when its buffer frees up) is an L2 hit.
      if (w0) {
        if (elect_one_sync()) {
          if (it == 0) {
            for (int s = 0; s < 2; ++s) {
              mbar_expect_tx(&rfull[s], GL_RES_BYTES);
              tma_load_2d(res_wg + s * GL_RES_BYTES, &tmX, &rfull[s], gcol_wg + 16 * s, row0);
            }
            tma_prefetch_2d(&tmX, gcol_wg + 32, row0);
          }
          if (tile + npairs < m_tiles)
            for (int s = 0; s < GL_NSUB; ++s) tma_prefetch_2d(&tmX, gcol_wg + 16 * s, (tile + npairs) * GT_BM);
        }
        __syncwarp();
      }
      if (tm_ && it < 8) tm_[8 * it + 0] = clock64();
      mbar_wait(&tfull_bar[b], (it >> 1) & 1);
      fence_after_sync();
      if (tm_ && it < 8) tm_[8 * it + 1] = clock64();
      // ---- pass 1: x = acc + bias + residual -> global (TMA store) and back into TMEM; half-row sum ----
      float sum = 0.f;
#pragma unroll 1
      for (int s = 0; s < GL_NSUB; ++s) {
        float v[16];
        tmem_ld16(trow + 16 * s, v);
        if (s & 1) mbar_wait(&rfull[1], nuse1++ & 1);
        else mbar_wait(&rfull[0], nuse0++ & 1);
        unsigned char* rowp = res_wg + (s & 1) * GL_RES_BYTES + r * 64;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float4* p = reinterpret_cast<float4*>(rowp + ((j ^ sw64) << 4));
          const float4 xo = *p;
          const float4 bb = *reinterpret_cast<const float4*>(sbias + col_wg + 16 * s + 4 * j);
          v[4 * j + 0] += bb.x + xo.x;
          v[4 * j + 1] += bb.y + xo.y;
          v[4 * j + 2] += bb.z + xo.z;
          v[4 * j + 3] += bb.w + xo.w;
          *p = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          sum += (v[4 * j] + v[4 * j + 1]) + (v[4 * j + 2] + v[4 * j + 3]);
        }
        if (do_ln) tmem_st16_f(trow + 16 * s, v);
        fence_proxy_async();
        wg_bar_sync(1 + wg);
        if (w0) {
          if (elect_one_sync()) {
            tma_store_2d(&tmX, res_wg + (s & 1) * GL_RES_BYTES, gcol_wg + 16 * s, row0);
            tma_store_commit();
            if (s + 2 < GL_NSUB) {
              tma_store_wait_read<0>();                         // the buffer is free again once the store has read it
              mbar_expect_tx(&rfull[s & 1], GL_RES_BYTES);
              tma_load_2d(res_wg + (s & 1) * GL_RES_BYTES, &tmX, &rfull[s & 1], gcol_wg + 16 * (s + 2), row0);
            }
          }
          __syncwarp();
        }
      }
      if (w0 && tile + npairs < m_tiles) {
        if (elect_one_sync()) {
          tma_store_wait_read<0>();                             // the x stores of this tile have read both buffers
          for (int s = 0; s < 2; ++s) {
            mbar_expect_tx(&rfull[s], GL_RES_BYTES);
            tma_load_2d(res_wg + s * GL_RES_BYTES, &tmX, &rfull[s], gcol_wg + 16 * s, (tile + npairs) * GT_BM);
          }
        }
        __syncwarp();
      }
      if (!do_ln) {
        fence_before_sync();
        mbar_arrive(&tempty_bar[b]);
        continue;
      }
      tmem_st_wait();
      if (tm_ && it < 8) tm_[8 * it + 2] = clock64();
      // ---- half-row mean ----
      part[wg * GT_BM + r].x = sum;
      epi_bar_sync_all();
      if (tm_ && it < 8) tm_[8 * it + 3] = clock64();
      const float hsum = (part[r].x + part[GT_BM + r].x) + (part[2 * GT_BM + r].x + part[3 * GT_BM + r].x);
      const float hmean = hsum * (1.0f / GL_HN);
      // ---- pass 2: centred sum of squares of the half row ----
      float sq = 0.f;
#pragma unroll 1
      for (int s = 0; s < GL_NSUB; ++s) {
        float v[16];
        tmem_ld16(trow + 16 * s, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float d = v[i] - hmean;
          sq = fmaf(d, d, sq);
        }
      }
      part[wg * GT_BM + r].y = sq;
      epi_bar_sync_all();
      if (tm_ && it < 8) tm_[8 * it + 4] = clock64();
      const float hm2 = (part[r].y + part[GT_BM + r].y) + (part[2 * GT_BM + r].y + part[3 * GT_BM + r].y);
      // ---- exchange with the peer CTA (the other 192 columns of the same rows) ----
      if (wg == 0) {
        st_cluster_f2(peer_mail + (uint32_t)((b * GT_BM + r) * sizeof(float2)), hsum, hm2);
        mbar_arrive_cluster(peer_bar + b * (uint32_t)sizeof(uint64_t));
      }
      mbar_wait_cluster(&mail_bar[b], (it >> 1) & 1);
      if (tm_ && it < 8) tm_[8 * it + 5] = clock64();
      const float2 pm = mail[b * GT_BM + r];
      const float mean = (hsum + pm.x) * (1.0f / GL_N);
      const float dm = hmean - pm.x * (1.0f / GL_HN);
      const float var = (hm2 + pm.y + dm * dm * (0.25f * GL_N)) * (1.0f / GL_N);   // Chan: n_a n_b / (n_a + n_b) = 96
      const float rstd = rsqrtf(var + eps);
      // ---- pass 3: normalise -> 16 bit -> TMA store ----
#pragma unroll 1
      for (int s = 0; s < GL_NSUB; ++s) {
        float v[16];
        tmem_ld16(trow + 16 * s, v);
        if (s + 1 == GL_NSUB) {
          fence_before_sync();
          mbar_arrive(&tempty_bar[b]);                          // last TMEM read of this tile
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int c = col_wg + 16 * s + i;
          v[i] = (v[i] - mean) * rstd * sgamma[c] + sbeta[c];
        }
        uint4 p[2];
        pack16<T>(v, p);
        stage_store16(&tmXn, xn_wg, r, wg, p, gcol_wg + 16 * s, row0);
      }
      if (tm_ && it < 8) tm_[8 * it + 6] = clock64();
    }
    if (w0) {
      if (elect_one_sync()) tma_store_wait_all();
      __syncwarp();
    }
  }
  fence_before_sync();
  cluster_sync_all();                       // nobody exits while the peer may still write into its shared memory
  if (warp == 1) {
    fence_after_sync();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace tc
