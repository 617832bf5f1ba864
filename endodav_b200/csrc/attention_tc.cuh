// tcgen05 flash attention for the spatial (per-frame) self-attention of the ViT encoder:
//   out[f, i, h, :] = softmax_j(q[f,i,h,:] . k[f,j,h,:]) v[f,j,h,:]     head dim 64, S ~ 1.4k tokens
// Replaces Attention.forward's q@k^T / softmax / @v (layers/attention.py:60-66); q is
// pre-scaled by 64^-0.5 at pack time, so the kernel applies no extra scale.
//
// PERSISTENT kernel: one CTA per SM walks a static list of work items; an item is 256 queries (two 128-row
// tiles, A and B; the last item of a (frame, head) may hold tile A only) of one (frame, head), whose keys /
// values are streamed in 128-row tiles.  384 threads = 3 warpgroups; setmaxnreg moves registers from warpgroup 0
// (56/thread) to the softmax warpgroups (224/thread):
//   warp 0       TMA producer: Q tiles of the item into one of two Q buffers, then K_j | V_j into a 4-stage
//                128B-swizzled ring.  The ring and the Q double buffer run ACROSS item boundaries, so the loads of
//                the next item (and the HBM burst when every CTA starts at once) hide under the current one.
//   warp 1       TMEM allocator + MMA issuer, WARP-UNIFORM (tc_common.cuh elect_one_sync):  S_t = Q_t K_j^T
//                (SS, 128x128x64, 4 x 64 cycles) and O_t += P_t V_j (A = P from TMEM, B = V tile MN-major,
//                128x64x128, 8 x 32 cycles).  The first S of the next item is issued during the last key block of
//                the current one.
//   warps 2,3    idle (fill warpgroup 0)
//   warps 4..7   softmax warpgroup of tile A: thread = query row.  tcgen05.ld the 128 scores of
//   warps 8..11  softmax warpgroup of tile B  the row into registers, row max (FMNMX3) / exp2 / row sum (packed
//                FFMA2 / FADD2) entirely thread-local, P rounded to 16 bit and written back to TMEM with
//                tcgen05.st, O rescaled in TMEM only when the running max grew by more than 2^8 (lazy rescale),
//                final O / l written straight to global.
// Software pipeline: S_t(j+1) is issued as soon as warpgroup t has pulled S_t(j) into registers (barrier s_free),
// i.e. it runs UNDER the softmax of S_t(j); the exponentials of block j are computed BEFORE waiting for
// O_t += P_t(j-1) V_{j-1} (only the P store and the rare O rescale need it).  The kernel is MUFU(ex2) bound:
// 2 x 128 x 128 exponentials per key block at 16 / clock / SM = 2048 cycles, against 1024 cycles of tensor work
// (tools/microbench.cu).  Measured timeline (edv_op_attention_timeline): ld 330 + max 310 + exp 1880 + wait 230 +
// store 130 cycles per key block when both warpgroups run in lockstep -- the MUFU idles while both are in their
// non-MUFU phases -- so warpgroup B starts FA_STAGGER cycles late: one warpgroup's exponentials then run under
// the other's load / max / store phases.
//
// TMEM columns (512): S_A [0,128) S_B [128,256) O_A [256,320) O_B [320,384) P_A [384,448) P_B [448,512)
#pragma once
#include "attention_simt.cuh"
#include "ops.h"

#include "tc_common.cuh"

namespace tc {

constexpr int FA_BM = 128;      // query rows per tile
constexpr int FA_BN = 128;      // keys per iteration
constexpr int FA_HD = 64;
constexpr int FA_STAGES = 4;
constexpr uint32_t FA_TILE_BYTES = FA_BM * FA_HD * 2;  // 16 KB: one 128 x 64 16-bit tile
constexpr int FA_QBUF = 2;           // Q double buffer (items i and i+1)
constexpr int FA_THREADS = 384;      // producer warpgroup + two softmax warpgroups (see the header)
constexpr int FA_STAGGER = 1000;     // cycles warpgroup B starts behind warpgroup A (see the header)
constexpr size_t FA_SMEM = 1024 + (2 * FA_QBUF + 2 * FA_STAGES) * (size_t)FA_TILE_BYTES + 256;   // + barriers

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_pair(float a, float b, bf16) {
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ uint32_t pack_pair(float a, float b, f16) {
  __half2 t = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}

__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
      "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}

// ---- packed fp32x2 helpers (FFMA2 / FADD2 / FMNMX3 on sm_100: half the issue slots of the scalar forms) ----
__device__ __forceinline__ void fma2_bcast(float& d0, float& d1, float a0, float a1, float b, float c) {
  uint64_t ra, rb, rc, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %1};" : "=l"(rb) : "f"(b));
  asm("mov.b64 %0, {%1, %1};" : "=l"(rc) : "f"(c));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d0), "=f"(d1) : "l"(rd));
}
__device__ __forceinline__ void add2(float& d0, float& d1, float a0, float a1) {
  uint64_t ra, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rd) : "f"(d0), "f"(d1));
  asm("add.rn.f32x2 %0, %0, %1;" : "+l"(rd) : "l"(ra));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d0), "=f"(d1) : "l"(rd));
}
__device__ __forceinline__ float max3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}

struct FaItem {
  int f, h, q0, nt;
};
__device__ __forceinline__ FaItem fa_item(int w, int nx, int heads, int S) {
  FaItem it;
  const int x = w % nx;
  const int r = w / nx;
  it.h = r % heads;
  it.f = r / heads;
  it.q0 = x * (2 * FA_BM);
  it.nt = (it.q0 + FA_BM) < S ? 2 : 1;   // tile B holds at least one real query
  return it;
}

// Two threads per query row (four softmax warpgroups, row max / sum exchanged through shared memory) and evaluating
// part of the exponentials as a polynomial on the FMA pipe were both measured slower than one thread per row with every
// exp2 on the MUFU (DESIGN.md section 5, profiles/r2_fa_variants_timeline.txt).
template <typename T>
__global__ void __launch_bounds__(FA_THREADS, 1)
    flash_attention_tc_kernel(const __grid_constant__ CUtensorMap tmQKV, T* __restrict__ out, int S, int heads, int nx,
                              int total_items, long long* __restrict__ tim) {
  pdl_launch();   // PDL: the next kernel of the stream may start its prologue (common.cuh)
  // tim: optional in-kernel timeline (clock64 stamps of the first 8 CTAs, 64 slots each; edv_op_attention_timeline):
  // 0 entry, 1 setup done, 2 first S ready, 3+j end of softmax iteration j of the FIRST item (tile A), 20 its O complete,
  // 21 stored, 24+j PV(j) issued, 44..48 phases of iteration 5 (S loaded, max, exps, PV(j-1) done, P stored),
  // 50+i end of item i (tile A, i < 12)
  long long* tm_ = (tim && blockIdx.x < 8) ? tim + blockIdx.x * 64 : nullptr;
  if (tm_ && threadIdx.x == 0) tm_[0] = clock64();
  extern __shared__ __align__(1024) unsigned char fa_smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(fa_smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* sQ = smem;                                        // FA_QBUF x 2 tiles
  unsigned char* sKV = smem + FA_QBUF * 2 * FA_TILE_BYTES;         // stages x (K | V)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sKV + (size_t)FA_STAGES * 2 * FA_TILE_BYTES);
  uint64_t* q_full = bars;                       // FA_QBUF
  uint64_t* q_empty = q_full + FA_QBUF;          // FA_QBUF: every S = Q K^T of the item has completed
  uint64_t* kv_full = q_empty + FA_QBUF;         // FA_STAGES
  uint64_t* kv_empty = kv_full + FA_STAGES;
  uint64_t* s_full = kv_empty + FA_STAGES;       // 2
  uint64_t* p_full = s_full + 2;                 // 2
  uint64_t* o_done = p_full + 2;                 // 2
  uint64_t* s_free = o_done + 2;                 // 2: warpgroup t holds S_t(j) in registers
  uint64_t* pv_done = s_free + 2;                // 2: O_t += P_t(j) V_j has completed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(pv_done + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int D = heads * FA_HD;
  const int n_iter = (S + FA_BN - 1) / FA_BN;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQKV);
    for (int b = 0; b < FA_QBUF; ++b) {
      mbar_init(&q_full[b], 1);
      mbar_init(&q_empty[b], 1);
    }
    for (int s = 0; s < FA_STAGES; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], 1);
    }
    for (int t = 0; t < 2; ++t) {
      mbar_init(&s_full[t], 1);
      mbar_init(&p_full[t], 128);
      mbar_init(&o_done[t], 1);
      mbar_init(&s_free[t], 128);
      mbar_init(&pv_done[t], 1);
    }
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();     // PDL: everything above ran under the previous kernel's tail; its results are visible from here
  if (tm_ && threadIdx.x == 0) tm_[1] = clock64();

  if (warp < 4) {
   asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
   if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      uint32_t kc = 0, it = 0;
      for (int w = blockIdx.x; w < total_items; w += gridDim.x, ++it) {
        const FaItem im = fa_item(w, nx, heads, S);
        const int row_base = im.f * S;
        const uint32_t qb = it % FA_QBUF;
        mbar_wait(&q_empty[qb], ((it / FA_QBUF) & 1) ^ 1);
        unsigned char* q = sQ + (size_t)qb * 2 * FA_TILE_BYTES;
        mbar_expect_tx(&q_full[qb], (uint32_t)im.nt * FA_TILE_BYTES);
        tma_load_2d(q, &tmQKV, &q_full[qb], im.h * FA_HD, row_base + im.q0);
        if (im.nt == 2) tma_load_2d(q + FA_TILE_BYTES, &tmQKV, &q_full[qb], im.h * FA_HD, row_base + im.q0 + FA_BM);
        for (int j = 0; j < n_iter; ++j, ++kc) {
          const int s = kc % FA_STAGES;
          mbar_wait(&kv_empty[s], ((kc / FA_STAGES) & 1) ^ 1);
          unsigned char* sk = sKV + (size_t)s * 2 * FA_TILE_BYTES;
          mbar_expect_tx(&kv_full[s], 2 * FA_TILE_BYTES);
          tma_load_2d(sk, &tmQKV, &kv_full[s], D + im.h * FA_HD, row_base + j * FA_BN);
          tma_load_2d(sk + FA_TILE_BYTES, &tmQKV, &kv_full[s], 2 * D + im.h * FA_HD, row_base + j * FA_BN);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: WARP-UNIFORM loop (all lanes wait and build descriptors), the elected lane issues =====
    constexpr uint32_t idesc_qk = make_idesc<T>(FA_BM, FA_BN, 0);   // K-major A and B
    constexpr uint32_t idesc_pv = make_idesc<T>(FA_BM, FA_HD, 1);   // B = V tile, MN-major
    const uint32_t leader = elect_one_sync();
    const uint32_t sq_addr = smem_u32(sQ), skv_addr = smem_u32(sKV);
    uint32_t kc = 0, it = 0;
    uint32_t n_qk[2] = {0, 0};   // S tiles issued so far per query tile (= s_free completions needed before the next)
    uint32_t n_pv[2] = {0, 0};   // PV batches issued so far per query tile
    // S_t = Q_t K^T for key stage `stage`, Q buffer `qb`; the S buffer must have been drained n_qk[t] times
    auto issue_qk = [&](int t, uint32_t qb, uint32_t stage) {
      if (n_qk[t] > 0) {
        mbar_wait(&s_free[t], (n_qk[t] - 1) & 1);
        fence_after_sync();
      }
      const uint64_t adesc = make_smem_desc(sq_addr + (qb * 2 + t) * FA_TILE_BYTES, 1024, 16, SWZ_128B);
      const uint64_t bdesc = make_smem_desc(skv_addr + stage * 2 * FA_TILE_BYTES, 1024, 16, SWZ_128B);
      if (leader) {
#pragma unroll
        for (int k = 0; k < FA_HD / 16; ++k)
          mma_ss(tmem_base + t * FA_BN, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc_qk, k ? 1u : 0u);
        mma_commit(&s_full[t]);
      }
      __syncwarp();
      ++n_qk[t];
    };
    if (blockIdx.x < total_items) {
      const FaItem first = fa_item(blockIdx.x, nx, heads, S);
      mbar_wait(&q_full[0], 0);
      mbar_wait(&kv_full[0], 0);
      fence_after_sync();
      for (int t = 0; t < first.nt; ++t) issue_qk(t, 0, 0);
    }
    for (int w = blockIdx.x; w < total_items; w += gridDim.x, ++it) {
      const FaItem im = fa_item(w, nx, heads, S);
      const uint32_t qb = it % FA_QBUF;
      const bool has_next = (w + (int)gridDim.x) < total_items;
      for (int j = 0; j < n_iter; ++j, ++kc) {
        const uint32_t s = kc % FA_STAGES;
        // 1) the next S: S_t(j+1) of this item, or S_t(0) of the NEXT item during the last key block
        if (j + 1 < n_iter) {
          const uint32_t s1 = (kc + 1) % FA_STAGES;
          mbar_wait(&kv_full[s1], ((kc + 1) / FA_STAGES) & 1);
          fence_after_sync();
          for (int t = 0; t < im.nt; ++t) issue_qk(t, qb, s1);
          if (j + 2 == n_iter) {
            if (leader) mma_commit(&q_empty[qb]);       // the last S of this item is in flight: Q buffer reusable when it completes
            __syncwarp();
          }
        } else {
          if (n_iter == 1) {
            if (leader) mma_commit(&q_empty[qb]);
            __syncwarp();
          }
          if (has_next) {
            const FaItem nx_im = fa_item(w + (int)gridDim.x, nx, heads, S);
            const uint32_t qb2 = (it + 1) % FA_QBUF;
            const uint32_t s1 = (kc + 1) % FA_STAGES;
            mbar_wait(&q_full[qb2], ((it + 1) / FA_QBUF) & 1);
            mbar_wait(&kv_full[s1], ((kc + 1) / FA_STAGES) & 1);
            fence_after_sync();
            for (int t = 0; t < nx_im.nt; ++t) issue_qk(t, qb2, s1);
          }
        }
        // 2) O_t (+)= P_t(j) V_j : A from TMEM (8 columns per 16-key step), B rows = keys (MN-major,
        //    128 B per key, 8-key groups 1024 B apart) -> +2048 B per 16-key step
        const uint64_t vdesc = make_smem_desc(skv_addr + s * 2 * FA_TILE_BYTES + FA_TILE_BYTES, 1024, 1024, SWZ_128B);
        for (int t = 0; t < im.nt; ++t) {
          mbar_wait(&p_full[t], n_pv[t] & 1);   // P_t(j) in TMEM, O_t rescaled (and, for j = 0, the previous item's O read out)
          fence_after_sync();
          if (leader) {
#pragma unroll
            for (int k = 0; k < FA_BN / 16; ++k)
              mma_ts(tmem_base + 256 + t * FA_HD, tmem_base + 384 + t * 64 + k * 8, vdesc + (uint64_t)(128 * k), idesc_pv,
                     (j | k) ? 1u : 0u);
            mma_commit(&pv_done[t]);
            if (t == im.nt - 1) mma_commit(&kv_empty[s]);   // K_j and V_j no longer needed once these complete
            if (j + 1 == n_iter) mma_commit(&o_done[t]);
            if (tm_ && it == 0 && t == im.nt - 1 && j < 16) tm_[24 + j] = clock64();
          }
          __syncwarp();
          ++n_pv[t];
        }
      }
    }
   }
  } else {
    // ===== softmax warpgroups =====
    asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
    const int t = (warp - 4) >> 2;        // softmax warpgroup = query tile (0: tile A, 1: tile B)
    const int q = warp & 3;               // TMEM lane quarter this warp may access
    const int r = q * 32 + lane;          // row inside the tile
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const uint32_t tS = tmem_base + lane_off + t * FA_BN;
    const uint32_t tO = tmem_base + lane_off + 256 + t * FA_HD;
    const uint32_t tP = tmem_base + lane_off + 384 + t * 64;
    constexpr float LOG2E = 1.4426950408889634f;
    const bool stamp = tm_ && t == 0 && r == 0;
    if (t == 1) {
      // start half a key block behind warpgroup A (see the header): the offset persists, both warpgroups run the same loop
      const long long c0 = clock64();
      while (clock64() - c0 < FA_STAGGER) {
      }
    }
    uint32_t cnt = 0, items = 0;          // key blocks / items processed by this query tile so far (barrier phases)
    uint32_t it = 0;
    for (int w = blockIdx.x; w < total_items; w += gridDim.x, ++it) {
      const FaItem im = fa_item(w, nx, heads, S);
      if (t >= im.nt) continue;
      const int row_base = im.f * S;
      float m_used = -INFINITY;           // max the exponentials are currently taken against (raw units)
      float l = 0.f;                      // row sum
      for (int j = 0; j < n_iter; ++j, ++cnt) {
        mbar_wait(&s_full[t], cnt & 1);
        fence_after_sync();
        if (stamp && cnt == 0) tm_[2] = clock64();
        uint32_t sv[FA_BN];
#pragma unroll
        for (int c = 0; c < FA_BN; c += 32) tmem_ld32_nowait(tS + c, sv + c);
        tmem_ld_wait();
        fence_before_sync();
        mbar_arrive(&s_free[t]);          // S_t(j) is in registers: the tensor core may overwrite it with the next S_t
        if (stamp && cnt == 5) tm_[44] = clock64();
        const int valid = S - j * FA_BN;  // keys of this block that belong to the frame
        if (valid < FA_BN) {
#pragma unroll
          for (int i = 0; i < FA_BN; ++i)
            if (i >= valid) sv[i] = 0xff800000u;  // -inf
        }
        // row max: 8 independent chains of 3-input maxima (FMNMX3)
        float pm[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) pm[i] = max3(__uint_as_float(sv[i]), __uint_as_float(sv[8 + i]), __uint_as_float(sv[16 + i]));
#pragma unroll
        for (int i = 24; i < FA_BN - 8; i += 16) {
#pragma unroll
          for (int c = 0; c < 8; ++c) pm[c] = max3(pm[c], __uint_as_float(sv[i + c]), __uint_as_float(sv[i + 8 + c]));
        }
#pragma unroll
        for (int c = 0; c < 8; ++c) pm[c] = fmaxf(pm[c], __uint_as_float(sv[FA_BN - 8 + c]));
        const float mx = fmaxf(max3(pm[0], pm[1], pm[2]), fmaxf(max3(pm[3], pm[4], pm[5]), fmaxf(pm[6], pm[7])));
        // lazy rescale: keep the old reference max unless the row max grew by more than 2^8
        float factor = 1.f;
        const bool grow = mx > m_used + 8.f / LOG2E;
        if (grow) {
          factor = ex2_approx((m_used - mx) * LOG2E);   // 0 on the first tile (m_used = -inf)
          m_used = mx;
          l *= factor;
        }
        // exponentials of the whole row BEFORE the wait on O_t += P_t(j-1) V_{j-1}: only the P store and the
        // (rare) O rescale need that MMA to have finished, so the softmax of block j runs under the PV of block j-1
        const float neg = -m_used * LOG2E;
        if (stamp && cnt == 5) tm_[45] = clock64();
        float ls0 = 0.f, ls1 = 0.f, ls2 = 0.f, ls3 = 0.f;   // two packed partial row sums
        uint32_t pv[FA_BN / 2];
#pragma unroll
        for (int i = 0; i < FA_BN / 2; ++i) {
          float x0, x1;
          fma2_bcast(x0, x1, __uint_as_float(sv[2 * i]), __uint_as_float(sv[2 * i + 1]), LOG2E, neg);
          const float p0 = ex2_approx(x0), p1 = ex2_approx(x1);
          if (i & 1) add2(ls2, ls3, p0, p1);
          else add2(ls0, ls1, p0, p1);
          pv[i] = pack_pair(p0, p1, T());
        }
        l += (ls0 + ls1) + (ls2 + ls3);
        if (stamp && cnt == 5) tm_[46] = clock64();
        if (j > 0) {
          mbar_wait(&pv_done[t], (cnt - 1) & 1);   // O_t += P_t(j-1) V_{j-1} done: O_t stable, P_t free
          fence_after_sync();
          if (stamp && cnt == 5) tm_[47] = clock64();
          if (__any_sync(0xffffffffu, grow)) {
#pragma unroll
            for (int c = 0; c < FA_HD; c += 32) {
              uint32_t ov[32];
              tmem_ld32_nowait(tO + c, ov);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 32; ++i) ov[i] = __float_as_uint(__uint_as_float(ov[i]) * factor);
              tmem_st32(tO + c, ov);
            }
          }
        }
        // (j == 0: the last PV of this tile's previous item completed before its epilogue read O -- o_done)
#pragma unroll
        for (int c = 0; c < FA_BN / 2; c += 32) tmem_st32(tP + c, pv + c);
        tmem_st_wait();
        fence_before_sync();
        mbar_arrive(&p_full[t]);
        if (stamp && cnt == 5) tm_[48] = clock64();
        if (stamp && cnt < 16) tm_[3 + cnt] = clock64();
      }
      // ---- epilogue: O / l -> global ----
      mbar_wait(&o_done[t], items & 1);
      fence_after_sync();
      if (stamp && items == 0) tm_[20] = clock64();
      const float inv = 1.f / l;
      const int qi = im.q0 + t * FA_BM + r;
      T* orow = out + ((long long)row_base + qi) * D + im.h * FA_HD;
#pragma unroll
      for (int c = 0; c < FA_HD; c += 32) {
        uint32_t ov[32];
        tmem_ld32_nowait(tO + c, ov);
        tmem_ld_wait();
        if (qi < S) {
          float o[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) o[i] = __uint_as_float(ov[i]) * inv;
          store_vec<T, 32>(orow + c, o);
        }
      }
      fence_before_sync();                // the O loads are complete before this thread's next p_full arrive lets PV(0) overwrite O
      if (stamp && items == 0) tm_[21] = clock64();
      if (stamp && items < 12) tm_[50 + items] = clock64();
      ++items;
    }
  }
  __syncthreads();
  if (warp == 1) {
    fence_after_sync();
    tmem_dealloc(tmem_base, 512);
  }
}

template <typename T>
void launch_attention_tc(edv::Launch& L, int dtype, const void* qkv, void* out, int F, int S, int heads, long long* timeline = nullptr) {
  const uint64_t D = heads * FA_HD;
  CUtensorMap tm;
  if (!edv::make_tmap_2d(L, &tm, dtype, qkv, 3 * D, (uint64_t)F * S, 3 * D * 2, FA_HD, FA_BM, 128)) return;
  constexpr auto kern = flash_attention_tc_kernel<T>;
  edv::smem_opt_in<kern>((int)FA_SMEM);
  const int nx = (S + 2 * FA_BM - 1) / (2 * FA_BM);
  const long long total = (long long)nx * heads * F;
  if (total > 0x7fffffffLL) return L.fail(EDV_ERR_ARG, "flash_attention_tc: too many work items");
  const int grid = (int)std::min<long long>(total, edv::num_sms());
  edv::launch_k(kern, dim3(grid), dim3(FA_THREADS), FA_SMEM, L.stream, tm, (T*)out, S, heads, nx, (int)total, timeline);
  L.check("flash_attention_tc");
}

}  // namespace tc
