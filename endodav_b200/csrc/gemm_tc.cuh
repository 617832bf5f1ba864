// Persistent tcgen05 GEMM / implicit-GEMM 3x3 convolution for sm_100a.
//
//   C[M,N] = A[M,K] * W[N,K]^T   (16-bit operands, fp32 accumulation in TMEM)
//
// One CTA per SM loops over 128 x BN output tiles (static round-robin, n fastest so that CTAs
// running together share A tiles through L2).  640 threads:
//   warp 0       TMA producer  -- cp.async.bulk.tensor loads of the A and W k-blocks into a ring
//                of 128B(64B)-swizzled shared-memory stages, completion on mbarriers; the ring
//                runs ahead across tile boundaries
//   warp 1       TMEM allocator + MMA issuer -- one lane issues tcgen05.mma (M=128, N=BN, K=16)
//                into one of TWO accumulator buffers in TMEM; tcgen05.commit releases the smem
//                stage / hands the finished accumulator to its epilogue warpgroup
//   warps 2,3    idle (keep the epilogue warpgroups 4-warp aligned for the TMEM lane quarters)
//   warps 4..19  four epilogue warpgroups: warpgroup wg drains columns [half*BN/2, +BN/2) of
//                accumulator buffer (wg & 1) (even / odd tiles of this CTA), half = wg >> 1
//                tcgen05.ld (lane = row), fused bias / row-bias / GELU / GEGLU / residual / ReLU /
//                pixel-shuffle / disparity-head epilogue (common.cuh), 16-byte vector stores.
// So the epilogue of tile i overlaps the mainloop of tile i+1 -- with K = 384 (ViT-S) the
// epilogue is as long as the mainloop and hiding it is what matters.
//
// CONV=false: A is a row-major [M,K] matrix (2-D tensor map), M tail rows are zero-filled by
//             TMA and masked in the epilogue.
// CONV=true : A is an NHWC activation [F,H,W,C]; the M tile is a TH x TW pixel patch of one
//             frame and k-block (tap, c0) is the patch shifted by the tap offset, fetched
//             with a 4-D tensor map whose out-of-bounds fill supplies the zero padding.
//             K = 9*C in (ky,kx,c) order.
#pragma once
#include "tc_common.cuh"

namespace tc {

struct ConvTile {
  int H, W, C;          // NHWC input == output spatial size (stride 1, pad 1)
  int th, tw;           // tile shape, th*tw == 128
  int tiles_y, tiles_x; // per frame
};

constexpr int GT_BM = 128;
constexpr int GT_PF_KB = 8;   // L2 prefetch distance of the A operand in k-blocks (tc_common.cuh tma_prefetch_2d)
constexpr int GT_THREADS = 640;

template <int BN, int BK> constexpr int gt_stage_bytes() { return (GT_BM + BN) * BK * 2; }
template <int BN> constexpr uint32_t gt_tmem_cols() { return 2 * BN <= 64 ? 64 : 2 * BN <= 128 ? 128 : 2 * BN <= 256 ? 256 : 512; }

constexpr int GT_STG_WORDS = 32 * 32;   // per-warp transposition buffer: 32 rows x 32 fp32, 16-byte chunks XOR-swizzled

// Row-owner -> row-segment transposition of one warp's 32 x 32 fp32 block through shared memory.
// write: thread = row, 8 x STS.128 with the 16-byte chunk index XORed by (row & 7)  (conflict-free)
// read : lane = (row it*4 + lane/8, columns 4*(lane%8)..+3), LDS.128                (conflict-free)
__device__ __forceinline__ void gt_stage_write(uint32_t* stg, int lane, const float* v) {
#pragma unroll
  for (int j = 0; j < 8; ++j)
    *reinterpret_cast<float4*>(stg + lane * 32 + ((j ^ (lane & 7)) << 2)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}
__device__ __forceinline__ float4 gt_stage_read(const uint32_t* stg, int rr, int j) {
  return *reinterpret_cast<const float4*>(stg + rr * 32 + ((j ^ (rr & 7)) << 2));
}

__device__ __forceinline__ void f4_add(float4& a, const float4& b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
template <typename T> __device__ __forceinline__ float4 ld4_as_f32(const void* p, int is_f32, long long off) {
  if (is_f32) return *reinterpret_cast<const float4*>((const float*)p + off);   // plain loads: may alias the output (x += ...)
  float v[4];
  load_vec<T, 4>((const T*)p + off, v);
  return make_float4(v[0], v[1], v[2], v[3]);
}

// Compile-time epilogue kinds.  The runtime-flag version of this code is a chain of
// `if (flag) { unrolled block }`: every skipped block is a taken branch to a far target, and with
// the epilogue far larger than the L0 instruction cache each of them is an instruction-fetch stall
// (ncu: stall_no_inst on every other line, ~2 500 cycles per 32-column chunk).  The hot call sites
// of the forward therefore get straight-line instantiations (F >= 0: bit mask below); anything
// else (row-bias tables, pixel shuffle, sigmoid) runs the generic F = -1 version.
// (the EF_* bit mask is declared in common.cuh: the launcher side needs it without the kernels)

// The fused epilogue on NS row segments (4 consecutive columns starting at n of rows mm[it] ->
// output rows oo[it], oo < 0 = masked).  Same order of operations as epi_apply (common.cuh):
// bias, per-frame row bias, GELU, residual(s), ReLU / sigmoid, stores.  Every stage is a loop over
// the NS segments so the loads of a stage are all in flight together.
template <typename T, int NS, int F>
__device__ __forceinline__ void gt_applyN(const Epi& e, float4* a, const int* mm, const int* oo, int n,
                                          const float* bias4) {
  constexpr bool S = F >= 0;
  const bool has_bias = S ? ((F & EF_BIAS) != 0) : (bias4 != nullptr);
  const bool do_gelu = S ? ((F & EF_GELU) != 0) : (e.act == ACT_GELU);
  const bool do_relu = S ? ((F & EF_RELU) != 0) : (e.act == ACT_RELU);
  const bool has_res1 = S ? ((F & (EF_RES1_F32 | EF_RES1_T)) != 0) : (e.res1 != nullptr);
  const int res1_f32 = S ? ((F & EF_RES1_F32) != 0) : e.res1_f32;
  const bool has_res2 = S ? ((F & EF_RES2_T) != 0) : (e.res2 != nullptr);
  const int res2_f32 = S ? 0 : e.res2_f32;
  const bool has_out = S ? true : (e.out != nullptr);
  const int out_f32 = S ? ((F & EF_OUT_F32) != 0) : e.out_f32;
  const bool has_out_relu = S ? ((F & EF_OUT_RELU) != 0) : (e.out_relu != nullptr);
  if (has_bias) {
    // the bias slice was staged in shared memory before the accumulator wait (with ~200 KB of the
    // SM's memory carved out as shared, L1 holds almost nothing)
    const float4 b = *reinterpret_cast<const float4*>(bias4);
#pragma unroll
    for (int it = 0; it < NS; ++it) f4_add(a[it], b);
  }
  const bool has_rowbias = S ? ((F & EF_ROWBIAS) != 0) : (e.rowbias != nullptr);
  if (has_rowbias) {
#pragma unroll
    for (int it = 0; it < NS; ++it)
      if (oo[it] >= 0) f4_add(a[it], *reinterpret_cast<const float4*>(e.rowbias + (long long)((mm[it] / e.rb_div) % e.rb_mod) * e.rb_ld + n));
  }
  if (do_gelu) {
#pragma unroll
    for (int it = 0; it < NS; ++it) {
      a[it].x = gelu_act<T>(a[it].x); a[it].y = gelu_act<T>(a[it].y);
      a[it].z = gelu_act<T>(a[it].z); a[it].w = gelu_act<T>(a[it].w);
    }
  }
  long long orow[NS];
  int ocol = n;
  if (!S && e.map == MAP_PIXSHUF) {
    // m = (f, y, x) over the ps_h x ps_w grid; n = (ky*k + kx)*ps_c + c
    const int tap = n / e.ps_c;
    ocol = n - tap * e.ps_c;
    const int ky = tap / e.ps_k, kx = tap - ky * e.ps_k;
    const int hw = e.ps_h * e.ps_w;
#pragma unroll
    for (int it = 0; it < NS; ++it) {
      const int f = mm[it] / hw;
      const int r = mm[it] - f * hw;
      const int y = r / e.ps_w, x = r - y * e.ps_w;
      orow[it] = ((long long)f * (e.ps_h * e.ps_k) + (long long)y * e.ps_k + ky) * ((long long)e.ps_w * e.ps_k) + (long long)x * e.ps_k + kx;
    }
  } else {
#pragma unroll
    for (int it = 0; it < NS; ++it) orow[it] = oo[it];
  }
  if (has_res1) {
    float4 r[NS];
#pragma unroll
    for (int it = 0; it < NS; ++it) r[it] = (oo[it] >= 0) ? ld4_as_f32<T>(e.res1, res1_f32, orow[it] * e.ld_res1 + ocol) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int it = 0; it < NS; ++it) f4_add(a[it], r[it]);
  }
  if (has_res2) {
    float4 r[NS];
#pragma unroll
    for (int it = 0; it < NS; ++it) r[it] = (oo[it] >= 0) ? ld4_as_f32<T>(e.res2, res2_f32, orow[it] * e.ld_res2 + ocol) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int it = 0; it < NS; ++it) f4_add(a[it], r[it]);
  }
  if (do_relu) {
#pragma unroll
    for (int it = 0; it < NS; ++it) { a[it].x = fmaxf(a[it].x, 0.f); a[it].y = fmaxf(a[it].y, 0.f); a[it].z = fmaxf(a[it].z, 0.f); a[it].w = fmaxf(a[it].w, 0.f); }
  } else if (!S && e.act == ACT_SIGMOID) {
#pragma unroll
    for (int it = 0; it < NS; ++it) {
      a[it].x = 1.f / (1.f + __expf(-e.sig_sign * a[it].x)); a[it].y = 1.f / (1.f + __expf(-e.sig_sign * a[it].y));
      a[it].z = 1.f / (1.f + __expf(-e.sig_sign * a[it].z)); a[it].w = 1.f / (1.f + __expf(-e.sig_sign * a[it].w));
    }
  }
  if (has_out) {
    if (out_f32) {
#pragma unroll
      for (int it = 0; it < NS; ++it)
        if (oo[it] >= 0) *reinterpret_cast<float4*>((float*)e.out + orow[it] * e.ldo + ocol) = a[it];
    } else {
#pragma unroll
      for (int it = 0; it < NS; ++it)
        if (oo[it] >= 0) {
          uint2 w;
          w.x = pack2(from_f<T>(a[it].x), from_f<T>(a[it].y));
          w.y = pack2(from_f<T>(a[it].z), from_f<T>(a[it].w));
          *reinterpret_cast<uint2*>((T*)e.out + orow[it] * e.ldo + ocol) = w;
        }
    }
  }
  if (has_out_relu) {
#pragma unroll
    for (int it = 0; it < NS; ++it)
      if (oo[it] >= 0) {
        uint2 w;
        w.x = pack2(from_f<T>(fmaxf(a[it].x, 0.f)), from_f<T>(fmaxf(a[it].y, 0.f)));
        w.y = pack2(from_f<T>(fmaxf(a[it].z, 0.f)), from_f<T>(fmaxf(a[it].w, 0.f)));
        *reinterpret_cast<uint2*>((T*)e.out_relu + orow[it] * e.ldo + ocol) = w;
      }
  }
}

// The row-segment path of gt_epilogue for columns [half*BN/2, +BN/2) of one accumulator.
template <typename T, int BN, int F>
__device__ __forceinline__ void gt_epi_rows(const Epi& e, uint32_t trow, int m32, int o32, int n0, uint32_t* stg, int lane,
                                            int half, const float* bias_s) {
  constexpr int CH0 = (BN >= 64) ? BN / 2 : BN;
  const int j = lane & 7, rsub = lane >> 3;
#pragma unroll 1
  for (int c = half * CH0; c < (BN >= 64 ? (half + 1) * CH0 : BN); c += 32) {
    float v[32];
    tmem_ld32(trow + c, v);
    gt_stage_write(stg, lane, v);
    __syncwarp();
#pragma unroll
    for (int hb = 0; hb < 2; ++hb) {   // 2 x 4 row segments: keeps the epilogue under 96 registers
      float4 a[4];
      int mm[4], oo[4];
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        const int rr = (hb * 4 + it) * 4 + rsub;
        mm[it] = __shfl_sync(0xffffffffu, m32, rr);
        oo[it] = __shfl_sync(0xffffffffu, o32, rr);
        a[it] = gt_stage_read(stg, rr, j);
      }
      gt_applyN<T, 4, F>(e, a, mm, oo, n0 + c + 4 * j, bias_s ? bias_s + (c - half * CH0) + 4 * j : nullptr);
    }
    __syncwarp();
  }
}

// epilogue of one 128 x BN accumulator: thread = row `r` of the tile, TMEM address `trow`.
// The accumulator leaves TMEM in the row-owner domain (tcgen05.ld: lane = row) and is transposed
// per warp through `stg`, so that the fused epilogue math (common.cuh: epi_apply) and every
// global access -- bias / residual loads, stores -- run with 8 lanes covering 32 consecutive
// columns of one row (128-bit accesses, 4 full rows per instruction).
template <typename T, int BN>
__device__ __forceinline__ void gt_epilogue(const Epi& e, uint32_t trow, bool valid, long long m, long long orow_lin,
                                            int n0, int tile_n, uint32_t* stg, int lane, int half,
                                            const float* bias_s) {
  const int m32 = (int)m;                          // rows < 2^31 (checked by the launcher)
  const int o32 = valid ? (int)orow_lin : -1;
  const int j = lane & 7, rsub = lane >> 3;
  // the two warpgroups of an accumulator split its columns: [0, BN/2) and [BN/2, BN)
  [[maybe_unused]] constexpr int CH0 = (BN >= 64) ? BN / 2 : BN;
  if (e.act == ACT_HEAD) {
    // whole row in one tile (BN == N == 32): relu(conv+b) . w + b -> relu  (dpt.py:118-123)
    if (half != 0) return;
    if constexpr (BN == 32) {
      float v[32];
      tmem_ld32(trow, v);
      if (valid) {
        float s = e.head_b + __ldg(e.head_w + 32);  // head_w[32] carries the 1x1 conv bias
#pragma unroll
        for (int i = 0; i < 32; ++i) s = fmaf(fmaxf(v[i] + __ldg(e.bias + i), 0.f), __ldg(e.head_w + i), s);
        if (e.sig_sign == 0.f) s = fmaxf(s, 0.f);             // output_conv2: trailing ReLU
        else s = 1.f / (1.f + expf(-e.sig_sign * s));         // HeadDepth + sigmoid
        ((float*)e.out)[orow_lin] = s;
      }
    }
  } else if (e.act == ACT_GEGLU) {
    // BN == 128: columns [0,64) value, [64,128) gate (pack.py pairs them per tile)
    if constexpr (BN == 128) {
      {
        const int c = half * 32;
        float v[32];
        float4 hv[8];
        tmem_ld32(trow + c, v);
        gt_stage_write(stg, lane, v);
        __syncwarp();
#pragma unroll
        for (int it = 0; it < 8; ++it) hv[it] = gt_stage_read(stg, it * 4 + rsub, j);
        __syncwarp();
        tmem_ld32(trow + 64 + c, v);
        gt_stage_write(stg, lane, v);
        __syncwarp();
        const float4 bh = *reinterpret_cast<const float4*>(e.bias + n0 + c + 4 * j);
        const float4 bg = *reinterpret_cast<const float4*>(e.bias + n0 + 64 + c + 4 * j);
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int rr = it * 4 + rsub;
          const int oo = __shfl_sync(0xffffffffu, o32, rr);
          const float4 gv = gt_stage_read(stg, rr, j);
          if (oo >= 0) {
            float o[4];
            o[0] = (hv[it].x + bh.x) * gelu_act<T>(gv.x + bg.x);
            o[1] = (hv[it].y + bh.y) * gelu_act<T>(gv.y + bg.y);
            o[2] = (hv[it].z + bh.z) * gelu_act<T>(gv.z + bg.z);
            o[3] = (hv[it].w + bh.w) * gelu_act<T>(gv.w + bg.w);
            store_vec<T, 4>((T*)e.out + (long long)oo * e.ldo + tile_n * 64 + c + 4 * j, o);
          }
        }
        __syncwarp();
      }
    }
  } else {
    if (BN < 64 && half != 0) return;
    switch (e.kind) {
#define EDV_EPI_CASE(F_) case F_: gt_epi_rows<T, BN, F_>(e, trow, m32, o32, n0, stg, lane, half, bias_s); break;
      EDV_EPI_ROW_KINDS(EDV_EPI_CASE)
#undef EDV_EPI_CASE
      default: gt_epi_rows<T, BN, -1>(e, trow, m32, o32, n0, stg, lane, half, bias_s); break;
    }
  }
}

// ---- TMA-store epilogue (EF_TMA_OUT): 16-bit row-major outputs without residual --------------------------------
// The row-segment epilogue above costs ~6 000 cycles per 128 x 192 tile even with trivial math (in-kernel timeline,
// tools/gemm_timeline.py: transposition through shared memory, row-index shuffles, 4-row store instructions), which
// made qkv / fc1 epilogue-bound at 2 x their mainloop.  Here the accumulator stays in the row-owner domain:
// thread = row, 16 columns per step: tcgen05.ld -> bias / GELU / ReLU -> pack to 16 bit -> two 16-byte shared-memory
// stores at 32B-swizzled chunk positions (conflict-free) -> one elected thread issues a TMA store of the
// 128 x 16 sub-tile (coalescing, M-tail clipping and address arithmetic are the TMA unit's job).  4 KB staging
// sub-tiles per epilogue warpgroup; cp.async.bulk.wait_group.read gates their reuse.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void wg_bar_sync(int id) { asm volatile("bar.sync %0, 128;" ::"r"(id) : "memory"); }

__device__ __forceinline__ void add2_f32(float& d0, float& d1, float a0, float a1) {   // packed FADD2
  unsigned long long ra, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rd) : "f"(d0), "f"(d1));
  asm("add.rn.f32x2 %0, %0, %1;" : "+l"(rd) : "l"(ra));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d0), "=f"(d1) : "l"(rd));
}

constexpr int GT_OUT_SUB_BYTES = GT_BM * 16 * 2;   // staging of one 128-row x 16-column 16-bit sub-tile (32-byte rows, SWIZZLE_32B)

__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait_all() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// The staging steps shared by the TMA-store epilogue and gemm_ln.cuh's pass 3.  r = row of the tile = thread of the
// warpgroup; warp 0 of the warpgroup (r < 32) owns the bulk-store groups, its elected lane issues (warp-uniform branch:
// no uniformisation loops around UTMASTG).
template <typename T> __device__ __forceinline__ void pack16(const float* v, uint4* p) {
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    p[i].x = pack2(from_f<T>(v[8 * i + 0]), from_f<T>(v[8 * i + 1]));
    p[i].y = pack2(from_f<T>(v[8 * i + 2]), from_f<T>(v[8 * i + 3]));
    p[i].z = pack2(from_f<T>(v[8 * i + 4]), from_f<T>(v[8 * i + 5]));
    p[i].w = pack2(from_f<T>(v[8 * i + 6]), from_f<T>(v[8 * i + 7]));
  }
}
// this thread's row of a staging sub-tile; SWIZZLE_32B: 16-byte chunk index ^= address bit 7
__device__ __forceinline__ void stage_row16(unsigned char* sub, int r, const uint4* p) {
  const int sw = (r >> 2) & 1;
  unsigned char* row = sub + r * 32;
  *reinterpret_cast<uint4*>(row + ((0 ^ sw) << 4)) = p[0];
  *reinterpret_cast<uint4*>(row + ((1 ^ sw) << 4)) = p[1];
}
// the stores issued so far have read their staging sub-tiles
__device__ __forceinline__ void wg_staging_wait(int r) {
  if ((r >> 5) == 0) {
    if (elect_one_sync()) tma_store_wait_read<0>();
    __syncwarp();
  }
}
// TMA store of the NS sub-tiles staged at stg to columns [c0, c0 + 16 NS) of rows [row0, row0 + 128)
template <int NS> __device__ __forceinline__ void wg_store_staged(const CUtensorMap* tm, unsigned char* stg, int r, int c0, int row0) {
  if ((r >> 5) == 0) {
    if (elect_one_sync()) {
#pragma unroll
      for (int s = 0; s < NS; ++s) tma_store_2d(tm, stg + s * GT_OUT_SUB_BYTES, c0 + 16 * s, row0);
      tma_store_commit();
    }
    __syncwarp();
  }
}
// one step through a single staging sub-tile: wait for the previous store to have read it, stage, store
__device__ __forceinline__ void stage_store16(const CUtensorMap* tm, unsigned char* stg, int r, int wg, const uint4* p, int c0, int row0) {
  wg_staging_wait(r);
  wg_bar_sync(1 + wg);
  stage_row16(stg, r, p);
  fence_proxy_async();
  wg_bar_sync(1 + wg);
  wg_store_staged<1>(tm, stg, r, c0, row0);
}

// All FOUR epilogue warpgroups drain every tile, warpgroup wg columns [wg * BN/4, +BN/4) in 16-column steps
// (the next tcgen05.ld is in flight while the current step is computed), so the epilogue of tile i takes a quarter
// of a warpgroup-per-half schedule and runs under the mainloop of tile i+1 (other accumulator buffer).
// trow: TMEM address of this thread's row at the warpgroup's first column; stg_wg: NSTG x 4 KB of staging, either
//   NSTG = BN/64 (gemm_tc): a sub-tile per step; one wait for the previous tile's stores, one barrier before the first
//                write, all stores after the last step
//   NSTG = 1     (gemm_bres, whose shared memory is full): every step waits for the previous step's store and stores
// stamps (null, or gemm_tc's timeline slots [170..175]): [0] staging free, [1] first sub-tile computed, [2] barrier
// passed, [3] last sub-tile staged, [4] proxy fence done, [5] all sub-tiles staged
template <typename T, int BN, int F, int NSTG>
__device__ __forceinline__ void gt_epilogue_tma(const CUtensorMap* tmC, uint32_t trow, int row0, int col0, int r, int wg,
                                                unsigned char* stg_wg, const float* bias_s, uint64_t* tempty,
                                                long long* stamps) {
  constexpr int CW = BN / 4;
  constexpr int NSUB = CW / 16;
  static_assert(CW % 16 == 0 && NSUB >= 1, "TMA-store epilogue needs BN to be a multiple of 64");
  static_assert(NSTG == NSUB || NSTG == 1, "staging: one sub-tile per step, or a single one");
  constexpr bool ALL = NSTG == NSUB;
  uint32_t raw[2][16];
  tmem_ld16_nowait(trow, raw[0]);
  if (ALL) wg_staging_wait(r);                                // the previous tile's stores have read the staging
  if (stamps) stamps[0] = clock64();
#pragma unroll
  for (int s = 0; s < NSUB; ++s) {
    tmem_ld_wait_all();
    if (s + 1 < NSUB) tmem_ld16_nowait(trow + 16 * (s + 1), raw[(s + 1) & 1]);
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(raw[s & 1][i]);
    if (F & EF_BIAS) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 b = *reinterpret_cast<const float4*>(bias_s + 16 * s + 4 * i);   // warp-wide broadcast
        add2_f32(v[4 * i], v[4 * i + 1], b.x, b.y);
        add2_f32(v[4 * i + 2], v[4 * i + 3], b.z, b.w);
      }
    }
    if (F & EF_GELU) {
#pragma unroll
      for (int i = 0; i < 8; ++i) gelu_poly2(v[2 * i], v[2 * i + 1], v[2 * i], v[2 * i + 1]);
    }
    if (F & EF_RELU) {
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.f);
    }
    uint4 p[2];
    pack16<T>(v, p);
    if (ALL) {
      if (s == 0) {
        if (stamps) stamps[1] = clock64();
        wg_bar_sync(1 + wg);                                  // staging free (warp 0 has passed its wait above)
        if (stamps) stamps[2] = clock64();
      }
      stage_row16(stg_wg + s * GT_OUT_SUB_BYTES, r, p);
    }
    if (s + 1 == NSUB) {
      // every tcgen05.ld of this thread has completed: hand the accumulator back before the stores
      fence_before_sync();
      mbar_arrive(tempty);
    }
    if (!ALL) stage_store16(tmC, stg_wg, r, wg, p, col0 + 16 * s, row0);
  }
  if (ALL) {
    if (stamps) stamps[3] = clock64();
    fence_proxy_async();
    if (stamps) stamps[4] = clock64();
    wg_bar_sync(1 + wg);
    if (stamps) stamps[5] = clock64();
    wg_store_staged<NSUB>(tmC, stg_wg, r, col0, row0);
  }
}

// MMA issuer of one tile: all 32 lanes of warp 1 wait on the barriers and build the descriptors, the elected `leader`
// issues tcgen05.mma / tcgen05.commit (see elect_one_sync in tc_common.cuh).  Waits for the epilogue to have drained
// accumulator `acc` (tempty), then per k-block waits for its ring stage, issues BK/16 MMAs (M = 128, N) and releases
// the stage (empty_bar) once they have read it; finally hands the accumulator to the epilogue (tfull).  ab(s, kb)
// returns the shared-memory addresses of the A and B tiles of k-block kb (ring stage s).  kc counts the k-blocks of
// the whole kernel (ring position); it counts the tiles of this CTA.  tm_: optional timeline (slot table of
// gemm_tc_kernel).
template <typename T, int N, int BK, typename AB>
__device__ __forceinline__ void mma_tile(uint32_t leader, uint32_t acc, uint64_t* tempty, uint64_t* tfull, uint64_t* full_bar,
                                         uint64_t* empty_bar, int stages, int kblocks, uint32_t& kc, uint32_t it, AB ab,
                                         long long* tm_) {
  constexpr uint32_t idesc = make_idesc<T>(GT_BM, N, 0);
  constexpr uint32_t SBO = 8 * BK * 2;                      // 8-row swizzle atom of BK * 2-byte rows
  constexpr uint32_t SWZ = (BK == 64) ? SWZ_128B : SWZ_64B;
  mbar_wait(tempty, ((it >> 1) & 1) ^ 1);
  fence_after_sync();
  if (tm_ && leader && it < 20) tm_[8 + 4 * it] = clock64();
  for (int kb = 0; kb < kblocks; ++kb, ++kc) {
    const int s = kc % stages;
    if (tm_ && leader && it == 4 && kb < 30) tm_[200 + kb] = clock64();   // [200+kb]: before the wait for k-block kb
    mbar_wait(&full_bar[s], (kc / stages) & 1);
    fence_after_sync();
    if (tm_ && leader && it == 4 && kb < 30) tm_[130 + kb] = clock64();
    const uint2 op = ab(s, kb);
    const uint64_t adesc = make_smem_desc(op.x, SBO, 16, SWZ);
    const uint64_t bdesc = make_smem_desc(op.y, SBO, 16, SWZ);
    if (leader) {
#pragma unroll
      for (int k = 0; k < BK / 16; ++k) {
        // advance 16 elements (32 bytes) along K inside the swizzle atom: +2 in the >>4 address field
        mma_ss(acc, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) ? 1u : 0u);
      }
      mma_commit(&empty_bar[s]);  // stage reusable once these MMAs have read it
    }
    __syncwarp();
  }
  if (leader) mma_commit(tfull);    // accumulator complete
  if (tm_ && leader && it < 20) tm_[9 + 4 * it] = clock64();
  __syncwarp();
}

template <typename T, int BN, int BK, bool CONV>
__global__ void __launch_bounds__(GT_THREADS, 1) gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                const __grid_constant__ CUtensorMap tmB,
                                                                const __grid_constant__ CUtensorMap tmC, Epi e, int M,
                                                                int N, int K, int stages, ConvTile ct, int n_tiles,
                                                                int total_tiles) {
  pdl_launch();   // PDL: the next kernel of the stream may start its prologue (common.cuh)
  constexpr uint32_t ROW_BYTES = BK * 2;                    // 128 (BK=64) or 64 (BK=32)
  constexpr uint32_t A_BYTES = GT_BM * ROW_BYTES;
  constexpr uint32_t B_BYTES = BN * ROW_BYTES;
  constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr uint32_t TMEM_COLS = gt_tmem_cols<BN>();
  static_assert(BN % 32 == 0 && BN >= 32 && BN <= 256, "BN must be a multiple of 32 in [32,256]");

  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  // ring stages (multiples of 1 KB) | epilogue staging 64 KB (1 KB aligned: TMA-store source) | bias slices | barriers
  uint32_t* stg_base = reinterpret_cast<uint32_t*>(smem + (size_t)stages * STAGE_BYTES);   // 16 warps x GT_STG_WORDS
  float* bias_base = reinterpret_cast<float*>(stg_base + 16 * GT_STG_WORDS);               // 16 warps x 128 floats
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(bias_base + 16 * 128);
  uint64_t* empty_bar = full_bar + stages;
  uint64_t* tfull_bar = empty_bar + stages;   // 2: accumulator buffer b complete
  uint64_t* tempty_bar = tfull_bar + 2;       // 2: accumulator buffer b drained by its epilogue warpgroup
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kblocks = K / BK;
  // optional timeline (first 4 CTAs, 256 slots each): [0] entry, [1] setup done; per tile i < 20:
  // [8+4i] MMA: accumulator free (tempty wait done), [9+4i] MMA: last k-block issued, [10+4i] epilogue wg0/wg1: accumulator
  // complete (tfull wait done), [11+4i] epilogue wg0/wg1: tile stored; [100+i] producer: last load of tile i issued;
  // [130+kb] MMA: k-block kb of tile 4 ready (full_bar wait done)
  long long* tm_ = (e.tim && blockIdx.x < 4) ? e.tim + blockIdx.x * 256 : nullptr;
  if (tm_ && threadIdx.x == 0) tm_[0] = clock64();

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (e.kind >= 0 && (e.kind & EF_TMA_OUT)) tma_prefetch_desc(&tmC);
    for (int s = 0; s < stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], (!CONV && e.kind >= 0 && (e.kind & EF_TMA_OUT)) ? 512 : 256);   // TMA-store mode: all four warpgroups drain every tile
    }
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();     // PDL: everything above ran under the previous kernel's tail; its results are visible from here
  if (tm_ && threadIdx.x == 0) tm_[1] = clock64();

  if (warp == 0) {
    if (lane == 0) {
      const int cblocks = CONV ? ct.C / BK : 1;
      uint32_t kc = 0;  // k-blocks issued so far (ring position)
      int ti = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++ti) {
        const int tile_n = tile % n_tiles, tile_m = tile / n_tiles;
        int cf = 0, y0 = 0, x0 = 0;
        if (CONV) {
          const int per = ct.tiles_y * ct.tiles_x;
          cf = tile_m / per;
          const int r = tile_m - cf * per;
          const int tyi = r / ct.tiles_x;
          y0 = tyi * ct.th;
          x0 = (r - tyi * ct.tiles_x) * ct.tw;
        }
        for (int kb = 0; kb < kblocks; ++kb, ++kc) {
          const int s = kc % stages;
          mbar_wait(&empty_bar[s], ((kc / stages) & 1) ^ 1);
          unsigned char* sa = smem + (size_t)s * STAGE_BYTES;
          mbar_expect_tx(&full_bar[s], STAGE_BYTES);
          if (CONV) {
            const int tap = kb / cblocks;
            const int c0 = (kb - tap * cblocks) * BK;
            const int ky = tap / 3, kx = tap - ky * 3;
            tma_load_4d(sa, &tmA, &full_bar[s], c0, x0 + kx - 1, y0 + ky - 1, cf);
          } else {
            // L2 prefetch of the A k-block GT_PF_KB steps ahead (same tile, or the head of this CTA's next tile)
            {
              int pk = kb + GT_PF_KB, pt = tile;
              if (pk >= kblocks) { pk -= kblocks; pt += gridDim.x; }
              if (pk < kblocks && pt < total_tiles) tma_prefetch_2d(&tmA, pk * BK, (pt / n_tiles) * GT_BM);
            }
            tma_load_2d(sa, &tmA, &full_bar[s], kb * BK, tile_m * GT_BM);
          }
          tma_load_2d(sa + A_BYTES, &tmB, &full_bar[s], kb * BK, tile_n * BN);
        }
        if (tm_ && ti < 20) tm_[100 + ti] = clock64();
      }
    }
  } else if (warp == 1) {
    const uint32_t leader = elect_one_sync();
    const auto ab = [&](int s, int) {
      const uint32_t sa = smem_u32(smem + (size_t)s * STAGE_BYTES);
      return make_uint2(sa, sa + A_BYTES);
    };
    uint32_t kc = 0, it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const uint32_t b = it & 1;
      mma_tile<T, BN, BK>(leader, tmem_base + b * BN, &tempty_bar[b], &tfull_bar[b], full_bar, empty_bar, stages, kblocks, kc, it, ab, tm_);
    }
  } else if (warp >= 4) {
    // epilogue warpgroups 0..3: accumulator buffer g = wg & 1, column half = wg >> 1;
    // warp w may touch TMEM lanes [32*(w%4), +32)
    const uint32_t wg = (warp - 4) >> 2;
    const uint32_t g = wg & 1;
    const int half = wg >> 1;
    const int q = warp & 3;
    const int r = q * 32 + lane;  // row inside the tile
    uint32_t it = 0;
    const bool tma_out = !CONV && e.kind >= 0 && (e.kind & EF_TMA_OUT);
    if constexpr (!CONV && BN % 64 == 0) {
      if (tma_out) {
        // ---- TMA-store mode: warpgroup wg drains columns [wg * BN/4, +BN/4) of EVERY tile ----
        constexpr int CW = BN / 4;
        unsigned char* stg_wg = reinterpret_cast<unsigned char*>(stg_base) + wg * ((CW / 16) * GT_OUT_SUB_BYTES);
        float* bias_s = bias_base + (warp - 4) * 128;
        const int kind = e.kind & ~EF_TMA_OUT;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
          const uint32_t b = it & 1;
          const int tile_n = tile % n_tiles, tile_m = tile / n_tiles;
          if (kind & EF_BIAS) {
            __syncwarp();
            if (lane < CW) bias_s[lane] = __ldg(e.bias + tile_n * BN + wg * CW + lane);
            if (CW > 32 && lane + 32 < CW) bias_s[lane + 32] = __ldg(e.bias + tile_n * BN + wg * CW + lane + 32);
            __syncwarp();
          }
          mbar_wait(&tfull_bar[b], (it >> 1) & 1);
          fence_after_sync();
          const bool stamp = tm_ && wg == 0 && q == 0 && lane == 0 && it < 20;
          if (stamp) tm_[10 + 4 * it] = clock64();
          const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + b * BN + wg * CW;
          const int row0 = tile_m * GT_BM, col0 = tile_n * BN + wg * CW;
          long long* st = (stamp && it == 5) ? tm_ + 170 : nullptr;   // [170..175]: phases of tile 5 (see gt_epilogue_tma)
          switch (kind) {
#define EDV_TMA_CASE(F_) case F_: gt_epilogue_tma<T, BN, F_, BN / 64>(&tmC, trow, row0, col0, r, wg, stg_wg, bias_s, &tempty_bar[b], st); break;
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
    }
    if (!tma_out) {
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      if ((it & 1) != g) continue;
      const int tile_n = tile % n_tiles, tile_m = tile / n_tiles;
      long long m, orow;
      bool valid;
      if (CONV) {
        const int per = ct.tiles_y * ct.tiles_x;
        const int cf = tile_m / per;
        const int rr = tile_m - cf * per;
        const int tyi = rr / ct.tiles_x;
        const int dy = r / ct.tw, dx = r - dy * ct.tw;
        const int y = tyi * ct.th + dy, x = (rr - tyi * ct.tiles_x) * ct.tw + dx;
        valid = (y < ct.H) && (x < ct.W);
        m = ((long long)cf * ct.H + y) * ct.W + x;
        orow = m;
      } else {
        m = (long long)tile_m * GT_BM + r;
        valid = m < M;
        orow = epi_row(e, m);
      }
      // stage this warp's bias slice (columns [half*BN/2, +BN/2) of the tile) while the mainloop runs.  At BN = 32
      // warpgroup half 0 drains all columns and half 1 returns without them: staging there would read bias[N, N + 32)
      // on the last n-tile.
      float* bias_s = nullptr;
      if (e.bias && e.act != ACT_GEGLU && e.act != ACT_HEAD && (BN >= 64 || half == 0)) {
        constexpr int CH0 = (BN >= 64) ? BN / 2 : BN;
        bias_s = bias_base + (warp - 4) * 128;
        __syncwarp();
#pragma unroll
        for (int k = 0; k < (CH0 + 31) / 32; ++k)
          if (lane + 32 * k < CH0) bias_s[lane + 32 * k] = __ldg(e.bias + tile_n * BN + half * CH0 + lane + 32 * k);
        __syncwarp();
      }
      mbar_wait(&tfull_bar[g], (it >> 1) & 1);
      fence_after_sync();
      const bool stamp = tm_ && half == 0 && q == 0 && lane == 0 && it < 20;
      if (stamp) tm_[10 + 4 * it] = clock64();
      gt_epilogue<T, BN>(e, tmem_base + ((uint32_t)(q * 32) << 16) + g * BN, valid, m, orow, tile_n * BN, tile_n,
                         stg_base + (warp - 4) * GT_STG_WORDS, lane, half, bias_s);
      fence_before_sync();
      mbar_arrive(&tempty_bar[g]);
      if (stamp) tm_[11 + 4 * it] = clock64();
    }
    }
  }
  __syncthreads();
  if (warp == 1) {
    fence_after_sync();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

}  // namespace tc
