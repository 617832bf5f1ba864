// Pipe-rate microbenchmarks for sm_100a that the kernel designs in DESIGN.md lean on:
//   * tcgen05.mma issue interval for the tile shapes of the flash-attention kernel (SS / TS operands,
//     N = 32..256, K-major / MN-major B, same vs alternating accumulator)
//   * MUFU ex2 throughput in f32, f16x2 and bf16x2 form, FFMA vs fma.rn.f32x2, FMNMX
//   * tcgen05.ld / tcgen05.st throughput
// Build:  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o tools/microbench tools/microbench.cu
// Run  :  tools/microbench            (prints one line per measurement; cycles are SM clocks)
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../endodav_b200/csrc/tc_common.cuh"
#include "../endodav_b200/csrc/ops.h"
#include "../endodav_b200/csrc/attention_tc.cuh"

using namespace tc;

#define CK(x)                                                                    \
  do {                                                                           \
    cudaError_t e_ = (x);                                                        \
    if (e_ != cudaSuccess) {                                                     \
      printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); \
      exit(1);                                                                   \
    }                                                                            \
  } while (0)

// ---- tcgen05.mma -----------------------------------------------------------------------------
// One CTA: thread 32 issues `groups` x 4 MMAs (K = 16 each; 4 = one 64-wide k-block), commits, waits.
// TS: A operand from TMEM (as P in the attention kernel).  BMN: B stored MN-major (as V).
// ALT: alternate between two accumulators (independent chains) instead of one.
template <int N, bool TS, bool BMN, bool ALT, int MM = 128>
__global__ void __launch_bounds__(128, 1) mma_bench(long long* out, int groups) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* sA = smem;               // 128 x 64 x 2 = 16 KB
  unsigned char* sB = smem + 16384;       // 256 x 64 x 2 = 32 KB
  uint64_t* bar = reinterpret_cast<uint64_t*>(sB + 32768);
  uint32_t* slot = reinterpret_cast<uint32_t*>(bar + 1);
  for (int i = threadIdx.x; i < (16384 + 32768) / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0;
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  fence_proxy_async();
  if (threadIdx.x < 32) tmem_alloc(slot, 512);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tm = *slot;
  if (threadIdx.x == 32) {
    constexpr uint32_t idesc = make_idesc<f16>(MM, N, BMN ? 1 : 0);
    const uint64_t adesc = make_smem_desc(smem_u32(sA), 1024, 16, SWZ_128B);
    const uint64_t bdesc = BMN ? make_smem_desc(smem_u32(sB), 1024, 1024, SWZ_128B) : make_smem_desc(smem_u32(sB), 1024, 16, SWZ_128B);
    // warm-up
    for (int k = 0; k < 4; ++k) {
      if (TS) mma_ts(tm, tm + 448 + k * 8, bdesc + (uint64_t)(BMN ? 128 * k : 2 * k), idesc, 0);
      else mma_ss(tm, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(BMN ? 128 * k : 2 * k), idesc, 0);
    }
    mma_commit(bar);
    mbar_wait(bar, 0);
    const long long t0 = clock64();
    for (int g = 0; g < groups; ++g) {
      const uint32_t d = tm + ((ALT && (g & 1)) ? 256 : 0);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (TS) mma_ts(d, tm + 448 + k * 8, bdesc + (uint64_t)(BMN ? 128 * k : 2 * k), idesc, 1);
        else mma_ss(d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(BMN ? 128 * k : 2 * k), idesc, 1);
      }
    }
    mma_commit(bar);
    mbar_wait(bar, 1);
    const long long t1 = clock64();
    out[blockIdx.x] = t1 - t0;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    fence_after_sync();
    tmem_dealloc(tm, 512);
  }
}

__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred;
}

// Same measurement with a WARP-UNIFORM issue loop: every lane of warp 1 runs the loop and only the tcgen05
// instructions are predicated on elect.sync, so the descriptors live in uniform registers (no per-MMA
// R2UR.BROADCAST / BRA.U.ANY uniformisation loop as in the single-lane version above).
template <int N, bool TS, bool BMN, bool ALT>
__global__ void __launch_bounds__(128, 1) mma_bench_uniform(long long* out, int groups) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* sA = smem;
  unsigned char* sB = smem + 16384;
  uint64_t* bar = reinterpret_cast<uint64_t*>(sB + 32768);
  uint32_t* slot = reinterpret_cast<uint32_t*>(bar + 1);
  for (int i = threadIdx.x; i < (16384 + 32768) / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0;
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  fence_proxy_async();
  if (threadIdx.x < 32) tmem_alloc(slot, 512);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tm = *slot;
  if ((threadIdx.x >> 5) == 1) {
    constexpr uint32_t idesc = make_idesc<f16>(128, N, BMN ? 1 : 0);
    const uint64_t adesc = make_smem_desc(smem_u32(sA), 1024, 16, SWZ_128B);
    const uint64_t bdesc = BMN ? make_smem_desc(smem_u32(sB), 1024, 1024, SWZ_128B) : make_smem_desc(smem_u32(sB), 1024, 16, SWZ_128B);
    const uint32_t leader = elect_one();
    if (leader) {
      for (int k = 0; k < 4; ++k) {
        if (TS) mma_ts(tm, tm + 448 + k * 8, bdesc + (uint64_t)(BMN ? 128 * k : 2 * k), idesc, 0);
        else mma_ss(tm, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(BMN ? 128 * k : 2 * k), idesc, 0);
      }
      mma_commit(bar);
    }
    __syncwarp();
    mbar_wait(bar, 0);
    const long long t0 = clock64();
    for (int g = 0; g < groups; ++g) {
      const uint32_t d = tm + ((ALT && (g & 1)) ? 256 : 0);
      if (leader) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (TS) mma_ts(d, tm + 448 + k * 8, bdesc + (uint64_t)(BMN ? 128 * k : 2 * k), idesc, 1);
          else mma_ss(d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(BMN ? 128 * k : 2 * k), idesc, 1);
        }
      }
      __syncwarp();
    }
    if (leader) mma_commit(bar);
    __syncwarp();
    mbar_wait(bar, 1);
    const long long t1 = clock64();
    if (leader) out[blockIdx.x] = t1 - t0;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    fence_after_sync();
    tmem_dealloc(tm, 512);
  }
}

// ---- what slows tcgen05.mma down inside a real kernel? --------------------------------------------------------------
// The MMA stream of a GEMM mainloop (M = 128, N = 192, SS operands, warp-uniform issue) measured (a) alone, (b) while
// 16 other warps read a second accumulator with tcgen05.ld (the epilogue), (c) while a producer thread streams bulk
// copies into other shared-memory stages (the TMA ring), (d) both.
template <int N>
__global__ void __launch_bounds__(640, 1) mma_contention(long long* out, int groups, int with_ld, int with_copy, const unsigned char* gsrc) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* sA = smem;                 // 16 KB
  unsigned char* sB = smem + 16384;         // 32 KB
  unsigned char* sC = smem + 49152;         // 3 x 40 KB copy targets
  uint64_t* bar = reinterpret_cast<uint64_t*>(sC + 3 * 40960);
  uint64_t* cbar = bar + 1;                 // 3 copy barriers
  uint32_t* slot = reinterpret_cast<uint32_t*>(cbar + 3);
  volatile int* stop = reinterpret_cast<volatile int*>(slot + 1);
  for (int i = threadIdx.x; i < 49152 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0;
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    for (int i = 0; i < 3; ++i) mbar_init(&cbar[i], 1);
    *stop = 0;
    fence_barrier_init();
  }
  fence_proxy_async();
  const int warp = threadIdx.x >> 5;
  if (warp == 1) tmem_alloc(slot, 512);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tm = *slot;
  if (warp == 1) {
    constexpr uint32_t idesc = make_idesc<f16>(128, N, 0);
    const uint64_t adesc = make_smem_desc(smem_u32(sA), 1024, 16, SWZ_128B);
    const uint64_t bdesc = make_smem_desc(smem_u32(sB), 1024, 16, SWZ_128B);
    const uint32_t leader = elect_one();
    const long long t0 = clock64();
    for (int g = 0; g < groups; ++g) {
      if (leader) {
#pragma unroll
        for (int k = 0; k < 4; ++k) mma_ss(tm, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, 1);
      }
      __syncwarp();
    }
    if (leader) mma_commit(bar);
    __syncwarp();
    mbar_wait(bar, 0);
    const long long t1 = clock64();
    if (leader) out[blockIdx.x] = t1 - t0;
    *stop = 1;
  } else if (warp == 0) {
    if (with_copy && threadIdx.x == 0) {
      // stream 40 KB bulk copies global (L2 resident) -> shared, three in flight, until the MMA warp is done
      uint32_t n = 0;
      while (!*stop) {
        const uint32_t s = n % 3;
        if (n >= 3) mbar_wait(&cbar[s], ((n / 3) - 1) & 1);
        mbar_expect_tx(&cbar[s], 40960);
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sC + s * 40960)),
                     "l"(gsrc + (size_t)((blockIdx.x * 7 + n) % 64) * 40960), "r"(40960), "r"(smem_u32(&cbar[s]))
                     : "memory");
        ++n;
      }
      for (uint32_t i = (n > 3 ? n - 3 : 0); i < n; ++i) mbar_wait(&cbar[i % 3], (i / 3) & 1);
      out[1024 + blockIdx.x] = n;
    }
  } else if (warp >= 4 && with_ld) {
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    float acc = 0.f;
    while (!*stop) {
      float v[16];
      tmem_ld16(tm + lane_off + 256 + ((warp - 4) >> 2) * 48, v);
      acc += v[0];
    }
    if (acc == 12345.f) out[2048] = 1;
  }
  __syncthreads();
  if (warp == 1) {
    fence_after_sync();
    tmem_dealloc(tm, 512);
  }
}

// ---- per-k-block bookkeeping of a GEMM mainloop: which part is not hidden behind the MMAs? -------------------------
// groups of 4 MMAs (N = 192) with, per group: bit0 tcgen05.commit to an mbarrier, bit1 a wait on an already completed
// mbarrier, bit2 tcgen05.fence::after_thread_sync, bit3 rebuilding the two shared-memory descriptors, bit4 the
// accumulator alternates between TMEM columns 0 and 192 every 6 groups, bit5 the operands rotate over 4 A stages and
// 6 resident B k-blocks (212 KB footprint, as in gemm_bres_kernel).
__global__ void __launch_bounds__(128, 1) mma_loop_overheads(long long* out, int groups, int mode) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* sA = smem;                 // 4 x 16 KB
  unsigned char* sB = smem + 65536;         // 6 x 24 KB
  uint64_t* bar = reinterpret_cast<uint64_t*>(sB + 6 * 24576);
  uint64_t* done_bar = bar + 1;     // completed once: waits with parity 0 succeed immediately
  uint64_t* sink_bar = bar + 2;     // receives the per-group commits
  uint32_t* slot = reinterpret_cast<uint32_t*>(bar + 4);
  for (int i = threadIdx.x; i < (65536 + 6 * 24576) / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0;
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    mbar_init(done_bar, 1);
    mbar_init(sink_bar, 1);
    fence_barrier_init();
    mbar_arrive(done_bar);
  }
  fence_proxy_async();
  if (threadIdx.x < 32) tmem_alloc(slot, 512);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tm = *slot;
  if ((threadIdx.x >> 5) == 1) {
    constexpr uint32_t idesc = make_idesc<f16>(128, 192, 0);
    const uint32_t leader = elect_one();
    const uint32_t a_addr = smem_u32(sA), b_addr = smem_u32(sB);
    uint64_t adesc = make_smem_desc(a_addr, 1024, 16, SWZ_128B);
    uint64_t bdesc = make_smem_desc(b_addr, 1024, 16, SWZ_128B);
    const long long t0 = clock64();
    for (int g = 0; g < groups; ++g) {
      if (mode & 2) mbar_wait(done_bar, 0);
      if (mode & 4) fence_after_sync();
      if (mode & 8) {
        adesc = make_smem_desc(a_addr + ((mode & 32) ? (g & 3) * 16384 : 0), 1024, 16, SWZ_128B);
        bdesc = make_smem_desc(b_addr + ((mode & 32) ? (g % 6) * 24576 : 0), 1024, 16, SWZ_128B);
      }
      const uint32_t d = tm + (((mode & 16) && ((g / 6) & 1)) ? 192 : 0);
      if (leader) {
#pragma unroll
        for (int k = 0; k < 4; ++k) mma_ss(d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, 1);
        if (mode & 1) mma_commit(sink_bar);
      }
      __syncwarp();
    }
    if (leader) mma_commit(bar);
    __syncwarp();
    mbar_wait(bar, 0);
    const long long t1 = clock64();
    if (leader) out[blockIdx.x] = t1 - t0;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    fence_after_sync();
    tmem_dealloc(tm, 512);
  }
}

template <int N, bool TS, bool BMN, bool ALT> void run_mma_u(const char* what, long long* d_out, int nblocks) {
  auto kern = mma_bench_uniform<N, TS, BMN, ALT>;
  const int smem = 1024 + 16384 + 32768 + 64;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  const int groups = 256;
  kern<<<nblocks, 128, smem>>>(d_out, groups);
  CK(cudaDeviceSynchronize());
  std::vector<long long> h(nblocks);
  CK(cudaMemcpy(h.data(), d_out, nblocks * sizeof(long long), cudaMemcpyDeviceToHost));
  double s = 0;
  for (long long v : h) s += (double)v;
  const double per = s / nblocks / (groups * 4);
  printf("mma-uniform %-26s N=%3d ctas=%3d: %7.1f cycles / MMA (M=128,K=16)  -> %6.0f MAC/cycle/SM\n", what, N, nblocks, per,
         128.0 * N * 16 / per);
}

// M = 64 instructions (the "weights as A, pixels as B" formulation of the 64-channel convolutions)
template <int N, int MM> void run_mma_m(const char* what, long long* d_out, int nblocks) {
  const int groups = 512;
  auto kern = mma_bench<N, false, false, false, MM>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 1024 + 16384 + 32768 + 64));
  kern<<<nblocks, 128, 1024 + 16384 + 32768 + 64>>>(d_out, groups);
  CK(cudaDeviceSynchronize());
  std::vector<long long> h(nblocks);
  CK(cudaMemcpy(h.data(), d_out, nblocks * sizeof(long long), cudaMemcpyDeviceToHost));
  double s = 0;
  for (long long v : h) s += (double)v;
  const double per = s / nblocks / (groups * 4);
  printf("mma %-26s M=%3d N=%3d ctas=%3d: %7.1f cycles / MMA (K=16)  -> %6.0f MAC/cycle/SM\n", what, MM, N, nblocks, per, (double)MM * N * 16 / per);
}

template <int N, bool TS, bool BMN, bool ALT> void run_mma(const char* what, long long* d_out, int nblocks) {
  auto kern = mma_bench<N, TS, BMN, ALT>;
  const int smem = 1024 + 16384 + 32768 + 64;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  const int groups = 256;
  kern<<<nblocks, 128, smem>>>(d_out, groups);
  CK(cudaDeviceSynchronize());
  std::vector<long long> h(nblocks);
  CK(cudaMemcpy(h.data(), d_out, nblocks * sizeof(long long), cudaMemcpyDeviceToHost));
  double s = 0;
  for (long long v : h) s += (double)v;
  const double per = s / nblocks / (groups * 4);
  printf("mma %-34s N=%3d ctas=%3d: %7.1f cycles / MMA (M=128,K=16)  -> %6.0f MAC/cycle/SM\n", what, N, nblocks, per,
         128.0 * N * 16 / per);
}

// ---- ALU / MUFU pipes ---------------------------------------------------------------------------
enum { OP_EX2_F32 = 0, OP_EX2_F16X2 = 1, OP_EX2_BF16X2 = 2, OP_FFMA = 3, OP_FFMA2 = 4, OP_FMNMX = 5, OP_CVT_F16X2 = 6, OP_FADD = 7 };

template <int OP> __global__ void __launch_bounds__(1024) pipe_bench(float* out, long long* cyc, int iters) {
  constexpr int U = 8;
  float x[U];
  uint32_t h[U];
  unsigned long long p[U];
#pragma unroll
  for (int j = 0; j < U; ++j) {
    x[j] = -0.001f * (threadIdx.x + j);
    h[j] = 0xb800b400u + j;                 // two small negative halves
    p[j] = ((unsigned long long)__float_as_uint(0.999f) << 32) | __float_as_uint(0.998f);
  }
  const unsigned long long cst = ((unsigned long long)__float_as_uint(1e-9f) << 32) | __float_as_uint(1e-9f);
  __syncthreads();
  const long long t0 = clock64();
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int j = 0; j < U; ++j) {
      if (OP == OP_EX2_F32) asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(x[j]));
      if (OP == OP_EX2_F16X2) asm volatile("ex2.approx.f16x2 %0, %0;" : "+r"(h[j]));
      if (OP == OP_EX2_BF16X2) asm volatile("ex2.approx.ftz.bf16x2 %0, %0;" : "+r"(h[j]));
      if (OP == OP_FFMA) asm volatile("fma.rn.f32 %0, %0, %1, %2;" : "+f"(x[j]) : "f"(0.999f), "f"(1e-9f));
      if (OP == OP_FFMA2) asm volatile("fma.rn.f32x2 %0, %0, %1, %2;" : "+l"(p[j]) : "l"(p[(j + 1) % U]), "l"(cst));
      if (OP == OP_FMNMX) asm volatile("max.f32 %0, %0, %1;" : "+f"(x[j]) : "f"(x[(j + 1) % U]));
      if (OP == OP_CVT_F16X2) asm volatile("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(h[j]) : "f"(x[j]), "f"(x[(j + 1) % U]));
      if (OP == OP_FADD) asm volatile("add.f32 %0, %0, %1;" : "+f"(x[j]) : "f"(1e-9f));
    }
  }
  const long long t1 = clock64();
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < U; ++j) s += x[j] + __uint_as_float(h[j]) + __uint_as_float((uint32_t)p[j]);
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
  if (threadIdx.x == 0) cyc[blockIdx.x] = t1 - t0;
}

template <int OP> void run_pipe(const char* what, float* d_f, long long* d_out, int warps) {
  const int iters = 2048;
  pipe_bench<OP><<<1, warps * 32>>>(d_f, d_out, iters);
  CK(cudaDeviceSynchronize());
  long long c;
  CK(cudaMemcpy(&c, d_out, sizeof c, cudaMemcpyDeviceToHost));
  const double instr_per_smsp = (double)iters * 8 * warps / 4.0;
  printf("pipe %-16s warps/SM=%2d: %6.2f cycles per warp-instruction per SMSP  (%5.1f lanes/clk/SM)\n", what, warps,
         (double)c / instr_per_smsp, 32.0 * 4 * instr_per_smsp / (double)c);
}


// ---- the exponential phase of the flash-attention softmax, as an instruction mix ---------------------------------
__device__ __forceinline__ void fma2(float& d0, float& d1, float a0, float a1, float b0, float b1, float c0, float c1) {
  uint64_t ra, rb, rc, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b0), "f"(b1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c0), "f"(c1));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d0), "=f"(d1) : "l"(rd));
}
// 2^x for a PAIR on the FMA / ALU pipes (no MUFU), packed fp32x2: x = n + f (round to nearest), degree-3 minimax
// polynomial for 2^f on [-0.5, 0.5] (max relative error 1.1e-4 < the 16-bit rounding of P: 4.9e-4 fp16,
// 3.9e-3 bf16), exponent inserted with one integer multiply-add.
__device__ __forceinline__ void ex2_poly2(float& p0, float& p1, float x0, float x1) {
  x0 = fmaxf(x0, -125.f);
  x1 = fmaxf(x1, -125.f);
  float t0 = x0, t1 = x1;
  add2(t0, t1, 12582912.f, 12582912.f);            // 1.5 * 2^23: n lands in the low mantissa bits
  float n0 = t0, n1 = t1;
  add2(n0, n1, -12582912.f, -12582912.f);
  float f0, f1;
  fma2_bcast(f0, f1, n0, n1, -1.0f, 0.f);          // -n
  add2(f0, f1, x0, x1);                            // f = x - n
  float q0, q1;
  fma2_bcast(q0, q1, f0, f1, 0.05550410866f, 0.2402265069f);
  fma2(q0, q1, q0, q1, f0, f1, 0.6931471806f, 0.6931471806f);
  fma2(q0, q1, q0, q1, f0, f1, 1.0f, 1.0f);
  p0 = __int_as_float(__float_as_int(q0) + (__float_as_int(t0) << 23));
  p1 = __int_as_float(__float_as_int(q1) + (__float_as_int(t1) << 23));
}

// Each thread owns NP pairs of scores in registers and runs, per "key block":  x = s * log2e - m (FFMA2), p = ex2(x)
// (2 MUFU), row sum (FADD2), 16-bit pack (F2FP) -- attention_tc.cuh's loop.  MODE bit 0: drop the pack, bit 1: drop the
// row sum, bit 2: every 4th pair through the FMA-pipe polynomial.  Reports cycles per MUFU warp-instruction per SMSP
// (the pipe alone: 8.0), i.e. how close this mix can get to the MUFU roofline with 1 / 2 / 4 warps per scheduler.
template <int NP, int MODE> __global__ void __launch_bounds__(512, 1) softmax_mix_bench(const float* in, float* out, long long* cyc, int iters) {
  float sv[2 * NP];
#pragma unroll
  for (int i = 0; i < 2 * NP; ++i) sv[i] = in[(threadIdx.x * 2 * NP + i) & 4095];
  float acc = 0.f;
  uint32_t px = 0;
  float neg = -1.0f;
  __syncthreads();
  const long long t0 = clock64();
  for (int it = 0; it < iters; ++it) {
    float ls0 = 0.f, ls1 = 0.f, ls2 = 0.f, ls3 = 0.f;
    uint32_t pv[NP];
#pragma unroll
    for (int i = 0; i < NP; ++i) {
      float x0, x1, p0, p1;
      fma2_bcast(x0, x1, sv[2 * i], sv[2 * i + 1], 1.4426950408889634f, neg);
      if ((MODE & 4) && (i & 3) == 3) {
        ex2_poly2(p0, p1, x0, x1);
      } else {
        p0 = ex2_approx(x0);
        p1 = ex2_approx(x1);
      }
      if (!(MODE & 2)) {
        if (i & 1) add2(ls2, ls3, p0, p1);
        else add2(ls0, ls1, p0, p1);
      } else {
        ls0 = p0; ls1 = p1;
      }
      if (!(MODE & 1)) pv[i] = pack_pair(p0, p1, f16());
      else pv[i] = __float_as_uint(p0) ^ __float_as_uint(p1);
    }
    acc += (ls0 + ls1) + (ls2 + ls3);
#pragma unroll
    for (int i = 0; i < NP; ++i) px ^= pv[i];
    neg = -1.0f - 1e-6f * (float)(px & 1);     // loop-carried: the compiler cannot hoist the block
  }
  const long long t1 = clock64();
  out[blockIdx.x * blockDim.x + threadIdx.x] = acc + __uint_as_float(px);
  if (threadIdx.x == 0) cyc[blockIdx.x] = t1 - t0;
}
template <int NP, int MODE> void run_softmax_mix(const char* what, const float* d_in, float* d_f, long long* d_out, int warps) {
  const int iters = 256;
  softmax_mix_bench<NP, MODE><<<1, warps * 32>>>(d_in, d_f, d_out, iters);
  CK(cudaDeviceSynchronize());
  long long c;
  CK(cudaMemcpy(&c, d_out, sizeof c, cudaMemcpyDeviceToHost));
  const double mufu_per_smsp = (double)iters * 2 * NP * ((MODE & 4) ? 0.75 : 1.0) * warps / 4.0;
  printf("softmax-mix %-34s pairs/thread=%2d warps/SM=%2d: %6.2f cycles per MUFU per SMSP, %7.1f cycles per key block of %d scores/thread\n", what, NP,
         warps, (double)c / mufu_per_smsp, (double)c / iters, 2 * NP);
}

// ---- tcgen05.ld / st ------------------------------------------------------------------------------
__global__ void __launch_bounds__(256, 1) tmem_bench(long long* out, float* sink, int iters, int nwarps_active) {
  __shared__ uint32_t slot;
  if (threadIdx.x < 32) tmem_alloc(&slot, 512);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tm = slot;
  const int warp = threadIdx.x >> 5;
  const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
  float acc = 0.f;
  long long t_ld = 0, t_st = 0;
  if (warp < nwarps_active) {
    float v[32];
    uint32_t r[16];
    for (int i = 0; i < 16; ++i) r[i] = i;
    for (int c = 0; c < 512; c += 16) tmem_st16(tm + lane_off + c, r);
    tmem_st_wait();
    __syncwarp();
    long long t0 = clock64();
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int c = 0; c < 128; c += 32) {
        tmem_ld32(tm + lane_off + (warp >> 2) * 128 + c, v);
        acc += v[0] + v[31];
      }
    }
    long long t1 = clock64();
    t_ld = t1 - t0;
    t0 = clock64();
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int c = 0; c < 64; c += 16) tmem_st16(tm + lane_off + 256 + (warp >> 2) * 64 + c, r);
      tmem_st_wait();
    }
    t1 = clock64();
    t_st = t1 - t0;
  }
  sink[threadIdx.x] = acc;
  if (threadIdx.x == 0) {
    out[0] = t_ld;
    out[1] = t_st;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    fence_after_sync();
    tmem_dealloc(tm, 512);
  }
}

static void run_mix_all(float* d_f, long long* d_out) {
  {
    float* d_in;
    CK(cudaMalloc(&d_in, 4096 * sizeof(float)));
    std::vector<float> hin(4096);
    for (int i = 0; i < 4096; ++i) hin[i] = -0.01f * (i % 97);
    CK(cudaMemcpy(d_in, hin.data(), 4096 * sizeof(float), cudaMemcpyHostToDevice));
    for (int w : {4, 8, 16}) {
      run_softmax_mix<64, 0>("ffma2 + 2 ex2 + fadd2 + f2fp", d_in, d_f, d_out, w);
      run_softmax_mix<64, 1>("... without the pack", d_in, d_f, d_out, w);
      run_softmax_mix<64, 2>("... without the row sum", d_in, d_f, d_out, w);
      run_softmax_mix<64, 3>("ffma2 + 2 ex2 only", d_in, d_f, d_out, w);
      run_softmax_mix<64, 4>("full mix, every 4th pair polynomial", d_in, d_f, d_out, w);
      run_softmax_mix<32, 0>("full mix", d_in, d_f, d_out, w);
      run_softmax_mix<32, 4>("full mix, every 4th pair polynomial", d_in, d_f, d_out, w);
    }
    CK(cudaFree(d_in));
  }
}

int main(int argc, char** argv) {
  const bool only_mix = argc > 1 && std::string(argv[1]) == "mix";   // tools/microbench mix: the softmax instruction mix only
  long long* d_out;
  float* d_f;
  CK(cudaMalloc(&d_out, 4096 * sizeof(long long)));
  CK(cudaMalloc(&d_f, 1 << 20));
  int sms = 0;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
  printf("SMs: %d\n", sms);
  if (argc > 1 && std::string(argv[1]) == "m64") {
    for (int nb : {1, sms}) {
      run_mma_m<32, 64>("SS K-major", d_out, nb);
      run_mma_m<64, 64>("SS K-major", d_out, nb);
      run_mma_m<128, 64>("SS K-major", d_out, nb);
      run_mma_m<256, 64>("SS K-major", d_out, nb);
      run_mma_m<64, 128>("SS K-major", d_out, nb);
      run_mma_m<128, 128>("SS K-major", d_out, nb);
      run_mma_m<256, 128>("SS K-major", d_out, nb);
    }
    printf("done\n");
    return 0;
  }
  if (only_mix) {
    run_mix_all(d_f, d_out);
    printf("done\n");
    return 0;
  }
  for (int nb : {1, sms}) {
    run_mma<32, false, false, false>("SS K-major", d_out, nb);
    run_mma<64, false, false, false>("SS K-major", d_out, nb);
    run_mma<128, false, false, false>("SS K-major", d_out, nb);
    run_mma<192, false, false, false>("SS K-major", d_out, nb);
    run_mma<256, false, false, false>("SS K-major", d_out, nb);
    run_mma<128, false, false, true>("SS K-major, alternating D", d_out, nb);
    run_mma<64, false, true, false>("SS B MN-major", d_out, nb);
    run_mma<64, true, true, false>("TS (A in TMEM) B MN-major", d_out, nb);
    run_mma<64, true, true, true>("TS B MN-major, alternating D", d_out, nb);
    run_mma<128, true, true, false>("TS (A in TMEM) B MN-major", d_out, nb);
    run_mma<64, true, false, false>("TS (A in TMEM) B K-major", d_out, nb);
  }
  for (int nb : {1, sms}) {
    run_mma_u<32, false, false, false>("SS K-major", d_out, nb);
    run_mma_u<64, false, false, false>("SS K-major", d_out, nb);
    run_mma_u<128, false, false, false>("SS K-major", d_out, nb);
    run_mma_u<256, false, false, false>("SS K-major", d_out, nb);
    run_mma_u<64, true, true, false>("TS B MN-major", d_out, nb);
    run_mma_u<64, true, true, true>("TS B MN-major, alt D", d_out, nb);
    run_mma_u<32, false, false, true>("SS K-major, alt D", d_out, nb);
  }
  {
    const int smem = 1024 + 65536 + 6 * 24576 + 128;
    CK(cudaFuncSetAttribute(mma_loop_overheads, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    for (int mode : {0, 15, 16, 8 + 32, 15 + 16 + 32}) {
      const int groups = 512;
      mma_loop_overheads<<<sms, 128, smem>>>(d_out, groups, mode);
      CK(cudaDeviceSynchronize());
      std::vector<long long> h(sms);
      CK(cudaMemcpy(h.data(), d_out, sms * sizeof(long long), cudaMemcpyDeviceToHost));
      double s = 0;
      for (long long v : h) s += (double)v;
      printf("mma-loop N=192, per group of 4:%s%s%s%s%s -> %7.1f cycles per group (MMA alone: 384)\n", mode == 0 ? " nothing" : "",
             (mode & 1) ? " commit" : "", (mode & 2) ? " wait(done)" : "", (mode & 4) ? " fence" : "", (mode & 8) ? " descriptors" : "",
             s / sms / groups);
      if (mode & 48) printf("      (+%s%s)\n", (mode & 16) ? " accumulator alternates between columns 0 / 192" : "", (mode & 32) ? " operands rotate over 4 A stages x 6 B blocks" : "");
    }
  }
  {
    unsigned char* gsrc;
    CK(cudaMalloc(&gsrc, 64 * 40960));
    CK(cudaMemset(gsrc, 0, 64 * 40960));
    auto kern = mma_contention<192>;
    const int smem = 1024 + 49152 + 3 * 40960 + 128;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    for (int mode = 0; mode < 4; ++mode) {
      const int groups = 512;
      CK(cudaMemset(d_out, 0, 4096 * sizeof(long long)));
      kern<<<sms, 640, smem>>>(d_out, groups, mode & 1, (mode >> 1) & 1, gsrc);
      CK(cudaDeviceSynchronize());
      std::vector<long long> h(2048);
      CK(cudaMemcpy(h.data(), d_out, 2048 * sizeof(long long), cudaMemcpyDeviceToHost));
      double s = 0, c = 0;
      for (int i = 0; i < sms; ++i) { s += (double)h[i]; c += (double)h[1024 + i]; }
      printf("mma-contention N=192 SS, %s%s: %7.1f cycles / MMA;  bulk copies per CTA %.0f (%.1f B/cycle/SM into smem)\n",
             (mode & 1) ? "16 warps tcgen05.ld " : "", (mode & 2) ? "+ 40 KB bulk copies" : ((mode & 1) ? "" : "alone"), s / sms / (groups * 4),
             c / sms, c / sms * 40960.0 / (s / sms));
    }
    CK(cudaFree(gsrc));
  }
  for (int w : {4, 8, 16}) {
    run_pipe<OP_EX2_F32>("ex2.f32", d_f, d_out, w);
    run_pipe<OP_EX2_F16X2>("ex2.f16x2", d_f, d_out, w);
    run_pipe<OP_EX2_BF16X2>("ex2.bf16x2", d_f, d_out, w);
    run_pipe<OP_FFMA>("fma.f32", d_f, d_out, w);
    run_pipe<OP_FFMA2>("fma.f32x2", d_f, d_out, w);
    run_pipe<OP_FMNMX>("max.f32", d_f, d_out, w);
    run_pipe<OP_CVT_F16X2>("cvt.f16x2.f32", d_f, d_out, w);
    run_pipe<OP_FADD>("add.f32", d_f, d_out, w);
  }
  run_mix_all(d_f, d_out);
  for (int w : {4, 8}) {
    const int iters = 512;
    tmem_bench<<<1, 256>>>(d_out, d_f, iters, w);
    CK(cudaDeviceSynchronize());
    long long c[2];
    CK(cudaMemcpy(c, d_out, sizeof c, cudaMemcpyDeviceToHost));
    printf("tmem warps=%d: ld 128 cols x 32 lanes: %.1f cycles per warp (%.1f B/cycle/SM);  st 64 cols + wait: %.1f cycles per warp (%.1f B/cycle/SM)\n",
           w, (double)c[0] / iters, (double)w * 128 * 32 * 4 * iters / c[0], (double)c[1] / iters, (double)w * 64 * 32 * 4 * iters / c[1]);
  }
  printf("done\n");
  return 0;
}
