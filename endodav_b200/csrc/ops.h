// Host-side launcher interface shared by the translation units of the library: launch
// bookkeeping, TMA descriptor encoding, GEMM arguments, and the declarations of the launchers
// whose kernels live in their own .cu files (so that nvcc compiles them in parallel).
// Everything is stream-ordered; no allocation, no synchronisation.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <string>

#include "../../include/endodav_b200.h"
#include "launch.h"
#include "common.cuh"

namespace edv {

inline size_t dtype_size(int dtype) { return dtype == EDV_F32 ? 4 : 2; }

// ---- TMA descriptor encoding (driver entry point fetched through the runtime, so the
// library carries no link-time dependency on libcuda) --------------------------------------
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_tmapEncodeTiled get_encode_fn() {
  static PFN_tmapEncodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
  }
  return fn;
}

// rank-R tiled map over a 16-bit (or, dtype == EDV_F32, float32) tensor; dims/box innermost first; strides in bytes for dims 1..R-1
inline bool make_tmap(Launch& L, CUtensorMap* m, int dtype, const void* base, int rank, const uint64_t* dims,
                      const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes) {
  PFN_tmapEncodeTiled fn = get_encode_fn();
  if (!fn) {
    L.fail(EDV_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
    return false;
  }
  cuuint64_t gd[5];
  cuuint64_t gs[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gd[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
  }
  for (int i = 0; i < rank - 1; ++i) gs[i] = strides_bytes[i];
  CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                          : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                          : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                                : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUtensorMapDataType dt = dtype == EDV_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                           : dtype == EDV_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                              : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUresult r = fn(m, dt, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[256];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled failed (%d): rank %d dims %llu,%llu box %u,%u", (int)r, rank,
             (unsigned long long)dims[0], (unsigned long long)dims[1], box[0], box[1]);
    L.fail(EDV_ERR_CUDA, buf);
    return false;
  }
  return true;
}
// 2-D map over a row-major [outer][inner] tensor whose rows are pitch_bytes apart
inline bool make_tmap_2d(Launch& L, CUtensorMap* m, int dtype, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
                         uint32_t box_inner, uint32_t box_outer, int swizzle_bytes) {
  const uint64_t dims[2] = {inner, outer};
  const uint32_t box[2] = {box_inner, box_outer};
  return make_tmap(L, m, dtype, base, 2, dims, &pitch_bytes, box, swizzle_bytes);
}

// ---- GEMM -----------------------------------------------------------------------------------
struct GemmArgs {
  const void* A = nullptr;   // [M,K] (lda) or NHWC activation for conv
  const void* W = nullptr;   // [N,K]
  int M = 0, N = 0, K = 0;
  long long lda = 0;
  Epi e{};
  // conv (3x3, pad 1)
  bool conv = false;
  int F = 0, H = 0, Wd = 0, C = 0, stride = 1;
};

inline Epi epi_zero() {
  Epi e;
  memset(&e, 0, sizeof e);
  e.rb_div = 1;
  e.rb_mod = 1;
  return e;
}

// Epi::kind as launchers report it: the EF_* mask in hex, or -1 (generic epilogue)
inline std::string kind_label(int kind) {
  char b[16];
  if (kind < 0) snprintf(b, sizeof b, "-1");
  else snprintf(b, sizeof b, "0x%x", (unsigned)kind);
  return b;
}

inline void note_gemm(Launch& L, const GemmArgs& a, size_t es) {
  // algorithmic work: 2*M*N*K; bytes: A (conv: the activation once) + W + C once
  const double a_elems = a.conv ? (double)a.F * a.H * a.Wd * a.C : (double)a.M * a.K;
  L.note(2.0 * a.M * a.N * a.K, (a_elems + (double)a.N * a.K + (double)a.M * a.N) * es);
}

inline int num_sms() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  }
  return n;
}

// choose the conv tile shape (th*tw == 128) wasting the fewest pixels
inline void pick_conv_tile(int H, int W, int* th, int* tw) {
  const int cand[6][2] = {{8, 16}, {16, 8}, {4, 32}, {32, 4}, {2, 64}, {1, 128}};
  long long best = -1;
  for (auto& c : cand) {
    long long cover = (long long)((H + c[0] - 1) / c[0]) * c[0] * ((W + c[1] - 1) / c[1]) * c[1];
    if (best < 0 || cover < best) {
      best = cover;
      *th = c[0];
      *tw = c[1];
    }
  }
}

// ---- launchers defined in other translation units ---------------------------------------------
// gemm_tc_lin_{f16,bf16}.cu / gemm_tc_conv_{f16,bf16}.cu: tcgen05 GEMM and implicit-GEMM 3x3 conv
template <typename T> void launch_gemm_tc_lin(Launch& L, int dtype, const GemmArgs& a);
template <typename T> void launch_gemm_tc_conv(Launch& L, int dtype, const GemmArgs& a);
// gemm_tc_lin_*.cu: x += A W^T + bias (fp32, in place) fused with xn = LayerNorm(x) (gemm_ln.cuh; N = 384 only)
bool gemm_ln_supported(int dtype, int N, int K);
void gemm_ln(Launch& L, int dtype, const void* A, const void* W, const float* bias, float* x, void* xn, const float* gamma,
             const float* beta, float eps, int M, int N, int K, int do_ln, long long* tim = nullptr);
// attention.cu: spatial flash attention (tcgen05) / CUDA-core attention, temporal attention
void attention(Launch& L, int dtype, int engine, const void* qkv, void* out, int F, int S, int heads,
               long long* timeline = nullptr);
void temporal_attention(Launch& L, int dtype, const void* qkv, void* out, int B, int Tn, int hw, int C,
                        const float* rope = nullptr);
// head.cu: fused upsample -> conv3x3 -> ReLU -> 1x1 -> ReLU|sigmoid
bool head_fused_supported(int dtype, int Cin);
void head_fused(Launch& L, int dtype, const void* x, const void* w, const float* bias, const float* head_w, float* out,
                int F, int H1, int W1, int OH, int OW, int Cin, float sig_sign);

#define EDV_DISPATCH_T(dtype, ...)                      \
  do {                                                  \
    if ((dtype) == EDV_F32) { using T = float; __VA_ARGS__; } \
    else if ((dtype) == EDV_BF16) { using T = bf16; __VA_ARGS__; } \
    else { using T = f16; __VA_ARGS__; }                \
  } while (0)

inline unsigned nblk(long long n, int per) { return (unsigned)((n + per - 1) / per); }

}  // namespace edv
