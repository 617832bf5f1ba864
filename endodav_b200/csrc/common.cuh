// Shared device helpers: element types, vector load/store, epilogue description.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

typedef __nv_bfloat16 bf16;
typedef __half f16;

// ---------------------------------------------------------------------------------------
// element conversion
// ---------------------------------------------------------------------------------------
// ---- programmatic dependent launch (PDL) --------------------------------------------------------------------------
// Every kernel of the forward starts with pdl_launch() -- "the next kernel of the stream may be scheduled now" -- and
// calls pdl_wait() before its first access to global memory: the wait returns when the PREVIOUS kernel of the stream
// has completed and its writes are visible.  The next kernel's CTAs therefore become resident, run their prologue
// (barrier init, TMEM allocation, tensor-map prefetch, index arithmetic) under the tail of the current one, and the
// ~2-3 us launch gap between dependent kernels disappears.  Both are no-ops in a kernel launched without the
// cudaLaunchAttributeProgrammaticStreamSerialization attribute (launch.h: launch_k).
__device__ __forceinline__ void pdl_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename T> __device__ __forceinline__ float to_f(T v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<bf16>(bf16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f<f16>(f16 v) { return __half2float(v); }

template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f<bf16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ f16 from_f<f16>(float v) { return __float2half_rn(v); }

__device__ __forceinline__ uint32_t pack2(bf16 a, bf16 b) {
  __nv_bfloat162 t = __halves2bfloat162(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ uint32_t pack2(f16 a, f16 b) {
  __half2 t = __halves2half2(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}

// load NV consecutive elements as float; pointer must be aligned to NV*sizeof(T) when
// NV*sizeof(T) is 8 or 16 bytes (all call sites guarantee it: leading dims are multiples of 8).
template <typename T, int NV> __device__ __forceinline__ void load_vec(const T* __restrict__ p, float* v) {
  if constexpr (sizeof(T) == 4) {
    if constexpr (NV % 4 == 0) {
#pragma unroll
      for (int i = 0; i < NV / 4; ++i) {
        float4 t = reinterpret_cast<const float4*>(p)[i];
        v[4 * i + 0] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < NV; ++i) v[i] = to_f<T>(p[i]);
    }
  } else {
    if constexpr (NV % 8 == 0) {
#pragma unroll
      for (int i = 0; i < NV / 8; ++i) {
        uint4 t = reinterpret_cast<const uint4*>(p)[i];
        const T* e = reinterpret_cast<const T*>(&t);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[8 * i + j] = to_f<T>(e[j]);
      }
    } else if constexpr (NV % 4 == 0) {
#pragma unroll
      for (int i = 0; i < NV / 4; ++i) {
        uint2 t = reinterpret_cast<const uint2*>(p)[i];
        const T* e = reinterpret_cast<const T*>(&t);
#pragma unroll
        for (int j = 0; j < 4; ++j) v[4 * i + j] = to_f<T>(e[j]);
      }
    } else {
#pragma unroll
      for (int i = 0; i < NV; ++i) v[i] = to_f<T>(p[i]);
    }
  }
}

template <typename T, int NV> __device__ __forceinline__ void store_vec(T* __restrict__ p, const float* v) {
  if constexpr (sizeof(T) == 4) {
    if constexpr (NV % 4 == 0) {
#pragma unroll
      for (int i = 0; i < NV / 4; ++i)
        reinterpret_cast<float4*>(p)[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    } else {
#pragma unroll
      for (int i = 0; i < NV; ++i) p[i] = from_f<T>(v[i]);
    }
  } else {
    if constexpr (NV % 8 == 0) {
#pragma unroll
      for (int i = 0; i < NV / 8; ++i) {
        uint4 t;
        t.x = pack2(from_f<T>(v[8 * i + 0]), from_f<T>(v[8 * i + 1]));
        t.y = pack2(from_f<T>(v[8 * i + 2]), from_f<T>(v[8 * i + 3]));
        t.z = pack2(from_f<T>(v[8 * i + 4]), from_f<T>(v[8 * i + 5]));
        t.w = pack2(from_f<T>(v[8 * i + 6]), from_f<T>(v[8 * i + 7]));
        reinterpret_cast<uint4*>(p)[i] = t;
      }
    } else if constexpr (NV % 4 == 0) {
#pragma unroll
      for (int i = 0; i < NV / 4; ++i) {
        uint2 t;
        t.x = pack2(from_f<T>(v[4 * i + 0]), from_f<T>(v[4 * i + 1]));
        t.y = pack2(from_f<T>(v[4 * i + 2]), from_f<T>(v[4 * i + 3]));
        reinterpret_cast<uint2*>(p)[i] = t;
      }
    } else {
#pragma unroll
      for (int i = 0; i < NV; ++i) p[i] = from_f<T>(v[i]);
    }
  }
}

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }

// GELU(erf) for the 16-bit paths: gelu(x) = relu(x) - 0.5 |x| P(t) exp(-x^2/2), t = 1/(1 + p|x|/sqrt2),
// P the Abramowitz-Stegun 7.1.26 erfc polynomial (|erf error| <= 1.5e-7, far below 16-bit output
// rounding); written without the 1 - erf cancellation.  2 MUFU + ~12 FMA-pipe instructions
// instead of erff()'s ~25, which matters because the fc1 epilogue is as long as its mainloop.
__device__ __forceinline__ float gelu_fast(float x) {
  const float ax = fabsf(x);
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(ax, 0.3275911f * 0.70710678118654752440f, 1.0f)));
  float p = fmaf(t, 1.061405429f, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  p *= t;
  float ex;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ex) : "f"(x * x * (-0.5f * 1.4426950408889634f)));
  return fmaf(-0.5f * ax * p, ex, fmaxf(x, 0.f));
}
#define GELU_ZA 9.182736455e-02f
#define GELU_Q0 3.027377123e-01f
#define GELU_Q1 -1.496531036e-01f
#define GELU_Q2 1.075239210e-01f
#define GELU_Q3 -8.094775278e-02f
#define GELU_Q4 5.954273902e-02f
#define GELU_Q5 -4.183582460e-02f
#define GELU_Q6 2.565362346e-02f
#define GELU_Q7 -1.271499527e-02f
#define GELU_Q8 8.149412674e-03f
#define GELU_Q9 -6.645919508e-03f
#define GELU_Q10 2.464738470e-03f
// GELU(erf) for a PAIR without MUFU, in packed fp32x2 arithmetic (FFMA2 / FMUL2; sm_100): erf(x / sqrt2) = xc * Q(xc^2)
// with xc = clamp(x, +-4.6669) (erf(3.3) = 1 - 3e-6) and Q a degree-10 minimax polynomial evaluated in
// z = xc^2 * GELU_ZA - 1 in [-1, 1] (the power basis in xc^2 itself loses 5 digits in float32); max |erf error| 3e-6
// in float32 arithmetic, far below the 16-bit output rounding.  ~9 issue slots per value instead of ~14 + 2 MUFU: the fc1 epilogue is
// issue / MUFU bound, not math bound (tools/gemm_timeline.py).
__device__ __forceinline__ void gelu_poly2(float& y0, float& y1, float x0, float x1) {
  // symmetric clamp in ONE instruction per value: min(|x|, c) with the sign of x (min.xorsign.abs, c > 0)
  float c0, c1;
  asm("min.xorsign.abs.f32 %0, %1, %2;" : "=f"(c0) : "f"(x0), "f"(4.66690475f));
  asm("min.xorsign.abs.f32 %0, %1, %2;" : "=f"(c1) : "f"(x1), "f"(4.66690475f));
  unsigned long long xc, xx, t, q, k, r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(xc) : "f"(c0), "f"(c1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(xx) : "f"(x0), "f"(x1));
  asm("mul.rn.f32x2 %0, %1, %1;" : "=l"(t) : "l"(xc));
  {
    unsigned long long za, m1;
    asm("mov.b64 %0, {%1, %1};" : "=l"(za) : "f"(GELU_ZA));
    asm("mov.b64 %0, {%1, %1};" : "=l"(m1) : "f"(-1.0f));
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(t) : "l"(t), "l"(za), "l"(m1));
  }
  // Q' = Q / 2: Phi(x) = 0.5 + xc * Q'(z)
#define EDV_GELU_K(v) asm("mov.b64 %0, {%1, %1};" : "=l"(k) : "f"(0.5f * (v)))
  EDV_GELU_K(GELU_Q10);
  q = k;
#define EDV_GELU_STEP(v) EDV_GELU_K(v); asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(q) : "l"(q), "l"(t), "l"(k))
  EDV_GELU_STEP(GELU_Q9);
  EDV_GELU_STEP(GELU_Q8);
  EDV_GELU_STEP(GELU_Q7);
  EDV_GELU_STEP(GELU_Q6);
  EDV_GELU_STEP(GELU_Q5);
  EDV_GELU_STEP(GELU_Q4);
  EDV_GELU_STEP(GELU_Q3);
  EDV_GELU_STEP(GELU_Q2);
  EDV_GELU_STEP(GELU_Q1);
  EDV_GELU_STEP(GELU_Q0);
#undef EDV_GELU_STEP
  asm("mov.b64 %0, {%1, %1};" : "=l"(k) : "f"(0.5f));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(q) : "l"(q), "l"(xc), "l"(k));   // Phi(x) = 0.5 (1 + erf(x / sqrt2))
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(q), "l"(xx));               // x Phi(x)
#undef EDV_GELU_K
  asm("mov.b64 {%0, %1}, %2;" : "=f"(y0), "=f"(y1) : "l"(r));
}

template <typename T> __device__ __forceinline__ float gelu_act(float x) {
  if constexpr (sizeof(T) == 4) return gelu_erf(x);
  else return gelu_fast(x);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---------------------------------------------------------------------------------------
// GEMM / conv epilogue description (shared by the CUDA-core and tcgen05 kernels)
// ---------------------------------------------------------------------------------------
enum { ACT_NONE = 0, ACT_GELU = 1, ACT_RELU = 2, ACT_GEGLU = 3, ACT_HEAD = 4, ACT_SIGMOID = 5 };
enum { MAP_LINEAR = 0, MAP_TOKENS = 1, MAP_PIXSHUF = 2 };

struct Epi {
  void* out;             // primary output, element (orow, ocol) at out[orow*ldo + ocol]
  void* out_relu;        // optional copy relu(value) in the activation dtype, same indexing
  const float* bias;     // [N] or null
  const float* rowbias;  // table [(m / rb_div) % rb_mod][rb_ld] or null
  const void* res1;      // optional residual, indexed like out (ld_res)
  const void* res2;
  const float* head_w;   // ACT_HEAD: 1x1 conv weights [N] and bias (dpt.py:121-123)
  long long ldo, ld_res1, ld_res2, rb_ld;
  int rb_div, rb_mod;
  int out_f32, res1_f32, res2_f32;  // 1: that tensor is float32 regardless of T
  int act;
  int map;
  int map_p;       // MAP_TOKENS: patches per frame
  int ps_k, ps_h, ps_w, ps_c;  // MAP_PIXSHUF: k, grid h, grid w, channels per tap (padded)
  float head_b;
  float sig_sign;  // ACT_SIGMOID: sigmoid(sig_sign * x)
  int kind;        // tcgen05 epilogue specialisation (gemm_tc.cuh EF_* mask) or -1: set by the launcher
  long long* tim;  // optional in-kernel timeline of gemm_tc_kernel (edv_op_linear_timeline), else null
};

// maps GEMM row m -> output row for the column-independent mappings
__device__ __forceinline__ long long epi_row(const Epi& e, long long m) {
  if (e.map == MAP_TOKENS) return m + m / e.map_p + 1;
  return m;
}

// Apply the epilogue to NV consecutive columns [n0, n0+NV) of GEMM row m and store.
// `orow` is the output row for MAP_LINEAR/MAP_TOKENS (conv kernels pass their own pixel row).
template <typename T, int NV>
__device__ __forceinline__ void epi_apply(const Epi& e, long long m, long long orow, int n0, float* v) {
  if (e.bias) {
    float b[NV];
    load_vec<float, NV>(e.bias + n0, b);   // n0 is a multiple of 4 at every call site
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] += b[i];
  }
  if (e.rowbias) {
    float b[NV];
    load_vec<float, NV>(e.rowbias + (long long)((m / e.rb_div) % e.rb_mod) * e.rb_ld + n0, b);
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] += b[i];
  }
  if (e.act == ACT_GELU) {
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = gelu_act<T>(v[i]);
  }
  long long ocol = n0;
  if (e.map == MAP_PIXSHUF) {
    // m = (f, y, x) over the ps_h x ps_w grid; n = (ky*k + kx)*ps_c + c
    int tap = n0 / e.ps_c;
    ocol = n0 - tap * e.ps_c;
    int ky = tap / e.ps_k, kx = tap - ky * e.ps_k;
    long long hw = (long long)e.ps_h * e.ps_w;
    long long f = m / hw;
    int r = (int)(m - f * hw);
    int y = r / e.ps_w, x = r - y * e.ps_w;
    orow = (f * (e.ps_h * e.ps_k) + (long long)y * e.ps_k + ky) * ((long long)e.ps_w * e.ps_k) + (long long)x * e.ps_k + kx;
  }
  if (e.res1) {
    float r[NV];
    if (e.res1_f32) load_vec<float, NV>((const float*)e.res1 + orow * e.ld_res1 + ocol, r);
    else load_vec<T, NV>((const T*)e.res1 + orow * e.ld_res1 + ocol, r);
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] += r[i];
  }
  if (e.res2) {
    float r[NV];
    if (e.res2_f32) load_vec<float, NV>((const float*)e.res2 + orow * e.ld_res2 + ocol, r);
    else load_vec<T, NV>((const T*)e.res2 + orow * e.ld_res2 + ocol, r);
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] += r[i];
  }
  if (e.act == ACT_RELU) {
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = fmaxf(v[i], 0.f);
  } else if (e.act == ACT_SIGMOID) {
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = 1.f / (1.f + __expf(-e.sig_sign * v[i]));
  }
  if (e.out) {
    if (e.out_f32) store_vec<float, NV>((float*)e.out + orow * e.ldo + ocol, v);
    else store_vec<T, NV>((T*)e.out + orow * e.ldo + ocol, v);
  }
  if (e.out_relu) {
    float r[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) r[i] = fmaxf(v[i], 0.f);
    store_vec<T, NV>((T*)e.out_relu + orow * e.ldo + ocol, r);
  }
}

// compile-time epilogue kinds of the tcgen05 GEMM (gemm_tc.cuh); Epi::kind holds one of these masks or -1
namespace tc {
enum { EF_BIAS = 1, EF_GELU = 2, EF_RELU = 4, EF_RES1_F32 = 8, EF_RES1_T = 16, EF_RES2_T = 32, EF_OUT_F32 = 64, EF_OUT_RELU = 128, EF_ROWBIAS = 256,
       EF_TMA_OUT = 512 /* 16-bit output written through shared memory + TMA store (gt_epilogue_tma) */ };
}
// The kinds that get their own instantiation, as X-macro lists: the host (ops.cuh epi_kind, gemm_tc_inst.cuh
// gemm_tma_out_ok) accepts exactly the kinds that the device switches (gemm_tc.cuh, gemm_bres.cuh) dispatch.
// Row-segment epilogue (gt_epi_rows); any other epilogue runs its generic F = -1 version.
#define EDV_EPI_ROW_KINDS(X)                                                                  \
  X(EF_BIAS)                                                  /* qkv, projects, out_conv, output_conv1 */ \
  X(EF_BIAS | EF_GELU)                                        /* fc1 */                      \
  X(EF_BIAS | EF_RES1_F32 | EF_OUT_F32)                       /* attn.proj, fc2, temporal to_out: x += ... */ \
  X(EF_BIAS | EF_OUT_F32)                                     /* temporal proj_in */         \
  X(EF_BIAS | EF_RES1_F32)                                    /* temporal ff.net.2 */        \
  X(EF_BIAS | EF_RES1_T)                                      /* temporal proj_out, RCU conv2 */ \
  X(EF_BIAS | EF_RES1_T | EF_OUT_RELU)                                                       \
  X(EF_BIAS | EF_RES1_T | EF_RES2_T)                                                         \
  X(EF_BIAS | EF_RES1_T | EF_RES2_T | EF_OUT_RELU)                                           \
  X(EF_BIAS | EF_RELU)                                        /* RCU conv1 */                \
  X(EF_OUT_RELU)                                              /* layer*_rn */                \
  X(0)                                                        /* temporal q|k|v (no bias) */
// TMA-store epilogue (gt_epilogue_tma): 16-bit row-major output with bias / GELU / ReLU only
#define EDV_EPI_TMA_KINDS(X) X(EF_BIAS) X(EF_BIAS | EF_GELU) X(EF_BIAS | EF_RELU) X(0)
