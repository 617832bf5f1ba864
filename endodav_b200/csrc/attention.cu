// Attention launchers: spatial flash attention (tcgen05, attention_tc.cuh) with its CUDA-core
// cross-check, and the short-sequence temporal attention (mma.sync / CUDA-core).
#include "ops.h"
#include "attention_simt.cuh"
#include "attention_temporal_mma.cuh"
#include "attention_tc.cuh"

namespace edv {

void attention(Launch& L, int dtype, int engine, const void* qkv, void* out, int F, int S, int heads, long long* timeline) {
  if (!L.ok()) return;
  // QK^T + PV: 4*S*S*64 per (frame, head); q,k,v read once, o written once
  L.note(4.0 * F * heads * (double)S * S * 64, 4.0 * F * S * heads * 64 * dtype_size(dtype));
  if (dtype != EDV_F32 && engine == EDV_ENGINE_TC) {
    if (dtype == EDV_BF16) tc::launch_attention_tc<bf16>(L, dtype, qkv, out, F, S, heads, timeline);
    else tc::launch_attention_tc<f16>(L, dtype, qkv, out, F, S, heads, timeline);
    return;
  }
  dim3 grid((S + 127) / 128, heads, F);
  EDV_DISPATCH_T(dtype, { spatial_attention_simt_kernel<T><<<grid, 128, 0, L.stream>>>((const T*)qkv, (T*)out, S, heads); });
  L.check("spatial_attention_simt");
}

template <typename T, int HD>
void launch_temporal(Launch& L, const void* qkv, void* out, int B, int Tn, int hw, int C, const float* rope) {
  const int heads = 8;
  // shared memory per (position, head): K and V in fp32, q/o in T
  const size_t per = (size_t)Tn * HD * (8 + sizeof(T));
  int hg = heads;
  while (hg > 1 && hg * per > 64 * 1024) hg >>= 1;
  int pb = (int)((64 * 1024) / (hg * per));
  if (pb < 1) pb = 1;
  if (pb > 4) pb = 4;
  while (pb > 1 && 32 * hg * pb > ta_max_threads<HD>()) --pb;
  while (hg > 1 && 32 * hg * pb > ta_max_threads<HD>()) hg >>= 1;
  if (pb > hw) pb = hw;
  const size_t smem = (size_t)pb * hg * per + (size_t)Tn * 16 + 16;
  constexpr auto kern = temporal_attention_kernel<T, HD>;
  smem_opt_in<kern>(200 * 1024);
  dim3 grid((hw + pb - 1) / pb, B, heads / hg);
  L.note(4.0 * B * hw * heads * (double)Tn * Tn * HD, 4.0 * B * Tn * hw * C * sizeof(T));
  kern<<<grid, 32 * hg * pb, smem, L.stream>>>((const T*)qkv, (T*)out, Tn, hw, C, pb, hg, (const float2*)rope);   // fp32 CUDA-core path: no PDL hooks, plain launch
  L.check("temporal_attention");
}

template <typename T, int HD, int PB>
void launch_temporal_mma_pb(Launch& L, const void* qkv, void* out, int B, int Tn, int hw, const float* rope) {
  constexpr auto kern = tmma::temporal_attention_mma_kernel<T, HD, PB>;
  const size_t smem = PB * tmma::ta_smem_per_pos<HD>();
  smem_opt_in<kern>((int)smem);
  dim3 grid((hw + PB - 1) / PB, B);
  const int C = 8 * HD;
  L.note(4.0 * B * hw * 8 * (double)Tn * Tn * HD, 4.0 * B * Tn * hw * C * sizeof(T));
  edv::launch_k(kern, dim3(grid), dim3(tmma::TA_WARPS * 32), smem, L.stream, (const T*)qkv, (T*)out, Tn, hw, (const float2*)rope);
  L.check("temporal_attention");
}

// 16-bit paths: warp-level tensor-core kernel (attention_temporal_mma.cuh); PB positions per CTA so that the
// staging fits ~96 KB (two CTAs per SM) and every warp gets at least one (position, head) task
template <typename T, int HD>
void launch_temporal_mma(Launch& L, const void* qkv, void* out, int B, int Tn, int hw, const float* rope) {
  constexpr size_t per = tmma::ta_smem_per_pos<HD>();
  if constexpr (4 * per <= 96 * 1024) {
    if (hw >= 4) return launch_temporal_mma_pb<T, HD, 4>(L, qkv, out, B, Tn, hw, rope);
  }
  if constexpr (2 * per <= 96 * 1024) {
    if (hw >= 2) return launch_temporal_mma_pb<T, HD, 2>(L, qkv, out, B, Tn, hw, rope);
  }
  launch_temporal_mma_pb<T, HD, 1>(L, qkv, out, B, Tn, hw, rope);
}

void temporal_attention(Launch& L, int dtype, const void* qkv, void* out, int B, int Tn, int hw, int C,
                               const float* rope) {
  if (!L.ok()) return;
  if (Tn > 32 || Tn < 1) return L.fail(EDV_ERR_ARG, "temporal attention: T must be in [1,32] (motion_module.py:185-197)");
  if (C % 8 != 0) return L.fail(EDV_ERR_ARG, "temporal attention: C must be a multiple of 8");
  const int hd = C / 8;
  if (dtype != EDV_F32) {
#define EDV_TM_CASE(HD_)                                                                                   \
    if (hd == HD_) {                                                                                       \
      if (dtype == EDV_BF16) launch_temporal_mma<bf16, HD_>(L, qkv, out, B, Tn, hw, rope);                 \
      else launch_temporal_mma<f16, HD_>(L, qkv, out, B, Tn, hw, rope);                                     \
      return;                                                                                              \
    }
    EDV_TM_CASE(8)
    EDV_TM_CASE(24)
    EDV_TM_CASE(32)
    EDV_TM_CASE(48)
    EDV_TM_CASE(128)
#undef EDV_TM_CASE
  }
#define EDV_TA_CASE(HD_)                                                                   \
  if (hd == HD_) {                                                                         \
    EDV_DISPATCH_T(dtype, { launch_temporal<T, HD_>(L, qkv, out, B, Tn, hw, C, rope); });        \
    return;                                                                                \
  }
  EDV_TA_CASE(8)
  EDV_TA_CASE(24)
  EDV_TA_CASE(32)
  EDV_TA_CASE(48)
  EDV_TA_CASE(128)
#undef EDV_TA_CASE
  L.fail(EDV_ERR_ARG, "temporal attention: unsupported head dim (supported 8,24,32,48,128)");
}

}  // namespace edv
