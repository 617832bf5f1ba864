// Launchers of the memory-bound kernels and the GEMM dispatcher; included by engine.cu only.
// The tensor-core kernels live in their own translation units (ops.h).
#pragma once
#include "ops.h"
#include "elementwise.cuh"
#include "gemm_simt.cuh"

namespace edv {

template <typename T> void launch_gemm_simt(Launch& L, const GemmArgs& a) {
  note_gemm(L, a, sizeof(T));
  L.kernel = "gemm_simt";
  dim3 grid((unsigned)((a.M + SG_BM - 1) / SG_BM), (a.N + SG_BN - 1) / SG_BN);
  ConvGeom g{};
  if (a.conv) {
    g.H = a.H; g.W = a.Wd; g.C = a.C; g.stride = a.stride;
    g.OH = (a.H - 1) / a.stride + 1;
    g.OW = (a.Wd - 1) / a.stride + 1;
    gemm_simt_kernel<T, true><<<grid, 256, 0, L.stream>>>((const T*)a.A, (const T*)a.W, a.e, a.M, a.N, a.K, a.lda, g);
  } else {
    gemm_simt_kernel<T, false><<<grid, 256, 0, L.stream>>>((const T*)a.A, (const T*)a.W, a.e, a.M, a.N, a.K, a.lda, g);
  }
  L.check("gemm_simt");
}

// which compile-time epilogue instantiation (gemm_tc.cuh EF_*) matches this epilogue, or -1
inline int epi_kind(const Epi& e) {
  using namespace tc;
  if (e.rowbias || e.map == MAP_PIXSHUF || e.act == ACT_SIGMOID || e.act == ACT_GEGLU || e.act == ACT_HEAD || !e.out) return -1;
  if (e.res2 && (e.res2_f32 || !e.res1)) return -1;
  int f = 0;
  if (e.bias) f |= EF_BIAS;
  if (e.act == ACT_GELU) f |= EF_GELU;
  if (e.act == ACT_RELU) f |= EF_RELU;
  if (e.res1) f |= e.res1_f32 ? EF_RES1_F32 : EF_RES1_T;
  if (e.res2) f |= EF_RES2_T;
  if (e.out_f32) f |= EF_OUT_F32;
  if (e.out_relu) f |= EF_OUT_RELU;
  switch (f) {
#define EDV_KIND_LABEL(F_) case F_:
    EDV_EPI_ROW_KINDS(EDV_KIND_LABEL) return f;
#undef EDV_KIND_LABEL
    default: return -1;
  }
}

// dispatch on dtype / engine.  GEGLU and HEAD epilogues exist only in the tcgen05 kernel;
// the CUDA-core path composes them from a plain GEMM plus a small kernel (see engine.cu).
inline void gemm(Launch& L, int dtype, int engine, const GemmArgs& a_in) {
  if (!L.ok()) return;
  GemmArgs a = a_in;
  a.e.kind = epi_kind(a.e);
  if (dtype == EDV_F32) return launch_gemm_simt<float>(L, a);
  if (engine == EDV_ENGINE_SIMT) {
    if (dtype == EDV_BF16) return launch_gemm_simt<bf16>(L, a);
    return launch_gemm_simt<f16>(L, a);
  }
  if (dtype == EDV_BF16) return a.conv ? launch_gemm_tc_conv<bf16>(L, dtype, a) : launch_gemm_tc_lin<bf16>(L, dtype, a);
  return a.conv ? launch_gemm_tc_conv<f16>(L, dtype, a) : launch_gemm_tc_lin<f16>(L, dtype, a);
}

inline void layernorm(Launch& L, int dtype, const float* x, const float* g, const float* b, void* y, long long Mout,
                      int D, float eps, int grp = 0, int skip = 0, const float* add = nullptr, int add_div = 1,
                      int add_mod = 1) {
  if (!L.ok()) return;
  if (D % 4 != 0 || D > 1024) return L.fail(EDV_ERR_ARG, "layernorm: D must be a multiple of 4 and <= 1024");
  const int maxv = (D + 127) / 128;
  const unsigned blocks = nblk(((Mout + 1) / 2) * 32, 256);   // one warp per two rows
  L.note(0, (double)Mout * D * (4 + dtype_size(dtype)));
  EDV_DISPATCH_T(dtype, {
    if (maxv <= 1) edv::launch_k(layernorm_kernel<T, 1>, dim3(blocks), dim3(256), 0, L.stream, x, g, b, (T*)y, Mout, D, eps, grp, skip, add, add_div, add_mod);
    else if (maxv <= 2) edv::launch_k(layernorm_kernel<T, 2>, dim3(blocks), dim3(256), 0, L.stream, x, g, b, (T*)y, Mout, D, eps, grp, skip, add, add_div, add_mod);
    else if (maxv <= 3) edv::launch_k(layernorm_kernel<T, 3>, dim3(blocks), dim3(256), 0, L.stream, x, g, b, (T*)y, Mout, D, eps, grp, skip, add, add_div, add_mod);
    else if (maxv <= 4) edv::launch_k(layernorm_kernel<T, 4>, dim3(blocks), dim3(256), 0, L.stream, x, g, b, (T*)y, Mout, D, eps, grp, skip, add, add_div, add_mod);
    else edv::launch_k(layernorm_kernel<T, 8>, dim3(blocks), dim3(256), 0, L.stream, x, g, b, (T*)y, Mout, D, eps, grp, skip, add, add_div, add_mod);
  });
  L.check("layernorm");
}

constexpr int GN_MAX_SPLIT = 64;   // groupnorm stats scratch: F*32*(1+GN_MAX_SPLIT) float2

inline void groupnorm(Launch& L, int dtype, const void* x, const float* g, const float* b, void* y, float2* stats,
                      int F, int hw, int C, float eps) {
  if (!L.ok()) return;
  if (C % 32 != 0 || C % 8 != 0) return L.fail(EDV_ERR_ARG, "groupnorm: C must be a multiple of 32");
  if (dtype == EDV_F32 || C / 8 > 256) {
    // fp32 path: two-pass (mean, then centred variance) per (frame, group)
    EDV_DISPATCH_T(dtype, {
      L.note(0, (double)F * hw * C * sizeof(T));
      edv::launch_k(groupnorm_stats_kernel<T>, dim3(32, F), dim3(256), 0, L.stream, (const T*)x, stats, hw, C, eps);
    });
    L.check("groupnorm_stats");
  } else {
    const int per_px = 256 / (C / 8);
    int split = (hw + per_px * 8 - 1) / (per_px * 8);     // ~8 pixels per thread
    if (split < 1) split = 1;
    if (split > GN_MAX_SPLIT) split = GN_MAX_SPLIT;
    float2* part = stats + (size_t)F * 32;                 // caller provides F*32*(1+GN_MAX_SPLIT) entries
    EDV_DISPATCH_T(dtype, {
      L.note(0, (double)F * hw * C * sizeof(T));
      edv::launch_k(groupnorm_partial_kernel<T>, dim3(F, split), dim3(256), 0, L.stream, (const T*)x, part, hw, C);
    });
    L.check("groupnorm_stats");
    edv::launch_k(groupnorm_finalize_kernel, dim3(nblk((long long)F * 32, 256)), dim3(256), 0, L.stream, part, stats, F * 32, split, (float)hw * (C / 32), eps);
    L.check("groupnorm_finalize");
  }
  EDV_DISPATCH_T(dtype, {
    long long total8 = (long long)F * hw * C / 8;
    L.note(0, 2.0 * F * hw * C * sizeof(T));
    edv::launch_k(groupnorm_apply_kernel<T>, dim3(nblk(total8, 256)), dim3(256), 0, L.stream, (const T*)x, stats, g, b, (T*)y, total8, hw, C);
  });
  L.check("groupnorm_apply");
}

inline void upsample(Launch& L, int dtype, const void* x, void* y, int F, int h, int w, int oh, int ow, int C) {
  if (!L.ok()) return;
  if (C % 8 != 0) return L.fail(EDV_ERR_ARG, "upsample: C must be a multiple of 8");
  const long long bands = (long long)F * ((oh + UP_ROWS - 1) / UP_ROWS), per_row = (long long)ow * (C / 8);
  if (bands > 0x7fffffffLL || per_row > 65535LL * 256) return L.fail(EDV_ERR_ARG, "upsample: map too large");
  L.note(0, ((double)F * h * w + (double)F * oh * ow) * C * dtype_size(dtype));
  const dim3 grid((unsigned)bands, (unsigned)((per_row + 255) / 256));
  EDV_DISPATCH_T(dtype, { edv::launch_k(upsample_nhwc_kernel<T>, dim3(grid), dim3(256), 0, L.stream, (const T*)x, (T*)y, F, h, w, oh, ow, C); });
  L.check("upsample");
}

inline void resize_f32(Launch& L, const float* x, float* y, int F, int h, int w, int oh, int ow) {
  if (!L.ok()) return;
  long long total = (long long)F * oh * ow;
  L.note(0, ((double)F * h * w + (double)F * oh * ow) * 4);
  edv::launch_k(resize_f32_kernel, dim3(nblk(total, 256)), dim3(256), 0, L.stream, x, y, F, h, w, oh, ow);
  L.check("resize_f32");
}

// K1: frames (float32 [F,3,H,W] or, u8, uint8 [F,H,W,3] at network resolution) -> out [F*(h/14)*(w/14), Kp]
inline void preprocess_patches(Launch& L, int dtype, const void* src, bool u8, void* out, int F, int H, int W, int h, int w,
                               int Kp, int normalize) {
  if (!L.ok()) return;
  const long long tot = (long long)F * (h / 14) * (w / 14) * Kp;
  const unsigned blocks = nblk(tot / 8, 256);
  L.note(0, (double)F * 3 * H * W * (u8 ? 1 : 4) + (double)tot * dtype_size(dtype));
  EDV_DISPATCH_T(dtype, {
    if (u8) preprocess_patches_kernel<T, true><<<blocks, 256, 0, L.stream>>>(src, (T*)out, F, H, W, h, w, Kp, normalize);
    else preprocess_patches_kernel<T, false><<<blocks, 256, 0, L.stream>>>(src, (T*)out, F, H, W, h, w, Kp, normalize);
  });
  L.check("preprocess");
}

// patch rows of the fp32 residual stream x [Mp/P frames][P + cls][D] -> out [Mp, D] in `dtype`
inline void tokens_to_patches(Launch& L, int dtype, const float* x, void* out, long long Mp, int P, int D, int cls) {
  if (!L.ok()) return;
  EDV_DISPATCH_T(dtype, { tokens_to_patches_kernel<T><<<nblk(Mp * (D / 4), 256), 256, 0, L.stream>>>(x, (T*)out, Mp, P, D, cls); });
  L.check("tokens_to_patches");
}

// y [M, C] = act(LN over the first Cr of the C channels of x), padding columns Cr..C-1 written as 0
inline void rowln_act(Launch& L, int dtype, const void* x, const float* gamma, const float* beta, void* y, long long M, int C,
                      int Cr, float eps, int gelu, const char* what = "rowln_act") {
  if (!L.ok()) return;
  EDV_DISPATCH_T(dtype, { rowln_act_kernel<T><<<nblk(M * 32, 256), 256, 0, L.stream>>>((const T*)x, gamma, beta, (T*)y, M, C, Cr, eps, gelu); });
  L.check(what);
}

// x (fp32 residual stream, in place): patch row p of every frame += LN(r[p]); cls rows untouched
inline void resblock_add(Launch& L, int dtype, float* x, const void* r, const float* gamma, const float* beta, long long Mp, int P,
                         int D, float eps, int cls) {
  if (!L.ok()) return;
  EDV_DISPATCH_T(dtype, { resblock_add_kernel<T><<<nblk(Mp * 32, 256), 256, 0, L.stream>>>(x, (const T*)r, gamma, beta, Mp, P, D, eps, cls); });
  L.check("res add");
}

// 3x3 pad-1 im2col of NHWC x [F,H,W,C] -> out [F*OH*OW, 9*C] in (ky,kx,c) order
inline void im2col3x3(Launch& L, int dtype, const void* x, void* out, int F, int H, int W, int C, int OH, int OW, int stride) {
  if (!L.ok()) return;
  const long long tot = (long long)F * OH * OW * 9 * (C / 8);
  EDV_DISPATCH_T(dtype, { edv::launch_k(im2col3x3_kernel<T>, dim3(nblk(tot, 256)), dim3(256), 0, L.stream, (const T*)x, (T*)out, F, H, W, C, OH, OW, stride); });
  L.check("im2col");
}

// out [M, C4] = value * gelu(gate) of hg [M, 2*C4] in pack.py's [64 value | 64 gate] column pairs (CUDA-core GEGLU)
inline void geglu_pair(Launch& L, int dtype, const void* hg, void* out, long long M, int C4) {
  if (!L.ok()) return;
  EDV_DISPATCH_T(dtype, { geglu_pair_kernel<T><<<nblk(M * C4, 256), 256, 0, L.stream>>>((const T*)hg, (T*)out, M, C4); });
  L.check("geglu");
}

// out[m] = x[m] . w[0..C-1] + w[C], then ReLU (sig_sign == 0) or sigmoid(sig_sign * .) (CUDA-core disparity head)
inline void head_dot(Launch& L, int dtype, const void* x, const float* w, float* out, long long M, int C, float sig_sign) {
  if (!L.ok()) return;
  EDV_DISPATCH_T(dtype, {
    head_dot_kernel<T><<<nblk(M, 256), 256, 0, L.stream>>>((const T*)x, w, out, M, C, sig_sign == 0.f, sig_sign, sig_sign != 0.f);
  });
  L.check("head_dot");
}

}  // namespace edv
