// Memory-bound kernels of the EndoDAV forward: preprocessing, normalisations, resampling.
// All activations are NHWC / token-major; T is the activation dtype (float, bf16, f16).
#pragma once
#include "common.cuh"

// ---------------------------------------------------------------------------------------
// K1: resize (bilinear, align_corners=True) + ImageNet normalise + im2col for the 14x14
// patch embedding.  Replaces endodav.py:153,155 and the unfold implied by
// patch_embed.py:75-77.  Output A0[(f*P + py*pw + px), Kp] with k = c*196 + ky*14 + kx
// (the flatten order of the conv weight), zero padded to Kp.
// ---------------------------------------------------------------------------------------
template <typename T, bool U8>
__global__ void preprocess_patches_kernel(const void* __restrict__ src, T* __restrict__ out, int F, int H, int W,
                                          int h, int w, int Kp, int normalize) {
  pdl_launch();
  pdl_wait();
  // one thread = 8 consecutive k of one patch row (one aligned 16-byte store for 16-bit T)
  const int ph = h / 14, pw = w / 14;
  const int kch = Kp / 8;
  const long long total = (long long)F * ph * pw * kch;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int k0 = (int)(i % kch) * 8;
  const long long row = i / kch;
  const int px = (int)(row % pw);
  const long long t = row / pw;
  const int py = (int)(t % ph);
  const int f = (int)(t / ph);
  const float sy = (h > 1) ? (float)(H - 1) / (float)(h - 1) : 0.f;
  const float sx = (w > 1) ? (float)(W - 1) / (float)(w - 1) : 0.f;
  int c = k0 / 196, r = k0 - c * 196;
  int ky = r / 14, kx = r - ky * 14;
  float val[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float o = 0.f;
    if (k0 + j < 588) {
      const int y = py * 14 + ky, x = px * 14 + kx;
      float v;
      if (U8) {
        // uint8 HWC frames already at network resolution (infer_video_depth path)
        const uint8_t* sp = (const uint8_t*)src;
        v = (float)sp[(((long long)f * H + y) * W + x) * 3 + c] / 255.0f;
      } else {
        const float* sp = (const float*)src + ((long long)f * 3 + c) * H * W;
        if (H == h && W == w) {
          v = sp[(long long)y * W + x];
        } else {
          // area_pixel_compute_source_index with align_corners=True
          const float fy = sy * y, fx = sx * x;
          const int y0 = (int)fy, x0 = (int)fx;
          const int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
          const float ly = fy - y0, lx = fx - x0;
          const float v00 = sp[(long long)y0 * W + x0], v01 = sp[(long long)y0 * W + x1];
          const float v10 = sp[(long long)y1 * W + x0], v11 = sp[(long long)y1 * W + x1];
          v = (1.f - ly) * ((1.f - lx) * v00 + lx * v01) + ly * ((1.f - lx) * v10 + lx * v11);
        }
      }
      const float mean = (c == 0) ? 0.485f : (c == 1 ? 0.456f : 0.406f);
      const float stdv = (c == 0) ? 0.229f : (c == 1 ? 0.224f : 0.225f);
      o = normalize ? (v - mean) / stdv : v;
    }
    val[j] = o;
    if (++kx == 14) { kx = 0; if (++ky == 14) { ky = 0; ++c; } }
  }
  store_vec<T, 8>(out + row * Kp + k0, val);
}

// ---------------------------------------------------------------------------------------
// Host preprocessing of infer_video_depth moved to the GPU (SURVEY.md 8(f)-1):
//   frames[i].astype(float32) / 255 -> cv2.resize(INTER_CUBIC) -> HWC->CHW
// (endodav.py:195; util/transform.py:109-113,139-158).  Restates OpenCV's float bicubic:
// A = -0.75, half-pixel centres (fx = (dx + 0.5) * W/w - 0.5), border replicate, horizontal pass
// then vertical pass, no anti-aliasing.  src uint8 [n_src,H,W,3] at element strides (st_n, st_y, st_x, st_c) -> dst float32
// [N,3,h,w]; output frame i reads source frame frames.src[i] (frames.count == 0: frame i).  Consecutive threads take
// consecutive dx, so one tap of a warp reads one run of about 32 * W / w source pixels along x: interleaved RGB for NHWC
// (st_x = 3), the same run in each of the three planes for NCHW memory (st_x = 1).  DESIGN.md section 6 has the
// measured time of both layouts.
// ---------------------------------------------------------------------------------------
// The source frame of every output frame of one launch, passed by value in the kernel parameters: no device
// allocation, copy or synchronisation, and the host validates every entry before the launch.
struct FrameTable {
  static constexpr int kMax = 256;
  int count;
  int src[kMax];
};

__device__ __forceinline__ void cubic_coeffs(float x, float* c) {
  const float A = -0.75f;
  c[0] = ((A * (x + 1) - 5 * A) * (x + 1) + 8 * A) * (x + 1) - 4 * A;
  c[1] = ((A + 2) * x - (A + 3)) * x * x + 1;
  c[2] = ((A + 2) * (1 - x) - (A + 3)) * (1 - x) * (1 - x) + 1;
  c[3] = 1.f - c[0] - c[1] - c[2];
}

__global__ void cubic_resize_u8_kernel(const uint8_t* __restrict__ src, float* __restrict__ dst, int N, int H, int W,
                                       int h, int w, long long st_n, long long st_y, long long st_x, long long st_c,
                                       const __grid_constant__ FrameTable frames) {
  const long long total = (long long)N * h * w;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int dx = (int)(i % w);
  const long long t = i / w;
  const int dy = (int)(t % h);
  const int n = (int)(t / h);
  const double scale_x = (double)W / w, scale_y = (double)H / h;
  // source coordinate in double, fraction rounded to float last (a float coordinate near 300 would lose
  // 3e-5 of the fraction; OpenCV 4.x is accurate to 2e-7 against the exact cubic)
  const double fxd = (dx + 0.5) * scale_x - 0.5, fyd = (dy + 0.5) * scale_y - 0.5;
  const int sx = (int)floor(fxd), sy = (int)floor(fyd);
  const float fx = (float)(fxd - sx), fy = (float)(fyd - sy);
  float cx[4], cy[4];
  cubic_coeffs(fx, cx);
  cubic_coeffs(fy, cy);
  int xs[4], ys[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    xs[k] = min(max(sx + k - 1, 0), W - 1);
    ys[k] = min(max(sy + k - 1, 0), H - 1);
  }
  const uint8_t* base = src + (long long)(frames.count ? frames.src[n] : n) * st_n;
  float acc[3] = {0.f, 0.f, 0.f};
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const uint8_t* row = base + ys[r] * st_y;
    float hs[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint8_t* px = row + xs[k] * st_x;
#pragma unroll
      for (int c = 0; c < 3; ++c) hs[c] += ((float)px[c * st_c] / 255.0f) * cx[k];
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) acc[c] += hs[c] * cy[r];
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) dst[(((size_t)n * 3 + c) * h + dy) * w + dx] = acc[c];
}

// cls row of every frame: x[f, 0, :] = cls_token + pos_embed[0]  (vision_transformer.py:225-227)
__global__ void cls_row_kernel(float* __restrict__ x, const float* __restrict__ cls_row, int F, int N, int D) {
  pdl_launch();
  pdl_wait();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= F * D) return;
  int f = i / D, d = i - f * D;
  x[(long long)f * N * D + d] = cls_row[d];
}

// ---------------------------------------------------------------------------------------
// LayerNorm over D (one warp per row), float32 in -> T out.  With grp>0 the input is
// [.., grp rows] per frame and the first `skip` rows of every frame are dropped from the
// (compact) output: the final norm on the four taps + cls split
// (vision_transformer.py:318-321).  Two-pass statistics in registers.
// ---------------------------------------------------------------------------------------
template <typename TOut, int MAXV>
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, TOut* __restrict__ out,
                                                        long long Mout, int D, float eps, int grp, int skip,
                                                        const float* __restrict__ add, int add_div, int add_mod) {
  pdl_launch();
  pdl_wait();
  // one warp normalises TWO consecutive rows: both rows' loads are in flight before the first
  // reduction (the kernel is pure streaming: fp32 in, 16-bit out)
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const long long mo0 = warp * 2;
  if (mo0 >= Mout) return;
  float v[2][MAXV * 4];
  bool live[2];
  long long mo[2];
#pragma unroll
  for (int rw = 0; rw < 2; ++rw) {
    mo[rw] = mo0 + rw;
    live[rw] = mo[rw] < Mout;
    long long mi = mo[rw];
    if (grp > 0) {
      // skip >= 0: drop the first `skip` rows of every group of `grp`; skip < 0: keep ONLY the first -skip rows
      const int per = skip >= 0 ? grp - skip : -skip;
      mi = (mo[rw] / per) * grp + (skip >= 0 ? skip : 0) + (mo[rw] % per);
    }
    const float* xr = x + mi * D;
#pragma unroll
    for (int it = 0; it < MAXV; ++it) {
      const int c = (it * 32 + lane) * 4;
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      if (live[rw] && c < D) t = *reinterpret_cast<const float4*>(xr + c);
      v[rw][4 * it] = t.x; v[rw][4 * it + 1] = t.y; v[rw][4 * it + 2] = t.z; v[rw][4 * it + 3] = t.w;
    }
  }
  float g[MAXV * 4], b[MAXV * 4];
#pragma unroll
  for (int it = 0; it < MAXV; ++it) {
    const int c = (it * 32 + lane) * 4;
    float4 tg = make_float4(0.f, 0.f, 0.f, 0.f), tb = tg;
    if (c < D) {
      tg = *reinterpret_cast<const float4*>(gamma + c);
      tb = *reinterpret_cast<const float4*>(beta + c);
    }
    g[4 * it] = tg.x; g[4 * it + 1] = tg.y; g[4 * it + 2] = tg.z; g[4 * it + 3] = tg.w;
    b[4 * it] = tb.x; b[4 * it + 1] = tb.y; b[4 * it + 2] = tb.z; b[4 * it + 3] = tb.w;
  }
#pragma unroll
  for (int rw = 0; rw < 2; ++rw) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV * 4; ++i) s += v[rw][i];     // columns >= D hold zeros
    const float mean = warp_sum(s) / (float)D;
    float q = 0.f;
#pragma unroll
    for (int it = 0; it < MAXV; ++it) {
      const int c = (it * 32 + lane) * 4;
      if (c < D) {
#pragma unroll
        for (int j = 0; j < 4; ++j) { const float d = v[rw][4 * it + j] - mean; q += d * d; }
      }
    }
    const float rstd = rsqrtf(warp_sum(q) / (float)D + eps);
    if (!live[rw]) continue;
    TOut* orow = out + mo[rw] * D;
    // optional per-frame additive table (temporal positional encoding, motion_module.py:236-237)
    const float* arow = add ? add + (long long)((mo[rw] / add_div) % add_mod) * D : nullptr;
#pragma unroll
    for (int it = 0; it < MAXV; ++it) {
      const int c = (it * 32 + lane) * 4;
      if (c < D) {
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = (v[rw][4 * it + j] - mean) * rstd * g[4 * it + j] + b[4 * it + j];
        if (arow) {
          const float4 t = *reinterpret_cast<const float4*>(arow + c);
          o[0] += t.x; o[1] += t.y; o[2] += t.z; o[3] += t.w;
        }
        store_vec<TOut, 4>(orow + c, o);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------
// GroupNorm(32) statistics per (frame, group) over (C/32) x hw elements, NHWC input.
// Two passes (mean, then centred variance); the second pass hits L2.  stats[f*32+g] = {mean, rstd}
// ---------------------------------------------------------------------------------------
template <typename T>
__global__ void groupnorm_stats_kernel(const T* __restrict__ x, float2* __restrict__ stats, int hw, int C, float eps) {
  pdl_launch();
  pdl_wait();
  const int f = blockIdx.y, g = blockIdx.x;
  const int cpg = C / 32;
  const T* base = x + (long long)f * hw * C + g * cpg;
  __shared__ float red[32];
  __shared__ float s_mean;
  const int total = hw * cpg;
  float s = 0.f;
  for (int i = threadIdx.x; i < total; i += blockDim.x) {
    int p = i / cpg, c = i - p * cpg;
    s += to_f<T>(base[(long long)p * C + c]);
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) s_mean = t / (float)total;
  }
  __syncthreads();
  const float mean = s_mean;
  float q = 0.f;
  for (int i = threadIdx.x; i < total; i += blockDim.x) {
    int p = i / cpg, c = i - p * cpg;
    float d = to_f<T>(base[(long long)p * C + c]) - mean;
    q += d * d;
  }
  q = warp_sum(q);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = q;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) stats[f * 32 + g] = make_float2(mean, rsqrtf(t / (float)total + eps));
  }
}

// Coalesced statistics for the 16-bit paths: grid (F, NSPLIT); a block streams whole pixel rows
// (16-byte loads), keeps per-thread sums of its 8 channels and reduces them through shared memory
// in a FIXED order (no atomics: the forward must stay bit-reproducible) to one (sum, sum of
// squares) per group, written to part[(f*NSPLIT + split)*32 + g].  fp32 sums over <= a few 10^4
// values of O(1): the E[x^2]-E[x]^2 form is far inside 16-bit accuracy.
template <typename T>
__global__ void __launch_bounds__(256) groupnorm_partial_kernel(const T* __restrict__ x, float2* __restrict__ part, int hw, int C) {
  pdl_launch();
  pdl_wait();
  __shared__ float cs[2][2048];                // [sum|sq][pixel lane][channel], per_px * C <= 2048
  const int f = blockIdx.x;
  const int c8n = C / 8;                       // 16-byte chunks per pixel
  const int cpg = C / 32;
  const int per_px = blockDim.x / c8n;         // pixel lanes per block
  const int c8 = threadIdx.x % c8n, pl = threadIdx.x / c8n;
  if (pl < per_px) {
    float s[8], q[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j] = 0.f; q[j] = 0.f; }
    const T* base = x + (long long)f * hw * C + c8 * 8;
    for (int p = blockIdx.y * per_px + pl; p < hw; p += gridDim.y * per_px) {
      float v[8];
      load_vec<T, 8>(base + (long long)p * C, v);
#pragma unroll
      for (int j = 0; j < 8; ++j) { s[j] += v[j]; q[j] = fmaf(v[j], v[j], q[j]); }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) { cs[0][pl * C + c8 * 8 + j] = s[j]; cs[1][pl * C + c8 * 8 + j] = q[j]; }
  }
  __syncthreads();
  if (threadIdx.x < 64) {
    const int g = threadIdx.x & 31, which = threadIdx.x >> 5;
    float a = 0.f;
    for (int pp = 0; pp < per_px; ++pp)
      for (int c = g * cpg; c < (g + 1) * cpg; ++c) a += cs[which][pp * C + c];
    float* dst = reinterpret_cast<float*>(&part[((long long)f * gridDim.y + blockIdx.y) * 32 + g]);
    dst[which] = a;
  }
}

// partial (sum, sumsq) over the splits (fixed order) -> (mean, rstd) in stats[f*32+g]
__global__ void groupnorm_finalize_kernel(const float2* __restrict__ part, float2* __restrict__ stats, int n, int nsplit,
                                          float count, float eps) {
  pdl_launch();
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int f = i >> 5, g = i & 31;
  float sx = 0.f, sq = 0.f;
  for (int k = 0; k < nsplit; ++k) {
    const float2 r = part[((long long)f * nsplit + k) * 32 + g];
    sx += r.x;
    sq += r.y;
  }
  const float mean = sx / count;
  const float var = fmaxf(sq / count - mean * mean, 0.f);
  stats[i] = make_float2(mean, rsqrtf(var + eps));
}

template <typename T>
__global__ void groupnorm_apply_kernel(const T* __restrict__ x, const float2* __restrict__ stats,
                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                       T* __restrict__ y, long long total8, int hw, int C) {
  pdl_launch();
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total8) return;
  long long e0 = i * 8;
  int c0 = (int)(e0 % C);
  int f = (int)(e0 / ((long long)hw * C));
  const int cpg = C / 32;
  float v[8];
  load_vec<T, 8>(x + e0, v);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    int c = c0 + j;
    float2 st = stats[f * 32 + c / cpg];
    v[j] = (v[j] - st.x) * st.y * __ldg(gamma + c) + __ldg(beta + c);
  }
  store_vec<T, 8>(y + e0, v);
}

// ---------------------------------------------------------------------------------------
// Bilinear resize, align_corners=True, NHWC, 8 channels per thread.
// (util/blocks.py:156-158; dpt_pyramid.py:90-92)
// ---------------------------------------------------------------------------------------
// Separable evaluation, bit-identical to the direct form  o = (1-ly)*((1-lx)*a + lx*b) + ly*((1-lx)*c + lx*d)  (ATen's
// association): a thread owns ONE (output column, 8-channel chunk) and walks a band of UP_ROWS output rows.  The
// horizontal lerp of a source row, H(r) = fma(lx, x[r,x1], (1-lx)*x[r,x0]), depends only on the column, so it is kept
// in registers and reused by every output row that touches source row r (each source row serves ~2 output rows as y0
// and ~2 as y1 when upsampling x2): 1.5 lerps and 0.5 source conversions per output instead of 3 and 4, and the column
// index / weight arithmetic is done once per thread instead of once per output.  (The direct kernel was issue-bound:
// ncu issue slots 78 % busy at 1.8 TB/s.)
// grid.x = F * ceil(oh / UP_ROWS) bands, grid.y covers the ow*C/8 16-byte chunks of a row.
constexpr int UP_ROWS = 16;
template <typename T>
__global__ void __launch_bounds__(256) upsample_nhwc_kernel(const T* __restrict__ x, T* __restrict__ y, int F, int h, int w, int oh, int ow,
                                                             int C) {
  pdl_launch();
  const int c8 = C / 8;
  const int j = blockIdx.y * blockDim.x + threadIdx.x;      // chunk within the output row
  const int bands = (oh + UP_ROWS - 1) / UP_ROWS;
  const int f = blockIdx.x / bands, oy0 = (blockIdx.x - f * bands) * UP_ROWS;
  const float sy = (oh > 1) ? (float)(h - 1) / (float)(oh - 1) : 0.f;
  const float sx = (ow > 1) ? (float)(w - 1) / (float)(ow - 1) : 0.f;
  const bool live = j < ow * c8;
  const int ox = live ? j / c8 : 0, c = live ? (j - ox * c8) * 8 : 0;
  const float fx = sx * ox;
  const int x0 = (int)fx;
  const int x1 = min(x0 + 1, w - 1);
  const float lx = fx - x0, wx0 = 1.f - lx;
  const T* b0 = x + (long long)f * h * w * C + (long long)x0 * C + c;
  const T* b1 = x + (long long)f * h * w * C + (long long)x1 * C + c;
  pdl_wait();
  if (!live) return;
  auto hrow = [&](int r, float* H) {
    float a[8], bq[8];
    load_vec<T, 8>(b0 + (long long)r * w * C, a);
    load_vec<T, 8>(b1 + (long long)r * w * C, bq);
#pragma unroll
    for (int i = 0; i < 8; ++i) H[i] = wx0 * a[i] + lx * bq[i];
  };
  float H0[8], H1[8];
  int r0 = -1, r1 = -1;                                     // source rows held in H0 / H1
  const int oy_end = min(oy0 + UP_ROWS, oh);
  for (int oy = oy0; oy < oy_end; ++oy) {
    const float fy = sy * oy;
    const int y0 = (int)fy;
    const int y1 = min(y0 + 1, h - 1);
    const float ly = fy - y0, wy0 = 1.f - ly;
    if (y0 != r0) {                                         // (uniform over the CTA: every thread shares oy)
      if (y0 == r1) {
#pragma unroll
        for (int i = 0; i < 8; ++i) H0[i] = H1[i];
      } else {
        hrow(y0, H0);
      }
      r0 = y0;
    }
    if (y1 != r1) {
      if (y1 == r0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) H1[i] = H0[i];
      } else {
        hrow(y1, H1);
      }
      r1 = y1;
    }
    float o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = wy0 * H0[i] + ly * H1[i];
    store_vec<T, 8>(y + (((long long)f * oh + oy) * ow + ox) * C + c, o);
  }
}

// single-channel float32 bilinear resize (align_corners=True): disparity pyramid
// (dpt_pyramid.py:95-97) and the final per-window resize (endodav.py:205).
__global__ void resize_f32_kernel(const float* __restrict__ x, float* __restrict__ y, int F, int h, int w, int oh,
                                  int ow) {
  pdl_launch();
  pdl_wait();
  const long long total = (long long)F * oh * ow;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int ox = (int)(i % ow);
  long long t = i / ow;
  int oy = (int)(t % oh);
  int f = (int)(t / oh);
  const float sy = (oh > 1) ? (float)(h - 1) / (float)(oh - 1) : 0.f;
  const float sx = (ow > 1) ? (float)(w - 1) / (float)(ow - 1) : 0.f;
  float fy = sy * oy, fx = sx * ox;
  int y0 = (int)fy, x0 = (int)fx;
  int y1 = min(y0 + 1, h - 1), x1 = min(x0 + 1, w - 1);
  float ly = fy - y0, lx = fx - x0;
  const float* b = x + (long long)f * h * w;
  float v = (1.f - ly) * ((1.f - lx) * b[(long long)y0 * w + x0] + lx * b[(long long)y0 * w + x1]) +
            ly * ((1.f - lx) * b[(long long)y1 * w + x0] + lx * b[(long long)y1 * w + x1]);
  y[i] = v;
}

__global__ void sigmoid_inplace_kernel(float* __restrict__ x, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = 1.f / (1.f + expf(-x[i]));
}

// explicit im2col for the single stride-2 3x3 conv (resize_layers[3], dpt.py:85-90):
// out[(f,oy,ox), (ky,kx,c)] with zero padding 1.
template <typename T>
__global__ void im2col3x3_kernel(const T* __restrict__ x, T* __restrict__ out, int F, int H, int W, int C, int OH,
                                 int OW, int stride) {
  pdl_launch();
  pdl_wait();
  const int c8 = C / 8;
  const long long total = (long long)F * OH * OW * 9 * c8;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int c = (int)(i % c8) * 8;
  long long t = i / c8;
  int tap = (int)(t % 9);
  long long p = t / 9;
  int ox = (int)(p % OW);
  long long t2 = p / OW;
  int oy = (int)(t2 % OH);
  int f = (int)(t2 / OH);
  int ky = tap / 3, kx = tap - ky * 3;
  int iy = oy * stride + ky - 1, ix = ox * stride + kx - 1;
  float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (iy >= 0 && iy < H && ix >= 0 && ix < W) load_vec<T, 8>(x + (((long long)f * H + iy) * W + ix) * C + c, v);
  store_vec<T, 8>(out + (p * 9 + tap) * C + c, v);
}

// strided channel copy NHWC [.., Cs] -> [.., Cd] (first min(Cs,Cd) channels), debug taps of padded maps
template <typename T>
__global__ void copy_channels_f32_kernel(const T* __restrict__ x, float* __restrict__ y, long long rows, int Cs, int Cd) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * Cd) return;
  long long r = i / Cd;
  int c = (int)(i - r * Cd);
  y[i] = to_f<T>(x[r * Cs + c]);
}

// channels-first LayerNorm of ResBottleneckBlock on NHWC rows (layers/utils.py:171-179),
// optional exact GELU, one warp per pixel; in/out dtype T.  Rows hold C (padded) channels of
// which the first Cr are real; padded outputs are written as zero.
template <typename T>
__global__ void rowln_act_kernel(const T* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                                 T* __restrict__ y, long long M, int C, int Cr, float eps, int gelu) {
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= M) return;
  const T* xr = x + warp * C;
  float s = 0.f;
  for (int c = lane; c < Cr; c += 32) s += to_f<T>(xr[c]);
  const float mean = warp_sum(s) / (float)Cr;
  float q = 0.f;
  for (int c = lane; c < Cr; c += 32) { float d = to_f<T>(xr[c]) - mean; q += d * d; }
  const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)Cr + eps);
  for (int c = lane; c < C; c += 32) {
    float v = 0.f;
    if (c < Cr) {
      v = (to_f<T>(xr[c]) - mean) * rstd * __ldg(gamma + c) + __ldg(beta + c);
      if (gelu) v = gelu_erf(v);
    }
    y[warp * C + c] = from_f<T>(v);
  }
}

// x[f, 1+p, :] += LN_cf(r[f*P+p, :])   -- the residual-block add into patch tokens (block.py:146-150)
template <typename T>
__global__ void resblock_add_kernel(float* __restrict__ x, const T* __restrict__ r, const float* __restrict__ gamma,
                                    const float* __restrict__ beta, long long Mp, int P, int D, float eps, int cls) {
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= Mp) return;
  const T* rr = r + warp * D;
  float s = 0.f;
  for (int c = lane; c < D; c += 32) s += to_f<T>(rr[c]);
  const float mean = warp_sum(s) / (float)D;
  float q = 0.f;
  for (int c = lane; c < D; c += 32) { float d = to_f<T>(rr[c]) - mean; q += d * d; }
  const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)D + eps);
  float* xr = x + (cls ? warp + warp / P + 1 : warp) * D;   // cls: skip the frame's cls row
  for (int c = lane; c < D; c += 32)
    xr[c] += (to_f<T>(rr[c]) - mean) * rstd * __ldg(gamma + c) + __ldg(beta + c);
}

// compact copy of the patch tokens of the fp32 residual stream into T (drops cls rows)
template <typename T>
__global__ void tokens_to_patches_kernel(const float* __restrict__ x, T* __restrict__ y, long long Mp, int P, int D, int cls) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = Mp * (D / 4);
  if (i >= total) return;
  long long r = i / (D / 4);
  int c = (int)(i - r * (D / 4)) * 4;
  float v[4];
  load_vec<float, 4>(x + (cls ? r + r / P + 1 : r) * D + c, v);
  store_vec<T, 4>(y + r * D + c, v);
}
