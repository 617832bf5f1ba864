/*
 * endodav_b200 -- C ABI of the B200-native (sm_100a) EndoDAV video-depth forward path.
 *
 * The reference (Zanue/EndoDAV) has no FFI of its own: its boundary for this path is the
 * Python class `endodav` (models/endodav/endodav.py:52-160).  This header is the thin
 * C-ABI extension that the Python host class `endodav_b200.endodav` binds with ctypes;
 * each entry point names the reference code it replaces.
 *
 * Conventions
 *   - every function returns 0 on success or a negative edv_status; never throws;
 *   - all pointers called *_dev are CUDA device pointers owned by the caller (the Python
 *     host allocates them with torch); the library never allocates activation memory;
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it;
 *   - no global state, no internal threads; one edv_ctx per (device, model).
 *   - dtype: EDV_F32 runs fp32 CUDA-core kernels (the "tight" path); EDV_BF16 / EDV_F16
 *     run the tcgen05 tensor-core kernels with 16-bit operands and fp32 accumulation.
 */
#ifndef ENDODAV_B200_H
#define ENDODAV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct edv_ctx edv_ctx;

/* Bumped whenever an entry point's argument list or a struct layout changes.  The ctypes host
 * (endodav_b200/engine.py) mirrors the signatures by hand, so it refuses a library whose
 * edv_abi_version() differs from its own constant instead of calling it with a stale layout. */
#define EDV_ABI_VERSION 13
int edv_abi_version(void);

enum edv_status {
  EDV_OK = 0,
  EDV_ERR_ARG = -1,      /* bad argument / unsupported shape */
  EDV_ERR_CUDA = -2,     /* a CUDA runtime / driver call failed (see edv_last_error) */
  EDV_ERR_WEIGHT = -3,   /* a required packed weight is missing or has the wrong size */
  EDV_ERR_STATE = -4,    /* call order violated (e.g. forward before plan) */
  EDV_ERR_NO_DEVICE = -5 /* no sm_100 device */
};

enum edv_dtype { EDV_F32 = 0, EDV_BF16 = 1, EDV_F16 = 2 };

/* Which matmul engine a 16-bit ctx uses.  EDV_ENGINE_TC (tcgen05/TMEM/TMA) is the product
 * path; EDV_ENGINE_SIMT exists so tests can cross-check the tensor-core kernels against the
 * CUDA-core ones on identical 16-bit operands.  EDV_F32 always uses the SIMT kernels. */
enum edv_engine { EDV_ENGINE_TC = 0, EDV_ENGINE_SIMT = 1 };

/* Model hyper-parameters: mirrors the constructor of the reference class
 * (models/endodav/endodav.py:53-73) after resolving the encoder table
 * (models/backbones/vision_transformer.py:351-398). */
typedef struct edv_config {
  int32_t dim;             /* ViT embed dim: 384 (vits) / 1024 (vitl) */
  int32_t depth;           /* 12 / 24 */
  int32_t heads;           /* 6 / 16 (head dim must be 64) */
  int32_t taps[4];         /* block indices tapped: {2,5,8,11} / {4,11,17,23} (endodav.py:76-79) */
  int32_t features;        /* DPT features: 64 / 256 */
  int32_t out_channels[4]; /* {48,96,192,384} / {256,512,1024,1024} */
  int32_t num_frames;      /* temporal_max_len (<= 32) */
  int32_t conv_head;       /* 0: output_conv1/2 path (disable_conv_head=True); 1: HeadDepth x4 */
  int32_t out_sigmoid;     /* dpt_pyramid.py:98-102 */
  int32_t inv_sigmoid;     /* dpt_pyramid.py:105 */
  int32_t res_blocks;      /* bit i set: ViT block i has a ResBottleneckBlock (block.py:146-150) */
  int32_t rope;            /* 0: sinusoidal APE rows added by the LayerNorm that feeds q|k|v; 1: RoPE on q,k */
  int32_t dtype;           /* edv_dtype */
  int32_t engine;          /* edv_engine */
  int32_t no_motion;       /* 1: no temporal modules -- the `endodac` image model (models/endodac/endodac.py:14-127) */
  int32_t no_normalize;    /* 1: frames enter the patch embedding un-normalised (endodac pre_norm=False, endodac.py:208-211) */
  int32_t use_clstoken;    /* 1: readout projects (dpt.py:92-99; dpt_pyramid.py:54-57): tap' = GELU(Linear(2D, D)([token | class token])) */
  int32_t no_cls;          /* 1: include_cls_token=False -- the ViT runs on the patch tokens only (vision_transformer.py:214-228,
                              319-324; block.py:131-133): S = P tokens, no cls row, pos-embed = the patch rows */
} edv_config;

/* --- context ---------------------------------------------------------------------------- */

/* Replaces: endodav.__init__ + .cuda() (endodav.py:53-147; evaluate_depth_video.py:84-95). */
int edv_create(const edv_config* cfg, edv_ctx** out);
void edv_destroy(edv_ctx* ctx);
const char* edv_last_error(const edv_ctx* ctx); /* ctx may be NULL: last creation error */

/* Register one packed weight tensor (device pointer, borrowed until replaced/destroy).
 * Names and layouts are produced by endodav_b200/pack.py (LoRA merged, LayerScale and
 * q-scale folded, channels padded, conv weights in (ky,kx,c) order).
 * Replaces: load_state_dict (evaluate_depth_video.py:91-93). */
int edv_set_weight(edv_ctx* ctx, const char* name, const void* dev_ptr, size_t bytes);

/* Shape-specialise for clips [B,T,3,H,W] run at network resolution (net_h,net_w)
 * (= image_shape, multiples of 14).  Returns the workspace size the caller must supply. */
int edv_plan(edv_ctx* ctx, int B, int T, int H, int W, int net_h, int net_w, size_t* workspace_bytes);

/* Replaces: endodav.forward (endodav.py:150-160).
 *   frames_dev : [B,T,3,H,W] float32 in [0,1]  (NCHW per frame, as the reference takes it)
 *   disp_dev[s]: [B*T,1,h_s,w_s] float32, s = 0..3 (any may be NULL to skip writing it);
 *                sizes from edv_output_shape.
 *   resized_dev: optional [B*T, out_h, out_w] float32 -- disp0 bilinearly resized
 *                (align_corners=True) to (out_h,out_w): the per-window resize of
 *                infer_video_depth (endodav.py:205); NULL to skip. */
int edv_forward(edv_ctx* ctx, const float* frames_dev, float* const disp_dev[4], float* resized_dev, int out_h,
                int out_w, void* workspace_dev, void* stream);

/* As edv_forward, but frames are uint8 [B*T,H,W,3] (what infer_video_depth receives,
 * endodav.py:162,195) already at network resolution: x/255 -> normalise -> patches. */
int edv_forward_u8(edv_ctx* ctx, const uint8_t* frames_dev, float* const disp_dev[4], float* resized_dev, int out_h,
                   int out_w, void* workspace_dev, void* stream);

int edv_output_shape(const edv_ctx* ctx, int scale, int* h, int* w);

/* CUDA-graph replay.  After the first (eager) forward of a plan, edv_forward captures its launch sequence into a
 * cudaGraphExec keyed by the external INPUT pointers of the call (frames, resized, workspace) and replays it on later
 * calls with the same pointers: no tensor-map encoding and one host launch instead of ~170 -- what the reference's
 * production resolution (224x280, evaluate_depth_video.py:86) needs, where the forward is launch bound.  The disparity
 * pyramid is produced in the plan's own buffers inside the graph and copied to disp[] behind the replay, so callers
 * whose OUTPUT tensors are fresh on every call (any PyTorch caller) still replay.  A pointer set is captured the second
 * time it is seen (callers whose input buffers never repeat stay eager); up to 32 are cached per plan (LRU); edv_plan,
 * edv_set_weight (new pointer) and edv_set_debug drop them; profiling (edv_profile) and debug taps run eagerly.
 * Default on (environment EDV_GRAPH=0 turns it off). */
int edv_set_graph_mode(edv_ctx* ctx, int on);
int edv_graph_count(const edv_ctx* ctx);
/* "ok" after a successful capture, otherwise why the last attempt fell back to eager launches (never NULL). */
const char* edv_graph_status(const edv_ctx* ctx);

/* Number of kernels the last edv_forward launched (bench.py's gpu_launches). */
int edv_launch_count(const edv_ctx* ctx);

/* Live per-launch timing for bench.py's roofline numbers.  With edv_profile(ctx,1) every kernel
 * launch of edv_forward is followed by a CUDA event on the caller's stream; edv_profile_collect
 * waits for them and accumulates, per call site ("gemm_tc:blk.qkv", "spatial_attention_tc", ...),
 * the device time, launch count and the algorithmic FLOPs / bytes of DESIGN.md.  Returns the
 * number of call sites; edv_profile_get reads entry `index`. */
int edv_profile(edv_ctx* ctx, int on);
int edv_profile_reset(edv_ctx* ctx);
int edv_profile_collect(edv_ctx* ctx);
int edv_profile_get(edv_ctx* ctx, int index, char* name, int name_cap, double* ms, long long* count, double* flops,
                    double* bytes);

/* Debug / parity taps.  edv_set_debug(ctx,1) before edv_plan makes edv_forward keep float32
 * snapshots of the stages the oracle records ("tokens0","block0","tap0".."tap3","layer1".."layer4",
 * "mm0","mm1","path4_pre","path3","path1"; NHWC / token-major, real channels only) inside the
 * caller's workspace; edv_debug_tap returns where. */
int edv_set_debug(edv_ctx* ctx, int on);
int edv_debug_tap(edv_ctx* ctx, const char* name, size_t* offset_bytes, long long* rows, int* cols);

/* Enumerate the named workspace buffers of the current plan: index 0,1,... until EDV_ERR_ARG.  elem_bytes is 2
 * for 16-bit activations, 4 for float32 buffers (residual stream, disparities), 8 for float2 statistics.  Used by
 * the fp16 range / saturation tests (tests/test_gpu_fullsize.py) to scan every intermediate for inf / near-overflow. */
int edv_plan_buffer(edv_ctx* ctx, int index, char* name, int name_cap, size_t* offset_bytes, size_t* bytes, int* elem_bytes);

/* --- per-kernel entry points (unit parity tests + ncu) ---------------------------------- */

/* One GEMM / 3x3 convolution through the forward's own dispatcher and kernels, with any epilogue the forward uses:
 *   out = epilogue(A[M,K] * W[N,K]^T)   (A, W in `dtype`, fp32 accumulate; engine as in edv_config)
 * The fields after the conv geometry are those of the library's epilogue description (csrc/common.cuh: Epi), in the
 * order it applies them: + bias[n], + rowbias[(m / rb_div) % rb_mod][n] (row pitch rb_ld), GELU (act 1), row map
 * (map 1 tokens: out row m + m / map_p + 1; map 2 pixel shuffle: column (ky*ps_k + kx)*ps_c + c of grid cell m ->
 * pixel (ps_k y + ky, ps_k x + kx) of a [ps_h ps_k, ps_w ps_k] map), + res1, + res2, ReLU (act 2) or
 * sigmoid(sig_sign x) (act 5), store to out and relu(value) to out_relu.  act 3 (GEGLU: column pairs of 64 value | 64
 * gate per 128, out has N/2 columns) and act 4 (disparity head, N = 32: relu(relu(v + bias) . head_w[0..31] +
 * head_w[32]) or its sigmoid(sig_sign .), one float per row) exist on the tensor-core engine only.
 * *_f32 = 1: that tensor is float32, else `dtype`.  Leading dimensions are in elements and multiples of 8.
 * conv = 1: A is an NHWC activation [F,H,Wd,C], padding 1, K = 9*C in (ky,kx,c) order, M = F*OH*OW; stride 2 runs on
 * the CUDA-core engine only.  struct_bytes must equal sizeof(edv_gemm_desc).
 * `kernel` (may be NULL) receives the kernel instance that ran, e.g. "gemm_tc<BN=32,BK=64,kind=0x9,tma=0>".
 * Replaces: every nn.Linear / 1x1 / 3x3 conv on the path (attention.py:58,67; mlp.py:34-37; dpt.py:100-117; ...). */
typedef struct edv_gemm_desc {
  int32_t struct_bytes;
  const void* A;
  const void* W;
  int32_t M, N, K;
  int64_t lda;
  int32_t conv, F, H, Wd, C, stride;
  void* out;
  void* out_relu;
  const float* bias;
  const float* rowbias;
  const void* res1;
  const void* res2;
  const float* head_w;
  int64_t ldo, ld_res1, ld_res2, rb_ld;
  int32_t rb_div, rb_mod;
  int32_t out_f32, res1_f32, res2_f32;
  int32_t act, map, map_p;
  int32_t ps_k, ps_h, ps_w, ps_c;
  float sig_sign;
} edv_gemm_desc;
int edv_op_gemm(int dtype, int engine, const edv_gemm_desc* d, char* kernel, int kernel_cap, void* stream);

/* C[M,N] = A[M,K] W[N,K]^T (+bias), act 0 none / 1 GELU / 2 ReLU, on the tcgen05 kernel (16-bit dtypes), recording the
 * kernel's own timeline: 4 CTAs x 256 clock64 stamps (per-tile accumulator-free / issued / complete / stored times,
 * slot table in csrc/gemm_tc.cuh). */
int edv_op_linear_timeline(int dtype, const void* A, const void* W, const float* bias, void* C, int M, int N, int K, int act,
                           long long* timeline_dev, void* stream);

/* Row-owning GEMM with fused residual add and LayerNorm (ViT-S, N = 384 only; 16-bit dtypes):
 *   x_inout[M,N] (float32, in place) += A[M,K] W[N,K]^T + bias;  xn_out[M,N] (`dtype`) = LayerNorm(x; gamma, beta, eps).
 * gamma / beta / xn_out NULL: residual update only.  timeline_dev: optional 64 clock64 stamps of the first cluster's
 * epilogue (slot table in csrc/gemm_ln.cuh), else NULL.  Replaces `x = x + ls(proj(.))` / `x = x + ls(fc2(.))` followed by
 * the next norm (layers/block.py:110-116,143-145; LayerScale is folded into W / bias by pack.py). */
int edv_op_linear_residual_ln(int dtype, const void* A, const void* W, const float* bias, float* x_inout, const float* gamma,
                              const float* beta, float eps, void* xn_out, int M, int N, int K, long long* timeline_dev, void* stream);

/* Spatial multi-head attention over token-major qkv [F*S, 3*heads*64] (q pre-scaled) ->
 * out [F*S, heads*64].  Replaces: Attention.forward's softmax(qk^T)v (attention.py:60-66). */
int edv_op_attention(int dtype, int engine, const void* qkv, void* out, int F, int S, int heads, void* stream);

/* edv_op_attention (tcgen05 kernel, 16-bit dtypes) that also records the kernel's own timeline: timeline_dev gets
 * 8 CTAs x 64 clock64 stamps (entry, setup, per-iteration softmax / MMA-issue times; slot table in
 * csrc/attention_tc.cuh).  Diagnostic evidence for the cycle budget in DESIGN.md. */
int edv_op_attention_timeline(int dtype, const void* qkv, void* out, int F, int S, int heads, long long* timeline_dev,
                              void* stream);

/* Temporal attention over the frame axis: qkv [B*T*hw, 3C] (q pre-scaled by hd^-0.5) ->
 * out [B*T*hw, C]; 8 heads; one softmax per (clip, position, head) over T<=32 frames.
 * Replaces: TemporalAttention/CrossAttention._attention (motion_module.py:232-295;
 * motion_module/attention.py:182-211). */
int edv_op_temporal_attention(int dtype, const void* qkv, void* out, int B, int T, int hw, int C, void* stream);

/* Fused disparity-head tail on an NHWC map X[F,H1,W1,Cin] (16-bit, Cin in {32,128}):
 * bilinear resize (align_corners=True) to (OH,OW) -> 3x3 conv Wt[32, 9*Cin] + bias -> ReLU ->
 * 1x1 conv head_w[0..31] + head_w[32] -> ReLU (sig_sign == 0) or sigmoid(sig_sign * x) -> out[F,OH,OW] f32.
 * Replaces dpt_pyramid.py:90-93 + dpt.py:118-124 (output_conv2); layers.py:211-217 (HeadDepth). */
int edv_op_disp_head(int dtype, const void* X, const void* Wt, const float* bias, const float* head_w, float* out, int F,
                     int H1, int W1, int OH, int OW, int Cin, float sig_sign, void* stream);

/* Host preprocessing of infer_video_depth on the GPU: uint8 RGB frames [N,H,W,3] -> float32 [N,3,h,w] =
 * cv2.resize(frame / 255, (w,h), INTER_CUBIC) in CHW order (OpenCV's float bicubic: A=-0.75, half-pixel
 * centres, replicated border).  Replaces endodav.py:195 + util/transform.py:109-113,139-158. */
int edv_op_cubic_resize_u8(const uint8_t* src, float* dst, int N, int H, int W, int h, int w, void* stream);

/* LayerNorm over the last dim: X[M,D] float32 -> Y[M,D] `dtype`. */
int edv_op_layernorm(int dtype, const float* X, const float* gamma, const float* beta, void* Y, int M, int D,
                     float eps, void* stream);

/* GroupNorm(32 groups) over NHWC X[F,hw,C] (`dtype`) -> Y same layout.
 * Replaces: TemporalTransformer3DModel.norm (motion_module.py:84,110). */
int edv_op_groupnorm(int dtype, const void* X, const float* gamma, const float* beta, void* Y, int F, int hw, int C,
                     float eps, void* stream);

/* Bilinear resize, align_corners=True, NHWC `dtype`: X[F,h,w,C] -> Y[F,oh,ow,C].
 * Replaces: F.interpolate calls at util/blocks.py:156-158, dpt_pyramid.py:90-92. */
int edv_op_upsample(int dtype, const void* X, void* Y, int F, int h, int w, int oh, int ow, int C, void* stream);

/* Bilinear resize of single-channel float32 maps (align_corners=True): disp pyramid
 * (dpt_pyramid.py:95-97) and the final resize of infer_video_depth (endodav.py:205). */
int edv_op_resize_f32(const float* X, float* Y, int F, int h, int w, int oh, int ow, void* stream);

/* On-GPU stitching of infer_video_depth, one window per call (stream-ordered, no host sync):
 * window k [32,H,W] float32 (already resized to the frame size) is aligned to the frames stitched so
 * far by the reference's least-squares (scale, shift) over the 8 overlap frames, clamped at 0, its
 * overlap cross-faded into out_dev's last 8 frames and its 22 fresh frames appended; k = 0 copies the
 * 32 frames.  Windows must be submitted in order k = 0,1,2,...  out_dev holds 32 + 22*(n_windows-1)
 * frames; scale_shift_dev [n_windows][2] receives (scale, shift) of every window.
 * Replaces endodav.py:213-254 + utils/util.py:40-74 (compute_scale_and_shift_full,
 * get_interpolate_frames) BIT-EXACTLY: float32 arithmetic op for op without FMA contraction, and the
 * np.sum reductions in numpy's own pairwise association order.  That order is a function of
 * n = 8*H*W only; edv_op_stitch_plan (host-only, no GPU needed) writes it as an int32 table
 * (returns the number of int32 it needs; call with plan_host = NULL to size it; negative on error,
 * e.g. 8*H*W >= 2^24).  The caller uploads the table (plan_dev), passes n_leaves = plan[0] and a
 * 16-byte-aligned scratch of 4*(plan[0]+plan[1]) floats. */
long long edv_op_stitch_plan(int H, int W, int32_t* plan_host, long long cap);
int edv_op_stitch_window(const float* win_dev, int k, int H, int W, float* out_dev, const int32_t* plan_dev, int n_leaves,
                         float* scratch_dev, float* scale_shift_dev, void* stream);

/* Depth conversion of the evaluate scripts on the GPU: scaled_disp = 1/max_depth + (1/min_depth - 1/max_depth) * disp,
 * depth = 1 / scaled_disp over n float32 elements (scaled_disp_dev may be NULL).  float32 arithmetic op for op, so the
 * result is bit-identical to the numpy expression.  Replaces disp_to_depth (utils/layers.py:11-20) as called at
 * evaluate_depth_video.py:170. */
int edv_op_disp_to_depth(const float* disp_dev, float* scaled_disp_dev, float* depth_dev, long long n, double min_depth,
                         double max_depth, void* stream);

/* Per-frame depth metrics: out_dev[f][0..7] = abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3, valid-pixel count (float64)
 * for frames f of gt_dev / pred_dev [frames][hw] float32.  Valid pixels: mask_dev (uint8 [frames][hw]) when given, else
 * gt in (gt_lo, gt_hi); pred is multiplied by pred_scale and clamped to [clamp_lo, clamp_hi] first (clamp_lo > clamp_hi
 * skips the clamp).  One block per frame, fixed summation order (bit-reproducible); a frame without valid pixels gives
 * NaNs like numpy.  Replaces compute_errors (utils/utils.py:112-133) and the per-frame masking / scaling / clamping
 * loop around it (evaluate_depth_video.py:197-204). */
int edv_op_compute_errors(const float* gt_dev, const float* pred_dev, const uint8_t* mask_dev, int frames, long long hw,
                          float gt_lo, float gt_hi, float pred_scale, float clamp_lo, float clamp_hi, double* out_dev,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ENDODAV_B200_H */
