"""The forward's non-GEMM launches, each through the launcher the forward calls, at the arguments it passes, against a
float64 reference.

One case per call site of csrc/engine.cu (preprocess_patches, tokens_to_patches, rowln_act, resblock_add, im2col3x3,
geglu_pair, head_dot, the LayerNorm row-selection and frame-table modes, out_sigmoid), with the shapes the forward
passes for ViT-S (D = 384), ViT-B (endodac base, D = 768) and ViT-L (D = 1024), at 518 x 518 (37 x 37 patches) and at a
small shape with tails.  As in test_gpu_epilogues.py: operands are rounded to the dtype first, the reference is float64
on those operands, outputs live in NaN-filled buffers whose guard rows must stay NaN, and side tables are followed in
the same allocation by at least as many NaN rows as they have, so that a row index running past a table reads NaN.

test_every_kernel_is_covered (no GPU) keeps a table of every __global__ kernel of csrc/ and the tests that reach it."""
import ast
import os
import re

import pytest
import torch
import torch.nn.functional as F

from endodav_b200 import engine as eng

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda"
DTYPES = [torch.float32, torch.bfloat16, torch.float16]
GUARD = 136
NAN = float("nan")
D_VIT = [384, 768, 1024]                       # ViT-S, ViT-B (endodac base), ViT-L
GRIDS = [(2, 37, 37), (3, 5, 7)]               # (frames, patch rows, patch cols): 518 x 518 and a 70 x 98 tail


def _rand(shape, dtype, seed, scale=1.0, shift=0.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(shape, generator=g, device=DEV) * scale + shift).to(dtype)


def _tol(dtype):
    # relative output rounding: bf16 2^-8, f16 2^-11, fp32 accumulate-order noise
    return {torch.float32: 2e-5, torch.bfloat16: 2 ** -8, torch.float16: 2 ** -11}[dtype]


WORST = {}   # case -> worst error as a fraction of its tolerance (printed at the end of the module)


def _close(got, ref, dtype, what, slack=2.0):
    """|got - ref| <= slack * tol(dtype) * max(|ref|, 1) + 1e-5; records the worst fraction of that bound."""
    err = (got.double() - ref).abs()
    bound = slack * _tol(dtype) * ref.abs().clamp_min(1.0) + 1e-5
    bad = ~(err <= bound)
    assert not bool(bad.any()), "%s: max err %.4g (ref max %.4g), %d / %d over tolerance" % (
        what, float(err.nan_to_num(float("inf")).max()), float(ref.abs().max()), int(bad.sum()), bad.numel())
    _note(what.split(" ")[0], float((err / bound).max()) if err.numel() else 0.0)


def _note(name, frac):
    WORST[name] = max(WORST.get(name, 0.0), frac)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        print("\nworst error / tolerance per case:")
        for k in sorted(WORST):
            print("  %-32s %.3f" % (k, WORST[k]))


def _nan_rows(rows, cols, dtype):
    return torch.full((rows + GUARD, cols), NAN, dtype=dtype, device=DEV)


def _guard_ok(buf, rows, what):
    assert bool(buf[rows:].float().isnan().all()), "%s: guard rows beyond the output were written" % what


def _dt_id(dtype):
    return str(dtype).replace("torch.", "")


# ---- K1: resize + normalise + 14 x 14 im2col (engine.cu run, preprocess_patches) ------------------------------------
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


def _patches_ref(img, normalize):
    """img float32 [F,3,h,w] -> float64 [F*(h/14)*(w/14), 588]."""
    x = img.double()
    if normalize:
        x = (x - torch.tensor(MEAN, dtype=torch.float64, device=DEV).view(1, 3, 1, 1)) / \
            torch.tensor(STD, dtype=torch.float64, device=DEV).view(1, 3, 1, 1)
    return F.unfold(x, 14, stride=14).transpose(1, 2).reshape(-1, 588)


def _check_patches(out, ref, M, dtype, what):
    _guard_ok(out, M, what)
    assert bool((out[:M, 588:] == 0).all()), "%s: padding columns 588..639 are not zero" % what
    _close(out[:M, :588], ref, dtype, what)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt_id)
@pytest.mark.parametrize("normalize", [1, 0])
@pytest.mark.parametrize("H,W,h,w", [(256, 320, 224, 280), (80, 112, 70, 98), (42, 56, 42, 56), (480, 640, 518, 518)])
def test_preprocess_patches(H, W, h, w, normalize, dtype):
    Fr = 2
    frames = torch.rand(Fr, 3, H, W, generator=torch.Generator(device=DEV).manual_seed(H + W), device=DEV)
    M = Fr * (h // 14) * (w // 14)
    out = _nan_rows(M, 640, dtype)
    eng.op_preprocess_patches(frames, h, w, out, normalize=bool(normalize))
    # source coordinates in float32 exactly like ATen's upsample_bilinear2d (see test_gpu_ops.test_resize_f32)
    img = frames if (H, W) == (h, w) else F.interpolate(frames, size=(h, w), mode="bilinear", align_corners=True)
    _check_patches(out, _patches_ref(img, normalize), M, dtype, "preprocess %dx%d->%dx%d norm=%d %s" % (H, W, h, w, normalize, dtype))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt_id)
@pytest.mark.parametrize("normalize", [1, 0])
@pytest.mark.parametrize("h,w", [(518, 518), (70, 98)])
def test_preprocess_patches_u8(h, w, normalize, dtype):
    Fr = 3
    g = torch.Generator(device=DEV).manual_seed(h * w)
    frames = torch.randint(0, 256, (Fr, h, w, 3), generator=g, device=DEV, dtype=torch.uint8)
    M = Fr * (h // 14) * (w // 14)
    out = _nan_rows(M, 640, dtype)
    eng.op_preprocess_patches(frames, h, w, out, normalize=bool(normalize))
    img = (frames.float() / 255.0).permute(0, 3, 1, 2)          # x / 255 in float32, as the kernel divides
    _check_patches(out, _patches_ref(img, normalize), M, dtype, "preprocess_u8 %dx%d norm=%d %s" % (h, w, normalize, dtype))


# ---- ResBottleneckBlock (engine.cu res_block) -------------------------------------------------------------------------
def _tokens(BT, P, D, cls, seed):
    """float32 [BT*(P + cls), D] token stream; cls rows are NaN so that reading one shows."""
    x = _rand((BT, P + cls, D), torch.float32, seed, 2.0)
    if cls:
        x[:, 0] = NAN
    return x.reshape(-1, D)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt_id)
@pytest.mark.parametrize("cls", [1, 0])
@pytest.mark.parametrize("D", D_VIT)
@pytest.mark.parametrize("BT,ph,pw", GRIDS)
def test_tokens_to_patches(BT, ph, pw, D, cls, dtype):
    P = ph * pw
    Mp = BT * P
    x = _tokens(BT, P, D, cls, 21)
    out = _nan_rows(Mp, D, dtype)
    eng.op_tokens_to_patches(x, out, Mp, P, D, cls)
    _guard_ok(out, Mp, "tokens_to_patches")
    assert torch.equal(out[:Mp], x.view(BT, P + cls, D)[:, cls:].reshape(Mp, D).to(dtype))
    _note("tokens_to_patches", 0.0)


def _ln_gelu_ref(x, g, b, Cr, eps):
    v = x[:, :Cr].double()
    y = F.layer_norm(v, (Cr,), g[:Cr].double(), b[:Cr].double(), eps)
    return F.gelu(y)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt_id)
@pytest.mark.parametrize("Cr,C", [(48, 64), (96, 128), (128, 128)])     # round_up(D/8, 64) for D = 384, 768, 1024
@pytest.mark.parametrize("BT,ph,pw", GRIDS)
def test_rowln_act(BT, ph, pw, Cr, C, dtype):
    M = BT * ph * pw
    x = _rand((M, C), dtype, 22, 1.5, 0.7)
    x[:, Cr:] = NAN                                            # padding channels must never be read
    g, b = _rand((C,), torch.float32, 23, 0.3, 1.0), _rand((C,), torch.float32, 24, 0.2)
    y = _nan_rows(M, C, dtype)
    eng.op_rowln_act(x, g, b, y, M, C, Cr, 1e-6, True)
    _guard_ok(y, M, "rowln_act")
    pad = y[:M, Cr:].float()
    assert bool((pad == 0).all()) and not bool(torch.signbit(pad).any()), "rowln_act: padding columns are not +0"
    _close(y[:M, :Cr], _ln_gelu_ref(x, g, b, Cr, 1e-6), dtype, "rowln_act Cr=%d C=%d %s" % (Cr, C, dtype))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt_id)
@pytest.mark.parametrize("cls", [1, 0])
@pytest.mark.parametrize("D", D_VIT)
@pytest.mark.parametrize("BT,ph,pw", GRIDS)
def test_resblock_add(BT, ph, pw, D, cls, dtype):
    P = ph * pw
    Mp, rows = BT * P, BT * (P + cls)
    buf = _nan_rows(rows, D, torch.float32)
    buf[:rows] = _rand((rows, D), torch.float32, 25, 2.0)
    before = buf.clone()
    r = _rand((Mp, D), dtype, 26, 1.5, 0.3)
    g, b = _rand((D,), torch.float32, 27, 0.3, 1.0), _rand((D,), torch.float32, 28, 0.2)
    eng.op_resblock_add(buf, r, g, b, Mp, P, D, cls)
    _guard_ok(buf, rows, "resblock_add")
    view, old = buf[:rows].view(BT, P + cls, D), before[:rows].view(BT, P + cls, D)
    if cls:
        assert torch.equal(view[:, 0], old[:, 0]), "resblock_add: cls rows changed"
    ref = old[:, cls:].double() + F.layer_norm(r.double(), (D,), g.double(), b.double(), 1e-6).view(BT, P, D)
    _close(view[:, cls:], ref, torch.float32, "resblock_add D=%d cls=%d %s" % (D, cls, dtype))


# ---- resize_layers[3] on the tensor-core path (engine.cu run, im2col3x3) ----------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt_id)
@pytest.mark.parametrize("Fr,H,W,C", [(2, 37, 37, 384), (1, 3, 4, 384), (1, 5, 7, 1024), (2, 16, 20, 768)])
def test_im2col3x3(Fr, H, W, C, dtype):
    x = _rand((Fr, H, W, C), dtype, 29)
    OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    M = Fr * OH * OW
    out = _nan_rows(M, 9 * C, dtype)
    eng.op_im2col3x3(x, out, stride=2)
    _guard_ok(out, M, "im2col3x3")
    cols = F.unfold(x.permute(0, 3, 1, 2).float(), 3, padding=1, stride=2)           # [F, (c,ky,kx), L]
    ref = cols.view(Fr, C, 9, OH * OW).permute(0, 3, 2, 1).reshape(M, 9 * C).to(dtype)
    assert torch.equal(out[:M], ref)
    _note("im2col3x3", 0.0)


# ---- the CUDA-core engine's GEGLU and head tail (engine.cu motion / disp_head) ----------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt_id)
@pytest.mark.parametrize("C", [64, 192, 384, 256, 1024])               # ViT-S / ViT-B / ViT-L temporal-module channels
@pytest.mark.parametrize("M", [2 * 37 * 37, 3 * 5 * 7])
def test_geglu_pair(M, C, dtype):
    C4 = 4 * C
    hg = _rand((M, 2 * C4), dtype, 30, 1.5)
    out = _nan_rows(M, C4, dtype)
    eng.op_geglu_pair(hg, out, M, C4)
    _guard_ok(out, M, "geglu_pair")
    t = hg.double().view(M, C4 // 64, 2, 64)                    # column blocks [64 value | 64 gate] (pack.py)
    ref = (t[:, :, 0] * F.gelu(t[:, :, 1])).reshape(M, C4)
    _close(out[:M], ref, dtype, "geglu_pair C=%d %s" % (C, dtype))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt_id)
@pytest.mark.parametrize("sig", [0.0, 1.0, -1.0])
@pytest.mark.parametrize("M", [2 * 518 * 518, 3 * 70 * 98 + 5])
def test_head_dot(M, sig, dtype):
    x = F.relu(_rand((M, 32), torch.float32, 31, 1.0, 0.2)).to(dtype)   # the ReLU'd 32-channel map
    w = _rand((33,), torch.float32, 32, 0.3)
    w[32] = 0.5                                                 # the 1x1 bias sits in w[32]
    out = torch.full((M + GUARD,), NAN, dtype=torch.float32, device=DEV)
    eng.op_head_dot(x, w, out, M, 32, sig)
    _guard_ok(out, M, "head_dot")
    xd = x.double()
    s = xd @ w[:32].double() + float(w[32])
    ref = F.relu(s) if sig == 0.0 else torch.sigmoid(sig * s)
    # fp32 dot product of 32 terms: about 1e-5 of sum |x| |w| (sigmoid only shrinks the error)
    bound = 1e-5 * (xd.abs() @ w[:32].double().abs() + abs(float(w[32])))
    err = (out[:M].double() - ref).abs()
    assert bool((err <= bound).all()), "head_dot sig=%g: max err %.3g" % (sig, float(err.max()))
    _note("head_dot", float((err / bound).max()))


# ---- LayerNorm modes (engine.cu run: taps + cls split, use_clstoken readout; motion: + PE of the frame) ---------------
LN_D = [64, 192, 384, 768, 1024]                          # every MAXV instance the forward launches (1, 2, 3, 8)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt_id)
@pytest.mark.parametrize("D", LN_D)
@pytest.mark.parametrize("BT,ph,pw", GRIDS)
def test_layernorm_row_selection(BT, ph, pw, D, dtype):
    """grp = N, skip = 1 (the four tap norms without the cls rows) equals, bit for bit, the plain norm of the patch rows;
    skip = -1 (the class tokens of the readout) equals the plain norm of the cls rows."""
    P = ph * pw
    N = P + 1
    x = _rand((BT * N, D), torch.float32, 33, 3.0, 1.5)
    g, b = _rand((D,), torch.float32, 34), _rand((D,), torch.float32, 35)
    xv = x.view(BT, N, D)
    patches, clsr = xv[:, 1:].reshape(-1, D).contiguous(), xv[:, 0].contiguous()
    plain = eng.op_layernorm(patches, g, b, 1e-6, dtype)
    _close(plain, F.layer_norm(patches.double(), (D,), g.double(), b.double(), 1e-6), dtype, "layernorm D=%d %s" % (D, dtype), 4.0)
    out = _nan_rows(BT * P, D, dtype)
    eng.op_layernorm(x, g, b, 1e-6, dtype, grp=N, skip=1, out=out)
    _guard_ok(out, BT * P, "layernorm skip=1")
    assert torch.equal(out[:BT * P], plain)
    cout = _nan_rows(BT, D, dtype)
    eng.op_layernorm(x, g, b, 1e-6, dtype, grp=N, skip=-1, out=cout)
    _guard_ok(cout, BT, "layernorm skip=-1")
    assert torch.equal(cout[:BT], eng.op_layernorm(clsr, g, b, 1e-6, dtype))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=_dt_id)
@pytest.mark.parametrize("D", LN_D)
@pytest.mark.parametrize("T,hw", [(5, 7), (32, 7), (5, 19 * 19), (32, 37)])
def test_layernorm_frame_table(T, hw, D, dtype):
    """+ pe[frame] after the affine, rows (b, f, position) of B = 2 clips: add_div = hw, add_mod = T."""
    B = 2
    M = B * T * hw
    x = _rand((M, D), torch.float32, 36, 3.0, 1.5)
    g, b = _rand((D,), torch.float32, 37), _rand((D,), torch.float32, 38)
    table = torch.full((2 * T, D), NAN, dtype=torch.float32, device=DEV)       # T rows, then T NaN guard rows
    table[:T] = _rand((T, D), torch.float32, 39)
    out = _nan_rows(M, D, dtype)
    eng.op_layernorm(x, g, b, 1e-5, dtype, add=table, add_div=hw, add_mod=T, out=out)
    _guard_ok(out, M, "layernorm add")
    frame = (torch.arange(M, device=DEV) // hw) % T
    ref = F.layer_norm(x.double(), (D,), g.double(), b.double(), 1e-5) + table[:T].double()[frame]
    _close(out[:M], ref, dtype, "layernorm_pe D=%d T=%d %s" % (D, T, dtype), 4.0)


# ---- out_sigmoid (engine.cu run, !conv_head: sigmoid_inplace over the pyramid) ----------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["fp32", "fp16"])
def test_out_sigmoid_is_sigmoid_of_the_pyramid(dtype):
    import endodav_b200 as E
    from golden_util import oracle_cfg
    from oracle import weights

    ctor = dict(encoder="vits", features=64, out_channels=[48, 96, 192, 384], r=4, lora_type="dvlora", image_shape=(70, 98),
                disable_conv_head=True, residual_block_indexes=[])
    sd = weights.make_state_dict(oracle_cfg(ctor), 7)
    x = weights.make_frames(1, 3, 80, 112, 8).cuda()
    outs = []
    for sig in (False, True):
        model = E.endodav(dtype=dtype, out_sigmoid=sig, **ctor)
        model.load_state_dict(sd, strict=True)
        model = model.cuda().eval()
        o = model(x)
        outs.append([o[("disp", s)].clone() for s in range(4)])
    for s in range(4):
        raw, got = outs[0][s], outs[1][s]
        assert got.shape == raw.shape and bool(torch.isfinite(got).all())
        err = float((got.double() - torch.sigmoid(raw.double())).abs().max())
        assert err <= 1e-6, (s, err)
        _note("out_sigmoid", err / 1e-6)


# ---- every kernel has a test (no GPU) -----------------------------------------------------------------------------------
# kernel -> "test module::test function" that runs it
COVERED = {
    "preprocess_patches_kernel": ["test_gpu_forward_kernels::test_preprocess_patches", "test_gpu_forward_kernels::test_preprocess_patches_u8"],
    "tokens_to_patches_kernel": ["test_gpu_forward_kernels::test_tokens_to_patches"],
    "rowln_act_kernel": ["test_gpu_forward_kernels::test_rowln_act"],
    "resblock_add_kernel": ["test_gpu_forward_kernels::test_resblock_add"],
    "im2col3x3_kernel": ["test_gpu_forward_kernels::test_im2col3x3"],
    "geglu_pair_kernel": ["test_gpu_forward_kernels::test_geglu_pair"],
    "head_dot_kernel": ["test_gpu_forward_kernels::test_head_dot"],
    "sigmoid_inplace_kernel": ["test_gpu_forward_kernels::test_out_sigmoid_is_sigmoid_of_the_pyramid"],
    "layernorm_kernel": ["test_gpu_ops::test_layernorm", "test_gpu_forward_kernels::test_layernorm_row_selection",
                         "test_gpu_forward_kernels::test_layernorm_frame_table"],
    "cubic_resize_u8_kernel": ["test_gpu_ops::test_cubic_resize_u8_matches_cv2"],
    "groupnorm_stats_kernel": ["test_gpu_ops::test_groupnorm"],
    "groupnorm_partial_kernel": ["test_gpu_ops::test_groupnorm"],
    "groupnorm_finalize_kernel": ["test_gpu_ops::test_groupnorm"],
    "groupnorm_apply_kernel": ["test_gpu_ops::test_groupnorm"],
    "upsample_nhwc_kernel": ["test_gpu_ops::test_upsample_nhwc"],
    "resize_f32_kernel": ["test_gpu_ops::test_resize_f32"],
    "temporal_attention_mma_kernel": ["test_gpu_ops::test_temporal_attention"],
    "temporal_attention_kernel": ["test_gpu_ops::test_temporal_attention"],
    "spatial_attention_simt_kernel": ["test_gpu_ops::test_attention_fp32", "test_gpu_ops::test_attention_16bit",
                                      "test_gpu_attention::test_attention_forward_shapes", "test_gpu_attention::test_attention_tails",
                                      "test_gpu_attention::test_attention_frames_are_independent",
                                      "test_gpu_attention::test_attention_poisoned_neighbour",
                                      "test_gpu_attention::test_attention_lazy_rescale"],
    "flash_attention_tc_kernel": ["test_gpu_ops::test_attention_16bit", "test_gpu_attention::test_attention_forward_shapes",
                                  "test_gpu_attention::test_attention_tails", "test_gpu_attention::test_attention_frames_are_independent",
                                  "test_gpu_attention::test_attention_poisoned_neighbour",
                                  "test_gpu_attention::test_attention_lazy_rescale"],
    "gemm_simt_kernel": ["test_gpu_ops::test_linear_fp32", "test_gpu_epilogues::test_epilogue_matches_reference"],
    "gemm_tc_kernel": ["test_gpu_ops::test_linear_16bit", "test_gpu_epilogues::test_epilogue_matches_reference"],
    "gemm_bres_kernel": ["test_gpu_ops::test_linear_kernels_agree_bitwise", "test_gpu_epilogues::test_epilogue_matches_reference"],
    "conv3x3_halo_kernel": ["test_gpu_ops::test_conv3x3_16bit", "test_gpu_epilogues::test_epilogue_matches_reference"],
    "gemm_ln_kernel": ["test_gpu_gemm_ln::test_gemm_ln_forward_shapes", "test_gpu_gemm_ln::test_gemm_ln_grid_edges",
                       "test_gpu_gemm_ln::test_gemm_ln_ring_edges", "test_gpu_gemm_ln::test_gemm_ln_families",
                       "test_gpu_gemm_ln::test_gemm_ln_shapes", "test_gpu_gemm_ln::test_gemm_ln_rows_do_not_depend_on_position",
                       "test_gpu_gemm_ln::test_gemm_ln_dependent_launches"],
    "head_fused_kernel": ["test_gpu_head::test_head_dpt_shapes", "test_gpu_head::test_head_conv_head_shapes",
                          "test_gpu_head::test_head_tails", "test_gpu_head::test_head_small_shapes",
                          "test_gpu_head::test_head_grid_sizes", "test_gpu_head::test_head_frames_are_independent",
                          "test_gpu_head::test_head_poisoned_neighbour"],
    "stitch_leaf_kernel": ["test_gpu_stitch::test_stitch_matches_numpy_chain"],
    "stitch_tree_solve_kernel": ["test_gpu_stitch::test_stitch_matches_numpy_chain"],
    "stitch_identity_kernel": ["test_gpu_stitch::test_stitch_matches_numpy_chain"],
    "stitch_apply_kernel": ["test_gpu_stitch::test_stitch_matches_numpy_chain"],
    "disp_to_depth_kernel": ["test_metrics::test_gpu_disp_to_depth_is_bit_exact"],
    "compute_errors_kernel": ["test_metrics::test_gpu_compute_errors_matches_reference"],
}
# kernel -> (why it has no per-kernel test, the test that still runs it)
EXCLUDED = {
    "copy_channels_f32_kernel": ("debug taps only", "test_gpu_forward::test_stage_taps_fp32_match_oracle"),
    "copy_pyramid_kernel": ("copies the four disparity levels behind a graph replay; every level is compared",
                            "test_gpu_forward::test_cuda_graph_replay_on_default_stream_is_bit_identical"),
    "cls_row_kernel": ("fp32-only, the same instance in every dtype; held to 3e-4 by the tokens0 tap",
                       "test_gpu_forward::test_stage_taps_fp32_match_oracle"),
}


def _kernels():
    csrc = os.path.join(ROOT, "endodav_b200", "csrc")
    names = set()
    for f in os.listdir(csrc):
        if f.endswith((".cu", ".cuh", ".h")):
            with open(os.path.join(csrc, f)) as fh:
                src = re.sub(r"//[^\n]*|/\*.*?\*/", "", fh.read(), flags=re.S)
            names.update(re.findall(r"__global__\s+(?:void\s+|(?:__launch_bounds__|__cluster_dims__)\s*\((?:[^()]|\([^()]*\))*\)\s*)*"
                                    r"(\w+)\s*\(", src))
    return names


def _test_functions(module):
    with open(os.path.join(ROOT, "tests", module + ".py")) as f:
        tree = ast.parse(f.read())
    return {n.name for n in tree.body if isinstance(n, ast.FunctionDef) and n.name.startswith("test_")}


def test_every_kernel_is_covered():
    kernels = _kernels()
    assert "layernorm_kernel" in kernels and "copy_pyramid_kernel" in kernels and len(kernels) >= 30, sorted(kernels)
    missing = kernels - set(COVERED) - set(EXCLUDED)
    assert not missing, "kernels without a test (add one, or an EXCLUDED reason): %s" % sorted(missing)
    stale = (set(COVERED) | set(EXCLUDED)) - kernels
    assert not stale, "listed kernels that no longer exist: %s" % sorted(stale)
    assert not set(COVERED) & set(EXCLUDED)
    for k, tests in list(COVERED.items()) + [(k, [t]) for k, (_, t) in EXCLUDED.items()]:
        for t in tests:
            mod, fn = t.split("::")
            assert fn in _test_functions(mod), "%s: %s does not exist" % (k, t)
