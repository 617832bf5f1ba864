"""Per-kernel parity on a real B200, through the C ABI (endodav_b200.engine.op_*).

Each kernel is compared with a plain fp32 PyTorch statement of the same op on the same
(already rounded) operands; tolerances are written beside each comparison.  The fp32
CUDA-core kernels are held to fp32 round-off, the 16-bit tensor-core kernels to the output
rounding of their dtype (operands are identical on both sides, accumulation is fp32)."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from endodav_b200 import engine as eng  # noqa: E402

DEV = "cuda"
DT16 = [torch.bfloat16, torch.float16]


def _rand(shape, dtype, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(dtype).to(DEV)


def _tol(dtype):
    # relative output rounding: bf16 2^-8, f16 2^-11, fp32 accumulate-order noise
    return {torch.float32: 2e-5, torch.bfloat16: 2 ** -8, torch.float16: 2 ** -11}[dtype]


def _close(got, ref, dtype, what, slack=2.0):
    got = got.float()
    err = (got - ref).abs()
    bound = slack * _tol(dtype) * ref.abs().clamp_min(1.0) + 1e-5
    bad = err > bound
    assert not bool(bad.any()), "%s: max err %.4g (ref max %.4g), %d / %d over tolerance" % (
        what, float(err.max()), float(ref.abs().max()), int(bad.sum()), bad.numel())


# ---- linear -------------------------------------------------------------------------------
LIN_SHAPES = [(128, 128, 64), (300, 384, 384), (1000, 1152, 384), (257, 64, 32), (77, 96, 1536), (2568, 1536, 384),
              (130, 32, 96), (4000, 256, 192)]


@pytest.mark.parametrize("M,N,K", LIN_SHAPES)
@pytest.mark.parametrize("act", [0, 1, 2])
def test_linear_fp32(M, N, K, act):
    A, W, b = _rand((M, K), torch.float32, 1), _rand((N, K), torch.float32, 2, K ** -0.5), _rand((N,), torch.float32, 3)
    got = eng.op_linear(A, W, b, act, eng.ENGINE_SIMT)
    ref = F.linear(A.double(), W.double(), b.double())
    ref = F.gelu(ref) if act == 1 else F.relu(ref) if act == 2 else ref
    _close(got, ref.float(), torch.float32, "linear fp32", slack=4.0)


@pytest.mark.parametrize("dtype", DT16)
@pytest.mark.parametrize("engine", [eng.ENGINE_TC, eng.ENGINE_SIMT])
@pytest.mark.parametrize("M,N,K", LIN_SHAPES)
@pytest.mark.parametrize("act", [0, 1, 2])
def test_linear_16bit(dtype, engine, M, N, K, act):
    A, W, b = _rand((M, K), dtype, 1), _rand((N, K), dtype, 2, K ** -0.5), _rand((N,), torch.float32, 3)
    got = eng.op_linear(A, W, b, act, engine)
    ref = F.linear(A.double(), W.double(), b.double())
    ref = F.gelu(ref) if act == 1 else F.relu(ref) if act == 2 else ref
    _close(got, ref.float(), dtype, "linear %s engine %d" % (dtype, engine))


def test_linear_tc_equals_simt_bitwise_inputs():
    """Same 16-bit operands through both engines: only fp32 summation order may differ."""
    A, W = _rand((1370, 384), torch.bfloat16, 5), _rand((1536, 384), torch.bfloat16, 6, 0.05)
    a = eng.op_linear(A, W, None, 0, eng.ENGINE_TC).float()
    b = eng.op_linear(A, W, None, 0, eng.ENGINE_SIMT).float()
    assert float((a - b).abs().max()) <= 2 ** -7 * float(b.abs().max())


# ---- conv3x3 ------------------------------------------------------------------------------
CONV_SHAPES = [(2, 16, 20, 64, 64), (3, 5, 7, 64, 64), (1, 37, 37, 192, 64), (2, 19, 19, 384, 64), (1, 64, 80, 64, 32),
               (2, 33, 47, 32, 32), (1, 8, 10, 128, 128), (1, 128, 160, 64, 64)]


def _conv_ref(X, Wt, b, relu):
    Fr, H, W, C = X.shape
    O = Wt.shape[0]
    w4 = Wt.double().reshape(O, 3, 3, C).permute(0, 3, 1, 2)
    y = F.conv2d(X.double().permute(0, 3, 1, 2), w4, b.double() if b is not None else None, padding=1).permute(0, 2, 3, 1)
    return (F.relu(y) if relu else y).float()


@pytest.mark.parametrize("Fr,H,W,C,O", CONV_SHAPES)
def test_conv3x3_fp32(Fr, H, W, C, O):
    X, Wt, b = _rand((Fr, H, W, C), torch.float32, 1), _rand((O, 9 * C), torch.float32, 2, (9 * C) ** -0.5), _rand((O,), torch.float32, 3)
    got = eng.op_conv3x3(X, Wt, b, True, eng.ENGINE_SIMT)
    _close(got, _conv_ref(X, Wt, b, True), torch.float32, "conv fp32", slack=4.0)


@pytest.mark.parametrize("dtype", DT16)
@pytest.mark.parametrize("engine", [eng.ENGINE_TC, eng.ENGINE_SIMT])
@pytest.mark.parametrize("Fr,H,W,C,O", CONV_SHAPES)
def test_conv3x3_16bit(dtype, engine, Fr, H, W, C, O):
    X, Wt, b = _rand((Fr, H, W, C), dtype, 1), _rand((O, 9 * C), dtype, 2, (9 * C) ** -0.5), _rand((O,), torch.float32, 3)
    got = eng.op_conv3x3(X, Wt, b, False, engine)
    _close(got, _conv_ref(X, Wt, b, False), dtype, "conv %s engine %d" % (dtype, engine))


# ---- spatial attention --------------------------------------------------------------------
def _attn_ref(qkv, Fr, S, heads):
    D = heads * 64
    t = qkv.double().reshape(Fr, S, 3, heads, 64).permute(2, 0, 3, 1, 4)
    o = (t[0] @ t[1].transpose(-1, -2)).softmax(-1) @ t[2]
    return o.transpose(1, 2).reshape(Fr * S, D).float()


ATT_SHAPES = [(2, 321, 6), (1, 1370, 6), (3, 17, 6), (1, 128, 2), (2, 129, 16), (1, 26, 1), (1, 256, 3), (1, 300, 6)]


@pytest.mark.parametrize("Fr,S,heads", ATT_SHAPES)
def test_attention_fp32(Fr, S, heads):
    qkv = _rand((Fr * S, 3 * heads * 64), torch.float32, 7, 0.5)
    got = eng.op_attention(qkv, Fr, S, heads, eng.ENGINE_SIMT)
    _close(got, _attn_ref(qkv, Fr, S, heads), torch.float32, "attention fp32", slack=8.0)


@pytest.mark.parametrize("dtype", DT16)
@pytest.mark.parametrize("engine", [eng.ENGINE_TC, eng.ENGINE_SIMT])
@pytest.mark.parametrize("Fr,S,heads", ATT_SHAPES)
def test_attention_16bit(dtype, engine, Fr, S, heads):
    qkv = _rand((Fr * S, 3 * heads * 64), dtype, 7, 0.5)
    got = eng.op_attention(qkv, Fr, S, heads, engine)
    # the tensor-core kernel rounds P to 16 bits before P@V: allow 2x the output rounding
    _close(got, _attn_ref(qkv, Fr, S, heads), dtype, "attention %s engine %d" % (dtype, engine), slack=3.0)


def test_attention_peaked_softmax():
    """Large logits (|s| ~ 40): online softmax must not overflow or lose the dominant key."""
    Fr, S, heads = 1, 400, 2
    qkv = _rand((Fr * S, 3 * heads * 64), torch.bfloat16, 9, 1.0)
    qkv[:, : heads * 64] *= 4.0
    for engine in (eng.ENGINE_TC, eng.ENGINE_SIMT):
        got = eng.op_attention(qkv, Fr, S, heads, engine)
        assert bool(torch.isfinite(got.float()).all())
        _close(got, _attn_ref(qkv, Fr, S, heads), torch.bfloat16, "peaked attention", slack=4.0)


# ---- temporal attention ---------------------------------------------------------------------
def _tattn_ref(qkv, B, T, hw, C):
    hd = C // 8
    t = qkv.double().reshape(B, T, hw, 3, 8, hd).permute(3, 0, 2, 4, 1, 5)  # which, B, hw, head, T, hd
    o = (t[0] @ t[1].transpose(-1, -2)).softmax(-1) @ t[2]                   # B, hw, head, T, hd
    return o.permute(0, 3, 1, 2, 4).reshape(B * T * hw, C).float()


def _rope_table(T, C):
    """pack.py's RoPE table [T][C/2] (cos, sin) as float32 [T, C], followed by T NaN guard rows in the same allocation."""
    freqs = 1.0 / (10000.0 ** (torch.arange(0, C, 2, dtype=torch.float64)[: C // 2] / C))
    ang = torch.outer(torch.arange(T, dtype=torch.float64), freqs)
    tab = torch.full((2 * T, C), float("nan"), dtype=torch.float32)
    tab[:T] = torch.stack([ang.cos(), ang.sin()], -1).reshape(T, C).float()
    return tab.to(DEV)


def _rope_apply(qkv, B, T, hw, C, tab, dtype):
    """q and k of every row rotated in float64 by the (float32) table row of its frame; the tensor-core kernel rounds
    the rotated q and k to the 16-bit dtype, so the reference does too."""
    t = qkv.double().reshape(B, T, hw, 3, C // 2, 2).clone()
    cs = tab[:T].double().reshape(1, T, 1, C // 2, 2)
    c, s = cs[..., 0], cs[..., 1]
    for w in (0, 1):
        a, b = t[:, :, :, w, :, 0].clone(), t[:, :, :, w, :, 1].clone()
        t[:, :, :, w, :, 0] = a * c - b * s
        t[:, :, :, w, :, 1] = a * s + b * c
    t = t.reshape(B * T * hw, 3 * C)
    if dtype != torch.float32:
        t[:, : 2 * C] = t[:, : 2 * C].to(dtype).double()
    return t


def _ta_instance(dtype, T, hw, C):
    """The instance attention.cu launches: tensor-core PB from ta_smem_per_pos (<= 96 KB per CTA), CUDA-core PB / HG
    from the 64 KB staging budget of launch_temporal."""
    hd = C // 8
    if dtype != torch.float32:
        per = 3 * 32 * (8 * hd + 8) * 2
        pb = 4 if 4 * per <= 96 * 1024 and hw >= 4 else 2 if 2 * per <= 96 * 1024 and hw >= 2 else 1
        return "temporal_attention_mma<HD=%d,PB=%d>" % (hd, pb)
    per, hg, mt = T * hd * 12, 8, 256 if hd >= 64 else 512
    while hg > 1 and hg * per > 64 * 1024:
        hg >>= 1
    pb = min(4, max(1, (64 * 1024) // (hg * per)))
    while pb > 1 and 32 * hg * pb > mt:
        pb -= 1
    while hg > 1 and 32 * hg * pb > mt:
        hg >>= 1
    return "temporal_attention_simt<HD=%d,PB=%d,HG=%d>" % (hd, min(pb, hw), hg)


# every head dim the forward plans (8, 24, 32, 48, 128) at T up to 32 (the second 16-query m-tile starts at T = 17), B = 2,
# hw with a tail of the PB = 4 (HD 8) / PB = 2 (HD 24) instances
TA_SHAPES = [pytest.param(B, T, hw, C, False, id="%d-%d-%d-%d" % (B, T, hw, C))
             for B, T, hw, C in [(1, 32, 320, 192), (2, 8, 80, 384), (1, 32, 100, 64), (3, 5, 7, 64), (1, 1, 9, 192), (1, 16, 30, 256),
                                 (1, 32, 12, 1024)]]
TA_SHAPES += [pytest.param(2, T, hw, 8 * hd, rope, id="2-%d-%d-%d-%s" % (T, hw, 8 * hd, "rope" if rope else "ape"))
              for hd, hw in ((8, 7), (24, 5), (32, 3), (48, 2), (128, 3)) for T in (1, 5, 16, 17, 32) for rope in (False, True)]


@pytest.mark.parametrize("dtype", [torch.float32] + DT16)
@pytest.mark.parametrize("B,T,hw,C,rope", TA_SHAPES)
def test_temporal_attention(dtype, B, T, hw, C, rope):
    qkv = _rand((B * T * hw, 3 * C), dtype, 11, 0.7)
    tab = _rope_table(T, C) if rope else None
    got, kernel = eng.op_temporal_attention_kernel(qkv, B, T, hw, C, tab)
    assert kernel == _ta_instance(dtype, T, hw, C)
    ref_in = _rope_apply(qkv, B, T, hw, C, tab, dtype) if rope else qkv
    _close(got, _tattn_ref(ref_in, B, T, hw, C), dtype, "temporal attention %s" % dtype, slack=4.0)
    if rope:
        # the identity rotation (cos 1, sin 0) must leave q and k bit for bit as they are
        ident = torch.zeros(T, C, dtype=torch.float32, device=DEV)
        ident[:, 0::2] = 1.0
        assert torch.equal(eng.op_temporal_attention_kernel(qkv, B, T, hw, C, ident)[0], eng.op_temporal_attention(qkv, B, T, hw, C))


# ---- norms ------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32] + DT16)
@pytest.mark.parametrize("M,D,eps", [(2568, 384, 1e-6), (100, 1024, 1e-6), (321, 64, 1e-5), (77, 192, 1e-5), (5, 256, 1e-5)])
def test_layernorm(dtype, M, D, eps):
    X = _rand((M, D), torch.float32, 13, 3.0) + 1.5
    g, b = _rand((D,), torch.float32, 14), _rand((D,), torch.float32, 15)
    got = eng.op_layernorm(X, g, b, eps, dtype)
    ref = F.layer_norm(X.double(), (D,), g.double(), b.double(), eps).float()
    _close(got, ref, dtype, "layernorm", slack=4.0)


@pytest.mark.parametrize("dtype", [torch.float32] + DT16)
@pytest.mark.parametrize("Fr,hw,C", [(4, 320, 192), (3, 80, 384), (2, 1280, 64), (1, 7, 64), (2, 30, 1024)])
def test_groupnorm(dtype, Fr, hw, C):
    X = (_rand((Fr, hw, C), torch.float32, 16, 2.0) + 0.5).to(dtype)
    g, b = _rand((C,), torch.float32, 17), _rand((C,), torch.float32, 18)
    got = eng.op_groupnorm(X, g, b, 1e-6)
    ref = F.group_norm(X.double().permute(0, 2, 1), 32, g.double(), b.double(), 1e-6).permute(0, 2, 1).float()
    _close(got, ref, dtype, "groupnorm", slack=4.0)


# ---- resampling ---------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32] + DT16)
@pytest.mark.parametrize("Fr,h,w,oh,ow,C", [(2, 16, 20, 32, 40, 64), (1, 19, 19, 37, 37, 64), (1, 128, 160, 224, 280, 32),
                                             (2, 5, 7, 5, 7, 8), (1, 1, 1, 4, 4, 16)])
def test_upsample_nhwc(dtype, Fr, h, w, oh, ow, C):
    X = _rand((Fr, h, w, C), dtype, 19)
    got = eng.op_upsample(X, oh, ow)
    ref = F.interpolate(X.double().permute(0, 3, 1, 2), size=(oh, ow), mode="bilinear", align_corners=True).permute(0, 2, 3, 1).float()
    _close(got, ref, dtype, "upsample", slack=2.0)


@pytest.mark.parametrize("Fr,h,w,oh,ow", [(3, 224, 280, 256, 320), (2, 518, 518, 259, 259), (1, 28, 35, 14, 17), (1, 70, 98, 80, 112)])
def test_resize_f32(Fr, h, w, oh, ow):
    X = _rand((Fr, h, w), torch.float32, 20)
    got = eng.op_resize_f32(X, oh, ow)
    # source coordinates are computed in float32 exactly like ATen's upsample_bilinear2d
    # (a float64 reference differs by up to 1.4e-4 at 518 -> 259 through the coordinate rounding)
    ref = F.interpolate(X[:, None], size=(oh, ow), mode="bilinear", align_corners=True)[:, 0]
    _close(got, ref, torch.float32, "resize_f32", slack=1.0)


def test_pyramid_downscale_matches_scale_factor_half():
    """dpt_pyramid.py:95-97 uses scale_factor=0.5 (floor) with align_corners=True."""
    X = _rand((2, 70, 98), torch.float32, 21)
    got = eng.op_resize_f32(X, 35, 49)
    ref = F.interpolate(X[:, None], scale_factor=0.5, mode="bilinear", align_corners=True)[:, 0]
    assert float((got - ref).abs().max()) <= 1e-5


def test_linear_kernels_agree_bitwise():
    """The tcgen05 linear kernels that shape selects between must agree bit for bit on the same operands (same fp32
    accumulation order per output element), for act = none and ReLU:
      A [20000, 384], W [1152, 384]   M >= 2048      -> B-resident gemm_bres, TMA-store epilogue
      A[:2000]                        M < 2048       -> streaming gemm_tc at BN = 192, TMA-store epilogue
      A[:2000], W[:1120]              N % 64 != 0    -> streaming gemm_tc at BN = 32, row-segment epilogue"""
    g = torch.Generator().manual_seed(3)
    A = torch.randn(20000, 384, generator=g).half().cuda()
    W = (torch.randn(1152, 384, generator=g) * 0.05).half().cuda()
    b = torch.randn(1152, generator=g).cuda()
    for act, kind in ((0, "0x1"), (2, "0x5")):
        bres = torch.empty(20000, 1152, dtype=torch.half, device=DEV)
        tc192 = torch.empty(2000, 1152, dtype=torch.half, device=DEV)
        tc32 = torch.empty(2000, 1120, dtype=torch.half, device=DEV)
        assert eng.op_gemm(A, W, bres, bias=b, act=act) == "gemm_bres<BN=192>"
        assert eng.op_gemm(A[:2000], W, tc192, bias=b, act=act) == "gemm_tc<BN=192,BK=64,kind=%s,tma=1>" % kind
        assert eng.op_gemm(A[:2000], W[:1120], tc32, bias=b[:1120], act=act) == "gemm_tc<BN=32,BK=64,kind=%s,tma=0>" % kind
        assert torch.equal(bres[:2000], tc192)
        assert torch.equal(tc192[:, :1120], tc32)


# ---- GPU-side preprocessing of the long-video driver ------------------------------------------------
@pytest.mark.parametrize("N,H,W,h,w", [(3, 256, 320, 224, 280), (2, 48, 64, 28, 42), (1, 100, 90, 140, 126), (2, 37, 53, 37, 53)])
def test_cubic_resize_u8_matches_cv2(N, H, W, h, w):
    """frame/255 -> cv2.resize(INTER_CUBIC) -> CHW, as endodav.py:195 / util/transform.py:109-113 do on the host."""
    import cv2
    import numpy as np

    g = torch.Generator().manual_seed(41)
    fr = torch.randint(0, 256, (N, H, W, 3), generator=g, dtype=torch.uint8)
    got = eng.op_cubic_resize_u8(fr.cuda(), h, w).cpu().numpy()
    ref = np.stack([np.transpose(cv2.resize(f.numpy().astype(np.float32) / 255.0, (w, h), interpolation=cv2.INTER_CUBIC), (2, 0, 1))
                    for f in fr])
    assert got.shape == ref.shape
    # same arithmetic, different association / FMA contraction than OpenCV's SIMD loops: <= 2e-6 on values in [-0.2, 1.2]
    assert float(np.abs(got - ref).max()) <= 2e-6, float(np.abs(got - ref).max())
