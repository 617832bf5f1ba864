"""Every GEMM epilogue the forward uses, on every kernel that runs it, against a float64 reference.

One case per call site of csrc/engine.cu that hands an epilogue to gemm() (ops.cuh), with the forward's own N / K / C
(ViT-S: D = 384, features 64, projected channels 64 / 128 / 192 / 384) and buffer roles, sent through edv_op_gemm, so
that the product's own kernel selection decides which kernel runs; every case asserts which one did.  Each tensor-core
case runs at a shape with an M tail (or a map that is no multiple of the conv tile) and at one with more than 4 x SM
count tiles, so that every persistent CTA drains both TMEM accumulators in both barrier phases.  Outputs live in
NaN-filled buffers with guard rows and 8 padding columns that must stay untouched.

Operands are rounded to the dtype first; the reference is float64 on those operands, in epi_apply's order of operations
(common.cuh).  Tolerances follow test_gpu_ops.py: 16-bit outputs the output rounding of their dtype, float32 outputs
fp32 accumulation noise."""
import math
import os
import re

import pytest
import torch
import torch.nn.functional as F

from endodav_b200 import engine as eng
from packed_emulator import _pixshuf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda"
DT16 = [torch.bfloat16, torch.float16]
PAD = 8        # padding columns of every output buffer (ldo = columns + PAD)
GUARD = 136    # guard rows after every output buffer (more than one 128-row tile)
NAN = float("nan")


# ---- the epilogue kinds the kernels instantiate (EDV_EPI_*_KINDS in csrc/common.cuh) -------------------------------
def _kind_lists():
    with open(os.path.join(ROOT, "endodav_b200", "csrc", "common.cuh")) as f:
        src = f.read()
    ef = {k: int(v) for k, v in re.findall(r"\b(EF_\w+)\s*=\s*(\d+)", src)}
    lines = src.split("\n")

    def macro(name):
        head = "#define %s(X)" % name
        i = next(k for k, l in enumerate(lines) if l.startswith(head))
        body = lines[i]
        while body.rstrip().endswith("\\"):
            i += 1
            body = body.rstrip()[:-1] + " " + lines[i]
        body = re.sub(r"/\*.*?\*/", "", body)[len(head):]
        return [int(eval(x, {"__builtins__": {}}, ef)) for x in re.findall(r"X\(([^()]*)\)", body)]

    return ef, macro("EDV_EPI_ROW_KINDS"), macro("EDV_EPI_TMA_KINDS")


EF, ROW_KINDS, TMA_KINDS = _kind_lists()


def _hex(kind):
    return "0x%x" % kind


# ---- helpers --------------------------------------------------------------------------------------------------------
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _rand(shape, dtype, seed, scale=1.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(shape, generator=g, device=DEV) * scale).to(dtype)


def _tol(dtype):
    # relative output rounding: bf16 2^-8, f16 2^-11, fp32 accumulate-order noise
    return {torch.float32: 2e-5, torch.bfloat16: 2 ** -8, torch.float16: 2 ** -11}[dtype]


WORST = {}   # case -> worst error as a fraction of its tolerance (printed at the end of the module)


def _close(got, ref, dtype, what, slack):
    """|got - ref| <= slack * tol(dtype) * max(|ref|, 1) + 1e-5; returns the worst fraction of that bound."""
    err = (got.double() - ref).abs()
    bound = slack * _tol(dtype) * ref.abs().clamp_min(1.0) + 1e-5
    bad = ~(err <= bound)
    assert not bool(bad.any()), "%s: max err %.4g (ref max %.4g), %d / %d over tolerance" % (
        what, float(err.nan_to_num(float("inf")).max()), float(ref.abs().max()), int(bad.sum()), bad.numel())
    return float((err / bound).max()) if err.numel() else 0.0


def _note(name, frac):
    WORST[name] = max(WORST.get(name, 0.0), frac)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        print("\nworst error / tolerance per case:")
        for k in sorted(WORST):
            print("  %-40s %.3f" % (k, WORST[k]))


def _nan_buf(rows, cols, dtype):
    return torch.full((rows + GUARD, cols + PAD), NAN, dtype=dtype, device=DEV)


def _lin_acc(A, W):
    return A.double() @ W.double().t()


def _conv_acc(X, Wt, stride=1):
    """3x3, pad 1 convolution of NHWC X with Wt [O, 9C] in (ky,kx,c) order, as a float64 [F*OH*OW, O] matrix."""
    Fr, H, W, C = X.shape
    O = Wt.shape[0]
    cols = F.unfold(X.double().permute(0, 3, 1, 2), 3, padding=1, stride=stride)      # [F, C*9 (c,ky,kx), L]
    w = Wt.double().reshape(O, 3, 3, C).permute(0, 3, 1, 2).reshape(O, C * 9)
    return (w @ cols).permute(0, 2, 1).reshape(-1, O)


def _pick_conv_tile(H, W):   # ops.h pick_conv_tile
    best, bt = -1, None
    for th, tw in ((8, 16), (16, 8), (4, 32), (32, 4), (2, 64), (1, 128)):
        cover = -(-H // th) * th * (-(-W // tw) * tw)
        if best < 0 or cover < best:
            best, bt = cover, (th, tw)
    return bt


def epi_ref(acc, e, R):
    """The epilogue of common.cuh epi_apply on the float64 GEMM result acc [M, N], in its order of operations:
    bias, row bias, GELU (GEGLU / head), row map, res1, res2, ReLU / sigmoid.  -> (value [R, cols] in output rows, NaN
    where no row is written; relu copy)."""
    M = acc.shape[0]
    v = acc
    if e.get("bias") is not None:
        v = v + e["bias"].double()
    if e.get("rowbias") is not None:
        idx = (torch.arange(M, device=acc.device) // e["rb_div"]) % e["rb_mod"]
        v = v + e["rowbias"].double()[idx]
    act = e.get("act", eng.ACT_NONE)
    if act == eng.ACT_GELU:
        v = F.gelu(v)                                                   # exact erf
    elif act == eng.ACT_GEGLU:
        hg = v.reshape(M, -1, 2, 64)                                    # tile pairs [64 value | 64 gate] (pack.py)
        v = (hg[:, :, 0] * F.gelu(hg[:, :, 1])).reshape(M, -1)
    elif act == eng.ACT_HEAD:
        s = F.relu(v) @ e["head_w"][:32].double() + e["head_w"][32].double()
        v = (F.relu(s) if e["sig_sign"] == 0.0 else torch.sigmoid(e["sig_sign"] * s))[:, None]
    mp = e.get("map", eng.MAP_LINEAR)
    if mp == eng.MAP_TOKENS:
        img = torch.full((R, v.shape[1]), NAN, dtype=torch.float64, device=acc.device)
        m = torch.arange(M, device=acc.device)
        img[m + m // e["map_p"] + 1] = v
    elif mp == eng.MAP_PIXSHUF:
        k, ph, pw, c = e["ps"]
        img = _pixshuf(v, M // (ph * pw), ph, pw, k, c).reshape(R, c)
    else:
        img = v
    cols = img.shape[1]
    if e.get("res1") is not None:
        img = img + e["res1"][:R, :cols].double()
    if e.get("res2") is not None:
        img = img + e["res2"][:R, :cols].double()
    if act == eng.ACT_RELU:
        img = F.relu(img)
    elif act == eng.ACT_SIGMOID:
        img = torch.sigmoid(e["sig_sign"] * img)
    return img, F.relu(img)


def _check_buf(buf, ref, R, cols, dtype, what, slack):
    """buf [R + GUARD, cols + PAD]: the logical region matches ref (rows where ref is NaN stay NaN), the padding columns
    and guard rows are untouched."""
    written = ~ref[:, 0].isnan()
    assert bool(buf[:R][~written].isnan().all()), "%s: rows the epilogue must not write (cls rows) were written" % what
    assert bool(buf[:, cols:].isnan().all()), "%s: padding columns beyond N were written" % what
    assert bool(buf[R:].isnan().all()), "%s: guard rows beyond the output were written" % what
    return _close(buf[:R, :cols][written], ref[written], dtype, what, slack)


# ---- the call sites -------------------------------------------------------------------------------------------------
# geo: "tail" / "big" geometry, each a dict or a function of the SM count S.  Linear: M, or (BT, ph, pw) for the
# token / pixel-shuffle maps (M = BT ph pw).  Conv: (F, H, W).  tc: expected tensor-core kernel per shape (None: the
# tensor-core engine rejects the case).  simt: False when the CUDA-core engine rejects it.
def _m_big(S, n_tiles):        # M with an M tail and ceil(M / 128) * n_tiles > 4 S
    return ((4 * S) // n_tiles + 1) * 128 - 9


def _bt_big(S, n_tiles, hw=37 * 37):
    return dict(BT=(4 * S * 128) // (n_tiles * hw) + 1, ph=37, pw=37)


def _f_big(S):                 # 130 x 130 maps: 153 tiles of 128 pixels per frame for both conv kernels
    return dict(F=(4 * S) // 153 + 1, H=130, W=130)


TAIL_M = dict(M=300)
TAIL_TOK = dict(BT=3, ph=7, pw=10)
TAIL_CONV = dict(F=2, H=19, W=23)


def _lin(name, site, N, K, tail, big, n_big, tc_tail, tc_big, simt=True, **epi):
    return dict(name=name, site=site, conv=False, N=N, K=K, geo=dict(tail=tail, big=(lambda S: dict(M=_m_big(S, n_big)))
                if big is None else big), tc=dict(tail=tc_tail, big=tc_big), simt=simt, epi=epi)


def _cnv(name, site, N, C, tc_tail, tc_big, simt=True, stride=1, tail=TAIL_CONV, **epi):
    return dict(name=name, site=site, conv=True, N=N, C=C, stride=stride, geo=dict(tail=tail, big=_f_big), simt=simt,
                tc=None if tc_tail is None else dict(tail=tc_tail, big=tc_big), epi=epi)


def _tc(BN, kind, tma, BK=64):
    return "gemm_tc<BN=%d,BK=%d,kind=%s,tma=%d>" % (BN, BK, "-1" if kind < 0 else _hex(kind), tma)


def _tcc(BN, kind, BK=64):
    return "gemm_tc_conv<BN=%d,BK=%d,kind=%s>" % (BN, BK, "-1" if kind < 0 else _hex(kind))


def _halo(BN, kind):
    return "conv_halo<BN=%d,kind=%s>" % (BN, "-1" if kind < 0 else _hex(kind))


B, G, R_, OF, R1F, R1T, R2T, ORL = (EF["EF_BIAS"], EF["EF_GELU"], EF["EF_RELU"], EF["EF_OUT_F32"], EF["EF_RES1_F32"],
                                    EF["EF_RES1_T"], EF["EF_RES2_T"], EF["EF_OUT_RELU"])
BRES192 = "gemm_bres<BN=192>"

CASES = [
    # patch embedding (engine.cu:418-422): fp32 tokens, pos-embed row bias, cls rows left to cls_row_kernel
    _lin("patch_embed", "engine.cu:418", 384, 640, TAIL_TOK, lambda S: _bt_big(S, 2), 2, _tc(192, -1, 0), _tc(192, -1, 0),
         out_f32=True, rowbias="pos", map=eng.MAP_TOKENS),
    _lin("patch_embed_nocls", "engine.cu:419", 384, 640, TAIL_TOK, lambda S: _bt_big(S, 2), 2, _tc(192, -1, 0), _tc(192, -1, 0),
         out_f32=True, rowbias="pos"),
    # TMA-store kinds (16-bit row-major output, bias / GELU / none); M >= 2048 with K <= 384 is gemm_bres
    _lin("qkv", "engine.cu:440", 1152, 384, TAIL_M, None, 6, _tc(192, B, 1), BRES192, bias=True),
    _lin("fc1", "engine.cu:455", 1536, 384, TAIL_M, None, 8, _tc(256, B | G, 1), BRES192, bias=True, act=eng.ACT_GELU),
    _lin("proj2", "engine.cu:538", 192, 384, TAIL_M, None, 1, _tc(192, B, 1), BRES192, bias=True),
    _lin("proj3", "engine.cu:550", 384, 384, TAIL_M, None, 2, _tc(192, B, 1), BRES192, bias=True),
    _lin("resize3", "engine.cu:561", 384, 9 * 384, TAIL_M, None, 2, _tc(192, B, 1), _tc(192, B, 1), bias=True),
    _lin("out_conv", "engine.cu:351", 64, 64, TAIL_M, None, 1, _tc(64, B, 1), "gemm_bres<BN=64>", bias=True),
    _lin("temporal_qkv", "engine.cu:281", 3 * 192, 192, TAIL_M, None, 3, _tc(192, 0, 1), BRES192),
    # x += ... in place on the fp32 residual stream
    _lin("proj_unfused", "engine.cu:449", 384, 384, TAIL_M, None, 2, _tc(192, B | R1F | OF, 0), _tc(192, B | R1F | OF, 0),
         bias=True, out_f32=True, res1="inplace"),
    _lin("fc2_unfused", "engine.cu:470", 384, 1536, TAIL_M, None, 2, _tc(192, B | R1F | OF, 0), _tc(192, B | R1F | OF, 0),
         bias=True, out_f32=True, res1="inplace"),
    _lin("temporal_to_out", "engine.cu:284", 192, 192, TAIL_M, None, 1, _tc(192, B | R1F | OF, 0), _tc(192, B | R1F | OF, 0),
         bias=True, out_f32=True, res1="inplace"),
    _lin("temporal_proj_in", "engine.cu:272", 384, 384, TAIL_M, None, 2, _tc(192, B | OF, 0), _tc(192, B | OF, 0),
         bias=True, out_f32=True),
    _lin("temporal_ff2", "engine.cu:304", 64, 256, TAIL_M, None, 1, _tc(64, B | R1F, 0), _tc(64, B | R1F, 0),
         bias=True, res1="f32"),
    _lin("temporal_proj_out", "engine.cu:309", 192, 192, TAIL_M, None, 1, _tc(192, B | R1T, 0), _tc(192, B | R1T, 0),
         bias=True, res1="T"),
    _lin("temporal_geglu", "engine.cu:291", 8 * 64, 64, TAIL_M, None, 4, _tc(128, -1, 0), _tc(128, -1, 0), simt=False,
         bias=True, act=eng.ACT_GEGLU),
    # readout projects: w2 on the BT class tokens, w1 with the per-frame row bias + GELU
    _lin("readout_w2", "engine.cu:493", 384, 384, dict(M=3), None, 2, _tc(192, B | OF, 0), _tc(192, B | OF, 0),
         bias=True, out_f32=True),
    _lin("readout_w1", "engine.cu:498", 384, 384, TAIL_TOK, lambda S: _bt_big(S, 2), 2, _tc(192, -1, 0), _tc(192, -1, 0),
         rowbias="readout", act=eng.ACT_GELU),
    # projects[0..1] merged with their ConvTranspose: pixel shuffle
    _lin("proj0_pixshuf", "engine.cu:529", 16 * 64, 384, TAIL_TOK, lambda S: _bt_big(S, 4), 4, _tc(256, -1, 0), _tc(256, -1, 0),
         bias=True, map=eng.MAP_PIXSHUF, ps=(4, 64)),
    _lin("proj1_pixshuf", "engine.cu:534", 4 * 128, 384, TAIL_TOK, lambda S: _bt_big(S, 2), 2, _tc(256, -1, 0), _tc(256, -1, 0),
         bias=True, map=eng.MAP_PIXSHUF, ps=(2, 128)),
    # scratch.layer*_rn: no bias, relu copy for the RCUs
    _cnv("layer1_rn", "engine.cu:546", 64, 64, _halo(64, ORL), _halo(64, ORL), out_relu=True),
    _cnv("layer2_rn", "engine.cu:544", 64, 128, _tcc(64, ORL), _tcc(64, ORL), out_relu=True),
    _cnv("layer3_rn", "engine.cu:542", 64, 192, _tcc(64, ORL), _tcc(64, ORL), out_relu=True),
    _cnv("layer4_rn", "engine.cu:572", 64, 384, _tcc(64, ORL), _tcc(64, ORL), out_relu=True),
    # ResidualConvUnit: c1 bias + ReLU; c2 + x [+ extra] [relu copy]
    _cnv("rcu_c1", "engine.cu:319", 64, 64, _halo(64, B | R_), _halo(64, B | R_), bias=True, act=eng.ACT_RELU),
    _cnv("rcu_c2", "engine.cu:322", 64, 64, _halo(64, B | R1T), _halo(64, B | R1T), bias=True, res1="T"),
    _cnv("rcu_c2_relu", "listed kind, no call site", 64, 64, _halo(64, B | R1T | ORL), _halo(64, B | R1T | ORL), bias=True, res1="T",
         out_relu=True),
    _cnv("rcu_c2_extra", "listed kind, no call site", 64, 64, _halo(64, B | R1T | R2T), _halo(64, B | R1T | R2T), bias=True, res1="T",
         res2=True),
    _cnv("rcu_c2_extra_relu", "engine.cu:346", 64, 64, _halo(64, B | R1T | R2T | ORL), _halo(64, B | R1T | R2T | ORL),
         bias=True, res1="T", res2=True, out_relu=True),
    # disparity head: output_conv1 (32 channels), the unfused conv + 1x1 head (ReLU / sigmoid(sign .)), a sigmoid map
    _cnv("oc1", "engine.cu:363", 32, 64, _halo(32, B), _halo(32, B), bias=True),
    _cnv("head_unfused", "engine.cu:375", 32, 64, _tcc(32, -1), _tcc(32, -1), simt=False, bias=True, act=eng.ACT_HEAD,
         sig_sign=0.0),
    _cnv("head_unfused_sigmoid", "engine.cu:375", 32, 64, _tcc(32, -1), _tcc(32, -1), simt=False, bias=True,
         act=eng.ACT_HEAD, sig_sign=-1.0),
    _cnv("sigmoid_generic", "common.cuh:289", 64, 64, _halo(64, -1), _halo(64, -1), bias=True, act=eng.ACT_SIGMOID,
         sig_sign=-1.0),
    # resize_layers[3] on the CUDA-core path: stride-2 conv (the tensor-core path runs im2col + the resize3 GEMM)
    _cnv("resize3_stride2", "engine.cu:563", 384, 384, None, None, stride=2, tail=dict(F=2, H=37, W=37), bias=True),
]

# the ViT-L RCUs (features 256) run the same four c2 kinds on the implicit-GEMM conv kernel
for _n, _k, _e in (("", B | R1T, {}), ("_relu", B | R1T | ORL, dict(out_relu=True)), ("_extra", B | R1T | R2T, dict(res2=True)),
                   ("_extra_relu", B | R1T | R2T | ORL, dict(res2=True, out_relu=True))):
    CASES.append(_cnv("rcu_c2" + _n + "_vitl", "engine.cu:322", 256, 256, _tcc(256, _k), None, bias=True, res1="T", **_e))


def _params():
    out = []
    for c in CASES:
        if c["tc"] is not None:
            for shape in ("tail", "big"):
                if c["tc"].get(shape) is None:
                    continue
                for dt in DT16:
                    out.append(pytest.param(c, shape, dt, eng.ENGINE_TC, id="%s-%s-%s-tc" % (c["name"], shape, str(dt)[6:])))
        if c["simt"]:
            for dt in [torch.float32] + DT16:
                out.append(pytest.param(c, "tail", dt, eng.ENGINE_SIMT, id="%s-tail-%s-simt" % (c["name"], str(dt)[6:])))
    return out


def _geometry(c, shape, S):
    g = c["geo"][shape]
    return g(S) if callable(g) else dict(g)


def _operands(c, geo, dtype):
    """-> (A, W, M, conv tuple or None, map geometry (BT, ph, pw) or None)"""
    N = c["N"]
    if c["conv"]:
        s = c["stride"]
        Fr, H, Wd = geo["F"], geo["H"], geo["W"]
        A = _rand((Fr, H, Wd, c["C"]), dtype, 1)
        W = _rand((N, 9 * c["C"]), dtype, 2, (9 * c["C"]) ** -0.5)
        return A, W, Fr * ((H - 1) // s + 1) * ((Wd - 1) // s + 1), (Fr, H, Wd, c["C"], s), None
    M = geo["M"] if "M" in geo else geo["BT"] * geo["ph"] * geo["pw"]
    A = _rand((M, c["K"]), dtype, 1)
    W = _rand((N, c["K"]), dtype, 2, c["K"] ** -0.5)
    return A, W, M, None, (geo["BT"], geo["ph"], geo["pw"]) if "BT" in geo else None


def _tiles(kernel, c, geo, M):
    BN = int(re.search(r"BN=(\d+)", kernel).group(1))
    if kernel.startswith("conv_halo"):
        return geo["F"] * -(-geo["H"] // 16) * -(-geo["W"] // 8)
    if kernel.startswith("gemm_tc_conv"):
        th, tw = _pick_conv_tile(geo["H"], geo["W"])
        return geo["F"] * -(-geo["H"] // th) * -(-geo["W"] // tw) * (c["N"] // BN)
    return -(-M // 128) * (c["N"] // BN)


def _run_case(c, shape, dtype, engine):
    """-> (edv status, kernel, dict of what to check)"""
    S = _sms()
    geo = _geometry(c, shape, S)
    A, W, M, conv, tok = _operands(c, geo, dtype)
    e = c["epi"]
    N, act = c["N"], e.get("act", eng.ACT_NONE)
    ref_e = dict(act=act, sig_sign=e.get("sig_sign", 0.0))
    kw = dict(act=act, sig_sign=e.get("sig_sign", 0.0), conv=conv, M=M)
    out_dt = torch.float32 if (e.get("out_f32") or act == eng.ACT_HEAD) else dtype
    # output rows / columns
    cols, R = N, M
    if act == eng.ACT_GEGLU:
        cols = N // 2
    if e.get("map") == eng.MAP_TOKENS:
        BT, ph, pw = tok
        R = BT * (ph * pw + 1)
        kw.update(map=eng.MAP_TOKENS, map_p=ph * pw)
        ref_e.update(map=eng.MAP_TOKENS, map_p=ph * pw)
    elif e.get("map") == eng.MAP_PIXSHUF:
        BT, ph, pw = tok
        k, cp = e["ps"]
        cols, R = cp, BT * k * ph * k * pw
        kw.update(map=eng.MAP_PIXSHUF, ps=(k, ph, pw, cp))
        ref_e.update(map=eng.MAP_PIXSHUF, ps=(k, ph, pw, cp))
    if e.get("bias"):
        kw["bias"] = ref_e["bias"] = _rand((N,), torch.float32, 3)
    if e.get("rowbias") == "pos":
        P = tok[1] * tok[2] if tok else M
        tbl = _rand((P, N), torch.float32, 4)
        kw.update(rowbias=tbl, rb_ld=N, rb_div=1, rb_mod=P)
        ref_e.update(rowbias=tbl, rb_div=1, rb_mod=P)
    elif e.get("rowbias") == "readout":
        BT, P = tok[0], tok[1] * tok[2]
        tbl = _rand((BT, N), torch.float32, 4)
        kw.update(rowbias=tbl, rb_ld=N, rb_div=P, rb_mod=BT)
        ref_e.update(rowbias=tbl, rb_div=P, rb_mod=BT)
    if act == eng.ACT_HEAD:
        kw["head_w"] = ref_e["head_w"] = _rand((33,), torch.float32, 5, 0.3)
        out = torch.full((M + GUARD,), NAN, dtype=torch.float32, device=DEV)
        kw["ldo"] = 1
    else:
        out = _nan_buf(R, cols, out_dt)
        kw["ldo"] = cols + PAD
    r1 = e.get("res1")
    if r1 == "inplace":
        x0 = _rand((R, cols), torch.float32, 6, 2.0)
        out[:R, :cols] = x0
        kw.update(res1=out, ld_res1=cols + PAD)
        ref_e["res1"] = x0
    elif r1 is not None:
        res = _rand((R, cols + PAD), torch.float32 if r1 == "f32" else dtype, 6)
        kw.update(res1=res, ld_res1=cols + PAD)
        ref_e["res1"] = res
    if e.get("res2"):
        res = _rand((R, cols + PAD), dtype, 7)
        kw.update(res2=res, ld_res2=cols + PAD)
        ref_e["res2"] = res
    out_relu = _nan_buf(R, cols, dtype) if e.get("out_relu") else None
    kw["out_relu"] = out_relu
    rc, kernel = eng.op_gemm_status(eng._dt(A), engine, eng.gemm_desc(A, W, out, **kw))
    if rc != 0:
        return rc, kernel, None
    acc = _conv_acc(A, W, conv[4]) if conv else _lin_acc(A, W)
    return rc, kernel, dict(S=S, geo=geo, M=M, R=R, cols=cols, out=out, out_relu=out_relu, out_dt=out_dt, acc=acc, ref_e=ref_e)


@pytest.mark.gpu
@pytest.mark.parametrize("c,shape,dtype,engine", _params())
def test_epilogue_matches_reference(c, shape, dtype, engine):
    rc, kernel, r = _run_case(c, shape, dtype, engine)
    assert rc == 0, "%s: edv_op_gemm failed (%d)" % (c["name"], rc)
    want = c["tc"][shape] if engine == eng.ENGINE_TC else "gemm_simt"
    assert kernel == want, "%s (%s): ran %s, written for %s" % (c["name"], c["site"], kernel, want)
    if shape == "big":
        assert _tiles(kernel, c, r["geo"], r["M"]) > 4 * r["S"]
    torch.cuda.synchronize()
    ref, ref_relu = epi_ref(r["acc"], r["ref_e"], r["R"])
    what = "%s %s %s %s" % (c["name"], shape, dtype, kernel)
    # 16-bit outputs: output rounding of the dtype; fp32 outputs: fp32 accumulation noise (head: + a 33-term dot)
    slack = 2.0 if r["out_dt"] != torch.float32 else (8.0 if c["epi"].get("act") == eng.ACT_HEAD else 4.0)
    if c["epi"].get("act") == eng.ACT_HEAD:
        out = r["out"]
        assert bool(out[r["M"]:].isnan().all()), "%s: guard rows written" % what
        frac = _close(out[:r["M"]], ref[:, 0], torch.float32, what, slack)
    else:
        frac = _check_buf(r["out"], ref, r["R"], r["cols"], r["out_dt"], what, slack)
    if r["out_relu"] is not None:
        frac = max(frac, _check_buf(r["out_relu"], ref_relu, r["R"], r["cols"], dtype, what + " out_relu", 2.0))
    _note(c["name"], frac)


def _rejected():
    out = []
    for c in CASES:
        if not c["simt"]:
            for dt in [torch.float32] + DT16:
                out.append(pytest.param(c, dt, eng.ENGINE_SIMT, id="%s-%s-simt" % (c["name"], str(dt)[6:])))
        if c["tc"] is None:
            for dt in DT16:
                out.append(pytest.param(c, dt, eng.ENGINE_TC, id="%s-%s-tc" % (c["name"], str(dt)[6:])))
    return out


@pytest.mark.parametrize("c,dtype,engine", _rejected())
def test_unsupported_epilogue_is_rejected(c, dtype, engine):
    """GEGLU and the head epilogue exist only in the tcgen05 kernel (the CUDA-core forward composes them from a plain
    GEMM and a small kernel), stride-2 convs only in the CUDA-core one: edv_op_gemm refuses before any launch (no GPU
    needed)."""
    e = c["epi"]
    K = 9 * c["C"] if c["conv"] else c["K"]
    A, W = torch.zeros(16, K, dtype=dtype), torch.zeros(c["N"], K, dtype=dtype)
    out = torch.zeros(16, c["N"], dtype=torch.float32)
    kw = dict(act=e.get("act", 0), bias=torch.zeros(c["N"]), ldo=c["N"])
    if c["conv"]:
        kw.update(conv=(1, 4, 4, c["C"], c["stride"]), M=None)
        A = torch.zeros(1, 4, 4, c["C"], dtype=dtype)
    if e.get("act") == eng.ACT_HEAD:
        kw.update(head_w=torch.zeros(33), ldo=1)
    rc, kernel = eng.op_gemm_status(eng._dt(A), engine, eng.gemm_desc(A, W, out, **kw))
    assert rc == -1 and kernel == ""                                  # EDV_ERR_ARG, nothing launched


def test_bad_descriptor_is_rejected():
    A, W, out = torch.zeros(16, 64, dtype=torch.bfloat16), torch.zeros(64, 64, dtype=torch.bfloat16), torch.zeros(16, 72)
    for kw in (dict(ldo=68), dict(ldo=72, res1=out, ld_res1=68), dict(ldo=72, lda=60), dict(ldo=72, rowbias=out, rb_ld=4)):
        assert eng.op_gemm_status(eng.EDV_BF16, eng.ENGINE_TC, eng.gemm_desc(A, W, out, **kw))[0] == -1, kw
    d = eng.gemm_desc(A, W, out, ldo=72)
    d.out = None
    assert eng.op_gemm_status(eng.EDV_BF16, eng.ENGINE_TC, d)[0] == -1
    d = eng.gemm_desc(A, W, out, ldo=72)
    d.struct_bytes -= 8                                               # a stale mirror of edv_gemm_desc
    assert eng.op_gemm_status(eng.EDV_BF16, eng.ENGINE_TC, d)[0] == -1


# ---- bitwise: each compile-time kind equals the generic epilogue ----------------------------------------------------
def _kind_operands(kind, path, dtype):
    """A launch of `kind` on `path` ("lin": gemm_tc at BN = 192, row-segment epilogue; "halo": conv_halo; "conv":
    implicit-GEMM conv).  -> (A, W, epilogue kwargs without out / out_relu, M, N, out dtype)"""
    if path == "lin":
        M, N, K = 300, 192, 128
        A, W, conv = _rand((M, K), dtype, 21), _rand((N, K), dtype, 22, K ** -0.5), None
    else:
        C, N = (64, 64) if path == "halo" else (128, 64)
        Fr, H, Wd = 2, 19, 23
        M, conv = Fr * H * Wd, (Fr, H, Wd, C, 1)
        A, W = _rand((Fr, H, Wd, C), dtype, 21), _rand((N, 9 * C), dtype, 22, (9 * C) ** -0.5)
    kw = dict(conv=conv, M=M, ldo=N + PAD)
    if kind & EF["EF_BIAS"]:
        kw["bias"] = _rand((N,), torch.float32, 23)
    kw["act"] = eng.ACT_GELU if kind & EF["EF_GELU"] else eng.ACT_RELU if kind & EF["EF_RELU"] else eng.ACT_NONE
    if kind & (EF["EF_RES1_F32"] | EF["EF_RES1_T"]):
        kw.update(res1=_rand((M, N + PAD), torch.float32 if kind & EF["EF_RES1_F32"] else dtype, 24), ld_res1=N + PAD)
    if kind & EF["EF_RES2_T"]:
        kw.update(res2=_rand((M, N + PAD), dtype, 25), ld_res2=N + PAD)
    return A, W, kw, M, N, torch.float32 if kind & EF["EF_OUT_F32"] else dtype


def _kind_launch(kind, path, dtype, rowbias):
    A, W, kw, M, N, out_dt = _kind_operands(kind, path, dtype)
    # 8 bytes past a 16-byte boundary: a 16-bit output that the TMA-store epilogue cannot take, so the TMA kinds run
    # their row-segment instance here (ldo = N + 8 would not do it: the TMA store clips its tensor map at N columns)
    buf = torch.full(((M + GUARD) * (N + PAD) + 8,), NAN, dtype=out_dt, device=DEV)
    out = buf[4:]
    out_relu = _nan_buf(M, N, dtype) if kind & EF["EF_OUT_RELU"] else None
    if rowbias:
        kw.update(rowbias=torch.zeros(N, device=DEV), rb_ld=0)       # all rows read the same zero row: + 0 is exact
    kernel = eng.op_gemm(A, W, out, out_relu=out_relu, **kw)
    return kernel, out, out_relu


def _same(a, b):
    nan = a.isnan()
    return torch.equal(nan, b.isnan()) and torch.equal(a[~nan], b[~nan])


def _kind_params():
    out = []
    for k in ROW_KINDS:
        for path in ("lin", "halo", "conv"):
            if path == "halo" and k & EF["EF_GELU"]:
                continue            # conv_halo has no GELU epilogue: such convs run the implicit-GEMM kernel
            out.append(pytest.param(k, path, id="%s-%s" % (_hex(k), path)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16)
@pytest.mark.parametrize("kind,path", _kind_params())
def test_row_kind_instance_equals_generic(kind, path, dtype):
    """Every EDV_EPI_ROW_KINDS instantiation gives bit for bit what the generic F = -1 epilogue gives with the same
    flags: an all-zero row-bias table (rb_ld = 0) forces the generic version and adds an exact +0."""
    k1, out1, rl1 = _kind_launch(kind, path, dtype, False)
    k2, out2, rl2 = _kind_launch(kind, path, dtype, True)
    name = {"lin": "gemm_tc<BN=192,BK=64,kind=%s,tma=0>", "halo": "conv_halo<BN=64,kind=%s>",
            "conv": "gemm_tc_conv<BN=64,BK=64,kind=%s>"}[path]
    assert k1 == name % _hex(kind) and k2 == name % "-1", (k1, k2)
    assert not bool(out1.isnan().all())
    assert _same(out1, out2)
    if rl1 is not None:
        assert _same(rl1, rl2)


# ---- bitwise: TMA-store epilogue vs row-segment epilogue ------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16)
@pytest.mark.parametrize("N,BN", [(64, 64), (128, 128), (576, 192), (1024, 256)])
@pytest.mark.parametrize("kind", TMA_KINDS, ids=_hex)
def test_tma_store_equals_row_segment(kind, N, BN, dtype):
    """The TMA-store and row-segment epilogues of a kind agree bit for bit at the same BN (same fp32 math); BIAS|GELU
    uses a different GELU in each (gelu_poly2 / gelu_fast), so both are held to the float64 reference instead."""
    M, K = 300, 128
    A, W = _rand((M, K), dtype, 31), _rand((N, K), dtype, 32, K ** -0.5)
    b = _rand((N,), torch.float32, 33) if kind & EF["EF_BIAS"] else None
    act = eng.ACT_GELU if kind & EF["EF_GELU"] else eng.ACT_RELU if kind & EF["EF_RELU"] else eng.ACT_NONE
    tma = torch.full((M + GUARD, N), NAN, dtype=dtype, device=DEV)
    k1 = eng.op_gemm(A, W, tma, bias=b, act=act)
    seg = torch.full(((M + GUARD) * N + 8,), NAN, dtype=dtype, device=DEV)
    k2 = eng.op_gemm(A, W, seg[4:], bias=b, act=act)                  # 8-byte aligned output: no TMA store
    seg = seg[4:4 + (M + GUARD) * N].view(M + GUARD, N)
    assert k1 == _tc(BN, kind, 1) and k2 == _tc(BN, kind, 0), (k1, k2)
    assert bool(tma[M:].isnan().all()) and bool(seg[M:].isnan().all()), "rows beyond M written"
    if act == eng.ACT_GELU:
        ref, _ = epi_ref(_lin_acc(A, W), dict(bias=b, act=act), M)
        _note("tma_vs_rows_gelu", max(_close(tma[:M], ref, dtype, "TMA store", 2.0), _close(seg[:M], ref, dtype, "row segment", 2.0)))
    else:
        assert torch.equal(tma[:M], seg[:M])


# ---- every listed kind has a case -----------------------------------------------------------------------------------
def test_every_listed_kind_has_a_case():
    """A kind added to EDV_EPI_ROW_KINDS / EDV_EPI_TMA_KINDS (common.cuh) must get a call-site case above, or at least
    the kind tests: this fails until it does."""
    assert ROW_KINDS and TMA_KINDS and set(TMA_KINDS) <= set(ROW_KINDS)
    row, tma = set(), set()
    for c in CASES:
        for k in (c["tc"] or {}).values():
            m = re.search(r"kind=(0x[0-9a-f]+)", k or "")
            if m:
                (tma if "tma=1" in k else row).add(int(m.group(1), 16))
    # test_tma_store_equals_row_segment runs every TMA kind in both forms (BIAS|RELU has no call site in the forward)
    row |= set(TMA_KINDS)
    tma |= set(TMA_KINDS)
    assert set(ROW_KINDS) <= row, "row-segment kinds without a case: %s" % [_hex(k) for k in sorted(set(ROW_KINDS) - row)]
    assert set(TMA_KINDS) <= tma, "TMA-store kinds without a case: %s" % [_hex(k) for k in sorted(set(TMA_KINDS) - tma)]
    covered = {p.values[0] for p in _kind_params()}
    assert covered == set(ROW_KINDS)
