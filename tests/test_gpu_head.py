"""The fused disparity head (edv_op_disp_head: head_fused_kernel) at the forward's shapes, against a float64 reference.

head_fused_kernel writes every output pixel of the 16-bit tensor-core forward for Cin = features / 2 in {32, 128}:
bilinear upsample (align_corners=True) -> 3x3 conv Cin -> 32 + bias -> ReLU -> 1x1 conv + head_w[32] -> ReLU, or
sigmoid(sig * s) for the conv head.  It is persistent: one CTA per SM walks 16 x 8 output tiles, with a halo ring 4 deep
at Cin = 32 and 2 deep at Cin = 128 and a double-buffered accumulator.  So the shapes here run many tiles per CTA at
both ring depths, every tail class of OH mod 16 and OW mod 8, grids below, at and above the SM count, and frames of a
multi-tile launch must equal, bit for bit, the same frame launched alone or next to different neighbours.  A poisoned
neighbour (frame f+1 scaled by 2^10) makes any read of the wrong frame dominate.

X is a view of the first F frames of an allocation whose next frame is NaN, and outputs go to the front of a NaN-filled
buffer whose guard frame must stay NaN.  b and head_w are chosen so that about half the conv channels and half the
ReLU-head outputs are clipped, and the sigmoid inputs stay within about |s| < 4.  Every case asserts which instance ran.

Reference (_reference): float64 on the same 16-bit X and Wt.  Source coordinates, ly, lx and the four bilinear weights
are float32, computed exactly as the kernel (and ATen) computes them; after that everything is float64.

Tolerance: a per-pixel bound from the kernel's error model (_reference, `bound`), carried through every stage:
  halo      bf16: one fp32 lerp rounded once to bf16, |d| <= (u + (1 + u) g4) sum_i |w_i x_i|, u = 2^-8.
            f16: the four weights rounded to half, then HMUL2 and three HFMA2 (hf_lerp4).  The corner read first is
            rounded 5 times (weight, HMUL2, 3 x HFMA2), the next 4, 3 and 2 times, so
            |d| <= sum_i ((1 + u)^k_i - 1) |w_i x_i|, k = (5, 4, 3, 2), u = 2^-11, plus 2^-25 (1 + u)^4 (sum_i |x_i| + 4)
            for roundings that fall into the subnormal range.
  conv      (|W_i| * d)(p) + gK (|W_i| * (|up| + d))(p): the 16-bit products are exact in fp32, the tensor core sums
            K = 9 Cin of them, gK = K 2^-23 / (1 - K 2^-23) (one truncation-sized ulp per addition).
  epilogue  + bias rounds once; ReLU is 1-Lipschitz and exact where the reference is clipped by more than the bound;
            the fma chain over 32 channels rounds 32 times (g32 on the absolute terms); the final ReLU is exact where
            the reference is clipped by more than the bound (bound 0 there).  The sigmoid multiplies the error by
            |sig| / 4 and adds expf (2 ulp), 1 + e and the division: 2^-21 of the output.
test_head_bound_rejects_known_bugs (no GPU) holds a CPU model of the kernel's arithmetic to the same bound, which must
pass well inside it, and nine known bugs injected into that model, which must each exceed it at least tenfold."""
import ctypes
import math

import pytest
import torch
import torch.nn.functional as F

from endodav_b200 import engine as eng

DEV = "cuda"
NAN = float("nan")
TH, TW = 16, 8                       # output tile of head_fused_kernel
U32 = 2.0 ** -24
ETA16 = 2.0 ** -25                   # absolute error of an f16 rounding in the subnormal range
PERIOD = 3                           # the forward-shape inputs repeat every PERIOD frames
DT16 = [torch.bfloat16, torch.float16]


def _dt_id(d):
    return str(d).replace("torch.", "")


def _expected_kernel(dtype, cin):
    return "head_fused<%s,CIN=%d>" % ({torch.bfloat16: "bf16", torch.float16: "f16"}[dtype], cin)


def _tiles(F_, OH, OW):
    return F_ * -(-OH // TH) * -(-OW // TW)


def _gamma(n, unit):
    return n * unit / (1.0 - n * unit)


# ---- reference ---------------------------------------------------------------------------------------------------------
def _coords(n_in, n_out, device):
    """(i0, i1, l): the two source rows (columns) of every output row (column) and the float32 fraction, exactly as
    head_fused_kernel computes them: s = float(n_in - 1) / float(n_out - 1) (0 for n_out = 1), f = s * o, i0 = (int)f,
    l = f - i0, i1 = i0 + 1 clamped to the map."""
    if n_out > 1:
        s = torch.tensor(float(n_in - 1), dtype=torch.float32) / torch.tensor(float(n_out - 1), dtype=torch.float32)
    else:
        s = torch.tensor(0.0, dtype=torch.float32)
    f = s.to(device) * torch.arange(n_out, dtype=torch.float32, device=device)
    i0 = f.long()
    l = f - i0.float()
    i0 = i0.clamp(0, n_in - 1)
    return i0, (i0 + 1).clamp(max=n_in - 1), l


def _weights(ly, lx):
    """float32 [4, OH, OW] bilinear weights (w00, w01, w10, w11) as the kernel rounds them."""
    ly, lx = ly[:, None], lx[None, :]
    return torch.stack([(1.0 - ly) * (1.0 - lx), (1.0 - ly) * lx, ly * (1.0 - lx), ly * lx])


def _corners(xf, cy, cx):
    """The four source pixels of every output pixel of one frame xf [H1, W1, C]: [4, OH, OW, C] in the weights' order."""
    r0, r1 = xf[cy[0]], xf[cy[1]]
    return torch.stack([r0[:, cx[0]], r0[:, cx[1]], r1[:, cx[0]], r1[:, cx[1]]])


def _halo_error(w, xc, dtype):
    """float64 [OH, OW, C] bound on |rounded halo value - float64 lerp| (module docstring)."""
    w = w.double()[..., None]
    a = w * xc.abs()
    if dtype == torch.bfloat16:
        u = 2.0 ** -8
        return (u + (1 + u) * _gamma(4, U32)) * a.sum(0)
    u = 2.0 ** -11
    k = [(1 + u) ** n - 1 for n in (5, 4, 3, 2)]
    return sum(k[i] * a[i] for i in range(4)) + ETA16 * (1 + u) ** 4 * (xc.abs().sum(0) + 4)


def _w4(Wt):
    cin = Wt.shape[1] // 9
    return Wt.view(32, 3, 3, cin).permute(0, 3, 1, 2)


def _epilogue(y, E, b, hw, sig):
    """(ref, bound) [..., OH, OW] from the conv outputs y [.., 32, OH, OW] (float64, no bias) and their error bound E."""
    b, hw = b.double().view(32, 1, 1), hw.double()
    z = y + b
    Ez = E + U32 * (z.abs() + E)
    R = torch.where(z >= 0, Ez, (z + Ez).clamp_min(0.0))        # ReLU: exact where clipped by more than the bound
    r = z.clamp_min(0.0)
    hwv = hw[:32].view(32, 1, 1)
    S = hw[32] + (r * hwv).sum(-3)
    Es = (R * hwv.abs()).sum(-3) + _gamma(32, U32) * (hw[32].abs() + ((r + R) * hwv.abs()).sum(-3))
    if sig == 0.0:
        return S.clamp_min(0.0), torch.where(S >= 0, Es, (S + Es).clamp_min(0.0))
    # sigmoid: its slope, at most 1/4, is at most that at the end of [sig S - e, sig S + e] nearest to 0
    e = abs(sig) * (Es + U32 * (S.abs() + Es))
    p = torch.sigmoid((abs(sig) * S.abs() - e).clamp_min(0.0))
    return torch.sigmoid(sig * S), p * (1 - p) * e + 2.0 ** -21


def _reference(xf, Wt, b, hw, OH, OW, sig, dtype):
    """float64 (ref, bound) [OH, OW] of one frame xf [H1, W1, Cin] (module docstring)."""
    H1, W1, cin = xf.shape
    cy, cx = _coords(H1, OH, xf.device), _coords(W1, OW, xf.device)
    w = _weights(cy[2], cx[2])
    xc = _corners(xf.double(), cy, cx)                              # [4, OH, OW, C]
    up = (w.double()[..., None] * xc).sum(0)
    d = _halo_error(w, xc, dtype)
    del xc
    gk = _gamma(9 * cin, 2.0 ** -23)
    m = (1 + gk) * d + gk * up.abs()
    w4 = _w4(Wt).double()
    y = F.conv2d(up.permute(2, 0, 1)[None], w4, padding=1)[0]
    del up, d
    E = F.conv2d(m.permute(2, 0, 1)[None], w4.abs(), padding=1)[0]
    return _epilogue(y, E, b, hw, sig)


def _excess(err, bound):
    """Worst err / bound (inf where the bound is 0 and the error is not, or where err is NaN)."""
    err = err.nan_to_num(float("inf"))
    r = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, float("inf"), 0.0))
    return float(r.max())


# ---- inputs ------------------------------------------------------------------------------------------------------------
def _randn(shape, g, device):
    return torch.randn(shape, generator=g, device=device)


def _make_inputs(F_, H1, W1, OH, OW, cin, dtype, seed, sig=0.0, period=None, device=DEV):
    """(X, Wt, b, head_w).  X [F_, H1, W1, cin] (dtype, N(0, 1)) is a view of an allocation whose frame F_ is NaN; with
    `period` its frames repeat every `period` frames.  Wt ~ N(0, 1 / (9 cin)) in dtype.  b ~ N(0, 0.1^2): about half
    of every conv channel is clipped by ReLU.  head_w[:32] ~ N(1, 1), scaled so that the 1x1 output of frame 0 (estimated with
    the unfused float32 chain) has unit spread (1.2 for the sigmoid), and head_w[32] is minus its median: about half
    the ReLU-head outputs are clipped, the sigmoid inputs stay within about |s| < 4, and head_w[32] is a few times that
    spread (dropping it is visible)."""
    g = torch.Generator(device=device).manual_seed(seed)
    n = F_ if period is None else min(period, F_)
    base = _randn((n, H1, W1, cin), g, device).to(dtype)
    buf = torch.full((F_ + 1, H1, W1, cin), NAN, dtype=dtype, device=device)
    X = buf[:F_]
    X.copy_(base[torch.arange(F_, device=device) % n])
    Wt = (_randn((32, 9 * cin), g, device) * (9 * cin) ** -0.5).to(dtype)
    b = _randn((32,), g, device) * 0.1
    hw = _randn((33,), g, device) + 1.0
    up = F.interpolate(base[:1].float().permute(0, 3, 1, 2), size=(OH, OW), mode="bilinear", align_corners=True)
    r = F.conv2d(up, _w4(Wt).float(), b, padding=1).clamp_min(0.0)[0]
    t = (r * hw[:32].view(32, 1, 1)).sum(0)
    sd = float(t.std()) if t.numel() > 1 else 0.0
    scale = (1.0 if sig == 0.0 else 1.2) / (sd if sd > 1e-6 else 1.0)
    hw[:32] *= scale
    hw[32] = -float((t * scale).median())
    return X, Wt, b, hw


# ---- CPU model of head_fused_kernel ------------------------------------------------------------------------------------
BUGS = ["halo_shift", "taps_transposed", "frame_minus_one", "lx_ly_swapped", "replicate_padding", "last_k_step_dropped",
        "previous_tile", "head_bias_dropped", "sigmoid_sign_ignored"]


def _emulate(X, Wt, b, hw, OH, OW, sig, dtype, bug=None, grid=5):
    """float64 [F, OH, OW] from a model of the kernel's arithmetic: float32 coordinates and weights; the f16 halo in
    packed half arithmetic (weights rounded to half, HMUL2, three HFMA2, each rounded once), the bf16 halo as an fp32
    lerp rounded once; the conv in fp32 on the rounded halo; bias, ReLU, the 1x1 dot and ReLU | sigmoid in fp32.
    `bug` injects one of BUGS; `grid` is the number of CTAs the previous_tile bug assumes."""
    F_, H1, W1, cin = X.shape
    if bug == "frame_minus_one":
        X = torch.cat([X[:1], X[:-1]])
    cy, cx = _coords(H1, OH, X.device), _coords(W1, OW, X.device)
    if bug == "lx_ly_swapped":
        # the kernel's weight expressions with lx where ly belongs and ly where lx belongs
        ly, lx = cx[2][None, :].expand(OH, OW), cy[2][:, None].expand(OH, OW)
        w = torch.stack([(1.0 - ly) * (1.0 - lx), (1.0 - ly) * lx, ly * (1.0 - lx), ly * lx])
    else:
        w = _weights(cy[2], cx[2])
    w4 = _w4(Wt).float()
    if bug == "taps_transposed":
        w4 = w4.transpose(2, 3)
    if bug == "last_k_step_dropped":
        w4 = w4.clone()
        w4[:, cin - 16:] = 0.0
    ty, tx = -(-OH // TH), -(-OW // TW)
    out = torch.empty(F_, ty * TH, tx * TW, dtype=torch.float64)
    for f in range(F_):
        xc = _corners(X[f].float(), cy, cx)                         # [4, OH, OW, C] values of dtype
        if dtype == torch.float16:
            wh = w.half().float()[..., None]
            t = (wh[0] * xc[0]).half()
            for i in (1, 2, 3):                                     # HFMA2: exact product + sum, one rounding
                t = (wh[i].double() * xc[i].double() + t.double()).float().half()
            up = t.float()
        else:
            ww = w[..., None]
            up = (ww[0] * xc[0] + ww[1] * xc[1] + ww[2] * xc[2] + ww[3] * xc[3]).bfloat16().float()
        up = up.permute(2, 0, 1)
        # the halo beyond the image is zero, also on the padded tile canvas
        canvas = torch.zeros(cin, ty * TH, tx * TW)
        canvas[:, :OH, :OW] = up
        if bug == "halo_shift":
            canvas = torch.cat([canvas[:, :, 1:], torch.zeros(cin, ty * TH, 1)], 2)
        if bug == "replicate_padding":
            pad = F.pad(canvas[None, :, :OH, :OW], (1, 1, 1, 1), mode="replicate")
            acc = torch.zeros(32, ty * TH, tx * TW)
            acc[:, :OH, :OW] = F.conv2d(pad, w4)[0]
        else:
            acc = F.conv2d(canvas[None], w4, padding=1)[0]
        r = (acc + b.view(32, 1, 1)).clamp_min(0.0)
        hb = torch.tensor(0.0) if bug == "head_bias_dropped" else hw[32].clone()
        s = hb.expand_as(r[0]).clone()
        for i in range(32):
            s = s + r[i] * hw[i]
        if sig == 0.0:
            s = s.clamp_min(0.0)
        else:
            sg = 1.0 if bug == "sigmoid_sign_ignored" else sig
            s = 1.0 / (1.0 + torch.exp(-sg * s))
        out[f] = s.double()
    if bug == "previous_tile":
        # CTA c runs tiles c, c + grid, ...: each tile after a CTA's first gets the previous tile's accumulator
        t = out.view(F_, ty, TH, tx, TW).permute(0, 1, 3, 2, 4).reshape(-1, TH, TW)
        t = torch.cat([t[:grid], t[:-grid]])
        out = t.view(F_, ty, tx, TH, TW).permute(0, 1, 3, 2, 4).reshape(F_, ty * TH, tx * TW)
    return out[:, :OH, :OW]


# ---- harness -----------------------------------------------------------------------------------------------------------
WORST = {}   # family -> worst error as a fraction of its bound (printed at the end of the module)


def _note(name, frac):
    WORST[name] = max(WORST.get(name, 0.0), frac)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        print("\nworst error / bound per family:")
        for k in sorted(WORST):
            print("  %-36s %.3f" % (k, WORST[k]))


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _run(X, Wt, b, hw, OH, OW, sig):
    """Launch into the front of a NaN-filled buffer with one guard frame; asserts the instance, the guard and that every
    in-range pixel is finite; returns the [F, OH, OW] output."""
    F_, cin = X.shape[0], X.shape[3]
    buf = torch.full((F_ + 1, OH, OW), NAN, dtype=torch.float32, device=DEV)
    _, kernel = eng.op_disp_head_kernel(X, Wt, b, hw, OH, OW, sig, out=buf)
    torch.cuda.synchronize()
    assert kernel == _expected_kernel(X.dtype, cin), kernel
    assert bool(buf[F_].isnan().all()), "the guard frame behind the output was written"
    got = buf[:F_]
    assert bool(got.isfinite().all()), "%d pixels are not finite" % int((~got.isfinite()).sum())
    return got


def _check(got, X, Wt, b, hw, OH, OW, sig, frames, what, family):
    for f in frames:
        ref, bound = _reference(X[f], Wt, b, hw, OH, OW, sig, X.dtype)
        err = (got[f].double() - ref).abs()
        bad = ~(err <= bound)
        if bool(bad.any()):
            i = int(torch.argmax(torch.where(bad, err - bound, -1.0).flatten()))
            y, x = divmod(i, OW)
            raise AssertionError("%s: frame %d: %d / %d pixels over the bound; worst at (%d, %d): got %r ref %.8g bound %.3g"
                                 % (what, f, int(bad.sum()), bad.numel(), y, x, float(got[f, y, x]), float(ref[y, x]),
                                    float(bound[y, x])))
        _note(family, _excess(err, bound))


def _check_periodic(got, what):
    """Frames of a periodic input equal, bit for bit, the frame PERIOD earlier."""
    for f in range(PERIOD, got.shape[0]):
        assert torch.equal(got[f], got[f % PERIOD]), "%s: frame %d differs from frame %d (same input)" % (what, f, f % PERIOD)


def _run_and_check(F_, H1, W1, OH, OW, cin, dtype, sig, seed, family, periodic=False):
    X, Wt, b, hw = _make_inputs(F_, H1, W1, OH, OW, cin, dtype, seed, sig, period=PERIOD if periodic else None)
    got = _run(X, Wt, b, hw, OH, OW, sig)
    what = "head %s %dx%dx%dx%d -> %dx%d sig=%g" % (_dt_id(dtype), F_, H1, W1, cin, OH, OW, sig)
    frames = range(min(PERIOD, F_)) if periodic else range(F_)
    _check(got, X, Wt, b, hw, OH, OW, sig, frames, what, "%s %s" % (family, _dt_id(dtype)))
    if periodic:
        _check_periodic(got, what)
    return got


# ---- the forward's shapes ----------------------------------------------------------------------------------------------
# DPT head (output_conv2, sig = 0): 8 ph x 8 pw -> net resolution, ViT-S (Cin 32) and ViT-L (Cin 128), at 518^2 and
# 224 x 280, BT = 8 and 32; ViT-L at BT = 128 is the vitl_518_t32_b4 config (274 560 tiles)
DPT_SHAPES = [(bt, h, w, oh, ow, c) for (h, w, oh, ow) in ((296, 296, 518, 518), (128, 160, 224, 280))
              for bt in (8, 32) for c in (32, 128)] + [(128, 296, 296, 518, 518, 128)]
# conv head (HeadDepth, sig = +-1, Cin 32): (ph, pw) -> (2ph, 2pw), ..., (8ph, 8pw) -> (16ph, 16pw)
CONV_HEAD_SHAPES = [(4, k * ph, k * pw, 2 * k * ph, 2 * k * pw, 32) for (ph, pw) in ((37, 37), (16, 20)) for k in (1, 2, 4, 8)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
@pytest.mark.parametrize("BT,H1,W1,OH,OW,cin", DPT_SHAPES)
def test_head_dpt_shapes(BT, H1, W1, OH, OW, cin, dtype):
    """Inputs repeat every PERIOD frames: the first PERIOD frames are held to the float64 reference, every later frame
    must equal its repeat bit for bit."""
    assert _tiles(BT, OH, OW) > 4 * _sms()
    _run_and_check(BT, H1, W1, OH, OW, cin, dtype, 0.0, 1000 + BT + OH + cin, "dpt", periodic=True)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
@pytest.mark.parametrize("sig", [1.0, -1.0])
@pytest.mark.parametrize("BT,H1,W1,OH,OW,cin", CONV_HEAD_SHAPES)
def test_head_conv_head_shapes(BT, H1, W1, OH, OW, cin, sig, dtype):
    _run_and_check(BT, H1, W1, OH, OW, cin, dtype, sig, 2000 + OH + OW + int(sig), "conv head", periodic=True)


# ---- tails and small grids ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
@pytest.mark.parametrize("cin", [32, 128])
@pytest.mark.parametrize("OW", [1, 7, 8, 9])
@pytest.mark.parametrize("OH", [1, 2, 15, 16, 17, 31])
def test_head_tails(OH, OW, cin, dtype):
    """Every class of OH mod 16 and OW mod 8, including OH = 1 and OW = 1 (source step 0), from a 5 x 4 map."""
    _run_and_check(2, 5, 4, OH, OW, cin, dtype, 0.0, 3000 + 32 * OH + OW, "tails")


# (F, H1, W1, OH, OW, cin, sig): single source rows / columns (step 0 on that axis), identity resizes, and the shapes of
# the test this module replaces (40 x 56 -> 70 x 98, 128 x 160 -> 224 x 280, Cin 128 at 16 x 24 -> 28 x 42,
# 9 x 13 -> 18 x 26 with sig = 1, 5 x 5 -> 5 x 5 with sig = -1, 296^2 -> 518^2)
SMALL_SHAPES = [(2, 1, 6, 17, 9, 32, 0.0), (2, 6, 1, 17, 9, 128, 0.0), (1, 1, 1, 5, 7, 32, 1.0), (3, 1, 1, 1, 1, 128, 0.0),
                (2, 17, 9, 17, 9, 32, 0.0), (1, 31, 9, 31, 9, 128, -1.0),
                (2, 40, 56, 70, 98, 32, 0.0), (1, 128, 160, 224, 280, 32, 0.0), (1, 16, 24, 28, 42, 128, 0.0),
                (2, 9, 13, 18, 26, 32, 1.0), (1, 5, 5, 5, 5, 32, -1.0), (1, 296, 296, 518, 518, 32, 0.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
@pytest.mark.parametrize("F_,H1,W1,OH,OW,cin,sig", SMALL_SHAPES)
def test_head_small_shapes(F_, H1, W1, OH, OW, cin, sig, dtype):
    _run_and_check(F_, H1, W1, OH, OW, cin, dtype, sig, 4000 + OH * OW + cin, "small")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
@pytest.mark.parametrize("cin", [32, 128])
@pytest.mark.parametrize("grid", ["half", "sms-1", "sms", "sms+1", "1.5sms", "2sms-1"])
def test_head_grid_sizes(grid, cin, dtype):
    """Total tiles below, at and just above the SM count, and between 1x and 2x it (CTAs run unequal tile counts):
    one frame of one tile row, OW = 8 n - 3."""
    s = _sms()
    n = {"half": s // 2, "sms-1": s - 1, "sms": s, "sms+1": s + 1, "1.5sms": s + s // 2, "2sms-1": 2 * s - 1}[grid]
    OH, OW = 13, 8 * n - 3
    assert _tiles(1, OH, OW) == n
    _run_and_check(1, 7, OW // 2 + 1, OH, OW, cin, dtype, 0.0, 5000 + n + cin, "grid")


# ---- frames ------------------------------------------------------------------------------------------------------------
# (F, H1, W1, OH, OW, cin): 3 920 tiles, 26 per CTA on 148 SMs, at each ring depth
INDEPENDENT = [(8, 128, 160, 224, 280, 32), (8, 128, 160, 224, 280, 128)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
@pytest.mark.parametrize("F_,H1,W1,OH,OW,cin", INDEPENDENT)
def test_head_frames_are_independent(F_, H1, W1, OH, OW, cin, dtype):
    """A pixel's arithmetic does not depend on the CTA or on what it ran before: frames 0, F/2 and F-1 of the launch
    equal, bit for bit, the same frame launched alone and the same frames in a launch whose other frames differ."""
    assert _tiles(F_, OH, OW) > 4 * _sms()
    X, Wt, b, hw = _make_inputs(F_, H1, W1, OH, OW, cin, dtype, 6000 + cin)
    full = _run(X, Wt, b, hw, OH, OW, 0.0).clone()
    keep = (0, F_ // 2, F_ - 1)
    for f in keep:
        xs = torch.full((2, H1, W1, cin), NAN, dtype=dtype, device=DEV)
        xs[0] = X[f]
        alone = _run(xs[:1], Wt, b, hw, OH, OW, 0.0)
        assert torch.equal(alone[0], full[f]), "frame %d differs when launched alone" % f
    other, _, _, _ = _make_inputs(F_, H1, W1, OH, OW, cin, dtype, 6100 + cin)
    for f in keep:
        other[f] = X[f]
    mixed = _run(other, Wt, b, hw, OH, OW, 0.0)
    for f in keep:
        assert torch.equal(mixed[f], full[f]), "frame %d depends on the other frames" % f
    _check(full, X, Wt, b, hw, OH, OW, 0.0, keep, "independent %s cin=%d" % (_dt_id(dtype), cin), "independent " + _dt_id(dtype))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
@pytest.mark.parametrize("sig", [0.0, -1.0])
@pytest.mark.parametrize("F_,H1,W1,OH,OW,cin", [(7, 64, 80, 112, 140, 32), (7, 64, 80, 112, 140, 128)])
def test_head_poisoned_neighbour(F_, H1, W1, OH, OW, cin, sig, dtype):
    """Odd frames are scaled by 2^10: a read of frame f +- 1 for frame f dominates frame f's output (F odd: after the
    last, unscaled frame comes the NaN frame)."""
    X, Wt, b, hw = _make_inputs(F_, H1, W1, OH, OW, cin, dtype, 7000 + cin)
    X[1::2] *= 1024.0
    got = _run(X, Wt, b, hw, OH, OW, sig)
    _check(got, X, Wt, b, hw, OH, OW, sig, range(F_), "poisoned neighbour %s cin=%d sig=%g" % (_dt_id(dtype), cin, sig),
           "poison " + _dt_id(dtype))


# ---- rejections --------------------------------------------------------------------------------------------------------
# each entry overrides one argument of a valid call (F = 2, 8 x 8 -> 16 x 16, Cin = 32, bf16)
BAD_ARGS = [dict(X=0), dict(Wt=0), dict(bias=0), dict(head_w=0), dict(out=0), dict(X_off=2), dict(X_off=8), dict(Wt_off=4),
            dict(dtype=eng.EDV_F32), dict(dtype=3), dict(dtype=-1), dict(Cin=64), dict(Cin=16), dict(Cin=0), dict(F=0),
            dict(F=-1), dict(H1=0), dict(W1=0), dict(H1=-2), dict(OH=0), dict(OW=0), dict(OW=-8),
            dict(F=1 << 30, OH=1024, OW=1024)]   # 2^43 tiles


def _call(lib, a, name, stream):
    return lib.edv_op_disp_head(a["dtype"], ctypes.c_void_p(a["X"] and a["X"] + a.get("X_off", 0)),
                                ctypes.c_void_p(a["Wt"] and a["Wt"] + a.get("Wt_off", 0)), ctypes.c_void_p(a["bias"]),
                                ctypes.c_void_p(a["head_w"]), ctypes.c_void_p(a["out"]), a["F"], a["H1"], a["W1"], a["OH"],
                                a["OW"], a["Cin"], ctypes.c_float(0.0), name, 64, stream)


def test_head_rejects_bad_arguments():
    """edv_op_disp_head returns EDV_ERR_ARG, before any launch, for each argument it cannot run.  The pointers are fake,
    so this runs only where there is no device: a check that went missing fails with EDV_ERR_CUDA instead."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = eng.load_library()
    ok = dict(dtype=eng.EDV_BF16, X=1 << 20, Wt=2 << 20, bias=3 << 20, head_w=4 << 20, out=5 << 20, F=2, H1=8, W1=8, OH=16,
              OW=16, Cin=32)
    name = ctypes.create_string_buffer(64)
    for bad in BAD_ARGS:
        name.value = b"stale"
        rc = _call(lib, dict(ok, **bad), name, ctypes.c_void_p(0))
        assert rc == -1, (bad, rc)                                  # EDV_ERR_ARG
        assert lib.edv_last_error(ctypes.c_void_p(0)), bad
        assert name.value == b"", (bad, name.value)                # no kernel ran


@pytest.mark.gpu
def test_head_rejections_leave_the_output_untouched():
    """The same rejections with real buffers on the device: nothing is launched, the NaN output stays NaN; the valid call
    then runs and writes every pixel."""
    lib = eng.load_library()
    X, Wt, b, hw = _make_inputs(2, 8, 8, 16, 16, 32, torch.bfloat16, 8000)
    out = torch.full((3, 16, 16), NAN, device=DEV)
    ok = dict(dtype=eng.EDV_BF16, X=X.data_ptr(), Wt=Wt.data_ptr(), bias=b.data_ptr(), head_w=hw.data_ptr(),
              out=out.data_ptr(), F=2, H1=8, W1=8, OH=16, OW=16, Cin=32)
    name = ctypes.create_string_buffer(64)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for bad in BAD_ARGS:
        name.value = b"stale"
        assert _call(lib, dict(ok, **bad), name, stream) == -1, bad
        assert name.value == b"", (bad, name.value)
    torch.cuda.synchronize()
    assert bool(out.isnan().all()), "a rejected call wrote the output"
    assert _call(lib, ok, name, stream) == 0
    torch.cuda.synchronize()
    assert name.value == b"head_fused<bf16,CIN=32>", name.value
    assert bool(out[:2].isfinite().all()) and bool(out[2].isnan().all())


# ---- the bound itself, without a GPU -----------------------------------------------------------------------------------
# (F, H1, W1, OH, OW, cin, sig): multi-tile, multi-frame, non-square scales (lx != ly), partial tiles; the forward's
# combinations: the DPT head (sig = 0) at Cin 32 and 128, the conv head (sig = +-1) at Cin 32
MODEL_SHAPES = [(3, 9, 13, 37, 26, 32, 0.0), (2, 6, 5, 21, 17, 128, 0.0), (2, 7, 10, 20, 27, 32, -1.0),
                (2, 5, 6, 18, 23, 32, 1.0)]


@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
def test_head_bound_rejects_known_bugs(dtype):
    """On the CPU: the model of the kernel's arithmetic (_emulate) passes the bound well inside 1 on small multi-tile,
    multi-frame shapes, and each known bug injected into that model exceeds it at least tenfold on every shape it
    applies to."""
    worst = {}
    for shape in MODEL_SHAPES:
        F_, H1, W1, OH, OW, cin, sig = shape
        assert _tiles(F_, OH, OW) > 2 * 5                          # CTAs of the 5-CTA model run 2 or more tiles
        X, Wt, b, hw = _make_inputs(F_, H1, W1, OH, OW, cin, dtype, 9000 + OH + cin, sig, device="cpu")
        refs = [_reference(X[f], Wt, b, hw, OH, OW, sig, dtype) for f in range(F_)]
        ref = torch.stack([r[0] for r in refs])
        bound = torch.stack([r[1] for r in refs])
        frac = _excess((_emulate(X, Wt, b, hw, OH, OW, sig, dtype) - ref).abs(), bound)
        worst["model"] = max(worst.get("model", 0.0), frac)
        assert frac <= 0.5, (shape, frac)
        for bug in BUGS:
            if bug == "sigmoid_sign_ignored" and sig != -1.0:
                continue
            frac = _excess((_emulate(X, Wt, b, hw, OH, OW, sig, dtype, bug) - ref).abs(), bound)
            worst[bug] = min(worst.get(bug, math.inf), frac)
            assert frac >= 10.0, (bug, shape, frac)
    print("\n%s: model %.3f of the bound; each bug at least:" % (_dt_id(dtype), worst.pop("model")))
    for bug in BUGS:
        print("  %-24s %.3g x the bound" % (bug, worst[bug]))
