"""The fused GEMM + residual + LayerNorm (edv_op_linear_residual_ln: gemm_ln_kernel) at the forward's shapes, against a
float64 reference.

gemm_ln_kernel runs the ViT-S `blk.proj` (K = 384) and `blk.fc2` (K = 1536) call sites of the 16-bit forward:
x += A W^T + b on the fp32 residual stream in place, and xn = LayerNorm(x) in 16 bit (fc2 of the last block, and of a
block followed by a residual bottleneck, skips the LayerNorm).  A cluster of two CTAs owns a 128-row tile, CTA `rank`
the columns [192 rank, +192); pairs walk tiles tile = pair, pair + npairs, ... with two TMEM accumulators and two
mailboxes for the peer's half-row statistics, both by tile parity.  So the shapes here run up to 9 - 10 tiles per pair
(npairs = 74 on 148 SMs), grids below, at and just above one tile per pair, and 1 to 48 k-blocks against the 3-stage ring.
Rows launched alone through pointer-offset views must equal, bit for bit, the same rows of a large launch, and two
back-to-back launches on one stream (programmatic dependent launch) must equal the same launches with a synchronise
between them.

A is a view of the first M rows of an allocation whose next rows are NaN; x sits between rows of a finite sentinel
(a store past M would write sentinel + b + acc, which a NaN guard would not show), which must stay bit-identical; xn goes
to the front of a NaN-filled buffer whose guard rows must stay NaN.  Every case asserts which instance ran.

Input families (_make_inputs), each with per-row statistics from a hash of the row index, so that row r of tile t and of
tile t +- 1, t +- 2 differ by O(1):
  forward     mean in [-4, 4], spread in [0.5, 4], the two 192-column halves tilted by up to +-1 spread;
  split       halves at +-a, a = 1.5 .. 2.5 spreads: Chan's dm^2 term is most of the variance;
  massive     one column of each half at +-(50 .. 300) on a tilted bulk (the DINOv2 outlier channels);
  offset      250 .. 350 + a spread of 0.5 .. 2: the precision of the mean;
  degenerate  A rows zero, x0 = c - b exactly: half the rows have variance 0 (rstd = eps^-1/2), the others halves at
              +-t with t^2 < eps.

Reference and tolerance:
  x   x* = x0 + b + A W^T in float64 on the same 16-bit A and W, P = |A| |W|^T.  The kernel computes
      x^ = fl(acc + fl(b + x0)); the 16-bit products are exact in fp32, so
      |x^ - x*| <= gK P + u |b + x0| + u |x^|,  u = 2^-24, gK = K 2^-23 / (1 - K 2^-23).
  xn  LayerNorm in float64 of the kernel's own rows x^ (what it holds in TMEM), so the K-sum is checked once, by x.
      The bound (_ln_reference) follows the kernel's fp32 steps (gemm_ln.cuh):
        half sum    quads, 12 sequential adds, the tree of 4 warpgroup partials: depth 15; the half mean multiplies by
                    the rounded 1/192: |dh| <= g17 sum_half |x| / 192;
        mean        the pair sum and the rounded 1/384: |dmu| <= g18 sum |x| / 384;
        variance    the centred squares (fmaf, 48 per warpgroup) and the pair sum: g56 on M2a + M2b; centring on an
                    inexact half mean adds 192 dh^2 per half; Chan's 96 dm^2 with dm off by up to 2 dh; g9 on it;
        rstd        fl(var + eps), then rsqrtf (relative error <= 2^-22.9, PTX ISA);
        output      ((x - mean) rstd) gamma + beta with fma contraction allowed: the mean error times rstd |gamma|
                    stays in the bound (it dominates on large-offset rows and on rows with variance near eps), then
                    one 16-bit rounding (bf16 u = 2^-8, f16 u = 2^-11 plus 2^-25 for subnormals).
test_gemm_ln_bound_rejects_known_bugs (no GPU) holds a float32 model of the epilogue, in the kernel's order, to the
same bounds: it must pass the fp32 part of the xn bound within half of it, and each of ten known bugs injected into it
must exceed the bounds at least tenfold on every family it applies to."""
import ctypes
import math

import numpy as np
import pytest
import torch

from endodav_b200 import engine as eng

DEV = "cuda"
NAN = float("nan")
N, HN, BM = 384, 192, 128            # row width, columns per CTA of the pair, rows per tile
U32 = 2.0 ** -24
RSQRT_REL = 2.0 ** -22.9             # rsqrt.approx.f32 maximum relative error (PTX ISA)
EPS = float(np.float32(1e-6))        # the forward's eps as the kernel receives it
SENTINEL = 7777.25                   # guard rows around x
G = 3                                # guard rows
ETA16 = 2.0 ** -25
DT16 = [torch.bfloat16, torch.float16]
FAMILIES = ["forward", "split", "massive", "offset", "degenerate"]


def _dt_id(d):
    return str(d).replace("torch.", "")


def _expected_kernel(dtype):
    return "gemm_ln<%s>" % {torch.bfloat16: "bf16", torch.float16: "f16"}[dtype]


def _g(n, unit=U32):
    return n * unit / (1.0 - n * unit)


def _tiles(M):
    return -(-M // BM)


# ---- reference ---------------------------------------------------------------------------------------------------------
def _x_reference(A, W, b, x0, xh):
    """float64 (x*, bound) [M, 384] (module docstring)."""
    Ad, Wd = A.double(), W.double()
    bx = b.double() + x0.double()
    ref = bx + Ad @ Wd.T
    P = Ad.abs() @ Wd.abs().T
    K = A.shape[1]
    return ref, _g(K, 2.0 ** -23) * P + U32 * bx.abs() + U32 * xh.double().abs()


def _ln_reference(xh, gam, bet, dtype, eps=EPS):
    """float64 (ref, bound, bound32) [M, 384] of xn from the kernel's own fp32 rows xh (module docstring); bound32 is the
    part of the bound before the final 16-bit rounding."""
    v = xh.double()
    a, c = v[:, :HN], v[:, HN:]
    ma, mb = a.mean(1, keepdim=True), c.mean(1, keepdim=True)
    mu = v.mean(1, keepdim=True)
    d = v - mu
    m2a = ((a - ma) ** 2).sum(1, keepdim=True)
    m2b = ((c - mb) ** 2).sum(1, keepdim=True)
    vs = (d * d).mean(1, keepdim=True) + eps
    r = vs.rsqrt()
    g, be = gam.double(), bet.double()
    ref = d * r * g + be
    sa, sb = a.abs().sum(1, keepdim=True), c.abs().sum(1, keepdim=True)
    dh = _g(17) * torch.maximum(sa, sb) / HN             # half-mean error
    dmu = _g(18) * (sa + sb) / N                         # mean error
    dm = (ma - mb).abs()
    D = dm + 2 * dh
    e_var = (_g(56) * (m2a + m2b) + (2 + _g(56)) * N * dh * dh + N * dm * dh + _g(9) * 96 * D * D) / N
    e_w = e_var * (1 + U32) + U32 * vs
    assert bool((e_w < vs).all())
    rel_r = (1 + RSQRT_REL) * (1 - e_w / vs).rsqrt() - 1
    k = (1 + rel_r) * (1 + _g(3))
    ez = g.abs() * r * (d.abs() * (k - 1) + dmu * k)
    e32 = ez * (1 + U32) + U32 * ref.abs()
    u16, eta = (2.0 ** -8, 0.0) if dtype == torch.bfloat16 else (2.0 ** -11, ETA16)
    return ref, e32 + u16 * (ref.abs() + e32) + eta, e32


def _excess(err, bound):
    """Worst err / bound (inf where the bound is 0 and the error is not, or where err is NaN)."""
    err = err.nan_to_num(float("inf"))
    r = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, float("inf"), 0.0))
    return float(r.max())


# ---- inputs ------------------------------------------------------------------------------------------------------------
def _hash_u(rows, k):
    """Uniform [0, 1) per row index, stream k (an integer hash: neighbouring rows and tiles are unrelated)."""
    h = (rows * 0x5BD1E995 + (k + 1) * 0x27D4EB2D) & 0xFFFFFFFF
    h = h ^ (h >> 15)
    h = (h * 0x165667B1) & 0xFFFFFFFF
    h = h ^ (h >> 13)
    h = (h * 0x5BD1E995) & 0xFFFFFFFF
    h = h ^ (h >> 16)
    return (h.double() / 2.0 ** 32).float()[:, None]


def _make_inputs(M, K, dtype, family, seed, device=DEV):
    """(A, W, b, x0, gamma, beta).  A [M, K] (dtype) is a view of an allocation whose next G rows are NaN, W [384, K]
    ~ N(0, 0.25 / K) so that A W^T has spread 0.5, b ~ N(0, 0.1^2), gamma ~ 1 + N(0, 0.2^2), beta ~ N(0, 0.1^2);
    x0 [M, 384] float32 by family (module docstring)."""
    g = torch.Generator(device=device).manual_seed(seed)
    rows = torch.arange(M, device=device, dtype=torch.int64)
    u = [_hash_u(rows, 16 * seed + k) for k in range(10)]
    sgn = torch.ones(N, device=device)
    sgn[HN:] = -1.0
    buf = torch.full((M + G, K), NAN, dtype=dtype, device=device)
    A = buf[:M]
    A.copy_(torch.randn((M, K), generator=g, device=device))
    W = (torch.randn((N, K), generator=g, device=device) * (0.5 / math.sqrt(K))).to(dtype)
    b = torch.randn((N,), generator=g, device=device) * 0.1
    gam = 1.0 + 0.2 * torch.randn((N,), generator=g, device=device)
    bet = 0.1 * torch.randn((N,), generator=g, device=device)
    z = torch.randn((M, N), generator=g, device=device)
    mu, sd = -4.0 + 8.0 * u[0], 0.5 + 3.5 * u[1]
    if family == "forward":
        x0 = mu + sd * (z + (2.0 * u[2] - 1.0) * sgn)
    elif family == "split":
        a = (1.5 + u[2]) * sd * torch.where(u[3] < 0.5, -1.0, 1.0)
        x0 = mu + sd * z + a * sgn
    elif family == "massive":
        x0 = mu + sd * (z + (6.0 * u[2] - 3.0) * sgn)
        ca = (u[4] * HN).long().clamp(max=HN - 1)
        cb = HN + (u[5] * HN).long().clamp(max=HN - 1)
        va = (50.0 + 250.0 * u[6]) * torch.where(u[8] < 0.5, -1.0, 1.0)
        vb = (50.0 + 250.0 * u[7]) * torch.where(u[9] < 0.5, -1.0, 1.0)
        x0.scatter_(1, ca, va)
        x0.scatter_(1, cb, vb)
    elif family == "offset":
        x0 = 250.0 + 100.0 * u[0] + (0.5 + 1.5 * u[1]) * (z + (2.0 * u[2] - 1.0) * sgn)
    elif family == "degenerate":
        A.zero_()
        b = torch.round(b * 1024) / 1024                       # b, c and c - b exact in fp32: b + x0 == c
        c = torch.round(mu * 256) / 256
        t = (4e-4 + 5e-4 * u[2]) * torch.where(u[3] < 0.5, 0.0, 1.0) * torch.where(u[4] < 0.5, -1.0, 1.0)
        x0 = (c - b) + t * sgn
    else:
        raise ValueError(family)
    return A, W, b, x0.contiguous(), gam, bet


# ---- CPU model of the epilogue -----------------------------------------------------------------------------------------
BUGS = ["chan_term_dropped", "chan_weight_192", "mean_of_own_half", "mailbox_two_tiles_back", "bias_of_other_half",
        "gamma_beta_of_other_half", "residual_subtiles_swapped", "eps_dropped", "eps_outside_sqrt", "variance_over_383"]
# the families on which a bug changes xn by more than the bound allows for: eps matters only where the variance is
# below or near eps (degenerate rows); dividing by 383 changes xn - beta by 0.13 %, less than the mean-error allowance of
# offset rows (g18 * 300 * rstd) and than the eps-dominated rstd of degenerate rows
APPLIES = {bug: set(FAMILIES) for bug in BUGS}
APPLIES["eps_dropped"] = APPLIES["eps_outside_sqrt"] = {"degenerate"}
APPLIES["variance_over_383"] = {"forward", "split", "massive"}


def _rsqrt_worst(w):
    """rsqrtf at its worst-case relative error: the largest float32 at most (1 + 2^-22.9) / sqrt(w)."""
    with np.errstate(divide="ignore", invalid="ignore"):
        r64 = (1.0 + RSQRT_REL) / np.sqrt(w.astype(np.float64))
    r = r64.astype(np.float32)
    return np.where(r.astype(np.float64) > r64, np.nextafter(r, np.float32(0)), r)


def _model(A, W, b, x0, gam, bet, dtype, npairs, bug=None, eps=EPS):
    """(x^, xn, xn before its 16-bit rounding) from a float32 model of gemm_ln_kernel's epilogue in the kernel's own order (gemm_ln.cuh): pass 1 quads
    and 12 sequential adds per warpgroup, the tree of 4 warpgroup partials, the half mean, fmaf-centred squares, the
    mailbox by tile parity (pairs walk tile = pair, pair + npairs, ...), Chan's combination, rsqrtf at its worst-case
    error, ((x - mean) rstd) gamma + beta and one 16-bit rounding.  The accumulator is A W^T rounded once to fp32 (the
    tensor core's sum lies within the same bound).  `bug` injects one of BUGS."""
    f32 = np.float32
    M = A.shape[0]
    acc = (A.double().numpy() @ W.double().numpy().T).astype(f32)
    bias = b.numpy().astype(f32).copy()
    if bug == "bias_of_other_half":
        bias[HN:] = bias[:HN]                                   # col_half dropped: both CTAs read bias[0, 192)
    res = x0.numpy().astype(f32).copy()
    if bug == "residual_subtiles_swapped":
        r4 = res.reshape(M, 8, 3, 16)
        r4[:, :, [0, 1]] = r4[:, :, [1, 0]]
    xh = acc + (bias[None, :] + res)
    mp = _tiles(M) * BM
    xp = np.zeros((mp, N), f32)
    xp[:M] = xh
    v = xp.reshape(mp, 2, 4, 48)                                # [row, half, warpgroup, column]
    part = np.zeros((mp, 2, 4), f32)
    for k in range(12):
        q = v[..., 4 * k:4 * k + 4]
        part = part + ((q[..., 0] + q[..., 1]) + (q[..., 2] + q[..., 3]))
    hsum = (part[..., 0] + part[..., 1]) + (part[..., 2] + part[..., 3])          # [row, half]
    hmean = hsum * f32(1.0 / HN)
    sq = np.zeros((mp, 2, 4), f32)
    for i in range(48):
        dd = v[..., i] - hmean[..., None]
        sq = (dd.astype(np.float64) ** 2 + sq.astype(np.float64)).astype(f32)     # fmaf(d, d, sq)
    hm2 = (sq[..., 0] + sq[..., 1]) + (sq[..., 2] + sq[..., 3])
    pm_s, pm_m2 = hsum[:, ::-1].copy(), hm2[:, ::-1].copy()                         # the peer's half
    if bug == "mailbox_two_tiles_back":
        t = np.arange(mp) // BM
        late = t >= 2 * npairs                                  # a pair's third tile onwards
        src = np.arange(mp) - 2 * npairs * BM
        pm_s[late], pm_m2[late] = pm_s[src[late]], pm_m2[src[late]]
    mean = (hsum + pm_s) * f32(1.0 / N)
    if bug == "mean_of_own_half":
        mean = hmean
    dm = hmean - pm_s * f32(1.0 / HN)
    chan = dm * dm * f32(192.0 if bug == "chan_weight_192" else 0.25 * N)
    s = hm2 + pm_m2
    if bug != "chan_term_dropped":
        s = s + chan
    var = s * f32(1.0 / 383.0 if bug == "variance_over_383" else 1.0 / N)
    if bug == "eps_dropped":
        rstd = _rsqrt_worst(var)
    elif bug == "eps_outside_sqrt":
        rstd = _rsqrt_worst(var) + f32(eps)
    else:
        rstd = _rsqrt_worst(var + f32(eps))
    gm, bt = gam.numpy().astype(f32).reshape(2, HN), bet.numpy().astype(f32).reshape(2, HN)
    if bug == "gamma_beta_of_other_half":
        gm, bt = gm[::-1], bt[::-1]
    vh = xp.reshape(mp, 2, HN)
    with np.errstate(invalid="ignore", over="ignore"):
        y = ((vh - mean[..., None]) * rstd[..., None]) * gm[None] + bt[None]
    y = torch.from_numpy(y.reshape(mp, N)[:M].copy())
    return torch.from_numpy(xh), y.to(dtype), y


# ---- harness -----------------------------------------------------------------------------------------------------------
WORST = {}   # "family dtype x|xn" -> worst error as a fraction of its bound (printed at the end of the module)


def _note(name, frac):
    WORST[name] = max(WORST.get(name, 0.0), frac)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        print("\nworst error / bound per family and dtype:")
        for k in sorted(WORST):
            print("  %-32s %.3f" % (k, WORST[k]))


def _guarded(M, x0, dtype, ln):
    """(xbuf, x, xnbuf, xn): x0 copied into rows [G, G + M) of a SENTINEL buffer; xn the first M rows of a NaN buffer."""
    xbuf = torch.full((M + 2 * G, N), SENTINEL, dtype=torch.float32, device=DEV)
    x = xbuf[G:G + M]
    x.copy_(x0)
    xnbuf = torch.full((M + G, N), NAN, dtype=dtype, device=DEV) if ln else None
    return xbuf, x, xnbuf, (xnbuf[:M] if ln else None)


def _launch(A, W, b, x, gam, bet, xn):
    _, kernel = eng.op_linear_residual_ln_kernel(A, W, b, x, gam if xn is not None else None,
                                                 bet if xn is not None else None, EPS, xn=xn)
    assert kernel == _expected_kernel(A.dtype), kernel
    return kernel


def _check_guards(xbuf, x, xnbuf, xn, M):
    assert bool((xbuf[:G] == SENTINEL).all()) and bool((xbuf[G + M:] == SENTINEL).all()), "a guard row of x was written"
    assert bool(x.isfinite().all()), "%d x values are not finite" % int((~x.isfinite()).sum())
    if xn is not None:
        assert bool(xnbuf[M:].isnan().all()), "a guard row behind xn was written"
        assert bool(xn.isfinite().all()), "%d xn values are not finite" % int((~xn.isfinite()).sum())


def _run(A, W, b, x0, gam, bet, ln=True):
    """One launch with guards on every buffer; asserts the instance, the guards and finiteness; returns (x, xn)."""
    M = A.shape[0]
    xbuf, x, xnbuf, xn = _guarded(M, x0, A.dtype, ln)
    _launch(A, W, b, x, gam, bet, xn)
    torch.cuda.synchronize()
    _check_guards(xbuf, x, xnbuf, xn, M)
    return x, xn


def _fail(what, err, bound, got, ref):
    bad = ~(err <= bound)
    i = int(torch.argmax(torch.where(bad, err - bound, -1.0).flatten()))
    r, c = divmod(i, N)
    raise AssertionError("%s: %d / %d values over the bound; worst at row %d col %d: got %r ref %.8g bound %.3g"
                         % (what, int(bad.sum()), bad.numel(), r, c, float(got[r, c]), float(ref[r, c]), float(bound[r, c])))


def _check(x, xn, A, W, b, x0, gam, bet, what, family):
    dt = _dt_id(A.dtype)
    ref, bound = _x_reference(A, W, b, x0, x)
    err = (x.double() - ref).abs()
    if not bool((err <= bound).all()):
        _fail(what + " x", err, bound, x, ref)
    _note("%s %s x" % (family, dt), _excess(err, bound))
    del ref, bound, err
    if xn is not None:
        ref, bound, _ = _ln_reference(x, gam, bet, A.dtype)
        err = (xn.double() - ref).abs()
        if not bool((err <= bound).all()):
            _fail(what + " xn", err, bound, xn, ref)
        _note("%s %s xn" % (family, dt), _excess(err, bound))


def _run_and_check(M, K, dtype, family, seed, ln=True, residual_only_too=False):
    A, W, b, x0, gam, bet = _make_inputs(M, K, dtype, family, seed)
    what = "gemm_ln %s M=%d K=%d %s%s" % (_dt_id(dtype), M, K, family, "" if ln else " residual only")
    x, xn = _run(A, W, b, x0, gam, bet, ln)
    _check(x, xn, A, W, b, x0, gam, bet, what, family)
    if residual_only_too:
        # the residual-only form (the forward's fc2 before a bottleneck and of the last block) writes the same x
        x2, _ = _run(A, W, b, x0, gam, bet, ln=False)
        assert torch.equal(x2, x), "%s: the residual-only form writes a different x" % what


# ---- the forward's shapes ----------------------------------------------------------------------------------------------
# M = BT * (1 + h w / 196) tokens: bench 224 x 280 at BT 8 (2 568) and 32 (10 272: 81 tiles, 7 pairs run 2), 518^2 at BT
# 32 (43 840: 343 tiles, 47 pairs run 5, 27 run 4) and 64 (87 680: 685 tiles, 9 - 10 per pair); the golden configs'
# 36 ... 642 (102 and below are one partial tile)
FORWARD_M = [36, 39, 48, 65, 102, 144, 640, 642, 2568, 10272, 43840, 87680]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
@pytest.mark.parametrize("site", ["proj", "fc2"])
@pytest.mark.parametrize("M", FORWARD_M)
def test_gemm_ln_forward_shapes(M, site, dtype):
    """blk.proj (K = 384) and blk.fc2 (K = 1536), with the LayerNorm and, for fc2, in the residual-only form too."""
    K = 384 if site == "proj" else 1536
    _run_and_check(M, K, dtype, "forward", 100 + (M % 997) + K, residual_only_too=(site == "fc2"))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
@pytest.mark.parametrize("M", [1, 127, 128, 129, 9472, 9473, 18944])
def test_gemm_ln_grid_edges(M, dtype):
    """One row, one tile +- 1 row, exactly one tile per pair (9 472 = 74 x 128), one more row (pair 0's second tile has
    one row) and exactly two tiles per pair."""
    _run_and_check(M, 384, dtype, "forward", 200 + M % 997)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
@pytest.mark.parametrize("K", [64, 128, 192, 3072])
def test_gemm_ln_ring_edges(K, dtype):
    """1, 2 and 3 k-blocks against the 3-stage ring (the producer's prefetch reaches into the next tile), and 48, over
    157 tiles (2 - 3 per pair)."""
    _run_and_check(20000, K, dtype, "forward", 300 + K)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
@pytest.mark.parametrize("K", [384, 1536])
@pytest.mark.parametrize("family", FAMILIES)
def test_gemm_ln_families(family, K, dtype):
    """Every input family at the 518^2 BT 32 shape (4 - 5 tiles per pair)."""
    _run_and_check(43840, K, dtype, family, 400 + FAMILIES.index(family) + K)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
@pytest.mark.parametrize("M,K", [(128, 384), (300, 384), (2568, 1536), (1370 * 4 + 7, 384), (20000, 1536)])
def test_gemm_ln_shapes(M, K, dtype):
    """Single and partial tiles, and up to 157 tiles, with the residual-only form bit-identical in x."""
    _run_and_check(M, K, dtype, "forward", 500 + M % 997 + K, residual_only_too=True)


# ---- row position and dependent launches -------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
def test_gemm_ln_rows_do_not_depend_on_position(dtype):
    """Rows [a, a + n) launched alone, through pointer-offset views of A, x and xn, equal bit for bit the same rows of
    the M = 43 840 launch: a = 1 and 77 move every row to another thread of its tile, a = 9 473 to another pair and the
    other tile parity.  The rest of the x and xn buffers stays untouched."""
    M, K = 43840, 384
    A, W, b, x0, gam, bet = _make_inputs(M, K, dtype, "forward", 600)
    x_full, xn_full = _run(A, W, b, x0, gam, bet)
    _check(x_full, xn_full, A, W, b, x0, gam, bet, "position full %s" % _dt_id(dtype), "forward")
    for a, n in [(1, 300), (77, 1000), (9473, 517)]:
        xbuf, _, xnbuf, _ = _guarded(M, x0, dtype, True)
        x, xn = xbuf[G + a:G + a + n], xnbuf[a:a + n]
        _launch(A[a:a + n], W, b, x, gam, bet, xn)
        torch.cuda.synchronize()
        assert torch.equal(x, x_full[a:a + n]), "x rows [%d, %d) differ when launched alone" % (a, a + n)
        assert torch.equal(xn, xn_full[a:a + n]), "xn rows [%d, %d) differ when launched alone" % (a, a + n)
        assert torch.equal(xbuf[G:G + a], x0[:a]) and torch.equal(xbuf[G + a + n:G + M], x0[a + n:]), "x outside the rows"
        assert bool((xbuf[:G] == SENTINEL).all()) and bool((xbuf[G + M:] == SENTINEL).all())
        assert bool(xnbuf[:a].isnan().all()) and bool(xnbuf[a + n:].isnan().all()), "xn outside the rows was written"


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
def test_gemm_ln_dependent_launches(dtype):
    """A proj-like and then an fc2-like launch on the same x, back to back on one stream (the second starts its prologue
    under the first one's tail), equal bit for bit the same two launches with a synchronise between them."""
    M = 43840
    A1, W1, b1, x0, g1, be1 = _make_inputs(M, 384, dtype, "forward", 700)
    A2, W2, b2, _, g2, be2 = _make_inputs(M, 1536, dtype, "forward", 701)
    xbuf, x, xnbuf1, xn1 = _guarded(M, x0, dtype, True)
    xnbuf2 = torch.full((M + G, N), NAN, dtype=dtype, device=DEV)
    torch.cuda.synchronize()
    _launch(A1, W1, b1, x, g1, be1, xn1)
    _launch(A2, W2, b2, x, g2, be2, xnbuf2[:M])
    torch.cuda.synchronize()
    _check_guards(xbuf, x, xnbuf1, xn1, M)
    _check_guards(xbuf, x, xnbuf2, xnbuf2[:M], M)
    ybuf, y, ynbuf1, yn1 = _guarded(M, x0, dtype, True)
    ynbuf2 = torch.full((M + G, N), NAN, dtype=dtype, device=DEV)
    _launch(A1, W1, b1, y, g1, be1, yn1)
    torch.cuda.synchronize()
    y1 = y.clone()
    _launch(A2, W2, b2, y, g2, be2, ynbuf2[:M])
    torch.cuda.synchronize()
    assert torch.equal(xn1, yn1), "the first launch's xn differs when the second follows it directly"
    assert torch.equal(x, y), "x differs when the launches follow each other directly"
    assert torch.equal(xnbuf2[:M], ynbuf2[:M]), "the second launch's xn differs when it follows the first directly"
    _check(y1, yn1, A1, W1, b1, x0, g1, be1, "dependent proj %s" % _dt_id(dtype), "forward")
    _check(y, ynbuf2[:M], A2, W2, b2, y1, g2, be2, "dependent fc2 %s" % _dt_id(dtype), "forward")


# ---- rejections --------------------------------------------------------------------------------------------------------
# each entry overrides arguments of a valid call (M = 256, K = 384, bf16, with the LayerNorm)
BAD_ARGS = [dict(dtype=eng.EDV_F32), dict(dtype=3), dict(dtype=-1), dict(A=0), dict(W=0), dict(x=0), dict(A_off=2),
            dict(A_off=8), dict(W_off=4), dict(x_off=4), dict(x_off=8), dict(xn_off=2), dict(gamma=0), dict(beta=0),
            dict(xn=0), dict(gamma=0, beta=0), dict(gamma=0, xn=0), dict(beta=0, xn=0), dict(M=0), dict(M=-1),
            dict(M=2 ** 31 - 127), dict(M=2 ** 31 - 1), dict(N=383), dict(N=768), dict(N=0), dict(K=0), dict(K=32),
            dict(K=96), dict(K=-64), dict(eps=-1e-6), dict(eps=float("inf")), dict(eps=NAN)]


def _call(lib, a, name, stream):
    def p(k):
        return ctypes.c_void_p(a[k] and a[k] + a.get(k + "_off", 0))
    return lib.edv_op_linear_residual_ln(a["dtype"], p("A"), p("W"), ctypes.c_void_p(a["bias"]), p("x"),
                                         ctypes.c_void_p(a["gamma"]), ctypes.c_void_p(a["beta"]), ctypes.c_float(a["eps"]),
                                         p("xn"), a["M"], a["N"], a["K"], ctypes.c_void_p(0), name, 64, stream)


def test_gemm_ln_rejects_bad_arguments():
    """edv_op_linear_residual_ln returns EDV_ERR_ARG with a message, before any launch, for each argument it cannot run.
    The pointers are fake, so this runs only where there is no device: a check that went missing fails with
    EDV_ERR_CUDA instead."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = eng.load_library()
    ok = dict(dtype=eng.EDV_BF16, A=1 << 20, W=2 << 20, bias=3 << 20, x=4 << 20, gamma=5 << 20, beta=6 << 20, xn=7 << 20,
              M=256, N=384, K=384, eps=EPS)
    name = ctypes.create_string_buffer(64)
    for bad in BAD_ARGS:
        name.value = b"stale"
        rc = _call(lib, dict(ok, **bad), name, ctypes.c_void_p(0))
        assert rc == -1, (bad, rc)                                  # EDV_ERR_ARG
        assert b"edv_op_linear_residual_ln" in (lib.edv_last_error(ctypes.c_void_p(0)) or b""), bad
        assert name.value == b"", (bad, name.value)                # no kernel ran


@pytest.mark.gpu
def test_gemm_ln_rejections_leave_the_buffers_untouched():
    """The same rejections with real buffers on the device: nothing is launched, x keeps its bits and the NaN xn stays
    NaN; the valid call then runs and writes every row."""
    lib = eng.load_library()
    M = 256
    A, W, b, x0, gam, bet = _make_inputs(M, 384, torch.bfloat16, "forward", 800)
    xbuf, x, xnbuf, xn = _guarded(M, x0, torch.bfloat16, True)
    before = xbuf.clone()
    ok = dict(dtype=eng.EDV_BF16, A=A.data_ptr(), W=W.data_ptr(), bias=b.data_ptr(), x=x.data_ptr(), gamma=gam.data_ptr(),
              beta=bet.data_ptr(), xn=xn.data_ptr(), M=M, N=384, K=384, eps=EPS)
    name = ctypes.create_string_buffer(64)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for bad in BAD_ARGS:
        name.value = b"stale"
        assert _call(lib, dict(ok, **bad), name, stream) == -1, bad
        assert name.value == b"", (bad, name.value)
    torch.cuda.synchronize()
    assert torch.equal(xbuf, before), "a rejected call wrote x"
    assert bool(xnbuf.isnan().all()), "a rejected call wrote xn"
    assert _call(lib, ok, name, stream) == 0
    torch.cuda.synchronize()
    assert name.value == b"gemm_ln<bf16>", name.value
    _check_guards(xbuf, x, xnbuf, xn, M)
    _check(x, xn, A, W, b, x0, gam, bet, "after the rejections", "forward")


# ---- the bound itself, without a GPU -----------------------------------------------------------------------------------
# (M, K, npairs): 7 tiles on 2 pairs (4 and 3 tiles, the last partial) and 9 tiles on 3 pairs (3 each, the last
# partial): every pair reaches its third tile, where the mailbox of its first tile is reused
MODEL_SHAPES = [(859, 128, 2), (1100, 64, 3)]


@pytest.mark.parametrize("dtype", DT16, ids=_dt_id)
def test_gemm_ln_bound_rejects_known_bugs(dtype):
    """On the CPU: on small multi-tile shapes of every family, the model of the epilogue (_model) passes the fp32 part
    of the xn bound (the statistics, Chan's combination, rsqrtf and the normalisation, before the 16-bit rounding)
    within 0.5, and the x bound and the whole xn bound within 1.  (Those two end in roundings whose error alone can
    reach almost their whole term: u |b + x0| + u |x^| where A W^T is small against x, u16 |xn|.)  Each known bug
    injected into the model exceeds the bounds at least tenfold on every family it applies to."""
    worst = {}
    for M, K, npairs in MODEL_SHAPES:
        assert _tiles(M) > 2 * npairs
        for family in FAMILIES:
            A, W, b, x0, gam, bet = _make_inputs(M, K, dtype, family, 900 + FAMILIES.index(family), device="cpu")
            xref, xbound = None, None

            def excess(bug):
                """(fp32 xn against its bound, x and xn against theirs)"""
                nonlocal xref, xbound
                xh, xn, y32 = _model(A, W, b, x0, gam, bet, dtype, npairs, bug)
                if xref is None:
                    xref, xbound = _x_reference(A, W, b, x0, xh)
                ex = _excess((xh.double() - xref).abs(), xbound)
                ref, bound, bound32 = _ln_reference(xh, gam, bet, dtype)
                return _excess((y32.double() - ref).abs(), bound32), max(ex, _excess((xn.double() - ref).abs(), bound))

            frac32, frac = excess(None)
            for k, f in (("model fp32 ", frac32), ("model ", frac)):
                worst[k + family] = max(worst.get(k + family, 0.0), f)
            assert frac32 <= 0.5 and frac <= 1.0, (family, M, frac32, frac)
            for bug in BUGS:
                if family in APPLIES[bug]:
                    frac = excess(bug)[1]
                    worst[bug] = min(worst.get(bug, math.inf), frac)
                    assert frac >= 10.0, (bug, family, M, frac)
    print("\n%s: the model reaches, of the bound (fp32 xn; x and xn):" % _dt_id(dtype))
    for family in FAMILIES:
        print("  %-26s %.3f  %.3f" % (family, worst["model fp32 " + family], worst["model " + family]))
    print("each bug at least:")
    for bug in BUGS:
        print("  %-26s %.3g x the bound" % (bug, worst[bug]))
