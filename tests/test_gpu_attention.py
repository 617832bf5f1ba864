"""Spatial self-attention (edv_op_attention: flash_attention_tc_kernel and spatial_attention_simt_kernel) at the forward's
shapes, against a float64 reference.

The tcgen05 kernel is persistent: one CTA per SM walks (frame, head, 256-query) work items, and its Q double buffer, K|V
ring, barrier phases and per-item softmax state carry across item boundaries.  So the shapes here include launches with
more than 4 x SM-count items, and each frame of such a launch must equal, bit for bit, the same frame launched alone or
next to different neighbours.  Inputs built on purpose reach the lazy O rescale (row maxima growing by more than 8 ln2
per key block on half the rows of every warp, growth just below that, a dominant key first or in the partial last
block), and a poisoned next frame makes any key that leaks through the mask past S dominate the output.

Operands are rounded to the dtype first; the reference is float64 softmax(q k^T) v on those operands (q is pre-scaled
at pack time, the kernels apply no scale).  qkv is a view followed in the same allocation by NaN rows, and outputs go to
NaN-filled buffers whose guard rows must stay NaN.  Every case asserts which kernel ran.

Tolerance, per element: |got - ref| <= SLACK * u * (sum_j p_j |v_j| + |ref|), the error model of the kernels (_u):
a relative error on each weight p_j moves the output by at most that much of sum_j p_j |v_j - ref|, and a relative
error on the output (O / l rounded, or l summed) by that much of |ref|.  test_attention_bound_rejects_known_bugs
(no GPU) applies the same bound to a CPU model of the tcgen05 algorithm, which must pass, and to known bugs, which
must fail."""
import ctypes
import math

import pytest
import torch

from endodav_b200 import engine as eng

DEV = "cuda"
HD = 64
GUARD = 136                  # NaN rows after qkv and after every output (more than one 128-row TMA box)
NAN = float("nan")
SLACK = 2.0
LOG2E = 1.4426950408889634
TC, SIMT = eng.ENGINE_TC, eng.ENGINE_SIMT
# (dtype, engine): 16-bit on the tcgen05 kernel, every dtype on the CUDA-core kernel, and float32 with ENGINE_TC (no
# fp32 tensor-core kernel exists, so it runs the CUDA-core one)
CASES = [(torch.bfloat16, TC), (torch.float16, TC), (torch.float32, SIMT), (torch.bfloat16, SIMT), (torch.float16, SIMT),
         (torch.float32, TC)]
TC_CASES = CASES[:2]


def _case_id(c):
    return "%s-%s" % (str(c[0]).replace("torch.", ""), "tc" if c[1] == TC else "simt")


def _expected_kernel(dtype, engine):
    t = {torch.float32: "f32", torch.bfloat16: "bf16", torch.float16: "f16"}[dtype]
    return ("flash_attention_tc<%s>" if dtype != torch.float32 and engine == TC else "spatial_attention_simt<%s>") % t


def _items(F, S, heads):
    """Work items of flash_attention_tc_kernel: 256 queries of one (frame, head)."""
    return F * heads * -(-S // 256)


# ---- error model -------------------------------------------------------------------------------------------------------
def _u(dtype, S, qkv=None, heads=None):
    """Unit of the error model.  16-bit: P is rounded to the dtype before P V (tcgen05 kernel) and O / l is rounded to the
    dtype on the way out (both kernels): u = 2^-8 (bf16), 2^-11 (f16).

    float32 (spatial_attention_simt, fp32 math, u32 = 2^-24), every term relative to one p_j or to a sum of them:
      2 S       acc = sum_j p_j v_j and l = sum_j p_j are sequential fp32 sums over the S keys, (S - 1) u32 each
      64 A      each score is a 64-term fp32 dot product, off by at most 64 u32 sum_d |q_d k_d| <= 64 u32 |q| |k|;
                A = max |q| * max |k| over the launch (Cauchy-Schwarz), a relative error of exp(score)
      34 / tile __expf(x) = ex2.approx(x log2 e): 2 ulp, plus the rounding of x log2 e, <= 32 u32 for every key with a
                weight above e^-32 (the others weigh nothing in fp32); once for each p_j, and the running-max correction
                of each 32-key tile multiplies every earlier weight once more."""
    if dtype == torch.bfloat16:
        return 2.0 ** -8
    if dtype == torch.float16:
        return 2.0 ** -11
    D = heads * HD
    qn = qkv[:, :D].double().reshape(-1, heads, HD).norm(dim=-1).max()
    kn = qkv[:, D:2 * D].double().reshape(-1, heads, HD).norm(dim=-1).max()
    return 2.0 ** -24 * (2 * S + 64 * float(qn * kn) + 34 * (S // 32 + 1))


def _bound(ref, scl, u, slack=SLACK):
    return slack * u * (scl + ref.abs())


def _frac(got, ref, scl, u):
    """Worst |got - ref| / bound (inf where got is NaN)."""
    err = (got.double() - ref).abs().nan_to_num(float("inf"))
    return float((err / _bound(ref, scl, u)).max())


def _softmax_pv(q, k, v):
    """float64 (softmax(q k^T) v, softmax(q k^T) |v|) over the last two dims."""
    p = (q.double() @ k.double().transpose(-1, -2)).softmax(-1)
    return p @ v.double(), p @ v.double().abs()


def _reference(qkv, F, S, heads):
    """float64 (ref, scale) [F*S, heads*64], a few frames at a time: one (frame, head) at S = 1370 is a 15 MB float64
    matrix."""
    D = heads * HD
    ref = torch.empty(F * S, D, dtype=torch.float64, device=qkv.device)
    scl = torch.empty_like(ref)
    step = max(1, (1 << 28) // (heads * S * S * 8))
    for f0 in range(0, F, step):
        n = min(step, F - f0)
        t = qkv[f0 * S:(f0 + n) * S].view(n, S, 3, heads, HD).permute(2, 0, 3, 1, 4)
        o, s = _softmax_pv(t[0], t[1], t[2])                       # [n, heads, S, 64]
        ref[f0 * S:(f0 + n) * S] = o.transpose(1, 2).reshape(n * S, D)
        scl[f0 * S:(f0 + n) * S] = s.transpose(1, 2).reshape(n * S, D)
    return ref, scl


# ---- inputs ------------------------------------------------------------------------------------------------------------
def _qkv_buf(F, S, heads, dtype, device):
    """(buffer, view): the view is qkv [F*S, 3*heads*64], followed in the same allocation by GUARD NaN rows."""
    buf = torch.full((F * S + GUARD, 3 * heads * HD), NAN, dtype=dtype, device=device)
    return buf, buf[:F * S]


def _randn(shape, seed, scale, device):
    g = torch.Generator(device=device).manual_seed(seed)
    return torch.randn(shape, generator=g, device=device) * scale


def _make_qkv(F, S, heads, dtype, seed, kind="random", device=DEV):
    """qkv rounded to dtype.  kind:
      random       N(0, 0.5^2)
      poison       even frames' queries get q[0] = 1, odd frames' keys k[0] = 32: the keys of frame f+1 score about 30
                   above frame f's own keys against frame f's queries; every frame's own logits stay N(0, 2^2)
      ramp_grow    q[i, 0] = 1 on odd rows, 0 on even rows; k[j, 0] = j / 16: on odd rows the row max grows by 8 per
                   128-key block (> 8 ln2 = 5.55, the lazy-rescale threshold), on even rows it does not -- every warp
                   rescales O with mixed `grow`
      ramp_below   the same ramp at 5 per block: just below the threshold, P reaches e^5 ~ 2^7.2 between rescales
      peak_first   key 0 scores 12 above the others: the first block's max holds for the whole row
      peak_last    key S-1 (in the partial last block) scores 12 above the others: O is rescaled at the last block"""
    D = heads * HD
    scale = 0.25 if kind.startswith(("ramp", "peak")) else 0.5
    x = _randn((F, S, 3, heads, HD), seed, scale, device)
    q, k = x[:, :, 0, :, 0], x[:, :, 1, :, 0]
    if kind == "poison":
        q[0::2], k[0::2] = 1.0, 0.0
        q[1::2], k[1::2] = 0.0, 32.0
    elif kind.startswith("ramp"):
        q[:] = 0.0
        q[:, 1::2] = 1.0 if kind == "ramp_grow" else 5.0 / 8.0
        k[:] = (torch.arange(S, device=device, dtype=torch.float32) / 16.0).view(1, S, 1)
    elif kind.startswith("peak"):
        q[:] = 1.0
        k[:] = 0.0
        k[:, 0 if kind == "peak_first" else S - 1] = 12.0
    buf, view = _qkv_buf(F, S, heads, dtype, device)
    view.copy_(x.view(F * S, 3 * D).to(dtype))
    return buf, view


# ---- CPU model of flash_attention_tc_kernel ----------------------------------------------------------------------------
def _emulate_tc(qkv, F, S, heads, dtype, mask=True, rescale=True):
    """float64 [F*S, D] output of the tcgen05 algorithm, and statistics of the paths it took.  128-key blocks; scores in
    fp32 (exact 16-bit products summed in fp32); lazy max: the reference max moves only when the block max exceeds it by
    more than 8 ln2, then l and O are multiplied by exp(old - new); l sums the unrounded p, O += P V with P rounded to the
    dtype; out = O / l rounded to the dtype.  Keys past S are the next frame's rows (TMA zero fill after the last frame),
    removed by the mask.  mask / rescale False model the two bugs the tolerance must catch."""
    D = heads * HD
    pad = (-S) % 128
    rows = torch.cat([qkv.float(), torch.zeros(pad, 3 * D)])
    out = torch.empty(F * S, D, dtype=torch.float64)
    st = {"grow_rows": 0, "mixed_warps": 0, "pmax": 0.0}
    nw = S // 32                                                  # complete 32-row warps of each frame
    for f in range(F):
        for h in range(heads):
            c = h * HD
            q = rows[f * S:(f + 1) * S, c:c + HD]
            k = rows[f * S:(f + 1) * S + pad, D + c:D + c + HD]
            v = rows[f * S:(f + 1) * S + pad, 2 * D + c:2 * D + c + HD]
            s = q @ k.t()
            m = torch.full((S, 1), -math.inf)
            l = torch.zeros(S, 1)
            O = torch.zeros(S, HD)
            for j0 in range(0, S, 128):
                sb = s[:, j0:j0 + 128].clone()
                if mask:
                    sb[:, S - j0:] = -math.inf
                mx = sb.max(-1, keepdim=True).values
                grow = mx > m + 8.0 / LOG2E
                if j0 > 0:
                    g = grow[:nw * 32].view(nw, 32)
                    st["grow_rows"] += int(g.sum())
                    st["mixed_warps"] += int((g.any(1) & ~g.all(1)).sum())
                factor = torch.where(grow, torch.exp(m - mx), torch.ones_like(m)) if rescale else torch.ones_like(m)
                m = torch.where(grow, mx, m)
                l, O = l * factor, O * factor
                p = torch.exp(sb - m)
                st["pmax"] = max(st["pmax"], float(p.max()))
                l = l + p.sum(-1, keepdim=True)
                O = O + p.to(dtype).float() @ v[j0:j0 + 128]
            out[f * S:(f + 1) * S, c:c + HD] = (O * (1.0 / l)).to(dtype).double()
    return out, st


# ---- harness -----------------------------------------------------------------------------------------------------------
WORST = {}   # case -> worst error as a fraction of its bound (printed at the end of the module)


def _note(name, frac):
    WORST[name] = max(WORST.get(name, 0.0), frac)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        print("\nworst error / bound per case:")
        for k in sorted(WORST):
            print("  %-36s %.3f" % (k, WORST[k]))


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _run(qkv, F, S, heads, dtype, engine):
    """Launch into a NaN-filled buffer; asserts the kernel and the guard rows; returns the [F*S, D] output."""
    buf = torch.full((F * S + GUARD, heads * HD), NAN, dtype=dtype, device=DEV)
    _, kernel = eng.op_attention_kernel(qkv, F, S, heads, engine, out=buf)
    torch.cuda.synchronize()
    assert kernel == _expected_kernel(dtype, engine), kernel
    assert bool(buf[F * S:].float().isnan().all()), "guard rows beyond the output were written"
    return buf[:F * S]


def _check(got, qkv, F, S, heads, dtype, what, case):
    ref, scl = _reference(qkv, F, S, heads)
    u = _u(dtype, S, qkv, heads)
    err = (got.double() - ref).abs()
    bound = _bound(ref, scl, u)
    bad = ~(err <= bound)
    if bool(bad.any()):
        i = int(torch.argmax((err.nan_to_num(float("inf")) / bound).flatten()))
        r, col = divmod(i, heads * HD)
        raise AssertionError("%s: %d / %d over the bound; worst at frame %d row %d head %d dim %d: got %r ref %.6g bound %.3g"
                             % (what, int(bad.sum()), bad.numel(), r // S, r % S, col // HD, col % HD,
                                float(got[r, col]), float(ref[r, col]), float(bound[r, col])))
    _note(case, float((err / bound).max()))


# ---- the forward's shapes ----------------------------------------------------------------------------------------------
# (BT, N, heads): ViT-S / ViT-B / ViT-L (6 / 12 / 16 heads) at 518 x 518 (N = 1370 with the class token, 1369 without)
# and 224 x 280 (N = 321 / 320); MULTI shapes run more than 4 x SM-count work items on the tcgen05 kernel
MULTI = [(32, 1370, 6), (8, 1370, 16)]
FWD_SHAPES = MULTI + [(4, 1369, 12), (32, 321, 16), (6, 320, 6), (3, 1369, 16), (5, 321, 12)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
@pytest.mark.parametrize("BT,N,heads", FWD_SHAPES)
def test_attention_forward_shapes(BT, N, heads, case):
    dtype, engine = case
    if (BT, N, heads) in MULTI and engine == TC and dtype != torch.float32:
        assert _items(BT, N, heads) > 4 * _sms(), "%d work items" % _items(BT, N, heads)
    _, qkv = _make_qkv(BT, N, heads, dtype, 100 + N + heads)
    got = _run(qkv, BT, N, heads, dtype, engine)
    _check(got, qkv, BT, N, heads, dtype, "attention %s %dx%dx%d" % (_case_id(case), BT, N, heads), "shapes " + _case_id(case))


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
@pytest.mark.parametrize("S", [1, 2, 127, 128, 129, 255, 256, 257, 384, 385])
def test_attention_tails(S, case):
    """A tile-A-only item (S % 256 <= 128), one valid key in the last block (S % 128 == 1), exactly full blocks."""
    dtype, engine = case
    F, heads = 3, 2
    _, qkv = _make_qkv(F, S, heads, dtype, 200 + S)
    got = _run(qkv, F, S, heads, dtype, engine)
    _check(got, qkv, F, S, heads, dtype, "attention tail S=%d %s" % (S, _case_id(case)), "tails " + _case_id(case))


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES[:5], ids=_case_id)
@pytest.mark.parametrize("BT,N,heads", MULTI)
def test_attention_frames_are_independent(BT, N, heads, case):
    """A row's arithmetic does not depend on which CTA runs its item or what ran before it there: frames 0, BT/2 and
    BT-1 of the multi-frame launch equal, bit for bit, the same frame launched alone, and the same frames in a launch
    whose every other frame holds different values."""
    dtype, engine = case
    if engine == TC:
        assert _items(BT, N, heads) > 4 * _sms()
    buf, qkv = _make_qkv(BT, N, heads, dtype, 300 + heads)
    full = _run(qkv, BT, N, heads, dtype, engine).clone()
    keep = (0, BT // 2, BT - 1)
    for f in keep:
        alone = _run(qkv[f * N:(f + 1) * N], 1, N, heads, dtype, engine)
        assert torch.equal(alone, full[f * N:(f + 1) * N]), "frame %d differs when launched alone" % f
    _, other = _make_qkv(BT, N, heads, dtype, 301 + heads)
    for f in keep:
        other[f * N:(f + 1) * N] = qkv[f * N:(f + 1) * N]
    mixed = _run(other, BT, N, heads, dtype, engine)
    for f in keep:
        assert torch.equal(mixed[f * N:(f + 1) * N], full[f * N:(f + 1) * N]), "frame %d depends on the other frames" % f
    _note("independent " + _case_id(case), 0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
@pytest.mark.parametrize("F,S,heads", [(8, 1369, 6), (5, 321, 2)])
def test_attention_poisoned_neighbour(F, S, heads, case):
    """The last key block of frame f holds frame f+1's first keys, which score ~30 above frame f's own keys: any that
    leaks through the key mask dominates frame f's output (F odd: the last frame's tail is zero fill, then NaN rows)."""
    dtype, engine = case
    _, qkv = _make_qkv(F, S, heads, dtype, 400 + S, "poison")
    got = _run(qkv, F, S, heads, dtype, engine)
    _check(got, qkv, F, S, heads, dtype, "poisoned neighbour %dx%dx%d %s" % (F, S, heads, _case_id(case)),
           "poison " + _case_id(case))


RESCALE_KINDS = ["ramp_grow", "ramp_below", "peak_first", "peak_last"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
@pytest.mark.parametrize("kind", RESCALE_KINDS)
def test_attention_lazy_rescale(kind, case):
    """The lazy O rescale in TMEM (see _make_qkv for what each input does), at 11 key blocks, 576 work items."""
    dtype, engine = case
    F, S, heads = 16, 1370, 6
    _, qkv = _make_qkv(F, S, heads, dtype, 500, kind)
    got = _run(qkv, F, S, heads, dtype, engine)
    _check(got, qkv, F, S, heads, dtype, "lazy rescale %s %s" % (kind, _case_id(case)), "rescale %s %s" % (kind, _case_id(case)))


# ---- without a GPU -----------------------------------------------------------------------------------------------------
def test_attention_rejects_bad_arguments():
    """edv_op_attention returns EDV_ERR_ARG, before any launch, for what neither kernel can run.  The pointers are
    fake, so this only runs where there is no device: a check that went missing fails with EDV_ERR_CUDA instead."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = eng.load_library()
    bf16, f32 = eng.EDV_BF16, eng.EDV_F32
    ok = dict(dtype=bf16, engine=TC, qkv=1 << 20, out=2 << 20, F=2, S=321, heads=6)
    bad = [dict(qkv=0), dict(out=0), dict(F=0), dict(S=0), dict(heads=0), dict(S=-5), dict(engine=2), dict(engine=-1),
           dict(dtype=3), dict(qkv=(1 << 20) + 8), dict(out=(2 << 20) + 2),
           dict(engine=SIMT, heads=65536), dict(engine=SIMT, F=65536), dict(dtype=f32, engine=TC, F=65536)]
    name = ctypes.create_string_buffer(64)
    for b in bad:
        a = dict(ok, **b)
        name.value = b"stale"
        rc = lib.edv_op_attention(a["dtype"], a["engine"], ctypes.c_void_p(a["qkv"]), ctypes.c_void_p(a["out"]), a["F"], a["S"],
                                  a["heads"], name, 64, ctypes.c_void_p(0))
        assert rc == -1, (b, rc)                                    # EDV_ERR_ARG
        assert lib.edv_last_error(ctypes.c_void_p(0)), b
        assert name.value == b"", (b, name.value)                  # no kernel ran


# ---- the bound itself, without a GPU ----------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=lambda d: str(d).replace("torch.", ""))
def test_attention_bound_rejects_known_bugs(dtype):
    """On the CPU: the model of the tcgen05 algorithm (_emulate_tc) passes the bound on the inputs the GPU tests use, and
    reaches the paths those inputs are for; a dropped last key, an unmasked poisoned neighbour, query rows shifted by one
    and a skipped O rescale each fail it."""
    u = _u(dtype, 0)
    F, S, heads = 2, 321, 1

    def ref_of(qkv, F, S):
        return _reference(qkv.double(), F, S, heads)

    # random inputs: the model passes; the last key dropped and query rows shifted by one fail
    _, qkv = _make_qkv(F, S, heads, dtype, 7, device="cpu")
    ref, scl = ref_of(qkv, F, S)
    got, _ = _emulate_tc(qkv, F, S, heads, dtype)
    assert _frac(got, ref, scl, u) <= 1.0
    t = qkv.double().view(F, S, 3, HD)
    dropped = torch.cat([_softmax_pv(t[f, :, 0], t[f, :S - 1, 1], t[f, :S - 1, 2])[0] for f in range(F)])
    assert _frac(dropped, ref, scl, u) > 1.0, "dropping the last key passes the bound"
    shifted = torch.cat([ref[f * S:(f + 1) * S].roll(1, 0) for f in range(F)])
    assert _frac(shifted, ref, scl, u) > 1.0, "query rows shifted by one pass the bound"

    # poisoned neighbour: the masked model passes, the unmasked one fails
    _, qkv = _make_qkv(F, S, heads, dtype, 8, "poison", device="cpu")
    ref, scl = ref_of(qkv, F, S)
    assert _frac(_emulate_tc(qkv, F, S, heads, dtype)[0], ref, scl, u) <= 1.0
    assert _frac(_emulate_tc(qkv, F, S, heads, dtype, mask=False)[0], ref, scl, u) > 1.0, "an unmasked tail passes"

    # the rescale inputs at the GPU test's S: the model passes and takes the intended paths; skipping the rescale fails
    F, S = 1, 1370
    for kind in RESCALE_KINDS:
        _, qkv = _make_qkv(F, S, heads, dtype, 500, kind, device="cpu")
        ref, scl = ref_of(qkv, F, S)
        got, st = _emulate_tc(qkv, F, S, heads, dtype)
        assert _frac(got, ref, scl, u) <= 1.0, kind
        warps = S // 32                                              # complete 32-row warps (what the statistics count)
        if kind == "ramp_grow":
            # every warp in every full block after the first (the partial last block grows by only ~5.6)
            assert st["mixed_warps"] >= warps * (S // 128 - 1), st
            assert _frac(_emulate_tc(qkv, F, S, heads, dtype, rescale=False)[0], ref, scl, u) > 1.0, "a skipped rescale passes"
        elif kind == "ramp_below":
            assert st["grow_rows"] > 0 and st["pmax"] > 2.0 ** 7, st
        elif kind == "peak_first":
            assert st["grow_rows"] == 0, st
        else:
            assert st["grow_rows"] == warps * 32, st                 # every row rescales at the last block, nowhere else
