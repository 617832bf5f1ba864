"""End-to-end parity of the CUDA path (through the drop-in class -> ctypes -> C ABI) on a B200.

Gates (BASELINE.json north_star), all against golden vectors written by the UNMODIFIED
reference (tests/golden, oracle/make_golden.py):
  * fp32 path:  |ours - ref| <= 2e-4 * max(|ref|, 1);
  * fp16 tensor-core path (the default): per-pixel relative disparity error <= 1e-2,
    AbsRel <= 1e-3 and delta<1.25 >= 0.999 with the reference output as ground truth
    (utils/utils.py:112-133);
  * bf16 tensor-core path: 8-bit mantissas cannot meet 1e-2 on these synthetic weights -- the
    CPU oracle with ONLY its contraction operands rounded to bf16 (fp32 everything else) is
    already 1.5-2.4 % of the mean disparity off per pixel and 3e-3 AbsRel (DESIGN.md, accuracy
    table) -- so bf16 is held to that operand-rounding floor, measured per case in the test:
    <= max(2e-2, 2.5 x floor) per pixel (never above 8e-2), AbsRel <= 1e-2, delta<1.25 >= 0.999.
The relative error's denominator is floored at half the clip's mean disparity, and AbsRel / delta
are taken over pixels above a quarter of the mean: pixels sitting on the final ReLU's kink
(reference disparity ~ 0, several golden cases have them) have no meaningful relative error.
/root/reference is never read here."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import endodav_b200 as E  # noqa: E402
from oracle import endodav_oracle as orc  # noqa: E402
from oracle import weights  # noqa: E402
from golden_util import load_case, manifest, oracle_cfg, subsample_like_golden  # noqa: E402

FP32_RTOL = 2e-4
GATES = {"fp16": dict(rel=1e-2, absrel=1e-3, a1=0.999), "bf16": dict(rel=6e-2, absrel=1e-2, a1=0.999)}


def _rel(got, ref):
    return np.abs(got - ref) / np.maximum(np.abs(ref), 0.5 * float(np.abs(ref).mean()))


def _report_16bit(name, dtype, rel, absrel, a1, gate):
    """Measured margins of every golden case, brought back in gpurun_out/ for DESIGN.md."""
    import json
    import os
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "golden_16bit_margins.json")
    try:
        os.makedirs(os.path.dirname(path), exist_ok=True)
        data = json.load(open(path)) if os.path.exists(path) else {}
        data["%s.%s" % (name, dtype)] = dict(rel_max=rel, absrel=absrel, a1=a1, gate=gate)
        json.dump(data, open(path, "w"), indent=1, sort_keys=True)
    except OSError:
        pass


def _build(ctor, seed, dtype):
    kw = dict(ctor)
    kw["image_shape"] = tuple(kw["image_shape"])
    model = E.endodav(dtype=dtype, **kw)
    cfg = oracle_cfg(ctor)
    sd = weights.make_state_dict(cfg, seed)
    model.load_state_dict(sd, strict=True)
    return model.cuda().eval(), cfg, sd


def _metrics(pred, gt):
    """compute_errors (utils/utils.py:112-133) with the reference output as gt."""
    pred, gt = pred.astype(np.float64).ravel(), gt.astype(np.float64).ravel()
    m = gt > 0.25 * gt.mean()   # the eval scripts mask invalid (near-zero) ground truth the same way
    pred, gt = np.maximum(pred[m], 1e-9), gt[m]
    thresh = np.maximum(gt / pred, pred / gt)
    return float(np.mean(np.abs(gt - pred) / gt)), float((thresh < 1.25).mean())


FWD = [k for k, v in manifest().items() if v["kind"] == "forward"]   # includes the pe='rope' configuration


@pytest.mark.parametrize("name", FWD)
def test_forward_fp32_matches_reference_golden(name):
    m, arrays = load_case(name)
    model, cfg, sd = _build(m["ctor"], m["weight_seed"], "fp32")
    B, T, H, W = m["input"]
    x = weights.make_frames(B, T, H, W, m["frame_seed"]).cuda()
    out = model(x)
    assert model._eng.launch_count() > 0
    for s in range(4):
        got = subsample_like_golden(name, s, out[("disp", s)].cpu().numpy())
        ref = arrays["disp%d" % s]
        assert got.shape == ref.shape
        err = np.abs(got - ref) / np.maximum(np.abs(ref), 1.0)
        assert err.max() <= FP32_RTOL, (name, s, float(err.max()))


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("name", FWD)
def test_forward_16bit_within_tolerance(name, dtype):
    _check_16bit(name, dtype)


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("name", ["fwd_vits_lora_res_convhead", "fwd_vits_rope"])
def test_forward_16bit_cuda_core_engine_within_tolerance(name, dtype, monkeypatch):
    """The same gates on the CUDA-core 16-bit engine (ENDODAV_ENGINE=simt), the only product path that runs
    geglu_pair, head_dot and the unfused disparity head in 16 bits."""
    monkeypatch.setenv("ENDODAV_ENGINE", "simt")
    _check_16bit(name, dtype, "simt")


def _check_16bit(name, dtype, engine="tc"):
    m, arrays = load_case(name)
    model, cfg, sd = _build(m["ctor"], m["weight_seed"], dtype)
    B, T, H, W = m["input"]
    x = weights.make_frames(B, T, H, W, m["frame_seed"]).cuda()
    out = model(x)
    got = subsample_like_golden(name, 0, out[("disp", 0)].cpu().numpy())
    ref = arrays["disp0"]
    gate = dict(GATES[dtype])
    if dtype == "bf16":
        # bf16 is held to its operand-rounding floor, measured on THIS case: the fp32 oracle with only its contraction
        # operands rounded to bf16 (everything else fp32).  The CUDA path may be at most 2.5x that floor (and never
        # above the absolute 8e-2); which rounding realisation hits the worst pixel next to the ReLU kink is chance.
        with torch.no_grad():
            emu = orc.forward(sd, x.cpu(), cfg, tuple(m["ctor"]["image_shape"]), emulate_bf16=True)[("disp", 0)].numpy()
        floor = float(_rel(subsample_like_golden(name, 0, emu), ref).max())
        gate["rel"] = min(8e-2, max(2e-2, 2.5 * floor))
    rel = _rel(got, ref)
    absrel, a1 = _metrics(got, ref)
    assert rel.max() <= gate["rel"], (name, dtype, float(rel.max()))
    assert absrel <= gate["absrel"] and a1 >= gate["a1"], (name, dtype, absrel, a1)
    for s in range(1, 4):
        g = subsample_like_golden(name, s, out[("disp", s)].cpu().numpy())
        r = arrays["disp%d" % s]
        assert _rel(g, r).max() <= gate["rel"], (name, dtype, s)
    _report_16bit(name, dtype if engine == "tc" else dtype + "." + engine, float(rel.max()), absrel, a1, gate["rel"])


def test_stage_taps_fp32_match_oracle():
    """Every intermediate the engine can snapshot agrees with the oracle's record (fp32)."""
    m, _ = load_case("fwd_vits_dvlora")
    model, cfg, sd = _build(m["ctor"], m["weight_seed"], "fp32")
    B, T, H, W = m["input"]
    x = weights.make_frames(B, T, H, W, m["frame_seed"])
    rec = {}
    orc.forward(sd, x, cfg, tuple(m["ctor"]["image_shape"]), record=rec)
    h, w = m["ctor"]["image_shape"]
    eng = model._ensure_engine(h // 14, w // 14)
    eng.set_debug(True)
    model(x.cuda())
    for name, ref in rec.items():
        got = eng.debug_tap(name).cpu()
        if ref.dim() == 4:  # oracle keeps NCHW, the engine NHWC rows
            ref = ref.permute(0, 2, 3, 1)
        ref = ref.reshape(-1, ref.shape[-1])
        assert tuple(got.shape) == tuple(ref.shape), (name, got.shape, ref.shape)
        err = float((got - ref).abs().max())
        assert err <= 3e-4 * max(1.0, float(ref.abs().max())), (name, err)


def test_forward_is_deterministic_and_replans():
    m, _ = load_case("fwd_vits_b2")
    model, cfg, sd = _build(m["ctor"], m["weight_seed"], "fp16")
    x = weights.make_frames(2, 3, 56, 56, 3).cuda()
    a = model(x)[("disp", 0)].clone()
    y = weights.make_frames(1, 2, 40, 60, 4).cuda()     # different B,T,H,W -> re-plan
    model(y)
    b = model(x)[("disp", 0)]
    assert torch.equal(a, b)


def test_weight_update_is_repacked():
    """nn.Module protocol: loading new weights after a forward must change the output."""
    m, _ = load_case("fwd_vits_b2")
    model, cfg, sd = _build(m["ctor"], m["weight_seed"], "fp16")
    x = weights.make_frames(1, 2, 56, 56, 3).cuda()
    a = model(x)[("disp", 0)].clone()
    model.load_state_dict(weights.make_state_dict(cfg, 999))
    b = model(x)[("disp", 0)]
    assert not torch.equal(a, b)


def test_frame_order_matters():
    """Temporal modules must see the frame axis: permuting frames changes per-frame outputs."""
    m, _ = load_case("fwd_vits_dvlora")
    model, cfg, sd = _build(m["ctor"], m["weight_seed"], "fp32")
    x = weights.make_frames(1, 4, 70, 98, 5).cuda()
    a = model(x)[("disp", 0)]
    b = model(x[:, [1, 0, 2, 3]])[("disp", 0)]
    assert float((a[0] - b[1]).abs().max()) > 1e-5


@pytest.mark.parametrize("n_case", ["video_n5", "video_n45"])
def test_infer_video_depth_matches_reference_golden(n_case):
    m, arrays = load_case(n_case)
    model, cfg, sd = _build(m["ctor"], m["weight_seed"], "fp32")
    N, H, W = m["input"]
    v = weights.make_video_u8(N, H, W, m["frame_seed"])
    got = model.infer_video_depth(v)
    assert got.dtype == np.float32 and got.shape == arrays["depth"].shape
    err = np.abs(got - arrays["depth"]) / np.maximum(np.abs(arrays["depth"]), 1.0)
    assert err.max() <= 5e-4, float(err.max())


def test_vitl_full_size_clip_runs():
    """BASELINE config 4 shape family (ViT-L, 518 x 518, T=32; one clip): finite, non-degenerate, deterministic.
    (Parity at full size against the oracle is in tests/test_gpu_fullsize.py: ViT-S 32 x 518 x 518 and ViT-L 2 x 518 x 518.)"""
    ctor = dict(encoder="vitl", features=256, out_channels=[256, 512, 1024, 1024], r=4, lora_type="dvlora",
                image_shape=(518, 518), disable_conv_head=True, residual_block_indexes=[])
    model, cfg, sd = _build(ctor, 61, "fp16")
    x = weights.make_frames(1, 32, 518, 518, 62).cuda()
    d0 = model(x)[("disp", 0)]
    assert tuple(d0.shape) == (32, 1, 518, 518)
    assert bool(torch.isfinite(d0).all()) and float(d0.std()) > 1e-4
    assert torch.equal(d0, model(x)[("disp", 0)])


def test_clip_batch_sweep_matches_single_clips():
    """BASELINE config 5 (Hamlyn-shaped clip batches at 256 x 320, network 224 x 280): a batch of B clips must
    equal the B clips run one by one (no cross-clip leakage in the temporal modules), for T in {8, 16}."""
    ctor = dict(encoder="vits", features=64, out_channels=[48, 96, 192, 384], r=4, lora_type="dvlora",
                image_shape=(224, 280), disable_conv_head=True, residual_block_indexes=[])
    model, cfg, sd = _build(ctor, 1234, "fp16")
    for T in (8, 16):
        x = weights.make_frames(3, T, 256, 320, 70 + T).cuda()
        full = model(x)[("disp", 0)].clone()
        for b in range(3):
            one = model(x[b:b + 1])[("disp", 0)]
            assert torch.equal(full[b * T:(b + 1) * T], one), (T, b)


def test_long_video_scared_shape():
    """BASELINE config 3 shape (256 x 320 frames, network 224 x 280, 32-frame windows with stride 22):
    4 windows; output shape / dtype, finiteness, and that the first window's frames are untouched by
    the stitching (they are the raw network output resized to the frame size)."""
    ctor = dict(encoder="vits", features=64, out_channels=[48, 96, 192, 384], r=4, lora_type="dvlora",
                image_shape=(224, 280), disable_conv_head=True, residual_block_indexes=[])
    model, cfg, sd = _build(ctor, 1234, "fp16")
    v = weights.make_video_u8(80, 256, 320, 9)
    out = model.infer_video_depth(v)
    assert out.shape == (80, 256, 320) and out.dtype == np.float32 and np.isfinite(out).all()
    first = model.infer_video_depth(v[:32])
    assert np.array_equal(out[:22], first[:22])


def test_gpu_preprocessing_equals_host_preprocessing(monkeypatch):
    """SURVEY.md 8(f)-1: the driver's default GPU cubic resize must reproduce the reference's host
    (cv2) preprocessing path end to end."""
    m, arrays = load_case("video_n45")
    model, cfg, sd = _build(m["ctor"], m["weight_seed"], "fp32")
    N, H, W = m["input"]
    v = weights.make_video_u8(N, H, W, m["frame_seed"])
    a = model.infer_video_depth(v)
    monkeypatch.setenv("ENDODAV_PREPROCESS", "host")
    b = model.infer_video_depth(v)
    assert float(np.abs(a - b).max()) <= 1e-4 * max(1.0, float(np.abs(b).max()))


def test_cuda_graph_replay_on_default_stream_is_bit_identical():
    """edv_forward captures the planned launch sequence (on its private capture stream, so torch's legacy default
    stream works too) and replays it: same bits as eager launches, one graph per pointer set, and the graph sees
    new input VALUES written into the same buffers."""
    m, _ = load_case("fwd_vits_dvlora")
    model, cfg, sd = _build(m["ctor"], m["weight_seed"], "fp16")
    B, T, H, W = m["input"]
    x = weights.make_frames(B, T, H, W, m["frame_seed"]).cuda()
    h, w = m["ctor"]["image_shape"]
    eng = model._ensure_engine(h // 14, w // 14)
    def pyramid(inp):   # all four levels: a replay hands them over with one copy_pyramid_kernel launch
        o = model(inp)
        return [o[("disp", s)].clone() for s in range(4)]

    eng.set_graph_mode(False)
    eager = pyramid(x)
    assert eng.graph_count() == 0
    eng.set_graph_mode(True)
    outs = [pyramid(x) for _ in range(4)]
    assert eng.graph_count() >= 1, eng.graph_status()
    assert eng.graph_status() == "ok"
    for o in outs:
        for s in range(4):
            assert torch.equal(o[s], eager[s]), s
    x2 = weights.make_frames(B, T, H, W, m["frame_seed"] + 1).cuda()
    eng.set_graph_mode(False)
    eager2 = pyramid(x2)
    eng.set_graph_mode(True)
    model(x)
    x.copy_(x2)           # same pointer, new values
    for _ in range(3):
        got2 = pyramid(x)
    assert eng.graph_count() >= 1
    for s in range(4):
        assert torch.equal(got2[s], eager2[s]), s
    assert not torch.equal(got2[0], eager[0])
