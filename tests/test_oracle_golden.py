"""Pins oracle/ against golden vectors produced by the UNMODIFIED reference
(oracle/make_golden.py) -- SURVEY.md section 8(c).  CPU only."""
import numpy as np
import pytest
import torch

from oracle import endodav_oracle as orc
from oracle import video_oracle as vo
from oracle import weights
from golden_util import assert_video_stub_matches, load_case, manifest, oracle_cfg, subsample_like_golden

FWD = [k for k, v in manifest().items() if v["kind"] == "forward"]
# fp32 CPU: summation order differs between the restatement (merged LoRA, functional ops)
# and the reference's module graph; observed <= 1e-5 absolute on O(1) disparities.
ATOL = 5e-5


@pytest.mark.parametrize("name", FWD)
def test_forward_matches_reference_golden(name):
    m, arrays = load_case(name)
    ctor = m["ctor"]
    cfg = oracle_cfg(ctor)
    sd = weights.make_state_dict(cfg, m["weight_seed"])
    assert len(sd) == m["keys"]
    B, T, H, W = m["input"]
    x = weights.make_frames(B, T, H, W, m["frame_seed"])
    out = orc.forward(sd, x, cfg, tuple(ctor["image_shape"]))
    for s in range(4):
        got = subsample_like_golden(name, s, out[("disp", s)].numpy())
        ref = arrays["disp%d" % s]
        assert got.shape == ref.shape
        assert np.abs(got - ref).max() <= ATOL, (name, s, float(np.abs(got - ref).max()))
    assert float(np.abs(arrays["disp0"]).mean()) > 0.05  # not the degenerate all-zero output


FULL = [k for k, v in manifest().items() if v["kind"] == "forward_full"]


@pytest.mark.parametrize("name", FULL)
def test_forward_full_size_matches_reference_golden(name):
    """BASELINE configs 2 and 4 at their real resolution (S = 1370 tokens, 37x37 -> 19x19 maps, T = 32 for ViT-S):
    the oracle against a strided sample of the UNMODIFIED reference's output (oracle/make_golden.py FULL_CASES)."""
    m, arrays = load_case(name)
    ctor = m["ctor"]
    cfg = oracle_cfg(ctor)
    sd = weights.make_state_dict(cfg, m["weight_seed"])
    B, T, H, W = m["input"]
    x = weights.make_frames(B, T, H, W, m["frame_seed"])
    with torch.no_grad():
        out = orc.forward(sd, x, cfg, tuple(ctor["image_shape"]))
    d0 = out[("disp", 0)].numpy()
    st = m["stride"]
    got = d0[m["frames"]][:, :, ::st, ::st]
    assert got.shape == arrays["disp0"].shape
    assert np.abs(got - arrays["disp0"]).max() <= ATOL, float(np.abs(got - arrays["disp0"]).max())
    got3 = out[("disp", 3)].numpy()[m["frames"]]
    assert np.abs(got3 - arrays["disp3"]).max() <= ATOL
    stats = arrays["stats"]
    assert abs(float(d0.mean()) - stats[0]) <= 1e-5 and abs(float(d0.std()) - stats[1]) <= 1e-5
    assert stats[1] > 0.1   # non-degenerate


def test_unmerged_lora_equals_merged():
    m, arrays = load_case("fwd_vits_dvlora")
    cfg = oracle_cfg(m["ctor"])
    sd = weights.make_state_dict(cfg, m["weight_seed"])
    B, T, H, W = m["input"]
    x = weights.make_frames(B, T, H, W, m["frame_seed"])
    a = orc.forward(sd, x, cfg, tuple(m["ctor"]["image_shape"]), unmerged=True)[("disp", 0)].numpy()
    assert np.abs(a - arrays["disp0"]).max() <= ATOL


@pytest.mark.parametrize("name", [k for k, v in manifest().items() if v["kind"] == "video"])
def test_video_matches_reference_golden(name):
    m, arrays = load_case(name)
    ctor = m["ctor"]
    cfg = oracle_cfg(ctor)
    sd = weights.make_state_dict(cfg, m["weight_seed"])
    N, H, W = m["input"]
    v = weights.make_video_u8(N, H, W, m["frame_seed"])
    ishape = tuple(ctor["image_shape"])
    got = vo.infer_video_depth(v, ishape, lambda clip: orc.forward(sd, clip, cfg, ishape)[("disp", 0)])
    assert got.dtype == np.float32 and got.shape == arrays["depth"].shape
    assert np.abs(got - arrays["depth"]).max() <= ATOL


def _stub(clip):
    f = clip.flatten(0, 1)
    return f.mean(1, keepdim=True) + 0.1 * f.mean(dim=(1, 2, 3), keepdim=True)


def test_video_stub_bit_exact():
    """Window / keyframe / stitch arithmetic is bit-exact against the reference when the
    network is replaced by the same deterministic stub on both sides."""
    m, _ = load_case("video_stub")
    H, W = m["input"]
    for N in m["n"]:
        v = weights.make_video_u8(N, H, W, 100 + N)
        got = vo.infer_video_depth(v, tuple(m["image_shape"]), _stub)
        assert_video_stub_matches(N, got)


def test_window_slots_closed_form():
    """SURVEY.md section 3.2: slot i of window k reads frame min(f, N-1) with
    f = i (k=0); 22k-16 (i=0); 22k-10 (i=1); 22k+i (i>=2)."""
    for N in (1, 5, 21, 22, 23, 32, 44, 45, 100, 200, 2000):
        slots = vo.window_slots(N)
        assert len(slots) == (N + 21) // 22
        for k, row in enumerate(slots):
            for i, f in enumerate(row):
                if k == 0:
                    e = i
                elif i == 0:
                    e = 22 * k - 16
                elif i == 1:
                    e = 22 * k - 10
                else:
                    e = 22 * k + i
                assert f == min(e, N - 1)
