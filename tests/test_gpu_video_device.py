"""Video frames already on the GPU: ``infer_video_depth`` of endodav and endodac reads a CUDA uint8 [N,H,W,3] tensor of
any strides in place and returns the stitched depth on that device, bit-identical to the host path on the same frames.
The gather form of the cubic resize (edv_op_cubic_resize_u8_gather) is pinned to the contiguous kernel bit for bit."""
import ctypes
import json
import os
import signal
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import endodav_b200 as E  # noqa: E402
from endodav_b200 import engine as eng  # noqa: E402
from endodav_b200 import synthetic  # noqa: E402
from endodav_b200 import video as V  # noqa: E402
from oracle import weights  # noqa: E402
from golden_util import load_case, oracle_cfg  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = dict(encoder="vits", features=64, out_channels=[48, 96, 192, 384], r=4, lora_type="dvlora",
             image_shape=(28, 42), disable_conv_head=True, residual_block_indexes=[])


# ---- kernel ----------------------------------------------------------------------------------------
def _view(layout, n, H, W, seed):
    """A uint8 [n,H,W,3] CUDA view in the given memory layout (never made contiguous)."""
    g = torch.Generator().manual_seed(seed)
    rnd = lambda *s: torch.randint(0, 256, s, generator=g, dtype=torch.uint8).cuda()  # noqa: E731
    if layout == "nhwc":
        return rnd(n, H, W, 3)
    if layout == "nchw":
        return rnd(n, 3, H, W).permute(0, 2, 3, 1)
    if layout == "step2":
        return rnd(2 * n, H, W, 3)[::2]
    return rnd(n, H + 16, W + 8, 3)[:, 8:-8, 4:-4]          # spatial crop


def _tables(n):
    """Index tables: the driver's windows over a short video (repeats and the clamped tail), and 300 random entries
    with repeats (two launches of at most 256 frames)."""
    wins = np.concatenate([V.window_frame_indices(k, n) for k in range(V.num_windows(n))])
    rnd = np.random.default_rng(n).integers(0, n, 300)
    return [wins, rnd]


@pytest.mark.parametrize("h,w", [(28, 42), (70, 98), (48, 64)])          # downscale, upscale, identity
@pytest.mark.parametrize("layout", ["nhwc", "nchw", "step2", "crop"])
def test_gather_resize_equals_contiguous_resize(layout, h, w):
    n, H, W = 40, 48, 64
    x = _view(layout, n, H, W, 11)
    assert not x.is_contiguous() or layout == "nhwc"
    for idx in _tables(n) + [None]:
        m = n if idx is None else len(idx)
        buf = torch.full((m + 2, 3, h, w), float("nan"), device="cuda")
        got = eng.op_cubic_resize_u8(x, h, w, out=buf[1:-1], index=idx)
        sel = x if idx is None else x[torch.from_numpy(idx).cuda()]
        ref = eng.op_cubic_resize_u8(sel.contiguous(), h, w)
        assert torch.equal(got, ref), (layout, h, w, None if idx is None else len(idx))
        assert bool(buf[0].isnan().all()) and bool(buf[-1].isnan().all())     # guard rows untouched


def test_gather_resize_rejects_bad_arguments():
    """EDV_ERR_ARG before any launch: dst stays all NaN."""
    lib = eng.load_library()
    n_src, H, W, h, w = 4, 16, 20, 8, 10
    x = _view("nhwc", n_src, H, W, 3)
    dst = torch.full((3, 3, h, w), float("nan"), device="cuda")
    idx = np.array([0, 3, 1], dtype=np.int64)
    S = (H * W * 3, W * 3, 3, 1)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(src=x.data_ptr(), ns=n_src, strides=S, index=idx, n=3, out=dst.data_ptr()):
        ip = index.ctypes.data_as(ctypes.c_void_p) if index is not None else None
        return lib.edv_op_cubic_resize_u8_gather(src, ns, H, W, *strides, ip, n, out, h, w, stream)

    bad = [dict(src=None), dict(out=None), dict(index=None), dict(n=0), dict(ns=0),
           dict(index=np.array([0, -1, 1], np.int64)), dict(index=np.array([0, 4, 1], np.int64)),
           dict(strides=(0,) + S[1:]), dict(strides=S[:1] + (0,) + S[2:]), dict(strides=S[:2] + (-3,) + S[3:]),
           dict(strides=S[:3] + (0,)), dict(strides=(1 << 62,) + S[1:])]
    for kw in bad:
        assert call(**kw) == -1, kw                       # EDV_ERR_ARG
    torch.cuda.synchronize()
    assert bool(dst.isnan().all())
    assert call() == 0                                    # the same call with valid arguments writes dst
    torch.cuda.synchronize()
    assert not bool(dst.isnan().any())


# ---- endodav driver --------------------------------------------------------------------------------
def _golden_model(case):
    m, arrays = load_case(case)
    kw = dict(m["ctor"])
    kw["image_shape"] = tuple(kw["image_shape"])
    model = E.endodav(dtype="fp32", **kw)
    model.load_state_dict(weights.make_state_dict(oracle_cfg(m["ctor"]), m["weight_seed"]), strict=True)
    N, H, W = m["input"]
    return model.cuda().eval(), weights.make_video_u8(N, H, W, m["frame_seed"]), arrays["depth"]


def _assert_same(dev_out, host_out):
    assert isinstance(dev_out, torch.Tensor) and dev_out.is_cuda and dev_out.dtype == torch.float32
    assert dev_out.is_contiguous() and tuple(dev_out.shape) == host_out.shape
    assert torch.equal(dev_out.cpu(), torch.from_numpy(host_out))


@pytest.mark.parametrize("case", ["video_n45", "video_n5"])
def test_device_frames_match_host_path_and_golden(case):
    model, v, ref = _golden_model(case)
    host = model.infer_video_depth(v)
    got = model.infer_video_depth(torch.from_numpy(v).cuda())
    _assert_same(got, host)
    err = np.abs(got.cpu().numpy() - ref) / np.maximum(np.abs(ref), 1.0)
    assert err.max() <= 5e-4, float(err.max())


def _small():
    """The small fp16 network, with the same weights in every process (its base init draws from the global RNG)."""
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(0)
        model = E.endodav(dtype="fp16", **SMALL)
    synthetic.randomize_(model, 5)
    return model.cuda().eval()


@pytest.fixture(scope="module")
def small_model():
    return _small()


SETTINGS = {"default": {}, "stitch_host": {"ENDODAV_STITCH": "host"}, "wb1": {"ENDODAV_WINDOW_BATCH": "1"},
            "wb3": {"ENDODAV_WINDOW_BATCH": "3"}, "gather_single": {"ENDODAV_GATHER": "single"}, "nchw": {}}


@pytest.mark.parametrize("setting", list(SETTINGS))
@pytest.mark.parametrize("n", [1, 31, 32, 33, 54, 300])
def test_device_frames_bit_identical_under_every_schedule(small_model, monkeypatch, n, setting):
    for k, val in SETTINGS[setting].items():
        monkeypatch.setenv(k, val)
    v = weights.make_video_u8(n, 40, 56, 100 + n)
    host = small_model.infer_video_depth(v)
    if setting == "nchw":          # an NCHW decoder batch presented as [N,H,W,3]
        x = torch.from_numpy(np.ascontiguousarray(v.transpose(0, 3, 1, 2))).cuda().permute(0, 2, 3, 1)
    else:
        x = torch.from_numpy(v).cuda()
    _assert_same(small_model.infer_video_depth(x), host)


def test_device_frames_strided_views(small_model):
    """Frame slices and spatial crops are read in place, equal to the host path on the same frames."""
    base = torch.from_numpy(weights.make_video_u8(90, 56, 72, 9)).cuda()
    for x in (base[::2], base[:, 8:-8, 4:-4]):
        _assert_same(small_model.infer_video_depth(x), small_model.infer_video_depth(x.cpu().numpy()))


def test_device_frames_large_frames_take_host_stitching(small_model):
    """8*H*W >= 2^24: the windows go to the host, the stitched result is uploaded once."""
    v = weights.make_video_u8(24, 1024, 2048, 3)
    host = small_model.infer_video_depth(v)
    _assert_same(small_model.infer_video_depth(torch.from_numpy(v).cuda()), host)


def test_device_frames_on_second_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    model = _small()
    v = weights.make_video_u8(54, 40, 56, 4)
    host = model.infer_video_depth(v)
    got = model.infer_video_depth(torch.from_numpy(v).to("cuda:1"))
    assert got.device == torch.device("cuda:1")
    _assert_same(got, host)


def test_device_frames_move_no_bulk_data_between_host_and_device(small_model, tmp_path):
    """Under torch.profiler (CUDA activity) a warmed-up default call copies nothing larger than 64 KB between host
    and device (the stitch plan table, 24.6 KB at 128 x 160, is the largest upload)."""
    from torch.profiler import ProfilerActivity, profile

    x = torch.from_numpy(weights.make_video_u8(120, 128, 160, 6)).cuda()
    small_model.infer_video_depth(x)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        small_model.infer_video_depth(x)
        torch.cuda.synchronize()
    path = str(tmp_path / "trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    assert any(e.get("cat") == "kernel" for e in events), "no CUDA activity recorded"
    copies = [e for e in events if e.get("cat") == "gpu_memcpy" and ("HtoD" in e["name"] or "DtoH" in e["name"])]
    big = [(e["name"], e["args"].get("bytes")) for e in copies if e["args"].get("bytes", 0) > 64 * 1024]
    assert not big, big


def test_device_frames_rejections(small_model):
    x = torch.from_numpy(weights.make_video_u8(5, 40, 56, 1)).cuda()
    with pytest.raises(ValueError):
        small_model.infer_video_depth(x.float())
    with pytest.raises(ValueError):
        small_model.infer_video_depth(x[..., :2])
    with pytest.raises(ValueError):
        small_model.infer_video_depth(x[0])
    with pytest.raises(ValueError):                       # a broadcast view: one plane expanded to three channels
        small_model.infer_video_depth(x[..., :1].expand(-1, -1, -1, 3))
    with pytest.raises(ValueError):
        small_model.infer_video_depth(x, device="cuda:%d" % (x.device.index + 1))
    with pytest.raises(ValueError):
        small_model.infer_video_depth(x, device="cpu")


# ---- endodac ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("batch_size", [1, 3, 8])
def test_endodac_device_frames_match_host_path(batch_size):
    from test_gpu_endodac import _build

    m, arrays = load_case("dac_video_n11")
    model = _build(m, "fp32")
    N, H, W = m["input"]
    v = weights.make_video_u8(N, H, W, m["frame_seed"])
    host = model.infer_video_depth(v, batch_size=batch_size)
    _assert_same(model.infer_video_depth(torch.from_numpy(v).cuda(), batch_size=batch_size), host)


# ---- two ranks -------------------------------------------------------------------------------------
_RANK_SCRIPT = r'''
import os, sys
import numpy as np
import torch
import torch.distributed as dist
import endodav_b200 as E
from endodav_b200 import synthetic
from oracle import weights

rank = int(os.environ["RANK"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl")
torch.manual_seed(0)
model = E.endodav(dtype="fp16", **{kw})
synthetic.randomize_(model, 5)
model = model.cuda().eval()
x = torch.from_numpy(weights.make_video_u8({n}, 40, 56, 8)).cuda()
for gather in ("rounds", "single"):
    os.environ["ENDODAV_GATHER"] = gather
    got = model.infer_video_depth(x)
    if rank == 0:
        assert got.is_cuda and got.device == x.device
        np.save(os.path.join(sys.argv[1], gather + ".npy"), got.cpu().numpy())
    else:
        assert got is None
dist.destroy_process_group()
'''


def test_two_ranks_device_frames_match_single_gpu(small_model, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    n = 300
    script = tmp_path / "ranks.py"
    script.write_text(_RANK_SCRIPT.format(kw=repr(SMALL), n=n))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, os.environ.get("PYTHONPATH", "")]))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", "2", str(script), str(tmp_path)]
    proc = subprocess.Popen(cmd, env=env, cwd=ROOT, start_new_session=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    try:
        log, _ = proc.communicate(timeout=600)
    finally:
        if proc.poll() is None:
            os.killpg(proc.pid, signal.SIGKILL)
            proc.wait()
    assert proc.returncode == 0, log.decode(errors="replace")[-4000:]
    single = small_model.infer_video_depth(torch.from_numpy(weights.make_video_u8(n, 40, 56, 8)).cuda()).cpu().numpy()
    for gather in ("rounds", "single"):
        assert np.array_equal(np.load(str(tmp_path / (gather + ".npy"))), single), gather
