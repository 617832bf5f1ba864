"""Multi-rank path of the long-video driver on CPU: world_size-2 ``gloo`` processes run
``endodav_b200.video.infer_video_depth`` with an injected per-window forward (the network is
replaced by the same deterministic stub on every rank), so window sharding, the gather to
rank 0 and the rank-0 stitching are exercised without a GPU.  The result must be bit-identical
to the single-process run and to the golden vectors written by the UNMODIFIED reference driver
with the same stub (tests/golden/video_stub.npz, oracle/make_golden.py)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from endodav_b200 import video
from oracle import weights
from golden_util import assert_video_stub_matches, load_case


class _Shape:
    """Stands in for the model: the driver only reads ``image_shape`` when forward_window is injected."""

    def __init__(self, image_shape):
        self.image_shape = tuple(image_shape)


def _stub(clip):
    f = clip.flatten(0, 1)
    return f.mean(1, keepdim=True) + 0.1 * f.mean(dim=(1, 2, 3), keepdim=True)


def _fw(clip, size):
    d = _stub(clip)  # [32,1,h,w]
    return torch.nn.functional.interpolate(d, size=size, mode="bilinear", align_corners=True)[:, 0]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, n, hw, image_shape, out_path):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        v = weights.make_video_u8(n, hw[0], hw[1], 100 + n)
        got = video.infer_video_depth(_Shape(image_shape), v, forward_window=_fw)
        if rank == 0:
            np.save(out_path, got)
        else:
            assert got is None
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("n", [5, 45, 100])
def test_two_rank_gloo_matches_single_process_and_reference(n, tmp_path):
    m, _ = load_case("video_stub")
    hw, ishape = m["input"], m["image_shape"]
    out = str(tmp_path / "r0.npy")
    mp.spawn(_worker, args=(2, _free_port(), n, hw, ishape, out), nprocs=2, join=True)
    dist2 = np.load(out)
    v = weights.make_video_u8(n, hw[0], hw[1], 100 + n)
    single = video.infer_video_depth(_Shape(ishape), v, forward_window=_fw, distributed=False)
    assert np.array_equal(dist2, single)
    assert_video_stub_matches(n, single)       # the reference's own driver, same stub


def test_shards_partition_the_window_list():
    for n in (1, 22, 23, 45, 2000):
        nw = video.num_windows(n)
        for world in (1, 2, 4, 8):
            shards = [video.shard_windows(nw, r, world) for r in range(world)]
            assert sorted(k for s in shards for k in s) == list(range(nw))
            assert max(len(s) for s in shards) - min(len(s) for s in shards) <= 1


def test_window_indices_match_oracle():
    from oracle import video_oracle as vo

    for n in (1, 5, 21, 22, 23, 32, 44, 45, 100, 2000):
        slots = vo.window_slots(n)
        assert len(slots) == video.num_windows(n)
        for k, row in enumerate(slots):
            assert list(video.window_frame_indices(k, n)) == list(row)


def test_final_frame_ranges_tile_the_video():
    """GPU stitcher bookkeeping (video._GpuStitcher): the frames each window finalises are disjoint, in order,
    cover [0, n) exactly, and never include the 8-frame tail the next window still cross-fades."""
    from endodav_b200 import video as V

    for n in (1, 5, 21, 22, 23, 32, 33, 44, 45, 54, 100, 2000):
        nwin = V.num_windows(n)
        pos = 0
        for k in range(nwin):
            lo, hi = V.final_frame_range(k, nwin, n)
            assert lo == min(pos, n) and hi >= lo
            if k < nwin - 1:
                assert hi <= max(V.INFER_LEN + V.STEP * k - V.INTERP_LEN, 0)
            pos = max(pos, hi)
        assert pos == n
