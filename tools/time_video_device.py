"""Video frames already on the GPU against host frames, and the gather-resize kernel, on the B200.

    python tools/time_video_device.py [--frames N] [--out PATH]
    python -m torch.distributed.run --standalone --nproc-per-node G tools/time_video_device.py [--frames N] [--out PATH]

End to end (BASELINE config 3: a 256x320 SCARED-shaped synthetic video, ViT-S at 224x280): ``infer_video_depth`` with
host uint8 frames (returns a numpy array) and with the same frames as a CUDA tensor (returns a CUDA tensor), the two
alternated within one process; each timed call ends with its result complete (host: the array is filled; device: the
stream is synchronised).  The device frames are uploaded once before timing, as a GPU decoder would leave them.  Under
torch.distributed every rank passes its own copy of the same video and the time is the max over ranks between
barriers.

Kernel (one process only): ``edv_op_cubic_resize_u8_gather``, for NHWC frames and for NCHW memory viewed as [N,H,W,3],
at 256x320 -> 224x280 and 1920x1080 -> the resize target of a 518x518 network.  The table is four windows of the driver
(128 output frames, 98 distinct source frames).  Each launch's duration comes from torch.profiler's CUDA activity, with
L2 overwritten before every launch.  Bandwidth is given for the distinct bytes (each named source frame once + the
float32 output) and for the logical bytes (one source frame per output frame + the output).

Writes one JSON file (default profiles/video_device_<G>gpu.json) with the card name and power limit of the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import endodav_b200 as E  # noqa: E402
from endodav_b200 import engine, synthetic, video  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=2000)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--out", default=None)
args = ap.parse_args()

rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
if world > 1:
    dist.init_process_group("nccl")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip())


def barrier():
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def time_e2e():
    torch.manual_seed(0)   # the base init draws from the global RNG: every rank builds the same weights
    model = E.endodav(encoder="vits", features=64, out_channels=[48, 96, 192, 384], r=4, lora_type="dvlora",
                      image_shape=(224, 280), disable_conv_head=True, residual_block_indexes=[])
    synthetic.randomize_(model, 1234)
    model = model.cuda().eval()
    n = args.frames
    host = np.random.default_rng(0).integers(0, 256, size=(n, 256, 320, 3), dtype=np.uint8)
    dev = torch.from_numpy(host).cuda()
    inputs = {"host": host, "device": dev}
    for x in inputs.values():                  # warm-up: plans, graphs, NCCL, the pinned output of the host path
        model.infer_video_depth(x)
    times = {k: [] for k in inputs}
    outs = {}
    for _ in range(args.reps):
        for k, x in inputs.items():
            barrier()
            t0 = time.perf_counter()
            outs[k] = model.infer_video_depth(x)
            barrier()
            times[k].append(time.perf_counter() - t0)
    res = {}
    for k, ts in times.items():
        t = torch.tensor([min(ts)], device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res[k] = dict(best_s=float(t), all_s=ts, frames_per_s=n / float(t))
    if rank == 0:
        res["device_equals_host"] = bool(torch.equal(outs["device"].cpu(), torch.from_numpy(outs["host"])))
    return res


def time_kernel():
    """Kernel durations from torch.profiler's CUDA activity (not host-side events around a Python loop, which would
    time the enqueue).  Before every launch a 256 MB buffer is written, so the 126 MB L2 holds none of the frames."""
    import tempfile

    from torch.profiler import ProfilerActivity, profile

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    out = []
    for (H, W), (ih, iw) in (((256, 320), (224, 280)), ((1080, 1920), (518, 518))):
        w, h = video.resize_target(W, H, iw, ih)
        n_src = 4 * video.STEP + video.INFER_LEN
        idx = np.concatenate([video.window_frame_indices(k, n_src) for k in range(4)])
        g = torch.Generator().manual_seed(0)
        base = torch.randint(0, 256, (n_src, 3, H, W), generator=g, dtype=torch.uint8).cuda()
        layouts = {"nhwc": base.permute(0, 2, 3, 1).contiguous(), "nchw_memory": base.permute(0, 2, 3, 1)}
        dst = torch.empty(len(idx), 3, h, w, dtype=torch.float32, device="cuda")
        out_bytes = dst.numel() * 4
        # every source frame the table names is read at least once; a frame that two windows share is read twice by the
        # kernel but may then hit L2, so DRAM traffic lies between these two counts
        distinct_bytes = len(np.unique(idx)) * H * W * 3 + out_bytes
        logical_bytes = len(idx) * H * W * 3 + out_bytes
        for name, x in layouts.items():
            for _ in range(3):
                engine.op_cubic_resize_u8(x, h, w, out=dst, index=idx)
            torch.cuda.synchronize()
            reps = 20
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(reps):
                    flush.fill_(1)
                    engine.op_cubic_resize_u8(x, h, w, out=dst, index=idx)
                torch.cuda.synchronize()
            with tempfile.TemporaryDirectory() as tmp:
                path = os.path.join(tmp, "trace.json")
                prof.export_chrome_trace(path)
                with open(path) as f:
                    events = json.load(f)["traceEvents"]
            durs = [e["dur"] for e in events if e.get("cat") == "kernel" and "cubic_resize_u8_kernel" in e.get("name", "")]
            assert len(durs) == reps, (name, len(durs))
            us = float(np.median(durs))
            out.append(dict(layout=name, src=[H, W], dst=[h, w], frames=len(idx), distinct_src_frames=int(len(np.unique(idx))),
                            kernel_us_median=us, kernel_us_min=float(min(durs)), l2_flushed=True,
                            distinct_bytes=distinct_bytes, logical_bytes=logical_bytes,
                            gb_per_s_distinct=distinct_bytes / us / 1e3, gb_per_s_logical=logical_bytes / us / 1e3))
    return out


result = dict(gpus=world, card=card(), frames=args.frames, shape=[256, 320], network=[224, 280], e2e=time_e2e())
if world == 1:
    result["gather_resize_kernel"] = time_kernel()
if rank == 0:
    path = args.out or os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                    "video_device_%dgpu.json" % world)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))
if world > 1:
    dist.destroy_process_group()
