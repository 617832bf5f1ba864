#!/usr/bin/env python
"""Benchmark of the EndoDAV video-depth forward on B200 (BASELINE.json metric:
frames/sec on 32-frame 518 px clips at 1/2/4/8 GPUs, with roofline fractions).

  python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
  python bench.py --impl reference --steps K --warmup W    # the reference algorithm on host cores
  python bench.py ... --dump-outputs DIR                   # also save the last timed step's disparity maps

A step is one ``endodav.forward`` over one synthetic 32-frame 518x518 clip per GPU (ViT-S,
DV-LoRA, 16-bit tcgen05 path: fp16 operands by default, --dtype bf16 runs the same kernels) -- BASELINE.json configs[1].  At N > 1 every rank runs its own
window (the long-video driver shards independent 32-frame windows, SURVEY.md 8(e)) and each
step ends with the NCCL gather of the per-window disparity to rank 0: weak scaling.

Prints ONE JSON line on rank 0 (see the keys at the bottom of main()).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it (it may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: ctor kwargs, (B, T, H, W)
    "vits_518_t32": (dict(encoder="vits", features=64, out_channels=[48, 96, 192, 384], r=4, lora_type="dvlora",
                          image_shape=(518, 518), disable_conv_head=True, residual_block_indexes=[]), (1, 32, 518, 518)),
    "vits_224x280_t32": (dict(encoder="vits", features=64, out_channels=[48, 96, 192, 384], r=4, lora_type="dvlora",
                              image_shape=(224, 280), disable_conv_head=True, residual_block_indexes=[]), (1, 32, 224, 280)),
    "vits_224x280_t8": (dict(encoder="vits", features=64, out_channels=[48, 96, 192, 384], r=4, lora_type="dvlora",
                             image_shape=(224, 280), disable_conv_head=True, residual_block_indexes=[]), (1, 8, 224, 280)),
    "vitl_518_t32": (dict(encoder="vitl", features=256, out_channels=[256, 512, 1024, 1024], r=4, lora_type="dvlora",
                          image_shape=(518, 518), disable_conv_head=True, residual_block_indexes=[]), (1, 32, 518, 518)),
    # BASELINE config 4: ViT-L, batch of 4 x 32-frame 518x518 clips (spatial + temporal attention stress)
    "vitl_518_t32_b4": (dict(encoder="vitl", features=256, out_channels=[256, 512, 1024, 1024], r=4, lora_type="dvlora",
                             image_shape=(518, 518), disable_conv_head=True, residual_block_indexes=[]), (4, 32, 518, 518)),
}
METRIC = "frames/sec, 32-frame 518px clips"
UNIT = "frames/s"
DUMP_LIMIT_BYTES = 64 * 10 ** 6


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), power_w_max=max(pw), samples=len(sm), reasons=sorted(reasons))


# --------------------------------------------------------------------------------------------
# reference algorithm on the host (oracle/ is test infrastructure: only this leg may run it)
# --------------------------------------------------------------------------------------------
def cpu_reference_fps(ctor, shape, sample_frames, steps, warmup):
    import torch

    from oracle import endodav_oracle as orc
    from oracle import weights

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = weights.full_cfg({k: v for k, v in ctor.items() if k != "image_shape"})
    sd = weights.make_state_dict(cfg, 1234)
    B, T, H, W = shape
    t = min(sample_frames, T)
    x = weights.make_frames(1, t, H, W, 4321)
    with torch.no_grad():
        for _ in range(warmup):
            orc.forward(sd, x[:, :1], cfg, ctor["image_shape"])
        t0 = time.perf_counter()
        for _ in range(steps):
            orc.forward(sd, x, cfg, ctor["image_shape"])
        dt = time.perf_counter() - t0
    return dict(value=t * steps / dt, unit=UNIT, cores=cores, kind="port",
                sample="%d of %d frames of the %dx%d clip per step, %d step(s), fp32 torch CPU restatement of the reference "
                       "(oracle/endodav_oracle.py), %.1f s" % (t, T, H, W, steps, dt)), dt


def run_reference_eager_gpu(args):
    """BASELINE.md section 4 sanity line: the SAME restatement of the reference (plain PyTorch eager ops, ATen / cuBLAS /
    cuDNN kernels) on this B200, fp32 and under autocast(bf16), full clip, CUDA-event timed.  Not the reference arm (that is
    the CPU run below) and never the product path -- it says what "move the reference to the GPU unchanged" buys."""
    import torch

    from oracle import endodav_oracle as orc
    from oracle import weights

    ctor, shape = WORKLOADS[args.workload]
    cfg = weights.full_cfg({k: v for k, v in ctor.items() if k != "image_shape"})
    dev = torch.device("cuda:0")
    sd = {k: v.to(dev) for k, v in weights.make_state_dict(cfg, 1234).items()}
    B, T, H, W = shape
    x = weights.make_frames(B, T, H, W, 4321).to(dev)
    out = {}
    steps, warm = max(2, min(args.steps, 5)), max(1, min(args.warmup, 2))
    for name, ctx in (("fp32", torch.autocast("cuda", enabled=False)), ("autocast_bf16", torch.autocast("cuda", dtype=torch.bfloat16))):
        with torch.no_grad(), ctx:
            for _ in range(warm):
                orc.forward(sd, x, cfg, ctor["image_shape"])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                orc.forward(sd, x, cfg, ctor["image_shape"])
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[name] = dict(ms_per_step=ms, frames_per_s=B * T / (ms * 1e-3), steps=steps)
    print(json.dumps({"impl": "reference-eager-gpu", "metric": METRIC, "unit": UNIT, "n_gpus": 1, "data": "synthetic",
                      "config": {"workload": args.workload, "frames_per_clip": T, "frame": [H, W]},
                      "note": "oracle/endodav_oracle.py (PyTorch eager restatement of the reference) on cuda:0; library kernels, not this repo's",
                      "value": out["fp32"]["frames_per_s"], "results": out}))
    return 0


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    if args.reference_device == "cuda":
        return run_reference_eager_gpu(args)
    ctor, shape = WORKLOADS[args.workload]
    base, dt = cpu_reference_fps(ctor, shape, args.cpu_frames, max(1, args.steps), min(args.warmup, 1))
    steps = max(1, args.steps)
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "clips_per_gpu_per_step": shape[0], "frames_per_clip": shape[1], "frame": [shape[2], shape[3]],
                   "network_resolution": list(ctor["image_shape"]), "weights": "random-init, de-degenerated (oracle/weights.py, same recipe)",
                   "l2": "n/a (host)", "parallelism": "host cores",
                   "sample_frames": min(args.cpu_frames, shape[1]),
                   "note": "reference algorithm (CPU port) on host cores; each step is a bounded sample of the clip"},
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------------------------
def dump_outputs(out, directory):
    """Write the disparity pyramid that a caller of the timed forward receives as DIR/disp<s>.npy (float32), so that
    two builds can be compared output for output.  A pyramid above DUMP_LIMIT_BYTES is cut to the same share of every
    map: a sorted sample of flat indices drawn with a fixed seed, identical from run to run."""
    import numpy as np

    arrays = {"disp%d" % s: out[("disp", s)].float().cpu().numpy() for s in range(4)}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_LIMIT_BYTES:
            keep = a.size * DUMP_LIMIT_BYTES // total
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


def time_forward(E, synthetic, workload, dtype, dev, steps, warmup):
    """Device-timed forward of another workload / dtype on this rank (resident inputs): ms per step, frames/s."""
    import torch

    ctor, (B, T, H, Wd) = WORKLOADS[workload]
    model = E.endodav(dtype=dtype, **ctor)
    synthetic.randomize_(model, 1234)
    model = model.to(dev).eval()
    x = torch.rand(B, T, 3, H, Wd, generator=torch.Generator().manual_seed(4321)).to(dev)
    for _ in range(max(3, warmup)):
        model(x)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        model(x)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    out = dict(workload=workload, dtype=dtype, ms_per_step=ms, frames_per_s=B * T / (ms * 1e-3), steps=steps,
               gpu_launches_per_step=model._eng.launch_count(), cuda_graphs=model._eng.graph_count())
    del model
    torch.cuda.empty_cache()
    return out


def time_config5_sweep(E, synthetic, dtype, dev):
    """BASELINE config 5 (Hamlyn-shaped clip-batch sweep at 256x320, network resolution 224x280), a bounded subset of
    tools/sweep_clips.py: frames/s of endodav.forward and the temporal-attention kernel's share / bandwidth."""
    import torch

    ctor, _ = WORKLOADS["vits_224x280_t32"]
    model = E.endodav(dtype=dtype, **ctor)
    synthetic.randomize_(model, 1234)
    model = model.to(dev).eval()
    rows = []
    for T in (8, 32):
        for B in (1, 8, 64):
            x = torch.rand(B, T, 3, 256, 320, device=dev)
            for _ in range(3):
                model(x)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 10 if B * T <= 512 else 3
            e0.record()
            for _ in range(reps):
                model(x)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / reps
            eng = model._eng
            eng.profile(True)
            model(x)
            tab = eng.profile_collect()
            eng.profile(False)
            tot = sum(r["ms"] for r in tab) or 1.0
            ta = sum(r["ms"] for r in tab if r["name"].startswith("temporal_attention"))
            tb = sum(r["bytes"] for r in tab if r["name"].startswith("temporal_attention"))
            rows.append(dict(clips=B, T=T, ms=ms, frames_per_s=B * T / ms * 1e3, temporal_attention_share=ta / tot,
                             temporal_attention_gbs=tb / (ta * 1e-3) / 1e9 if ta else 0.0))
            del x
    del model
    torch.cuda.empty_cache()
    return dict(frame=[256, 320], network_resolution=[224, 280], dtype=dtype, rows=rows)


def time_video_config3(E, synthetic, dev, world, rank, dist, n_frames=2000):
    """BASELINE config 3: SCARED-shaped 2 000-frame 256x320 video through infer_video_depth, windows sharded over the
    ranks (strong scaling: the video is fixed).  Host uint8 frames in, host float32 depth out; wall clock between
    barriers, max over ranks.  Rank 0 also runs the single-GPU driver and reports whether the results are bit-identical."""
    import numpy as np
    import torch

    ctor, _ = WORKLOADS["vits_224x280_t32"]
    torch.manual_seed(0)   # the base init draws from the global RNG: every rank must build the same weights
    model = E.endodav(dtype="fp16", **ctor)
    synthetic.randomize_(model, 1234)
    model = model.to(dev).eval()
    rng = np.random.default_rng(2024)
    frames = rng.integers(0, 256, size=(n_frames, 256, 320, 3), dtype=np.uint8)
    from endodav_b200 import video as V

    def run(distributed):
        if world > 1 and distributed:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = V.infer_video_depth(model, frames, device=dev, distributed=distributed)
        torch.cuda.synchronize()
        if world > 1 and distributed:
            dist.barrier()
        return out, time.perf_counter() - t0

    run(True)                     # warm-up: plans, pinned buffers, CUDA graphs
    out, secs = run(True)
    t = torch.tensor([secs], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    secs = float(t.item())
    res = dict(frames=n_frames, frame=[256, 320], windows=V.num_windows(n_frames), seconds=secs, frames_per_s=n_frames / secs,
               scaling="strong", n_gpus=world)
    if world > 1:
        if rank == 0:
            run(False)                # warm-up of the single-GPU schedule (its own plan / graphs / pinned ring)
            single, s1 = run(False)
            res["bitwise_equal_to_1gpu"] = bool(np.array_equal(out, single))
            res["seconds_1gpu_same_process"] = s1
        dist.barrier()
    del model
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="vits_518_t32", choices=sorted(WORKLOADS))
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16", "fp32"])
    ap.add_argument("--cpu-frames", type=int, default=16, help="frames per step of the CPU baseline sample")
    ap.add_argument("--cpu-steps", type=int, default=4, help="steps of the CPU baseline sample in the GPU arm (~10 s of CPU work)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--kernels-out", default=None, help="write the per-call-site kernel table (JSON) here")
    ap.add_argument("--reference-device", default="cpu", choices=["cpu", "cuda"],
                    help="with --impl reference: 'cuda' prints the eager-PyTorch-on-this-GPU sanity line instead of the CPU reference arm")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra measured lines (bf16, 224x280 workloads, video config 3)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the disparity maps of the last timed step (rank 0) to DIR/disp<s>.npy, float32, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    import endodav_b200 as E
    from endodav_b200 import synthetic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the sm_100a path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    W = max(3, args.warmup)
    K = args.steps

    ctor, (B, T, H, Wd) = WORKLOADS[args.workload]
    torch.manual_seed(0)   # the base init draws from the global RNG: the same weights in every run and on every rank
    model = E.endodav(dtype=args.dtype, **ctor)
    synthetic.randomize_(model, 1234)
    model = model.to(dev).eval()
    g = torch.Generator().manual_seed(4321 + rank)
    host = torch.rand(B, T, 3, H, Wd, generator=g).pin_memory()
    x = host.to(dev)
    frames_per_step = B * T

    gather_bufs = None
    side = torch.cuda.Stream()

    pending = []

    def step(inp):
        out = model(inp)
        d0 = out[("disp", 0)]
        if world > 1:
            # the one collective of the path: per-window disparity -> rank 0 (SURVEY.md 8(e)).  Issued
            # asynchronously on NCCL's stream so that it overlaps the next window's kernels; at most
            # two are in flight (the gathers themselves serialise on NCCL's stream).
            if len(pending) >= 2:
                pending.pop(0).wait()
            pending.append(dist.gather(d0, gather_bufs if rank == 0 else None, dst=0, async_op=True))
        return out

    def drain():
        while pending:
            pending.pop(0).wait()

    if world > 1 and rank == 0:
        oh, ow = ctor["image_shape"]
        gather_bufs = [torch.empty(B * T, 1, oh, ow, dtype=torch.float32, device=dev) for _ in range(world)]

    def barrier():
        drain()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(W):
        step(x)
    eng = model._eng
    launches_per_step = eng.launch_count()
    ws_gb = eng.workspace.numel() / 1e9

    # ---- timed region: K steps, inputs resident in HBM ---------------------------------------
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        out = step(x)
    drain()          # the current stream waits for the outstanding gathers: they are inside the timed region
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    t_ms = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms = float(t_ms.item())
    value = world * frames_per_step * K / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    del out

    # ---- same K steps with one CUDA event per launch: per-kernel device time ---------------------
    eng.profile(True)
    barrier()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for _ in range(K):
        model(x)
    p1.record()
    torch.cuda.synchronize()
    prof_ms = p0.elapsed_time(p1)
    table = eng.profile_collect()
    eng.profile(False)

    # ---- end to end through the public API with HOST buffers -------------------------------------
    # Every step copies its clip from pinned host memory and reads its disparity back to pinned host
    # memory.  The copies run on their own streams, double buffered, so the H2D of step i+1 and the
    # D2H of step i-1 overlap the kernels of step i -- the way a streaming caller (the long-video
    # driver) uses the API.  Timed with the host clock around K complete steps.
    out_host = [torch.empty(B * T, 1, *ctor["image_shape"], dtype=torch.float32).pin_memory() for _ in range(2)]
    xbuf = [torch.empty_like(x) for _ in range(2)]
    h2d_s, d2h_s = torch.cuda.Stream(), torch.cuda.Stream()
    main_s = torch.cuda.current_stream()

    def e2e_loop(n):
        h2d_ev = [None, None]
        free_ev = [None, None]     # compute that read xbuf[j] has finished
        d2h_ev = [None, None]      # D2H that wrote out_host[j] has finished
        for i in range(n):
            j = i & 1
            with torch.cuda.stream(h2d_s):
                if free_ev[j] is not None:
                    h2d_s.wait_event(free_ev[j])
                xbuf[j].copy_(host, non_blocking=True)
                h2d_ev[j] = torch.cuda.Event()
                h2d_ev[j].record(h2d_s)
            main_s.wait_event(h2d_ev[j])
            d0 = step(xbuf[j])[("disp", 0)]
            free_ev[j] = torch.cuda.Event()
            free_ev[j].record(main_s)
            with torch.cuda.stream(d2h_s):
                d2h_s.wait_event(free_ev[j])
                if d2h_ev[j] is not None:
                    d2h_ev[j].synchronize()      # the caller has consumed out_host[j] of step i-2
                out_host[j].copy_(d0, non_blocking=True)
                d0.record_stream(d2h_s)
                d2h_ev[j] = torch.cuda.Event()
                d2h_ev[j].record(d2h_s)
        torch.cuda.synchronize()

    e2e_loop(8)     # warm-up: every (input buffer, output block) pointer set the allocator cycles through gets its CUDA graph captured here, not in the timed loop
    barrier()
    t0 = time.perf_counter()
    e2e_loop(K)
    barrier()
    e2e_s = time.perf_counter() - t0
    t_e = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_val = world * frames_per_step * K / float(t_e.item())

    # ---- extra measured lines (not the headline): bf16 beside the fp16 default, the reference's own resolution,
    # and BASELINE config 3 (long video, strong scaling over the ranks) ------------------------------------
    extra = {}
    if not args.no_extras and args.workload == "vits_518_t32":
        if rank == 0:
            other = "bf16" if args.dtype != "bf16" else "fp16"
            jobs = [(other, lambda: time_forward(E, synthetic, "vits_518_t32", other, dev, max(3, K // 3), 3))]
            if world == 1:
                jobs += [("config1_vits_224x280_t8", lambda: time_forward(E, synthetic, "vits_224x280_t8", args.dtype, dev, 50, 10)),
                         ("vits_224x280_t32", lambda: time_forward(E, synthetic, "vits_224x280_t32", args.dtype, dev, 50, 10)),
                         ("config4_vitl_518_t32_b4", lambda: time_forward(E, synthetic, "vitl_518_t32_b4", args.dtype, dev, 3, 3)),
                         ("config5_sweep", lambda: time_config5_sweep(E, synthetic, args.dtype, dev))]
            for name, fn in jobs:
                try:
                    extra[name] = fn()
                except Exception as exc:  # the headline line must survive a failure of an extra
                    extra[name] = dict(error=repr(exc)[:300])
        if world > 1:
            dist.barrier()
        try:
            extra["video_config3"] = time_video_config3(E, synthetic, dev, world, rank, dist if world > 1 else None)
        except Exception as exc:  # the headline line must survive a failure of an extra
            extra["video_config3"] = dict(error=repr(exc)[:300])

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel ------------------------------------------------------
    peaks = measured_peaks()
    table.sort(key=lambda r: -r["ms"])
    tot = sum(r["ms"] for r in table) or 1.0
    ridge = peaks["bf16_tflops"] * 1e12 / (peaks["hbm_gbs"] * 1e9)
    for r in table:
        r["share"] = r["ms"] / tot
        r["avg_us"] = 1e3 * r["ms"] / max(1, r["count"])
        r["tflops"] = r["flops"] / (r["ms"] * 1e-3) / 1e12 if r["ms"] > 0 else 0.0
        r["gbs"] = r["bytes"] / (r["ms"] * 1e-3) / 1e9 if r["ms"] > 0 else 0.0
        r["bound"] = "tensor" if (r["bytes"] > 0 and r["flops"] / r["bytes"] >= ridge) else "hbm"
    top = table[0] if table else None
    roofline = None
    if top:
        if top["bound"] == "tensor":
            # the bench runs a fraction of a second at full clocks (see "clocks"): the BURST cuBLAS figure is the honest
            # denominator; the sustained one (seconds-long loop under the power cap) is printed beside it
            roofline = dict(kernel=top["name"], bound="tensor", achieved=top["tflops"], peak=peaks["bf16_tflops"],
                            unit="TFLOP/s", frac=top["tflops"] / peaks["bf16_tflops"],
                            peak_sustained=peaks["bf16_tflops_sustained"], frac_of_sustained=top["tflops"] / peaks["bf16_tflops_sustained"])
        else:
            roofline = dict(kernel=top["name"], bound="hbm", achieved=top["gbs"], peak=peaks["hbm_gbs"], unit="GB/s",
                            frac=top["gbs"] / peaks["hbm_gbs"])
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "r2_ncu_full_summary_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            if top["name"] in tj:
                traffic = tj[top["name"]]["bytes"]
                traffic_src = "ncu --set full dram__bytes_read+write.sum of one launch at this shape (profiles/r2_ncu_full_summary.txt)"
        roofline.update(traffic=traffic, traffic_source=traffic_src, share_of_step=top["share"], avg_launch_us=top["avg_us"], launches_per_step=top["count"] // K,
                        peak_source=peaks["source"] + (", burst bf16 (frac_of_sustained beside it)" if top["bound"] == "tensor" else ""))
        # whole-forward tensor utilisation: all contraction FLOPs / step time
        roofline["step_tflops"] = sum(r["flops"] for r in table) / K / (ms / K * 1e-3) / 1e12
        if top["name"] == "flash_attention_tc":
            # The kernel's real limiter (DESIGN.md section 5): every score costs one MUFU ex2, 16 per clock per SM, against
            # 2 x 64 MACs of tensor work -- at head dim 64 the exponentials need twice the cycles of the MMAs.  Stated beside the
            # contract's tensor roofline so that the fraction can be read against the pipe that actually bounds the kernel.
            h_, w_ = ctor["image_shape"]
            S = (h_ // 14) * (w_ // 14) + 1
            heads = {"vits": 6, "vitb": 12, "vitl": 16}[ctor["encoder"]]
            blk = (S + 127) // 128 * 128
            exps = float(B * T * heads) * blk * blk
            mhz = (clocks or {}).get("sm_mhz") or 1965.0
            peak = 16.0 * 148 * mhz * 1e6
            roofline["mufu"] = dict(exp_per_launch=exps, peak_exp_per_s=peak, achieved_exp_per_s=exps / (top["avg_us"] * 1e-6),
                                    frac=exps / (top["avg_us"] * 1e-6) / peak,
                                    note="ex2 on the MUFU pipe: 16 / clock / SM x 148 SMs at the sampled SM clock; the softmax instruction mix "
                                         "reaches at most 86 % of it with two warps per scheduler (profiles/r2_microbench_softmax_mix.txt)")
    if args.kernels_out:
        with open(args.kernels_out, "w") as f:
            json.dump(dict(workload=args.workload, steps=K, profiled_ms_per_step=prof_ms / K, ms_per_step=ms / K, kernels=table), f, indent=1)

    cpu_base = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_base, _ = cpu_reference_fps(ctor, (B, T, H, Wd), args.cpu_frames, max(1, args.cpu_steps), 1)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": args.workload, "clips_per_gpu_per_step": B, "frames_per_clip": T, "frame": [H, Wd],
                   "network_resolution": list(ctor["image_shape"]), "weights": "random-init, de-degenerated (endodav_b200/synthetic.py)",
                   "l2": "no flush: per-step working set %.2f GB of activations >> 126 MB L2" % ws_gb,
                   "parallelism": "window-sharded dp%d + NCCL gather to rank 0" % world if world > 1 else "single GPU"},
        "roofline": roofline, "cpu_baseline": cpu_base,
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": host.numel() * 4, "d2h_bytes_per_step": out_host[0].numel() * 4,
                "note": "pinned host clip in, pinned host disparity out, copies double-buffered on side streams"},
        "gpu_launches": launches_per_step * K * world, "clocks": clocks,
        "profiled_ms_per_step": prof_ms / K, "cuda_graphs": eng.graph_count(), "extra": extra,
        "top_kernels": [dict(name=r["name"], share=round(r["share"], 4), avg_us=round(r["avg_us"], 1), tflops=round(r["tflops"], 1),
                             gbs=round(r["gbs"], 1)) for r in table[:8]],
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
