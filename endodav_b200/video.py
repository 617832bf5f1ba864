"""Sliding-window long-video driver (re-host of ``endodav.infer_video_depth``,
models/endodav/endodav.py:162-254) with windows sharded across the GPUs of one box.

Reference behaviour that is preserved exactly:
  * 32-frame windows, stride 22, 10 overlap slots fed from the previous window's *input*
    slots KEYFRAMES=[6,12,24..31] (endodav.py:47-50,193-199);
  * per-frame aspect-keeping cubic resize on the host (util/transform.py:62-122);
  * per-window bilinear resize of the disparity back to the frame size (endodav.py:205);
  * sequential scale/shift alignment + 8-frame linear cross-fade on rank 0 in float32 numpy,
    op for op (endodav.py:213-254; utils/util.py:40-74).

What is new: window inputs are a pure function of (k, N) (SURVEY.md section 3.2), so windows
are independent.  Rank r of W runs windows k = r, r+W, ... and one NCCL gather moves the
per-window disparity to rank 0 (``torch.distributed``); there is no collective inside the
network.  With torch.distributed not initialised this is the single-GPU path.
"""
import os
import time

import numpy as np
import torch

INFER_LEN = 32
OVERLAP = 10
KEYFRAMES = [6, 12, 24, 25, 26, 27, 28, 29, 30, 31]
INTERP_LEN = 8
STEP = INFER_LEN - OVERLAP


def num_windows(n_frames):
    return (n_frames + STEP - 1) // STEP


def window_frame_indices(k, n_frames):
    """Closed form of the source frame of every slot of window k.

    Unrolling endodav.py:185-199: slot i of window k>0 is slot KEYFRAMES[i] of window k-1 for
    i<10; KEYFRAMES[2:] = 24..31 are fresh slots of window k-1 (frames 22(k-1)+24.. = 22k+2..),
    while KEYFRAMES[0:2] = 6,12 are themselves fresh slots of window k-1 when k-1>0
    (22(k-1)+6 = 22k-16, 22(k-1)+12 = 22k-10) and plain frames 6,12 when k-1 == 0 (same
    formula).  Padding replicates the last frame, hence the clamp."""
    idx = np.empty(INFER_LEN, dtype=np.int64)
    if k == 0:
        idx[:] = np.arange(INFER_LEN)
    else:
        idx[0] = STEP * k - 16
        idx[1] = STEP * k - 10
        idx[2:] = STEP * k + np.arange(2, INFER_LEN)
    return np.minimum(idx, n_frames - 1)


def shard_windows(n_windows, rank, world):
    """Round-robin window ownership: rank r owns k = r, r+world, ...  (SURVEY.md section 8(e))."""
    return list(range(rank, n_windows, world))


def resize_target(width, height, want_w, want_h, multiple=14):
    """Output size of the reference's Resize(keep_aspect_ratio=True, 'lower_bound',
    ensure_multiple_of=14) (util/transform.py:49-107)."""
    scale_h, scale_w = want_h / height, want_w / width
    if scale_w > scale_h:
        scale_h = scale_w
    else:
        scale_w = scale_h

    def fit(x, lo):
        y = int(np.round(x / multiple) * multiple)
        if y < lo:
            y = int(np.ceil(x / multiple) * multiple)
        return y

    return fit(scale_w * width, want_w), fit(scale_h * height, want_h)


def lsq_scale_shift(pred, target):
    """compute_scale_and_shift_full with an all-ones mask, float32 numpy sums
    (utils/util.py:40-62); det == 0 -> (1, 0)."""
    pred = pred.astype(np.float32)
    target = target.astype(np.float32)
    ones = np.ones_like(target, dtype=np.float32)
    a00 = np.sum(ones * pred * pred)
    a01 = np.sum(ones * pred)
    a11 = np.sum(ones)
    b0 = np.sum(ones * pred * target)
    b1 = np.sum(ones * target)
    det = a00 * a11 - a01 * a01
    if det != 0:
        return (a11 * b0 - a01 * b1) / det, (-a01 * b0 + a00 * b1) / det
    return 1, 0


def stitch_windows(windows, n_frames):
    """windows: sequence over k of float32 [32,H,W] -> float32 [n_frames,H,W].

    Sequential by construction: (scale, shift) of window k is fitted against the already
    aligned tail of windows < k (endodav.py:231-244)."""
    fade = [0.0] + [i * (1.0 / (INTERP_LEN - 1)) for i in range(1, INTERP_LEN - 1)] + [1.0]
    seq = []
    for k, win in enumerate(windows):
        if k == 0:
            seq.extend(win[i] for i in range(INFER_LEN))
            continue
        pre = seq[-INTERP_LEN:]
        post = [win[i] for i in range(OVERLAP - INTERP_LEN, OVERLAP)]
        scale, shift = lsq_scale_shift(np.concatenate(post), np.concatenate(pre))
        aligned_post = []
        for f in post:
            g = f * scale + shift
            g[g < 0] = 0
            aligned_post.append(g)
        seq[-INTERP_LEN:] = [pre[i] * (1 - fade[i]) + aligned_post[i] * fade[i] for i in range(INTERP_LEN)]
        for i in range(OVERLAP, INFER_LEN):
            g = win[i] * scale + shift
            g[g < 0] = 0
            seq.append(g)
    return np.stack(seq[:n_frames], axis=0)


class _FrameCache:
    """Host-side preprocessing of the reference (endodav.py:195): float32/255 -> cv2 cubic
    resize -> CHW.  Each source frame is resized once even when several windows read it."""

    def __init__(self, frames, new_w, new_h):
        import cv2

        self.cv2 = cv2
        self.frames = frames
        self.size = (new_w, new_h)
        self.cache = {}

    def get(self, idx):
        t = self.cache.get(idx)
        if t is None:
            img = self.frames[idx].astype(np.float32) / 255.0
            img = self.cv2.resize(img, self.size, interpolation=self.cv2.INTER_CUBIC)
            t = np.ascontiguousarray(np.transpose(img, (2, 0, 1))).astype(np.float32)
            self.cache[idx] = t
        return t


class _Stager:
    """Host-side staging of the raw uint8 frames of window batches into pinned memory, off the launching thread.

    A batch is WB windows x 32 frames; window k > 0 is two single frames plus ONE contiguous run of 30 frames
    (``window_frame_indices``), so staging is three bulk copies per window.  Done inline it costs 10-17 ms per batch of four
    256x320 windows when eight ranks stage at once -- more than the 9.5 ms the GPU needs for that batch, and the first
    batch delayed every rank's first kernel (measured with ENDODAV_TRACE=1: the 8-GPU long-video run was bound by exactly
    this).  Here every window of a batch is copied by its own worker thread (torch's copy releases the GIL), and the
    next two batches of the caller's (sequential) schedule are staged while the current one is uploaded and computed.
    Ring of three pinned buffers; a buffer is rewritten only after the H2D copy that read it has completed."""

    RING = 3

    def __init__(self, frames, n_frames, mine, WB, H, W):
        from concurrent.futures import ThreadPoolExecutor

        self.frames, self.n, self.mine, self.WB = frames, n_frames, mine, WB
        pin = torch.cuda.is_available()   # (the CPU unit test of the staging logic runs without CUDA)
        self.bufs = [torch.empty(WB * INFER_LEN, H, W, 3, dtype=torch.uint8, pin_memory=pin) for _ in range(self.RING)]
        self.h2d_done = [None] * self.RING
        self.pool = ThreadPoolExecutor(max_workers=max(1, min(4, WB)))
        import weakref
        weakref.finalize(self, self.pool.shutdown, False)   # the worker threads go away with the stager
        self.tasks = {}          # (j, nb) -> (slot, futures)
        self.slot_futs = [[] for _ in range(self.RING)]   # fill tasks last submitted per buffer (possibly never fetched)
        self.count = 0

    def _fill(self, slot, b, k, ev):
        if ev is not None:
            ev.synchronize()     # the earlier upload out of this buffer has finished
        dst = self.bufs[slot][b * INFER_LEN:(b + 1) * INFER_LEN]
        idx = window_frame_indices(k, self.n)
        if int(idx[-1]) - int(idx[2]) == INFER_LEN - 3:
            dst[2:].copy_(torch.from_numpy(self.frames[int(idx[2]): int(idx[-1]) + 1]))
            dst[0].copy_(torch.from_numpy(self.frames[int(idx[0])]))
            dst[1].copy_(torch.from_numpy(self.frames[int(idx[1])]))
        else:                    # the clamped tail of the video: frame by frame
            np.take(self.frames, idx, axis=0, out=dst.numpy())

    def submit(self, j, nb):
        if nb <= 0 or j >= len(self.mine) or (j, nb) in self.tasks:
            return
        slot = self.count % self.RING
        self.count += 1
        ev, self.h2d_done[slot] = self.h2d_done[slot], None
        self.tasks = {k: v for k, v in self.tasks.items() if v[0] != slot}   # a stale prefetch in this buffer is forgotten
        for f in self.slot_futs[slot]:
            f.result()           # a prefetch that was never fetched (non-sequential caller) must not still be writing this buffer
        futs = [self.pool.submit(self._fill, slot, b, self.mine[j + b], ev) for b in range(nb)]
        self.slot_futs[slot] = futs
        self.tasks[(j, nb)] = (slot, futs)

    def fetch(self, j, nb):
        """-> (slot, pinned uint8 [nb*32,H,W,3]) for windows mine[j:j+nb]; stages the next two batches of a sequential
        schedule in the background."""
        self.submit(j, nb)
        slot, futs = self.tasks.pop((j, nb))
        for ahead in (1, 2):
            jn = j + ahead * nb
            self.submit(jn, min(nb, len(self.mine) - jn))
        for f in futs:
            f.result()
        return slot, self.bufs[slot][: nb * INFER_LEN]

    def uploaded(self, slot, event):
        self.h2d_done[slot] = event

    def close(self):
        self.pool.shutdown(wait=True)


def final_frame_range(k, n_windows, n_frames):
    """Output frames that become final once window k is stitched: everything but the 8-frame tail the next
    window will cross-fade (the last window finalises its tail too), clipped to the video length."""
    lo = 0 if k == 0 else INFER_LEN + STEP * (k - 1) - INTERP_LEN
    hi = INFER_LEN + STEP * (n_windows - 1) if k == n_windows - 1 else INFER_LEN + STEP * k - INTERP_LEN
    return min(lo, n_frames), min(hi, n_frames)


class _GpuStitcher:
    """Device-side replacement of ``stitch_windows`` (endodav.py:213-254): windows are pushed in order, each
    one is aligned and cross-faded by ``edv_op_stitch_window`` on the current stream (no host sync), and the
    frames it makes final are copied asynchronously into the pinned host array that ``finish`` returns
    (float32 [n_frames,H,W]; torch's pinned-memory cache recycles it once the caller drops it), or into the
    caller's device tensor ``out`` (then no pinned memory is allocated and ``finish`` returns that tensor).

    Device memory is bounded: only a segment of ``8 + 22*chunk`` frames of the stitched sequence lives on the
    GPU (frames older than the 8-frame cross-fade tail are final and already on their way to the host); when
    a window would run past the segment, the tail is moved to its start.  ``edv_op_stitch_window`` addresses
    the sequence from a base pointer, so the segment is presented to it through a shifted (virtual) base."""

    SEGMENT_BYTES = 256 << 20

    def __init__(self, n_windows, n_frames, H, W, device, plan=None, out=None):
        from . import engine as _engine

        self._op = _engine.op_stitch_window
        self.nwin, self.n, self.k = n_windows, n_frames, 0
        self.hw = H * W
        chunk = max(1, min(n_windows, self.SEGMENT_BYTES // (STEP * H * W * 4)))
        self.cap = max(INFER_LEN, INTERP_LEN + STEP * chunk)
        self.seg = torch.empty(self.cap, H, W, dtype=torch.float32, device=device)
        self.base = 0                          # global frame index of seg[0]
        if plan is None:
            plan = _engine.stitch_plan(H, W)   # numpy's pairwise-sum tree for the 8*H*W overlap elements
        self.n_leaves = int(plan[0])
        self.plan = torch.from_numpy(plan).to(device)
        self.scratch = torch.empty(4 * int(plan[0] + plan[1]), dtype=torch.float32, device=device)
        self.scale_shift = torch.empty(n_windows, 2, dtype=torch.float32, device=device)
        self.out = out if out is not None else torch.empty(n_frames, H, W, dtype=torch.float32, pin_memory=True)

    def push(self, win):
        """win: [32,H,W] float32 device tensor = window ``self.k`` resized to the frame size."""
        k = self.k
        if k > 0:
            pos = INFER_LEN + STEP * (k - 1)                       # frames aligned so far
            if pos + STEP - self.base > self.cap:                  # would run past the segment: move the tail to its start
                tail = self.seg[pos - INTERP_LEN - self.base: pos - self.base].clone()
                self.seg[:INTERP_LEN].copy_(tail)
                self.base = pos - INTERP_LEN
        self._op(win, k, self.seg, self.plan, self.n_leaves, self.scratch, self.scale_shift, base_frame=self.base)
        self.k += 1
        lo, hi = final_frame_range(k, self.nwin, self.n)
        if hi > lo:
            self.out[lo:hi].copy_(self.seg[lo - self.base: hi - self.base], non_blocking=True)

    def finish(self):
        assert self.k == self.nwin
        torch.cuda.current_stream().synchronize()
        return self.out if self.out.is_cuda else self.out.numpy()


def _stitch_plan_or_none(H, W):
    """The on-GPU stitching needs 8*H*W < 2^24 (np.sum(ones) must stay exact in float32, edv_op_stitch_plan);
    larger frames (>= ~2.1 MP: 2048x1080, 4K) use the reference's numpy chain on the host instead."""
    from . import engine as _engine

    try:
        return _engine.stitch_plan(H, W)
    except _engine.EndoDAVError:
        return None


def _dist():
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized():
        return dist, dist.get_rank(), dist.get_world_size()
    return None, 0, 1


def frames_device(frames, device):
    """The device the driver runs on for CUDA frames, which is theirs, or None for host frames.  CUDA frames must be a
    uint8 tensor of logical shape [N,H,W,3] with positive strides (any layout, but no broadcast view); ``device`` may be
    "cuda" without an index or name the same device."""
    if not (isinstance(frames, torch.Tensor) and frames.is_cuda):
        return None
    if frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[3] != 3:
        raise ValueError("CUDA frames must be a uint8 [N,H,W,3] tensor, got %s %s" % (frames.dtype, tuple(frames.shape)))
    if any(st < 1 and d > 1 for st, d in zip(frames.stride(), frames.shape)):
        # a broadcast view (e.g. one grayscale plane expanded to three channels): the resize reads positive strides
        raise ValueError("CUDA frames must not be a broadcast view (strides %s); materialise it first" % (frames.stride(),))
    want = torch.device(device)
    if want.type != "cuda" or (want.index is not None and want != frames.device):
        raise ValueError("frames are on %s but device=%r names another device" % (frames.device, device))
    return frames.device


def infer_video_depth(model, frames, device="cuda", forward_window=None, distributed=True):
    """frames: uint8 [N,H,W,3] -> float32 [N,H,W] on rank 0 (other ranks return None).

    Host frames (a numpy array, or anything numpy can read) give a numpy array.  A CUDA uint8 tensor of any positive strides
    (an NCHW decoder batch as ``x.permute(0, 2, 3, 1)``, frame slices, crops) is read in place on its own device and
    gives a contiguous float32 tensor there, bit-identical to the host path on the same frames.

    ``forward_window(clip[1,32,3,h,w] float32 tensor, (H,W)) -> [32,H,W] float32 tensor`` can be
    injected by tests (index/stitch logic on CPU, host frames only); by default it is the model's CUDA engine
    with the final resize fused into the same launch sequence."""
    frames_dev = frames_device(frames, device)
    if frames_dev is None:
        frames = np.ascontiguousarray(frames)
    elif forward_window is not None:
        raise ValueError("forward_window takes host frames only")
    if frames.ndim != 4 or frames.shape[-1] != 3:
        raise ValueError("frames must be [N,H,W,3], got %s" % (tuple(frames.shape),))
    n, H, W = frames.shape[:3]
    ih, iw = model.image_shape
    new_w, new_h = resize_target(W, H, iw, ih)
    cache = _FrameCache(frames, new_w, new_h) if frames_dev is None else None

    def deliver(result):
        """the stitched frames of device input go back to their device in one upload"""
        return torch.from_numpy(result).to(frames_dev) if frames_dev is not None else result

    def sink():
        """the device tensor that receives the stitched frames of device input; None: the stitcher's pinned host array"""
        return torch.empty(n, H, W, dtype=torch.float32, device=frames_dev) if frames_dev is not None else None
    dist, rank, world = _dist() if distributed else (None, 0, 1)
    nwin = num_windows(n)
    mine = shard_windows(nwin, rank, world)

    if forward_window is None:
        dev = frames_dev if frames_dev is not None else torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("endodav_b200 has no CPU path (device=%r)" % (device,))
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        if next(model.parameters()).device != dev:
            model.to(dev)
        eng = model._ensure_engine(ih // 14, iw // 14)
        from . import engine as _engine

        gpu_pre = frames_dev is not None or os.environ.get("ENDODAV_PREPROCESS", "gpu").lower() != "host"
        if frames_dev is None and frames.dtype != np.uint8:
            # the reference accepts any dtype through ``.astype(np.float32) / 255`` (endodav.py:195); the GPU cubic
            # resize is written for uint8 frames, so other dtypes take the reference's host preprocessing path
            gpu_pre = False
        # two pinned staging buffers: the host fills window j+1 while the GPU runs window j.
        # gpu_pre (default): the raw uint8 frames of the window are uploaded (4x fewer bytes than the
        # resized float clip) and the reference's /255 + cv2 INTER_CUBIC resize + HWC->CHW runs in a
        # CUDA kernel (edv_op_cubic_resize_u8); ENDODAV_PREPROCESS=host keeps the reference's host path for host frames.
        # Device frames are neither staged nor uploaded: the resize reads them from the caller's tensor.
        # Windows are independent, so WB of them go through the network as one [WB,32,...] clip batch (the
        # engine's batched result is bit-identical to the clips run one by one, test_clip_batch_sweep_*):
        # at 224x280 four windows take 9.1 ms instead of 4 x 3.7 ms.
        gpu_stitch = os.environ.get("ENDODAV_STITCH", "gpu").lower() != "host"
        splan = _stitch_plan_or_none(H, W) if gpu_stitch else None
        if splan is None:
            gpu_stitch = False
        # default: 4 windows at 224x280 (measured best of 1/2/4/6/8 on a B200: 0.35/0.29/0.25/0.30/0.30 s for
        # 2000 frames), fewer at larger network resolutions (the workspace grows with WB*32 frames)
        wb_default = max(1, min(4, int(round(4.0 * 224 * 280 / (new_h * new_w)))))
        if world > 1:
            # few windows per rank: keep at least ~4 rounds so that the rank-0 tail (stitch + D2H of the LAST round) stays a
            # small share -- measured at 8 GPUs on the 2 000-frame video (12 windows per rank): 46.9 / 41.8 / 42.7 ms for 4 / 3 / 2
            wb_default = max(1, min(wb_default, -(-((nwin + world - 1) // world) // 4)))
        WB = max(1, int(os.environ.get("ENDODAV_WINDOW_BATCH", wb_default))) if (gpu_stitch or world > 1) else 1
        stager = None
        if gpu_pre:
            # the staging buffers hold raw frames: bound them by the FRAME size too (256 MB each; 1080p -> one window)
            WB = max(1, min(WB, (256 << 20) // (INFER_LEN * H * W * 3)))
            stager = _Stager(frames, n, mine, WB, H, W) if frames_dev is None else None
            pinned = None
        else:
            pinned = [torch.empty(WB, INFER_LEN, 3, new_h, new_w, dtype=torch.float32, pin_memory=True) for _ in range(2)]
        copied = [None, None]
        calls = [0]
        # device staging is allocated once and reused (two slots): besides saving allocator traffic this keeps the
        # external pointers of edv_forward stable, so the captured CUDA graph of the forward is replayed for every
        # window batch instead of re-launching ~190 kernels from the host
        dev_u8 = ([torch.empty(WB * INFER_LEN, H, W, 3, dtype=torch.uint8, device=dev) for _ in range(2)]
                  if stager is not None else None)
        dev_x = [torch.empty(WB * INFER_LEN, 3, new_h, new_w, dtype=torch.float32, device=dev) for _ in range(2)]
        dev_out = [None, None]

        def launch(j, nb=1, out=None):
            """enqueue windows mine[j:j+nb]: H2D of their frames, (cubic resize,) forward, resize back ->
            device tensor [nb*32,H,W]"""
            slot = calls[0] & 1
            calls[0] += 1
            x = dev_x[slot][: nb * INFER_LEN]
            if frames_dev is not None:
                idx = np.concatenate([window_frame_indices(mine[j + b], n) for b in range(nb)])
                _engine.op_cubic_resize_u8(frames, new_h, new_w, out=x, index=idx)
            else:
                if gpu_pre:
                    pslot, buf = stager.fetch(j, nb)
                    xu8 = dev_u8[slot][: nb * INFER_LEN]
                    xu8.copy_(buf, non_blocking=True)
                else:
                    if copied[slot] is not None:
                        copied[slot].synchronize()  # the earlier H2D copy out of this buffer has finished
                    buf = pinned[slot]
                    idx = np.concatenate([window_frame_indices(mine[j + b], n) for b in range(nb)])
                    flat = buf.view(WB * INFER_LEN, 3, new_h, new_w)
                    for i, src in enumerate(idx):
                        flat[i].copy_(torch.from_numpy(cache.get(int(src))))
                    x.copy_(flat[: nb * INFER_LEN], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record()
                if gpu_pre:
                    stager.uploaded(pslot, ev)
                    _engine.op_cubic_resize_u8(xu8, new_h, new_w, out=x)
                else:
                    copied[slot] = ev
            if out is None:
                if dev_out[slot] is None:
                    dev_out[slot] = torch.empty(WB * INFER_LEN, H, W, dtype=torch.float32, device=dev)
                out = dev_out[slot][: nb * INFER_LEN]
            eng.plan(nb, INFER_LEN, new_h, new_w, ih, iw)
            return eng.forward(x.view(nb, INFER_LEN, 3, new_h, new_w), resize_to=(H, W), want_pyramid=False, resized_out=out)[1]

        if world == 1 and gpu_stitch:
            # Single GPU, default: every window is aligned / cross-faded on the device right behind its forward
            # (edv_op_stitch_window, no host sync); the frames a window makes final are copied back through a
            # small pinned ring while the next windows run.
            with torch.cuda.device(dev):
                st = _GpuStitcher(nwin, n, H, W, dev, splan, sink())
                for j in range(0, nwin, WB):
                    nb = min(WB, nwin - j)
                    d = launch(j, nb).view(nb, INFER_LEN, H, W)
                    for b in range(nb):
                        st.push(d[b])
                return st.finish()
        if world == 1:
            # ENDODAV_STITCH=host -- the reference's numpy chain: stream the windows.  Window j+2 is enqueued before window j is handed to the
            # (strictly sequential, host-side) stitching, and every result comes back through a small
            # ring of pinned buffers, so GPU work, D2H copies and the numpy stitching overlap.
            AHEAD, RING = 2, 3
            ring = [torch.empty(INFER_LEN, H, W, dtype=torch.float32, pin_memory=True) for _ in range(RING)]
            done = [None] * RING

            def stream():
                with torch.cuda.device(dev):
                    def enqueue(j):
                        ring[j % RING].copy_(launch(j), non_blocking=True)
                        done[j % RING] = torch.cuda.Event()
                        done[j % RING].record()

                    for j in range(min(AHEAD, len(mine))):
                        enqueue(j)
                    for j in range(len(mine)):
                        if j + AHEAD < len(mine):
                            enqueue(j + AHEAD)   # reuses the slot of window j-1, which the consumer has finished with
                        done[j % RING].synchronize()
                        arr = ring[j % RING].numpy()
                        yield arr.copy() if j == 0 else arr   # window 0's frames are kept by reference in the output list

            return deliver(stitch_windows(stream(), n))

        per = (nwin + world - 1) // world
        if gpu_stitch and os.environ.get("ENDODAV_GATHER", "rounds").lower() != "single":
            # Default multi-GPU schedule: the gather to rank 0 is issued per round of WB windows per rank
            # (asynchronously, on NCCL's stream) instead of once at the end, and rank 0 stitches round r-1 and
            # copies its final frames to the host on a side stream while every rank computes round r.  Same
            # collective, same data, same stitching order k = 0,1,2,... -> bit-identical result; only the
            # serial tail (gather + 91 stitch steps + 655 MB D2H for config 3) shrinks to the last round.
            with torch.cuda.device(dev):
                side = torch.cuda.Stream(device=dev) if rank == 0 else None
                st = None
                if rank == 0:
                    dest = sink()                     # allocated on this stream, which hands the result to the caller
                    with torch.cuda.stream(side):
                        st = _GpuStitcher(nwin, n, H, W, dev, splan, dest)
                # Three rotating sets of gather buffers (round r uses set r % 3): bounded memory however long the video,
                # and stable pointers, so the forward's captured CUDA graph is replayed.  Set r % 3 is reused by round
                # r + 3 once (a) this rank has waited for round r's gather (its `send` is free) and (b) on rank 0 the
                # side stream has stitched round r out of its receive buffers (`consumed` event).
                POOL = 3
                sends = [torch.empty(WB, INFER_LEN, H, W, dtype=torch.float32, device=dev) for _ in range(POOL)]
                recvs = [[torch.empty(WB, INFER_LEN, H, W, dtype=torch.float32, device=dev) for _ in range(world)]
                         for _ in range(POOL)] if rank == 0 else None
                works = [None] * POOL
                consumed = [None] * POOL

                def consume(r, j0, nb, bufs, work):
                    with torch.cuda.stream(side):
                        work.wait()                                   # side stream waits for this round's gather
                        for s_ in range(nb):
                            for w_ in range(world):
                                if (j0 + s_) * world + w_ < nwin:
                                    st.push(bufs[w_][s_])
                        consumed[r % POOL] = torch.cuda.Event()
                        consumed[r % POOL].record(side)

                prev = None
                trace = [] if os.environ.get("ENDODAV_TRACE") else None     # host-side timeline of the rounds (ms since entry)
                t_entry = time.perf_counter()

                def mark(what):
                    if trace is not None:
                        trace.append("%s@%.1f" % (what, 1e3 * (time.perf_counter() - t_entry)))

                for r, j0 in enumerate(range(0, per, WB)):
                    nb = min(WB, per - j0)
                    have = max(0, min(nb, len(mine) - j0))             # real windows of this rank in the round
                    if works[r % POOL] is not None:
                        works[r % POOL].wait()                         # round r-3's gather has read this send buffer
                    if rank == 0 and consumed[r % POOL] is not None:
                        torch.cuda.current_stream().wait_event(consumed[r % POOL])
                    send = sends[r % POOL][:nb]
                    mark("r%d:ready" % r)
                    if have:
                        launch(j0, have, send[:have].view(have * INFER_LEN, H, W))
                    mark("launched")
                    if have < nb:
                        send[have:].zero_()
                    bufs = [t[:nb] for t in recvs[r % POOL]] if rank == 0 else None
                    work = dist.gather(send, bufs, dst=0, async_op=True)
                    works[r % POOL] = work
                    mark("gather")
                    if rank == 0:
                        if prev is not None:
                            consume(*prev)
                        prev = (r, j0, nb, bufs, work)
                        mark("consumed")
                if rank == 0:
                    consume(*prev)
                    mark("last-consume")
                    with torch.cuda.stream(side):
                        result = st.finish()
                    mark("finish")
                    torch.cuda.current_stream().synchronize()
                    mark("sync")
                    if trace is not None:
                        print("[endodav trace rank 0] " + " ".join(trace), flush=True)
                    return result
                for work in works:
                    if work is not None:
                        work.wait()
                torch.cuda.current_stream().synchronize()
                mark("sync")
                if trace is not None and rank in (1, world - 1):
                    print("[endodav trace rank %d] " % rank + " ".join(trace), flush=True)
                return None
        # ENDODAV_GATHER=single: every window's disparity is written straight into this rank's (padded) slice of
        # ONE gather issued after the last window
        with torch.cuda.device(dev):
            local_t = torch.empty(per, INFER_LEN, H, W, dtype=torch.float32, device=dev)
            for j in range(0, len(mine), WB):
                nb = min(WB, len(mine) - j)
                launch(j, nb, local_t[j:j + nb].view(nb * INFER_LEN, H, W))
            if len(mine) < per:
                local_t[len(mine):].zero_()
    else:
        local = []
        for k in mine:
            clip = torch.from_numpy(np.stack([cache.get(int(i)) for i in window_frame_indices(k, n)], 0)).unsqueeze(0)
            local.append(forward_window(clip, (H, W)).reshape(INFER_LEN, H, W).float())
        local_t = torch.stack(local, 0) if local else torch.empty(0, INFER_LEN, H, W, dtype=torch.float32)

    if world == 1:
        wins = local_t.cpu().numpy()
        return stitch_windows([wins[i] for i in range(nwin)], n)

    # one gather of per-window disparity to rank 0 (padded to the largest shard)
    per = (nwin + world - 1) // world
    if local_t.shape[0] == per:
        pad = local_t
    else:
        pad = torch.zeros(per, INFER_LEN, H, W, dtype=torch.float32, device=local_t.device)
        pad[: local_t.shape[0]] = local_t
    gathered = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
    dist.gather(pad, gathered, dst=0)
    if rank != 0:
        return None
    if forward_window is None and gpu_stitch:
        with torch.cuda.device(local_t.device):
            st = _GpuStitcher(nwin, n, H, W, local_t.device, splan, sink())
            for k in range(nwin):
                st.push(gathered[k % world][k // world])
            return st.finish()
    host = [g.cpu().numpy() for g in gathered]
    wins = [host[k % world][k // world] for k in range(nwin)]
    return deliver(stitch_windows(wins, n))
