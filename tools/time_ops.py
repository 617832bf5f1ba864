"""CUDA-event timing of single kernels at the BASELINE config-2 shapes (development aid).
  python tools/time_ops.py attn [reps]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from endodav_b200 import engine as eng  # noqa: E402

dt = torch.float16
M = 32 * 1370
g = torch.Generator().manual_seed(0)


def rnd(*s, scale=1.0):
    return (torch.randn(*s, generator=g) * scale).to(dt).cuda()


def timeit(fn, reps=20):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


which = sys.argv[1]
if which == "attn":
    qkv = rnd(M, 1152, scale=0.5)
    ref = None
    us = timeit(lambda: eng.op_attention(qkv, 32, 1370, 6))
    out = eng.op_attention(qkv, 32, 1370, 6).float()
    t = qkv[:1370 * 2].float().reshape(2, 1370, 3, 6, 64).permute(2, 0, 3, 1, 4)
    r = ((t[0] @ t[1].transpose(-1, -2)).softmax(-1) @ t[2]).transpose(1, 2).reshape(2 * 1370, 384)
    print("attn: %.1f us  (%.1f TFLOP/s)  max err vs fp32 %.3g" % (
        us, 4 * 32 * 6 * 1370 * 1370 * 64 / us / 1e6, float((out[:2740] - r).abs().max())))
elif which in ("qkv", "fc1", "fc2", "proj"):
    N, K, act = {"qkv": (1152, 384, 0), "fc1": (1536, 384, 1), "fc2": (384, 1536, 0), "proj": (384, 384, 0)}[which]
    A, W, b = rnd(M, K), rnd(N, K, scale=K ** -0.5), torch.zeros(N).cuda()
    us = timeit(lambda: eng.op_linear(A, W, b, act))
    got = eng.op_linear(A[:512], W, b, act).float()
    ref = torch.nn.functional.linear(A[:512].float(), W.float())
    ref = torch.nn.functional.gelu(ref) if act else ref
    print("%s: %.1f us (%.0f TFLOP/s) max err %.3g" % (which, us, 2.0 * M * N * K / us / 1e6, float((got - ref).abs().max())))
elif which == "ln":
    x = torch.randn(M, 384, generator=g).cuda()
    gam, bet = torch.ones(384).cuda(), torch.zeros(384).cuda()
    # rotate over 4 inputs so that successive launches do not find x in L2
    xs = [x.clone() for _ in range(4)]
    it = [0]

    def f():
        it[0] += 1
        eng.op_layernorm(xs[it[0] & 3], gam, bet, 1e-6, dt)

    us = timeit(f, 40)
    got = eng.op_layernorm(x[:64], gam, bet, 1e-6, dt).float()
    ref = torch.nn.functional.layer_norm(x[:64], (384,), gam, bet, 1e-6)
    print("ln: %.1f us (%.0f GB/s incl. output alloc) max err %.3g" % (us, M * 384 * 6 / us / 1e3, float((got - ref).abs().max())))
