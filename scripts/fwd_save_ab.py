"""Fused forward kernel at C3 size (4096 rays x 128): inference launch vs training launch (activation save + ReLU bitmasks).
Kernel-only CUDA-event times around the C-ABI call.  Never a benchmark."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from texpose_b200 import _C, synth  # noqa: E402
from texpose_b200.config import AttrDict, adapt_gan_opt  # noqa: E402
from texpose_b200.layers.nerf_static_transient_light import NeRF  # noqa: E402
import texpose_b200.mlp_tc as tc_mod  # noqa: E402

DEV = "cuda:0"
opt = adapt_gan_opt(device=DEV)
opt.b200 = AttrDict(mlp="bf16")
torch.manual_seed(0)
m = NeRF(opt).to(DEV)
B, R, N = 16, 256, 128
g = torch.Generator().manual_seed(4)
center = (torch.randn(B, R, 3, generator=g) * 0.02 + torch.tensor([0.3, 0.2, -8.0])).to(DEV)
ray = (torch.randn(B, R, 3, generator=g) * 0.05 + torch.tensor([0.0, 0.0, 1.0])).to(DEV)
depth = ((torch.rand(B, R, N, 1, generator=g) + torch.arange(N)[None, None, :, None]) / N * 2.5 + 6.7).to(DEV)
lt, ll = [t.to(DEV) for t in synth.latents(B)]

times = []
orig = _C.call


def timing_call(name, *a):
    if name == "tp_tc_nerf_stl_forward":
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig(name, *a)
        e1.record()
        times.append((e0, e1))
    else:
        orig(name, *a)


for mod in (tc_mod,):
    mod._C.call = timing_call
_C.call = timing_call


def run(train, iters=12):
    times.clear()
    for _ in range(iters):
        if train:
            m.train()
            out = m.forward_samples(opt, center, ray, depth, lt, ll, mode="train")
        else:
            with torch.no_grad():
                out = m.forward_samples(opt, center, ray, depth, lt, ll, mode="val")
        del out
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in times[2:])
    return ms[len(ms) // 2], ms[0]


for label, train in (("inference", False), ("training (save)", True), ("inference", False), ("training (save)", True)):
    med, best = run(train)
    print(f"{label:18s} kernel median {med * 1e3:8.1f} us   best {best * 1e3:8.1f} us", flush=True)
