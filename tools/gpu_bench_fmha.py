"""FMHA timings at the shapes of the sampling paths: DiT-L/2 self-attention (16 samples) and cond-only
cross-attention (8 samples, 77 text tokens), DiT2 decoder in-plane (24 x 256 tokens) and global (8 x 768)
attention at 8 latents, and I23D self-attention over 768 latent + 256 DINO tokens (16 samples)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from ln3diff_b200 import ops

dev = "cuda"
torch.manual_seed(0)
H, D = 16, 16 * 64


def timeit(fn, iters=30):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3


def self_attn(B, L):
    qkv = (torch.randn(B, L, 3 * D, device=dev) * 0.5).bfloat16()
    return lambda: ops.fmha(qkv[:, :, :D], qkv[:, :, D:2 * D], qkv[:, :, 2 * D:], H)


qc = (torch.randn(8, 768, D, device=dev) * 0.5).bfloat16()
kvc = (torch.randn(8, 77, 2 * D, device=dev) * 0.5).bfloat16()
qi = (torch.randn(16, 768, 3 * D, device=dev) * 0.5).bfloat16()
kd = (torch.randn(16, 256, 2 * D, device=dev) * 0.5).bfloat16()
cases = [
    ("self(16x16x768x768)", 16 * 768 * 768, self_attn(16, 768)),
    ("cross(8x16x768x77)", 8 * 768 * 77, lambda: ops.fmha(qc, kvc[:, :, :D], kvc[:, :, D:], H)),
    ("inplane(24x16x256x256)", 24 * 256 * 256, self_attn(24, 256)),
    ("global(8x16x768x768)", 8 * 768 * 768, self_attn(8, 768)),
    ("i23d(16x16x768x(768+256))", 16 * 768 * 1024,
     lambda: ops.fmha(qi[:, :, :D], qi[:, :, D:2 * D], qi[:, :, 2 * D:], H, k2=kd[:, :, :D], v2=kd[:, :, D:])),
]
for name, qk_pairs, fn in cases:
    us = timeit(fn)
    print(f"{name} {us:.1f} us ({4.0 * H * qk_pairs * 64 / us / 1e6:.0f} TF/s)", flush=True)
