"""Timing / profiling driver for the t_sae path: python tests/prof_tsae.py [B] [iters] [exact]"""
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from quantizedsae_b200 import _lib as L  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 10
exact = bool(int(sys.argv[3])) if len(sys.argv) > 3 else False
H, D = 32768, 512
dev = torch.device("cuda:0")
g = torch.Generator(device=dev).manual_seed(0)
We = ((torch.rand((H, D), device=dev, generator=g) * 2 - 1) * (6.0 / (H + D)) ** 0.5).bfloat16().float()
be = torch.zeros(H, device=dev)
Wd = 0.4824 * torch.randn((D, H), device=dev, generator=g)
xs = [torch.randn((B, D), device=dev, generator=g).bfloat16().float() for _ in range(3)]
w_parts = L.split_bf16x3(We) if exact else (L.cast_bf16(We),)
t_bf16, _ = L.pack_ternary(Wd)
for i in range(3):
    h, r = L.tsae_forward(xs[i % 3], w_parts, be, t_bf16, exact)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
k0.record(); k1.record()
L.check(L.load().qsae_set_encode_kernel_events(k0.cuda_event, k1.cuda_event))
e0.record()
for i in range(iters):
    h, r = L.tsae_forward(xs[i % 3], w_parts, be, t_bf16, exact)
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / iters
L.check(L.load().qsae_set_encode_kernel_events(None, None))
print(f"dense encoder kernel: {k0.elapsed_time(k1) * 1e3:.1f} us")
print(f"t_sae fwd B={B} exact={exact}: {ms:.3f} ms/step, {B / ms * 1e3 / 1e6:.2f} Mtok/s, "
      f"{4.0 * B * H * D / ms / 1e9:.0f} TFLOP/s (two GEMMs)")
hi, lo = L.split_bf16(h)
for name, fn in (("decode 1-pass", lambda: L.decode_dense(hi, None, t_bf16)), ("decode 2-pass", lambda: L.decode_dense(hi, lo, t_bf16))):
    fn(); torch.cuda.synchronize()
    e0.record()
    for i in range(iters):
        fn()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    print(f"  {name}: {ms:.3f} ms, {2.0 * B * H * D / ms / 1e9:.0f} TFLOP/s per pass-equivalent")
