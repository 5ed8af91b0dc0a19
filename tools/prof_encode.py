"""Timing / profiling driver for the fused encoder (GPU box). python tests/prof_encode.py B k iters"""
import os, sys
from pathlib import Path
import torch
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from quantizedsae_b200 import _lib as L
B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
k = int(sys.argv[2]) if len(sys.argv) > 2 else 32
iters = int(sys.argv[3]) if len(sys.argv) > 3 else 20
H, D = 32768, 512
dev = torch.device("cuda:0")
g = torch.Generator(device=dev).manual_seed(0)
x = torch.randn((B, D), device=dev, generator=g).bfloat16().float()
W = ((torch.rand((H, D), device=dev, generator=g) * 2 - 1) * (6.0 / (H + D)) ** 0.5).bfloat16().float()
b = torch.zeros(H, device=dev)
Wb = L.cast_bf16(W)
sample = L.prepare_sample(Wb, b) if os.environ.get('QSAE_NO_SAMPLE') is None else None
for _ in range(3):
    L.encode_topk(x, Wb, None, b, k, sample=sample)
torch.cuda.synchronize()
s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
s.record()
for _ in range(iters):
    L.encode_topk(x, Wb, None, b, k, sample=sample)
e.record()
torch.cuda.synchronize()
t = s.elapsed_time(e) / iters
print(f"B={B} k={k}: {t*1e3:.1f} us  {2.0*B*H*D/t/1e9:.1f} TFLOP/s  {B/t/1e3:.2f} Mtok/s", flush=True)
