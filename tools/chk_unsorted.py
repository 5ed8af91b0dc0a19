import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from quantizedsae_b200 import _lib as L
B, H, D, k = (int(sys.argv[2]) if len(sys.argv) > 2 else 512), 131072, 512, int(sys.argv[1]) if len(sys.argv) > 1 else 2097
dev = torch.device("cuda:0")
g = torch.Generator(device=dev).manual_seed(0)
x = torch.randn((B, D), device=dev, generator=g).bfloat16().float()
W = ((torch.rand((H, D), device=dev, generator=g) * 2 - 1) * (6.0 / (H + D)) ** 0.5).bfloat16().float()
b = torch.zeros(H, device=dev)
Wb = L.cast_bf16(W)
sample = L.prepare_sample(Wb, b)
outs = {}
for u in ("0", "1"):
    os.environ["QSAE_TOPK_UNSORTED"] = u
    L.check(L.load().qsae_reload_tuning())
    v, i, f = L.encode_topk(x, Wb, None, b, k, exact=False, want_flags=True, sample=sample)
    torch.cuda.synchronize()
    outs[u] = (v.clone(), i.clone())
    cand = L.pack_candidates(v, i).unsqueeze(0).contiguous()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    L.merge_candidates(cand, H, k); torch.cuda.synchronize()
    e0.record(); mv, mi = L.merge_candidates(cand, H, k); e1.record(); torch.cuda.synchronize()
    print("unsorted", u, "merge ms", e0.elapsed_time(e1), "min idx", int(i.min()), "dups per row max",
          int(max(k - len(set(r.tolist())) for r in i[:8].cpu())))
    outs["m" + u] = (mv.clone(), mi.clone())
s0 = torch.sort(outs["0"][1], dim=1).values
s1 = torch.sort(outs["1"][1], dim=1).values
print("local sets equal:", bool(torch.equal(s0, s1)))
print("merged sets equal:", bool(torch.equal(torch.sort(outs["m0"][1], 1).values, torch.sort(outs["m1"][1], 1).values)))
