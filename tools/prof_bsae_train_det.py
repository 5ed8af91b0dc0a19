"""Timing of the deterministic b_sae backward (model.deterministic = True, qsae_bsae_backward; DESIGN 5.10).

    python tools/prof_bsae_train_det.py --out profiles/r8_bsae_train_det.md

b_sae 512 -> 32768, n_bits = 4, k = 32 and 65, B = 4096 and 65536:
1. qsae_bsae_backward on its own by CUDA events, alternating with the atomic backward that is the default
   (_BinarySAEFn.backward with deterministic = False: a zero-filled [H, D] G, rows_scatter_add into it,
   bsae_logit_grad, column_sum, rows_gather_dot, two zero-filled rows_scatter_add targets), on the same inputs in the
   same run. Neither computes grad x.
2. The whole trainer step (forward, 0.5 * mse + lambda * polarize, backward, Adam) with each backward, fast forward,
   and exact forward at B = 4096 (its forward after a weight update takes seconds at 65536).
3. Each kernel of both backwards over many launches, from torch.profiler in a separate pass: the fused
   bsae_latent_reduce_kernel against the bsae_logit_grad + atomic scatters + zero fills it replaces.
4. Both backwards on a skewed dictionary: one latent wins every row, 32 more get a raised bias.
Bytes from shapes: the fused pass reads the logits and writes their gradient, 2 H D n 4 bytes, writes grad W_enc,
H D 4, and reads the x and g rows of every entry, B k 2 D 4 (partly from L2). The card's name, power limit and
maximum SM clock are read in the same run and printed with the numbers.
"""
import argparse
import subprocess
import sys
import time
from pathlib import Path

import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

import quantizedsae_b200 as Q  # noqa: E402
from quantizedsae_b200 import _lib as L  # noqa: E402

PEAK_HBM = 7.7e12
D, H, NB = 512, 32768, 4
LAM = 0.1


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name()


def time_ms(fn, n, min_s=0.5):
    """Mean ms per call over a window of at least n calls and at least min_s seconds."""
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    n = max(n, int(min_s / max(time.perf_counter() - t0, 1e-6)) + 1)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def model(dev, B, k, exact, skew=False, seed=5):
    torch.manual_seed(seed)
    m = Q.BinarySAE(D, H, 4.0, NB)
    m.k = (k + 0.5) / H
    m.to(dev)
    m.exact, m.autograd, m.return_dense = exact, True, False
    if skew:
        with torch.no_grad():
            m.encoder[0].bias.zero_()
            m.encoder[0].bias[0] = 100.0
            m.encoder[0].bias[1:33] = 0.45
    x = torch.randn((B, D), device=dev).bfloat16().float()
    return m, x


def atomic(x, sl, g, rows, logits, q, gp):
    """_BinarySAEFn.backward's default path, without grad x."""
    G = torch.zeros((H, D), device=x.device)
    L.rows_scatter_add(sl.values, sl.indices, g, G, scale=q)
    glog = torch.empty_like(logits)
    L.bsae_logit_grad(logits, G, D, NB, gp, glog, accumulate=False)
    gbd = L.column_sum(g)
    gv = L.rows_gather_dot(g, rows, sl.indices, scale=q)
    gwe = torch.zeros((H, D), device=x.device)
    gbe = torch.zeros((H,), device=x.device)
    L.rows_scatter_add(gv, sl.indices, x, gwe, scale=1.0, dst_col=gbe)
    return gwe, gbe, glog, gbd


def det(x, sl, g, rows, logits, q, gp):
    return L.bsae_backward(x, sl.values, sl.indices, g, rows, logits, q, gp, None, NB, False)[:4]


def inputs(m, x):
    with torch.no_grad():
        sl = m.encode_topk(x)
    g = torch.randn_like(x) / x.numel()
    dec = m.decoder
    return sl, g, dec._soft_rows(), dec.weight.detach(), float(dec.quantization_step), torch.tensor(LAM, device=x.device)


def alternate(args, iters):
    t_det, t_atom = [], []
    for _ in range(3):
        t_det.append(time_ms(lambda: det(*args), iters))
        t_atom.append(time_ms(lambda: atomic(*args), iters))
    a, b = det(*args), atomic(*args)
    diff = max(float((p - q).abs().max() / q.abs().max().clamp_min(1e-30)) for p, q in zip(a, b))
    return min(t_det), min(t_atom), diff


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=50)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    lines = [f"# b_sae deterministic backward (512 -> 32768, n_bits = 4)", "", f"Card: {card()}", ""]
    lines += ["## Backward call, same inputs", "",
              "| B | k | deterministic ms | atomic ms | det / atomic | det GB/s (2 H D n 4 + H D 4 + B k 2 D 4) | "
              "max rel diff |", "|---|---|---|---|---|---|---|"]
    prof = []
    for B in (4096, 65536):
        for k in (32, 65):
            m, x = model(dev, B, k, exact=False)
            args = (x, *inputs(m, x))
            td, ta, diff = alternate(args, a.iters)
            nbytes = 2 * H * D * NB * 4 + H * D * 4 + B * k * 2 * D * 4
            lines.append(f"| {B} | {k} | {td:.3f} | {ta:.3f} | {td / ta:.2f} | {nbytes / td / 1e6:.0f} | {diff:.1e} |")
            print(lines[-1], flush=True)
            prof.append((f"B={B} k={k}", args))
    lines += ["", "Best of three alternating windows, each of at least 0.5 s and 50 calls. max rel diff: the largest |det - atomic| over "
              "max |atomic| across the four gradients.", ""]
    # trainer step
    lines += ["## Trainer step (forward, 0.5 mse + 0.1 polarize, backward, Adam)", "",
              "| B | k | forward | deterministic step ms | atomic step ms |", "|---|---|---|---|---|"]
    for B in (4096, 65536):
        for k in (32, 65):
            for exact in ((False, True) if B == 4096 else (False,)):     # exact: ~0.2 s (4096) to ~2 s (65536) a step
                m, x = model(dev, B, k, exact)
                opt = torch.optim.Adam(m.parameters(), lr=1e-4)

                def step():
                    opt.zero_grad(set_to_none=True)
                    _, r, pol = m(x)
                    (0.5 * F.mse_loss(r, x) + LAM * pol).backward()
                    opt.step()

                n = a.iters if not exact else 3
                ts = {}
                for _ in range(2):
                    for flag in (True, False):
                        m.deterministic = flag
                        ts.setdefault(flag, []).append(time_ms(step, n))
                lines.append(f"| {B} | {k} | {'exact' if exact else 'fast'} | {min(ts[True]):.3f} | {min(ts[False]):.3f} |")
                print(lines[-1], flush=True)
    lines += ["", "Steps with weight updates in between: each forward sees new weights (a fresh bf16 cast and sample).", ""]
    # exact forward on unchanged weights, for comparison with the step
    m, x = model(dev, 4096, 32, exact=True)
    with torch.no_grad():
        f_same = time_ms(lambda: m(x), a.iters)
    lines += [f"Exact forward on unchanged weights, B = 4096, k = 32, no_grad: {f_same:.3f} ms.", ""]
    # skewed dictionary
    lines += ["## Skewed dictionary (latent 0 in every row, latents 1..32 with a raised bias), k = 32", "",
              "| B | deterministic ms | atomic ms | rows of latent 0 | mean share of latents 1..32 |", "|---|---|---|---|---|"]
    for B in (4096, 65536):
        m, x = model(dev, B, 32, exact=False, skew=True)
        args = (x, *inputs(m, x))
        td, ta, _ = alternate(args, a.iters)
        c = torch.bincount(args[1].indices.reshape(-1).long(), minlength=H)
        lines.append(f"| {B} | {td:.3f} | {ta:.3f} | {int(c[0])} | {float(c[1:33].float().mean()) / B:.2f} |")
        print(lines[-1], flush=True)
        if B == 4096:
            prof.append(("skew B=4096 k=32", args))
    # per-kernel times, a separate profiled pass
    lines += ["", "## Kernels of both backwards (torch.profiler)", "",
              "| case | path | kernel | calls | mean us |", "|---|---|---|---|---|"]
    from torch.profiler import ProfilerActivity, profile

    for label, args in prof:
        for path, fn in (("deterministic", det), ("atomic", atomic)):
            for _ in range(3):
                fn(*args)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as p:
                for _ in range(a.iters):
                    fn(*args)
                torch.cuda.synchronize()
            for ev in p.key_averages():
                t = getattr(ev, "device_time_total", 0) or getattr(ev, "cuda_time_total", 0)
                if t <= 0 or ev.key.startswith("cuda"):
                    continue
                name = ev.key.replace("void ", "").replace("qsae::(anonymous namespace)::", "").split("(")[0]
                lines.append(f"| {label} | {path} | `{name[:70]}` | {ev.count} | {t / ev.count:.1f} |")
                print(lines[-1], flush=True)
    text = "\n".join(lines) + "\n"
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(text)
    print(text)


if __name__ == "__main__":
    main()
