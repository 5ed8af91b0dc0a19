"""Timing of the baseline_sae training step (quantizedsae_b200/training.py `baseline_forward`, DESIGN 5.10).

    python tools/prof_baseline_train.py --out profiles/r7_baseline_train.md

baseline_sae 512 -> 32768, k = 32 (BASELINE config 2), B = 4096 and 65536, exact and fast forward:
1. forward with grad (one autograd node), loss.backward() alone, and the whole trainer step (forward, 0.5 * mse,
   backward, normalize_decoder_weights, Adam), by CUDA events over many steps.
2. qsae_baseline_backward on its own by events, alternating with the composition of existing kernels it replaces
   (rows_gather_dot for gv, two zero-filled [H, D] rows_scatter_add targets, the [H, D] -> [D, H] transpose and its
   add into the gradient), on the same inputs in the same run.
3. Each kernel of the backward over many launches, from torch.profiler in a separate pass.
4. The same backward on a skewed dictionary: one latent wins every row, 32 more get a raised bias (their share of
   the rows is printed).
Bytes from shapes: the latent-major pass reads the x and g rows of every entry, B k 2 D 4 bytes (mostly from L2), and
writes both weight gradients once, 2 H D 4 bytes to HBM (7.7 TB/s data-sheet figure). The card's name and power limit
are read in the same run and printed with the numbers.
"""
import argparse
import subprocess
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

import quantizedsae_b200 as Q  # noqa: E402
from quantizedsae_b200 import _lib as L  # noqa: E402

PEAK_HBM = 7.7e12
D, H, K = 512, 32768, 32


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name()


def time_ms(fn, n):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def model(dev, B, exact, skew=False, seed=5):
    torch.manual_seed(seed)
    m = Q.BaselineSparseAutoencoder(D, H).to(dev)
    m.exact, m.autograd = exact, True
    if skew:
        with torch.no_grad():
            m.encoder[0].bias.zero_()
            m.encoder[0].bias[0] = 100.0
            m.encoder[0].bias[1:33] = 0.45
    x = torch.randn((B, D), device=dev).bfloat16().float()
    return m, x


def composition(x, sl, g, rows, w_enc):
    """The same gradients from the existing kernels (atomic scatters into [H, D] scratch, then a transpose)."""
    gv = L.rows_gather_dot(g, rows, sl.indices)
    gwe = torch.zeros((H, D), device=x.device)
    gbe = torch.zeros((H,), device=x.device)
    L.rows_scatter_add(gv, sl.indices, x, gwe, scale=1.0, dst_col=gbe)
    M = torch.zeros((H, D), device=x.device)
    L.rows_scatter_add(sl.values, sl.indices, g, M, scale=1.0)
    gwd = torch.zeros((D, H), device=x.device)
    gwd.add_(L.transpose(M))
    return gwe, gbe, gwd, L.column_sum(g)


def backward_call(x, sl, g, rows, w_enc):
    return L.baseline_backward(x, sl.values, sl.indices, g, None, None, w_enc, rows, want_grad_x=False)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=50)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    lines = [f"# baseline_sae training step (512 -> 32768, k = 32)", "", f"Card: {card()}", ""]
    lines += ["## Step and backward", "",
              "| B | forward | fwd (grad) ms | loss.backward() ms | trainer step ms | backward call ms | composition ms | "
              "backward GB/s (B k 2 D 4 + 2 H D 4) | HBM-write floor ms |", "|---|---|---|---|---|---|---|---|---|"]
    prof_rows = []
    for B in (4096, 65536):
        for exact in (True, False):
            m, x = model(dev, B, exact)
            opt = torch.optim.Adam(m.parameters(), lr=1e-4)
            fwd = time_ms(lambda: m(x), a.iters)

            def fwd_bwd():
                m.zero_grad(set_to_none=True)
                _, r = m(x)
                (0.5 * F.mse_loss(r, x)).backward()

            fb = time_ms(fwd_bwd, a.iters)

            def step():
                opt.zero_grad(set_to_none=True)
                _, r = m(x)
                (0.5 * F.mse_loss(r, x)).backward()
                m.normalize_decoder_weights()
                opt.step()

            st = time_ms(step, a.iters)
            with torch.no_grad():
                sl = m.encode_topk(x)
            g = torch.randn_like(x)
            rows, w = m._dec_rows(), m.encoder[0].weight.detach()
            # alternate the two so both see the same machine state
            t_new, t_old = [], []
            for _ in range(3):
                t_new.append(time_ms(lambda: backward_call(x, sl, g, rows, w), a.iters))
                t_old.append(time_ms(lambda: composition(x, sl, g, rows, w), a.iters))
            new, old = min(t_new), min(t_old)
            ref = composition(x, sl, g, rows, w)
            got = backward_call(x, sl, g, rows, w)
            diff = max(float((p - q).abs().max() / q.abs().max().clamp_min(1e-30)) for p, q in zip(got[:4], ref))
            nbytes = B * K * 2 * D * 4 + 2 * H * D * 4
            lines.append(f"| {B} | {'exact' if exact else 'fast'} | {fwd:.3f} | {fb - fwd:.3f} | {st:.3f} | {new:.3f} | "
                         f"{old:.3f} | {nbytes / new / 1e6:.0f} | {2 * H * D * 4 / PEAK_HBM * 1e3:.4f} |")
            print(lines[-1], f"(composition agrees to {diff:.1e} of max |grad|)", flush=True)
            if exact:
                prof_rows.append((B, x, sl, g, rows, w))
    lines += ["", "Backward call and composition: the best of three alternating windows of "
              f"{a.iters} calls each. The composition's atomics make it non-deterministic; the two agree to fp32 "
              "rounding (printed in the run log).", ""]
    # skewed dictionary
    lines += ["## Skewed dictionary (latent 0 in every row, latents 1..32 with a raised bias)", "",
              "| B | backward call ms | composition ms | rows of latent 0 | mean share of latents 1..32 |", "|---|---|---|---|---|"]
    for B in (4096, 65536):
        m, x = model(dev, B, False, skew=True)
        with torch.no_grad():
            sl = m.encode_topk(x)
        g = torch.randn_like(x)
        rows, w = m._dec_rows(), m.encoder[0].weight.detach()
        t_new, t_old = [], []
        for _ in range(3):
            t_new.append(time_ms(lambda: backward_call(x, sl, g, rows, w), a.iters))
            t_old.append(time_ms(lambda: composition(x, sl, g, rows, w), a.iters))
        c = torch.bincount(sl.indices.reshape(-1).long(), minlength=H)
        lines.append(f"| {B} | {min(t_new):.3f} | {min(t_old):.3f} | {int(c[0])} | {float(c[1:33].float().mean()) / B:.2f} |")
        print(lines[-1], flush=True)
    # per-kernel times, a separate profiled pass
    lines += ["", "## Kernels of the backward (torch.profiler, uniform dictionary, exact forward)", "",
              "| B | kernel | calls | mean us |", "|---|---|---|---|"]
    from torch.profiler import ProfilerActivity, profile

    for B, x, sl, g, rows, w in prof_rows:
        for _ in range(3):
            backward_call(x, sl, g, rows, w)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as p:
            for _ in range(a.iters):
                backward_call(x, sl, g, rows, w)
            torch.cuda.synchronize()
        for ev in p.key_averages():
            if "bwd_" in ev.key or "memset" in ev.key.lower():
                name = ev.key.replace("void ", "").replace("qsae::(anonymous namespace)::", "").split("(")[0]
                t = getattr(ev, "device_time_total", 0) or getattr(ev, "cuda_time_total", 0)
                lines.append(f"| {B} | `{name}` | {ev.count} | {t / ev.count:.1f} |")
                print(lines[-1], flush=True)
    text = "\n".join(lines) + "\n"
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(text)
    print(text)


if __name__ == "__main__":
    main()
