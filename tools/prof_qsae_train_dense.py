"""Timing of the q_sae decoder-side training step at any activity (quantizedsae_b200/training.py, DESIGN 5.10).

    python tools/prof_qsae_train_dense.py --out profiles/r6_qsae_train_dense.md

q_sae 512 -> 32768, n_bits = 4, B = 4096 (the BASELINE shape):
1. The untrained model (zero encoder bias, ~50 % active), exact and fast mode: the whole decoder-side step
   (qsae_trainer_decoder_grads) by CUDA events, and its stages in a separate torch.profiler pass: the dense forward
   with its mask, the gradient parts, the mask^T g product with the STE epilogue, z2, the secant step. The product's
   rate counts 2 B H D per bf16 product (1 product fast, 3 exact) against the 2250 TFLOP/s bf16 dense data-sheet
   figure; its memory floor is the read-modify-write of grad_w / grad_w_mirror and the reads of w / w_mirror (24 H D
   bytes) plus the operands, against 7.7 TB/s. The unfused alternative (one wgrad product writing M, then the finish
   kernel of the sparse route) is timed beside the fused product for one level in fast mode.
2. The sparse / dense crossover: models with encoder biases set for L0 = 33 .. 16384 (z ~ N(b, 2 D / (H + D)) for
   xavier weights and unit x), the step through (a) the active lists and the scatter, (b) the same lists scattered
   into a mask and the product, (c) the dense forward and the product.
The card's name and power limit are read in the same run and printed with the numbers.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import torch
from scipy.stats import norm

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

import quantizedsae_b200 as Q  # noqa: E402
from quantizedsae_b200 import _lib as L  # noqa: E402
from quantizedsae_b200 import training as TR  # noqa: E402
from quantizedsae_b200.analysis import _scatter_lists  # noqa: E402

PEAK_BF16 = 2250e12
PEAK_HBM = 7.7e12
D, H, NB, B = 512, 32768, 4, 4096


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


def model(dev, enc_bias, seed=3):
    torch.manual_seed(seed)
    with torch.device(dev):
        m = Q.QuantizedMatryoshkaSAE(D, H, 32, abs_range=4.0, n_bits=NB)
    with torch.no_grad():
        m.encoder[0].bias.fill_(enc_bias)
    return m


def kernel_times(fn, names):
    """-> {kernel name fragment: mean ms per call} over 5 calls, from a torch.profiler pass of its own"""
    fn()
    torch.cuda.synchronize()
    acts = [torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts) as prof:
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in names}
    for ev in prof.key_averages():
        for k in names:
            if k in ev.key:
                out[k] += ev.device_time_total / 1e3 / 5     # device_time_total: microseconds
    return out


def init_rows(dev):
    rows = []
    x = torch.randn((B, D), device=dev, generator=torch.Generator(device=dev).manual_seed(4))
    for exact in (True, False):
        m = model(dev, 0.0)
        m.exact = exact

        def step():
            m.zero_grad(set_to_none=False)
            TR.qsae_trainer_decoder_grads(m, x)

        step()
        assert m.last_path == "dense"
        step_ms = time_ms(step, 10)
        out = m.forward_dense_active(x)
        mask = out["active_mask"]
        grads = [(r - x) / float(B * D) for r in out["reconstruction_levels"]]

        def ste():
            TR.qsae_ste_backward(m.decoder, mask, grads, exact=exact)

        ste_ms = time_ms(ste, 20)
        fwd_ms = time_ms(lambda: m.forward_dense_active(x), 10)
        names = ["matryoshka_ste_dense_kernel", "mask_column_count_kernel", "split_bf16x3_kernel", "cast_bf16_kernel",
                 "matryoshka_grad_finish_kernel"]
        kt = kernel_times(step, names)
        n_prod = 3 if exact else 1
        flop = 2.0 * B * H * D * n_prod
        t_prod = kt["matryoshka_ste_dense_kernel"]
        bytes_prod = 24.0 * H * D + 2.0 * B * H + 2.0 * n_prod * NB * B * D
        rows.append(dict(what="init step", exact=exact, active_fraction=float(mask.float().mean()), step_ms=step_ms,
                         dense_forward_with_mask_ms=fwd_ms, ste_backward_ms=ste_ms,
                         kernels_ms={k: round(v, 4) for k, v in kt.items()},
                         product_tflops=flop / (t_prod / 1e3) / 1e12 if t_prod else None,
                         product_share_of_bf16_peak=flop / PEAK_BF16 / (t_prod / 1e3) if t_prod else None,
                         product_floor_mma_ms=flop / PEAK_BF16 * 1e3, product_floor_hbm_ms=bytes_prod / PEAK_HBM * 1e3,
                         z2_floor_hbm_ms=2.0 * B * H / PEAK_HBM * 1e3))
        if not exact:
            # unfused pair for one level (n_levels = 1): wgrad writes M [H, D], the finish kernel applies the STE factor
            g16 = L.cast_bf16(grads[0].contiguous())
            gw = torch.zeros((H, D), device=dev)
            gwm = torch.zeros((H, D), device=dev)
            _, alpha = m.decoder._packed()
            w, wm = m.decoder.weight.detach(), m.decoder.weight_mirror.detach()

            def unfused():
                M = L.wgrad([mask], [g16])
                L.matryoshka_backward_finish(w, wm, M, None, alpha, [0, H], 0.0, 0, gw, gwm)

            def fused():
                L.matryoshka_backward_dense(mask, [grads[0].contiguous()], [0, H], w, wm, alpha, False, gw, gwm)

            ku = kernel_times(unfused, ["wgrad_kernel", "matryoshka_grad_finish_kernel"])
            kf = kernel_times(fused, ["matryoshka_ste_dense_kernel"])
            rows.append(dict(what="fused vs unfused, one level, fast", fused_product_ms=kf["matryoshka_ste_dense_kernel"],
                             unfused_wgrad_ms=ku["wgrad_kernel"], unfused_finish_ms=ku["matryoshka_grad_finish_kernel"],
                             unfused_total_ms=ku["wgrad_kernel"] + ku["matryoshka_grad_finish_kernel"]))
        del m
        torch.cuda.empty_cache()
    return rows


def crossover_rows(dev):
    rows = []
    x = torch.randn((B, D), device=dev, generator=torch.Generator(device=dev).manual_seed(5))
    sigma = (2.0 * D / (H + D)) ** 0.5
    for l0 in (33, 128, 256, 512, 1024, 2048, 4096, 8192, 16384):
        m = model(dev, float(sigma * norm.ppf(l0 / H)))
        r = m._forward_lists(x, 256)
        row = dict(what="crossover", target_L0=l0)
        if r is not None:
            mean_l0 = float(r["level_counts"].sum()) / B
            row.update(L0=mean_l0, L0_over_H=mean_l0 / H)

            def sparse():
                m.zero_grad(set_to_none=False)
                o = m._forward_lists(x, 256)
                gr = [(v - x) / float(B * D) for v in o["reconstruction_levels"]]
                TR.qsae_ste_backward(m.decoder, o["active_idx"], gr, B, exact=m.exact)
                TR.qsae_apply_secant_grad(m.decoder)

            def lists_mask():
                m.zero_grad(set_to_none=False)
                o = m._forward_lists(x, 256)
                mask = torch.zeros((B, H), dtype=torch.bfloat16, device=dev)
                _scatter_lists(mask, o["active_idx"], None)
                gr = [(v - x) / float(B * D) for v in o["reconstruction_levels"]]
                TR.qsae_ste_backward(m.decoder, mask, gr, B, exact=m.exact)
                TR.qsae_apply_secant_grad(m.decoder)

            row.update(sparse_ms=time_ms(sparse, 5), lists_mask_product_ms=time_ms(lists_mask, 5))
        else:
            row.update(L0=None, sparse_ms=None, lists_mask_product_ms=None, note="rows overflow the active lists")

        def dense():
            m.zero_grad(set_to_none=False)
            o = m.forward_dense_active(x)
            gr = [(v - x) / float(B * D) for v in o["reconstruction_levels"]]
            TR.qsae_ste_backward(m.decoder, o["active_mask"], gr, B, exact=m.exact)
            TR.qsae_apply_secant_grad(m.decoder)

        row["dense_forward_product_ms"] = time_ms(dense, 5)
        rows.append(row)
        del m
        torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_qsae_train_dense: no CUDA device")
    dev = torch.device("cuda:0")
    name = card()
    t0 = time.perf_counter()
    rows = init_rows(dev) + crossover_rows(dev)
    lines = [f"# q_sae decoder-side training step at any activity: {name}", "", "```"]
    lines += [json.dumps(r) for r in rows]
    lines += ["```", "", f"router constant in use: mean list length / H > {TR._DENSE_TRAIN_L0_OVER_H}",
              f"(run took {time.perf_counter() - t0:.0f} s)"]
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
