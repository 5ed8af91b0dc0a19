"""Timing of the analysis consumers' dense route on the GPU (quantizedsae_b200/analysis.py, DESIGN 5.9).

    python tools/prof_dense_analysis.py --out profiles/r5_dense_analysis.md

1. qsae_coactivation_dense alone, H = 32768, K = 4096 and 65536, 50 % dense random mask: CUDA events over many
   launches; rate against the 2250 TFLOP/s bf16 dense data-sheet figure and the int32 read-modify-write of the
   [H, H] matrix (8 H^2 bytes) against 7.7 TB/s.
2. analyze_dataset on an untrained q_sae 512 -> 32768 (zero encoder bias, ~50 % active) over 65536 tokens
   (16 batches of 4096; token_ids omitted, so no per-feature token lists).
3. The sparse / dense crossover: the same random lists (B = 4096, k = 32 .. 2048 per row) through the list kernels
   (qsae_activation_counts + qsae_coactivation) and through scatter + qsae_coactivation_dense, at H = 32768 and 8192.
The card's name and power limit are read in the same run and printed with the numbers.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

import quantizedsae_b200 as Q  # noqa: E402
from quantizedsae_b200 import _lib as L  # noqa: E402
from quantizedsae_b200 import analysis as AN  # noqa: E402
from quantizedsae_b200.inference import framework as FW  # noqa: E402

PEAK_BF16 = 2250e12
PEAK_HBM = 7.7e12


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


def kernel_rows(dev):
    H = 32768
    cooc = torch.zeros((H, H), dtype=torch.int32, device=dev)
    out = []
    for K, n in [(4096, 30), (65536, 4)]:
        mask = (torch.rand((K, H), device=dev) < 0.5).to(torch.bfloat16)
        ms = time_ms(lambda: L.coactivation_dense(mask, cooc), n)
        flop = 2.0 * K * H * (H + 1) / 2
        rmw = 8.0 * H * H
        t_mma, t_mem = flop / PEAK_BF16, (rmw + K * H * 2) / PEAK_HBM
        out.append(dict(what="coactivation_dense", H=H, K=K, launches=n, ms=ms, tflops=flop / ms / 1e9,
                        share_of_bf16_peak=flop / PEAK_BF16 / (ms / 1e3), floor_mma_ms=t_mma * 1e3,
                        floor_hbm_ms=t_mem * 1e3, bound="mma" if t_mma >= t_mem else "hbm"))
        del mask
    del cooc
    torch.cuda.empty_cache()
    return out


def analyze_row(dev):
    D, H = 512, 32768
    torch.manual_seed(3)
    with torch.device(dev):
        m = Q.QuantizedMatryoshkaSAE(D, H, 32, abs_range=4.0, n_bits=4)
    m.eval()
    sae = FW.SAEWrapper(FW.SAE_REGISTRY["q_sae"], m, dev)
    g = torch.Generator(device=dev).manual_seed(4)
    batches = [torch.randn((4096, D), device=dev, generator=g) for _ in range(16)]
    AN.analyze_dataset(sae, batches[:1], token_ids=None, tokens_per_context=1, device="cuda")   # warm-up, regime
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = AN.analyze_dataset(sae, batches, token_ids=None, tokens_per_context=1, device="cuda")
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    # the same per-batch work without the final copy of the 4.3 GB matrix to the host
    acc = AN._StatsAccumulator(H, dev, None, 1)
    sq = torch.zeros((), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    for x in batches:
        fr = AN.forward_with_active(sae, x)
        L.sq_error_accumulate(fr["reconstruction"].contiguous(), x, sq)
        acc.add(fr)
    torch.cuda.synchronize()
    dt_dev = time.perf_counter() - t1
    return dict(what="analyze_dataset", model="q_sae 512->32768 untrained", tokens=65536, s=dt, tokens_per_s=65536 / dt,
                batches_on_device_s=dt_dev, batches_on_device_tokens_per_s=65536 / dt_dev,
                host_copy_and_rest_s=dt - dt_dev, path=m.last_path,
                mean_active=float(r["activation_counts"].sum()) / 65536)


def crossover_rows(dev):
    out = []
    B = 4096
    for H in (32768, 8192):
        cooc = torch.zeros((H, H), dtype=torch.int32, device=dev)
        counts = torch.zeros(H, dtype=torch.int64, device=dev)
        for k in (32, 64, 128, 256, 512, 1024, 2048):
            if k > H // 2:
                continue
            idx = torch.rand((B, H), device=dev).topk(k, dim=1).indices.to(torch.int32).contiguous()

            def sparse():
                L.activation_counts(idx, None, counts)
                L.coactivation(idx, None, cooc)

            def dense():
                mask = torch.zeros((B, H), dtype=torch.bfloat16, device=dev)
                AN._scatter_lists(mask, idx, None)
                L.coactivation_dense(mask, cooc, counts)

            n = 5
            ts, td = time_ms(sparse, n), time_ms(dense, n)
            out.append(dict(what="crossover", B=B, H=H, k=k, k_over_H=k / H, sparse_ms=ts, dense_ms=td,
                            faster="sparse" if ts <= td else "dense"))
        del cooc
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_dense_analysis: no CUDA device")
    dev = torch.device("cuda:0")
    name = card()
    rows = kernel_rows(dev) + [analyze_row(dev)] + crossover_rows(dev)
    lines = [f"# Dense analysis route: {name}", "", "```"]
    lines += [json.dumps(r) for r in rows]
    lines += ["```", "", f"router constant in use: k / H > {AN._DENSE_ROUTE_K_OVER_H}"]
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
