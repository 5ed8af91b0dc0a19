"""Timing of the dictionary-sharded baseline_sae training step (quantizedsae_b200/sharded.py, _ShardedBaselineFn;
DESIGN 5.10 and 8) against the single-GPU BaselineSparseAutoencoder step.

    python tools/prof_sharded_baseline_train.py [--out FILE.jsonl]                     (one GPU)
    torchrun --nproc-per-node G tools/prof_sharded_baseline_train.py [--out FILE.jsonl]  (G GPUs)

B = 4096, D = 512, H = 2^20, k = 32 and 2097, fast and exact. The step is the reference trainer's: forward,
0.5 * mse, loss.backward(), normalize_decoder_weights(), Adam; its time is split into forward (with the loss),
backward and optimizer (normalisation + Adam) by CUDA events, mean over --steps steps after --warmup, the slowest rank's.
The inputs rotate through 32 batches (256 MB, more than the 126 MB L2). The dictionary is tools/prof_sharded_baseline.py's.
1. One GPU: BaselineSparseAutoencoder (autograd = True) and DictionaryShardedBaselineSAE at world size 1.
2. One GPU, --virtual G: one rank's compute in a G-way split without the exchanges, as in r9: the local forward (local
   top-k, merge of G copies of this rank's list, owner decode), backward_local on the winners this rank owns, Adam on
   the shard. In a separate profiled pass (torch.profiler, CUDA activities) the backward's kernels are summed by
   step: grouping (compaction, scans, sort), gv (the dot kernel), reduce (chunk + latent reduce), b_dec column sums.
   G = 1 is the same emulation on the whole dictionary, and also the single-GPU qsae_baseline_backward (no compaction).
   Also the rank-order sum of G value-gradient blocks [B, k] (the backward's local part of collective 2).
3. torchrun, G >= 2: the whole sharded step over both forward transports, and the backward's two all-gathers alone.
The card's name and power limit are read in the same run and printed with the numbers.
"""
import argparse
import json
import os
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
sys.path.insert(0, str(Path(__file__).resolve().parent))

import quantizedsae_b200 as Q  # noqa: E402
from quantizedsae_b200 import _lib  # noqa: E402
from quantizedsae_b200.sharded import DictionaryShardedBaselineSAE  # noqa: E402
from prof_sharded_baseline import B, D, H, N_INPUTS, card, dictionary_rows  # noqa: E402

KS = (32, 2097)


def load(m, a, b, dev):
    we, be, wd, _ = dictionary_rows(a, b, dev)
    with torch.no_grad():
        m.encoder[0].weight.copy_(we)
        m.encoder[0].bias.copy_(be)
        m.decoder.weight.copy_(wd)
        m.decoder.bias.copy_(torch.randn(D, device=dev, generator=torch.Generator(device=dev).manual_seed(3)))


def time_phases(phases, xs, steps, warmup, dist=None, world=1):
    """phases: callables run in order per step, phases[0] takes the input. -> mean ms per phase (slowest rank)."""
    for i in range(warmup):
        s = phases[0](xs[i % len(xs)])
        for f in phases[1:]:
            s = f(s)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(len(phases) + 1)] for _ in range(steps)]
    for i in range(steps):
        ev[i][0].record()
        s = phases[0](xs[i % len(xs)])
        ev[i][1].record()
        for j, f in enumerate(phases[1:], 2):
            s = f(s)
            ev[i][j].record()
    torch.cuda.synchronize()
    ms = torch.tensor([sum(e[j].elapsed_time(e[j + 1]) for e in ev) / steps for j in range(len(phases))],
                      dtype=torch.float64, device=xs[0].device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return [float(v) for v in ms.tolist()]


def trainer_phases(m, opt, rows_of):
    def fwd(x):
        lat, rows = m(x)
        a, b = rows_of(x.shape[0])
        return 0.5 * ((rows - x[a:b]) ** 2).sum() / (x.shape[0] * D)

    def bwd(loss):
        opt.zero_grad(set_to_none=True)
        loss.backward()

    def step(_):
        m.normalize_decoder_weights()
        opt.step()

    return [fwd, bwd, step]


def kernel_split(fn, xs, n=20):
    """Mean CUDA time per call of fn, by step of the backward (torch.profiler, a separate pass)."""
    from torch.profiler import ProfilerActivity, profile

    fn(xs[0])
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(n):
            fn(xs[i % len(xs)])
        torch.cuda.synchronize()
    split = {"grouping_us": 0.0, "compaction_us": 0.0, "gv_us": 0.0, "reduce_us": 0.0, "colsum_us": 0.0}
    for e in prof.key_averages():
        t = e.device_time_total / n
        name = e.key
        if "bwd_own_" in name or "bwd_scan" in name or "bwd_sort_" in name:
            split["grouping_us"] += t
            if "bwd_own_" in name:
                split["compaction_us"] += t
        elif "bwd_latent_grad" in name:
            split["gv_us"] += t
        elif "bwd_chunk" in name or "bwd_latent_reduce" in name:
            split["reduce_us"] += t
        elif "bwd_colsum" in name:
            split["colsum_us"] += t
    return split


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file (rank 0)")
    ap.add_argument("--virtual", type=int, nargs="*", default=[1, 2, 8])
    ap.add_argument("--ks", type=int, nargs="*", default=list(KS))
    args = ap.parse_args()

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    head = {"card": card(), "world": world, "B": B, "D": D, "H": H, "steps": args.steps}
    lines = []

    def emit(rec):
        rec = {**head, **rec}
        lines.append(rec)
        if rank == 0:
            print(json.dumps(rec), flush=True)

    gx = torch.Generator(device=dev).manual_seed(7)
    xs = [torch.randint(-31, 32, (B, D), device=dev, generator=gx).float() for _ in range(N_INPUTS)]

    def trainer(name, m, rows_of, k, exact):
        m.topk, m.exact, m.autograd = k, exact, True
        opt = torch.optim.Adam(m.parameters(), lr=1e-4)
        f, bw, o = time_phases(trainer_phases(m, opt, rows_of), xs, args.steps, args.warmup, dist, world)
        emit({"module": name, "k": k, "mode": "exact" if exact else "fast", "forward_ms": f, "backward_ms": bw,
              "optimizer_ms": o, "step_ms": f + bw + o, "transport": getattr(m, "transport", None)})
        del opt

    if world == 1:
        for k in args.ks:
            for exact in (False, True):
                single = Q.BaselineSparseAutoencoder(D, H).to(dev)
                load(single, 0, H, dev)
                single.return_dense = False
                trainer("single_gpu_baseline", single, lambda n: (0, n), k, exact)
                del single
                torch.cuda.empty_cache()
                sh = DictionaryShardedBaselineSAE(D, H, rank=0, world_size=1).to(dev)
                load(sh, 0, H, dev)
                trainer("sharded_baseline_ws1", sh, sh.plan.row_range, k, exact)
                del sh
                torch.cuda.empty_cache()

        # one rank's compute of a G-way split, no exchanges (r9's emulation, with the backward and the optimizer)
        for G in args.virtual:
            vb = DictionaryShardedBaselineSAE(D, H, rank=0, world_size=G).to(dev)
            load(vb, 0, H // G, dev)
            opt = torch.optim.Adam(vb.parameters(), lr=1e-4)
            gg = torch.Generator(device=dev).manual_seed(11)
            g_rows = torch.randn((B, D), device=dev, generator=gg) * 1e-4
            for k in args.ks:
                for exact in (False, True):
                    vb.topk, vb.exact = k, exact
                    plan = vb.plan
                    g_vals = torch.zeros((B, k), device=dev)

                    def fwd(x, G=G, k=k):
                        with torch.no_grad():
                            cand = vb.ops.local_candidates(x, plan.k_local(k))
                            gv, gi = vb.ops.merge(cand.unsqueeze(0).expand((G,) + tuple(cand.shape)).contiguous(),
                                                  plan.shard_latents, k)
                            vb.ops.decode_partial(gv, gi, plan, with_bias=True)
                        return x, gv, gi

                    def bwd(s, g_vals=g_vals):
                        x, gv, gi = s
                        gwe, gbe, gwd, gbd = vb.ops.backward_local(x, gv, gi, g_rows, g_vals, plan)
                        for p, gr in zip((vb.encoder[0].weight, vb.encoder[0].bias, vb.decoder.weight, vb.decoder.bias),
                                         (gwe, gbe, gwd, gbd)):
                            p.grad = gr

                    def step(_):
                        vb.normalize_decoder_weights()
                        opt.step()

                    f, bw, o = time_phases([fwd, bwd, step], xs, args.steps, args.warmup)
                    split = kernel_split(lambda x: bwd(fwd(x)), xs)
                    x0, gv0, gi0 = fwd(xs[0])
                    owned = int(((gi0 >= plan.latent_begin) & (gi0 < plan.latent_begin + plan.shard_latents)).sum())
                    rec = {"module": "sharded_baseline", "world": G, "transport": "none (one rank's compute only)", "k": k,
                           "mode": "exact" if exact else "fast", "forward_ms": f, "backward_ms": bw, "optimizer_ms": o,
                           "step_ms": f + bw + o, "owned_entries": owned, **split}
                    if G == 1:
                        rows_full = vb.ops._dec_rows()
                        rec["full_backward_split"] = kernel_split(
                            lambda x: _lib.baseline_backward(x, gv0, gi0, g_rows, None, g_vals, None, rows_full, False), xs)
                    else:
                        parts = torch.randn((G, B, k), device=dev, generator=gg)

                        def rank_sum(_, parts=parts):
                            s = parts[0].clone()
                            for r in range(1, G):
                                s += parts[r]
                            return s

                        rec["gvals_rank_sum_ms"] = time_phases([rank_sum], xs, args.steps, args.warmup)[0]
                    emit(rec)
            del vb, opt
            torch.cuda.empty_cache()
        emit({"module": "sharded_baseline", "world": "2 or more GPUs", "note": "not measured: this run had one GPU"})
    else:
        hs = H // world
        m = DictionaryShardedBaselineSAE(D, H).to(dev)
        load(m, rank * hs, (rank + 1) * hs, dev)
        for k in args.ks:
            for transport in ("nccl", "p2p"):
                for exact in (False, True):
                    m.transport = transport
                    trainer("sharded_baseline", m, m.plan.row_range, k, exact)
            per = m.plan.padded_batch(B) // world
            rows = torch.randn((per, D), device=dev)
            vals = torch.randn((B, k), device=dev)
            ag_rows, = time_phases([lambda x: m._gather_rows(rows, B)], xs, args.steps, args.warmup, dist, world)
            ag_vals, = time_phases([lambda x: m._all_gather(vals)], xs, args.steps, args.warmup, dist, world)
            emit({"module": "sharded_baseline_backward_collectives", "k": k, "all_gather_rows_ms": ag_rows,
                  "all_gather_vals_ms": ag_vals})
        if m._peer is not None:
            torch.cuda.synchronize()
            m._peer.close()
            m._peer = None

    if rank == 0 and args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
