"""Timing of the dictionary-sharded baseline_sae forward (quantizedsae_b200/sharded.py, DESIGN 8) against the
single-GPU BaselineSparseAutoencoder and the dictionary-sharded b_sae on the same inputs.

    torchrun --nproc-per-node G tools/prof_sharded_baseline.py [--out FILE.jsonl]

B = 4096, D = 512, H = 2^20, k = 32 (b_sae: n_bits = 4, gamma = 4, its k fraction set to 32 / H):
1. DictionaryShardedBaselineSAE, fast and exact, over NCCL and over peer memory (p2p).
2. DictionaryShardedBinarySAE (polarised logits, the same encoder), the same four variants.
3. BaselineSparseAutoencoder on one GPU (rank 0, the others wait), fast and exact.
4. Run on one GPU (no torchrun), 1. and 2. are the world-size-1 modules, and for G in --virtual the tool times one
   rank's compute in a G-way split instead: local top-k over H / G latents, merge of G candidate lists, owner decode.
   That is a lower bound of a sharded step: the exchanges are not in it.
A step is one forward; its time is the mean over >= 100 steps by CUDA events, the slowest rank's (the step ends when
every rank has its rows). The inputs rotate through 32 batches (256 MB, more than the 126 MB L2). The dictionary is
the same for every G: blocks of 2^17 latents drawn from per-block seeds. The encoder weights and the inputs lie on a
grid that every summation order computes exactly (integers times 2^-12 and integers), so the in-run oracle check can
demand the exact indices: on 8 rows spread over the batch, every rank scores its shard in numpy, rank 0 merges the
candidates and sums the partial reconstructions, and compares with what the CUDA path returned (`parity_checked`).
The card's name and power limit are read in the same run and printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

import quantizedsae_b200 as Q  # noqa: E402
from oracle import qsae_oracle as O  # noqa: E402
from quantizedsae_b200.sharded import DictionaryShardedBaselineSAE, DictionaryShardedBinarySAE  # noqa: E402

B, D, H, K = 4096, 512, 2 ** 20, 32
N_BITS, GAMMA = 4, 4.0
BLOCK = 2 ** 17
N_INPUTS = 32


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name()


def dictionary_rows(a, b, dev, with_logits=False):
    """Latents [a, b) of the fixed 2^20-latent dictionary -> (We [n, D], be [n], Wd [D, n], logits [n, D n_bits] | None)."""
    parts = []
    for blk in range(a // BLOCK, -(-b // BLOCK)):
        g = torch.Generator(device=dev).manual_seed(1000 + blk)
        we = torch.randint(-127, 128, (BLOCK, D), device=dev, generator=g).float() * 2.0 ** -12
        be = torch.randint(-4096, 4097, (BLOCK,), device=dev, generator=g).float() * 2.0 ** -12
        wd = torch.randn((D, BLOCK), device=dev, generator=g) * (2.0 / (D + H)) ** 0.5
        lg = (torch.where(torch.rand((BLOCK, D * N_BITS), device=dev, generator=g) < 0.5, 110.0, -110.0)
              if with_logits else None)
        lo, hi = max(a, blk * BLOCK) - blk * BLOCK, min(b, (blk + 1) * BLOCK) - blk * BLOCK
        parts.append((we[lo:hi], be[lo:hi], wd[:, lo:hi], None if lg is None else lg[lo:hi]))
    we = torch.cat([p[0] for p in parts])
    be = torch.cat([p[1] for p in parts])
    wd = torch.cat([p[2] for p in parts], 1).contiguous()
    lg = torch.cat([p[3] for p in parts]) if with_logits else None
    return we, be, wd, lg


def time_ms(fn, xs, steps, warmup, dist, world):
    for i in range(warmup):
        fn(xs[i % len(xs)])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        fn(xs[i % len(xs)])
    b.record()
    torch.cuda.synchronize()
    ms = torch.tensor([a.elapsed_time(b) / steps], dtype=torch.float64, device=xs[0].device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def parity(m, x, rank, world, dist, dict_rows, scale, n_rows=8):
    """In-run oracle check of one sharded forward on `n_rows` rows spread over the batch (True on every rank)."""
    m.gather_output = True
    with torch.no_grad():
        out = m(x)
    m.gather_output = False
    lat, rows = out[0], out[1]
    R = np.linspace(0, x.shape[0] - 1, n_rows).astype(np.int64).tolist()
    lin = m.encoder[0]
    z = O.encode_pre(x[R].cpu().numpy(), lin.weight.detach().cpu().numpy(), lin.bias.detach().cpu().numpy())
    lv, li = O.topk_rows(z, min(K, z.shape[1]))
    a, b = m.plan.latent_range()
    gi = lat.indices[R].cpu().numpy().astype(np.int64)
    gv = lat.values[R].cpu().numpy()
    mine = (gi >= a) & (gi < b)
    loc = np.where(mine, gi - a, 0)
    need = np.unique(loc[mine])
    dr = np.zeros((b - a, D), dtype=np.float32)
    if len(need):
        dr[need] = dict_rows(torch.from_numpy(need).to(x.device))
    partial = O.decode_rows(np.where(mine, gv, np.float32(0)), loc, dr, scale, None).astype(np.float64)
    payload = (lv, li.astype(np.int64) + a, partial)
    gathered = [payload]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, payload)
    ok = True
    if rank == 0:
        v = np.concatenate([g[0] for g in gathered], 1)
        i = np.concatenate([g[1] for g in gathered], 1)
        order = np.lexsort((i, -v.astype(np.float64)), axis=1)[:, :K]
        ri, rv = np.take_along_axis(i, order, 1), np.take_along_axis(v, order, 1)
        ok = bool(np.array_equal(gi, ri) and np.all(np.abs(gv - rv) <= 1e-5 * np.maximum(1.0, np.abs(rv))))
        ref = sum(g[2] for g in gathered) + m.decoder.bias.detach().cpu().numpy().astype(np.float64)
        got = rows[R].cpu().numpy()
        rms = float(np.sqrt(np.mean(ref ** 2))) + 1e-30
        ok = ok and bool(np.allclose(got, ref, rtol=1e-4, atol=1e-4 * rms))
    flag = torch.tensor([int(ok)], device=x.device)
    if world > 1:
        dist.broadcast(flag, 0)
    return bool(flag.item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file (rank 0)")
    ap.add_argument("--no-single", action="store_true", help="skip the single-GPU BaselineSparseAutoencoder")
    ap.add_argument("--virtual", type=int, nargs="*", default=[2, 8],
                    help="world size 1 only: time one rank's compute (no exchange) of these G-way splits")
    args = ap.parse_args()

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    head = {"card": card(), "world": world, "B": B, "D": D, "H": H, "k": K, "steps": args.steps}
    lines = []

    def emit(rec):
        rec = {**head, **rec}
        lines.append(rec)
        if rank == 0:
            print(json.dumps(rec), flush=True)

    gx = torch.Generator(device=dev).manual_seed(7)               # the same inputs on every rank (replicated batch)
    xs = [torch.randint(-31, 32, (B, D), device=dev, generator=gx).float() for _ in range(N_INPUTS)]

    hs = H // world
    a, b = rank * hs, (rank + 1) * hs
    we, be, wd, lg = dictionary_rows(a, b, dev, with_logits=True)
    base = DictionaryShardedBaselineSAE(D, H, rank=rank, world_size=world)
    bsae = DictionaryShardedBinarySAE(D, H, GAMMA, N_BITS, rank=rank, world_size=world)
    with torch.no_grad():
        base.to(dev).eval()
        base.encoder[0].weight.copy_(we)
        base.encoder[0].bias.copy_(be)
        base.decoder.weight.copy_(wd)
        base.decoder.bias.copy_(torch.randn(D, device=dev, generator=torch.Generator(device=dev).manual_seed(3)))
        bsae.to(dev).eval()
        bsae.encoder[0].weight.copy_(we)
        bsae.encoder[0].bias.copy_(be)
        bsae.decoder.weight.copy_(lg)
        bsae.decoder.bias.copy_(base.decoder.bias)
    del lg
    bsae.k = K / H
    qstep = GAMMA / 2 ** (N_BITS - 1)
    base_rows = lambda i: base.decoder.weight.detach()[:, i].t().cpu().numpy()                       # noqa: E731
    bsae_rows = lambda i: O.dequant_hard(bsae.decoder.weight.detach()[i].cpu().numpy(), N_BITS).astype(np.float32)  # noqa: E731

    for name, m, rows_fn, scale in (("sharded_baseline", base, base_rows, 1.0), ("sharded_bsae", bsae, bsae_rows, qstep)):
        for transport in ("nccl", "p2p"):
            if transport == "p2p" and world == 1:
                continue
            for exact in (False, True):
                m.transport, m.exact = transport, exact
                with torch.no_grad():
                    ms = time_ms(lambda x: m(x), xs, args.steps, args.warmup, dist, world)
                if m._peer is not None:
                    m._peer.check()
                ok = parity(m, xs[0], rank, world, dist, rows_fn, scale)
                emit({"module": name, "transport": transport, "mode": "exact" if exact else "fast", "ms_per_step": ms,
                      "tokens_per_s": B / (ms * 1e-3), "parity_checked": ok, "k_send": m.last_k_send,
                      "exchange": m.last_exchange})
        if m._peer is not None:
            torch.cuda.synchronize()
            m._peer.close()
            m._peer = None
    del base, bsae, we, be, wd
    torch.cuda.empty_cache()

    if world == 1:
        # one GPU cannot run the exchanges; what it can show is one rank's compute in a G-way split: the local top-k
        # over H / G latents, the merge of G candidate lists (rank 0's list in every slot: the same G * k entries
        # and the same share of owned winners, k / G, as a real step) and the owner decode. No exchange is timed.
        for G in args.virtual:
            we, be, wd, lg = dictionary_rows(0, H // G, dev, with_logits=True)
            vb = DictionaryShardedBaselineSAE(D, H, rank=0, world_size=G).to(dev).eval()
            vs = DictionaryShardedBinarySAE(D, H, GAMMA, N_BITS, rank=0, world_size=G).to(dev).eval()
            with torch.no_grad():
                for mm in (vb, vs):
                    mm.encoder[0].weight.copy_(we)
                    mm.encoder[0].bias.copy_(be)
                vb.decoder.weight.copy_(wd)
                vs.decoder.weight.copy_(lg)
            del lg
            for name, mm in (("sharded_baseline", vb), ("sharded_bsae", vs)):
                for exact in (False, True):
                    mm.exact = exact

                    def step(x, mm=mm, G=G):
                        cand = mm.ops.local_candidates(x, mm.plan.k_local(K))
                        gv, gi = mm.ops.merge(cand.unsqueeze(0).expand((G,) + tuple(cand.shape)).contiguous(),
                                              mm.plan.shard_latents, K)
                        return mm.ops.decode_partial(gv, gi, mm.plan, with_bias=True)

                    with torch.no_grad():
                        ms = time_ms(step, xs, args.steps, args.warmup, None, 1)
                        local = time_ms(lambda x: mm.ops.local_candidates(x, mm.plan.k_local(K)), xs, args.steps,
                                        args.warmup, None, 1)
                    emit({"module": name, "world": G, "transport": "none (one rank's compute only)",
                          "mode": "exact" if exact else "fast", "ms_per_step": ms, "local_topk_ms": local,
                          "parity_checked": None})
            del vb, vs, we, be, wd
            torch.cuda.empty_cache()

    if not args.no_single:
        if world > 1:
            dist.barrier()
        if rank == 0:
            we, be, wd, _ = dictionary_rows(0, H, dev)
            single = Q.BaselineSparseAutoencoder(D, H).to(dev).eval()
            with torch.no_grad():
                single.encoder[0].weight.copy_(we)
                single.encoder[0].bias.copy_(be)
                single.decoder.weight.copy_(wd)
                single.decoder.bias.copy_(torch.randn(D, device=dev, generator=torch.Generator(device=dev).manual_seed(3)))
            single.return_dense = False
            R = np.linspace(0, B - 1, 8).astype(np.int64).tolist()
            for exact in (False, True):
                single.exact = exact
                with torch.no_grad():
                    ms = time_ms(lambda x: single(x), xs, args.steps, args.warmup, None, 1)
                    lat, rec = single(xs[0])
                rv, ri, rr = O.baseline_forward(xs[0][R].cpu().numpy(), we.cpu().numpy(), be.cpu().numpy(),
                                                wd.cpu().numpy(), single.decoder.bias.detach().cpu().numpy(), k=K)
                rms = float(np.sqrt(np.mean(rr.astype(np.float64) ** 2))) + 1e-30
                ok = bool(np.array_equal(lat.indices[R].cpu().numpy(), ri)
                          and np.allclose(rec[R].cpu().numpy(), rr, rtol=1e-4, atol=1e-4 * rms))
                emit({"module": "single_gpu_baseline", "world": 1, "transport": None, "mode": "exact" if exact else "fast",
                      "ms_per_step": ms, "tokens_per_s": B / (ms * 1e-3), "parity_checked": ok})
        if world > 1:
            dist.barrier()

    if rank == 0 and args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
