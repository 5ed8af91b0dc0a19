"""GPU parity of the dictionary-sharded b_sae (C ABI: qsae_pack_candidates, qsae_merge_candidates,
qsae_decode_int4_range). On one GPU the G shards are evaluated one after the other and the gathered
candidate tensor is assembled by hand (the collectives are covered by tests/test_sharded_gloo.py and,
when the box has >= 2 GPUs, by the NCCL test below). Indices bit-exact, values 1e-5, recon 1e-4."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import qsae_oracle as O
from quantizedsae_b200 import _lib as L
from quantizedsae_b200.sharded import DictionaryShardedBinarySAE, ShardPlan
from tests.sharded_common import full_state_dict, sharded_case

pytestmark = pytest.mark.gpu


def _recon_close(got, ref):
    rms = float(np.sqrt(np.mean(np.square(ref, dtype=np.float64)))) + 1e-30
    np.testing.assert_allclose(got, ref, rtol=1e-4, atol=1e-4 * rms)


@pytest.mark.parametrize("G,D,H,B,k", [(4, 64, 2048, 37, 4), (8, 512, 16384, 130, 32), (2, 256, 8192, 64, 65),
                                       (8, 64, 4096, 20, 200), (8, 512, 65536, 96, 128)])
def test_virtual_shards_match_full_dictionary(cuda_device, G, D, H, B, k):
    cfg, inp = sharded_case(D=D, H=H, B=B, seed=G + k)
    dev = cuda_device
    x = torch.from_numpy(inp["x"]).to(dev)
    bd = torch.from_numpy(inp["bd"]).to(dev)
    qstep = cfg["gamma"] / 2 ** (cfg["n_bits"] - 1)
    cands, packs = [], []
    for g in range(G):
        plan = ShardPlan(H, G, g)
        a, b = plan.latent_range()
        We = torch.from_numpy(inp["We"][a:b]).to(dev)
        be = torch.from_numpy(inp["be"][a:b]).to(dev)
        kl = plan.k_local(k)
        w_bf16 = L.cast_bf16(We)
        vals, idx, _ = L.encode_topk(x, w_bf16, None, be, kl, sample=L.prepare_sample(w_bf16, be))
        assert int(idx.min()) >= 0 and int(idx.max()) < plan.shard_latents          # shard-local indices
        cands.append(L.pack_candidates(vals, idx))
        packs.append(L.pack_bitplanes(torch.from_numpy(inp["logits"][a:b]).to(dev), D, cfg["n_bits"])[0])
    cand_all = torch.stack(cands, 0).contiguous()                                    # what the all-gather delivers
    gv, gi = L.merge_candidates(cand_all, H // G, k)
    rv, ri, rr, _ = O.bsae_forward(inp["x"], inp["We"], inp["be"], inp["logits"], inp["bd"], n_bits=cfg["n_bits"],
                                   gamma=cfg["gamma"], k=k, mode="hard")
    assert np.array_equal(gi.cpu().numpy(), ri)
    assert np.all(np.abs(gv.cpu().numpy() - rv) <= 1e-5 * np.maximum(1.0, np.abs(rv)))
    total = torch.zeros((B, D), device=dev)
    for g in range(G):
        part = L.decode_range(gv, gi, packs[g], H // G, g * (H // G), D, qstep, bd if g == 0 else None, cfg["n_bits"])
        total += part                                                                # stands in for the reduce-scatter
    _recon_close(total.cpu().numpy(), rr)
    # ownership: the partial of shard g only depends on winners inside its range
    g = G - 1
    masked = torch.where((gi >= g * (H // G)) & (gi < (g + 1) * (H // G)), gi, torch.full_like(gi, -1))
    p1 = L.decode_range(gv, masked, packs[g], H // G, g * (H // G), D, qstep, None, cfg["n_bits"])
    p2 = L.decode_range(gv, gi, packs[g], H // G, g * (H // G), D, qstep, None, cfg["n_bits"])
    assert torch.equal(p1, p2)


@pytest.mark.parametrize("G,D,H,B,k", [(8, 64, 131072, 24, 262), (4, 128, 65536, 10, 1000)])
def test_virtual_shards_large_k(cuda_device, G, D, H, B, k):
    """k > QSAE_MAX_K (int(0.002 H) = 262 at H = 2^17, 2097 at 2^20): every shard contributes its own
    top-k through the block-level path, the merge radix-selects the global top-k of the G * k
    candidates. Compared with the near-tie-aware rule (thousands of adjacent order statistics)."""
    from tests.test_gpu_parity import assert_topk_matches

    cfg, inp = sharded_case(D=D, H=H, B=B, seed=G + k)
    dev = cuda_device
    x = torch.from_numpy(inp["x"]).to(dev)
    bd = torch.from_numpy(inp["bd"]).to(dev)
    qstep = cfg["gamma"] / 2 ** (cfg["n_bits"] - 1)
    cands, packs = [], []
    for g in range(G):
        plan = ShardPlan(H, G, g)
        a, b = plan.latent_range()
        We = torch.from_numpy(inp["We"][a:b]).to(dev)
        be = torch.from_numpy(inp["be"][a:b]).to(dev)
        w_bf16 = L.cast_bf16(We)
        vals, idx, _ = L.encode_topk(x, w_bf16, None, be, plan.k_local(k), sample=L.prepare_sample(w_bf16, be))
        cands.append(L.pack_candidates(vals, idx))
        packs.append(L.pack_bitplanes(torch.from_numpy(inp["logits"][a:b]).to(dev), D, cfg["n_bits"])[0])
    gv, gi = L.merge_candidates(torch.stack(cands, 0).contiguous(), H // G, k)
    z = O.encode_pre(inp["x"], inp["We"], inp["be"])
    assert_topk_matches(gv.cpu().numpy(), gi.cpu().numpy(), z, k)
    total = torch.zeros((B, D), device=dev)
    for g in range(G):
        total += L.decode_range(gv, gi, packs[g], H // G, g * (H // G), D, qstep, bd if g == 0 else None, cfg["n_bits"])
    ref = O.decode_rows(gv.cpu().numpy(), gi.cpu().numpy(), O.dequant_hard(inp["logits"], cfg["n_bits"]).astype(np.float32),
                        qstep, inp["bd"])
    _recon_close(total.cpu().numpy(), ref)


def test_world_size_one_module_equals_bsae(cuda_device):
    cfg, inp = sharded_case(D=64, H=4096, B=50)
    m = DictionaryShardedBinarySAE(cfg["D"], cfg["H"], cfg["gamma"], cfg["n_bits"], rank=0, world_size=1)
    m.load_state_dict(full_state_dict(inp), strict=True)
    m.to(cuda_device).eval()
    with torch.no_grad():
        lat, rows, pol = m(torch.from_numpy(inp["x"]).to(cuda_device))
    k = int(cfg["H"] * 0.002)
    rv, ri, rr, rp = O.bsae_forward(inp["x"], inp["We"], inp["be"], inp["logits"], inp["bd"], n_bits=cfg["n_bits"],
                                    gamma=cfg["gamma"], k=k, mode="hard")
    assert np.array_equal(lat.indices.cpu().numpy(), ri)
    _recon_close(rows.cpu().numpy(), rr)
    assert float(pol) == rp == 0.0


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, out, D, H, B, kfrac, transport="nccl", ordered=True):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        cfg, inp = sharded_case(D=D, H=H, B=B, seed=5)
        m = DictionaryShardedBinarySAE(cfg["D"], cfg["H"], cfg["gamma"], cfg["n_bits"])
        m.load_state_dict(m.plan.shard_state_dict(full_state_dict(inp), cfg["n_bits"]), strict=True)
        m.to(dev).eval()
        m.k = kfrac
        m.transport = transport
        if not ordered:
            m.exact = False
            m.ordered_latents = False
        with torch.no_grad():
            for _ in range(3 if transport == "p2p" else 1):     # p2p: several exchanges through the two buffer slots
                lat, rows, pol = m(torch.from_numpy(inp["x"]).to(dev))
        torch.cuda.synchronize()
        if transport == "p2p":
            m._peer.check()                                     # no flag wait timed out
        out[rank] = (lat.values.cpu().numpy(), lat.indices.cpu().numpy(), rows.cpu().numpy(), float(pol),
                     m.plan.row_range(cfg["B"]), m.last_exchange)
    finally:
        dist.destroy_process_group()


# k = 32 of 32768 latents; and the reference default fraction 0.002 on 2^17 latents (k = 262 > QSAE_MAX_K:
# block-level selection on every shard, radix-select merge of G * 262 candidates)
@pytest.mark.parametrize("D,H,B,kfrac,transport", [(512, 32768, 203, 2 ** -10, "nccl"), (128, 131072, 61, 0.002, "nccl"),
                                                   (512, 32768, 203, 2 ** -10, "p2p"), (128, 131072, 61, 0.002, "p2p")])
def test_dictionary_sharded_forward_under_nccl(cuda_device, D, H, B, kfrac, transport):
    """transport "nccl": all-gather / reduce-scatter; "p2p": the same exchanges through CUDA IPC peer memory, read
    inside the merge / reduce kernels (NCCL only carries the IPC handles once)."""
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    from tests.test_gpu_parity import assert_topk_matches

    port = _free_port()
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_nccl_worker, args=(world, port, out, D, H, B, kfrac, transport), nprocs=world, join=True)
        res = {r: out[r] for r in range(world)}
    cfg, inp = sharded_case(D=D, H=H, B=B, seed=5)
    k = int(H * kfrac)
    z = O.encode_pre(inp["x"], inp["We"], inp["be"])
    hard = O.dequant_hard(inp["logits"], cfg["n_bits"]).astype(np.float32)
    qstep = cfg["gamma"] / 2 ** (cfg["n_bits"] - 1)
    for r in range(world):
        v, i, rows, pol, (a, b), exchange = res[r]
        assert exchange == ("truncated" if k >= 256 else "full")
        assert np.array_equal(i, res[0][1]) and np.array_equal(v, res[0][0])       # identical on every rank
        assert_topk_matches(v, i, z, k)
        _recon_close(rows, O.decode_rows(v, i, hard, qstep, inp["bd"])[a:b])
        assert pol == 0.0


def test_merge_candidates_truncated_lists(cuda_device):
    """Shards that send only part of their candidates: the merge must report a list that was used up."""
    rng = np.random.default_rng(4)
    G, B, kin, kout, shard = 4, 6, 100, 300, 4096
    vals = rng.standard_normal((G, B, kin)).astype(np.float32)
    vals[0, 2] += 10.0                                          # row 2: shard 0's whole list wins
    vals = -np.sort(-vals, axis=2)
    idx = np.stack([np.stack([rng.choice(shard, kin, replace=False) for _ in range(B)]) for _ in range(G)]).astype(np.int32)
    cand = np.empty((G, B, kin, 2), dtype=np.int32)
    cand[..., 0] = vals.view(np.int32)
    cand[..., 1] = idx

    def run(c):
        gv, gi, flag = L.merge_candidates(torch.from_numpy(np.ascontiguousarray(c)).to(cuda_device), shard, kout, truncated=True)
        gv2, gi2 = L.merge_candidates(torch.from_numpy(np.ascontiguousarray(c)).to(cuda_device), shard, kout)
        assert torch.equal(gv, gv2) and torch.equal(gi, gi2)    # the check does not change the result
        return int(flag.item())

    assert run(cand) == 1
    ok = cand.copy()
    ok[0, 2, :, 0] = (vals[0, 2] - 10.0).view(np.int32)       # back to an ordinary row: ~75 of 100 selected per shard
    assert run(ok) == 0


@pytest.mark.parametrize("G,B,kin,kout", [(8, 33, 32, 32), (4, 17, 65, 65), (8, 9, 128, 100), (2, 5, 7, 9), (8, 6, 224, 224),
                                          (8, 5, 263, 2097), (8, 3, 2097, 2097), (4, 4, 1000, 4000)])
def test_merge_candidates_tie_rule(cuda_device, G, B, kin, kout):
    """Heavily tied candidate values: the merge must order by (value desc, global index asc) exactly."""
    rng = np.random.default_rng(G * 1000 + kin)
    shard = 4096
    vals = rng.integers(0, 4, size=(G, B, kin)).astype(np.float32)       # only 4 distinct values
    vals[:, 0] = 1.0                                                      # a row where everything ties
    idx = np.stack([np.stack([rng.choice(shard, kin, replace=False) for _ in range(B)]) for _ in range(G)]).astype(np.int32)
    cand = np.empty((G, B, kin, 2), dtype=np.int32)
    cand[..., 0] = vals.view(np.int32)
    cand[..., 1] = idx
    gv, gi = L.merge_candidates(torch.from_numpy(cand).to(cuda_device), shard, kout)
    gidx = idx.astype(np.int64) + (np.arange(G) * shard)[:, None, None]
    v = vals.transpose(1, 0, 2).reshape(B, -1)
    i = gidx.transpose(1, 0, 2).reshape(B, -1)
    order = np.lexsort((i, -v.astype(np.float64)), axis=1)[:, :kout]
    assert np.array_equal(gi.cpu().numpy(), np.take_along_axis(i, order, 1))
    assert np.array_equal(gv.cpu().numpy(), np.take_along_axis(v, order, 1))


@pytest.mark.parametrize("G,D,H,B,k", [(8, 64, 131072, 24, 262), (4, 128, 65536, 10, 1000), (1, 512, 131072, 40, 2097)])
def test_unordered_large_k_selection_is_the_same_set(cuda_device, G, D, H, B, k):
    """qsae_set_unordered_topk: the block-level selections and the candidate merge skip the sort of the winners; the
    winner SETS (and therefore the reconstruction) are those of the ordered path."""
    cfg, inp = sharded_case(D=D, H=H, B=B, seed=G + k)
    dev = cuda_device
    x = torch.from_numpy(inp["x"]).to(dev)
    res = {}
    for unordered in (False, True):
        with L.unordered_topk(unordered):
            cands = []
            for g in range(G):
                plan = ShardPlan(H, G, g)
                a, b = plan.latent_range()
                We = torch.from_numpy(inp["We"][a:b]).to(dev)
                be = torch.from_numpy(inp["be"][a:b]).to(dev)
                w_bf16 = L.cast_bf16(We)
                vals, idx, _ = L.encode_topk(x, w_bf16, None, be, plan.k_local(k), sample=L.prepare_sample(w_bf16, be))
                cands.append(L.pack_candidates(vals, idx))
            gv, gi = L.merge_candidates(torch.stack(cands, 0).contiguous(), H // G, k)
        res[unordered] = (gv.cpu().numpy(), gi.cpu().numpy())
    (v0, i0), (v1, i1) = res[False], res[True]
    o0, o1 = np.argsort(i0, axis=1), np.argsort(i1, axis=1)
    assert np.array_equal(np.take_along_axis(i0, o0, 1), np.take_along_axis(i1, o1, 1))
    assert np.array_equal(np.take_along_axis(v0, o0, 1), np.take_along_axis(v1, o1, 1))
    assert np.all(np.diff(v0, axis=1) <= 0)                       # the ordered path is ordered
    # after the block the default is restored
    with L.unordered_topk(False):
        pass
    gv2, _ = L.merge_candidates(torch.stack(cands, 0).contiguous(), H // G, k)
    assert np.all(np.diff(gv2.cpu().numpy(), axis=1) <= 0)


def test_dictionary_sharded_forward_unordered_latents_under_nccl(cuda_device):
    """ordered_latents = False (fast mode): same winner sets and reconstruction rows on every rank, both transports."""
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp

    D, H, B, kfrac = 128, 131072, 61, 0.002
    cfg, inp = sharded_case(D=D, H=H, B=B, seed=5)
    k = int(H * kfrac)
    z = O.encode_pre(inp["x"], inp["We"], inp["be"])
    rv, ri = O.topk_rows(z, k)
    hard = O.dequant_hard(inp["logits"], cfg["n_bits"]).astype(np.float32)
    qstep = cfg["gamma"] / 2 ** (cfg["n_bits"] - 1)
    for transport in ("nccl", "p2p"):
        port = _free_port()
        with mp.Manager() as mgr:
            out = mgr.dict()
            mp.spawn(_nccl_worker, args=(world, port, out, D, H, B, kfrac, transport, False), nprocs=world, join=True)
            res = {r: out[r] for r in range(world)}
        for r in range(world):
            v, i, rows, pol, (a, b), exchange = res[r]
            # the same SET on every rank (the emission order of an unordered selection depends on warp timing)
            assert np.array_equal(np.sort(i, axis=1), np.sort(res[0][1], axis=1))
            # same sets as the oracle except near-ties at the cut (fp32 accumulation order): at most 0.5 % of the entries
            diff = sum(len(set(i[q].tolist()) ^ set(ri[q].tolist())) for q in range(B))
            assert diff <= max(2, int(0.005 * i.size)), diff
            assert all(len(set(i[q].tolist())) == k for q in range(B))
            _recon_close(rows, O.decode_rows(v, i, hard, qstep, inp["bd"])[a:b])
