"""Host logic of the dictionary-sharded baseline_sae on CPU: gloo processes run the shared collective choreography
(all-gather of candidates, truncated round and full retry, deterministic merge, owner-only decode from the shard's
decoder columns, reduce-scatter of the partial rows) with the numpy ops backend, and must reproduce the
single-process oracle forward over the full dictionary."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import qsae_oracle as O
from quantizedsae_b200.sharded import DictionaryShardedBaselineSAE, ShardPlan
from tests.sharded_baseline_common import NumpyBaselineShardOps, baseline_case, full_baseline_state_dict


def test_baseline_slicer_matches_manual_slicing():
    cfg, inp = baseline_case(D=64, H=2048)
    full = full_baseline_state_dict(inp)
    for G in (1, 2, 4, 8):
        for r in range(G):
            sd = ShardPlan(cfg["H"], G, r).shard_baseline_state_dict(full)
            a, b = r * (cfg["H"] // G), (r + 1) * (cfg["H"] // G)
            assert torch.equal(sd["encoder.0.weight"], torch.from_numpy(inp["We"][a:b]))
            assert torch.equal(sd["encoder.0.bias"], torch.from_numpy(inp["be"][a:b]))
            assert torch.equal(sd["decoder.weight"], torch.from_numpy(inp["Wd"][:, a:b]))       # columns: [D, H/G]
            assert sd["decoder.weight"].is_contiguous()
            assert torch.equal(sd["decoder.bias"], torch.from_numpy(inp["bd"]))
            m = DictionaryShardedBaselineSAE(cfg["D"], cfg["H"], rank=r, world_size=G, ops=False)
            m.load_state_dict(sd, strict=True)                                                  # the module's own layout
    # the b_sae slicer is unchanged: rows of decoder.weight
    sd = ShardPlan(cfg["H"], 4, 1).shard_state_dict(full, 4)
    assert torch.equal(sd["decoder.weight"], torch.from_numpy(inp["Wd"][512:1024]))


def test_module_defaults_and_k_out_of_range():
    m = DictionaryShardedBaselineSAE(64, 256, rank=0, world_size=1, ops=False)
    assert m.topk == 32 and m.exact and m.transport == "nccl" and not m.gather_output and m.ordered_latents
    assert m.trim_min_k == 256 and m.last_exchange is None and m.last_k_send is None and m._peer is None
    m.ops = NumpyBaselineShardOps(m)
    m.topk = 257
    with pytest.raises(RuntimeError, match="out of range"):
        m(torch.zeros(3, 64))


def test_normalize_decoder_weights_is_the_shard_of_the_full_formula():
    cfg, inp = baseline_case(D=64, H=2048)
    w = torch.from_numpy(inp["Wd"])
    ref = w / torch.clamp(torch.norm(w, dim=0, keepdim=True), min=1e-8)
    for r in range(4):
        plan = ShardPlan(cfg["H"], 4, r)
        m = DictionaryShardedBaselineSAE(cfg["D"], cfg["H"], rank=r, world_size=4, ops=False)
        m.load_state_dict(plan.shard_baseline_state_dict(full_baseline_state_dict(inp)), strict=True)
        m.normalize_decoder_weights()
        a, b = plan.latent_range()
        assert torch.equal(m.decoder.weight.detach(), ref[:, a:b])


def test_world_size_one_matches_oracle():
    cfg, inp = baseline_case(D=64, H=2048, B=13)
    m = DictionaryShardedBaselineSAE(cfg["D"], cfg["H"], rank=0, world_size=1, ops=False)
    m.ops = NumpyBaselineShardOps(m)
    m.load_state_dict(full_baseline_state_dict(inp), strict=True)
    with torch.no_grad():
        lat, rows = m(torch.from_numpy(inp["x"]))
    rv, ri, rr = O.baseline_forward(inp["x"], inp["We"], inp["be"], inp["Wd"], inp["bd"], k=32)
    assert np.array_equal(lat.indices.numpy(), ri) and np.array_equal(lat.values.numpy(), rv)
    assert lat.shape == (cfg["B"], cfg["H"]) and m.last_exchange == "full"
    np.testing.assert_allclose(rows.numpy(), rr, rtol=1e-5, atol=1e-5)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, topk, B, gather, skew, out):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        cfg, inp = baseline_case(B=B, skew=skew)
        m = DictionaryShardedBaselineSAE(cfg["D"], cfg["H"], ops=False)
        m.ops = NumpyBaselineShardOps(m)
        m.load_state_dict(m.plan.shard_baseline_state_dict(full_baseline_state_dict(inp)), strict=True)
        m.topk = topk
        m.gather_output = gather
        with torch.no_grad():
            lat, rows = m(torch.from_numpy(inp["x"]))
        out[rank] = (lat.values.numpy(), lat.indices.numpy(), rows.numpy(), m.plan.row_range(B), m.last_exchange,
                     m.last_k_send)
    finally:
        dist.destroy_process_group()


# k = 32: every shard sends its full top-k. k = 409 of 2048 latents: truncated first round (307 candidates per shard
# at G = 2, 179 at G = 4). Skewed: the first half of the dictionary wins everything, a shard's truncated list is used
# up, and the full exchange follows. Batches 37, 9, 11, 7 and 10 are not multiples of G: the reduce-scatter pads.
@pytest.mark.parametrize("world,topk,B,gather,skew,exchange", [
    (2, 32, 37, False, False, "full"), (2, 32, 9, True, False, "full"), (4, 32, 37, False, False, "full"),
    (2, 409, 11, False, False, "truncated"), (2, 409, 7, True, True, "full"), (4, 409, 10, True, False, "truncated"),
    (4, 409, 6, False, True, "full")])
def test_dictionary_sharded_baseline_under_gloo(world, topk, B, gather, skew, exchange):
    import torch.multiprocessing as mp

    port = _free_port()
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(world, port, topk, B, gather, skew, out), nprocs=world, join=True)
        res = {r: out[r] for r in range(world)}
    cfg, inp = baseline_case(B=B, skew=skew)
    rv, ri, rr = O.baseline_forward(inp["x"], inp["We"], inp["be"], inp["Wd"], inp["bd"], k=topk)
    plan0 = ShardPlan(cfg["H"], world, 0)
    k_send = plan0.k_send(topk) if exchange == "truncated" else plan0.k_local(topk)
    rms = float(np.sqrt(np.mean(rr.astype(np.float64) ** 2)))
    for r in range(world):
        v, i, rows, (a, b), got_exchange, got_k_send = res[r]
        assert got_exchange == exchange and got_k_send == k_send
        assert np.array_equal(i, ri), f"rank {r}: global top-k indices differ from the single-process oracle"
        np.testing.assert_array_equal(v, rv)
        ref_rows = rr if gather else rr[a:b]
        assert rows.shape == ref_rows.shape
        np.testing.assert_allclose(rows, ref_rows, rtol=1e-4, atol=1e-4 * rms)
    assert [res[r][3] for r in range(world)] == [ShardPlan(cfg["H"], world, r).row_range(B) for r in range(world)]
