"""GPU parity of the dictionary-sharded baseline_sae (quantizedsae_b200.sharded.DictionaryShardedBaselineSAE; C ABI:
qsae_encode_topk, qsae_pack_candidates, qsae_merge_candidates, qsae_decode_rows_f32_range). On one GPU the G shards
are G modules evaluated one after the other, and the gathered candidate tensor is stacked by hand (the collectives
are covered by tests/test_sharded_baseline_gloo.py and, when the box has >= 2 GPUs, by the NCCL / p2p test below).
Indices bit-exact, values 1e-5 * max(1, |v|), recon rtol 1e-4, atol 1e-4 * rms."""
import os
import socket

import numpy as np
import pytest
import torch

import quantizedsae_b200 as Q
from oracle import qsae_oracle as O
from quantizedsae_b200 import _lib as L
from quantizedsae_b200.sharded import DictionaryShardedBaselineSAE
from tests.golden import cases
from tests.sharded_baseline_common import exact_grid_case, full_baseline_state_dict

pytestmark = pytest.mark.gpu


def _recon_close(got, ref):
    rms = float(np.sqrt(np.mean(np.square(ref, dtype=np.float64)))) + 1e-30
    np.testing.assert_allclose(got, ref, rtol=1e-4, atol=1e-4 * rms)


def _vals_close(got, ref):
    assert np.all(np.abs(got - ref) <= 1e-5 * np.maximum(1.0, np.abs(ref)))


def _shards(cfg, inp, G, dev, exact=True):
    full = full_baseline_state_dict(inp)
    ms = []
    for g in range(G):
        m = DictionaryShardedBaselineSAE(cfg["D"], cfg["H"], rank=g, world_size=G)
        m.load_state_dict(m.plan.shard_baseline_state_dict(full), strict=True)
        m.to(dev).eval()
        m.exact = exact
        ms.append(m)
    return ms


def _virtual_forward(ms, x, k):
    """The sharded forward with the all-gather and the reduce-scatter done by hand on one device."""
    G, H = len(ms), ms[0].hidden_dim
    with torch.no_grad():
        cands = [m.ops.local_candidates(x, m.plan.k_local(k)) for m in ms]
        gv, gi = ms[0].ops.merge(torch.stack(cands, 0).contiguous(), H // G, k)
        total = torch.zeros((x.shape[0], ms[0].input_dim), device=x.device)
        for m in ms:
            total += m.ops.decode_partial(gv, gi, m.plan, with_bias=(m.plan.rank == 0))
    return gv, gi, total


# k = 32 at H = 65536; k = 300 and 1000: block-level selections (k > 224) on every shard and a radix-select merge
@pytest.mark.parametrize("G,D,H,B,k,exact", [(2, 64, 4096, 37, 32, True), (4, 256, 16384, 64, 32, False),
                                             (8, 512, 65536, 96, 32, True), (8, 512, 65536, 40, 32, False),
                                             (8, 256, 65536, 24, 300, False), (4, 512, 32768, 20, 1000, True),
                                             (2, 64, 8192, 16, 500, False)])
def test_virtual_shards_match_full_dictionary(cuda_device, G, D, H, B, k, exact):
    cfg, inp = exact_grid_case(D, H, B, seed=G * 7 + k)
    ms = _shards(cfg, inp, G, cuda_device, exact)
    gv, gi, total = _virtual_forward(ms, torch.from_numpy(inp["x"]).to(cuda_device), k)
    rv, ri, rr = O.baseline_forward(inp["x"], inp["We"], inp["be"], inp["Wd"], inp["bd"], k=k)
    assert np.array_equal(gi.cpu().numpy(), ri)
    _vals_close(gv.cpu().numpy(), rv)
    _recon_close(total.cpu().numpy(), rr)


def test_golden_baseline_through_eight_virtual_shards(cuda_device, golden_dir):
    name = "baseline_d512_h32768"
    cfg = cases.BASELINE_CASES[name]
    g = np.load(golden_dir / f"{name}.npz")
    inp = cases.baseline_inputs(cfg)
    ms = _shards(cfg, inp, 8, cuda_device)
    gv, gi, total = _virtual_forward(ms, torch.from_numpy(inp["x"]).to(cuda_device), int(g["k"]))
    assert np.array_equal(gi.cpu().numpy(), g["latent_idx"])
    _vals_close(gv.cpu().numpy(), g["latent_vals"])
    _recon_close(total.cpu().numpy(), g["recon"])


@pytest.mark.parametrize("G,k", [(4, 32), (8, 300)])
def test_partial_depends_only_on_owned_winners(cuda_device, G, k):
    cfg, inp = exact_grid_case(256, 16384, 33, seed=11 + G)
    ms = _shards(cfg, inp, G, cuda_device, exact=False)
    gv, gi, _ = _virtual_forward(ms, torch.from_numpy(inp["x"]).to(cuda_device), k)
    for m in (ms[0], ms[-1]):
        a, b = m.plan.latent_range()
        mine = (gi >= a) & (gi < b)
        assert bool(mine.any()) and not bool(mine.all())
        masked = torch.where(mine, gi, torch.full_like(gi, -1))
        zeroed = torch.where(mine, gv, torch.zeros_like(gv))
        p = m.ops.decode_partial(gv, gi, m.plan, with_bias=True)
        assert torch.equal(p, m.ops.decode_partial(gv, masked, m.plan, with_bias=True))
        assert torch.equal(p, m.ops.decode_partial(zeroed, gi, m.plan, with_bias=True))
        # nobody else's winners: the partial is the bias alone
        none = m.ops.decode_partial(gv, torch.where(mine, torch.full_like(gi, -1), gi), m.plan, with_bias=True)
        assert torch.equal(none, m.decoder.bias.detach().expand_as(none))


def test_decode_rows_f32_range_rejects_misaligned_buffers(cuda_device):
    dev = cuda_device
    B, k, Hs, D = 8, 4, 64, 64
    vals = torch.rand((B, k), device=dev)
    idx = torch.randint(0, Hs, (B, k), device=dev, dtype=torch.int32)
    rows = torch.randn((Hs, D), device=dev)
    bias = torch.randn(D, device=dev)
    ref = L.decode_rows_f32_range(vals, idx, rows, 0, 1.0, bias)
    assert torch.equal(ref, L.decode_rows_f32(vals, idx, rows, Hs, D, 1.0, bias))
    spare = torch.zeros(B * D + 4, device=dev)
    with pytest.raises(L.QsaeError, match="16-byte aligned"):
        L.decode_rows_f32_range(vals, idx, rows, 0, 1.0, bias, out=spare[1:1 + B * D].view(B, D))
    with pytest.raises(L.QsaeError, match="16-byte aligned"):
        L.decode_rows_f32_range(vals, idx, rows, 0, 1.0, torch.cat([bias.new_zeros(1), bias])[1:])
    torch.cuda.synchronize()
    out = spare[4:4 + B * D].view(B, D)                       # an aligned slot inside a larger buffer is accepted
    L.decode_rows_f32_range(vals, idx, rows, 0, 1.0, bias, out=out)
    assert torch.equal(out, ref)


def _single_gpu(inp, D, H, dev, exact):
    m = Q.BaselineSparseAutoencoder(D, H)
    m.load_state_dict(full_baseline_state_dict(inp), strict=True)
    m.to(dev).eval()
    m.exact, m.return_dense = exact, False
    return m


@pytest.mark.parametrize("exact", [True, False])
@pytest.mark.parametrize("topk", [32, 300])
def test_world_size_one_equals_baseline_module(cuda_device, exact, topk):
    """Same encoder, a merge of one list, and the same decode kernel at offset 0 over the same entries: bit-identical."""
    cfg = cases.BASELINE_CASES["baseline_d512_h32768"]
    inp = cases.baseline_inputs(dict(cfg, B=200))
    ref = _single_gpu(inp, cfg["D"], cfg["H"], cuda_device, exact)
    ref.topk = topk
    m = DictionaryShardedBaselineSAE(cfg["D"], cfg["H"], rank=0, world_size=1)
    m.load_state_dict(full_baseline_state_dict(inp), strict=True)
    m.to(cuda_device).eval()
    m.exact, m.topk = exact, topk
    x = torch.from_numpy(inp["x"]).to(cuda_device)
    with torch.no_grad():
        lat_r, rec_r = ref(x)
        lat, rec = m(x)
    assert lat.shape == lat_r.shape
    assert torch.equal(lat.indices, lat_r.indices) and torch.equal(lat.values, lat_r.values)
    assert torch.equal(rec, rec_r)


def test_weight_updates_reach_the_next_forward(cuda_device):
    dev = cuda_device
    cfg, inp = exact_grid_case(128, 8192, 24, seed=3)
    m = DictionaryShardedBaselineSAE(cfg["D"], cfg["H"], rank=0, world_size=1)
    m.load_state_dict(full_baseline_state_dict(inp), strict=True)
    m.to(dev).eval()
    x = torch.from_numpy(inp["x"]).to(dev)

    def same_as_fresh_module():
        fresh = Q.BaselineSparseAutoencoder(cfg["D"], cfg["H"])
        fresh.load_state_dict({k: v.detach().cpu() for k, v in m.state_dict().items()}, strict=True)
        fresh.to(dev).eval()
        fresh.exact, fresh.return_dense = m.exact, False
        with torch.no_grad():
            lat, rec = m(x)
            lat_r, rec_r = fresh(x)
        return torch.equal(lat.indices, lat_r.indices) and torch.equal(lat.values, lat_r.values) and torch.equal(rec, rec_r)

    assert same_as_fresh_module()                      # caches built
    opt = torch.optim.SGD(m.parameters(), lr=0.05)
    g = torch.Generator(device=dev).manual_seed(1)
    for p in m.parameters():
        p.grad = torch.randn(p.shape, device=dev, generator=g)
    opt.step()
    assert same_as_fresh_module()
    _, other = exact_grid_case(128, 8192, 24, seed=4)
    m.load_state_dict(full_baseline_state_dict(other), strict=True)
    assert same_as_fresh_module()
    m.normalize_decoder_weights()
    assert same_as_fresh_module()
    with torch.no_grad():
        m.decoder.weight.data.mul_(-3.0)               # through .data: no version bump, the cache cannot see it
        m.encoder[0].weight.data.mul_(-1.0)
    m.invalidate()
    assert same_as_fresh_module()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, out, D, H, B, topk, transport, exact):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        cfg, inp = exact_grid_case(D, H, B, seed=5)
        m = DictionaryShardedBaselineSAE(cfg["D"], cfg["H"])
        m.load_state_dict(m.plan.shard_baseline_state_dict(full_baseline_state_dict(inp)), strict=True)
        m.to(dev).eval()
        m.topk, m.transport, m.exact = topk, transport, exact
        with torch.no_grad():
            for _ in range(3 if transport == "p2p" else 1):     # p2p: several exchanges through the two buffer slots
                lat, rows = m(torch.from_numpy(inp["x"]).to(dev))
        torch.cuda.synchronize()
        if transport == "p2p":
            m._peer.check()                                     # no flag wait timed out
        out[rank] = (lat.values.cpu().numpy(), lat.indices.cpu().numpy(), rows.cpu().numpy(), m.plan.row_range(B),
                     m.last_exchange)
    finally:
        dist.destroy_process_group()


# k = 32 of 32768 latents (full lists); k = 262 of 2^17 (block-level selection, truncated first round)
@pytest.mark.parametrize("exact", [True, False])
@pytest.mark.parametrize("transport", ["nccl", "p2p"])
@pytest.mark.parametrize("D,H,B,topk", [(512, 32768, 203, 32), (128, 131072, 61, 262)])
def test_dictionary_sharded_baseline_under_nccl(cuda_device, D, H, B, topk, transport, exact):
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp

    port = _free_port()
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_nccl_worker, args=(world, port, out, D, H, B, topk, transport, exact), nprocs=world, join=True)
        res = {r: out[r] for r in range(world)}
    cfg, inp = exact_grid_case(D, H, B, seed=5)
    rv, ri, rr = O.baseline_forward(inp["x"], inp["We"], inp["be"], inp["Wd"], inp["bd"], k=topk)
    for r in range(world):
        v, i, rows, (a, b), exchange = res[r]
        assert exchange == ("truncated" if topk >= 256 else "full")
        assert np.array_equal(i, ri)
        _vals_close(v, rv)
        _recon_close(rows, rr[a:b])
