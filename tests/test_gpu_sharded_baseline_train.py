"""GPU tests of dictionary-sharded baseline_sae training (quantizedsae_b200.sharded, _ShardedBaselineFn; C ABI:
qsae_baseline_backward_range). A shard's backward sums each of its latents over the same entries in the same order as
the single-GPU backward, so the criterion is exact: every shard's gradients are bit-equal to the matching slice of
qsae_baseline_backward over the full dictionary, and grad b_dec is bit-equal to its grad b_dec. On one GPU the G
shards are G calls one after the other; the collectives run in the NCCL test (>= 2 GPUs) and, on CPU, in
tests/test_sharded_baseline_train_gloo.py."""
import os
import socket

import numpy as np
import pytest
import torch

import quantizedsae_b200 as Q
from quantizedsae_b200 import _lib as L
from quantizedsae_b200.sharded import DictionaryShardedBaselineSAE, ShardPlan
from tests.sharded_baseline_common import exact_grid_case, full_baseline_state_dict

pytestmark = pytest.mark.gpu


def _winners(B, H, k, dev, seed, skew_latents=None):
    """Distinct indices per row in random order: (offset + j * step) mod H with an odd step (H is a power of two).
    skew_latents: every index falls in [0, skew_latents) (shard 0 of H / skew_latents shards), and the first half of
    the rows all select latents 0 .. k-1, so those latents have B / 2 entries (the chunk path above 256)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    span = H if skew_latents is None else skew_latents
    off = torch.randint(0, span, (B, 1), device=dev, generator=g)
    step = 2 * torch.randint(0, span // 2, (B, 1), device=dev, generator=g) + 1
    j = torch.arange(k, device=dev)[None, :]
    idx = (off + j * step) % span
    if skew_latents is not None:
        idx[: B // 2] = j
    perm = torch.argsort(torch.rand((B, k), device=dev, generator=g), dim=1)
    return torch.gather(idx, 1, perm).to(torch.int32).contiguous()


def _inputs(D, H, B, k, dev, seed, skew_latents=None, with_gv=True):
    g = torch.Generator(device=dev).manual_seed(seed + 1)
    x = torch.randn((B, D), device=dev, generator=g)
    vals = torch.randn((B, k), device=dev, generator=g)
    grec = torch.randn((B, D), device=dev, generator=g) * 1e-3
    gv = torch.randn((B, k), device=dev, generator=g) * 1e-2 if with_gv else None
    rows = torch.randn((H, D), device=dev, generator=g) / np.sqrt(D)          # decoder.weight^T
    return x, vals, _winners(B, H, k, dev, seed, skew_latents), grec, gv, rows


def _full(x, vals, idx, grec, gv, rows):
    gwe, gbe, gwd, gbd, _ = L.baseline_backward(x, vals, idx, grec, None, gv, None, rows, want_grad_x=False)
    return gwe, gbe, gwd, gbd


def _check_shards(G, x, vals, idx, grec, gv, rows, ref):
    H = rows.shape[0]
    gwe, gbe, gwd, gbd = ref
    for r in range(G):
        a, b = ShardPlan(H, G, r).latent_range()
        swe, sbe, swd, sbd = L.baseline_backward_range(x, vals, idx, grec, gv, rows[a:b].contiguous(), a)
        assert torch.equal(swe, gwe[a:b]), f"shard {r}: grad W_enc"
        assert torch.equal(sbe, gbe[a:b]), f"shard {r}: grad b_enc"
        assert torch.equal(swd, gwd[:, a:b]), f"shard {r}: grad W_dec"
        assert torch.equal(sbd, gbd), f"shard {r}: grad b_dec"


# k up to 1000; (256, 2048, 9, 300) at G = 4 and 8 has shards of 512 and 256 latents, fewer than k
@pytest.mark.parametrize("G", [2, 4, 8])
@pytest.mark.parametrize("D,H,B,k", [(512, 65536, 96, 32), (256, 65536, 24, 300), (512, 32768, 20, 1000),
                                     (64, 8192, 37, 32), (256, 2048, 9, 300)])
@pytest.mark.parametrize("with_gv", [True, False])
def test_virtual_shards_bit_equal_full_backward(cuda_device, G, D, H, B, k, with_gv):
    args = _inputs(D, H, B, k, cuda_device, seed=G * 31 + k + B, with_gv=with_gv)
    _check_shards(G, *args, _full(*args))


@pytest.mark.parametrize("G", [2, 4, 8])
@pytest.mark.parametrize("D,H,B,k", [(512, 65536, 600, 32), (128, 16384, 1030, 300)])
def test_skewed_dictionary_shard_zero_owns_everything(cuda_device, G, D, H, B, k):
    x, vals, idx, grec, gv, rows = _inputs(D, H, B, k, cuda_device, seed=7, skew_latents=H // G)
    ref = _full(x, vals, idx, grec, gv, rows)
    _check_shards(G, x, vals, idx, grec, gv, rows, ref)
    hs = H // G
    assert torch.count_nonzero(ref[0][hs:]) == 0 and torch.count_nonzero(ref[2][:, hs:]) == 0
    assert int(torch.bincount(idx.flatten().long(), minlength=H).max()) > 256        # the long-latent chunk path ran


def test_empty_batch(cuda_device):
    x, vals, idx, grec, gv, rows = _inputs(64, 4096, 0, 32, cuda_device, seed=1)
    ref = _full(x, vals, idx, grec, gv, rows)
    _check_shards(4, x, vals, idx, grec, gv, rows, ref)
    assert all(int(torch.count_nonzero(t)) == 0 for t in ref)


def test_baseline_shape_eight_shards(cuda_device):
    args = _inputs(512, 1 << 20, 4096, 32, cuda_device, seed=20)
    _check_shards(8, *args, _full(*args))


def test_full_range_and_determinism(cuda_device):
    x, vals, idx, grec, gv, rows = _inputs(512, 65536, 2048, 64, cuda_device, seed=3, skew_latents=8192)
    ref = _full(x, vals, idx, grec, gv, rows)
    full_range = L.baseline_backward_range(x, vals, idx, grec, gv, rows, 0)
    assert all(torch.equal(a, b) for a, b in zip(full_range, ref))
    a, b = 8192, 16384
    one = [t.clone() for t in L.baseline_backward_range(x, vals, idx, grec, gv, rows[a:b].contiguous(), a)]
    two = L.baseline_backward_range(x, vals, idx, grec, gv, rows[a:b].contiguous(), a)
    assert all(torch.equal(p, q) for p, q in zip(one, two))


def test_range_entry_rejects_bad_arguments(cuda_device):
    x, vals, idx, grec, gv, rows = _inputs(64, 4096, 8, 32, cuda_device, seed=2)
    with pytest.raises(L.QsaeError, match="out of int32"):
        L.baseline_backward_range(x, vals, idx, grec, gv, rows[:512].contiguous(), -1)
    with pytest.raises(L.QsaeError, match="QSAE_MAX_K_LARGE"):
        L.baseline_backward_range_workspace_bytes(8, 512, 64, L.QSAE_MAX_K_LARGE + 1)
    assert L.baseline_backward_range_workspace_bytes(8, 16, 64, 1000) > 0           # k > H_shard is legal


def _pair(cfg, inp, dev, k, exact):
    full = full_baseline_state_dict(inp)
    ref = Q.BaselineSparseAutoencoder(cfg["D"], cfg["H"])
    ref.load_state_dict(full, strict=True)
    sh = DictionaryShardedBaselineSAE(cfg["D"], cfg["H"], rank=0, world_size=1)
    sh.load_state_dict(sh.plan.shard_baseline_state_dict(full), strict=True)
    for m in (ref, sh):
        m.to(dev)
        m.topk, m.exact, m.autograd = k, exact, True
    ref.return_dense = False
    return ref, sh


def _step(m, x, l1=1e-3):
    B, D = x.shape
    lat, rows = m(x)
    return 0.5 * ((rows - x) ** 2).sum() / (B * D) + l1 * lat.values.abs().sum() / B


@pytest.mark.parametrize("exact", [True, False])
@pytest.mark.parametrize("k", [32, 300])
def test_world_size_one_matches_single_gpu_module(cuda_device, k, exact):
    cfg, inp = exact_grid_case(256, 16384, 200, seed=k)
    ref, sh = _pair(cfg, inp, cuda_device, k, exact)
    x = torch.from_numpy(inp["x"]).to(cuda_device)
    opts = [torch.optim.Adam(m.parameters(), lr=1e-3) for m in (ref, sh)]
    for step in range(5):
        for m, opt in zip((ref, sh), opts):
            opt.zero_grad(set_to_none=True)
            _step(m, x).backward()
        for (n, p), (n2, p2) in zip(ref.named_parameters(), sh.named_parameters()):
            assert n == n2 and torch.equal(p.grad, p2.grad), f"step {step}: {n}.grad"
        for m, opt in zip((ref, sh), opts):
            m.normalize_decoder_weights()
            opt.step()
    for (n, t), (n2, t2) in zip(ref.state_dict().items(), sh.state_dict().items()):
        assert n == n2 and torch.equal(t, t2), n


def test_plain_forward_unchanged_with_autograd_off(cuda_device):
    cfg, inp = exact_grid_case(128, 8192, 24, seed=9)
    _, sh = _pair(cfg, inp, cuda_device, 32, True)
    x = torch.from_numpy(inp["x"]).to(cuda_device)
    with torch.no_grad():
        lat0, rows0 = sh(x)
    sh.autograd = False
    lat1, rows1 = sh(x)
    assert not rows1.requires_grad and torch.equal(rows0, rows1) and torch.equal(lat0.indices, lat1.indices)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, out, D, H, B, topk, transport):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        cfg, inp = exact_grid_case(D, H, B, seed=5)
        full = full_baseline_state_dict(inp)
        m = DictionaryShardedBaselineSAE(cfg["D"], cfg["H"])
        m.load_state_dict(m.plan.shard_baseline_state_dict(full), strict=True)
        m.to(dev)
        m.topk, m.transport, m.autograd = topk, transport, True
        x = torch.from_numpy(inp["x"]).to(dev)
        seen = {}
        lat, rows = m(x)
        rows.register_hook(lambda g: seen.__setitem__("rows", g.detach().clone()))
        lat.values.register_hook(lambda g: seen.__setitem__("vals", g.detach().clone()))
        a, b = m.plan.row_range(B)
        loss = 0.5 * ((rows - x[a:b]) ** 2).sum() / (B * cfg["D"])
        if rank == 0:
            loss = loss + 1e-3 * lat.values.abs().sum() / B
        loss.backward()
        torch.cuda.synchronize()
        if transport == "p2p":
            m._peer.check()
        # the reference: the single-GPU backward over the full dictionary, fed the same winners, the concatenated row
        # gradients and rank 0's value gradient (the other ranks' losses do not read the values)
        g_rows = m._gather_rows(seen["rows"].contiguous(), B)
        g_vals = seen.get("vals", torch.zeros_like(lat.values))
        dist.broadcast(g_vals, src=0)
        rows_full = full["decoder.weight"].t().contiguous().to(dev)
        gwe, gbe, gwd, gbd, _ = L.baseline_backward(x, lat.values.detach(), lat.indices, g_rows.contiguous(), None,
                                                    g_vals.contiguous(), None, rows_full, want_grad_x=False)
        lo, hi = m.plan.latent_range()
        ok = {"encoder.0.weight": torch.equal(m.encoder[0].weight.grad, gwe[lo:hi]),
              "encoder.0.bias": torch.equal(m.encoder[0].bias.grad, gbe[lo:hi]),
              "decoder.weight": torch.equal(m.decoder.weight.grad, gwd[:, lo:hi]),
              "decoder.bias": torch.equal(m.decoder.bias.grad, gbd)}
        bias_all = m._all_gather(m.decoder.bias.grad)
        ok["bias identical on all ranks"] = all(torch.equal(bias_all[0], bias_all[r]) for r in range(world))
        out[rank] = ok
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("transport", ["nccl", "p2p"])
@pytest.mark.parametrize("D,H,B,topk", [(512, 32768, 203, 32), (128, 131072, 61, 262)])
def test_sharded_training_under_nccl(cuda_device, D, H, B, topk, transport):
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp

    port = _free_port()
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_nccl_worker, args=(world, port, out, D, H, B, topk, transport), nprocs=world, join=True)
        res = {r: out[r] for r in range(world)}
    for r in range(world):
        assert all(res[r].values()), f"rank {r}: {res[r]}"
