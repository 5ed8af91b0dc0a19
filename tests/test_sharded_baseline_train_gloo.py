"""Training of the dictionary-sharded baseline_sae on CPU: gloo processes run the backward's collective choreography
(all-gather of the row gradients, rank-order sum of the value gradients, the shard-local backward) with a numpy
backend, and every shard's gradients must equal the float64 oracle of the single-process backward over the full
dictionary, sliced to the shard. Also covers ShardPlan.merge_baseline_state_dicts and the training refusals."""
import os
import socket

import numpy as np
import pytest
import torch

from quantizedsae_b200.sae.baseline import BaselineSparseAutoencoder
from quantizedsae_b200.sharded import DictionaryShardedBaselineSAE, ShardPlan
from tests.baseline_oracle import baseline_training_grads
from tests.sharded_baseline_common import NumpyBaselineShardOps, baseline_case, full_baseline_state_dict

L1 = 0.05                      # the L1 term on lat.values, taken on rank 0 only


class NumpyBaselineTrainOps(NumpyBaselineShardOps):
    """CPU restatement of CudaBaselineShardOps.backward_local (test infrastructure only): float64 sums over the entries
    this shard owns, from its own parameters."""

    def backward_local(self, x, vals, idx, g, g_vals, plan):
        a, b = plan.latent_range()
        hs = b - a
        x64, g64 = x.numpy().astype(np.float64), g.numpy().astype(np.float64)
        wd = self.m.decoder.weight.detach().numpy().astype(np.float64)             # [D, H/G]
        i = idx.numpy().astype(np.int64)
        mine = (i >= a) & (i < b)
        li = np.where(mine, i - a, 0)
        gv = np.einsum("bd,bjd->bj", g64, wd.T[li]) + g_vals.numpy().astype(np.float64)
        gv = np.where(mine, gv, 0.0)
        v = np.where(mine, vals.numpy().astype(np.float64), 0.0)
        B = x64.shape[0]
        Gz = np.zeros((B, hs))
        Gv = np.zeros((B, hs))
        rows = np.broadcast_to(np.arange(B)[:, None], li.shape)
        np.add.at(Gz, (rows[mine], li[mine]), gv[mine])
        np.add.at(Gv, (rows[mine], li[mine]), v[mine])
        f32 = lambda t: torch.from_numpy(np.ascontiguousarray(t, dtype=np.float32))
        return f32(Gz.T @ x64), f32(Gz.sum(0)), f32(g64.T @ Gv), f32(g64.sum(0))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _loss(m, lat, rows, x, l1_here):
    B, D = x.shape
    a, b = m.plan.row_range(B)
    loss = 0.5 * ((rows - x[a:b]) ** 2).sum() / (B * D)
    if l1_here:
        loss = loss + L1 * lat.values.abs().sum() / B
    return loss


def _train(rank, world, topk, B, skew, l1, steps):
    """-> (grads of the first step, rows and winners of the first forward, state_dict after `steps` Adam steps)"""
    cfg, inp = baseline_case(B=B, skew=skew)
    m = DictionaryShardedBaselineSAE(cfg["D"], cfg["H"], rank=rank, world_size=world, ops=False)
    m.ops = NumpyBaselineTrainOps(m)
    m.load_state_dict(m.plan.shard_baseline_state_dict(full_baseline_state_dict(inp)), strict=True)
    m.topk = topk
    m.autograd = True
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    x = torch.from_numpy(inp["x"])
    first = None
    for step in range(steps):
        lat, rows = m(x)
        loss = _loss(m, lat, rows, x, l1 and rank == 0)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        if step == 0:
            first = dict(rows=rows.detach().numpy().copy(), vals=lat.values.detach().numpy().copy(),
                         idx=lat.indices.numpy().copy(), exchange=m.last_exchange,
                         grads={n: p.grad.numpy().copy() for n, p in m.named_parameters()})
        m.normalize_decoder_weights()
        opt.step()
    return first, {n: t.clone() for n, t in m.state_dict().items()}


def _worker(rank, world, port, topk, B, skew, l1, steps, out):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        out[rank] = _train(rank, world, topk, B, skew, l1, steps)
    finally:
        dist.destroy_process_group()


def test_merge_inverts_the_slicer():
    cfg, inp = baseline_case(D=64, H=2048)
    full = full_baseline_state_dict(inp)
    for G in (1, 2, 4, 8):
        plan = ShardPlan(cfg["H"], G, 0)
        shards = [ShardPlan(cfg["H"], G, r).shard_baseline_state_dict(full) for r in range(G)]
        merged = plan.merge_baseline_state_dicts(shards)
        assert merged.keys() == full.keys()
        for n in full:
            assert torch.equal(merged[n], full[n]), n
        ref = BaselineSparseAutoencoder(cfg["D"], cfg["H"])
        ref.load_state_dict(merged, strict=True)
    shards = [ShardPlan(cfg["H"], 4, r).shard_baseline_state_dict(full) for r in range(4)]
    shards[2]["decoder.bias"] = shards[2]["decoder.bias"] + 1e-7
    with pytest.raises(ValueError, match="decoder.bias of rank 2"):
        ShardPlan(cfg["H"], 4, 0).merge_baseline_state_dicts(shards)
    with pytest.raises(ValueError, match="expected 4"):
        ShardPlan(cfg["H"], 4, 0).merge_baseline_state_dicts(shards[:3])


def test_training_refusals_and_default():
    m = DictionaryShardedBaselineSAE(64, 256, rank=0, world_size=1, ops=False)
    assert m.autograd is False and "autograd" not in m.state_dict()
    m.ops = NumpyBaselineTrainOps(m)
    m.autograd = True
    m.gather_output = True
    with pytest.raises(RuntimeError, match="gather_output"):
        m(torch.zeros(3, 64))
    m.gather_output = False
    with pytest.raises(RuntimeError, match="requires_grad"):
        m(torch.zeros(3, 64, requires_grad=True))
    with torch.no_grad():                                   # grad mode off: the plain forward, gather_output allowed
        m.gather_output = True
        lat, rows = m(torch.zeros(3, 64))
        assert not rows.requires_grad


def _check_grads(res, world, topk, B, skew, l1):
    cfg, inp = baseline_case(B=B, skew=skew)
    H, D = cfg["H"], cfg["D"]
    rows = np.concatenate([res[r][0]["rows"] for r in range(world)], 0)
    idx, vals = res[0][0]["idx"], res[0][0]["vals"]
    for r in range(1, world):
        assert np.array_equal(res[r][0]["idx"], idx) and np.array_equal(res[r][0]["vals"], vals)
    g = (rows.astype(np.float64) - inp["x"]) / (B * D)
    g_h = np.zeros((B, H))
    if l1:
        np.put_along_axis(g_h, idx.astype(np.int64), L1 * np.sign(vals.astype(np.float64)) / B, axis=1)
    ref = baseline_training_grads(inp["x"], inp["We"], inp["be"], inp["Wd"], inp["bd"], g, g_h, idx=idx)
    for r in range(world):
        a, b = ShardPlan(H, world, r).latent_range()
        gr = res[r][0]["grads"]
        for name, want in (("encoder.0.weight", ref["grad_we"][a:b]), ("encoder.0.bias", ref["grad_be"][a:b]),
                           ("decoder.weight", ref["grad_wd"][:, a:b]), ("decoder.bias", ref["grad_bd"])):
            scale = max(1e-30, float(np.abs(want).max()))
            np.testing.assert_allclose(gr[name], want, rtol=1e-5, atol=1e-6 * scale, err_msg=f"rank {r} {name}")
        assert np.array_equal(gr["decoder.bias"], res[0][0]["grads"]["decoder.bias"]), "decoder.bias.grad differs by rank"


# k = 32; k = 409 of 2048 latents (truncated first exchange round); the skewed dictionary (shard 0 owns every winner,
# full retry); batches 37, 11, 9, 10 that are not multiples of G; an L1 term on the values on rank 0 only.
@pytest.mark.parametrize("world,topk,B,skew,l1,exchange", [
    (2, 32, 37, False, False, "full"), (2, 32, 9, False, True, "full"), (4, 32, 37, False, True, "full"),
    (2, 409, 11, False, True, "truncated"), (2, 409, 7, True, False, "full"), (4, 409, 10, False, False, "truncated"),
    (4, 409, 6, True, True, "full")])
def test_sharded_training_under_gloo(world, topk, B, skew, l1, exchange):
    import torch.multiprocessing as mp

    steps = 3
    port = _free_port()
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(world, port, topk, B, skew, l1, steps, out), nprocs=world, join=True)
        res = {r: out[r] for r in range(world)}
    assert all(res[r][0]["exchange"] == exchange for r in range(world))
    _check_grads(res, world, topk, B, skew, l1)
    # three Adam steps: the merged shards match one process running the same loop over the whole dictionary. The
    # reconstruction rows are summed in another order across shards, and Adam normalises a gradient by its own size,
    # so an element whose gradient is rounding noise may move by a fraction of lr = 1e-3 per step: atol 3e-5.
    cfg, _ = baseline_case(B=B, skew=skew)
    merged = ShardPlan(cfg["H"], world, 0).merge_baseline_state_dicts([res[r][1] for r in range(world)])
    _, single = _train(0, 1, topk, B, skew, l1, steps)
    for n, t in single.items():
        np.testing.assert_allclose(merged[n].numpy(), t.numpy(), rtol=1e-5, atol=3e-5, err_msg=n)
