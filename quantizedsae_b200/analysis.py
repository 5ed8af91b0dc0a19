"""Sparse-native analysis consumers: the functions of the reference's scripts/analysis/dynamic_analysis.py
with the same names, arguments and return structure, computed from the active sets the B200 forward already
produces.

The reference (dynamic_analysis.py) re-densifies everything: `_activation_mask` runs a second forward and
returns a [B, H] boolean matrix on the CPU (:30-73), `compute_activation_stats` / `analyze_dataset` form the
co-activation counts as a dense [H, B] x [B, H] product per batch (:344-345, :391) and ship a 4 GB matrix to the
host chunk by chunk. Here one forward yields (values, indices) [B, k] (b_sae, baseline) or per-row active lists
(q_sae, rq_sae); activation counts, the co-activation matrix and the squared-error sums are accumulated by
libqsae_b200 kernels into HBM-resident buffers (qsae_activation_counts, qsae_coactivation,
qsae_sq_error_accumulate) and leave the device once, at the end.

At high activity (a q_sae between initialisation, ~50 % of the latents active, and the end of its sparsity schedule)
the rows no longer fit the sparse lists. The q_sae / rq_sae forward then runs its dense path, which writes a bf16
activity mask [B, H] from the same decisions that form its output (forward_dense_active), and the co-activation
counts become a tensor-core product M^T M over the upper triangle (qsae_coactivation_dense). Lists whose mean length
passes the measured crossover with that product are scattered into a mask and take the same route. Both routes add
exact integers into the same buffers, so batches of either kind accumulate in any order.

`sae` is a quantizedsae_b200.inference.SAEWrapper (or any object with `.model`, `.to`, `.eval`); `loader` is any
iterable of [B, D] tensors or 1-tuples of them. CUDA only -- there is no CPU path.
"""
from __future__ import annotations

from typing import Any, Iterable, Optional

import torch

from . import _lib
from .sae.baseline import BaselineSparseAutoencoder
from .sae.binary import BinarySAE
from .sae.quantized_matryoshka import QuantizedMatryoshkaSAE
from .sae.residual_quantized import ResidualQuantizedSAE
from .sparse import SparseLatents


def _batch_tensor(batch: Any) -> torch.Tensor:
    if isinstance(batch, (list, tuple)):
        batch = batch[0]
    return batch


def _hidden_dim(sae) -> int:
    """dynamic_analysis.py:17-27"""
    model = sae.model
    if hasattr(model, "hidden_dim"):
        return int(model.hidden_dim)
    if isinstance(model, BaselineSparseAutoencoder):
        return int(model.decoder.weight.shape[1])
    if isinstance(model, ResidualQuantizedSAE):
        return int(sum(s.hidden_dim for s in model.saes))
    raise ValueError(f"Unable to determine hidden_dim for model type {type(model)}")


# Sparse / dense crossover of the co-activation counts: the list kernel costs ~k^2 atomic increments per row, the
# mask product ~H^2 / 2 multiply-adds per row, so the routes cross at a fixed mean list length per latent, k / H.
# Measured with tools/prof_dense_analysis.py on a B200 (1000 W limit; profiles/r5_dense_analysis.md), B = 4096 random
# lists: H = 32768, lists 2.70 ms at k = 128 and 10.3 ms at k = 256 against 4.3 ms for scatter + mask product; H = 8192,
# 0.12 ms at k = 32 and 0.43 ms at k = 64 against 0.38 ms. Both cross between k / H = 1/256 and 1/128 (k^2 fit:
# 1/203 and 1/147). Past the list kernel's 2048 entries per row only the mask route exists.
_DENSE_ROUTE_K_OVER_H = 1.0 / 192
_SPARSE_LIST_CAP = 2048


def _qsae_active(model: QuantizedMatryoshkaSAE, x: torch.Tensor, shared=None, col: int = 0) -> dict:
    """model.forward_active(x), or model.forward_dense_active(x) when the model's regime is already dense or the rows
    overflow the sparse lists (the regime is then recorded as dense, as model(x) does). shared: callable returning
    the [B, P] mask a dense result is written into at column `col` (rq_sae stages)."""
    if not model._known_dense():
        r = model._forward_lists(x)
        if r is not None:
            return r
        if model.dense_mode == "never":
            raise RuntimeError("q_sae: a row has more active latents than the sparse path holds and dense_mode is 'never'")
        model._regime = (model._weights_key(), "dense")
    return model.forward_dense_active(x, None if shared is None else shared(), col)


def _scatter_lists(mask: torch.Tensor, idx: torch.Tensor, vals: Optional[torch.Tensor]) -> None:
    """mask[b, idx[b, j]] = 1 for every active list entry (entries < 0 or >= the mask's width are empty)."""
    active = (idx >= 0) & (idx < mask.shape[1])
    if vals is not None:
        active &= vals > 0
    rows, slots = active.nonzero(as_tuple=True)
    mask[rows, idx[rows, slots].long()] = 1.0


def forward_with_active(sae, x: torch.Tensor) -> dict:
    """One forward of the wrapped model -> dict(reconstruction, reconstruction_levels | None, level_counts | None,
    and the activity in one of two forms:
      lists: active_idx [B, cap] int32 (-1 = empty), active_vals [B, cap] | None, active_cnt [B] | None;
      mask:  active_mask [B, H] bf16 1.0 / 0.0 (active_idx None) -- q_sae / rq_sae rows too long for the lists).

    Activity follows `_activation_mask` (:30-73): b_sae / baseline: top-k latent > 0; q_sae: sigmoid(z) > 0.5;
    rq_sae: the stages' activities concatenated along the latent axis, residual updated as in forward. An rq_sae batch
    takes the mask form when any stage is on the dense path; the other stages' lists go into their column slices."""
    model = sae.model
    x = x.contiguous().float()
    out = {"active_idx": None, "active_vals": None, "active_cnt": None, "active_mask": None}
    with torch.no_grad():
        if isinstance(model, (BinarySAE, BaselineSparseAutoencoder)):
            keep = model.return_dense
            model.return_dense = False
            try:
                res = model(x)
            finally:
                model.return_dense = keep
            latents: SparseLatents = res[0]
            out.update(reconstruction=res[1], reconstruction_levels=None, level_counts=None, active_idx=latents.indices,
                       active_vals=latents.values)
            return out
        if isinstance(model, QuantizedMatryoshkaSAE):
            r = _qsae_active(model, x)
            out.update(reconstruction=r["reconstruction_levels"][-1], reconstruction_levels=r["reconstruction_levels"],
                       level_counts=r["level_counts"], active_idx=r.get("active_idx"), active_cnt=r.get("active_cnt"),
                       active_mask=r.get("active_mask"))
            return out
        if isinstance(model, ResidualQuantizedSAE):
            H = _hidden_dim(sae)
            shared = []

            def mask():
                if not shared:
                    shared.append(torch.zeros((x.shape[0], H), dtype=torch.bfloat16, device=x.device))
                return shared[0]

            residual, start = x, 0
            levels, lists, counts, cnts = [], [], [], []
            for sub, size in zip(model.saes, model.sae_hidden_dims):
                r = _qsae_active(sub, residual, mask, start)
                recon = r["reconstruction_levels"][-1]
                if "active_idx" in r:
                    a = r["active_idx"]
                    lists.append(torch.where(a >= 0, a + start, a))
                    cnts.append(r["active_cnt"])
                counts.append(r["level_counts"][-1])
                levels.append(recon)
                residual = _lib.residual_update(residual, recon.contiguous())
                start += size
            out.update(reconstruction=levels[-1], reconstruction_levels=levels, level_counts=torch.stack(counts))
            if shared:
                for a in lists:
                    _scatter_lists(shared[0], a, None)
                out["active_mask"] = shared[0]
            else:
                out.update(active_idx=torch.cat(lists, dim=1).contiguous(), active_cnt=torch.stack(cnts).sum(0))
            return out
    raise TypeError(f"Unsupported SAE model type: {type(model)}")


def _activation_mask(sae, x: torch.Tensor) -> torch.Tensor:
    """Boolean [batch, hidden_dim] mask on the CPU, as the reference returns it (:30-73). Dense by
    definition -- the accumulating functions below never build it from lists."""
    r = forward_with_active(sae, x.to(_device_of(sae)))
    if r["active_mask"] is not None:
        return (r["active_mask"] != 0).cpu()
    idx, vals = r["active_idx"], r["active_vals"]
    H = _hidden_dim(sae)
    active = idx >= 0 if vals is None else (idx >= 0) & (vals > 0)
    mask = torch.zeros((idx.shape[0], H + 1), dtype=torch.bool, device=idx.device)
    mask.scatter_(1, torch.where(active, idx, torch.full_like(idx, H)).long(), True)
    return mask[:, :H].cpu()


def _device_of(sae) -> torch.device:
    return next(sae.model.parameters()).device


def _prepare(sae, device) -> torch.device:
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("quantizedsae_b200.analysis runs on CUDA only (no CPU fallback)")
    sae.to(dev).eval()
    return dev


def compute_reconstruction_error(sae, loader: Iterable, device: str = "cuda") -> float:
    """mean (recon - x)^2 over all tokens and dimensions (:76-100)."""
    dev = _prepare(sae, device)
    acc = torch.zeros((), dtype=torch.float64, device=dev)
    n = 0
    for batch in loader:
        x = _batch_tensor(batch).to(dev).contiguous().float()
        recon = forward_with_active(sae, x)["reconstruction"]
        _lib.sq_error_accumulate(recon.contiguous(), x, acc)
        n += x.numel()
    return float(acc.item()) / n


def compute_reconstruction_error_by_level(sae, loader: Iterable, device: str = "cuda") -> torch.Tensor:
    """Per-level MSE (:103-165): q_sae levels vs x; rq_sae stage t vs the residual it was given."""
    dev = _prepare(sae, device)
    model = sae.model
    if not isinstance(model, (QuantizedMatryoshkaSAE, ResidualQuantizedSAE)):
        return torch.tensor([compute_reconstruction_error(sae, loader, device=device)], dtype=torch.float64)
    sums: Optional[torch.Tensor] = None
    n = 0
    for batch in loader:
        x = _batch_tensor(batch).to(dev).contiguous().float()
        levels = forward_with_active(sae, x)["reconstruction_levels"]
        if sums is None:
            sums = torch.zeros(len(levels), dtype=torch.float64, device=dev)
        target = x
        for i, recon in enumerate(levels):
            recon = recon.contiguous()
            _lib.sq_error_accumulate(recon, target, sums[i])
            if isinstance(model, ResidualQuantizedSAE):
                target = _lib.residual_update(target, recon)
        n += x.numel()
    return (sums / n).cpu()


def compute_l0_by_level(sae, loader: Iterable, device: str = "cuda") -> torch.Tensor:
    """Average number of active latents per token and level (:168-252)."""
    dev = _prepare(sae, device)
    total: Optional[torch.Tensor] = None
    n_tokens = 0
    for batch in loader:
        x = _batch_tensor(batch).to(dev)
        r = forward_with_active(sae, x)
        if r["level_counts"] is not None:
            c = r["level_counts"].to(torch.float64)
        else:
            idx, vals = r["active_idx"], r["active_vals"]
            c = ((idx >= 0) & (vals > 0)).sum().to(torch.float64).reshape(1)
        total = c.clone() if total is None else total + c
        n_tokens += x.shape[0]
    return (total / max(n_tokens, 1.0)).cpu()


class _StatsAccumulator:
    """activation counts [H] int64, co-activation [H, H] int32 (HBM resident), (feature, token) pairs."""

    def __init__(self, H: int, dev: torch.device, token_ids: Optional[torch.Tensor], tokens_per_context: int):
        self.H, self.dev = H, dev
        self.counts = torch.zeros(H, dtype=torch.int64, device=dev)
        self.cooc = torch.zeros((H, H), dtype=torch.int32, device=dev)
        self.token_ids = None if token_ids is None else token_ids.to(dev)
        self.tpc = tokens_per_context
        self.pairs = []
        self.global_index = 0

    def add(self, r: dict) -> None:
        """One batch of forward_with_active: lists -> qsae_activation_counts / qsae_coactivation; a mask, or lists
        past the crossover with the mask product (or past the list kernel's limit) -> qsae_coactivation_dense."""
        mask, idx, vals = r["active_mask"], r["active_idx"], r["active_vals"]
        if mask is None and self.H % 8 == 0:
            cap = idx.shape[1]
            mean_len = float(r["active_cnt"].float().mean()) if r["active_cnt"] is not None else float(cap)
            if cap > _SPARSE_LIST_CAP or mean_len > _DENSE_ROUTE_K_OVER_H * self.H:
                mask = torch.zeros((idx.shape[0], self.H), dtype=torch.bfloat16, device=idx.device)
                _scatter_lists(mask, idx.contiguous(), None if vals is None else vals.contiguous())
        if mask is not None:
            mask = mask.contiguous()
            _lib.coactivation_dense(mask, self.cooc, self.counts)
            B = mask.shape[0]
            if self.token_ids is not None:
                rows, feat = mask.nonzero(as_tuple=True)
                self.pairs.append(feat * (1 << 40) + (rows + self.global_index))    # sort key: (feature, global token)
            self.global_index += B
            return
        idx = idx.contiguous()
        vals = None if vals is None else vals.contiguous()
        _lib.activation_counts(idx, vals, self.counts)
        _lib.coactivation(idx, vals, self.cooc)
        B = idx.shape[0]
        if self.token_ids is not None:
            active = (idx >= 0) if vals is None else (idx >= 0) & (vals > 0)
            rows, slots = active.nonzero(as_tuple=True)
            feat = idx[rows, slots].long()
            self.pairs.append(feat * (1 << 40) + (rows + self.global_index))      # sort key: (feature, global token)
        self.global_index += B

    def tokens_per_feature(self) -> list:
        out = [[] for _ in range(self.H)]
        if self.token_ids is None or not self.pairs:
            return out
        keys = torch.sort(torch.cat(self.pairs)).values
        feat = keys >> 40
        gidx = keys & ((1 << 40) - 1)
        toks = self.token_ids[torch.div(gidx, self.tpc, rounding_mode="floor"), gidx % self.tpc]
        per = torch.bincount(feat, minlength=self.H).cpu().tolist()
        toks = toks.cpu().tolist()
        pos = 0
        for f, c in enumerate(per):
            if c:
                out[f] = [int(t) for t in toks[pos:pos + c]]
                pos += c
        return out


def compute_activation_stats(sae, loader: Iterable, *, token_ids: torch.Tensor, tokens_per_context: int,
                             device: str = "cuda") -> dict:
    """activation_counts [H], coactivation [H, H] = A^T A, tokens_per_feature (:255-314); CPU tensors / lists
    like the reference's."""
    dev = _prepare(sae, device)
    acc = _StatsAccumulator(_hidden_dim(sae), dev, token_ids, tokens_per_context)
    for batch in loader:
        acc.add(forward_with_active(sae, _batch_tensor(batch).to(dev)))
    return {"activation_counts": acc.counts.cpu(), "coactivation": acc.cooc.cpu(),
            "tokens_per_feature": acc.tokens_per_feature()}


def analyze_dataset(sae, loader: Iterable, *, token_ids: torch.Tensor, tokens_per_context: int, device: str) -> dict:
    """One pass: final-reconstruction MSE + activation statistics (:317-440), one forward per batch."""
    dev = _prepare(sae, device)
    acc = _StatsAccumulator(_hidden_dim(sae), dev, token_ids, tokens_per_context)
    sq = torch.zeros((), dtype=torch.float64, device=dev)
    n = 0
    for batch in loader:
        x = _batch_tensor(batch).to(dev).contiguous().float()
        r = forward_with_active(sae, x)
        _lib.sq_error_accumulate(r["reconstruction"].contiguous(), x, sq)
        n += x.numel()
        acc.add(r)
    return {"mse_final": float(sq.item()) / max(n, 1), "mse_per_level": None, "l0_per_level": None,
            "activation_counts": acc.counts.cpu(), "coactivation": acc.cooc.cpu(),
            "tokens_per_feature": acc.tokens_per_feature()}
