"""q_sae: QuantizedMatryoshkaSAE / QuantizedMatryoshkaDecoder (sae/quantized_matryoshka.py) on
libqsae_b200.so.

forward(x) -> (latent_group: list[n_bits] of 0-d tensors, result: list[n_bits] of [B, D])   (:143)

Reference: sigmoid encoder, activity = sigmoid(z) > 0.5 (`top_k` is stored and never used, :204),
per level a dense `(scale * a) @ (S + S_mirror)` with host syncs (:85). Here: the tcgen05 encoder
collects each row's active latents in its epilogue (threshold mode) and a sparse decoder sums the
packed {-2,0,+2} rows per level, emitting the cumulative reconstructions in one pass.
When a row has more active latents than the survivor lists hold (1024 per sub-stream, e.g. an
untrained model with ~50 % activity) the forward is redone on the dense path: dense pre-activations,
A = active * scale as bf16 hi + lo and one tcgen05 GEMM per level (qsae_matryoshka_forward_dense).
`dense_mode`: "auto" (default), "always", "never" (sparse only; raise on overflow, one host sync per forward).
"auto" costs NO host synchronisation in the steady state (the reference itself syncs once per level, :85): the first
forward of a weight version checks the overflow flag synchronously and records the regime (sparse / dense);
afterwards a dense-regime model goes straight to the dense path, and a sparse-regime model reads the flag lazily --
it is copied to pinned host memory behind the forward and examined at the start of the next one. Should a later
batch overflow after all, its outputs are NaN (the kernel poisons them: never a silently wrong reconstruction), a
warning is issued at the next forward and the module switches to the dense regime. `overflowed()` checks now.
"""
from __future__ import annotations

import warnings

import torch
import torch.nn as nn

from .. import _lib
from .base import PreparedCache, invalidate_prepared, SparseAutoencoder, param_key, require_cuda_input


def nested_sizes(in_features: int, n_bits: int) -> list:
    """Level sizes: base pattern [1, 1, 2, 4, ...] scaled to in_features with int() truncation,
    remainder folded into the last level (sae/quantized_matryoshka.py:25-38)."""
    sizes = [1 if i < 2 else 2 ** (i - 1) for i in range(n_bits)]
    total = sum(sizes)
    if total != in_features:
        f = in_features / total
        sizes = [max(1, int(s * f)) for s in sizes]
        sizes[-1] = in_features - sum(sizes[:-1])
    return sizes


class QuantizedMatryoshkaDecoder(nn.Module):
    def __init__(self, in_features, out_features, abs_range=4, n_bits=8, top_k=None, joint_gradient=False,
                 allow_bias=True):
        super().__init__()
        self._ctx = [None] * n_bits            # training-only stash in the reference (:131-141); unused here
        self.joint_gradient = joint_gradient
        self.in_features = in_features
        self.out_features = out_features
        self.n_bits = n_bits
        self.abs_range = abs_range
        self.quant_step = abs_range / (2 ** (n_bits - 1))
        self.top_k = top_k
        self.allow_bias = allow_bias
        self.nested_dictionary_size = nested_sizes(in_features, n_bits)
        self.weight = nn.Parameter(torch.empty(in_features, out_features))
        self.weight_mirror = nn.Parameter(torch.empty(in_features, out_features))
        self.bias = nn.Parameter(torch.zeros(out_features))
        nn.init.xavier_uniform_(self.weight)
        nn.init.xavier_uniform_(self.weight_mirror)
        self._prep = PreparedCache()

    # ---- prepared dictionary ---------------------------------------------------------------

    def invalidate(self) -> None:
        """Forget the prepared copies of the weights (needed after in-place edits through `.data`, which bump no version
        counter; see sae/base.py)."""
        invalidate_prepared(self)

    refresh = invalidate
    def _levels(self):
        dev = self.weight.device

        def make():
            starts = [0]
            for s in self.nested_dictionary_size:
                starts.append(starts[-1] + s)
            factors = [2 ** (self.n_bits - i - 2) * self.quant_step for i in range(self.n_bits)]
            return (torch.tensor(starts, dtype=torch.int32, device=dev),
                    torch.tensor(factors, dtype=torch.float32, device=dev))

        return self._prep.get("levels", (str(dev), self.n_bits, self.in_features, self.quant_step), make)

    def _packed(self):
        if not self.weight.is_cuda:
            raise RuntimeError("QuantizedMatryoshkaDecoder runs only on CUDA (no CPU fallback)")
        ls, lf = self._levels()

        def make():
            packed, scale = _lib.pack_matryoshka(self.weight.detach().contiguous(), self.weight_mirror.detach().contiguous(),
                                                 ls, lf)
            # the reference warns on every forward when a row of S + S_mirror is all zero (:85-86); here once per
            # weight version, when the dictionary is packed (scale = factor / (norm + 1e-8): norm < 1e-6 <=> scale > factor * 1e6 / 1.01)
            starts = self._level_starts_host()
            for i in range(self.n_bits):
                sl = scale[starts[i]:starts[i + 1]]
                if sl.numel():
                    factor = float(lf[i])
                    norms = factor / sl - 1e-8
                    if bool((norms < 1e-6).any()):
                        print(f"Warning: Very small norm detected at level {i}: min={float(norms.min().clamp_min(0.0)):.2e}")
            return packed, scale

        return self._prep.get("packed", param_key(self.weight, self.weight_mirror), make)

    def _t_bf16(self):
        """T^T [D, H] bf16 for the dense level GEMMs (cached per weight version)."""
        return self._prep.get("t_bf16", param_key(self.weight, self.weight_mirror),
                              lambda: _lib.unpack_matryoshka_t(self._packed()[0], self.out_features))

    def _level_starts_host(self):
        starts = [0]
        for s in self.nested_dictionary_size:
            starts.append(starts[-1] + s)
        return starts

    def _finish(self, result, counts, overflow, B):
        if overflow is not None and int(overflow.item()) != 0:
            raise RuntimeError("q_sae: a row has more active latents than the sparse decoder holds "
                               "(1024 per sub-stream) and dense_mode is 'never'")
        groups = torch.true_divide(counts, float(max(B, 1))).to(torch.float32)   # int64 / float -> float32 in one kernel
        return [groups[i] for i in range(self.n_bits)], [result[i] for i in range(self.n_bits)]

    # ---- training-side (SURVEY 8f-4; quantizedsae_b200/training.py) --------------------------
    def ste_backward(self, active_idx, grad_levels, batch_size=None):
        """Accumulate the STE gradients of weight / weight_mirror / bias for upstream gradients
        grad_levels[i] = d loss / d result[i] (what loss.backward() leaves there in the reference, :94-124) at any
        activity: active_idx is the int32 active lists [B, cap] of QuantizedMatryoshkaSAE.forward_active, or the bf16
        activity mask [B, H] of forward_dense_active (a tensor-core product, fp32-accurate). Returns z2 (:137)."""
        from .. import training
        return training.qsae_ste_backward(self, active_idx, grad_levels, batch_size)

    def apply_secant_grad(self):
        """(:145-190) secant correction of weight.grad / weight_mirror.grad from the last ste_backward's context."""
        from .. import training
        training.qsae_apply_secant_grad(self)

    def forward(self, latent):
        """Reference signature: dense latent [B, H] (sigmoid outputs) -> (latent_group, result)."""
        if not latent.is_cuda:
            raise RuntimeError("QuantizedMatryoshkaDecoder runs only on CUDA (no CPU fallback)")
        B, H = latent.shape
        # active = latent > 0.5 (:99), compacted into per-row lists by qsae_compact_dense
        lists, _, cnt = _lib.compact_dense(latent.contiguous().float(), 1, 0.5, want_pairs=True)
        cap = lists.shape[1]
        packed, scale = self._packed()
        ls, _ = self._levels()
        result, counts = _lib.decode_matryoshka_lists(lists, cnt.contiguous(), cap, packed, scale, ls, self.n_bits,
                                                      H, self.out_features,
                                                      self.bias.detach() if self.allow_bias else None)
        return self._finish(result, counts, torch.zeros(1, dtype=torch.int32), B)


class QuantizedMatryoshkaSAE(SparseAutoencoder):
    def __init__(self, input_dim, hidden_dim, top_k, abs_range=4, n_bits=8, allow_bias=True):
        super().__init__(input_dim, hidden_dim)
        self.n_bits = n_bits
        self.abs_range = abs_range
        self.input_dim = input_dim
        self.hidden_dim = hidden_dim
        self.allow_bias = allow_bias
        self.top_k = top_k
        self.encoder = nn.Sequential(nn.Linear(input_dim, hidden_dim), nn.Sigmoid())
        nn.init.xavier_uniform_(self.encoder[0].weight, gain=1)
        nn.init.zeros_(self.encoder[0].bias)
        self.decoder = QuantizedMatryoshkaDecoder(hidden_dim, input_dim, abs_range=abs_range, n_bits=n_bits,
                                                  top_k=self.top_k, allow_bias=self.allow_bias)
        self.exact = True                    # decide activity from an fp32 re-scoring (any fp32 weights)
        self.dense_mode = "auto"             # "auto" | "always" | "never"
        self.last_path = None                # "sparse" / "dense": which path produced the last forward
        self.last_overflow = None            # device flag of the last sparse forward (1: lists overflowed, outputs NaN)
        self._regime = None                  # (weight key, "sparse" | "dense"): decided by the first forward of a weight version
        self._pending = None                 # (pinned host flag, event) of the last unchecked sparse forward
        self._train_l0_over_h = 0.0          # mean active latents per row / H of the last training step (training.py)
        self._prep = PreparedCache()

    def _w_bf16(self):
        w = self.encoder[0].weight
        return self._prep.get("w_bf16", param_key(w), lambda: _lib.cast_bf16(w.detach().contiguous()))

    def _w_parts(self):
        """(hi, mid, lo) bf16 parts of encoder.0.weight (dense path, exact mode)."""
        w = self.encoder[0].weight
        return self._prep.get("w_parts", param_key(w), lambda: _lib.split_bf16x3(w.detach().contiguous()))

    def _w_norm_max(self):
        w = self.encoder[0].weight
        return self._prep.get("w_norm", param_key(w), lambda: _lib.max_row_norm(w.detach().contiguous()))

    def encode(self, x):
        """Dense sigmoid latents [B, H] (sae/base.py:16-19); exact fp32 CUDA-core pre-activations."""
        x = require_cuda_input(x, self)
        lin = self.encoder[0]
        return torch.sigmoid(_lib.encode_dense(x, lin.weight.detach().contiguous(), lin.bias.detach()))

    def _dense_levels(self, x, mask=None, mask_col=0):
        """The dense path -> (result [n_bits, B, D], level counts); mask: also its activity (forward_dense_active)."""
        lin = self.encoder[0]
        dec = self.decoder
        _, scale = dec._packed()
        ls, _ = dec._levels()
        w_parts = self._w_parts() if self.exact else (self._w_bf16(),)
        result, counts = _lib.matryoshka_forward_dense(
            x, w_parts, lin.bias.detach(), dec._t_bf16(), scale, ls, dec._level_starts_host(),
            dec.bias.detach() if self.allow_bias else None, mask=mask, mask_col=mask_col)
        self.last_path = "dense"
        return result, counts

    def _forward_dense(self, x):
        result, counts = self._dense_levels(x)
        return self.decoder._finish(result, counts, None, x.shape[0])

    def forward_dense_active(self, x, mask=None, mask_col: int = 0):
        """The dense path's forward with its activity as a mask, for the analysis consumers at any activity
        (scripts/analysis/dynamic_analysis.py:30-73 builds the same [B, H] mask from `encoder(x) > 0.5`).
        -> dict(latent_groups, reconstruction_levels, level_counts int64 [n_bits], active_mask [B, H] bf16 1.0 / 0.0).
        The mask comes from the decisions that form the level GEMMs' operand, so it matches the forward bit for bit; it
        records activity, so a latent whose decoder row is all zero is still active. mask / mask_col: write into columns [mask_col, mask_col + H) of
        a caller's bf16 [B, P] mask instead (multiples of 8; rq_sae puts its stages side by side)."""
        x = require_cuda_input(x, self)
        if self.hidden_dim % 8 != 0:
            raise ValueError(f"q_sae: hidden_dim {self.hidden_dim} is not a multiple of 8, so there is no dense path "
                             "(its operands need 16-byte aligned rows) and no activity mask; use forward_active")
        if mask is None:
            mask = torch.empty((x.shape[0], self.hidden_dim), dtype=torch.bfloat16, device=x.device)
            mask_col = 0
        result, counts = self._dense_levels(x, mask, mask_col)
        groups, levels = self.decoder._finish(result, counts, None, x.shape[0])
        return {"latent_groups": groups, "reconstruction_levels": levels, "level_counts": counts,
                "active_mask": mask[:, mask_col:mask_col + self.hidden_dim]}

    def _known_dense(self) -> bool:
        """True when this weight version's regime is already known to be dense (model(x) takes the dense path)."""
        if self.dense_mode == "always":
            return True
        return (self.dense_mode == "auto" and self._regime is not None and self._regime[0] == self._weights_key()
                and self._regime[1] == "dense")

    def _forward_lists(self, x, active_cap: int = 256):
        """forward_active's body: the dict, or None when the rows overflow the sparse survivor lists."""
        lin = self.encoder[0]
        packed, scale = self.decoder._packed()
        ls, _ = self.decoder._levels()
        cap = max(32, int(active_cap))
        while True:
            result, counts, overflow, a_idx, a_cnt = _lib.matryoshka_forward(
                x, self._w_bf16(), lin.bias.detach(), packed, scale, ls, self.n_bits,
                self.decoder.bias.detach() if self.allow_bias else None,
                w_f32=lin.weight.detach().contiguous() if self.exact else None,
                w_norm_max=self._w_norm_max() if self.exact else None, active_cap=cap)
            if int(overflow.item()) != 0:
                return None
            need = int(a_cnt.max().item()) if a_cnt.numel() else 0
            if need <= cap:
                break
            cap = 1 << (need - 1).bit_length()
        self.last_path = "sparse"
        groups, levels = self.decoder._finish(result, counts, overflow, x.shape[0])
        return {"latent_groups": groups, "reconstruction_levels": levels, "level_counts": counts,
                "active_idx": a_idx, "active_cnt": a_cnt}

    def forward_active(self, x, active_cap: int = 256):
        """forward(x) plus each row's active latents in sparse form, for the analysis consumers
        (scripts/analysis/dynamic_analysis.py:30-73 builds a dense [B, H] mask from a second encoder pass).
        -> dict(latent_groups, reconstruction_levels, level_counts int64 [n_bits],
                active_idx [B, cap] int32 (-1 = empty, unordered), active_cnt [B] int32).
        Sparse path only: a model whose rows overflow the survivor lists (~50 % active, untrained) has no
        sparse active form and raises; forward_dense_active gives the same forward's activity as a dense mask."""
        x = require_cuda_input(x, self)
        r = self._forward_lists(x, active_cap)
        if r is None:
            raise RuntimeError("q_sae: rows with more active latents than the sparse path holds have no sparse "
                               "active-list form (dense activity); use forward_dense_active(x) or model.encode(x) > 0.5")
        return r

    def _forward_sparse(self, x, want_residual: bool = False):
        """The sparse path without the host-side overflow check: -> (result [n_bits, B, D], counts, overflow [1]
        [, next residual (x - result[-1]) * 2]). Callers that chain several forwards (rq_sae) read the flags once at
        the end instead of once per stage, and take the residual from the level decoder instead of a separate pass."""
        lin = self.encoder[0]
        packed, scale = self.decoder._packed()
        ls, _ = self.decoder._levels()
        return _lib.matryoshka_forward(
            x, self._w_bf16(), lin.bias.detach(), packed, scale, ls, self.n_bits,
            self.decoder.bias.detach() if self.allow_bias else None,
            w_f32=lin.weight.detach().contiguous() if self.exact else None,
            w_norm_max=self._w_norm_max() if self.exact else None, want_residual=want_residual)

    def _weights_key(self):
        lin = self.encoder[0]
        return param_key(lin.weight, lin.bias, self.decoder.weight, self.decoder.weight_mirror)

    def _take_pending(self, block: bool) -> bool:
        """-> True when the last unchecked sparse forward overflowed (block=False: only if its flag copy has landed)."""
        if self._pending is None:
            return False
        host, ev = self._pending
        if not block and not ev.query():
            return False
        ev.synchronize()
        self._pending = None
        return int(host[0]) != 0

    def overflowed(self) -> bool:
        """Synchronous check of the last sparse forward: True = its survivor lists overflowed and its outputs are NaN."""
        if self.last_overflow is None:
            return False
        return int(self.last_overflow.item()) != 0

    def forward(self, x):
        x = require_cuda_input(x, self)
        if self.dense_mode == "always":
            return self._forward_dense(x)
        key = self._weights_key()
        regime = self._regime[1] if (self._regime is not None and self._regime[0] == key) else None
        capturing = torch.cuda.is_current_stream_capturing()
        if self.dense_mode == "auto" and not capturing and self._take_pending(block=False):
            warnings.warn("q_sae: the previous forward overflowed the sparse survivor lists (its outputs were NaN); "
                          "switching this weight version to the dense path")
            self._regime = (key, "dense")
            regime = "dense"
        if self.dense_mode == "auto" and regime == "dense":
            return self._forward_dense(x)
        result, counts, overflow = self._forward_sparse(x)
        self.last_overflow = overflow
        if self.dense_mode == "never" or (regime is None and not capturing):
            # synchronous: "never" must raise now; the first forward of a weight version decides the regime
            if int(overflow.item()) != 0:
                if self.dense_mode == "never":
                    return self.decoder._finish(result, counts, overflow, x.shape[0])     # raises
                self._regime = (key, "dense")
                return self._forward_dense(x)
            self._regime = (key, "sparse")
        elif not capturing:
            host = torch.empty((1,), dtype=torch.int32).pin_memory() if self._pending is None else self._pending[0]
            host.copy_(overflow, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            self._pending = (host, ev)
        self.last_path = "sparse"
        return self.decoder._finish(result, counts, None, x.shape[0])
