"""t_sae: TernarySparseAutoencoder / STEWeights (sae/ternary.py) on libqsae_b200.so.

forward(x) -> (h, recon)                                                    (sae/ternary.py:116-122)

The reference forward does NOT apply top-k (the call is commented out, :119-120): h = relu(Linear(x))
is dense and the decoder is a dense F.linear with the hard ternary weights
T = sign(W) * (|W| >= 0.5) (:46-52; the STE expression evaluates to T exactly and the `mask` buffer
does not enter the forward value). So t_sae is two chained dense GEMMs:
  * encoder: the tcgen05 kernel of b_sae with a dense epilogue -- bias + ReLU, h written once as
    fp32 (the returned latents) and once as bf16 (A operand of the decoder) by TMA stores;
  * decoder: a second tcgen05 GEMM over K = hidden_dim with the exact-ternary bf16 matrix, split-K
    with a fixed-order reduction.
`exact` (default True, as for the other modules) reproduces the fp32 reference for arbitrary fp32
weights/inputs, still on the tensor cores: x and encoder.0.weight are split exactly into three bf16
parts each and the six partial products above 2^-24 are accumulated in three launches of the encoder;
the decoder runs two passes over the hi/lo split of h. exact = False is the throughput path, exact
when x and encoder.0.weight are bf16-representable (the benchmark's stated precondition) up to fp32
accumulation order and bf16 rounding of h in the decoder.

The dormant sparse mode `apply_topk_activation` (:102-114) is available on dense inputs and, opt-in,
as `forward_topk(x)`: fused encoder + top-k (ReLU epilogue) and an int8 ternary row gather.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .. import _lib
from ..sparse import SparseLatents
from .base import PreparedCache, invalidate_prepared, param_key, require_cuda_input


class STEWeights(nn.Module):
    def __init__(self, in_features, out_features):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(out_features, in_features))    # [D, H]
        self.threshold = 0.5
        self.register_buffer("mask", torch.ones(out_features, in_features))   # RigL mask: gradients only
        self.register_buffer("input_activations", None)
        self.register_buffer("output_grad", None)
        nn.init.kaiming_normal_(self.weight)
        self.exact = True
        self._prep = PreparedCache()


    def invalidate(self) -> None:
        """Forget the prepared copies of the weights (needed after in-place edits through `.data`, which bump no version
        counter; see sae/base.py)."""
        invalidate_prepared(self)

    refresh = invalidate
    def _ternary(self):
        """(T bf16 [D, H], T int8 rows [H, D]) for the current weights."""
        if not self.weight.is_cuda:
            raise RuntimeError("STEWeights runs only on CUDA (no CPU fallback)")
        return self._prep.get("ternary", param_key(self.weight) + (self.threshold,),
                              lambda: _lib.pack_ternary(self.weight.detach().contiguous(), self.threshold,
                                                        want_bf16=True, want_rows=True))

    # ---- RigL mask maintenance (sae/ternary.py:27-90; csrc/train.cu) ---------------------------
    def init_mask(self, sparsity):
        from .. import training
        training.rigl_init_mask(self, sparsity)

    def update_mask(self, f_decay, sparsity_rate=0.7):
        from .. import training
        training.rigl_update_mask(self, f_decay, sparsity_rate)

    def mask_grad(self):
        from .. import training
        training.rigl_mask_grad(self)

    def _ternary_t(self):
        """T^T as bf16 [H, D] for the current weights (B operand of the backward's g T, training.py)."""
        if not self.weight.is_cuda:
            raise RuntimeError("STEWeights runs only on CUDA (no CPU fallback)")
        return self._prep.get("ternary_t", param_key(self.weight) + (self.threshold,),
                              lambda: _lib.pack_ternary_t(self.weight.detach().contiguous(), self.threshold))

    def hard_weights(self) -> torch.Tensor:
        """sign(W) * (|W| >= threshold) as float32 [D, H] (sae/ternary.py:46-49)."""
        return self._ternary()[0].float()

    def forward(self, x):
        """Dense latents [B, H] -> reconstruction [B, D] (reference: F.linear(x, hard_weights), :52)."""
        if not x.is_cuda:
            raise RuntimeError("STEWeights runs only on CUDA (no CPU fallback)")
        x = x.contiguous().float()
        self.input_activations = x.detach()       # the reference's forward hook (:21-22)
        hi, lo = _lib.split_bf16(x, want_lo=self.exact)
        return _lib.decode_dense(hi, lo, self._ternary()[0])

    def decode_sparse(self, latents: SparseLatents) -> torch.Tensor:
        D, H = self.weight.shape
        return _lib.decode_int8(latents.values, latents.indices, self._ternary()[1], H, D, 1.0, None)


class TernarySparseAutoencoder(nn.Module):
    def __init__(self, input_dim, hidden_dim):
        super().__init__()
        self.encoder = nn.Sequential(nn.Linear(input_dim, hidden_dim), nn.ReLU())
        self.decoder = STEWeights(hidden_dim, input_dim)
        self.topk = int(hidden_dim * 0.002)
        self.input_dim = input_dim
        self.hidden_dim = hidden_dim
        self.exact = True
        # True: forward builds one autograd node (training.py, _TernarySAEFn) whenever grad mode is on, so the
        # trainer's loss.backward() fills encoder.0.weight / .bias, decoder.weight (and x) .grad and
        # decoder.output_grad
        self.autograd = False
        self._prep = PreparedCache()


    def invalidate(self) -> None:
        """Forget the prepared copies of the weights (needed after in-place edits through `.data`, which bump no version
        counter; see sae/base.py)."""
        invalidate_prepared(self)

    refresh = invalidate
    def _w_bf16(self):
        w = self.encoder[0].weight
        return self._prep.get("w_bf16", param_key(w), lambda: _lib.cast_bf16(w.detach().contiguous()))

    def _w_parts(self):
        """(hi, mid, lo) bf16 parts of encoder.0.weight, hi + mid + lo == W exactly."""
        w = self.encoder[0].weight
        return self._prep.get("w_parts", param_key(w), lambda: _lib.split_bf16x3(w.detach().contiguous()))

    def _sample(self):
        lin = self.encoder[0]
        return self._prep.get("sample", param_key(lin.weight, lin.bias),
                              lambda: _lib.prepare_sample(self._w_bf16(), lin.bias.detach()))

    def apply_topk_activation(self, h):
        """Dense [B, H] -> top-`topk` entries kept, non-positive ones zeroed (sae/ternary.py:102-114)."""
        if not h.is_cuda:
            raise RuntimeError("apply_topk_activation needs CUDA tensors (no CPU fallback)")
        vals, idx = _lib.topk_dense(h.contiguous().float(), int(self.topk))
        return _lib.densify(torch.clamp_min(vals, 0.0), idx, h.shape[1])

    def encode_topk(self, x) -> SparseLatents:
        """relu(Linear(x)) -> top-`topk` per row, as SparseLatents (opt-in sparse mode)."""
        x = require_cuda_input(x, self)
        lin = self.encoder[0]
        w32 = lin.weight.detach().contiguous()
        vals, idx, _ = _lib.encode_topk(x, self._w_bf16(), w32 if self.exact else None, lin.bias.detach(),
                                        int(self.topk), _lib.ACT_RELU, self.exact, sample=self._sample())
        return SparseLatents(vals, idx, (x.shape[0], self.hidden_dim))

    def forward_topk(self, x):
        """The reference's commented-out variant (:119-120): (sparse latents, decoder(h_sparse))."""
        latents = self.encode_topk(x)
        return latents, self.decoder.decode_sparse(latents)

    def _enc_parts(self):
        """The encoder weight as the forward contracts it: split_bf16x3 parts (exact) or (bf16(W),)."""
        return self._w_parts() if self.exact else (self._w_bf16(),)

    def _forward_dense(self, x):
        lin = self.encoder[0]
        return _lib.tsae_forward(x, self._enc_parts(), lin.bias.detach(), self.decoder._ternary()[0], self.exact)

    def forward(self, x):
        if self.autograd and torch.is_grad_enabled():
            from .. import training
            return training.tsae_forward(self, x)
        x = require_cuda_input(x, self)
        h, recon = self._forward_dense(x)
        self.decoder.input_activations = h        # the reference's forward hook (sae/ternary.py:21-22)
        return h, recon
