"""baseline_sae: BaselineSparseAutoencoder (sae/baseline.py) on libqsae_b200.so.

forward(x) -> (h_sparse, recon): Linear (no ReLU, sae/baseline.py:8-10) -> top-`topk` of the raw
pre-activations (:35) -> Linear decode (:29). The encoder + top-k is the same fused tcgen05
kernel as b_sae; the decoder gathers the selected columns of decoder.weight [D, H] from a
transposed [H, D] float32 copy cached per weight version.

`autograd = True` (training): the same forward behind one autograd node whose backward is the deterministic
latent-major kernel set of csrc/train.cu (training.py, `baseline_forward`).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .. import _lib
from ..sparse import SparseLatents
from .base import PreparedCache, invalidate_prepared, param_key, require_cuda_input


class BaselineSparseAutoencoder(nn.Module):
    def __init__(self, input_dim, hidden_dim):
        super().__init__()
        self.encoder = nn.Sequential(nn.Linear(input_dim, hidden_dim))
        self.decoder = nn.Linear(hidden_dim, input_dim)
        self.topk = 32
        self.input_dim = input_dim
        self.hidden_dim = hidden_dim
        self.return_dense = True
        self.exact = True
        # True: forward builds one autograd node (training.py, _BaselineSAEFn) whenever grad mode is on, so the
        # trainer's loss.backward() fills encoder.0.weight / .bias, decoder.weight / .bias (and x) .grad
        self.autograd = False
        self.last_flags = None
        self._prep = PreparedCache()


    def invalidate(self) -> None:
        """Forget the prepared copies of the weights (needed after in-place edits through `.data`, which bump no version
        counter; see sae/base.py)."""
        invalidate_prepared(self)

    refresh = invalidate
    def _w_bf16(self):
        w = self.encoder[0].weight
        return self._prep.get("w_bf16", param_key(w), lambda: _lib.cast_bf16(w.detach().contiguous()))

    def _sample(self):
        """Sampled dictionary rows for the prior-threshold pre-pass (None for small dictionaries)."""
        lin = self.encoder[0]
        return self._prep.get("sample", param_key(lin.weight, lin.bias),
                              lambda: _lib.prepare_sample(self._w_bf16(), lin.bias.detach()))

    def _dec_rows(self):
        w = self.decoder.weight                     # [D, H]: feature vectors are columns
        return self._prep.get("dec_rows", param_key(w), lambda: _lib.transpose(w.detach().contiguous()))

    def encode_topk(self, x) -> SparseLatents:
        x = require_cuda_input(x, self)
        lin = self.encoder[0]
        w32 = lin.weight.detach().contiguous()
        vals, idx, flags = _lib.encode_topk(x, self._w_bf16(), w32 if self.exact else None,
                                            lin.bias.detach(), int(self.topk), _lib.ACT_NONE,
                                            self.exact, want_flags=self.exact, sample=self._sample())
        self.last_flags = flags
        return SparseLatents(vals, idx, (x.shape[0], self.hidden_dim))

    def apply_topk_activation(self, h):
        """Dense [B, H] -> dense top-k-sparsified [B, H] (sae/baseline.py:34-40)."""
        if not h.is_cuda:
            raise RuntimeError("apply_topk_activation needs CUDA tensors (no CPU fallback)")
        vals, idx = _lib.topk_dense(h.contiguous().float(), int(self.topk))
        return _lib.densify(vals, idx, h.shape[1])

    def forward(self, x):
        if self.autograd and torch.is_grad_enabled():
            from .. import training
            return training.baseline_forward(self, x)
        latents = self.encode_topk(x)
        recon = _lib.decode_rows_f32(latents.values, latents.indices, self._dec_rows(), self.hidden_dim,
                                     self.input_dim, 1.0, self.decoder.bias.detach())
        return (latents.to_dense() if self.return_dense else latents), recon

    def normalize_decoder_weights(self):
        """Unit-norm decoder columns (training utility, sae/baseline.py:42-50)."""
        with torch.no_grad():
            w = self.decoder.weight.data
            self.decoder.weight.data = w / torch.clamp(torch.norm(w, dim=0, keepdim=True), min=1e-8)
