"""b_sae: BinarySAE / binary_decoder with the reference's constructor, attributes, state_dict
and forward return structure (sae/binary.py), running on libqsae_b200.so.

forward(x) -> (sparse_latent, reconstruction, polarize_loss)                (sae/binary.py:103)

What differs from the reference is only *how* it is computed:
  * encoder Linear + topk (sae/binary.py:92-94) -> one fused tcgen05 kernel, no dense [B,H] z;
  * mask/scatter/multiply (:96-99)             -> never executed; `sparse_latent` is built from
    the k survivors (dense on request, see `return_dense`);
  * sigmoid over all bit logits + weighted bit sum + dense matmul (:26-38), recomputed on every
    call by the reference -> a packed dictionary cached per weight version and a sparse gather.

decode_mode
  "auto" (default): use the packed two's-complement dictionary when the logits are polarised
          (max |sigmoid(w) - bit| <= polar_tol, i.e. the soft forward *is* the hard dictionary
          to float32 accuracy), otherwise the float32 soft dictionary -- either way the result
          matches the reference forward within the stated tolerance;
  "int":  always the hard dictionary == quantized_int_weights() * quantization_step, the
          deployed/quantised model (inference/framework.py:114-124);
  "soft": always the soft dictionary (reference forward semantics on any logits).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .. import _lib
from ..sparse import SparseLatents
from .base import PreparedCache, invalidate_prepared, SparseAutoencoder, param_key, require_cuda_input


class binary_decoder(nn.Module):
    def __init__(self, in_features, out_features, gamma=4.0, n_bits=8):
        super().__init__()
        self.in_features = in_features          # hidden_dim (dictionary rows)
        self.out_features = out_features        # input_dim
        self.n_bits = n_bits
        self.scale_factor = 2 ** n_bits
        self.gamma = gamma
        self.quantization_step = gamma / (2 ** (n_bits - 1))
        # bit i of output feature d lives at column d*n_bits + i (LSB first, sign bit last)
        self.weight = nn.Parameter(torch.empty(in_features, out_features * n_bits))
        self.bias = nn.Parameter(torch.zeros(out_features))
        nn.init.kaiming_normal_(self.weight)
        self.decode_mode = "auto"
        self.polar_tol = 1e-6
        self._prep = PreparedCache()

    # ---- cached device-side dictionaries -------------------------------------------------

    def invalidate(self) -> None:
        """Forget the prepared copies of the weights (needed after in-place edits through `.data`, which bump no version
        counter; see sae/base.py)."""
        invalidate_prepared(self)

    refresh = invalidate
    def _packed(self):
        """(packed dictionary, polarize_loss, max |p - bit|) for the current logits."""
        if not self.weight.is_cuda:
            raise RuntimeError("binary_decoder: the packed dictionary is built by a CUDA kernel; "
                               "move the module to the GPU (no CPU fallback)")
        return self._prep.get(
            "packed", param_key(self.weight),
            lambda: _lib.pack_bitplanes(self.weight.detach(), self.out_features, self.n_bits))

    def _soft_rows(self):
        return self._prep.get(
            "soft", param_key(self.weight),
            lambda: _lib.dequant_soft(self.weight.detach(), self.out_features, self.n_bits))

    def resolved_mode(self) -> str:
        if self.decode_mode in ("int", "soft"):
            return self.decode_mode
        if self.decode_mode != "auto":
            raise ValueError(f"unknown decode_mode {self.decode_mode!r}")
        return "int" if self._packed()[2] <= self.polar_tol else "soft"

    def polarize_loss(self) -> torch.Tensor:
        """mean(p (1-p) 2^i) (sae/binary.py:41-42); weight-only, cached per weight version."""
        return self._prep.get(
            "pol_t", param_key(self.weight),
            lambda: torch.tensor(self._packed()[1], dtype=torch.float32, device=self.weight.device))

    # ---- forward --------------------------------------------------------------------------
    def decode_sparse(self, latents: SparseLatents) -> torch.Tensor:
        H, D = self.in_features, self.out_features
        bias = self.bias.detach()
        if self.resolved_mode() == "int":
            packed = self._packed()[0]
            fn = _lib.decode_int4 if self.n_bits <= 4 else _lib.decode_int8
            return fn(latents.values, latents.indices, packed, H, D, self.quantization_step, bias)
        return _lib.decode_rows_f32(latents.values, latents.indices, self._soft_rows(), H, D,
                                    self.quantization_step, bias)

    def forward(self, latent, true_sum=None):
        """reference signature (latent, true_sum) -> (reconstruction, polarize_loss); the second
        argument is unused there too (sae/binary.py:24). `latent` may be SparseLatents or the
        dense [B, H] matrix the reference passes (rows with at most QSAE_MAX_K_LARGE non-zeros)."""
        if not isinstance(latent, SparseLatents):
            latent = sparsify_dense(latent)
        return self.decode_sparse(latent), self.polarize_loss()

    # ---- exports --------------------------------------------------------------------------
    def quantized_int_weights(self):
        """[H, D] float tensor of integers in [-2^(n-1), 2^(n-1)-1] (sae/binary.py:49-58)."""
        with torch.no_grad():
            packed = self._packed()[0]
            if self.n_bits <= 4:
                lo = (packed & 0xF).to(torch.int8)
                hi = (packed >> 4).to(torch.int8)
                both = torch.stack((lo, hi), dim=-1).reshape(packed.shape[0], -1)
                ints = torch.where(both >= 8, both - 16, both)
            else:
                ints = packed.view(torch.int8)
            return ints.to(self.weight.dtype)

    def quantized_int_weights_continuous(self):
        """Soft (sigmoid) effective weights (sae/binary.py:60-69)."""
        return self._soft_rows().clone()


def sparsify_dense(latent: torch.Tensor) -> SparseLatents:
    """Dense [B, H] latent (as the reference passes to its decoder, sae/binary.py:24) -> SparseLatents holding the
    non-zeros of each row in ascending latent order (qsae_compact_dense: one counting and one filling launch)."""
    if not latent.is_cuda:
        raise RuntimeError("binary_decoder.forward needs CUDA tensors (no CPU fallback)")
    latent = latent.contiguous().float()
    idx, vals, cnt = _lib.compact_dense(latent, 0, want_vals=True)
    if idx.shape[1] > _lib.QSAE_MAX_K_LARGE:
        raise RuntimeError(f"dense latent with {idx.shape[1]} non-zeros per row exceeds QSAE_MAX_K_LARGE={_lib.QSAE_MAX_K_LARGE}")
    return SparseLatents(vals, idx, tuple(latent.shape))


class BinarySAE(SparseAutoencoder):
    def __init__(self, input_dim, hidden_dim, gamma=4.0, n_bits=8):
        super().__init__(input_dim, hidden_dim)
        self.n_bits = n_bits
        self.input_dim = input_dim
        self.hidden_dim = hidden_dim
        self.k = 0.002                       # fraction of latents kept: int(hidden_dim * k)
        self.encoder = nn.Sequential(nn.Linear(input_dim, hidden_dim))
        nn.init.xavier_uniform_(self.encoder[0].weight, gain=1)
        nn.init.zeros_(self.encoder[0].bias)
        self.decoder = binary_decoder(hidden_dim, input_dim, gamma=gamma, n_bits=self.n_bits)
        # B200-path options (not constructor arguments, so positional construction is unchanged)
        self.return_dense = True             # reference returns a dense [B,H] latent
        self.exact = True                    # fp32 re-scoring of the tensor-core candidates
        self.last_flags = None               # rows whose selection was not certified (exact mode)
        self.autograd = False                # True: forward attaches the sparse backward (quantizedsae_b200/training.py)
        self.deterministic = False           # with autograd: the bit-deterministic latent-major backward (qsae_bsae_backward)
        self.ordered_latents = True          # False (fast mode, k > QSAE_MAX_K): sparse latents as unordered winner sets
        self._prep = PreparedCache()

    def _w_bf16(self):
        w = self.encoder[0].weight
        return self._prep.get("w_bf16", param_key(w), lambda: _lib.cast_bf16(w.detach().contiguous()))

    def _sample(self):
        """Sampled dictionary rows for the prior-threshold pre-pass (None for small dictionaries)."""
        lin = self.encoder[0]
        return self._prep.get("sample", param_key(lin.weight, lin.bias),
                              lambda: _lib.prepare_sample(self._w_bf16(), lin.bias.detach()))

    def encode(self, x):
        """Dense pre-activations [B, H] (sae/base.py:16-19). Exact fp32 CUDA-core kernel; the
        throughput path is forward()/encode_topk(), which never builds this matrix."""
        x = require_cuda_input(x, self)
        lin = self.encoder[0]
        return _lib.encode_dense(x, lin.weight.detach().contiguous(), lin.bias.detach())

    def encode_topk(self, x) -> SparseLatents:
        x = require_cuda_input(x, self)
        lin = self.encoder[0]
        k = int(self.hidden_dim * self.k)
        w32 = lin.weight.detach().contiguous()
        vals, idx, flags = _lib.encode_topk(x, self._w_bf16(), w32 if self.exact else None,
                                            lin.bias.detach(), k, _lib.ACT_NONE, self.exact,
                                            want_flags=self.exact, sample=self._sample())
        self.last_flags = flags
        return SparseLatents(vals, idx, (x.shape[0], self.hidden_dim))

    def forward(self, x):
        if not self.ordered_latents and not self.exact:
            with _lib.unordered_topk():
                return self._forward(x)
        return self._forward(x)

    def _forward(self, x):
        if self.autograd and torch.is_grad_enabled():
            # training (training/trainer.py:143-151): soft-bit forward with the sparse backward attached
            from .. import training
            return training.bsae_forward(self, x)
        if self.decoder.resolved_mode() == "int":
            # packed dictionary: encoder + top-k + sparse decode behind one C-ABI call (qsae_bsae_forward)
            x = require_cuda_input(x, self)
            lin, dec = self.encoder[0], self.decoder
            w32 = lin.weight.detach().contiguous()
            vals, idx, flags, recon = _lib.bsae_forward(
                x, self._w_bf16(), w32 if self.exact else None, lin.bias.detach(), int(self.hidden_dim * self.k),
                dec._packed()[0], self.n_bits, dec.quantization_step, dec.bias.detach(), exact=self.exact,
                want_flags=self.exact, sample=self._sample())
            self.last_flags = flags
            latents = SparseLatents(vals, idx, (x.shape[0], self.hidden_dim))
        else:
            latents = self.encode_topk(x)
            recon = self.decoder.decode_sparse(latents)
        out_latent = latents.to_dense() if self.return_dense else latents
        return out_latent, recon, self.decoder.polarize_loss()
