"""Training-side pieces adjacent to the forward (SURVEY.md 8f-4), on libqsae_b200.so (csrc/train.cu).

The reference trains with eager autograd over dense [B, H] latents and dense [H, D n_bits] soft-bit tensors
(training/trainer.py:88-173). The pieces of that backward that touch the quantised decoders are sparse in the same
way the forward is, and are provided here on the sparse forward quantities:

b_sae   `bsae_forward(model, x)` (what `BinarySAE.forward` runs when `model.autograd = True`): the reference's
        forward tuple, with `reconstruction` and `polarize_loss` attached to an autograd node, so the trainer's
        own lines -- loss = 0.5 * mse(recon, batch) + polarize_lambda * polarize_loss; loss.backward()
        (training/trainer.py:143-151) -- fill .grad of encoder.0.weight / encoder.0.bias / decoder.weight /
        decoder.bias. Backward of sae/binary.py:24-47 and :91-99: sparse outer products (16-byte vector reductions),
        row dots against the soft dictionary, one streaming pass over the bit logits that applies the sigmoid chain
        rule and adds the polarize gradient. The returned latent carries no gradient (the trainer only logs it).
        With model.deterministic = True the backward is qsae_bsae_backward instead: the baseline_sae latent-major
        pass below with gv = q <g, soft_rows[h]>, G[h] = q sum v g built per latent and the logit chain rule applied
        while G's row is in shared memory (G never reaches memory). Every gradient is then bit-deterministic.
q_sae   `QuantizedMatryoshkaDecoder.ste_backward(active, grad_levels)`: what loss.backward() leaves in
        decoder.weight.grad, weight_mirror.grad and bias.grad (STE through the sign, sae/quantized_matryoshka.py:94-124,
        joint_gradient = False), at any activity: from the active lists of `QuantizedMatryoshkaSAE.forward_active`
        (int32, a scatter of the level gradients) or from the bf16 activity mask of `forward_dense_active` (a
        tensor-core product mask^T g per level with the STE factor in its epilogue); `apply_secant_grad()`
        (:145-190). `qsae_trainer_decoder_grads` strings them together under the trainer's loss
        (training/trainer.py:88-113) and picks the route from the activity, so it runs from initialisation (~50 %
        of the latents active) to the end of the sparsity schedule.
        The encoder side of q_sae's backward is dense (the STE passes a gradient to every latent, :99) and is not
        built: its STE and sparsity-term semantics are not pinned here.
t_sae   `tsae_forward(model, x)` (what `TernarySparseAutoencoder.forward` runs when `model.autograd = True` and grad
        mode is on): the same (h, recon) as the plain forward, behind ONE autograd node, so the reference trainer's
        loop (training/trainer.py:152-173) runs as written: loss.backward() fills .grad of encoder.0.weight /
        encoder.0.bias / decoder.weight (and of x when it requires grad) and sets decoder.output_grad (the
        reference's backward hook, sae/ternary.py:24-25). With g = d loss / d recon and g_h = d loss / d h:
            gz = (g T + g_h) * 1[h > 0]: the dense encoder kernel over g against T^T with a ReLU-backward epilogue
                 (g T never reaches memory);
            grad W_enc = gz^T x, grad W_dec = mask * (g^T h) (the STE's weight * mask, sae/ternary.py:41-52),
            grad x = gz W_enc: tensor-core GEMMs over the batch (csrc/wgrad_sm100.cu) on the row-major batch
                 tensors as they are (MN-major operands, no transposes);
            grad b_enc = column sums of gz (atomics: not bit-deterministic, the other gradients are).
        model.exact (default) contracts three-part bf16 splits of every fp32 operand (fp32-accurate products);
        exact = False one bf16 product per GEMM.
        `STEWeights.init_mask / update_mask / mask_grad` (sae/ternary.py:27-90): exact RigL drop / grow by radix
        select on the device.
baseline_sae  `baseline_forward(model, x)` (what `BaselineSparseAutoencoder.forward` runs when `model.autograd = True` and
        grad mode is on): the same (h_sparse, recon) bits as the plain forward behind ONE autograd node (h_sparse, or
        latents.values when return_dense is off, is differentiable), so the reference trainer's baseline loop
        (training/trainer.py:168-173) runs as written: loss.backward() fills .grad of encoder.0.weight / encoder.0.bias /
        decoder.weight / decoder.bias (and of x when it requires grad). With g = d loss / d recon, g_h = d loss / d h and
        gv = <g, W_dec[:, h]> + g_h at each kept entry (qsae_baseline_backward, csrc/train.cu):
            grad W_enc[h] = sum gv x, grad b_enc[h] = sum gv, grad W_dec[:, h] = sum v g over the rows that selected h,
            from one latent-major pass over the entries grouped by latent (one writer per element, no atomics);
            grad b_dec = column sums of g (two fixed-order levels); grad x = gv W_enc (the sparse row decoder).
        Every gradient is bit-deterministic.
No CPU fallback: CUDA tensors only.
"""
from __future__ import annotations

import torch

from . import _lib
from .sparse import SparseLatents


def _acc_grad(p: torch.nn.Parameter) -> torch.Tensor:
    if p.grad is None:
        p.grad = torch.zeros_like(p, memory_format=torch.contiguous_format)
    return p.grad


class _BinarySAEFn(torch.autograd.Function):
    """(x, W_enc, b_enc, logits, b_dec) -> (values, indices, reconstruction, polarize_loss)."""

    @staticmethod
    def forward(ctx, x, w_enc, b_enc, logits, b_dec, model):
        dec = model.decoder
        lat = model.encode_topk(x)
        rows = dec._soft_rows()
        H, D = dec.in_features, dec.out_features
        recon = _lib.decode_rows_f32(lat.values, lat.indices, rows, H, D, dec.quantization_step, b_dec.detach())
        pol = dec.polarize_loss().detach().clone()
        ctx.save_for_backward(x, lat.values, lat.indices, logits, w_enc, rows)
        ctx.dims = (H, D, dec.n_bits, float(dec.quantization_step))
        ctx.deterministic = bool(model.deterministic)
        ctx.mark_non_differentiable(lat.values, lat.indices)
        return lat.values, lat.indices, recon, pol

    @staticmethod
    def backward(ctx, _g_vals, _g_idx, g_recon, g_pol):
        x, vals, idx, logits, w_enc, rows = ctx.saved_tensors
        H, D, n_bits, q = ctx.dims
        dev = x.device
        B = x.shape[0]
        g = (torch.zeros((B, D), dtype=torch.float32, device=dev) if g_recon is None
             else g_recon.contiguous().float())
        gp = 0.0 if g_pol is None else g_pol.detach().reshape(()).float().contiguous()
        if ctx.deterministic:
            want_x = ctx.needs_input_grad[0]
            gwe, gbe, glog, gbd, gx = _lib.bsae_backward(x.detach().contiguous(), vals, idx, g, rows,
                                                         logits.detach().contiguous(), q, gp,
                                                         w_enc.detach().contiguous() if want_x else None, n_bits, want_x)
            return gx, gwe, gbe, glog, gbd, None
        G = torch.zeros((H, D), dtype=torch.float32, device=dev)
        _lib.rows_scatter_add(vals, idx, g, G, scale=q)                       # d / d int_w
        grad_logits = torch.empty_like(logits, memory_format=torch.contiguous_format)
        _lib.bsae_logit_grad(logits.detach().contiguous(), G, D, n_bits, gp, grad_logits, accumulate=False)
        grad_bd = _lib.column_sum(g)
        grad_vals = _lib.rows_gather_dot(g, rows, idx, scale=q)               # d / d latent at the kept positions
        grad_we = torch.zeros((H, D), dtype=torch.float32, device=dev)
        grad_be = torch.zeros((H,), dtype=torch.float32, device=dev)
        _lib.rows_scatter_add(grad_vals, idx, x.detach().contiguous(), grad_we, scale=1.0, dst_col=grad_be)
        grad_x = None
        if ctx.needs_input_grad[0]:
            grad_x = _lib.decode_rows_f32(grad_vals, idx, w_enc.detach().contiguous(), H, D, 1.0, None)
        return grad_x, grad_we, grad_be, grad_logits, grad_bd, None


def bsae_forward(model, x):
    """BinarySAE.forward with an autograd node behind `reconstruction` and `polarize_loss` (see module docstring).
    Always decodes with the soft (sigmoid) dictionary: that is the function the reference differentiates
    (sae/binary.py:26-38), whatever `decode_mode` says about inference."""
    from .sae.base import require_cuda_input

    x = require_cuda_input(x, model)
    lin, dec = model.encoder[0], model.decoder
    vals, idx, recon, pol = _BinarySAEFn.apply(x, lin.weight, lin.bias, dec.weight, dec.bias, model)
    latents = SparseLatents(vals, idx, (x.shape[0], model.hidden_dim))
    return (latents.to_dense() if model.return_dense else latents), recon, pol


# ---- q_sae --------------------------------------------------------------------------------------------

def qsae_ste_backward(decoder, active_idx, grad_levels, batch_size: int | None = None, *, exact: bool = True) -> torch.Tensor:
    """Accumulate into decoder.weight.grad / weight_mirror.grad / bias.grad what autograd leaves there for upstream
    gradients grad_levels[i] = d loss / d result[i] (sae/quantized_matryoshka.py:94-124). `active_idx`: the int32
    active lists [B, cap] of forward_active, or the bf16 activity mask [B, H] of forward_dense_active (any activity;
    exact: the mask product takes three bf16 parts of each gradient, fp32-accurate, else one). Returns z2 [H] int32
    (the per-latent activity counts, :137) and stashes it for apply_secant_grad."""
    H, D = decoder.in_features, decoder.out_features
    dev = decoder.weight.device
    gl = [g.detach().contiguous().float() for g in grad_levels]
    if len(gl) != decoder.n_bits:
        raise ValueError(f"expected {decoder.n_bits} level gradients, got {len(gl)}")
    starts = decoder._level_starts_host()
    _, alpha = decoder._packed()
    if active_idx.dtype == torch.bfloat16:
        z2 = _lib.matryoshka_backward_dense(active_idx.contiguous(), gl, starts, decoder.weight.detach(),
                                            decoder.weight_mirror.detach(), alpha, exact, _acc_grad(decoder.weight),
                                            _acc_grad(decoder.weight_mirror))
    elif active_idx.dtype == torch.int32:
        M = torch.zeros((H, D), dtype=torch.float32, device=dev)
        z2 = torch.zeros((H,), dtype=torch.int32, device=dev)
        _lib.matryoshka_backward_scatter(active_idx, gl, starts, M, z2)
        _lib.matryoshka_backward_finish(decoder.weight.detach(), decoder.weight_mirror.detach(), M, None, alpha, starts, 0.0, 0,
                                        _acc_grad(decoder.weight), _acc_grad(decoder.weight_mirror))
    else:
        raise TypeError(f"ste_backward: int32 active lists or a bf16 activity mask expected, got {active_idx.dtype}")
    if decoder.allow_bias:
        _lib.column_sum(gl[0], 1.0, _acc_grad(decoder.bias))
    decoder._ctx = {"z2": z2, "batch_size": int(batch_size if batch_size is not None else active_idx.shape[0])}
    return z2


def qsae_apply_secant_grad(decoder) -> None:
    """decoder.apply_secant_grad() (sae/quantized_matryoshka.py:145-190): grad -= c m z2 alpha^2 Bsign s'(w)."""
    ctx = decoder._ctx
    if not isinstance(ctx, dict) or ctx.get("z2") is None:
        raise RuntimeError("apply_secant_grad: no training context; call forward_active + ste_backward first "
                           "(the reference stashes it in forward, sae/quantized_matryoshka.py:131-141)")
    _, alpha = decoder._packed()
    c = 1.0 / ctx["batch_size"] / decoder.out_features
    _lib.matryoshka_backward_finish(decoder.weight.detach(), decoder.weight_mirror.detach(), None, ctx["z2"], alpha,
                                    decoder._level_starts_host(), c, decoder.n_bits if decoder.joint_gradient else 0,
                                    _acc_grad(decoder.weight), _acc_grad(decoder.weight_mirror))


# Sparse / dense crossover of the decoder-side step: the sparse step (forward_active + scatter) grows with the mean
# list length L0 (the scatter issues L0 D reductions per row), the dense step (forward_dense_active + mask product)
# costs the same at any activity. Measured with tools/prof_qsae_train_dense.py on a B200 (1000 W limit;
# profiles/r6_qsae_train_dense.md), 512 -> 32768, n_bits 4, B = 4096, exact: sparse 0.93 ms at L0 = 33, 1.90 ms at
# 128, 2.59 ms at 256; dense 1.62-1.66 ms throughout. Linear between the first two, they cross at L0 ~ 100, L0 / H ~ 1/320.
# The step cannot know its own L0 before its forward, so the decision uses the previous step's (activity moves
# slowly under training); a step that overflows the lists goes dense at once.
_DENSE_TRAIN_L0_OVER_H = 1.0 / 320


def _qsae_train_active(model, x, active_cap: int) -> dict:
    """The forward of a training step with its activity: forward_active's lists, or forward_dense_active's bf16 mask
    when the model's regime is already dense, the previous step's mean list length passed the crossover, or the rows
    overflow the lists (the regime is then recorded as dense, as model(x) does). Records this step's L0 / H."""
    H = model.hidden_dim
    dense_ok = model.dense_mode != "never" and H % 8 == 0
    r = None
    if not model._known_dense() and not (dense_ok and model._train_l0_over_h > _DENSE_TRAIN_L0_OVER_H):
        r = model._forward_lists(x, active_cap)
        if r is None:
            if model.dense_mode == "never":
                raise RuntimeError("q_sae: a row has more active latents than the sparse path holds and dense_mode is 'never'")
            model._regime = (model._weights_key(), "dense")
    if r is None:
        r = model.forward_dense_active(x)
    model._train_l0_over_h = float(r["level_counts"].sum()) / max(1, x.shape[0] * H)
    return r


def qsae_trainer_decoder_grads(model, x, active_cap: int = 256):
    """One q_sae step of the reference trainer as far as the decoder is concerned (training/trainer.py:88-113):
    forward, recon_loss = sum_i 0.5 * mse(result_i, x), decoder gradients of it, apply_secant_grad. Any activity: the
    route (active lists and a scatter, or an activity mask and a tensor-core product) follows the activity, and
    model.last_path records which forward ran. -> dict(recon_losses [n_bits] device tensor, latent_groups,
    reconstruction_levels)."""
    x = x.contiguous().float()
    out = _qsae_train_active(model, x, active_cap)
    B, D = x.shape
    levels = out["reconstruction_levels"]
    grads = [(r - x) / float(B * D) for r in levels]
    active = out["active_mask"] if "active_mask" in out else out["active_idx"]
    qsae_ste_backward(model.decoder, active, grads, B, exact=model.exact)
    qsae_apply_secant_grad(model.decoder)
    losses = torch.stack([0.5 * ((r - x) ** 2).mean() for r in levels])
    return {"recon_losses": losses, "latent_groups": out["latent_groups"], "reconstruction_levels": levels}


# ---- t_sae: autograd node ------------------------------------------------------------------------------

class _TernarySAEFn(torch.autograd.Function):
    """(x, W_enc, b_enc, W_dec) -> (h, recon), one node: g T feeds the ReLU mask inside one epilogue."""

    @staticmethod
    def forward(ctx, x, w_enc, b_enc, w_dec, model):
        ctx.set_materialize_grads(False)
        h, recon = model._forward_dense(x.detach())
        dec = model.decoder
        # what the forward contracted, kept for the backward (the reference differentiates through these values)
        ctx.t_t = dec._ternary_t()
        ctx.mask = dec.mask.detach().contiguous().float()
        ctx.w_parts = model._enc_parts()
        ctx.exact = bool(model.exact)
        ctx.dec = dec
        ctx.save_for_backward(x, h)
        return h, recon

    @staticmethod
    def backward(ctx, g_h, g_recon):
        x, h = ctx.saved_tensors
        B, D = x.shape
        if g_recon is not None:
            g = g_recon.detach().contiguous().float()
            ctx.dec.output_grad = g                   # the reference's backward hook (sae/ternary.py:24-25)
        else:
            g = torch.zeros((B, D), dtype=torch.float32, device=x.device)
        gh = None if g_h is None else g_h.detach().contiguous().float()
        gwe, gbe, gwd, gx = _lib.tsae_backward(x.detach().contiguous(), h.detach(), g, gh, ctx.t_t, ctx.mask, ctx.w_parts,
                                               ctx.exact, want_grad_x=ctx.needs_input_grad[0])
        return gx, gwe, gbe, gwd, None


def tsae_forward(model, x):
    """TernarySparseAutoencoder.forward with an autograd node behind (h, recon) (see module docstring)."""
    from .sae.base import require_cuda_input

    x = require_cuda_input(x, model)
    lin = model.encoder[0]
    h, recon = _TernarySAEFn.apply(x, lin.weight, lin.bias, model.decoder.weight, model)
    model.decoder.input_activations = h.detach()  # the reference's forward hook (sae/ternary.py:21-22)
    return h, recon


# ---- baseline_sae: autograd node ------------------------------------------------------------------------

class _BaselineSAEFn(torch.autograd.Function):
    """(x, W_enc, b_enc, W_dec, b_dec) -> (h_sparse [B, H] or values [B, k], indices, recon)."""

    @staticmethod
    def forward(ctx, x, w_enc, b_enc, w_dec, b_dec, model):
        ctx.set_materialize_grads(False)
        lat = model.encode_topk(x.detach())
        rows = model._dec_rows()
        recon = _lib.decode_rows_f32(lat.values, lat.indices, rows, model.hidden_dim, model.input_dim, 1.0, b_dec.detach())
        ctx.dense = bool(model.return_dense)
        ctx.rows = rows
        ctx.save_for_backward(x, lat.values, lat.indices, w_enc)
        ctx.mark_non_differentiable(lat.indices)
        return (lat.to_dense() if ctx.dense else lat.values), lat.indices, recon

    @staticmethod
    def backward(ctx, g_lat, _g_idx, g_recon):
        x, vals, idx, w_enc = ctx.saved_tensors
        B, D = x.shape
        g = (torch.zeros((B, D), dtype=torch.float32, device=x.device) if g_recon is None
             else g_recon.detach().contiguous().float())
        gl = None if g_lat is None else g_lat.detach().contiguous().float()
        gwe, gbe, gwd, gbd, gx = _lib.baseline_backward(x.detach(), vals, idx, g, gl if ctx.dense else None,
                                                        None if ctx.dense else gl, w_enc.detach().contiguous(), ctx.rows,
                                                        want_grad_x=ctx.needs_input_grad[0])
        return gx, gwe, gbe, gwd, gbd, None


def baseline_forward(model, x):
    """BaselineSparseAutoencoder.forward with an autograd node behind (h_sparse, recon) (see module docstring)."""
    from .sae.base import require_cuda_input

    x = require_cuda_input(x, model)
    lin, dec = model.encoder[0], model.decoder
    h, idx, recon = _BaselineSAEFn.apply(x, lin.weight, lin.bias, dec.weight, dec.bias, model)
    if model.return_dense:
        return h, recon
    return SparseLatents(h, idx, (x.shape[0], model.hidden_dim)), recon


# ---- t_sae: RigL mask maintenance ---------------------------------------------------------------------

def rigl_init_mask(ste, sparsity: float) -> None:
    """STEWeights.init_mask (sae/ternary.py:27-39)."""
    w = ste.weight.data
    if not w.is_cuda:
        raise RuntimeError("STEWeights.init_mask runs only on CUDA (no CPU fallback)")
    n_inactive = int(w.numel() * sparsity)
    mask = torch.ones_like(w, memory_format=torch.contiguous_format)
    wc = w if w.is_contiguous() else w.contiguous()
    _lib.rigl_init_mask(wc, mask, n_inactive)
    if wc is not w:
        w.copy_(wc)
    ste.mask = mask
    ste.invalidate()


def rigl_update_mask(ste, f_decay: float, sparsity_rate: float = 0.7) -> None:
    """STEWeights.update_mask (sae/ternary.py:54-87)."""
    w = ste.weight.data
    if not w.is_cuda:
        raise RuntimeError("STEWeights.update_mask runs only on CUDA (no CPU fallback)")
    n_drop = int(f_decay * (1 - sparsity_rate) * w.numel())
    n_grow = n_drop
    a_mean = d_mean = None
    if n_grow > 0 and ste.input_activations is not None:
        if ste.output_grad is None:
            raise RuntimeError("update_mask: output_grad is not set (the reference captures it in a backward hook, "
                               "sae/ternary.py:24-25); set model.autograd = True and call loss.backward(), or assign "
                               "decoder.output_grad = d loss / d reconstruction")
        a = ste.input_activations.detach().contiguous().float()
        d = ste.output_grad.detach().contiguous().float()
        a_mean = _lib.column_sum(a, 1.0 / a.shape[0])
        d_mean = _lib.column_sum(d, 1.0 / d.shape[0])
    mask = ste.mask.contiguous().float()
    wc = w if w.is_contiguous() else w.contiguous()
    _lib.rigl_update_mask(wc, mask, a_mean, d_mean, n_drop, n_grow if a_mean is not None else 0)
    if wc is not w:
        w.copy_(wc)
    ste.mask = mask
    ste.invalidate()


def rigl_mask_grad(ste) -> None:
    """STEWeights.mask_grad (sae/ternary.py:89-90)."""
    g = ste.weight.grad
    if g is None:
        raise AttributeError("mask_grad: weight.grad is None")
    gc = g.data if g.is_contiguous() else g.data.contiguous()
    _lib.mul_inplace(gc, ste.mask.contiguous().float())
    if gc is not g.data:
        g.data.copy_(gc)
