"""CPU pin of tests/tsae_oracle.tsae_training_grads against torch float64 autograd on a restatement of the reference
t_sae forward: encoder = Linear + ReLU (sae/ternary.py:95-98), decoder = F.linear(h, ste) with
ste = (T - Wd * mask).detach() + Wd * mask, T = sign(Wd) * (|Wd| >= 0.5) (STEWeights.forward, :41-52).

No stored reference outputs exist for this step: the reference checkout is not part of this repository, so the
restatement above stands in for it (tests/golden holds only what was generated from the reference before)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import tsae_oracle as to


def _restated_forward(x, We, be, Wd, mask):
    h = F.relu(F.linear(x, We, be))
    T = torch.sign(Wd) * (Wd.abs() >= 0.5)
    ste = (T - Wd * mask).detach() + Wd * mask
    return h, F.linear(h, ste)


@pytest.mark.parametrize("B,D,H,with_gh", [(7, 8, 16, False), (33, 24, 40, True), (64, 64, 128, True)])
def test_tsae_training_grads_match_torch_autograd(B, D, H, with_gh):
    rng = np.random.default_rng(B * 1000 + H)
    x = rng.standard_normal((B, D))
    We = rng.standard_normal((H, D)) / np.sqrt(D)
    be = rng.standard_normal(H) * 0.1
    Wd = rng.standard_normal((D, H))
    mask = (rng.random((D, H)) > 0.3).astype(np.float64)
    lam = 0.01
    t = {k: torch.tensor(v, dtype=torch.float64, requires_grad=k != "mask") for k, v in
         dict(x=x, We=We, be=be, Wd=Wd, mask=mask).items()}
    h, recon = _restated_forward(t["x"], t["We"], t["be"], t["Wd"], t["mask"])
    # the reference trainer's loss (training/trainer.py:152-173), plus an L1 term on h for the g_h path
    loss = 0.5 * F.mse_loss(recon, t["x"].detach())
    if with_gh:
        loss = loss + lam * h.abs().mean()
    loss.backward()
    g = (recon.detach() - t["x"].detach()).numpy() / (B * D)
    g_h = lam * np.sign(h.detach().numpy()) / (B * H) if with_gh else None
    o = to.tsae_training_grads(x, We, be, Wd, mask, g, g_h)
    np.testing.assert_allclose(o["h"], h.detach().numpy(), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(o["recon"], recon.detach().numpy(), rtol=1e-12, atol=1e-12)
    for name, key in (("We", "grad_we"), ("be", "grad_be"), ("Wd", "grad_wd")):
        np.testing.assert_allclose(o[key], t[name].grad.numpy(), rtol=1e-10, atol=1e-14, err_msg=name)
    # x also feeds the mse target, detached in the trainer; the input gradient is the one through the encoder
    np.testing.assert_allclose(o["grad_x"], t["x"].grad.numpy(), rtol=1e-10, atol=1e-14)
    assert np.any(mask * (g.T @ h.detach().numpy()) != g.T @ h.detach().numpy())   # the mask gates something
