"""CPU pin of tests/baseline_oracle.baseline_training_grads against torch float64 autograd on a restatement of the
reference baseline forward (SURVEY A.2: Linear -> topk(k) -> zeros_like + scatter_ -> Linear, sae/baseline.py:17-40), the
restatement itself against the stored forward fixtures, and the host-side argument checks of qsae_baseline_backward."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from quantizedsae_b200 import _lib
from tests import baseline_oracle as bo
from tests.golden import cases


def _restated_forward(x, We, be, Wd, bd, k):
    z = F.linear(x, We, be)
    v, i = torch.topk(z, k)
    h = torch.zeros_like(z).scatter_(1, i, v)
    return h, F.linear(h, Wd, bd)


def _inputs(name):
    inp = cases.baseline_inputs(cases.BASELINE_CASES[name])
    return {k: torch.tensor(v.astype(np.float64), requires_grad=True) for k, v in inp.items()}


@pytest.mark.parametrize("name", list(cases.BASELINE_CASES))
def test_restated_forward_matches_golden(golden_dir, name):
    g = np.load(golden_dir / f"{name}.npz")
    t = _inputs(name)
    with torch.no_grad():
        h, recon = _restated_forward(t["x"], t["We"], t["be"], t["Wd"], t["bd"], int(g["k"]))
    h = h.numpy()
    B = h.shape[0]
    got_vals = h[np.arange(B)[:, None], g["latent_idx"]]
    assert np.all((h != 0).sum(1) == int(g["k"]))
    np.testing.assert_allclose(got_vals, g["latent_vals"], rtol=1e-5, atol=1e-6)   # the same entries are kept
    rms = float(np.sqrt(np.mean(g["recon"].astype(np.float64) ** 2)))
    np.testing.assert_allclose(recon.numpy(), g["recon"], rtol=1e-5, atol=1e-5 * rms)


@pytest.mark.parametrize("with_l1", [False, True])
@pytest.mark.parametrize("name", list(cases.BASELINE_CASES))
def test_baseline_training_grads_match_torch_autograd(name, with_l1):
    t = _inputs(name)
    k = 32
    h, recon = _restated_forward(t["x"], t["We"], t["be"], t["Wd"], t["bd"], k)
    h.retain_grad()
    recon.retain_grad()
    # the reference trainer's loss (training/trainer.py:168-173), plus an L1 term on h for the g_h path
    loss = 0.5 * F.mse_loss(recon, t["x"].detach())
    if with_l1:
        loss = loss + 0.01 * h.abs().mean()
    loss.backward()
    g = recon.grad.numpy()
    hd = h.detach().numpy()
    g_h = 0.01 * np.sign(hd) / hd.size if with_l1 else None     # the L1 term's own d / d h
    if with_l1:   # h.grad is that plus the reconstruction's share g Wd: the oracle adds the latter itself
        np.testing.assert_allclose(h.grad.numpy(), g_h + g @ t["Wd"].detach().numpy(), rtol=1e-10, atol=1e-15)
    o = bo.baseline_training_grads(*(t[n].detach().numpy() for n in ("x", "We", "be", "Wd", "bd")), g, g_h, k=k)
    np.testing.assert_allclose(o["h"], h.detach().numpy(), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(o["recon"], recon.detach().numpy(), rtol=1e-12, atol=1e-12)
    for name_, key in (("We", "grad_we"), ("be", "grad_be"), ("Wd", "grad_wd"), ("bd", "grad_bd"), ("x", "grad_x")):
        np.testing.assert_allclose(o[key], t[name_].grad.numpy(), rtol=1e-10, atol=1e-15, err_msg=name_)


def test_baseline_backward_validates_arguments_without_a_device():
    lib = _lib.load()
    n = C.c_size_t(0)
    assert lib.qsae_baseline_backward_workspace_bytes(16, 2048, 64, 32, C.byref(n)) == 0 and n.value > 0
    assert lib.qsae_baseline_backward_workspace_bytes(0, 2048, 64, 32, C.byref(n)) == 0
    assert lib.qsae_baseline_backward_workspace_bytes(16, 2048, 64, 32, None) == -1
    assert lib.qsae_baseline_backward_workspace_bytes(-1, 2048, 64, 32, C.byref(n)) == -1
    assert lib.qsae_baseline_backward_workspace_bytes(16, 2048, 520, 32, C.byref(n)) == -1          # D > 512
    assert lib.qsae_baseline_backward_workspace_bytes(16, 2048, 60, 32, C.byref(n)) == -1           # D % 8
    assert b"multiple of 8" in lib.qsae_last_error()
    assert lib.qsae_baseline_backward_workspace_bytes(16, 0, 64, 32, C.byref(n)) == -1              # H = 0
    assert lib.qsae_baseline_backward_workspace_bytes(16, 2048, 64, 0, C.byref(n)) == -1            # k = 0
    assert lib.qsae_baseline_backward_workspace_bytes(16, 2048, 64, 4096, C.byref(n)) == -5         # k > H
    assert lib.qsae_baseline_backward_workspace_bytes(1 << 20, 4096, 64, 4096, C.byref(n)) == -1    # B k >= 2^31
    assert lib.qsae_baseline_backward_workspace_bytes(16, 2048, 64, 32, C.byref(n)) == 0
    need = n.value
    p = 1 << 20           # never dereferenced: every call below fails its host-side checks
    args = lambda gh, gvals, ws_bytes, gwe=p: (p, p, p, p, gh, gvals, p, p, 16, 2048, 64, 32, gwe, p, p, p, None, p, ws_bytes, None)
    assert lib.qsae_baseline_backward(*args(p, p, need)) == -1                                       # both g_h forms
    assert b"not both" in lib.qsae_last_error()
    assert lib.qsae_baseline_backward(*args(None, None, need - 1)) == -2                             # workspace too small
    assert lib.qsae_baseline_backward(*args(None, None, need, gwe=None)) == -1                       # null gradient
    assert lib.qsae_baseline_backward(*args(None, None, need, gwe=p + 4)) == -1                      # alignment
    assert b"16-byte" in lib.qsae_last_error()
    bad = list(args(None, None, need))
    bad[10] = 520                                                                                     # D > 512
    assert lib.qsae_baseline_backward(*bad) == -1
    bad = list(args(None, None, need))
    bad[0] = None                                                                                     # x missing
    assert lib.qsae_baseline_backward(*bad) == -1
    bad = list(args(None, None, need))
    bad[6] = None                                                                                     # grad_x needs W_enc
    bad[16] = p
    assert lib.qsae_baseline_backward(*bad) == -1
    assert b"W_enc" in lib.qsae_last_error()


def test_baseline_autograd_has_no_cpu_path():
    import quantizedsae_b200 as Q

    m = Q.BaselineSparseAutoencoder(16, 64)
    assert m.autograd is False
    m.autograd = True
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros((4, 16)))
