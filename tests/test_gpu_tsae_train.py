"""t_sae training step on the GPU: the weight-gradient GEMM (qsae_wgrad), the backward node behind
TernarySparseAutoencoder.forward with autograd = True (qsae_tsae_backward), and the reference trainer's t_sae loop
(training/trainer.py:152-173): forward, loss, backward, mask_grad, optimizer step, update_mask.

Precision contract. The reference is the float64 product; its bound is S = |A|^T |B|, the elementwise sum of
absolute products (float64 as well). Exact mode (module default): every gradient within 2e-5 S; fast mode: within
2^-7 S. The gradients are checked against float64 products of the GPU's own forward quantities (h, and the upstream
gradients autograd hands to the node), which is what torch autograd on the reference differentiates. The largest
observed error is printed as a fraction of S. encoder.0.bias.grad is a column sum with atomics: not bit-deterministic.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import quantizedsae_b200 as Q
from oracle import train_oracle as TO
from quantizedsae_b200 import _lib as L
from tests import tsae_oracle
from tests.golden import cases

pytestmark = pytest.mark.gpu

TOL_EXACT = 2e-5
TOL_FAST = 2.0 ** -7


def _frac(got, ref, S):
    """max |got - ref| / S over all entries (an entry with S == 0 must be exact)."""
    err = (got.double() - ref).abs()
    if bool(((S == 0) & (err > 0)).any()):
        return float("inf")
    return float((err / S.clamp_min(1e-300)).max()) if err.numel() else 0.0


def _split(t, n_parts):
    return L.split_bf16x3(t) if n_parts == 3 else (L.cast_bf16(t),)


# ---------------------------------------------------------------------------------------------------------------
# the weight-gradient GEMM on its own
# ---------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n_parts", [1, 3])
@pytest.mark.parametrize("M,N", [(8, 16), (64, 2048), (512, 4096), (4096, 512), (248, 520)])
@pytest.mark.parametrize("B", [1, 37, 130, 4096])
def test_wgrad_vs_fp64(cuda_device, B, M, N, n_parts):
    g = torch.Generator(device=cuda_device).manual_seed(B * 7919 + M * 31 + N)
    a = torch.randn((B, M), device=cuda_device, generator=g)
    b = torch.randn((B, N), device=cuda_device, generator=g) * 3.0
    c = L.wgrad(_split(a, n_parts), _split(b, n_parts))
    ref = a.double().T @ b.double()
    S = a.double().abs().T @ b.double().abs()
    frac = _frac(c, ref, S)
    tol = TOL_EXACT if n_parts == 3 else TOL_FAST
    print(f"wgrad B={B} M={M} N={N} parts={n_parts}: max err / S = {frac:.3e} (bound {tol:.1e})")
    assert tuple(c.shape) == (M, N)
    assert frac <= tol


@pytest.mark.parametrize("n_parts", [1, 3])
@pytest.mark.parametrize("B,H,D", [(37, 264, 64), (256, 2048, 512), (130, 1000, 8)])
def test_wgrad_kmajor_a_vs_fp64(cuda_device, B, H, D, n_parts):
    """x.grad = gz W_enc: A = gz [B, H] is K-major (K = H), B = W_enc [H, D]."""
    g = torch.Generator(device=cuda_device).manual_seed(B + H + D)
    gz = torch.randn((B, H), device=cuda_device, generator=g)
    w = torch.randn((H, D), device=cuda_device, generator=g)
    c = L.wgrad(_split(gz, n_parts), _split(w, n_parts), a_kmajor=True)
    ref = gz.double() @ w.double()
    S = gz.double().abs() @ w.double().abs()
    frac = _frac(c, ref, S)
    tol = TOL_EXACT if n_parts == 3 else TOL_FAST
    print(f"wgrad K-major A B={B} H={H} D={D} parts={n_parts}: max err / S = {frac:.3e}")
    assert frac <= tol


# ---------------------------------------------------------------------------------------------------------------
# the module's backward node
# ---------------------------------------------------------------------------------------------------------------

ODD_CASES = {
    "b37_d64_h1000": dict(D=64, H=1000, B=37, bf16=False, seed=71),     # H % 128 != 0, B not a multiple of 128
    "b130_d8_h264": dict(D=8, H=264, B=130, bf16=False, seed=72),       # D = 8
    "b300_d512_h2056": dict(D=512, H=2056, B=300, bf16=True, seed=73),
    "b130_d392_h1000": dict(D=392, H=1000, B=130, bf16=False, seed=74),     # 7 K chunks, the last one partial
    "b300_d456_h2056": dict(D=456, H=2056, B=300, bf16=True, seed=75),      # 8 K chunks above D = 448, the last partial
}
STEP_CASES = {**cases.TSAE_CASES, **ODD_CASES}


def _model(cfg, dev, exact, mask_density=0.7):
    inp = cases.tsae_inputs(cfg)
    m = Q.TernarySparseAutoencoder(cfg["D"], cfg["H"])
    with torch.no_grad():
        m.encoder[0].weight.copy_(torch.from_numpy(inp["We"]))
        m.encoder[0].bias.copy_(torch.from_numpy(inp["be"]))
        m.decoder.weight.copy_(torch.from_numpy(inp["Wd"]))
    m.to(dev)
    m.exact = exact
    m.autograd = True
    rng = np.random.default_rng(cfg["seed"] + 1)
    m.decoder.mask = torch.from_numpy((rng.random((cfg["D"], cfg["H"])) < mask_density).astype(np.float32)).to(dev)
    return m, torch.from_numpy(inp["x"]).to(dev)


def _step(m, x, lam):
    """The reference trainer's loss (training/trainer.py:152-173), plus an L1 term on h when lam > 0.
    -> (loss, h, recon, g = d loss / d recon, g_h = d loss / d h or None) with g / g_h captured by hooks."""
    seen = {}
    h, recon = m(x)
    recon.register_hook(lambda g: seen.__setitem__("g", g.detach().clone()))
    loss = 0.5 * F.mse_loss(recon, x.detach())
    if lam > 0:
        h.register_hook(lambda g: seen.__setitem__("g_h", g.detach().clone()))
        loss = loss + lam * h.abs().mean()
    loss.backward()
    return loss, h, recon, seen["g"], seen.get("g_h")


def _reference(m, x, h, g, g_h, mask):
    """float64 gradients and bounds from the GPU's h and upstream gradients (what autograd on the reference computes)."""
    Wd = m.decoder.weight.detach().double()
    T = torch.sign(Wd) * (Wd.abs() >= 0.5)
    We = m.encoder[0].weight.detach().double()
    xd, hd, gd = x.double(), h.detach().double(), g.double()
    pos = hd > 0
    gz = gd @ T
    S_gz = gd.abs() @ T.abs()
    if g_h is not None:
        gz = gz + g_h.double()
        S_gz = S_gz + g_h.double().abs()
    gz = torch.where(pos, gz, torch.zeros_like(gz))
    S_gz = torch.where(pos, S_gz, torch.zeros_like(S_gz))
    agz = S_gz   # |gz| <= S_gz: bounds of the products built on gz use it
    md = mask.double()
    return {
        "grad_we": (gz.T @ xd, agz.T @ xd.abs()),
        "grad_be": (gz.sum(0), agz.sum(0)),
        "grad_wd": (md * (gd.T @ hd), md * (gd.abs().T @ hd.abs())),
        "grad_x": (gz @ We, agz @ We.abs()),
    }


@pytest.mark.parametrize("with_gh", [False, True])
@pytest.mark.parametrize("exact", [True, False])
@pytest.mark.parametrize("name", list(STEP_CASES))
def test_tsae_backward_matches_oracle(cuda_device, name, exact, with_gh):
    cfg = STEP_CASES[name]
    m, x = _model(cfg, cuda_device, exact)
    x = x.clone().requires_grad_(True)
    mask = m.decoder.mask.clone()
    loss, h, recon, g, g_h = _step(m, x, 1e-2 if with_gh else 0.0)
    # forward values are the plain forward's, bit for bit
    with torch.no_grad():
        h0, r0 = m._forward_dense(x.detach())
    assert torch.equal(h.detach(), h0) and torch.equal(recon.detach(), r0)
    # side effects of the reference hooks
    assert torch.equal(m.decoder.input_activations, h.detach())
    assert torch.equal(m.decoder.output_grad, g)
    ref = _reference(m, x.detach(), h, g, g_h, mask)
    got = {"grad_we": m.encoder[0].weight.grad, "grad_be": m.encoder[0].bias.grad, "grad_wd": m.decoder.weight.grad,
           "grad_x": x.grad}
    tol = TOL_EXACT if exact else TOL_FAST
    for k, (r, S) in ref.items():
        frac = _frac(got[k], r, S)
        print(f"{name} exact={exact} g_h={with_gh} {k}: max err / S = {frac:.3e} (bound {tol:.1e})")
        assert frac <= tol, k
    # the closed-form oracle (numpy float64 from the inputs alone) where its ReLU pattern is the GPU's: in exact mode h
    # is fp32-accurate, so the oracle's gradients meet the same bound
    if exact and cfg["B"] * cfg["H"] <= 1 << 20:
        o = tsae_oracle.tsae_training_grads(x.detach().cpu().numpy(), m.encoder[0].weight.detach().cpu().numpy(),
                                   m.encoder[0].bias.detach().cpu().numpy(), m.decoder.weight.detach().cpu().numpy(),
                                   mask.cpu().numpy(), g.cpu().numpy(), None if g_h is None else g_h.cpu().numpy())
        if np.array_equal(o["h"] > 0, h.detach().cpu().numpy() > 0):
            # the oracle's h is float64, the GPU's fp32-accurate: g^T h also carries h's own error, which is bounded
            # by the forward's S_h = |x| |We|^T + |be|, not by |h|
            xd, We = x.detach().double(), m.encoder[0].weight.detach().double()
            S_h = xd.abs() @ We.abs().T + m.encoder[0].bias.detach().double().abs()
            extra = {"grad_wd": mask.double() * (g.double().abs().T @ S_h)}
            for k, (r, S) in ref.items():
                S = S + extra.get(k, 0.0)
                assert _frac(got[k], torch.from_numpy(o[k]).to(cuda_device), S) <= tol, ("oracle", k)


def test_tsae_backward_recon_only_and_h_only(cuda_device):
    """Either upstream gradient may be absent: a loss on h alone leaves decoder.weight.grad = 0 and output_grad unset."""
    m, x = _model(cases.TSAE_CASES["tsae_d64_h2048"], cuda_device, True)
    h, recon = m(x)
    (h.abs().mean()).backward()
    assert m.decoder.output_grad is None
    assert float(m.decoder.weight.grad.abs().max()) == 0.0
    g_h = torch.sign(h.detach()) / h.numel()
    ref = _reference(m, x, h, torch.zeros_like(recon), g_h, m.decoder.mask)
    assert _frac(m.encoder[0].weight.grad, *ref["grad_we"]) <= TOL_EXACT


# ---------------------------------------------------------------------------------------------------------------
# the reference trainer's t_sae loop
# ---------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("exact", [True, False])
def test_tsae_trainer_sequence(cuda_device, exact):
    cfg = dict(D=64, H=2048, B=256, bf16=False, seed=91)
    m, x = _model(cfg, cuda_device, exact)
    m.decoder.mask = torch.ones_like(m.decoder.mask)
    m.decoder.init_mask(0.7)                                      # RigL start (sae/ternary.py:27-39)
    mask0 = m.decoder.mask.clone()
    assert 0.25 < float(mask0.mean()) < 0.35
    opt = torch.optim.SGD(m.parameters(), lr=0.5)
    losses = []
    tol = TOL_EXACT if exact else TOL_FAST
    for step in range(4):
        opt.zero_grad(set_to_none=True)
        loss, h, recon, g, g_h = _step(m, x, 1e-3)
        losses.append(float(loss))
        mask = m.decoder.mask.clone()
        ref = _reference(m, x, h, g, g_h, mask)
        m.decoder.mask_grad()                                     # (:89-90)
        for k, p in (("grad_we", m.encoder[0].weight), ("grad_be", m.encoder[0].bias), ("grad_wd", m.decoder.weight)):
            assert _frac(p.grad, *ref[k]) <= tol, (step, k)
        w_before = m.decoder.weight.detach().clone()
        opt.step()
        torch.testing.assert_close(m.decoder.weight.detach(), w_before - 0.5 * m.decoder.weight.grad, rtol=0, atol=0)
        # update_mask from the hooks' buffers (:54-87), against the oracle on the same GPU state
        w_np = m.decoder.weight.detach().cpu().numpy()
        m_np = m.decoder.mask.cpu().numpy()
        a_np = m.decoder.input_activations.cpu().numpy()
        d_np = m.decoder.output_grad.cpu().numpy()
        m.decoder.update_mask(0.3)
        om, ow = TO.rigl_update_mask(w_np, m_np, a_np, d_np, 0.3, 0.7)
        got_m = m.decoder.mask.cpu().numpy()
        # the batch means are column sums with atomics: only scores equal up to the last bits may swap at the cut
        assert got_m.sum() == om.sum()
        assert (got_m != om).mean() < 1e-3
        np.testing.assert_array_equal(m.decoder.weight.detach().cpu().numpy(), (w_np * got_m).astype(np.float32))
    print(f"t_sae trainer loop exact={exact}: losses {losses}")
    assert losses[-1] < losses[0]


# ---------------------------------------------------------------------------------------------------------------
# BASELINE config 3 shape: B = 4096, 512 -> 32768
# ---------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("exact", [True, False])
def test_tsae_backward_full_size(cuda_device, exact):
    B, D, H = 4096, 512, 32768
    cfg = dict(D=D, H=H, B=B, bf16=True, seed=33)
    m, x = _model(cfg, cuda_device, exact)
    # autograd = False and no_grad: the plain forward, the same launches and bits as a direct library call
    m.autograd = False
    h_plain, r_plain = m(x)
    h_lib, r_lib = L.tsae_forward(x, m._enc_parts(), m.encoder[0].bias.detach(), m.decoder._ternary()[0], exact)
    assert torch.equal(h_plain, h_lib) and torch.equal(r_plain, r_lib)
    m.autograd = True
    with torch.no_grad():
        h_ng, r_ng = m(x)
    assert h_ng.grad_fn is None and torch.equal(h_ng, h_plain) and torch.equal(r_ng, r_plain)
    loss, h, recon, g, g_h = _step(m, x, 1e-3)
    assert torch.equal(h.detach(), h_plain) and torch.equal(recon.detach(), r_plain)
    # sampled rows / columns against float64 products on the GPU
    gen = torch.Generator(device=cuda_device).manual_seed(5)
    rows = torch.randperm(H, device=cuda_device, generator=gen)[:512]
    Wd = m.decoder.weight.detach().double()
    T = torch.sign(Wd) * (Wd.abs() >= 0.5)
    hd = h.detach().double()
    gd = g.double()
    Ts = T[:, rows]
    gz = torch.where(hd[:, rows] > 0, gd @ Ts + g_h[:, rows].double(), torch.zeros((), dtype=torch.float64, device=x.device))
    agz = torch.where(hd[:, rows] > 0, gd.abs() @ Ts.abs() + g_h[:, rows].double().abs(),
                      torch.zeros((), dtype=torch.float64, device=x.device))
    xd = x.double()
    tol = TOL_EXACT if exact else TOL_FAST
    checks = {
        "grad_we": (m.encoder[0].weight.grad[rows], gz.T @ xd, agz.T @ xd.abs()),
        "grad_be": (m.encoder[0].bias.grad[rows], gz.sum(0), agz.sum(0)),
        "grad_wd": (m.decoder.weight.grad[:, rows], m.decoder.mask[:, rows].double() * (gd.T @ hd[:, rows]),
                    m.decoder.mask[:, rows].double() * (gd.abs().T @ hd[:, rows].abs())),
    }
    for k, (got, r, S) in checks.items():
        frac = _frac(got, r, S)
        print(f"B=4096 512->32768 exact={exact} {k}: max err / S = {frac:.3e} (bound {tol:.1e})")
        assert frac <= tol, k


def test_tsae_step_in_cuda_graph(cuda_device):
    """A whole forward + backward captured in a CUDA graph replays to the eager gradients (the bias gradient up to
    the atomics' summation order)."""
    cfg = dict(D=512, H=4096, B=512, bf16=True, seed=95)
    m, x = _model(cfg, cuda_device, True)
    params = list(m.parameters())
    for p in params:
        p.grad = None
    _step(m, x, 1e-3)
    eager = [p.grad.clone() for p in params]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            for p in params:
                p.grad = None
            hh, rr = m(x)
            (0.5 * F.mse_loss(rr, x) + 1e-3 * hh.abs().mean()).backward()
    torch.cuda.current_stream().wait_stream(s)
    for p in params:
        p.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        hh, rr = m(x)
        (0.5 * F.mse_loss(rr, x) + 1e-3 * hh.abs().mean()).backward()
    for p in params:
        p.grad.zero_()
    graph.replay()
    torch.cuda.synchronize()
    for p, e in zip(params, eager):
        if p is m.encoder[0].bias:
            torch.testing.assert_close(p.grad, e, rtol=1e-5, atol=1e-9)
        else:
            assert torch.equal(p.grad, e)


# ---------------------------------------------------------------------------------------------------------------
# argument validation
# ---------------------------------------------------------------------------------------------------------------

def test_new_entries_validate_arguments(cuda_device):
    import ctypes as C

    lib = L.load()
    a = torch.zeros((64, 64), dtype=torch.bfloat16, device=cuda_device)
    c = torch.zeros((64, 64), dtype=torch.float32, device=cuda_device)
    ptrs = (C.c_void_p * 3)(a.data_ptr(), a.data_ptr(), a.data_ptr())
    s = L._stream()
    assert lib.qsae_wgrad(ptrs, ptrs, 2, 64, 64, 64, 0, c.data_ptr(), s) == -1          # 1 or 3 parts
    assert lib.qsae_wgrad(ptrs, ptrs, 1, 60, 64, 64, 0, c.data_ptr(), s) == -1          # MN-major A: M % 8
    assert lib.qsae_wgrad(ptrs, ptrs, 1, 64, 60, 64, 0, c.data_ptr(), s) == -1          # N % 8
    assert lib.qsae_wgrad(ptrs, ptrs, 1, 64, 64, 60, 1, c.data_ptr(), s) == -1          # K-major A: K % 8
    assert lib.qsae_wgrad(ptrs, ptrs, 1, 64, 64, 0, 0, c.data_ptr(), s) == -1           # empty contraction
    assert lib.qsae_wgrad(ptrs, ptrs, 1, 64, 64, 64, 0, None, s) == -1
    assert lib.qsae_wgrad(ptrs, ptrs, 1, 64, 64, 64, 0, c.data_ptr() + 4, s) == -1      # alignment
    assert b"16-byte" in lib.qsae_last_error()
    n = C.c_size_t(0)
    assert lib.qsae_tsae_backward_workspace_bytes(16, 2048, 520, 1, C.byref(n)) == -1   # D > 512
    assert lib.qsae_tsae_backward_workspace_bytes(16, 2044, 64, 1, C.byref(n)) == -1    # H % 8
    assert lib.qsae_tsae_backward_workspace_bytes(16, 2048, 64, 1, C.byref(n)) == 0 and n.value > 0
    f = torch.zeros(1 << 20, dtype=torch.float32, device=cuda_device)
    p = f.data_ptr()
    assert lib.qsae_tsae_backward(p, p, p, None, p, None, None, None, None, 16, 2048, 64, 1, p, p, p, None, p, 1024, s) == -2
    assert lib.qsae_tsae_backward(p, p, None, None, p, None, None, None, None, 16, 2048, 64, 1, p, p, p, None, p, n.value,
                                  s) == -1
    # grad_x needs the encoder weight's parts
    assert lib.qsae_tsae_backward(p, p, p, None, p, None, p, None, None, 16, 2048, 64, 1, p, p, p, p, p, n.value, s) == -1
    with pytest.raises(ValueError):
        L.wgrad((a, a), (a, a))
    with pytest.raises(ValueError):
        L.wgrad((a,), (torch.zeros((32, 64), dtype=torch.bfloat16, device=cuda_device),))
    with pytest.raises(L.QsaeError):
        L.wgrad((torch.zeros((64, 60), dtype=torch.bfloat16, device=cuda_device),), (a,))
