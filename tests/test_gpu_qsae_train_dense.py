"""q_sae decoder training at any activity: the STE backward from the dense activity mask of forward_dense_active
(qsae_matryoshka_backward_dense: a tensor-core product mask^T g per level with the STE factor in its epilogue).

Checked against
  * the fixtures produced by torch autograd on the UNMODIFIED reference (tests/golden/train_qsae_*.npz), with the
    tolerances of the sparse route's test (test_gpu_train.py);
  * train_oracle.qsae_decoder_backward in float64, fed the GPU's own mask. With S[h, d] = alpha[h] sum_b a[b, h]
    |g_l(h)[b, d]|: exact mode (three bf16 parts of g, the mask exact in bf16, fp32 accumulation) within 2e-5 S, fast
    mode (one bf16 part, relative rounding 2^-9 per term) within 2^-8 S;
  * the sparse route on models where both exist.
"""
import ctypes as C

import numpy as np
import pytest
import torch
from scipy.stats import norm

import quantizedsae_b200 as Q
from oracle import train_oracle as TO
from quantizedsae_b200 import _lib as L
from quantizedsae_b200 import training
from tests.golden import cases
from tests.test_gpu_matryoshka_levels import activity_band

pytestmark = pytest.mark.gpu


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def close(got, want, rtol=2e-4, atol_frac=2e-6):
    """the sparse route's tolerance (test_gpu_train.py)"""
    want = np.asarray(want, dtype=np.float64)
    got = got.detach().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    atol = atol_frac * max(1e-30, float(np.abs(want).max()))
    np.testing.assert_allclose(got.astype(np.float64), want, rtol=rtol, atol=atol)


def load_model(inp, cfg, dev):
    m = Q.QuantizedMatryoshkaSAE(cfg["D"], cfg["H"], 32, cfg["abs_range"], cfg["n_bits"], cfg["allow_bias"])
    m.load_state_dict({"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
                       "decoder.weight": torch.from_numpy(inp["W"]), "decoder.weight_mirror": torch.from_numpy(inp["Wm"]),
                       "decoder.bias": torch.from_numpy(inp["bd"])}, strict=True)
    return m.to(dev)


def level_grads(levels, x):
    B, D = x.shape
    return [(r - x) / float(B * D) for r in levels]


def within_s(got, want, S, tol, what):
    err = np.abs(got.astype(np.float64) - want)
    bad = err > tol * S + 1e-30
    assert not bad.any(), f"{what}: {int(bad.sum())} elements beyond {tol:g} S, worst err/S " \
                          f"{float((err / np.maximum(S, 1e-300)).max()):.3g}"


def s_bound(mask64, grads, alpha, starts):
    """S[h, d] = alpha[h] sum_b a[b, h] |g_l(h)[b, d]| (float64)"""
    H = mask64.shape[1]
    S = np.zeros((H, grads[0].shape[1]))
    for l in range(len(starts) - 1):
        s0, s1 = starts[l], starts[l + 1]
        S[s0:s1] = alpha[s0:s1, None] * (np.abs(mask64[:, s0:s1]).T @ np.abs(grads[l]))
    return S


# ------------------------------------------------------------------------------------------
# 1. the reference's fixtures, through the dense route (exact mode)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(cases.TRAIN_QSAE))
def test_dense_route_matches_reference_fixtures(cuda_device, golden_dir, name):
    cfg = cases.QSAE_CASES[name]
    inp = cases.qsae_inputs(cfg)
    g = np.load(golden_dir / f"train_{name}.npz")
    assert str(g["input_sha"]) == cases.checksum(inp)
    m = load_model(inp, cfg, cuda_device)
    x = T(inp["x"], cuda_device)
    out = m.forward_dense_active(x)
    mask = out["active_mask"]
    z2 = m.decoder.ste_backward(mask, level_grads(out["reconstruction_levels"], x))
    # the rule of test_gpu_matryoshka_levels.py: a decision within the fp32 band of THR may go either way; the
    # latents with such a decision are named and left out, every other one compared as is
    _, band = activity_band(inp["x"], inp["We"], inp["be"])
    loose = np.flatnonzero(band.any(0))
    if loose.size:
        print(f"{name}: activity decisions within the fp32 band at latents {loose.tolist()}")
    keep_cols = np.setdiff1d(np.arange(cfg["H"]), loose)
    assert np.array_equal(z2.cpu().numpy()[keep_cols], g["z2"].astype(np.int64)[keep_cols])
    rows = np.asarray(g["rows"])
    sel = np.isin(rows, loose, invert=True)
    close(m.decoder.weight.grad[rows[sel]], g["ste_W"][sel])
    close(m.decoder.weight_mirror.grad[rows[sel]], g["ste_Wm"][sel])
    if cfg["allow_bias"]:
        close(m.decoder.bias.grad, g["grad_bias"])
    else:
        assert m.decoder.bias.grad is None
    m.decoder.apply_secant_grad()
    close(m.decoder.weight.grad[rows[sel]], g["secant_W"][sel])
    close(m.decoder.weight_mirror.grad[rows[sel]], g["secant_Wm"][sel])
    if not loose.size:
        sums = [float(t.double().abs().sum()) for t in (m.decoder.weight.grad, m.decoder.weight_mirror.grad)]
        np.testing.assert_allclose(sums, g["abs_sums"][2:], rtol=1e-5)


# ------------------------------------------------------------------------------------------
# 2. float64 on the GPU's own mask: level boundaries on and off the 128-row tiles, batch tails, narrow / wide D
# ------------------------------------------------------------------------------------------
SHAPES = [  # (H, n_bits, B, D)
    (1000, 1, 1, 16), (1000, 8, 65, 48), (1000, 4, 4097, 512),
    (2056, 2, 63, 272), (2056, 8, 4097, 16), (2056, 1, 65, 512),
    (2504, 4, 65, 512), (2504, 8, 1, 48), (2504, 2, 4097, 272),
    (4104, 8, 4097, 48), (4104, 4, 63, 512), (4104, 2, 65, 272), (4104, 1, 1, 16),
    (32776, 4, 65, 512), (32776, 8, 63, 16), (32776, 1, 4097, 48), (32776, 2, 1, 272),
]


def dense_case(H, nb, B, D, seed, enc_bias=0.0):
    cfg = dict(D=D, H=H, n_bits=nb, abs_range=4.0, B=B, enc_bias=enc_bias, bf16=False, allow_bias=False, seed=seed)
    return cfg, cases.qsae_inputs(cfg)


@pytest.mark.parametrize("exact", [True, False], ids=["exact", "fast"])
@pytest.mark.parametrize("H,nb,B,D", SHAPES, ids=[f"h{H}-nb{nb}-b{B}-d{D}" for H, nb, B, D in SHAPES])
def test_dense_route_vs_float64(cuda_device, H, nb, B, D, exact):
    cfg, inp = dense_case(H, nb, B, D, seed=7000 + H + nb + B + D)
    m = load_model(inp, cfg, cuda_device)
    x = T(inp["x"], cuda_device)
    mask = m.forward_dense_active(x)["active_mask"]
    rng = np.random.default_rng(H + B)
    grads = [rng.standard_normal((B, D)).astype(np.float32) * np.float32(10.0 ** (-l)) for l in range(nb)]
    z2 = training.qsae_ste_backward(m.decoder, mask, [T(gr, cuda_device) for gr in grads], exact=exact)
    a = mask.float().cpu().numpy().astype(np.float64)
    assert set(np.unique(a).tolist()) <= {0.0, 1.0}
    assert np.array_equal(z2.cpu().numpy(), a.sum(0).astype(np.int64))
    gW, gWm, _, z2_64 = TO.qsae_decoder_backward(a, inp["W"], inp["Wm"], grads, n_bits=nb, abs_range=4.0, allow_bias=False)
    assert np.array_equal(z2.cpu().numpy(), z2_64.astype(np.int64))
    alpha = m.decoder._packed()[1].double().cpu().numpy()
    S = s_bound(a, grads, alpha, m.decoder._level_starts_host())
    tol = 2e-5 if exact else 2.0 ** -8
    within_s(m.decoder.weight.grad.cpu().numpy(), gW, S, tol, "grad weight")
    within_s(m.decoder.weight_mirror.grad.cpu().numpy(), gWm, S, tol, "grad weight_mirror")
    assert m.decoder.bias.grad is None


# ------------------------------------------------------------------------------------------
# 3. the two routes agree where both exist
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["qsae_d64_h2048", "qsae_d512_h4096"])
def test_sparse_and_dense_routes_agree(cuda_device, name):
    cfg = dict(cases.QSAE_CASES[name], B=256, seed=cases.QSAE_CASES[name]["seed"] + 100)
    inp = cases.qsae_inputs(cfg)
    m = load_model(inp, cfg, cuda_device)
    x = T(inp["x"], cuda_device)
    lists = m.forward_active(x, active_cap=256)
    dense = m.forward_dense_active(x)
    grads = level_grads(lists["reconstruction_levels"], x)
    z2_s = m.decoder.ste_backward(lists["active_idx"], grads)
    gw_s, gwm_s = m.decoder.weight.grad.clone(), m.decoder.weight_mirror.grad.clone()
    m.zero_grad(set_to_none=True)
    z2_d = m.decoder.ste_backward(dense["active_mask"], grads)
    assert torch.equal(z2_s, z2_d)
    a = dense["active_mask"].float().cpu().numpy().astype(np.float64)
    S = s_bound(a, [gr.double().cpu().numpy() for gr in grads], m.decoder._packed()[1].double().cpu().numpy(),
                m.decoder._level_starts_host())
    within_s(m.decoder.weight.grad.cpu().numpy(), gw_s.double().cpu().numpy(), S, 2e-5, "grad weight")
    within_s(m.decoder.weight_mirror.grad.cpu().numpy(), gwm_s.double().cpu().numpy(), S, 2e-5, "grad weight_mirror")


# ------------------------------------------------------------------------------------------
# 4. accumulation, determinism, CUDA graphs
# ------------------------------------------------------------------------------------------
def test_accumulates_is_deterministic_and_replays_in_a_graph(cuda_device):
    cfg, inp = dense_case(4104, 8, 1000, 272, seed=77)
    m = load_model(inp, cfg, cuda_device)
    x = T(inp["x"], cuda_device)
    mask = m.forward_dense_active(x)["active_mask"]
    g = torch.Generator(device=cuda_device).manual_seed(5)
    grads = [torch.randn((1000, 272), device=cuda_device, generator=g) for _ in range(8)]
    dec = m.decoder

    def run(n=1):
        dec.zero_grad(set_to_none=True)
        for _ in range(n):
            dec.ste_backward(mask, grads)
        return dec.weight.grad.clone(), dec.weight_mirror.grad.clone()

    w1, wm1 = run()
    w1b, wm1b = run()
    assert torch.equal(w1, w1b) and torch.equal(wm1, wm1b)
    w2, wm2 = run(2)
    torch.testing.assert_close(w2, 2 * w1, rtol=1e-6, atol=0)
    torch.testing.assert_close(wm2, 2 * wm1, rtol=1e-6, atol=0)
    # capture one dense ste_backward into zeroed .grad buffers and replay it
    dec.weight.grad.zero_()
    dec.weight_mirror.grad.zero_()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        dec.ste_backward(mask, grads)     # warm-up on the capture stream: workspace and tensor maps
    torch.cuda.current_stream().wait_stream(s)
    dec.weight.grad.zero_()
    dec.weight_mirror.grad.zero_()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        z2 = dec.ste_backward(mask, grads)
    dec.weight.grad.zero_()
    dec.weight_mirror.grad.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(dec.weight.grad, w1) and torch.equal(dec.weight_mirror.grad, wm1)
    assert torch.equal(z2, mask.float().sum(0).to(torch.int32))


def test_argument_checks_and_empty_batch(cuda_device):
    lib = L.load()
    dev = cuda_device
    H, D, B = 64, 32, 4
    w = torch.zeros((H, D), device=dev)
    gw = torch.ones((H, D), device=dev)
    alpha = torch.ones(H, device=dev)
    z2 = torch.full((H,), 7, dtype=torch.int32, device=dev)
    gl = torch.zeros((B, D), device=dev)
    mask = torch.zeros((B, H), dtype=torch.bfloat16, device=dev)
    ws = L._workspace(dev, 1 << 20)
    starts = (C.c_int * 3)(0, 32, H)
    ptrs = (C.c_void_p * 2)(gl.data_ptr(), gl.data_ptr())

    def call(mask_p, B_, H_, D_, n=2, g=ptrs, gw_p=gw.data_ptr()):
        return lib.qsae_matryoshka_backward_dense(mask_p, B_, H_, D_, g, starts, n, w.data_ptr(), w.data_ptr(), alpha.data_ptr(), 1,
                                                  gw_p, gw_p, z2.data_ptr(), ws.data_ptr(), ws.numel(), L._stream())

    assert call(mask.data_ptr(), B, 60, D) != 0                 # H % 8
    assert call(mask.data_ptr(), B, H, 40) != 0                 # D % 16
    assert call(mask.data_ptr(), B, H, 528) != 0                # D > 512
    assert call(mask.data_ptr(), B, H, D, n=9) != 0             # levels
    assert call(mask.data_ptr() + 2, B, H, D) != 0              # misaligned mask
    assert call(mask.data_ptr(), B, H, D, gw_p=gw.data_ptr() + 4) != 0
    assert call(mask.data_ptr(), 0, H, D) == 0                  # empty batch: z2 = 0, gradients untouched
    torch.cuda.synchronize()
    assert int(z2.abs().sum()) == 0 and bool((gw == 1).all())


# ------------------------------------------------------------------------------------------
# 5. the BASELINE shape at initialisation: 512 -> 32768, n_bits = 4, B = 4096, ~50 % active
# ------------------------------------------------------------------------------------------
def test_trainer_step_at_initialisation_baseline_shape(cuda_device):
    torch.manual_seed(0)
    D, H, nb, B = 512, 32768, 4, 4096
    m = Q.QuantizedMatryoshkaSAE(D, H, 32, 4.0, nb).to(cuda_device)
    x = torch.randn((B, D), device=cuda_device)
    training.qsae_trainer_decoder_grads(m, x)
    assert m.last_path == "dense"
    gw, gwm = m.decoder.weight.grad.clone(), m.decoder.weight_mirror.grad.clone()
    z2 = m.decoder._ctx["z2"]
    out = m.forward_dense_active(x)                                # the same forward: the same mask and levels
    mask = out["active_mask"]
    assert 0.3 < float(mask.float().mean()) < 0.7
    assert torch.equal(z2, mask.float().sum(0).to(torch.int32))
    # the secant part from the (separately tested) finish kernel
    dW, dWm = torch.zeros_like(gw), torch.zeros_like(gwm)
    _, alpha = m.decoder._packed()
    starts = m.decoder._level_starts_host()
    L.matryoshka_backward_finish(m.decoder.weight.detach(), m.decoder.weight_mirror.detach(), None, z2, alpha, starts,
                                 1.0 / B / D, 0, dW, dWm)
    grads = level_grads(out["reconstruction_levels"], x)
    rng = np.random.default_rng(3)
    for l in range(nb):
        rows = np.unique(rng.integers(starts[l], starts[l + 1], size=6))
        rows = np.union1d(rows, [starts[l], starts[l + 1] - 1])
        r = torch.from_numpy(rows).to(cuda_device)
        a = mask[:, r].double()
        gl = grads[l].double()
        M = a.T @ gl
        S = (alpha[r].double()[:, None] * (a.T @ gl.abs())).cpu().numpy()
        for w, got, d in ((m.decoder.weight, gw, dW), (m.decoder.weight_mirror, gwm, dWm)):
            s = torch.sigmoid(w.detach()[r].double())
            want = (alpha[r].double()[:, None] * M * s * (1 - s) + d[r].double()).cpu().numpy()
            within_s(got[r].cpu().numpy(), want, S + 0.01 * np.abs(d[r].double().cpu().numpy()), 2e-5, f"level {l}")


# ------------------------------------------------------------------------------------------
# 6. routing of qsae_trainer_decoder_grads
# ------------------------------------------------------------------------------------------
def test_trainer_routing(cuda_device):
    # BASELINE-like activity (L0 ~ 33 of 32768): the sparse route with the launches of the sparse step
    cfg = cases.QSAE_CASES["qsae_d512_h32768"]
    inp = cases.qsae_inputs(cfg)
    m = load_model(inp, cfg, cuda_device)
    x = T(inp["x"], cuda_device)
    m.forward_active(x, active_cap=256)                            # warm the prepared dictionary
    n0 = L.launch_count()
    m.forward_active(x, active_cap=256)
    n_fwd = L.launch_count() - n0
    n0 = L.launch_count()
    training.qsae_trainer_decoder_grads(m, x)
    # forward + scatter + STE finish + bias column sum + secant finish
    assert L.launch_count() - n0 == n_fwd + 4
    assert m.last_path == "sparse"
    training.qsae_trainer_decoder_grads(m, x)                     # L0 / H ~ 1e-3 stays below the crossover
    assert m.last_path == "sparse"
    # lists that fit but pass the crossover (L0 ~ 512 of 32768): this step on the lists, the next one dense
    sigma = (2.0 * 512 / (32768 + 512)) ** 0.5
    cfg1, inp1 = dense_case(32768, 4, 64, 512, seed=11, enc_bias=float(sigma * norm.ppf(1 / 64)))
    m1 = load_model(inp1, cfg1, cuda_device)
    x1 = T(inp1["x"], cuda_device)
    training.qsae_trainer_decoder_grads(m1, x1)
    assert m1.last_path == "sparse" and m1._train_l0_over_h > training._DENSE_TRAIN_L0_OVER_H
    training.qsae_trainer_decoder_grads(m1, x1)
    assert m1.last_path == "dense"
    # an untrained model (~50 % active) overflows the lists and goes dense
    cfg2, inp2 = dense_case(32768, 4, 8, 512, seed=9)
    m2 = load_model(inp2, cfg2, cuda_device)
    x2 = T(inp2["x"], cuda_device)
    training.qsae_trainer_decoder_grads(m2, x2)
    assert m2.last_path == "dense"
    m3 = load_model(inp2, cfg2, cuda_device)
    m3.dense_mode = "never"
    with pytest.raises(RuntimeError, match="dense_mode is 'never'"):
        training.qsae_trainer_decoder_grads(m3, x2)
