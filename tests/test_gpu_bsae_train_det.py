"""b_sae training step with model.deterministic = True on the GPU: the autograd node behind BinarySAE.forward with
autograd = True calls qsae_bsae_backward (the latent-major kernels of csrc/train.cu with the logit chain rule fused
into the reduction) instead of the atomic scatters.

Precision contract. Every gradient is checked against float64 on the GPU's own forward selections (v, idx), its own
soft dictionary rows R = dequant_soft(logits) and the upstream gradients autograd hands to the node (g = d loss /
d recon and gp = d loss / d polarize_loss, captured by hooks). q is the quantization step, n_h the number of rows that
selected latent h, u = 2^-24, and S the same sum over absolute values:
  gv = q <g, R[h]>: an fp32 dot of D terms, then the product with q: |err| <= (D + 1) u S_gv;
  G[h] = q sum v g: n_h fma terms (in chunks, then chunk partials: fewer roundings than a serial sum) and the product
  with q: (n_h + 1) u S_G;
  grad W_enc[h] = sum gv x, grad b_enc[h] = sum gv: the error of each gv plus n_h additions: (D + n_h + 2) u S;
  grad b_dec = sum_b g: (B + 1) u S;   grad x = sum_j gv W_enc[idx]: the gv error plus k terms: (D + k + 2) u S.
Logit gradients: out = ((G c_i + T) s) with s = p (1 - p), T = gp 2^i (1 - 2p) / N and p the fast logistic, which
both kernels evaluate identically. The float64 G rounded to fp32, Gr, goes through the existing bsae_logit_grad. Its
input differs from the new kernel's G by at most bound_G + u |G|, which moves the output by |c_i| s times that; each
of the two evaluations adds at most two roundings (the sum and the product) of a value at most |G c_i| + |T| in
magnitude, 4 u s (|G c_i| + |T|) in all. Rows nobody selected have G = 0 exactly and must equal bsae_logit_grad with
G = NULL bit for bit.
Each case prints its largest error / bound ratio (<= 1 passes)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import quantizedsae_b200 as Q
from oracle import qsae_oracle as O
from oracle import train_oracle as TO
from quantizedsae_b200 import _lib as L
from tests.golden import cases

pytestmark = pytest.mark.gpu

U = 2.0 ** -24


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def close(got, want, rtol=2e-4, atol_frac=2e-6):
    """test_gpu_train.py's tolerance for the b_sae gradients."""
    want = np.asarray(want, dtype=np.float64)
    got = got.detach().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    atol = atol_frac * max(1e-30, float(np.abs(want).max()))
    np.testing.assert_allclose(got.astype(np.float64), want, rtol=rtol, atol=atol)


def _model(dev, D, H, n_bits, k, B, seed, gamma=4.0, skew=False):
    torch.manual_seed(seed)
    m = Q.BinarySAE(D, H, gamma, n_bits)
    m.k = (k + 0.5) / H                                   # int(H * m.k) == k
    m.to(dev)
    m.autograd, m.deterministic, m.return_dense = True, True, False
    if skew:
        with torch.no_grad():
            m.encoder[0].bias.zero_()
            m.encoder[0].bias[0] = 100.0                  # wins every row: 4096 entries -> the chunk path
            m.encoder[0].bias[1:33] = 0.45
    x = torch.randn((B, D), device=dev)
    return m, x


def _step(m, x, lam):
    """0.5 * mse + lam * polarize -> backward, with g and gp captured."""
    seen = {}
    lat, recon, pol = m(x)
    recon.register_hook(lambda g: seen.__setitem__("g", g.detach().clone()))
    pol.register_hook(lambda g: seen.__setitem__("gp", g.detach().clone()))
    (0.5 * F.mse_loss(recon, x.detach()) + lam * pol).backward()
    return lat, seen["g"], seen["gp"]


def _reference(x, vals, idx, g, R, We, q, chunk=4096):
    """float64 gv-derived gradients, G and their bounds from the GPU's (vals, idx), soft rows and g."""
    B, D = x.shape
    H = R.shape[0]
    dev = x.device
    Rd, Wed = R.double(), We.double()
    out = {n: torch.zeros(s, dtype=torch.float64, device=dev) for n, s in
           (("grad_we", (H, D)), ("grad_be", (H,)), ("G", (H, D)), ("grad_x", (B, D)))}
    S = {n: torch.zeros_like(t) for n, t in out.items()}
    for r0 in range(0, B, chunk):
        r = slice(r0, min(B, r0 + chunk))
        il = idx[r].long()
        xd, gd, vd = x[r].double(), g[r].double(), vals[r].double()
        rows = Rd[il]                                                  # [b, k, D]
        gv = q * torch.einsum("bd,bjd->bj", gd, rows)
        sgv = abs(q) * torch.einsum("bd,bjd->bj", gd.abs(), rows.abs())
        flat = il.reshape(-1)
        out["grad_we"].index_add_(0, flat, (gv[:, :, None] * xd[:, None, :]).reshape(-1, D))
        S["grad_we"].index_add_(0, flat, (sgv[:, :, None] * xd.abs()[:, None, :]).reshape(-1, D))
        out["G"].index_add_(0, flat, (q * vd[:, :, None] * gd[:, None, :]).reshape(-1, D))
        S["G"].index_add_(0, flat, (abs(q) * vd.abs()[:, :, None] * gd.abs()[:, None, :]).reshape(-1, D))
        out["grad_be"].index_add_(0, flat, gv.reshape(-1))
        S["grad_be"].index_add_(0, flat, sgv.reshape(-1))
        out["grad_x"][r] = torch.einsum("bj,bjd->bd", gv, Wed[il])
        S["grad_x"][r] = torch.einsum("bj,bjd->bd", sgv, Wed[il].abs())
        del rows
    out["grad_bd"], S["grad_bd"] = g.double().sum(0), g.double().abs().sum(0)
    n_h = torch.bincount(idx.reshape(-1).long(), minlength=H).double()
    k = idx.shape[1]
    factor = {"grad_we": (D + n_h + 2)[:, None], "grad_be": D + n_h + 2, "G": (n_h + 1)[:, None],
              "grad_bd": float(B + 1), "grad_x": float(D + k + 2)}
    return {n: (out[n], U * factor[n] * S[n]) for n in out}, n_h


def _ratio(got, ref, bound):
    """max |got - ref| / bound (an entry with bound 0 must be exact)."""
    err = (got.double() - ref).abs()
    if bool(((bound == 0) & (err > 0)).any()):
        return float("inf")
    return float((err / bound.clamp_min(1e-300)).max()) if err.numel() else 0.0


def _logit_check(m, G, G_bound, n_h, gp):
    """The fused logit gradients against bsae_logit_grad on the float64 G rounded to fp32 (bound in the header), and
    the unselected rows bit for bit against bsae_logit_grad with G = NULL."""
    dec = m.decoder
    H, D, nb = dec.in_features, dec.out_features, dec.n_bits
    logits = dec.weight.detach()
    got = dec.weight.grad
    ref = torch.empty_like(logits)
    L.bsae_logit_grad(logits, G.float().contiguous(), D, nb, gp, ref, accumulate=False)
    pol_only = torch.empty_like(logits)
    L.bsae_logit_grad(logits, None, D, nb, gp, pol_only, accumulate=False)
    un = n_h == 0
    if bool(un.any()):
        assert torch.equal(got[un], pol_only[un]), "unselected rows differ from bsae_logit_grad with G = 0"
    p = torch.sigmoid(logits.double()).reshape(H, D, nb)
    s = p * (1 - p)
    c = torch.from_numpy(O.bit_coefficients(nb).astype(np.float64)).to(G.device)
    pw = 2.0 ** torch.arange(nb, device=G.device, dtype=torch.float64)
    Tm = float(gp) * pw * (1 - 2 * p) / (H * D * nb)
    Gc = G[:, :, None].abs() * c.abs()
    bound = c.abs() * s * (G_bound + U * G.abs())[:, :, None] + 4 * U * s * (Gc + Tm.abs())
    return _ratio(got.reshape(H, D, nb), ref.double().reshape(H, D, nb), bound)


def _check(name, m, x, lat, g, gp, x_grad=None):
    dec, lin = m.decoder, m.encoder[0]
    ref, n_h = _reference(x, lat.values.detach(), lat.indices, g, dec._soft_rows(), lin.weight.detach(),
                          float(dec.quantization_step))
    got = {"grad_we": lin.weight.grad, "grad_be": lin.bias.grad, "grad_bd": dec.bias.grad, "grad_x": x_grad}
    worst = 0.0
    for key, (r, bound) in ref.items():
        if key == "G" or got[key] is None:
            continue
        q = _ratio(got[key], r, bound)
        worst = max(worst, q)
        assert q <= 1.0, (name, key, q)
    G, G_bound = ref["G"]
    q = _logit_check(m, G, G_bound, n_h, gp)
    assert q <= 1.0, (name, "grad_logits", q)
    worst = max(worst, q)
    un = n_h == 0
    assert bool((lin.weight.grad[un] == 0).all()) and bool((lin.bias.grad[un] == 0).all())
    print(f"{name}: max error / bound = {worst:.3e} (logits {q:.3e}); {int((n_h > 256).sum())} latents on the chunk path")
    return worst


# ------------------------------------------------------------------------------------------
# the reference's fixtures through the deterministic path
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(cases.TRAIN_BSAE))
def test_fixtures_through_deterministic_path(cuda_device, golden_dir, name):
    cfg = cases.BSAE_CASES[name]
    inp = cases.bsae_inputs(cfg)
    g = np.load(golden_dir / f"train_{name}.npz")
    assert str(g["input_sha"]) == cases.checksum(inp)
    lam = float(g["polarize_lambda"])
    m = Q.BinarySAE(cfg["D"], cfg["H"], cfg["gamma"], cfg["n_bits"]).to(cuda_device)
    m.load_state_dict({"encoder.0.weight": T(inp["We"], cuda_device), "encoder.0.bias": T(inp["be"], cuda_device),
                       "decoder.weight": T(inp["logits"], cuda_device), "decoder.bias": T(inp["bd"], cuda_device)})
    m.autograd, m.deterministic = True, True
    x = T(inp["x"], cuda_device)
    latent, recon, pol = m(x)
    recon_loss = 0.5 * F.mse_loss(recon, x)
    (recon_loss + lam * pol).backward()
    assert float(recon_loss.detach()) == pytest.approx(float(g["recon_loss"]), rel=1e-5)
    rows = g["rows"]
    close(m.decoder.weight.grad[rows], g["grad_logits_rows"])
    close(m.encoder[0].weight.grad[rows], g["grad_We_rows"])
    close(m.encoder[0].bias.grad, g["grad_be"])
    close(m.decoder.bias.grad, g["grad_bd"])
    assert float(m.decoder.weight.grad.double().abs().sum()) == pytest.approx(float(g["grad_logits_abs_sum"]), rel=1e-5)
    assert float(m.encoder[0].weight.grad.double().abs().sum()) == pytest.approx(float(g["grad_We_abs_sum"]), rel=1e-5)
    want = TO.bsae_training_grads(inp["x"], inp["We"], inp["be"], inp["logits"], inp["bd"], n_bits=cfg["n_bits"],
                                  gamma=cfg["gamma"], k=O.bsae_k(cfg["H"]), polarize_lambda=lam)
    for key, p in (("decoder.weight", m.decoder.weight), ("encoder.0.weight", m.encoder[0].weight),
                   ("encoder.0.bias", m.encoder[0].bias), ("decoder.bias", m.decoder.bias)):
        close(p.grad, want[key])
    # a second backward accumulates like autograd does
    _, recon, pol = m(x)
    (0.5 * F.mse_loss(recon, x) + lam * pol).backward()
    close(m.decoder.bias.grad, 2 * want["decoder.bias"])
    close(m.decoder.weight.grad, 2 * want["decoder.weight"])


# ------------------------------------------------------------------------------------------
# float64 bounds on the GPU's own selections
# ------------------------------------------------------------------------------------------
BOUND_CASES = {   # name: (D, H, n_bits, k, B, gamma, skew)
    "d8_h1000_1b_k1": (8, 1000, 1, 1, 37, 4.0, False),
    "d64_h2048_2b_k32": (64, 2048, 2, 32, 300, 4.0, False),
    "d256_h4096_4b_k65": (256, 4096, 4, 65, 512, 1.5, False),
    "d512_h4096_8b_k2097": (512, 4096, 8, 2097, 96, 4.0, False),
    "d512_h32768_4b_k32": (512, 32768, 4, 32, 4096, 4.0, False),
    "d512_h32768_4b_skew": (512, 32768, 4, 32, 4096, 4.0, True),
    "d64_h1m_4b_k16": (64, 1 << 20, 4, 16, 1024, 4.0, False),          # keys over [0, 2^20]: three radix passes
}


@pytest.mark.parametrize("x_grad", [False, True])
@pytest.mark.parametrize("name", list(BOUND_CASES))
def test_gradients_within_float64_bounds(cuda_device, name, x_grad):
    D, H, nb, k, B, gamma, skew = BOUND_CASES[name]
    m, x0 = _model(cuda_device, D, H, nb, k, B, seed=100 + list(BOUND_CASES).index(name), gamma=gamma, skew=skew)
    x = x0.clone().requires_grad_(x_grad)
    lat, g, gp = _step(m, x, 0.37)
    assert lat.indices.shape[1] == k
    _check(f"{name} x_grad={x_grad}", m, x0, lat, g, gp, x.grad if x_grad else None)
    assert (x.grad is not None) == x_grad


def test_gp_from_host_value_and_batch_zero(cuda_device):
    m, x = _model(cuda_device, 64, 2048, 4, 16, 64, seed=3)
    with torch.no_grad():
        sl = m.encode_topk(x)
    dec, W = m.decoder, m.encoder[0].weight.detach()
    g = torch.randn_like(x)
    args = (x, sl.values, sl.indices, g, dec._soft_rows(), dec.weight.detach(), dec.quantization_step)
    a = L.bsae_backward(*args, 0.5, W, 4, True)
    b = L.bsae_backward(*args, torch.tensor(0.5, device=cuda_device), W, 4, True)
    for p, q in zip(a, b):
        assert torch.equal(p, q)
    z = L.bsae_backward(x[:0], sl.values[:0], sl.indices[:0], g[:0], dec._soft_rows(), dec.weight.detach(),
                        dec.quantization_step, 0.5, W, 4, False)
    pol_only = torch.empty_like(dec.weight)
    L.bsae_logit_grad(dec.weight.detach(), None, 64, 4, 0.5, pol_only, accumulate=False)
    assert float(z[0].abs().max()) == 0 and float(z[1].abs().max()) == 0 and float(z[3].abs().max()) == 0
    assert torch.equal(z[2], pol_only)


# ------------------------------------------------------------------------------------------
# bit-determinism
# ------------------------------------------------------------------------------------------
def _raw(m, x, sl, g, gp=0.25):
    dec = m.decoder
    return L.bsae_backward(x, sl.values, sl.indices, g, dec._soft_rows(), dec.weight.detach(), dec.quantization_step, gp,
                           m.encoder[0].weight.detach(), dec.n_bits, True)


@pytest.mark.parametrize("B,skew", [(4096, False), (65536, False), (4096, True)])
def test_bit_deterministic(cuda_device, B, skew):
    m, x = _model(cuda_device, 512, 32768, 4, 32, B, seed=41, skew=skew)
    with torch.no_grad():
        sl = m.encode_topk(x)
    if skew:
        assert int((sl.indices == 0).sum()) == B        # one latent with B entries: the chunk path
    g = torch.randn_like(x) / (B * 512)
    a = _raw(m, x, sl, g)
    b = _raw(m, x, sl, g)
    for p, q in zip(a, b):
        assert torch.equal(p, q)


def test_cuda_graph_replay(cuda_device):
    m, x = _model(cuda_device, 512, 4096, 4, 32, 512, seed=42)
    with torch.no_grad():
        sl = m.encode_topk(x)
    dec = m.decoder
    sx, sv, si, sg = x.clone(), sl.values.clone(), sl.indices.clone(), torch.randn_like(x)
    gp = torch.tensor(0.3, device=cuda_device)
    rows, logits, W = dec._soft_rows(), dec.weight.detach(), m.encoder[0].weight.detach()
    call = lambda: L.bsae_backward(sx, sv, si, sg, rows, logits, dec.quantization_step, gp, W, 4, True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            call()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = call()
    x2 = torch.randn_like(x)
    with torch.no_grad():
        sl2 = m.encode_topk(x2)
    g2 = torch.randn_like(x)
    sx.copy_(x2); sv.copy_(sl2.values); si.copy_(sl2.indices); sg.copy_(g2); gp.fill_(0.7)
    graph.replay()
    torch.cuda.synchronize()
    direct = L.bsae_backward(x2, sl2.values, sl2.indices, g2, rows, logits, dec.quantization_step, 0.7, W, 4, True)
    for p, q in zip(outs, direct):
        assert torch.equal(p, q)


# ------------------------------------------------------------------------------------------
# against the atomic path, the trainer loop, and the default path
# ------------------------------------------------------------------------------------------
def _grads(m):
    return [p.grad.clone() for p in (m.encoder[0].weight, m.encoder[0].bias, m.decoder.weight, m.decoder.bias)]


def test_agrees_with_atomic_path_at_baseline_shape(cuda_device):
    m, x = _model(cuda_device, 512, 32768, 4, 65, 4096, seed=43)
    x = x.requires_grad_(True)
    out = {}
    for det in (False, True):
        m.zero_grad(set_to_none=True)
        x.grad = None
        m.deterministic = det
        _, recon, pol = m(x)
        (0.5 * F.mse_loss(recon, x) + 0.25 * pol).backward()
        out[det] = _grads(m) + [x.grad.clone()]
    for p, q in zip(out[True], out[False]):
        close(p, q.double().cpu().numpy())


def test_trainer_loop_state_dict_is_reproducible(cuda_device):
    def run():
        m, x = _model(cuda_device, 512, 32768, 4, 65, 4096, seed=44)
        opt = torch.optim.Adam(m.parameters(), lr=1e-3)
        losses = []
        for _ in range(5):
            opt.zero_grad(set_to_none=True)
            _, recon, pol = m(x)
            loss = 0.5 * F.mse_loss(recon, x) + 0.1 * pol
            loss.backward()
            opt.step()
            losses.append(float(loss))
        return m.state_dict(), losses

    a, la = run()
    b, lb = run()
    assert la == lb
    for key in a:
        assert torch.equal(a[key], b[key]), key
    print(f"b_sae deterministic trainer loop: losses {la}")
    assert la[-1] < la[0]


def test_default_path_and_forward_unchanged(cuda_device):
    m, x = _model(cuda_device, 512, 4096, 4, 32, 1024, seed=45)
    m.deterministic = False
    x = x.requires_grad_(True)
    # forward: the same launches and bits with the switch on and off
    _, r0, _ = m(x)
    n0 = L.launch_count()
    lat0, r0, p0 = m(x)
    fwd_off = L.launch_count() - n0
    m.deterministic = True
    n0 = L.launch_count()
    lat1, r1, p1 = m(x)
    fwd_on = L.launch_count() - n0
    assert fwd_on == fwd_off
    assert torch.equal(lat0.values, lat1.values) and torch.equal(lat0.indices, lat1.indices) and torch.equal(r0, r1)
    # backward with the switch off: exactly the atomic kernels' launches
    m.deterministic = False
    _, recon, pol = m(x)
    loss = 0.5 * F.mse_loss(recon, x) + 0.25 * pol
    n0 = L.launch_count()
    loss.backward()
    bwd_off = L.launch_count() - n0
    dec, W = m.decoder, m.encoder[0].weight.detach()
    H, D = 4096, 512
    g = torch.randn_like(x)
    n0 = L.launch_count()
    G = torch.zeros((H, D), device=cuda_device)
    L.rows_scatter_add(lat0.values.detach(), lat0.indices, g, G, scale=dec.quantization_step)
    gl = torch.empty_like(dec.weight)
    L.bsae_logit_grad(dec.weight.detach(), G, D, 4, 0.25, gl, accumulate=False)
    L.column_sum(g)
    gv = L.rows_gather_dot(g, dec._soft_rows(), lat0.indices, scale=dec.quantization_step)
    gwe, gbe = torch.zeros((H, D), device=cuda_device), torch.zeros((H,), device=cuda_device)
    L.rows_scatter_add(gv, lat0.indices, x.detach(), gwe, scale=1.0, dst_col=gbe)
    L.decode_rows_f32(gv, lat0.indices, W, H, D, 1.0, None)
    atomic = L.launch_count() - n0
    assert bwd_off == atomic, (bwd_off, atomic)
    # and the deterministic backward launches its own kernels
    m.deterministic = True
    m.zero_grad(set_to_none=True)
    _, recon, pol = m(x)
    loss = 0.5 * F.mse_loss(recon, x) + 0.25 * pol
    n0 = L.launch_count()
    loss.backward()
    print(f"b_sae backward launches: atomic {bwd_off}, deterministic {L.launch_count() - n0}; forward {fwd_off}")
