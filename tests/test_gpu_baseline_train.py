"""baseline_sae training step on the GPU: the autograd node behind BaselineSparseAutoencoder.forward with
autograd = True (qsae_baseline_backward, the deterministic latent-major kernels of csrc/train.cu) and the reference
trainer's baseline loop (training/trainer.py:168-173): forward, 0.5 * mse, backward, normalize_decoder_weights, Adam.

Precision contract. Every gradient is checked against float64 on the GPU's own forward selections (v, idx) and the
upstream gradients autograd hands to the node (captured by hooks). S is the same sum over absolute values, n_h the
number of rows that selected latent h, u = 2^-24:
  gv = <g, W_dec[:, h]> + g_h is an fp32 dot of D terms plus one add: |err| <= (D + 2) u S_gv;
  grad W_enc[h] = sum gv x and grad b_enc[h] = sum gv add n_h terms (in chunks, then chunk partials: fewer roundings
  than a serial sum): (D + n_h + 2) u S;
  grad W_dec[:, h] = sum v g: (n_h + 1) u S;   grad b_dec = sum_b g: (B + 1) u S;
  grad x = sum_j gv We[idx]: the gv error plus k terms: (D + k + 2) u S.
Each case prints its largest error / bound ratio (<= 1 passes).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import quantizedsae_b200 as Q
from quantizedsae_b200 import _lib as L
from tests import baseline_oracle
from tests.golden import cases

pytestmark = pytest.mark.gpu

U = 2.0 ** -24


def _model(cfg, dev, k=32, exact=True, return_dense=True):
    inp = cases.baseline_inputs(cfg)
    m = Q.BaselineSparseAutoencoder(cfg["D"], cfg["H"])
    m.load_state_dict({"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
                       "decoder.weight": torch.from_numpy(inp["Wd"]), "decoder.bias": torch.from_numpy(inp["bd"])})
    m.to(dev)
    m.topk, m.exact, m.return_dense, m.autograd = k, exact, return_dense, True
    return m, torch.from_numpy(inp["x"]).to(dev)


def _reference(x, vals, idx, g, g_h, g_vals, We, Wd, chunk=4096):
    """float64 gradients and their bounds S from the GPU's (vals, idx) and upstream gradients; rows in chunks."""
    B, D = x.shape
    H = We.shape[0]
    dev = x.device
    WdT, Wed = Wd.double().T.contiguous(), We.double()
    out = {n: torch.zeros(s, dtype=torch.float64, device=dev) for n, s in
           (("grad_we", (H, D)), ("grad_be", (H,)), ("grad_wd", (H, D)), ("grad_x", (B, D)))}
    S = {n: torch.zeros_like(t) for n, t in out.items()}
    for r0 in range(0, B, chunk):
        r = slice(r0, min(B, r0 + chunk))
        il = idx[r].long()
        xd, gd, vd = x[r].double(), g[r].double(), vals[r].double()
        cols = WdT[il]                                                   # [b, k, D]
        gv = torch.einsum("bd,bjd->bj", gd, cols)
        sgv = torch.einsum("bd,bjd->bj", gd.abs(), cols.abs())
        if g_h is not None:
            gh = torch.gather(g_h[r].double(), 1, il)
            gv, sgv = gv + gh, sgv + gh.abs()
        if g_vals is not None:
            gv, sgv = gv + g_vals[r].double(), sgv + g_vals[r].double().abs()
        flat = il.reshape(-1)
        for name, a, b in (("grad_we", gv, xd), ("grad_wd", vd, gd)):
            out[name].index_add_(0, flat, (a[:, :, None] * b[:, None, :]).reshape(-1, D))
        S["grad_we"].index_add_(0, flat, (sgv[:, :, None] * xd.abs()[:, None, :]).reshape(-1, D))
        S["grad_wd"].index_add_(0, flat, (vd.abs()[:, :, None] * gd.abs()[:, None, :]).reshape(-1, D))
        out["grad_be"].index_add_(0, flat, gv.reshape(-1))
        S["grad_be"].index_add_(0, flat, sgv.reshape(-1))
        out["grad_x"][r] = torch.einsum("bj,bjd->bd", gv, Wed[il])
        S["grad_x"][r] = torch.einsum("bj,bjd->bd", sgv, Wed[il].abs())
        del cols
    out["grad_wd"], S["grad_wd"] = out["grad_wd"].T, S["grad_wd"].T
    out["grad_bd"], S["grad_bd"] = g.double().sum(0), g.double().abs().sum(0)
    n_h = torch.bincount(idx.reshape(-1).long(), minlength=H).double()
    k = idx.shape[1]
    factor = {"grad_we": (D + n_h + 2)[:, None], "grad_be": D + n_h + 2, "grad_wd": (n_h + 1)[None, :],
              "grad_bd": float(B + 1), "grad_x": float(D + k + 2)}
    return {n: (out[n], U * factor[n] * S[n]) for n in out}


def _ratio(got, ref, bound):
    """max |got - ref| / bound (an entry with bound 0 must be exact)."""
    err = (got.double() - ref).abs()
    if bool(((bound == 0) & (err > 0)).any()):
        return float("inf")
    return float((err / bound.clamp_min(1e-300)).max()) if err.numel() else 0.0


def _step(m, x, lam):
    """0.5 * mse (+ lam * L1 of the latent) -> backward, with g = d loss / d recon and the latent's gradient captured."""
    seen = {}
    lat, recon = m(x)
    t = lat if m.return_dense else lat.values
    recon.register_hook(lambda g: seen.__setitem__("g", g.detach().clone()))
    loss = 0.5 * F.mse_loss(recon, x.detach())
    if lam > 0:
        t.register_hook(lambda g: seen.__setitem__("g_lat", g.detach().clone()))
        loss = loss + lam * t.abs().mean()
    loss.backward()
    return lat, recon, seen["g"], seen.get("g_lat")


def _check(name, m, x, lat, g, g_lat, x_grad=None):
    with torch.no_grad():
        sl = m.encode_topk(x)
    vals, idx = sl.values, sl.indices
    dense = m.return_dense
    ref = _reference(x, vals, idx, g, g_lat if dense else None, None if dense else g_lat, m.encoder[0].weight.detach(),
                     m.decoder.weight.detach())
    got = {"grad_we": m.encoder[0].weight.grad, "grad_be": m.encoder[0].bias.grad, "grad_wd": m.decoder.weight.grad,
           "grad_bd": m.decoder.bias.grad, "grad_x": x_grad}
    worst = 0.0
    for key, (r, bound) in ref.items():
        if got[key] is None:
            continue
        q = _ratio(got[key], r, bound)
        worst = max(worst, q)
        assert q <= 1.0, (name, key, q)
    print(f"{name}: max error / bound = {worst:.3e}")
    return worst


ODD = {
    "b37_d8_h1000": dict(D=8, H=1000, B=37, bf16=False, seed=81),
    "b300_d256_h2056": dict(D=256, H=2056, B=300, bf16=False, seed=82),
}
STEP_CASES = {**cases.BASELINE_CASES, **ODD}


@pytest.mark.parametrize("with_gh", [False, True])
@pytest.mark.parametrize("return_dense", [True, False])
@pytest.mark.parametrize("exact", [True, False])
@pytest.mark.parametrize("k", [1, 32, 65, 500])
@pytest.mark.parametrize("name", list(STEP_CASES))
def test_baseline_module_step(cuda_device, name, k, exact, return_dense, with_gh):
    cfg = STEP_CASES[name]
    m, x0 = _model(cfg, cuda_device, k=k, exact=exact, return_dense=return_dense)
    x_req = with_gh != return_dense                     # x.requires_grad on and off across the grid
    x = x0.clone().requires_grad_(x_req)
    # the forward bits (and flags) are the plain forward's
    m.autograd = False
    with torch.no_grad():
        lat0, r0 = m(x0)
    flags0 = None if m.last_flags is None else m.last_flags.clone()
    m.autograd = True
    lat, recon, g, g_lat = _step(m, x, 1e-2 if with_gh else 0.0)
    t0, t = (lat0, lat) if return_dense else (lat0.values, lat.values)
    assert torch.equal(t.detach(), t0) and torch.equal(recon.detach(), r0)
    if not return_dense:
        assert torch.equal(lat.indices, lat0.indices)
    if flags0 is not None:
        assert torch.equal(m.last_flags, flags0)
    _check(f"{name} k={k} exact={exact} dense={return_dense} g_h={with_gh} x_grad={x_req}", m, x0, lat, g, g_lat,
           x.grad if x_req else None)
    assert (x.grad is not None) == x_req


def test_baseline_step_matches_closed_form_oracle(cuda_device):
    """The numpy closed form of tests/baseline_oracle.py on the GPU's own selections, within the same bounds."""
    cfg = cases.BASELINE_CASES["baseline_d512_h4096"]
    m, x = _model(cfg, cuda_device)
    lat, recon, g, g_lat = _step(m, x, 1e-2)
    with torch.no_grad():
        sl = m.encode_topk(x)
    ref = _reference(x, sl.values, sl.indices, g, g_lat, None, m.encoder[0].weight.detach(), m.decoder.weight.detach())
    cpu = lambda t: t.detach().cpu().numpy()
    o = baseline_oracle.baseline_training_grads(cpu(x), cpu(m.encoder[0].weight), cpu(m.encoder[0].bias),
                                                cpu(m.decoder.weight), cpu(m.decoder.bias), cpu(g), cpu(g_lat),
                                                idx=cpu(sl.indices))
    got = {"grad_we": m.encoder[0].weight.grad, "grad_be": m.encoder[0].bias.grad, "grad_wd": m.decoder.weight.grad,
           "grad_bd": m.decoder.bias.grad}
    for key, t in got.items():
        # the oracle's v is float64 from the inputs, the GPU's fp32-accurate: grad W_dec carries v's own error as well
        r, bound = ref[key]
        extra = 1e-6 * bound / U if key == "grad_wd" else 0.0
        assert _ratio(t, torch.from_numpy(o[key]).to(cuda_device), bound + extra) <= 1.0, key


def _raw(x, sl, g, m, gx=True, out=None):
    W = m.encoder[0].weight.detach()
    return L.baseline_backward(x, sl.values, sl.indices, g, None, None, W, m._dec_rows(), want_grad_x=gx)


def test_outputs_are_written_and_unselected_latents_are_zero(cuda_device):
    import ctypes as C

    cfg = dict(D=64, H=2048, B=32, bf16=False, seed=21)
    m, x = _model(cfg, cuda_device)
    with torch.no_grad():
        sl = m.encode_topk(x)
    g = torch.randn((cfg["B"], cfg["D"]), device=cuda_device)
    B, H, D, k = cfg["B"], cfg["H"], cfg["D"], 32
    outs = [torch.full(s, float("nan"), device=cuda_device) for s in ((H, D), (H,), (D, H), (D,), (B, D))]
    n = L.baseline_backward_workspace_bytes(B, H, D, k)
    ws = torch.empty(n + 256, dtype=torch.uint8, device=cuda_device)
    wp = ws.data_ptr() + (-ws.data_ptr()) % 256
    L.check(L.load().qsae_baseline_backward(x.data_ptr(), sl.values.data_ptr(), sl.indices.data_ptr(), g.data_ptr(), None,
                                            None, m.encoder[0].weight.data_ptr(), m._dec_rows().data_ptr(), B, H, D, k,
                                            *[o.data_ptr() for o in outs], C.c_void_p(wp), n, L._stream()))
    torch.cuda.synchronize()
    for o in outs:
        assert not bool(torch.isnan(o).any())
    sel = torch.zeros(H, dtype=torch.bool, device=cuda_device)
    sel[sl.indices.reshape(-1).long()] = True
    assert int(sel.sum()) < H
    assert bool((outs[0][~sel] == 0).all()) and bool((outs[1][~sel] == 0).all()) and bool((outs[2][:, ~sel] == 0).all())
    # B = 0: zero gradients
    z = L.baseline_backward(x[:0], sl.values[:0], sl.indices[:0], g[:0], None, None, m.encoder[0].weight.detach(),
                            m._dec_rows(), want_grad_x=False)
    assert all(float(t.abs().max()) == 0.0 for t in z[:4])


def _skewed(dev, B, exact=False):
    cfg = dict(D=512, H=32768, B=B, bf16=True, seed=97)
    m, x = _model(cfg, dev, exact=exact, return_dense=False)
    with torch.no_grad():
        m.encoder[0].bias.zero_()
        m.encoder[0].bias[0] = 100.0          # wins every row
        m.encoder[0].bias[1:33] = 0.45        # raised: each wins about a quarter of the rows here
    return m, x


@pytest.mark.parametrize("B", [4096, 65536])
def test_skewed_dictionary(cuda_device, B):
    m, x = _skewed(cuda_device, B)
    x = x.clone().requires_grad_(True)
    lat, recon, g, g_lat = _step(m, x, 1e-3)
    counts = torch.bincount(lat.indices.reshape(-1).long(), minlength=m.hidden_dim)
    assert int(counts[0]) == B
    print(f"skew B={B}: latent 0 in {int(counts[0])} rows, latents 1..32 in {counts[1:33].float().mean().item() / B:.2f} "
          f"of the rows on average")
    _check(f"skew B={B}", m, x.detach(), lat, g, g_lat, x.grad)


def test_backward_is_bit_deterministic(cuda_device):
    m, x = _skewed(cuda_device, 4096)
    with torch.no_grad():
        sl = m.encode_topk(x)
    g = torch.randn_like(x)
    a = _raw(x, sl, g, m)
    b = _raw(x, sl, g, m)
    for p, q in zip(a, b):
        assert torch.equal(p, q)


def test_backward_in_cuda_graph(cuda_device):
    cfg = dict(D=512, H=4096, B=512, bf16=True, seed=95)
    m, x = _model(cfg, cuda_device)
    with torch.no_grad():
        sl = m.encode_topk(x)
    W, rows = m.encoder[0].weight.detach(), m._dec_rows()
    sx, sv, si, sg = x.clone(), sl.values.clone(), sl.indices.clone(), torch.randn_like(x)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            L.baseline_backward(sx, sv, si, sg, None, None, W, rows, want_grad_x=True)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = L.baseline_backward(sx, sv, si, sg, None, None, W, rows, want_grad_x=True)
    x2 = torch.randn_like(x)
    with torch.no_grad():
        sl2 = m.encode_topk(x2)
    g2 = torch.randn_like(x)
    sx.copy_(x2); sv.copy_(sl2.values); si.copy_(sl2.indices); sg.copy_(g2)
    graph.replay()
    torch.cuda.synchronize()
    direct = L.baseline_backward(x2, sl2.values, sl2.indices, g2, None, None, W, rows, want_grad_x=True)
    for p, q in zip(outs, direct):
        assert torch.equal(p, q)


def test_forward_launches_unchanged(cuda_device):
    m, x = _model(cases.BASELINE_CASES["baseline_d512_h4096"], cuda_device)
    m.autograd = False
    with torch.no_grad():
        m(x)
    n0 = L.launch_count()
    m(x)
    plain = L.launch_count() - n0
    m.autograd = True
    with torch.no_grad():
        n0 = L.launch_count()
        lat, _ = m(x)
        nograd = L.launch_count() - n0
    assert lat.grad_fn is None
    n0 = L.launch_count()
    lat, recon = m(x)
    with_node = L.launch_count() - n0
    assert recon.grad_fn is not None
    assert plain == nograd == with_node
    print(f"baseline forward: {plain} launches with autograd off, on under no_grad, and on with a node")


def test_baseline_trainer_sequence(cuda_device):
    cfg = dict(D=512, H=32768, B=4096, bf16=True, seed=23)
    m, x = _model(cfg, cuda_device)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    losses = []
    for step in range(5):
        opt.zero_grad(set_to_none=True)
        seen = {}
        lat, recon = m(x)
        recon.register_hook(lambda g: seen.__setitem__("g", g.detach().clone()))
        loss = 0.5 * F.mse_loss(recon, x)
        loss.backward()
        losses.append(float(loss))
        _check(f"trainer step {step}", m, x, lat, seen["g"], None)
        m.normalize_decoder_weights()
        opt.step()
        fresh = Q.BaselineSparseAutoencoder(cfg["D"], cfg["H"])
        fresh.load_state_dict(m.state_dict())
        fresh.to(cuda_device)
        with torch.no_grad():
            a, ra = m(x)
            b, rb = fresh(x)
        assert torch.equal(a, b) and torch.equal(ra, rb), step
    print(f"baseline trainer loop: losses {losses}")
    assert losses[-1] < losses[0]


def test_cpu_tensors_raise(cuda_device):
    m = Q.BaselineSparseAutoencoder(16, 64)
    m.autograd = True
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros((4, 16), requires_grad=True))
    m.to(cuda_device)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros((4, 16)))
