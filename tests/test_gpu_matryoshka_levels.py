"""q_sae (QuantizedMatryoshkaSAE) and rq_sae (ResidualQuantizedSAE) at every level count, with level boundaries on and
off the 8-grid, against the float64 oracle (oracle/qsae_oracle.py, oracle/train_oracle.py).

Two comparison rules (u = 2^-24):

Activity decisions. A latent is active when sigmoid_f32(z_f32) > 0.5, i.e. z_f32 >= THR = 1.5 u. z is computed here in
float64, and the fp32 dot product (D products and the bias) is within delta = (D + 1) u (sum_d |x_d W_hd| + |b_h|) of
it. Outside the band |z - THR| <= delta the kernel's decision must equal (z >= THR) exactly; inside it either decision
is accepted (such entries are rare and counted). The sparse path reports its own decisions (forward_active) and the
decoder's input shows them; there the level counts equal their sums exactly. The dense path does not report them: its
level counts must lie between the forced and the forced-plus-band sums, and each band entry may add its term to the
reconstruction, so it widens that row's bound by |scale_h T_hd|.

Reconstructions, level by level. The reference is the float64 level sum over the kernel's own activity set. The bound
comes from the magnitude the fp32 running sum went through, S_l[b, d] = |bias_d| + sum over the active h of levels
<= l of |scale_h T_hd|; n is the number of terms (active latents of levels <= l, plus the bias).
  sparse path: every term 2 scale_h is exact and enters the running sum by one fp32 addition, whose rounding is at
      most u of the running magnitude <= S_l: |got - ref| <= n 2^-23 S_l (a factor 2 of margin).
  dense path: the operand is scale as bf16 hi + lo, within 2^-18 of scale (2^-16 allowed); the level GEMMs add the
      exact products hi T, lo T in fp32 (tensor-core accumulation, split-K reduction, level chain, leftover columns),
      each addition at most 2^-23 of the running magnitude even when truncating; 2^-22 per addition and 32 additions
      for the splits, the chain and the leftover kernel: |got - ref| <= (2^-16 + (n + 32) 2^-22) S_l.
  Each level's increment result[l] - result[l - 1] is checked too, with the same bound in which n counts only the
  terms added at level l (the rounding of the earlier levels cancels in the difference). Both bounds are far below
  one last-level term (2 scale_h, a 2^-(n_bits - 1) fraction of a level-0 term): dropping or doubling one active
  latent of the last level violates them, which every sparse-activity case asserts.
"""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import quantizedsae_b200 as Q
from oracle import qsae_oracle as O
from oracle import train_oracle as TO
from quantizedsae_b200 import training
from tests.golden import cases

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
THR = 1.5 * U


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def report(msg):
    print(f"[levels] {msg}")


# ------------------------------------------------------------------------------------------
# shape matrix: (n_bits, H, D, B)
# ------------------------------------------------------------------------------------------
SHAPES = [
    (1, 1000, 48, 33), (2, 1000, 16, 130), (1, 4096, 512, 33), (2, 4096, 48, 1),   # NL = 1 outside rq_sae, NL = 2
    (5, 4096, 512, 130), (6, 4096, 16, 33),                                      # NL = 8, boundaries on the 128-grid
    (7, 4096, 48, 130), (8, 4096, 512, 33),                                      # 8-grid only; 64- and 32-wide levels
    (8, 32768, 512, 130),                                                        # headline size
    (8, 1000, 512, 130), (5, 1000, 16, 33),                                      # boundaries off the 8-grid
    (4, 2056, 48, 33), (4, 32776, 512, 1),                                       # one level boundary off the 8-grid
]
IDS = [f"nb{nb}-h{H}-d{D}-b{B}" for nb, H, D, B in SHAPES]
LEVEL_SIZES = {
    (8, 1000): [7, 7, 15, 31, 62, 125, 250, 503], (5, 1000): [62, 62, 125, 250, 501],
    (4, 2056): [257, 257, 514, 1028], (4, 32776): [4097, 4097, 8194, 16388], (8, 4096): [32, 32, 64, 128, 256, 512, 1024, 2048],
}


def qsae_cfg(nb, H, D, B, bf16=False, enc_bias=None, seed=None):
    # about 3 % of the latents active (z ~ N(0, 2 D / (H + D)) for xavier weights and unit x), ~0.1 % at H = 32768
    if enc_bias is None:
        enc_bias = -0.543 if H >= 32768 else -1.9 * (2.0 * D / (H + D)) ** 0.5
    return dict(D=D, H=H, n_bits=nb, abs_range=4.0, B=B, enc_bias=enc_bias, bf16=bf16, allow_bias=True,
                seed=seed if seed is not None else 1000 + nb * 7 + H + D + B)


def qsae_case(cfg):
    """cases.qsae_inputs plus edge weights: W / Wm entries of exactly 0.0 and -0.0 (sigmoid 0.5: sign +1), and one
    always-active dictionary row whose T is all zero (W = +, Wm = -: scale = factor / 1e-8) that must add nothing."""
    inp = cases.qsae_inputs(cfg)
    W, Wm, be = inp["W"], inp["Wm"], inp["be"]
    W[2, 0:16:2], W[2, 1:16:2] = 0.0, -0.0
    Wm[2, 0:16:2], Wm[2, 1:16:2] = -0.0, 0.0
    hz = zero_row(cfg)
    W[hz], Wm[hz] = np.abs(W[hz]), -np.abs(Wm[hz])
    be[hz] = 10.0
    return inp


def zero_row(cfg):
    starts = np.cumsum([0] + O.matryoshka_level_sizes(cfg["H"], cfg["n_bits"]))
    return int(starts[-2]) + 1 if cfg["H"] > 8 else 0   # in the last level, next to its first row


def make_qsae(inp, cfg, dev):
    m = Q.QuantizedMatryoshkaSAE(cfg["D"], cfg["H"], 32, cfg["abs_range"], cfg["n_bits"], cfg["allow_bias"])
    m.load_state_dict({"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
                       "decoder.weight": torch.from_numpy(inp["W"]), "decoder.weight_mirror": torch.from_numpy(inp["Wm"]),
                       "decoder.bias": torch.from_numpy(inp["bd"])}, strict=True)
    return m.to(dev).eval()


# ------------------------------------------------------------------------------------------
# the two rules
# ------------------------------------------------------------------------------------------
def activity_band(x, We, be, extra=0.0, chunk=256):
    """-> (forced [B, H] bool: z >= THR outside the band, band [B, H] bool), float64 z with the fp32 error band."""
    x64, W64, b64 = x.astype(np.float64), We.astype(np.float64), be.astype(np.float64)
    D = x.shape[1]
    forced = np.empty((x.shape[0], We.shape[0]), dtype=bool)
    band = np.empty_like(forced)
    for r in range(0, x.shape[0], chunk):
        xs = x64[r:r + chunk]
        z = xs @ W64.T + b64
        delta = (D + 1) * U * (np.abs(xs) @ np.abs(W64).T + np.abs(b64)) + extra
        band[r:r + chunk] = np.abs(z - THR) <= delta
        forced[r:r + chunk] = (z >= THR) & ~band[r:r + chunk]
    return forced, band


def check_decisions(act, forced, band, what):
    """The kernel's decisions act [B, H] against the rule; -> number of band entries."""
    wrong = (act != forced) & ~band
    assert not wrong.any(), f"{what}: {int(wrong.sum())} activity decisions outside the rounding band differ, " \
                            f"first at {np.argwhere(wrong)[:4].tolist()}"
    nb = int(band.sum())
    assert nb <= max(2, band.size // 1000), f"{what}: {nb} of {band.size} pre-activations within the rounding band"
    return nb


def level_sums_f64(act, rows, starts, bias):
    """Cumulative float64 level sums of act [B, H] over the dictionary rows [H, D] -> ([L, B, D], terms [L, B])."""
    A = sp.csr_matrix(act, dtype=np.float64)   # from the non-zeros: no dense float64 copy of a [B, H] mask
    B, D = act.shape[0], rows.shape[1]
    L = len(starts) - 1
    out, n = np.empty((L, B, D)), np.empty((L, B))
    acc = np.zeros((B, D)) + (bias if bias is not None else 0.0)
    for l in range(L):
        a = A[:, starts[l]:starts[l + 1]]
        acc = acc + a @ rows[starts[l]:starts[l + 1]]
        out[l], n[l] = acc, np.asarray(a.sum(1)).ravel()
    return out, n


def bound(S, n, dense):
    n = n[:, None]
    return (2.0 ** -16 + (n + 32) * 2.0 ** -22) * S if dense else n * 2.0 ** -23 * S


def check_levels(got, act, Tm, scale, starts, bias, dense, what, band=None, perturb=True):
    """got [L, B, D] fp32 against the float64 level sums over act, cumulative levels and increments. band [B, H]:
    undetermined decisions (dense path), each of which may add its term: the bound grows by their |scale T|. Shows on
    a row without band entries that dropping or doubling one active last-level latent breaks the bound.
    -> largest error / bound ratio."""
    rows = Tm.astype(np.float64) * scale.astype(np.float64)[:, None]
    b64 = bias.astype(np.float64) if bias is not None else None
    ref, n_inc = level_sums_f64(act, rows, starts, b64)
    S, _ = level_sums_f64(act, np.abs(rows), starts, np.abs(b64) if b64 is not None else None)
    if band is not None and band.any():
        E, n_band = level_sums_f64(band, np.abs(rows), starts, None)
    else:
        E, n_band = np.zeros_like(S), np.zeros_like(n_inc)
    n_inc = n_inc + n_band
    n_cum = np.cumsum(n_inc, 0) + 1
    got = np.asarray(got, dtype=np.float64)
    assert np.isfinite(got).all(), f"{what}: non-finite outputs"
    L = got.shape[0]
    worst = 0.0
    for l in range(L):
        checks = [("level", got[l], ref[l], bound(S[l] + E[l], n_cum[l], dense), E[l])]
        if l > 0:
            checks.append(("increment", got[l] - got[l - 1], ref[l] - ref[l - 1],
                           bound(S[l] + E[l], n_inc[l] + 1, dense), E[l] - E[l - 1]))
        for kind, g, r, b, slack in checks:
            err = np.abs(g - r)
            bad = err > b + slack
            assert not bad.any(), f"{what}: {kind} {l}: {int(bad.sum())} entries beyond the bound, first " \
                                  f"{np.argwhere(bad)[0].tolist()}: |err| {err[bad][0]:.3e} > {(b + slack)[bad][0]:.3e}"
            pos = (b > 0) & (slack == 0)   # the ratio is reported where no band decision widens the bound
            if pos.any():
                worst = max(worst, float((err[pos] / b[pos]).max()))
    if perturb:   # the clean row with the loosest last-level bound: one active latent more or less must not pass
        lo, hi = starts[L - 1], starts[L]
        last = act[:, lo:hi] & Tm[lo:hi].any(1)[None, :]
        if band is not None:
            last &= ~band.any(1)[:, None]
        b_last = bound(S[L - 1], n_cum[L - 1], dense)
        cand = np.nonzero(last.any(1))[0]
        assert len(cand), f"{what}: no row with an active last-level latent to perturb"
        r = int(cand[np.argmax(b_last[cand].max(1))])
        h = lo + int(np.nonzero(last[r])[0][-1])
        for f in (-1.0, 1.0):   # dropped, doubled
            assert np.any(np.abs(got[L - 1, r] - (ref[L - 1, r] + f * rows[h])) > b_last[r]), \
                f"{what}: a last-level latent {'dropped' if f < 0 else 'doubled'} would pass the bound"
    return worst


def sparse_decisions(a_idx, a_cnt, H):
    a_idx, a_cnt = a_idx.cpu().numpy(), a_cnt.cpu().numpy()
    B, cap = a_idx.shape
    assert np.all(a_cnt <= cap)
    act = np.zeros((B, H), dtype=bool)
    for b in range(B):
        lst = a_idx[b, :a_cnt[b]]
        assert np.all((lst >= 0) & (lst < H)) and len(set(lst.tolist())) == len(lst), f"row {b}: bad active list"
        assert np.all(a_idx[b, a_cnt[b]:] == -1)
        act[b, lst] = True
    return act


def level_sums(act, starts):
    return np.array([int(act[:, starts[l]:starts[l + 1]].sum()) for l in range(len(starts) - 1)])


def group_counts(groups, B):
    g = np.array([float(v) for v in groups], dtype=np.float64)
    cnt = np.rint(g * B).astype(np.int64)
    assert np.all(cnt < 2 ** 23)   # the float32 mean still identifies the integer count
    return cnt


def starts_of(cfg):
    return [int(v) for v in np.cumsum([0] + O.matryoshka_level_sizes(cfg["H"], cfg["n_bits"]))]


def dictionary(inp, cfg):
    Tm, scale, _, _ = O.qsae_dictionary(inp["W"], inp["Wm"], n_bits=cfg["n_bits"], abs_range=cfg["abs_range"])
    return Tm, scale


# ------------------------------------------------------------------------------------------
# pack / unpack
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nb,H,D,B", SHAPES, ids=IDS)
def test_pack_unpack_every_level_count(cuda_device, nb, H, D, B):
    cfg = qsae_cfg(nb, H, D, B)
    inp = qsae_case(cfg)
    m = make_qsae(inp, cfg, cuda_device)
    sizes = O.matryoshka_level_sizes(H, nb)
    assert m.decoder.nested_dictionary_size == sizes
    if (nb, H) in LEVEL_SIZES:
        assert sizes == LEVEL_SIZES[(nb, H)]
    packed, scale = m.decoder._packed()
    Tm, sref = dictionary(inp, cfg)
    codes = packed.cpu().numpy().view(np.uint32)
    ent = ((codes[:, :, None] >> (2 * np.arange(16, dtype=np.uint32))) & 3).reshape(H, -1)
    assert np.array_equal(np.where(ent & 1, np.where(ent & 2, -2, 2), 0).astype(np.int8), Tm)
    assert np.all(Tm[2, :16] == 2)                                   # sigmoid(+-0.0) = 0.5 -> +1 on both sides
    hz = zero_row(cfg)
    assert not Tm[hz].any()
    s = scale.cpu().numpy()
    np.testing.assert_allclose(s, sref, rtol=2e-7, atol=0)
    # the level factor on both sides of every boundary: scale (||T|| + 1e-8) = 2^(n_bits - l - 2) quant_step
    starts = starts_of(cfg)
    qstep = cfg["abs_range"] / 2 ** (nb - 1)
    norms = np.sqrt((Tm.astype(np.float64) ** 2).sum(1))
    for l in range(nb):
        for h in {starts[l], starts[l + 1] - 1}:
            assert s[h] * (norms[h] + 1e-8) == pytest.approx(2.0 ** (nb - l - 2) * qstep, rel=1e-6), (l, h)
    assert s[hz] == pytest.approx(2.0 ** (nb - (nb - 1) - 2) * qstep / 1e-8, rel=1e-6)
    tt = m.decoder._t_bf16()
    assert tuple(tt.shape) == (D, H)
    assert np.array_equal(tt.float().cpu().numpy(), Tm.T.astype(np.float32))


# ------------------------------------------------------------------------------------------
# sparse path
# ------------------------------------------------------------------------------------------
def run_sparse(m, inp, cfg, dev, what):
    x = T(inp["x"], dev)
    with torch.no_grad():
        out = m.forward_active(x)
        groups, result = m(x)
    assert m.last_path == "sparse"
    H, B = cfg["H"], cfg["B"]
    act = sparse_decisions(out["active_idx"], out["active_cnt"], H)
    forced, band = activity_band(inp["x"], inp["We"], inp["be"])
    n_band = check_decisions(act, forced, band, what)
    starts = starts_of(cfg)
    assert np.array_equal(out["level_counts"].cpu().numpy(), level_sums(act, starts))
    assert np.array_equal(group_counts(groups, B), level_sums(act, starts))
    for a, b in zip(result, out["reconstruction_levels"]):
        assert torch.equal(a, b)
    Tm, scale = dictionary(inp, cfg)
    got = torch.stack(result).cpu().numpy()
    ratio = check_levels(got, act, Tm, scale, starts, inp["bd"], False, what)
    report(f"{what}: sparse path, {int(act.sum(1).mean())} active per row, {n_band} band entries, max err/bound {ratio:.3g}")
    return act


@pytest.mark.parametrize("exact", [True, False], ids=["exact", "fast"])
@pytest.mark.parametrize("nb,H,D,B", SHAPES, ids=IDS)
def test_sparse_forward_levels(cuda_device, nb, H, D, B, exact):
    cfg = qsae_cfg(nb, H, D, B, bf16=not exact)
    inp = qsae_case(cfg)
    m = make_qsae(inp, cfg, cuda_device)
    m.exact = exact
    run_sparse(m, inp, cfg, cuda_device, f"sparse {'exact' if exact else 'fast'} nb={nb} H={H} D={D} B={B}")


def test_sparse_forward_levels_headline_batch(cuda_device):
    """B = 4096 at 512 -> 32768, n_bits = 8: every decision of 134 M checked, all levels of every row."""
    cfg = qsae_cfg(8, 32768, 512, 4096)
    inp = qsae_case(cfg)
    m = make_qsae(inp, cfg, cuda_device)
    run_sparse(m, inp, cfg, cuda_device, "sparse exact nb=8 H=32768 D=512 B=4096")


@pytest.mark.parametrize("nb,H,D,B", SHAPES, ids=IDS)
def test_decoder_alone_levels(cuda_device, nb, H, D, B):
    """m.decoder(m.encode(x)): dense sigmoid latents -> compact_dense -> decode_matryoshka_lists. torch's sigmoid rounds
    to exactly 0.5 for 0 < z <~ 1.2e-7 depending on its expf, so the band is widened by 2^-22."""
    cfg = qsae_cfg(nb, H, D, B)
    inp = qsae_case(cfg)
    m = make_qsae(inp, cfg, cuda_device)
    with torch.no_grad():
        lat = m.encode(T(inp["x"], cuda_device))
        groups, result = m.decoder(lat)
    act = (lat > 0.5).cpu().numpy()
    forced, band = activity_band(inp["x"], inp["We"], inp["be"], extra=2.0 ** -22)
    what = f"decoder nb={nb} H={H} D={D} B={B}"
    n_band = check_decisions(act, forced, band, what)
    starts = starts_of(cfg)
    assert np.array_equal(group_counts(groups, B), level_sums(act, starts))
    Tm, scale = dictionary(inp, cfg)
    ratio = check_levels(torch.stack(result).cpu().numpy(), act, Tm, scale, starts, inp["bd"], False, what)
    report(f"{what}: decoder alone, {n_band} band entries, max err/bound {ratio:.3g}")


# ------------------------------------------------------------------------------------------
# dense path
# ------------------------------------------------------------------------------------------
def check_dense(groups, result, inp, cfg, what, rows=None, perturb=True):
    """The dense path does not report its decisions: a decision inside the band may have gone either way, so the
    level counts lie between the forced and the forced-plus-band sums, and each band entry widens its row's bound."""
    x, B = inp["x"], cfg["B"]
    if rows is not None:
        x = x[rows]
    forced, band = activity_band(x, inp["We"], inp["be"])
    n_band = check_decisions(forced, forced, band, what)
    starts = starts_of(cfg)
    if rows is None:
        cnt = group_counts(groups, B)
        lo, nb = level_sums(forced, starts), level_sums(band, starts)
        assert np.all((lo <= cnt) & (cnt <= lo + nb)), f"{what}: level counts {cnt} outside [{lo}, {lo + nb}]"
    got = torch.stack(result).cpu().numpy()
    if rows is not None:
        got = got[:, rows]
    ratio = check_levels(got, forced, *dictionary(inp, cfg), starts, inp["bd"], True, what, band=band, perturb=perturb)
    report(f"{what}: dense path, {int(forced.sum(1).mean())} active per row, {n_band} band entries in "
           f"{int(band.any(1).sum())} rows, max err/bound {ratio:.3g}")


@pytest.mark.parametrize("exact", [True, False], ids=["exact", "fast"])
@pytest.mark.parametrize("nb,H,D,B", SHAPES, ids=IDS)
def test_dense_forward_levels(cuda_device, tuning, nb, H, D, B, exact):
    """dense_mode = "always" at every level count and boundary layout (H % 8 == 0). Where every boundary is a multiple
    of 128 the encoder epilogue writes the operand itself; that form must equal the streaming operand kernel's bits."""
    cfg = qsae_cfg(nb, H, D, B, bf16=not exact)
    inp = qsae_case(cfg)
    m = make_qsae(inp, cfg, cuda_device)
    m.dense_mode, m.exact = "always", exact
    x = T(inp["x"], cuda_device)
    with torch.no_grad():
        groups, result = m(x)
    assert m.last_path == "dense"
    what = f"dense {'exact' if exact else 'fast'} nb={nb} H={H} D={D} B={B}"
    check_dense(groups, result, inp, cfg, what)
    if all(s % 128 == 0 for s in starts_of(cfg)):
        tuning("QSAE_DENSE_STEP_FUSED", "0")
        with torch.no_grad():
            g0, r0 = m(x)
        assert [float(v) for v in g0] == [float(v) for v in groups]
        assert all(torch.equal(a, b) for a, b in zip(result, r0))


def test_dense_path_needs_hidden_dim_multiple_of_8(cuda_device):
    cfg = qsae_cfg(4, 1004, 16, 4)
    m = make_qsae(qsae_case(cfg), cfg, cuda_device)
    m.dense_mode = "always"
    with pytest.raises(RuntimeError, match=r"hidden_dim must be a multiple of 8, got 1004 \(the A operand and T\^T rows "
                                           r"are not padded"):
        with torch.no_grad():
            m(torch.randn((4, 16), device=cuda_device))


# ------------------------------------------------------------------------------------------
# overflow: NaN poisoning and the dense fallback
# ------------------------------------------------------------------------------------------
def test_overflow_poisons_every_level_at_eight_levels(cuda_device):
    """n_bits = 8: a batch that overflows the survivor lists is NaN at every level; "auto" then serves it densely."""
    import warnings

    cfg = qsae_cfg(8, 32768, 512, 64, seed=7)
    inp = qsae_case(cfg)
    m = make_qsae(inp, cfg, cuda_device)
    x = T(inp["x"], cuda_device)
    with torch.no_grad():
        m(x)
        assert m._regime[1] == "sparse"
        We = inp["We"]
        xbig = (inp["x"] * 40.0 + 30.0 * np.sign(We[:2000].sum(0))).astype(np.float32)   # thousands active per row
        g2, r2 = m(T(xbig, cuda_device))
        torch.cuda.synchronize()
        assert m.overflowed()
        assert all(bool(torch.isnan(r).all()) for r in r2)
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            g3, r3 = m(T(xbig, cuda_device))
    assert any("overflowed" in str(i.message) for i in w)
    assert m.last_path == "dense"
    rows = np.arange(8)
    check_dense(g3, r3, dict(inp, x=xbig), cfg, "overflow fallback nb=8 H=32768", rows=rows, perturb=False)


def test_untrained_model_off_grid_levels_falls_back_to_dense(cuda_device):
    """H = 32776, n_bits = 4: levels [4097, 4097, 8194, 16388]. An untrained model (zero encoder bias, ~50 % active)
    overflows the sparse lists; "auto" redoes the forward on the dense path, whose level GEMMs end at the 8-aligned
    cuts and whose leftover columns are added by the tail kernel."""
    cfg = qsae_cfg(4, 32776, 512, 48, enc_bias=0.0, seed=93)
    inp = qsae_case(cfg)
    m = make_qsae(inp, cfg, cuda_device)
    with torch.no_grad():
        groups, result = m(T(inp["x"], cuda_device))
    assert m.overflowed() and m.last_path == "dense"
    check_dense(groups, result, inp, cfg, "untrained nb=4 H=32776", perturb=False)
    rg, _, act = O.qsae_forward(inp["x"], inp["We"], inp["be"], inp["W"], inp["Wm"], inp["bd"], n_bits=4, abs_range=4.0)
    assert 15000 < act.sum(1).mean() < 18000
    np.testing.assert_allclose(np.array([float(v) for v in groups]), rg, rtol=2e-5)


# ------------------------------------------------------------------------------------------
# rq_sae at the default n_bits = 8
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H,D", [(1000, 64), (1000, 512), (2048, 64), (2048, 512)])
def test_rqsae_eight_stages(cuda_device, H, D):
    """Stage t is checked against the oracle on the kernel's own stage-t input r_t, rebuilt in fp32 as
    r_{t+1} = (r_t - recon_t) * 2 (a stage's error doubles at every later stage)."""
    nb = 8
    cfg = dict(D=D, H=H, n_bits=nb, abs_range=4.0, B=33, enc_bias=-1.9 * (2.0 * D / (H + D)) ** 0.5, seed=H + D)
    inp = cases.rqsae_inputs(cfg)
    m = Q.ResidualQuantizedSAE(D, H, 32, cfg["abs_range"], nb)
    assert m.sae_hidden_dims == O.matryoshka_level_sizes(H, nb)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in cases.rqsae_state_dict(inp, nb).items()}, strict=True)
    m.to(cuda_device).eval()
    x = T(inp["x"], cuda_device)
    with torch.no_grad():
        groups, recons = m(x)
        assert all(s.last_path == "sparse" for s in m.saes)
        m.saes[0].dense_mode = "never"                       # the stage-by-stage path with residual_update
        g1, r1 = m(x)
    for a, b in zip(recons, r1):
        assert torch.equal(a, b)
    np.testing.assert_allclose([float(v) for v in groups], [float(v) for v in g1], rtol=1e-6)
    r = inp["x"]
    for t, sae in enumerate(m.saes):
        stage = dict(D=D, H=m.sae_hidden_dims[t], n_bits=1, abs_range=4.0, B=cfg["B"])
        sinp = dict(x=r, We=inp[f"We{t}"], be=inp[f"be{t}"], W=inp[f"W{t}"], Wm=inp[f"Wm{t}"],
                    bd=inp[f"bd{t}"] if t == 0 else None)
        rt = T(r, cuda_device)
        with torch.no_grad():
            out = sae.forward_active(rt)
            *_, fused = sae._forward_sparse(rt, want_residual=True)
        assert torch.equal(out["reconstruction_levels"][0], recons[t])
        act = sparse_decisions(out["active_idx"], out["active_cnt"], stage["H"])
        what = f"rq_sae H={H} D={D} stage {t} (width {stage['H']})"
        forced, band = activity_band(r, sinp["We"], sinp["be"])
        check_decisions(act, forced, band, what)
        assert int(out["level_counts"][0]) == int(act.sum()) == round(float(groups[t]) * cfg["B"])
        Tm, scale = dictionary(sinp, stage)
        ratio = check_levels(recons[t].cpu().numpy()[None], act, Tm, scale, [0, stage["H"]], sinp["bd"], False, what)
        report(f"{what}: sparse path, max err/bound {ratio:.3g}")
        r = ((r - recons[t].cpu().numpy()) * np.float32(2)).astype(np.float32)
        assert np.array_equal(fused.cpu().numpy(), r), f"{what}: fused residual differs from (r - recon) * 2"


# ------------------------------------------------------------------------------------------
# q_sae training: decoder gradients of one trainer step
# ------------------------------------------------------------------------------------------
def close(got, want, rtol=2e-4, atol_frac=2e-6):
    want = np.asarray(want, dtype=np.float64)
    got = got.detach().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    atol = atol_frac * max(1e-30, float(np.abs(want).max()))
    np.testing.assert_allclose(got.astype(np.float64), want, rtol=rtol, atol=atol)


@pytest.mark.parametrize("nb,H,D,B,seed", [(1, 1000, 64, 33, 1001), (2, 4096, 48, 17, 4098), (5, 1000, 64, 33, 1005),
                                           (8, 1000, 512, 33, 1019), (8, 4096, 64, 40, 4106)])
def test_qsae_trainer_decoder_grads_levels(cuda_device, nb, H, D, B, seed):
    """The oracle decides activity on its own fp32 pre-activations; the seeds give inputs without band entries, where
    those decisions are the kernel's."""
    cfg = qsae_cfg(nb, H, D, B, seed=seed)
    inp = cases.qsae_inputs(cfg)
    _, band = activity_band(inp["x"], inp["We"], inp["be"])
    assert not band.any()
    m = make_qsae(inp, cfg, cuda_device)
    x = T(inp["x"], cuda_device)
    training.qsae_trainer_decoder_grads(m, x, active_cap=64)
    want = TO.qsae_training_decoder_grads(inp["x"], inp["We"], inp["be"], inp["W"], inp["Wm"], inp["bd"], n_bits=nb,
                                          abs_range=cfg["abs_range"])
    close(m.decoder.weight.grad, want["secant_W"])
    close(m.decoder.weight_mirror.grad, want["secant_Wm"])
    close(m.decoder.bias.grad, want["bias"])
    assert np.array_equal(m.decoder._ctx["z2"].cpu().numpy(), want["z2"].astype(np.int64))
    if nb == 8:   # joint_gradient: the secant term weighted by n_bits - level
        m.zero_grad(set_to_none=True)
        m.decoder.joint_gradient = True
        m.decoder.apply_secant_grad()
        dW, dWm = TO.qsae_secant_term(want["z2"], inp["W"], inp["Wm"], B, n_bits=nb, abs_range=cfg["abs_range"],
                                      joint_gradient=True)
        close(m.decoder.weight.grad, dW)
        close(m.decoder.weight_mirror.grad, dWm)
