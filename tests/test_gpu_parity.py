"""GPU parity tests (run on the B200 box: pytest -m gpu). Every call goes through the C ABI
(libqsae_b200.so via ctypes); results are checked against
  * the committed outputs of the unmodified reference (tests/golden/*.npz), and
  * the numpy oracle on seeded inputs, bit-exact for integer / index work.
Tolerances (stated once):
  dictionary integers, packed nibbles, top-k indices ........ bit exact
  latent values (bf16-representable inputs or exact mode) .... |dv| <= 1e-5 * max(1, |v|)
  reconstructions (fp32 accumulate) ........................... atol 1e-4 * rms(recon) + rtol 1e-4
"""
import numpy as np
import pytest
import torch

import quantizedsae_b200 as Q
from oracle import qsae_oracle as O
from quantizedsae_b200 import _lib as L
from tests.golden import cases

pytestmark = pytest.mark.gpu


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def assert_recon_close(got, ref):
    rms = float(np.sqrt(np.mean(np.square(ref, dtype=np.float64)))) + 1e-30
    np.testing.assert_allclose(got, ref, rtol=1e-4, atol=1e-4 * rms)


def assert_vals_close(got, ref):
    assert np.all(np.abs(got - ref) <= 1e-5 * np.maximum(1.0, np.abs(ref)))


def assert_topk_matches(gv, gi, z, k, eps=1e-6):
    """Index order must equal the oracle's (value desc, index asc) bit for bit, except where the
    oracle's own fp32 values are tied to within accumulation-order noise (|dz| <= eps * max(1,|z|)):
    there any order / choice among the near-equal entries is accepted. Near-ties must stay rare:
    at most 2 % of the rows for k <= 224; for the large-k paths (thousands of adjacent order
    statistics per row) at most 0.5 % of all (row, rank) positions."""
    rv, ri = O.topk_rows(z, k)
    bad_rows = np.nonzero((gi != ri).any(1))[0]
    for r in bad_rows:
        assert len(set(gi[r].tolist())) == k, f"row {r}: duplicate indices"
        got = z[r, gi[r].astype(np.int64)]
        assert np.all(np.abs(got - rv[r]) <= eps * np.maximum(1.0, np.abs(rv[r]))), \
            f"row {r}: differs from the oracle beyond a near-tie: {gi[r]} vs {ri[r]}"
    if k <= 224:
        assert len(bad_rows) <= max(1, gi.shape[0] // 50), f"{len(bad_rows)} rows rely on the near-tie rule"
    else:
        assert int((gi != ri).sum()) <= max(2, gi.size // 200), f"{int((gi != ri).sum())} positions rely on the near-tie rule"
    assert_vals_close(gv, np.take_along_axis(z, gi.astype(np.int64), axis=1))


def test_device_and_library(cuda_device):
    L.check(L.load().qsae_check_device())
    assert torch.cuda.get_device_capability(0)[0] == 10


# ------------------------------------------------------------------------------------------
# weight preparation
# ------------------------------------------------------------------------------------------
def test_cast_bf16_bit_exact(cuda_device):
    a = np.random.default_rng(0).standard_normal((1000, 77)).astype(np.float32)
    a[0, :4] = [0.0, -0.0, 1e-40, 3.3895314e38]
    got = L.cast_bf16(T(a, cuda_device)).float().cpu().numpy()
    assert np.array_equal(got, cases.round_bf16(a))


@pytest.mark.parametrize("name", list(cases.BSAE_CASES))
def test_pack_bitplanes_matches_reference_int_weights(cuda_device, golden_dir, name):
    cfg = cases.BSAE_CASES[name]
    g = np.load(golden_dir / f"{name}.npz")
    inp = cases.bsae_inputs(cfg)
    packed, pol, gap = L.pack_bitplanes(T(inp["logits"], cuda_device), cfg["D"], cfg["n_bits"])
    got = O.unpack_nibbles(packed.cpu().numpy()) if cfg["n_bits"] <= 4 else packed.cpu().numpy().view(np.int8)
    assert cases.int_weights_match(got, g)                     # reference quantized_int_weights()
    assert pol == pytest.approx(float(g["polarize"]), rel=1e-5, abs=1e-9)
    assert (gap == 0.0) == cfg["polar"]
    soft = L.dequant_soft(T(inp["logits"], cuda_device), cfg["D"], cfg["n_bits"]).cpu().numpy()
    np.testing.assert_allclose(soft[:4], g["soft_weights_row0"], rtol=1e-5, atol=2e-7 * 2 ** cfg["n_bits"])


def test_readme_known_answer_and_all_nibbles(cuda_device):
    pat = np.array([[(v >> i) & 1 for i in range(4)] for v in range(16)], dtype=np.float32)
    logits = np.where(pat.reshape(1, 64) > 0, 110.0, -110.0).astype(np.float32)
    packed, pol, gap = L.pack_bitplanes(T(logits, cuda_device), 16, 4)
    ints = O.unpack_nibbles(packed.cpu().numpy())[0]
    assert ints.tolist() == [v if v < 8 else v - 16 for v in range(16)]
    assert ints[0b0101 + 0] == 5 and ints[10] == -6             # README.md:100: bits [0,1,0,1] LSB-first -> -6
    vals = T(np.ones((1, 1), np.float32), cuda_device)
    idx = T(np.zeros((1, 1), np.int32), cuda_device)
    recon = L.decode_int4(vals, idx, packed, 1, 16, 4.0 / 8, None).cpu().numpy()[0]
    assert recon[10] == -3.0                                     # -6 * (4.0 / 8)
    assert pol == 0.0 and gap == 0.0


# ------------------------------------------------------------------------------------------
# sparse decoders, densify
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,k,H,D", [(1, 1, 256, 8), (37, 4, 2048, 64), (130, 32, 4096, 512), (9, 65, 1024, 256)])
def test_decoders_vs_oracle(cuda_device, B, k, H, D):
    rng = np.random.default_rng(B * 7 + k)
    iw = rng.integers(-8, 8, size=(H, D)).astype(np.int8)
    vals = rng.standard_normal((B, k)).astype(np.float32)
    idx = np.stack([rng.choice(H, k, replace=False) for _ in range(B)]).astype(np.int32)
    idx[0, -1] = -1                                              # empty slot is skipped
    bias = rng.standard_normal(D).astype(np.float32)
    vz = vals.copy()
    vz[0, -1] = 0
    iz = np.where(idx < 0, 0, idx)
    ref = O.decode_rows(vz, iz, iw.astype(np.float32), 0.5, bias)
    dv, di = T(vals, cuda_device), T(idx, cuda_device)
    assert_recon_close(L.decode_int4(dv, di, T(O.pack_nibbles(iw), cuda_device), H, D, 0.5, T(bias, cuda_device)).cpu().numpy(), ref)
    assert_recon_close(L.decode_int8(dv, di, T(iw, cuda_device), H, D, 0.5, T(bias, cuda_device)).cpu().numpy(), ref)
    rows = rng.standard_normal((H, D)).astype(np.float32)
    ref = O.decode_rows(vz, iz, rows, 1.0, None)
    assert_recon_close(L.decode_rows_f32(dv, di, T(rows, cuda_device), H, D, 1.0, None).cpu().numpy(), ref)
    dense = L.densify(T(vz, cuda_device), T(iz, cuda_device), H).cpu().numpy()
    assert np.array_equal(dense, O.densify(vz, iz, H))
    assert np.array_equal(L.transpose(T(rows, cuda_device)).cpu().numpy(), rows.T)


def test_decode_linearity_full_size(cuda_device):
    """Size-independent property at the headline shape: decode(a*v1 + v2-rows) is linear in vals."""
    H, D, B, k = 32768, 512, 4096, 32
    g = torch.Generator(device=cuda_device).manual_seed(1)
    packed = torch.randint(0, 256, (H, D // 2), dtype=torch.uint8, device=cuda_device, generator=g)
    idx = torch.randint(0, H, (B, k), dtype=torch.int32, device=cuda_device, generator=g)
    v1 = torch.randn((B, k), device=cuda_device, generator=g)
    v2 = torch.randn((B, k), device=cuda_device, generator=g)
    r1 = L.decode_int4(v1, idx, packed, H, D, 0.5, None)
    r2 = L.decode_int4(v2, idx, packed, H, D, 0.5, None)
    r12 = L.decode_int4(2.0 * v1 + v2, idx, packed, H, D, 0.5, None)
    torch.testing.assert_close(r12, 2.0 * r1 + r2, rtol=1e-4, atol=1e-3)
    # checksum against the oracle on a few rows
    rows = [0, 1, 777, B - 1]
    ref = O.decode_rows(v1[rows].cpu().numpy(), idx[rows].cpu().numpy(),
                        O.unpack_nibbles(packed.cpu().numpy()).astype(np.float32), 0.5, None)
    assert_recon_close(r1[rows].cpu().numpy(), ref)


# ------------------------------------------------------------------------------------------
# encoder + top-k
# ------------------------------------------------------------------------------------------
def _enc_case(B, H, D, seed, bf16=True):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((B, D)).astype(np.float32)
    W = cases.xavier_uniform(rng, H, D)
    if bf16:
        x, W = cases.round_bf16(x), cases.round_bf16(W)
    b = (0.01 * rng.standard_normal(H)).astype(np.float32)
    return x, W, b


@pytest.mark.parametrize("B,H,D", [(128, 256, 64), (200, 1024, 512), (77, 1000, 72), (1, 300, 8)])
def test_tensor_core_gemm_vs_fp32(cuda_device, B, H, D):
    x, W, b = _enc_case(B, H, D, 3)
    z = L.encode_dense_tc(T(x, cuda_device), L.cast_bf16(T(W, cuda_device)), T(b, cuda_device)).cpu().numpy()
    np.testing.assert_allclose(z, O.encode_pre(x, W, b), rtol=1e-5, atol=1e-5)
    zr = L.encode_dense_tc(T(x, cuda_device), L.cast_bf16(T(W, cuda_device)), T(b, cuda_device), act=L.ACT_RELU).cpu().numpy()
    np.testing.assert_allclose(zr, np.maximum(O.encode_pre(x, W, b), 0), rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("B,H,D,k", [
    (32, 2048, 64, 4), (48, 4096, 512, 8), (300, 8192, 256, 32), (130, 32768, 512, 65),
    (1, 512, 512, 1), (129, 1000, 72, 33), (5, 300, 8, 150), (64, 4096, 512, 224), (17, 64, 64, 64)])
def test_fused_topk_bit_exact_indices(cuda_device, B, H, D, k):
    x, W, b = _enc_case(B, H, D, 100 + k)
    vals, idx, _ = L.encode_topk(T(x, cuda_device), L.cast_bf16(T(W, cuda_device)), None, T(b, cuda_device), k)
    assert_topk_matches(vals.cpu().numpy(), idx.cpu().numpy(), O.encode_pre(x, W, b), k)


def test_fused_topk_exact_mode_fp32_inputs(cuda_device):
    """Arbitrary fp32 operands: bf16 candidates + fp32 re-scoring must reproduce the fp32 oracle."""
    B, H, D, k = 256, 32768, 512, 32
    x, W, b = _enc_case(B, H, D, 5, bf16=False)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    vals, idx, flags = L.encode_topk(dx, L.cast_bf16(dW), dW, db, k, exact=True, want_flags=True)
    z = O.encode_pre(x, W, b)
    assert_topk_matches(vals.cpu().numpy(), idx.cpu().numpy(), z, k)
    assert int(flags.sum()) == 0                                  # every row certified
    # and k = 65 (reference default at H = 32768)
    vals, idx, flags = L.encode_topk(dx, L.cast_bf16(dW), dW, db, 65, exact=True, want_flags=True)
    assert_topk_matches(vals.cpu().numpy(), idx.cpu().numpy(), z, 65)
    assert int(flags.sum()) == 0


def test_relu_and_tie_rule(cuda_device):
    """ReLU floods the stream with equal zeros: survivors must follow (value desc, index asc)."""
    B, H, D, k = 64, 4096, 64, 48
    x, W, b = _enc_case(B, H, D, 9)
    b = b - 0.6                                                   # most pre-activations negative
    vals, idx, _ = L.encode_topk(T(x, cuda_device), L.cast_bf16(T(W, cuda_device)), None, T(b, cuda_device), k, act=L.ACT_RELU)
    zr = np.maximum(O.encode_pre(x, W, b), 0).astype(np.float32)
    rv, ri = O.topk_rows(zr, k)
    assert (rv == 0).any(), "case should contain ties at zero"
    assert_topk_matches(vals.cpu().numpy(), idx.cpu().numpy(), zr, k)
    zero_rows = (rv == 0).any(1)                                  # exact ties: lowest index first, bit exact
    assert np.array_equal(idx.cpu().numpy()[zero_rows][rv[zero_rows] == 0], ri[zero_rows][rv[zero_rows] == 0])
    z = np.zeros((3, 5000), dtype=np.float32)
    z[:, 2500] = 1
    _, i2 = L.topk_dense(T(z, cuda_device), 4)
    assert i2.cpu().numpy().tolist() == [[2500, 0, 1, 2]] * 3


def test_topk_dense_and_simt_encoder(cuda_device):
    for (B, H, D, k) in [(20, 1000, 72, 5), (33, 4096, 512, 65), (5, 300, 8, 224)]:
        x, W, b = _enc_case(B, H, D, 2, bf16=False)
        z = L.encode_dense(T(x, cuda_device), T(W, cuda_device), T(b, cuda_device))
        np.testing.assert_allclose(z.cpu().numpy(), O.encode_pre(x, W, b), rtol=1e-4, atol=1e-5)
        vals, idx = L.topk_dense(z, k)
        rv, ri = O.topk_rows(z.cpu().numpy(), k)
        assert np.array_equal(idx.cpu().numpy(), ri) and np.array_equal(vals.cpu().numpy(), rv)


def test_edge_cases(cuda_device):
    x, W, b = _enc_case(4, 512, 64, 11)
    dW = L.cast_bf16(T(W, cuda_device))
    v, i, _ = L.encode_topk(T(x[:0], cuda_device), dW, None, T(b, cuda_device), 4)    # empty batch
    assert v.shape == (0, 4) and i.shape == (0, 4)
    with pytest.raises(RuntimeError, match="out of range"):                            # k > H like torch.topk
        L.encode_topk(T(x, cuda_device), dW, None, T(b, cuda_device), 513)
    with pytest.raises(L.QsaeError):
        L.encode_topk(T(x, cuda_device), dW, None, T(b, cuda_device), 0)
    with pytest.raises(L.QsaeError):                                                   # D not a multiple of 8
        L.encode_topk(torch.zeros(4, 12, device=cuda_device), torch.zeros(16, 12, device=cuda_device).bfloat16(),
                      None, torch.zeros(16, device=cuda_device), 2)


def test_full_size_properties(cuda_device):
    """Headline shape (B=4096, H=32768, D=512): oracle on a row sample + self-consistency."""
    B, H, D, k = 4096, 32768, 512, 32
    x, W, b = _enc_case(B, H, D, 21)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    vals, idx, _ = L.encode_topk(dx, L.cast_bf16(dW), None, db, k)
    rows = np.r_[0:16, 2040:2056, B - 16:B]
    assert_topk_matches(vals.cpu().numpy()[rows], idx.cpu().numpy()[rows], O.encode_pre(x[rows], W, b), k)
    v = vals.cpu().numpy()
    i = idx.cpu().numpy()
    assert np.all(np.diff(v, axis=1) <= 0)                                             # sorted descending
    assert all(len(set(r)) == k for r in i[::97])                                      # distinct indices
    assert i.min() >= 0 and i.max() < H
    # values agree with an independent CUDA-core fp32 evaluation of the same (row, index) pairs
    z = L.encode_dense(dx, dW, db, rows=T(np.arange(0, B, 64, dtype=np.int32), cuda_device)).cpu().numpy()
    sel = np.take_along_axis(z, i[::64].astype(np.int64), axis=1)
    assert_vals_close(v[::64], sel)
    assert_vals_close(v[::64, 0], z.max(1))                                            # row maximum is first
    assert np.all(np.sort(z, axis=1)[:, -k] <= v[::64, -1] + 1e-5)                     # nothing larger was left out
    # idempotence: densify -> dense top-k returns the same sparse form
    d = L.densify(vals[:64], idx[:64], H)
    v2, i2 = L.topk_dense(d, k)
    assert torch.equal(i2, idx[:64]) and torch.equal(v2, vals[:64])


def test_bench_size_properties(cuda_device):
    """The bench workload itself (B = 65536 rows, H = 32768, D = 512, k = 32, qsae_bsae_forward): oracle on a row
    sample, size-independent properties on everything."""
    B, H, D, k = 65536, 32768, 512, 32
    g = torch.Generator(device=cuda_device).manual_seed(11)
    x = torch.randn((B, D), device=cuda_device, generator=g).bfloat16().float()
    W = ((torch.rand((H, D), device=cuda_device, generator=g) * 2 - 1) * (6.0 / (H + D)) ** 0.5).bfloat16().float()
    b = (0.01 * torch.randn(H, device=cuda_device, generator=g)).float()
    packed = torch.randint(0, 256, (H, D // 2), dtype=torch.uint8, device=cuda_device, generator=g)
    bd = torch.randn(D, device=cuda_device, generator=g)
    wb = L.cast_bf16(W)
    vals, idx, _, recon = L.bsae_forward(x, wb, None, b, k, packed, 4, 0.5, bd, sample=L.prepare_sample(wb, b))
    assert bool((vals[:, :-1] >= vals[:, 1:]).all())                                   # sorted descending
    assert int(idx.min()) >= 0 and int(idx.max()) < H
    srt = torch.sort(idx, dim=1).values
    assert bool((srt[:, 1:] != srt[:, :-1]).all())                                     # distinct indices in every row
    rows = np.r_[0:24, 30000:30024, B - 24:B]
    xn, Wn, bn = x[rows].cpu().numpy(), W.cpu().numpy(), b.cpu().numpy()
    assert_topk_matches(vals[rows].cpu().numpy(), idx[rows].cpu().numpy(), O.encode_pre(xn, Wn, bn), k)
    ref = O.decode_rows(vals[rows].cpu().numpy(), idx[rows].cpu().numpy(),
                        O.unpack_nibbles(packed.cpu().numpy()).astype(np.float32), 0.5, bd.cpu().numpy())
    assert_recon_close(recon[rows].cpu().numpy(), ref)
    # every 256th row against an independent CUDA-core fp32 evaluation: nothing larger than the k-th value was left out
    sel = torch.arange(0, B, 256, device=cuda_device, dtype=torch.int32)
    z = L.encode_dense(x, W, b, rows=sel)
    kth = torch.sort(z, dim=1, descending=True).values[:, k - 1]
    assert bool((kth <= vals[::256, -1] + 1e-5).all()) and bool((vals[::256, 0] - z.max(1).values).abs().max() <= 1e-5)


def test_qsae_full_size_properties(cuda_device):
    """q_sae at the config-4 shape (512 -> 32768, n_bits = 4, bias -0.543, B = 4096): exact level counts against the
    oracle's activity over the whole batch, reconstructions against the oracle on a row sample, level structure."""
    cfg = dict(D=512, H=32768, n_bits=4, abs_range=4.0, B=4096, enc_bias=-0.543, bf16=False, allow_bias=True, seed=92)
    inp = cases.qsae_inputs(cfg)
    m = Q.QuantizedMatryoshkaSAE(cfg["D"], cfg["H"], 32, cfg["abs_range"], cfg["n_bits"], True)
    m.load_state_dict({"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
                       "decoder.weight": torch.from_numpy(inp["W"]), "decoder.weight_mirror": torch.from_numpy(inp["Wm"]),
                       "decoder.bias": torch.from_numpy(inp["bd"])}, strict=True)
    m.to(cuda_device).eval()
    with torch.no_grad():
        r = m.forward_active(T(inp["x"], cuda_device))
    assert m.last_path == "sparse"
    z = O.encode_pre(inp["x"], inp["We"], inp["be"])
    act = O.sigmoid_f32(z) > np.float32(0.5)
    edges = np.cumsum([0] + O.matryoshka_level_sizes(cfg["H"], cfg["n_bits"]))
    assert r["level_counts"].cpu().numpy().tolist() == [int(act[:, a:b].sum()) for a, b in zip(edges[:-1], edges[1:])]
    assert np.array_equal(r["active_cnt"].cpu().numpy(), act.sum(1))                   # per-row activity, exact
    ai = r["active_idx"].cpu().numpy()
    for row in (0, 1777, 4095):
        assert sorted(ai[row][ai[row] >= 0].tolist()) == np.nonzero(act[row])[0].tolist()
    rows = np.r_[0:32, 4064:4096]
    _, res, _ = O.qsae_forward(inp["x"][rows], inp["We"], inp["be"], inp["W"], inp["Wm"], inp["bd"], n_bits=cfg["n_bits"],
                               abs_range=cfg["abs_range"], allow_bias=True)
    for i in range(cfg["n_bits"]):
        assert_recon_close(r["reconstruction_levels"][i][rows].cpu().numpy(), res[i])
    # a level only adds vectors of norm 2^(n - l - 2) * quant_step per active latent (Appendix A.4): rows without an
    # active latent in level l have identical consecutive outputs
    lv = [t.cpu().numpy() for t in r["reconstruction_levels"]]
    for l in range(1, cfg["n_bits"]):
        quiet = ~act[:, edges[l]:edges[l + 1]].any(1)
        assert np.array_equal(lv[l][quiet], lv[l - 1][quiet])


# ------------------------------------------------------------------------------------------
# modules vs the reference's own outputs
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(cases.BSAE_CASES))
def test_bsae_module_matches_reference(cuda_device, golden_dir, name):
    cfg = cases.BSAE_CASES[name]
    g = np.load(golden_dir / f"{name}.npz")
    inp = cases.bsae_inputs(cfg)
    m = Q.BinarySAE(cfg["D"], cfg["H"], cfg["gamma"], cfg["n_bits"])
    m.load_state_dict({"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
                       "decoder.weight": torch.from_numpy(inp["logits"]), "decoder.bias": torch.from_numpy(inp["bd"])},
                      strict=True)
    m.to(cuda_device).eval()
    with torch.no_grad():
        latent, recon, pol = m(T(inp["x"], cuda_device))
    assert latent.shape == (cfg["B"], cfg["H"]) and recon.shape == (cfg["B"], cfg["D"]) and pol.dim() == 0
    vals, idx = cases.sparse_from_dense(latent.cpu().numpy())
    assert np.array_equal(idx, g["latent_idx"])                   # bit-exact top-k index sets and order
    assert_vals_close(vals, g["latent_vals"])
    assert_recon_close(recon.cpu().numpy(), g["recon"])
    assert float(pol) == pytest.approx(float(g["polarize"]), rel=1e-5, abs=1e-9)
    assert m.decoder.resolved_mode() == ("int" if cfg["polar"] else "soft")
    assert int(m.last_flags.sum()) == 0
    assert cases.int_weights_match(m.decoder.quantized_int_weights().cpu().numpy().astype(np.int8), g)
    # sparse return form carries the same information
    m.return_dense = False
    with torch.no_grad():
        sp, recon2, _ = m(T(inp["x"], cuda_device))
    assert torch.equal(sp.to_dense(), latent) and torch.equal(recon2, recon)
    # the standalone decoder accepts the dense latent the reference passes (sae/binary.py:101)
    with torch.no_grad():
        recon3, _ = m.decoder(latent, None)
    assert_recon_close(recon3.cpu().numpy(), g["recon"])
    # dense encode() agrees with the oracle pre-activations
    with torch.no_grad():
        z = m.encode(T(inp["x"], cuda_device)).cpu().numpy()
    np.testing.assert_allclose(z, O.encode_pre(inp["x"], inp["We"], inp["be"]), rtol=1e-4, atol=1e-5)


def test_bsae_forced_int_mode_is_the_hard_dictionary(cuda_device):
    cfg = cases.BSAE_CASES["bsae_soft_d64_h2048"]
    inp = cases.bsae_inputs(cfg)
    m = Q.BinarySAE(cfg["D"], cfg["H"], cfg["gamma"], cfg["n_bits"]).to(cuda_device)
    with torch.no_grad():
        m.encoder[0].weight.copy_(T(inp["We"], cuda_device)); m.encoder[0].bias.copy_(T(inp["be"], cuda_device))
        m.decoder.weight.copy_(T(inp["logits"], cuda_device)); m.decoder.bias.copy_(T(inp["bd"], cuda_device))
    m.decoder.decode_mode = "int"
    with torch.no_grad():
        _, recon, _ = m(T(inp["x"], cuda_device))
    k = O.bsae_k(cfg["H"])
    _, _, ref, _ = O.bsae_forward(inp["x"], inp["We"], inp["be"], inp["logits"], inp["bd"],
                                  n_bits=cfg["n_bits"], gamma=cfg["gamma"], k=k, mode="hard")
    assert_recon_close(recon.cpu().numpy(), ref)
    # cache invalidation: changing the logits in place must change the packed dictionary
    with torch.no_grad():
        m.decoder.weight.neg_()
        _, recon_neg, _ = m(T(inp["x"], cuda_device))
    _, _, ref_neg, _ = O.bsae_forward(inp["x"], inp["We"], inp["be"], -inp["logits"], inp["bd"],
                                      n_bits=cfg["n_bits"], gamma=cfg["gamma"], k=k, mode="hard")
    assert_recon_close(recon_neg.cpu().numpy(), ref_neg)


@pytest.mark.parametrize("name", list(cases.BASELINE_CASES))
def test_baseline_module_matches_reference(cuda_device, golden_dir, name):
    cfg = cases.BASELINE_CASES[name]
    g = np.load(golden_dir / f"{name}.npz")
    inp = cases.baseline_inputs(cfg)
    m = Q.BaselineSparseAutoencoder(cfg["D"], cfg["H"])
    m.load_state_dict({"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
                       "decoder.weight": torch.from_numpy(inp["Wd"]), "decoder.bias": torch.from_numpy(inp["bd"])},
                      strict=True)
    m.to(cuda_device).eval()
    with torch.no_grad():
        h, recon = m(T(inp["x"], cuda_device))
    vals, idx = cases.sparse_from_dense(h.cpu().numpy())
    assert np.array_equal(idx, g["latent_idx"])
    assert_vals_close(vals, g["latent_vals"])
    assert_recon_close(recon.cpu().numpy(), g["recon"])
    with torch.no_grad():
        z = T(O.encode_pre(inp["x"], inp["We"], inp["be"]), cuda_device)
        assert torch.equal(m.apply_topk_activation(z) != 0, h != 0)


def test_host_pipeline_entry(cuda_device):
    """qsae_bsae_forward_host: host buffers in, host buffers out, chunked and overlapped."""
    import ctypes as C

    cfg = cases.BSAE_CASES["bsae_polar_d512_h4096"]
    inp = cases.bsae_inputs(cfg)
    k = O.bsae_k(cfg["H"])
    lib = L.load()
    dW, db = T(inp["We"], cuda_device), T(inp["be"], cuda_device)
    dl, dbd = T(inp["logits"], cuda_device), T(inp["bd"], cuda_device)
    plan = C.c_void_p()
    L.check(lib.qsae_bsae_plan_create(dW.data_ptr(), db.data_ptr(), dl.data_ptr(), dbd.data_ptr(), cfg["H"], cfg["D"],
                                      cfg["n_bits"], cfg["gamma"], k, 20, C.byref(plan)))
    try:
        B = cfg["B"]
        x = torch.from_numpy(inp["x"]).pin_memory()
        vals = torch.empty((B, k), dtype=torch.float32).pin_memory()
        idx = torch.empty((B, k), dtype=torch.int32).pin_memory()
        recon = torch.empty((B, cfg["D"]), dtype=torch.float32).pin_memory()
        L.check(lib.qsae_bsae_forward_host(plan, x.data_ptr(), B, vals.data_ptr(), idx.data_ptr(), recon.data_ptr()))
    finally:
        lib.qsae_bsae_plan_destroy(plan)
    rv, ri, rr, _ = O.bsae_forward(inp["x"], inp["We"], inp["be"], inp["logits"], inp["bd"],
                                   n_bits=cfg["n_bits"], gamma=cfg["gamma"], k=k, mode="hard")
    assert np.array_equal(idx.numpy(), ri)
    assert_vals_close(vals.numpy(), rv)
    assert_recon_close(recon.numpy(), rr)


def test_host_pipeline_submit_wait_and_bf16_io(cuda_device):
    """qsae_bsae_submit_host / qsae_bsae_wait_host: several batches in flight, each bit-identical to the synchronous
    call; bf16 host input (exact for bf16-representable x) and bf16 / omitted reconstruction output."""
    import ctypes as C

    cfg = cases.BSAE_CASES["bsae_polar_d512_h4096"]
    inp = cases.bsae_inputs(cfg)
    k = O.bsae_k(cfg["H"])
    lib = L.load()
    dW, db = T(inp["We"], cuda_device), T(inp["be"], cuda_device)
    dl, dbd = T(inp["logits"], cuda_device), T(inp["bd"], cuda_device)
    B, D = cfg["B"], cfg["D"]
    plan = C.c_void_p()
    L.check(lib.qsae_bsae_plan_create(dW.data_ptr(), db.data_ptr(), dl.data_ptr(), dbd.data_ptr(), cfg["H"], D,
                                      cfg["n_bits"], cfg["gamma"], k, 48, C.byref(plan)))
    rng = np.random.default_rng(3)
    xs = [cases.round_bf16(inp["x"] * np.float32(1.0 + 0.25 * j) + rng.standard_normal(inp["x"].shape).astype(np.float32) * (j > 0))
          for j in range(5)]
    try:
        hx = [torch.from_numpy(x).pin_memory() for x in xs]
        outs = [(torch.empty((B, k), dtype=torch.float32).pin_memory(), torch.empty((B, k), dtype=torch.int32).pin_memory(),
                 torch.empty((B, D), dtype=torch.float32).pin_memory()) for _ in xs]
        ref = [(torch.empty((B, k), dtype=torch.float32).pin_memory(), torch.empty((B, k), dtype=torch.int32).pin_memory(),
                torch.empty((B, D), dtype=torch.float32).pin_memory()) for _ in xs]
        for x, (v, i, r) in zip(hx, ref):
            L.check(lib.qsae_bsae_forward_host(plan, x.data_ptr(), B, v.data_ptr(), i.data_ptr(), r.data_ptr()))
        tickets = []
        for x, (v, i, r) in zip(hx, outs):
            t = C.c_int(-1)
            L.check(lib.qsae_bsae_submit_host(plan, x.data_ptr(), B, v.data_ptr(), i.data_ptr(), r.data_ptr(), C.byref(t)))
            tickets.append(t.value)
        assert len(set(tickets)) == len(tickets)
        for t in tickets:
            L.check(lib.qsae_bsae_wait_host(plan, t))
        with pytest.raises(L.QsaeError):
            L.check(lib.qsae_bsae_wait_host(plan, tickets[0]))          # already waited for
        for (v, i, r), (rv, ri, rr) in zip(outs, ref):
            assert torch.equal(i, ri) and torch.equal(v, rv) and torch.equal(r, rr)
        rv, ri, rr, _ = O.bsae_forward(xs[3], inp["We"], inp["be"], inp["logits"], inp["bd"], n_bits=cfg["n_bits"],
                                       gamma=cfg["gamma"], k=k, mode="hard")
        assert np.array_equal(outs[3][1].numpy(), ri)
        assert_recon_close(outs[3][2].numpy(), rr)
        # bf16 host input, bf16 reconstruction out
        L.check(lib.qsae_bsae_plan_set_io(plan, 1, 1))
        xb = torch.from_numpy(xs[3]).bfloat16().pin_memory()
        v2 = torch.empty((B, k), dtype=torch.float32).pin_memory()
        i2 = torch.empty((B, k), dtype=torch.int32).pin_memory()
        r2 = torch.empty((B, D), dtype=torch.bfloat16).pin_memory()
        t = C.c_int(-1)
        L.check(lib.qsae_bsae_submit_host(plan, xb.data_ptr(), B, v2.data_ptr(), i2.data_ptr(), r2.data_ptr(), C.byref(t)))
        L.check(lib.qsae_bsae_wait_host(plan, t.value))
        assert torch.equal(i2, outs[3][1]) and torch.equal(v2, outs[3][0])
        assert torch.equal(r2, outs[3][2].bfloat16())
        # no reconstruction copied out
        L.check(lib.qsae_bsae_plan_set_io(plan, 1, 2))
        v3 = torch.zeros((B, k), dtype=torch.float32).pin_memory()
        i3 = torch.zeros((B, k), dtype=torch.int32).pin_memory()
        L.check(lib.qsae_bsae_forward_host(plan, xb.data_ptr(), B, v3.data_ptr(), i3.data_ptr(), None))
        assert torch.equal(i3, i2) and torch.equal(v3, v2)
    finally:
        lib.qsae_bsae_plan_destroy(plan)


def test_data_edits_need_invalidate(cuda_device):
    """In-place edits through `.data` (the reference's STEWeights.init_mask / update_mask do `weight.data *= mask`)
    bump no version counter: the prepared dictionary stays until invalidate() -- the documented contract."""
    D, H, B = 64, 2048, 32
    torch.manual_seed(1)
    with torch.device(cuda_device):
        m = Q.TernarySparseAutoencoder(D, H)
    with torch.no_grad():
        m.decoder.weight.copy_(0.6 * torch.randn(D, H, device=cuda_device))
    m.eval()
    x = torch.randn(B, D, device=cuda_device)
    with torch.no_grad():
        _, r0 = m(x)
        m.decoder.weight.data.mul_(0.0)            # every ternary weight becomes 0
        _, r1 = m(x)
        assert torch.equal(r0, r1)                 # stale prepared copy (documented)
        m.invalidate()
        _, r2 = m(x)
    assert float(r2.abs().max()) == 0.0


def test_native_library_was_used(cuda_device):
    assert L._lib is not None and L.launch_count() > 0


# ------------------------------------------------------------------------------------------
# prior threshold (sampled-latent pre-pass), count verification and the rescue kernel
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,exact", [(32, False), (65, False), (32, True), (65, True)])
def test_prior_threshold_path_matches_oracle(cuda_device, k, exact):
    B, H, D = 384, 32768, 512
    x, W, b = _enc_case(B, H, D, 40 + k, bf16=not exact)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    sample = L.prepare_sample(wb, db)
    assert sample is not None and sample[0].shape == (L.default_sample_rows(H), D) and L.default_sample_rows(H) == 2048
    vals, idx, flags = L.encode_topk(dx, wb, dW if exact else None, db, k, exact=exact, want_flags=True, sample=sample)
    assert_topk_matches(vals.cpu().numpy(), idx.cpu().numpy(), O.encode_pre(x, W, b), k)
    assert int((flags != 0).sum()) == 0
    # identical to the path without the prior
    v0, i0, _ = L.encode_topk(dx, wb, dW if exact else None, db, k, exact=exact)
    assert torch.equal(i0, idx) and torch.equal(v0, vals)


@pytest.mark.parametrize("k,exact", [(65, False), (65, True), (100, False)])
def test_prior_ranks_above_16_on_the_separate_prior_kernels(cuda_device, k, exact):
    """B = 9600 rows is past the single-launch prior kernel (2 x 75 row blocks > 148 SMs): cast, sample pre-pass (top-2 per
    column class) and the sorting prior kernel run as separate launches. With the H / 16 sample the prior ranks are
    18 (k_sel = 65), 20 (k_sel = 81, exact) and 23 (k_sel = 100): above the old limit of 16. Same result as without the
    sample, and the oracle's indices on a strided subset of the rows."""
    B, H, D = 9600, 32768, 512
    x, W, b = _enc_case(B, H, D, 80 + k, bf16=not exact)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    sample = L.prepare_sample(wb, db)
    vals, idx, flags = L.encode_topk(dx, wb, dW if exact else None, db, k, exact=exact, want_flags=True, sample=sample)
    assert int((flags != 0).sum()) == 0
    v0, i0, _ = L.encode_topk(dx, wb, dW if exact else None, db, k, exact=exact)
    assert torch.equal(i0, idx) and torch.equal(v0, vals)
    rows = np.arange(0, B, 25)
    assert_topk_matches(vals[rows].cpu().numpy(), idx[rows].cpu().numpy(), O.encode_pre(x[rows], W, b), k)


@pytest.mark.parametrize("k,exact", [(32, False), (65, False), (32, True)])
def test_heavy_tailed_activations(cuda_device, k, exact):
    """SURVEY 8d config 1, heavy-tail variant: 8 of the 512 input dimensions scaled by 20 (outlier residual-stream
    channels). The pre-activations of a row are then dominated by a few encoder columns -- a much heavier tail
    than the Gaussian case; the sampled prior is distribution-free and the result must stay exact."""
    B, H, D = 320, 32768, 512
    x, W, b = _enc_case(B, H, D, 60 + k, bf16=not exact)
    x[:, np.random.default_rng(1).choice(D, 8, replace=False)] *= 20.0
    if not exact:
        x = cases.round_bf16(x)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    vals, idx, flags = L.encode_topk(dx, wb, dW if exact else None, db, k, exact=exact, want_flags=True,
                                     sample=L.prepare_sample(wb, db))
    assert_topk_matches(vals.cpu().numpy(), idx.cpu().numpy(), O.encode_pre(x, W, b), k)
    assert int((flags != 0).sum()) == 0


def test_prior_failure_is_rescued_exactly(cuda_device):
    """Force the prior to fail: the sampled rows carry a huge bias that the real rows do not have,
    so every row's prior threshold is far above its true top-k and the count check must route
    all rows through the rescue kernel -- which has to reproduce the exact result."""
    B, H, D, k = 70, 16384, 256, 32
    x, W, b = _enc_case(B, H, D, 77)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    ws, bs = L.prepare_sample(wb, db, 512)
    for exact in (False, True):
        vals, idx, flags = L.encode_topk(dx, wb, dW if exact else None, db, k, exact=exact, want_flags=True,
                                         sample=(ws, bs + 100.0))
        assert_topk_matches(vals.cpu().numpy(), idx.cpu().numpy(), O.encode_pre(x, W, b), k)
        assert int((flags != 0).sum()) == 0          # rescued rows are exact by construction


@pytest.mark.parametrize("B,D,n_sample,m,act", [(300, 512, 1024, 10, 0), (4096, 512, 1024, 10, 0), (130, 256, 512, 7, 0),
                                                (6000, 512, 1024, 12, 0), (200, 512, 2048, 9, 1), (77, 512, 1000, 5, 0),
                                                (4096, 512, 2048, 13, 0), (1000, 512, 2048, 20, 0), (512, 512, 8192, 32, 0)])
def test_prior_prep_kernel_vs_numpy(cuda_device, B, D, n_sample, m, act):
    """The single-launch cast + sample pre-pass + prior: x_bf16 must be the round-to-nearest bf16 of x (bit exact: it is
    the sweep's operand) and prior[b] the m-th largest per-class maximum of row b's sampled pre-activations, classes =
    (CTA of the cluster, column half of the 256-wide tile, column mod 32). Checks the hand-written 128-byte swizzle of
    the x operand, the cluster exchange and the bisection."""
    rng = np.random.default_rng(B + m)
    x = rng.standard_normal((B, D)).astype(np.float32)
    ws = cases.round_bf16(cases.xavier_uniform(rng, n_sample, D))
    bs = (0.05 * rng.standard_normal(n_sample)).astype(np.float32)
    dws = T(ws, cuda_device).bfloat16()
    xb, prior, ns = L.prior_prep(T(x, cuda_device), (dws, T(bs, cuda_device)), m, act)
    assert ns in (2, 4)
    xr = cases.round_bf16(x)
    assert np.array_equal(xb.float().cpu().numpy(), xr)
    z = xr.astype(np.float64) @ ws.astype(np.float64).T + bs
    if act:
        z = np.maximum(z, 0.0)
    n_tiles = (n_sample + 255) // 256
    tiles_per_cta = (n_tiles + ns - 1) // ns
    col = np.arange(n_sample)
    cls = ((col // 256) // tiles_per_cta) * 64 + ((col % 256) // 128) * 32 + col % 32
    cmax = np.full((B, ns * 64), -np.inf)
    for c in range(ns * 64):
        sel = cls == c
        if sel.any():
            cmax[:, c] = z[:, sel].max(1)
    ref = -np.sort(-cmax, axis=1)[:, m - 1]
    got = prior.cpu().numpy().astype(np.float64)
    assert np.all(np.abs(got - ref) <= 2e-6 * np.maximum(1.0, np.abs(ref))), float(np.abs(got - ref).max())


@pytest.mark.parametrize("B,H,D,k,exact", [(4096, 32768, 512, 32, False), (1000, 32768, 512, 65, False), (2048, 16384, 512, 32, True),
                                           (333, 32768, 512, 32, False), (700, 16384, 256, 100, False)])
def test_range_schedule_is_bit_identical_to_the_grid_schedule(cuda_device, tuning, B, H, D, k, exact):
    """Small batches sweep with one CTA per SM over contiguous tile ranges (pieces of up to three row blocks per CTA,
    x tile reloaded in between, per-piece survivor lists); the (split, row block) grid must give the same bits, and
    both must match the oracle."""
    x, W, b = _enc_case(B, H, D, 31 + B, bf16=not exact)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    sample = L.prepare_sample(wb, db)
    packed = torch.randint(0, 256, (H, D // 2), dtype=torch.uint8, device=cuda_device)
    bd = torch.randn(D, device=cuda_device)
    outs = []
    for flag in ("1", "0"):
        tuning("QSAE_ENCODE_RANGE", flag)
        outs.append(L.bsae_forward(dx, wb, dW if exact else None, db, k, packed, 4, 0.5, bd, exact=exact, want_flags=True,
                                   sample=sample))
    for a, c in zip(outs[0], outs[1]):
        assert torch.equal(a, c)
    rows = np.random.default_rng(0).choice(B, min(B, 256), replace=False)
    z = O.encode_pre(x[rows], W, b)
    assert_topk_matches(outs[0][0].cpu().numpy()[rows], outs[0][1].cpu().numpy()[rows], z, k)
    assert int((outs[0][2] != 0).sum()) == 0


@pytest.mark.parametrize("B,H,D,k,exact", [(4096, 32768, 512, 32, False), (1536, 32768, 512, 65, True), (2048, 16384, 512, 32, False)])
def test_pair_range_schedule_is_bit_identical_to_the_single_cta_range_schedule(cuda_device, tuning, B, H, D, k, exact):
    """Batches of whole row-block pairs run the range schedule over cta_group::2 pairs (units = (pair of row blocks, tile),
    74 pairs on 148 SMs, x tiles of both CTAs reloaded between pieces): same bits as the single-CTA range schedule."""
    x, W, b = _enc_case(B, H, D, 77 + B, bf16=not exact)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    sample = L.prepare_sample(wb, db)
    packed = torch.randint(0, 256, (H, D // 2), dtype=torch.uint8, device=cuda_device)
    bd = torch.randn(D, device=cuda_device)
    outs = []
    for flag in ("1", "0"):
        tuning("QSAE_ENCODE_RANGE_PAIR", flag)
        outs.append(L.bsae_forward(dx, wb, dW if exact else None, db, k, packed, 4, 0.5, bd, exact=exact, want_flags=True,
                                   sample=sample))
    for a, c in zip(outs[0], outs[1]):
        assert torch.equal(a, c)
    rows = np.random.default_rng(1).choice(B, 128, replace=False)
    z = O.encode_pre(x[rows], W, b)
    assert_topk_matches(outs[0][0].cpu().numpy()[rows], outs[0][1].cpu().numpy()[rows], z, k)


def test_prior_prep_path_is_bit_identical_to_the_separate_kernels(cuda_device, tuning):
    B, H, D, k = 700, 32768, 512, 32
    x, W, b = _enc_case(B, H, D, 4242)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    sample = L.prepare_sample(wb, db)
    packed = torch.randint(0, 256, (H, D // 2), dtype=torch.uint8, device=cuda_device)
    bd = torch.randn(D, device=cuda_device)
    outs = []
    for flag in ("1", "0"):
        tuning("QSAE_PRIOR_PREP", flag)
        outs.append(L.bsae_forward(dx, wb, None, db, k, packed, 4, 0.5, bd, sample=sample))
    for a, c in zip(outs[0], outs[1]):
        if a is not None:
            assert torch.equal(a, c)
    assert_topk_matches(outs[0][0].cpu().numpy(), outs[0][1].cpu().numpy(), O.encode_pre(x, W, b), k)


@pytest.mark.parametrize("k,exact,shift", [(32, False, 0.12), (65, False, 0.2), (32, True, 0.12), (100, False, 0.3)])
def test_loose_prior_takes_the_two_pass_merge(cuda_device, k, exact, shift):
    """A prior that is too LOW (sampled rows carry a negative bias): every row keeps far more than the 512 survivors
    the merge warp holds in registers, so the whole batch goes through the in-warp two-pass prefilter (round 1: a
    second kernel tier). The result must not depend on the prior at all."""
    B, H, D = 300, 32768, 512
    x, W, b = _enc_case(B, H, D, 900 + k, bf16=not exact)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    ws, bs = L.prepare_sample(wb, db)
    v0, i0, _ = L.encode_topk(dx, wb, dW if exact else None, db, k, exact=exact, sample=(ws, bs))
    vals, idx, flags = L.encode_topk(dx, wb, dW if exact else None, db, k, exact=exact, want_flags=True,
                                     sample=(ws, bs - shift))
    assert_topk_matches(vals.cpu().numpy(), idx.cpu().numpy(), O.encode_pre(x, W, b), k)
    assert int((flags != 0).sum()) == 0
    assert torch.equal(i0, idx) and torch.equal(v0, vals)
    # and the fused decode of the same rows
    packed = torch.randint(0, 256, (H, D // 2), dtype=torch.uint8, device=cuda_device)
    bd = torch.randn(D, device=cuda_device)
    v1, i1, _, r1 = L.bsae_forward(dx, wb, dW if exact else None, db, k, packed, 4, 0.5, bd, exact=exact,
                                   sample=(ws, bs - shift))
    assert torch.equal(i1, idx) and torch.equal(v1, vals)
    assert torch.equal(r1, L.decode_int4(vals, idx, packed, H, D, 0.5, bd))


def test_prior_path_relu_flood_goes_through_the_tail_kernel(cuda_device):
    """ReLU with almost every pre-activation negative: the prior is 0, every list fills with equal zeros, the warp
    merge cannot separate them (all tie with the k-th value) and hands the rows to the block-per-row select of the
    tail kernel, which must apply the (value desc, index asc) rule exactly -- and decode the rows when fused."""
    B, H, D, k = 150, 16384, 512, 32
    x, W, b = _enc_case(B, H, D, 321)
    b = (b - 5.0).astype(np.float32)
    hot = np.random.default_rng(5).choice(H, 20, replace=False)
    b[hot] += 10.0
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    sample = L.prepare_sample(wb, db)
    vals, idx, _ = L.encode_topk(dx, wb, None, db, k, act=L.ACT_RELU, sample=sample)
    zr = np.maximum(O.encode_pre(x, W, b), 0).astype(np.float32)
    rv, ri = O.topk_rows(zr, k)
    assert (rv == 0).any(1).all(), "every row should end in a run of zeros"
    assert np.array_equal(idx.cpu().numpy(), ri)
    assert_vals_close(vals.cpu().numpy(), rv)


def test_class_bound_exact_mode_rescues_uncertified_rows(cuda_device):
    """H < 8192 has no sampled prior (class-bound sweep + block merge). Near-tied fp32 inputs that are not
    bf16-representable can leave a row uncertified; round 1 returned such rows flagged with their bf16-chosen
    candidates, now they are recomputed exactly: flags must be 0 and the indices exact."""
    B, H, D, k = 96, 4096, 512, 32
    rng = np.random.default_rng(77)
    x = rng.standard_normal((B, D)).astype(np.float32)
    W = cases.xavier_uniform(rng, H, D)
    # clusters of nearly identical dictionary rows: their scores differ by ~1e-6 relative, far inside the bf16 band
    base = rng.choice(H, 64, replace=False)
    for j in base:
        for t in range(1, 24):
            W[(j + t * 37) % H] = W[j] * np.float32(1.0 + 3e-7 * t)
    b = np.zeros(H, dtype=np.float32)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    vals, idx, flags = L.encode_topk(dx, L.cast_bf16(dW), dW, db, k, exact=True, want_flags=True)
    assert int((flags != 0).sum()) == 0
    z = O.encode_pre(x, W, b)
    rv, _ = O.topk_rows(z, k)
    gi = idx.cpu().numpy().astype(np.int64)
    assert all(len(set(r.tolist())) == k for r in gi)
    got = np.take_along_axis(z, gi, axis=1)           # the oracle's values at the selected columns, in our order
    assert np.all(np.abs(got - rv) <= 2e-6 * np.maximum(1.0, np.abs(rv))), "selection differs beyond the planted near-ties"
    assert_vals_close(vals.cpu().numpy(), got)


@pytest.mark.parametrize("B,H,D,k,n_bits,exact", [
    (1000, 32768, 512, 32, 4, False), (700, 32768, 512, 65, 4, False), (300, 32768, 512, 32, 4, True),
    (513, 16384, 512, 200, 4, False),      # rows with more survivors than the merge warp holds (two-pass prefilter)
    (200, 16384, 256, 32, 4, False),
    (150, 8192, 512, 16, 8, False),        # int8 dictionary
    (90, 2048, 512, 8, 4, False),          # no sampled prior
])
def test_bsae_forward_entry_is_bit_identical_to_the_two_calls(cuda_device, B, H, D, k, n_bits, exact):
    """qsae_bsae_forward (one call) vs qsae_encode_topk + qsae_decode_int4/int8."""
    x, W, b = _enc_case(B, H, D, 500 + k, bf16=not exact)
    rng = np.random.default_rng(k)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    sample = L.prepare_sample(wb, db)
    bd = T(rng.standard_normal(D).astype(np.float32), cuda_device)
    if n_bits <= 4:
        packed = torch.randint(0, 256, (H, D // 2), dtype=torch.uint8, device=cuda_device)
        dec = L.decode_int4
    else:
        packed = torch.randint(-128, 128, (H, D), dtype=torch.int8, device=cuda_device)
        dec = L.decode_int8
    v0, i0, f0 = L.encode_topk(dx, wb, dW if exact else None, db, k, exact=exact, want_flags=True, sample=sample)
    r0 = dec(v0, i0, packed, H, D, 0.5, bd)
    v1, i1, f1, r1 = L.bsae_forward(dx, wb, dW if exact else None, db, k, packed, n_bits, 0.5, bd, exact=exact,
                                    want_flags=True, sample=sample)
    assert torch.equal(i0, i1) and torch.equal(v0, v1) and torch.equal(f0, f1)
    assert torch.equal(r0, r1)
    if sample is not None:    # a failed prior sends every row through the rescue kernel + listed-rows decode
        ws, bs = sample
        v2, i2, _, r2 = L.bsae_forward(dx, wb, dW if exact else None, db, k, packed, n_bits, 0.5, bd, exact=exact,
                                       sample=(ws, bs + 100.0))
        assert_topk_matches(v2.cpu().numpy(), i2.cpu().numpy(), O.encode_pre(x, W, b), k)
        assert torch.equal(dec(v2, i2, packed, H, D, 0.5, bd), r2)


# ------------------------------------------------------------------------------------------
# k > QSAE_MAX_K: block-level radix select (reference default k = int(0.002 H) = 2097 at H = 2^20)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,H,D,k,exact", [
    (40, 16384, 256, 300, False),     # prior path, m ~ 27
    (33, 65536, 128, 2097, False),    # prior path at the reference-default k of a 2^20 dictionary
    (260, 32768, 512, 262, False),    # 2097 / 8 shards
    (24, 32768, 512, 300, True),      # arbitrary fp32 operands: fp32 re-scoring of k + 16 candidates
    (9, 2048, 64, 500, False),        # no sample: dense pre-activations + dense radix select
    (7, 2048, 64, 500, True),
    (5, 4096, 8, 4096, False),        # k == H
])
def test_large_k_topk_matches_oracle(cuda_device, B, H, D, k, exact):
    x, W, b = _enc_case(B, H, D, 300 + k, bf16=not exact)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    sample = L.prepare_sample(wb, db)
    assert (sample is not None) == (H >= 8192)
    vals, idx, flags = L.encode_topk(dx, wb, dW if exact else None, db, k, exact=exact, want_flags=True, sample=sample)
    assert_topk_matches(vals.cpu().numpy(), idx.cpu().numpy(), O.encode_pre(x, W, b), k)
    assert int((flags != 0).sum()) == 0


def test_large_k_relu_ties_and_failed_prior_are_rescued(cuda_device):
    """(a) ReLU zeros flood every survivor list (threshold 0 keeps all H latents): the rows must go
    through the exact dense recomputation and come back in (value desc, index asc) order, bit exact.
    (b) A prior that is far too high (sampled rows carry a bias the real rows lack) fails the count
    check on every row."""
    B, H, D, k = 20, 16384, 64, 1000
    x, W, b = _enc_case(B, H, D, 91)
    b = b - 0.6
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    sample = L.prepare_sample(wb, db)
    vals, idx, _ = L.encode_topk(dx, wb, None, db, k, act=L.ACT_RELU, sample=sample)
    zr = np.maximum(O.encode_pre(x, W, b), 0).astype(np.float32)
    rv, ri = O.topk_rows(zr, k)
    assert (rv == 0).any()
    assert_topk_matches(vals.cpu().numpy(), idx.cpu().numpy(), zr, k)
    zero = rv == 0
    assert np.array_equal(idx.cpu().numpy()[zero], ri[zero])
    ws, bs = sample
    for exact in (False, True):
        vals, idx, flags = L.encode_topk(dx, wb, dW if exact else None, db, 300, exact=exact, want_flags=True,
                                         sample=(ws, bs + 100.0))
        assert_topk_matches(vals.cpu().numpy(), idx.cpu().numpy(), O.encode_pre(x, W, b), 300)
        assert int((flags != 0).sum()) == 0


def test_large_k_dense_topk_and_decode(cuda_device):
    """dense top-k with k > QSAE_MAX_K (apply_topk_activation / binary_decoder.forward on dense latents)
    and the sparse decoders at the same k."""
    rng = np.random.default_rng(12)
    R, H, D, k = 11, 20000, 64, 700
    z = rng.standard_normal((R, H)).astype(np.float32)
    z[3] = np.round(z[3])                                               # heavy ties in one row
    vals, idx = L.topk_dense(T(z, cuda_device), k)
    rv, ri = O.topk_rows(z, k)
    assert np.array_equal(idx.cpu().numpy(), ri) and np.array_equal(vals.cpu().numpy(), rv)
    iw = rng.integers(-8, 8, size=(H, D)).astype(np.int8)
    bias = rng.standard_normal(D).astype(np.float32)
    ref = O.decode_rows(rv, ri, iw.astype(np.float32), 0.5, bias)
    got = L.decode_int4(vals, idx, T(O.pack_nibbles(iw), cuda_device), H, D, 0.5, T(bias, cuda_device)).cpu().numpy()
    assert_recon_close(got, ref)
    got = L.decode_int8(vals, idx, T(iw, cuda_device), H, D, 0.5, T(bias, cuda_device)).cpu().numpy()
    assert_recon_close(got, ref)


def test_bsae_module_reference_default_k_large_dictionary(cuda_device):
    """BinarySAE at H = 2^17 keeps int(0.002 H) = 262 latents per row (sae/binary.py:94): module forward
    vs the oracle restatement (the reference itself is pinned at smaller H by the golden fixtures)."""
    D, H, B, n_bits = 64, 2 ** 17, 48, 4
    rng = np.random.default_rng(8)
    x = cases.round_bf16(rng.standard_normal((B, D)).astype(np.float32))
    We = cases.round_bf16(cases.xavier_uniform(rng, H, D))
    be = np.zeros(H, np.float32)
    logits = np.where(rng.random((H, D * n_bits)) < 0.5, 110.0, -110.0).astype(np.float32)
    bd = rng.standard_normal(D).astype(np.float32)
    m = Q.BinarySAE(D, H, 4.0, n_bits)
    m.load_state_dict({"encoder.0.weight": torch.from_numpy(We), "encoder.0.bias": torch.from_numpy(be),
                       "decoder.weight": torch.from_numpy(logits), "decoder.bias": torch.from_numpy(bd)}, strict=True)
    m.to(cuda_device).eval()
    m.return_dense = False
    k = O.bsae_k(H)
    assert k == 262
    with torch.no_grad():
        sp, recon, pol = m(T(x, cuda_device))
    rv, ri, rr, rp = O.bsae_forward(x, We, be, logits, bd, n_bits=n_bits, gamma=4.0, k=k, mode="hard")
    assert_topk_matches(sp.values.cpu().numpy(), sp.indices.cpu().numpy(), O.encode_pre(x, We, be), k)
    assert_recon_close(recon.cpu().numpy(), rr)
    assert float(pol) == pytest.approx(rp, abs=1e-9)


def test_sample_rows_are_a_stratified_subset(cuda_device):
    H, D, n = 32768, 64, 1024
    W = torch.arange(H, device=cuda_device, dtype=torch.float32)[:, None].expand(H, D).contiguous()
    b = torch.arange(H, device=cuda_device, dtype=torch.float32)
    ws, bs = L.prepare_sample(L.cast_bf16(W), b, n)
    rows = bs.cpu().numpy().astype(np.int64)
    assert len(set(rows.tolist())) == n
    assert np.all(rows // (H // n) == np.arange(n))   # one row from each of the n equal slices


# ------------------------------------------------------------------------------------------
# q_sae (Quantized Matryoshka) vs the reference's own outputs
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(cases.QSAE_CASES))
def test_qsae_module_matches_reference(cuda_device, golden_dir, name):
    cfg = cases.QSAE_CASES[name]
    g = np.load(golden_dir / f"{name}.npz")
    inp = cases.qsae_inputs(cfg)
    m = Q.QuantizedMatryoshkaSAE(cfg["D"], cfg["H"], 32, cfg["abs_range"], cfg["n_bits"], cfg["allow_bias"])
    m.load_state_dict({"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
                       "decoder.weight": torch.from_numpy(inp["W"]), "decoder.weight_mirror": torch.from_numpy(inp["Wm"]),
                       "decoder.bias": torch.from_numpy(inp["bd"])}, strict=True)
    m.to(cuda_device).eval()
    assert m.decoder.nested_dictionary_size == g["level_sizes"].tolist()
    with torch.no_grad():
        groups, result = m(T(inp["x"], cuda_device))
    assert len(groups) == cfg["n_bits"] == len(result) and groups[0].dim() == 0
    np.testing.assert_allclose(np.array([float(v) for v in groups]), g["latent_group"], rtol=1e-6, atol=1e-6)
    for i in range(cfg["n_bits"]):
        assert_recon_close(result[i].cpu().numpy(), g["result"][i])
    # packed dictionary: bit exact against the oracle's T and scale
    packed, scale = m.decoder._packed()
    Tref, sref, _, _ = O.qsae_dictionary(inp["W"], inp["Wm"], n_bits=cfg["n_bits"], abs_range=cfg["abs_range"])
    codes = packed.cpu().numpy().view(np.uint32)
    ent = ((codes[:, :, None] >> (2 * np.arange(16, dtype=np.uint32))) & 3).reshape(cfg["H"], -1)
    Tgot = np.where(ent & 1, np.where(ent & 2, -2, 2), 0).astype(np.int8)
    assert np.array_equal(Tgot, Tref)
    np.testing.assert_allclose(scale.cpu().numpy(), sref, rtol=2e-7, atol=0)
    # the decoder alone, fed the dense sigmoid latents the reference passes (:219)
    with torch.no_grad():
        g2, r2 = m.decoder(m.encode(T(inp["x"], cuda_device)))
    for i in range(cfg["n_bits"]):
        assert_recon_close(r2[i].cpu().numpy(), g["result"][i])
    np.testing.assert_allclose(np.array([float(v) for v in g2]), g["latent_group"], rtol=1e-6, atol=1e-6)


def test_qsae_headline_shape_vs_oracle(cuda_device):
    """512 -> 32768, n_bits = 4, encoder bias -0.543 (mean L0 ~ 34, SURVEY 8d config 4)."""
    cfg = dict(D=512, H=32768, n_bits=4, abs_range=4.0, B=96, enc_bias=-0.543, bf16=False, allow_bias=True, seed=91)
    inp = cases.qsae_inputs(cfg)
    m = Q.QuantizedMatryoshkaSAE(cfg["D"], cfg["H"], 32, cfg["abs_range"], cfg["n_bits"], True)
    m.load_state_dict({"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
                       "decoder.weight": torch.from_numpy(inp["W"]), "decoder.weight_mirror": torch.from_numpy(inp["Wm"]),
                       "decoder.bias": torch.from_numpy(inp["bd"])}, strict=True)
    m.to(cuda_device).eval()
    with torch.no_grad():
        groups, result = m(T(inp["x"], cuda_device))
    rg, rr, act = O.qsae_forward(inp["x"], inp["We"], inp["be"], inp["W"], inp["Wm"], inp["bd"],
                                 n_bits=4, abs_range=4.0, allow_bias=True)
    assert 20 < act.sum(1).mean() < 50
    np.testing.assert_allclose(np.array([float(v) for v in groups]), rg, rtol=1e-6, atol=1e-6)
    for i in range(4):
        assert_recon_close(result[i].cpu().numpy(), rr[i])


# ------------------------------------------------------------------------------------------
# t_sae (ternary): dense ReLU latents + dense ternary decoder GEMM
#   h (exact mode or bf16-representable inputs) ........ |dh| <= 1e-5 * max(1, |h|)
#   recon, exact mode (hi/lo two-pass decoder) ......... atol 1e-4 * rms + rtol 1e-4
#   recon, fast mode (one bf16 pass over h) ............ atol 8e-3 * rms + rtol 8e-3
# ------------------------------------------------------------------------------------------
def assert_recon_close_bf16(got, ref):
    rms = float(np.sqrt(np.mean(np.square(ref, dtype=np.float64)))) + 1e-30
    np.testing.assert_allclose(got, ref, rtol=8e-3, atol=8e-3 * rms)


def test_pack_ternary_bit_exact(cuda_device):
    rng = np.random.default_rng(5)
    D, H = 70, 1000
    w = (0.4824 * rng.standard_normal((D, H))).astype(np.float32)
    w[0, :8] = [0.5, -0.5, np.nextafter(np.float32(0.5), np.float32(0)), -np.nextafter(np.float32(0.5), np.float32(0)),
                0.0, -0.0, 3.0, -3.0]
    t_bf16, t_rows = L.pack_ternary(T(w, cuda_device), 0.5, want_bf16=True, want_rows=True)
    ref = O.ternarize(w)
    assert np.array_equal(t_bf16.float().cpu().numpy().astype(np.int8), ref)
    assert np.array_equal(t_rows.cpu().numpy(), ref.T)
    assert ref[0, :8].tolist() == [1, -1, 0, 0, 0, 0, 1, -1]


@pytest.mark.parametrize("B,K,N", [(128, 1024, 512), (200, 4096, 64), (77, 1000, 256), (1, 72, 8), (300, 2048, 384),
                                   (33, 8, 64), (130, 32, 512), (1, 40, 16)])
def test_decode_dense_vs_fp64(cuda_device, B, K, N):
    rng = np.random.default_rng(B + K + N)
    a = np.maximum(rng.standard_normal((B, K)), 0).astype(np.float32)
    t = O.ternarize((0.4824 * rng.standard_normal((N, K))).astype(np.float32))
    bias = rng.standard_normal(N).astype(np.float32)
    ref = a.astype(np.float64) @ t.T.astype(np.float64) + bias
    hi, lo = L.split_bf16(T(a, cuda_device))
    tb = T(t.astype(np.float32), cuda_device).bfloat16().contiguous()
    # hi + lo reproduces a to 2^-17
    rec = hi.float().cpu().numpy().astype(np.float64) + lo.float().cpu().numpy()
    assert np.all(np.abs(rec - a) <= 2.0 ** -16 * np.abs(a) + 1e-38)
    two = L.decode_dense(hi, lo, tb, T(bias, cuda_device)).cpu().numpy()
    assert_recon_close(two, ref.astype(np.float32))
    one = L.decode_dense(hi, None, tb, T(bias, cuda_device)).cpu().numpy()
    assert_recon_close_bf16(one, ref.astype(np.float32))
    # the single pass is exact for the operand it was given: compare against bf16(a) in fp64
    ref_hi = hi.float().cpu().numpy().astype(np.float64) @ t.T.astype(np.float64) + bias
    assert_recon_close(one, ref_hi.astype(np.float32))


@pytest.mark.parametrize("B,H,D", [(128, 256, 64), (200, 1000, 512), (77, 2056, 72), (1, 304, 8), (300, 4096, 512)])
def test_dense_encoder_tma_store_epilogue(cuda_device, B, H, D):
    """fast t_sae path: h = relu(x W^T + b) written by TMA stores as fp32 (+ bf16 for the decoder)."""
    xn, Wn, bn = _enc_case(B, H, D, seed=B + H)
    inp = dict(x=xn, We=Wn, be=bn)
    rng = np.random.default_rng(3)
    wd = (0.4824 * rng.standard_normal((D, H))).astype(np.float32)
    We, be, x = (T(inp[k], cuda_device) for k in ("We", "be", "x"))
    t_bf16, _ = L.pack_ternary(T(wd, cuda_device))
    h, recon = L.tsae_forward(x, (L.cast_bf16(We),), be, t_bf16, exact=False)
    torch.cuda.synchronize()
    h_ref, r_ref = O.tsae_forward(inp["x"], inp["We"], inp["be"], wd)
    assert_vals_close(h.cpu().numpy(), h_ref)
    assert_recon_close_bf16(recon.cpu().numpy(), r_ref)
    # the decoder consumed bf16(h) of the h this kernel produced: recompute exactly that
    hb = h.bfloat16().float().cpu().numpy().astype(np.float64)
    assert_recon_close(recon.cpu().numpy(), (hb @ O.ternarize(wd).T.astype(np.float64)).astype(np.float32))


@pytest.mark.parametrize("name", list(cases.TSAE_CASES))
def test_tsae_module_matches_reference(cuda_device, golden_dir, name):
    cfg = cases.TSAE_CASES[name]
    g = np.load(golden_dir / f"{name}.npz")
    inp = cases.tsae_inputs(cfg)
    m = Q.TernarySparseAutoencoder(cfg["D"], cfg["H"])
    assert sorted(m.state_dict().keys()) == g["state_keys"].tolist()
    sd = m.state_dict()
    sd.update({"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
               "decoder.weight": torch.from_numpy(inp["Wd"])})
    m.load_state_dict(sd, strict=True)
    m.to(cuda_device).eval()
    assert m.topk == int(cfg["H"] * 0.002) and m.decoder.threshold == 0.5
    with torch.no_grad():
        h, recon = m(T(inp["x"], cuda_device))                       # exact mode (default)
    assert tuple(h.shape) == (cfg["B"], cfg["H"]) and tuple(recon.shape) == (cfg["B"], cfg["D"])
    assert_vals_close(h.cpu().numpy(), g["h"])
    assert_recon_close(recon.cpu().numpy(), g["recon"])
    assert sorted(m.state_dict().keys()) == g["state_keys_after_forward"].tolist()
    assert np.array_equal(m.decoder.hard_weights().cpu().numpy().astype(np.int8), O.ternarize(inp["Wd"]))
    # decoder alone on the dense latents, as callers of STEWeights use it
    with torch.no_grad():
        r2 = m.decoder(T(g["h"], cuda_device))
    assert_recon_close(r2.cpu().numpy(), g["recon"])
    if cfg["bf16"]:
        m.exact = False
        with torch.no_grad():
            h3, r3 = m(T(inp["x"], cuda_device))
        assert_vals_close(h3.cpu().numpy(), g["h"])
        assert_recon_close_bf16(r3.cpu().numpy(), g["recon"])


def test_tsae_topk_mode_vs_oracle(cuda_device):
    cfg = dict(D=512, H=8192, B=64, bf16=True, seed=77)
    inp = cases.tsae_inputs(cfg)
    m = Q.TernarySparseAutoencoder(cfg["D"], cfg["H"])
    sd = m.state_dict()
    sd.update({"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
               "decoder.weight": torch.from_numpy(inp["Wd"])})
    m.load_state_dict(sd, strict=True)
    m.to(cuda_device).eval()
    h_ref, _ = O.tsae_forward(inp["x"], inp["We"], inp["be"], inp["Wd"])
    with torch.no_grad():
        lat, recon = m.forward_topk(T(inp["x"], cuda_device))
        dense = m.apply_topk_activation(T(h_ref, cuda_device))
    assert_topk_matches(lat.values.cpu().numpy(), lat.indices.cpu().numpy(), h_ref, m.topk)
    rv, ri = O.tsae_topk_activation(h_ref, m.topk)
    ref_recon = O.decode_rows(rv, ri, np.ascontiguousarray(O.ternarize(inp["Wd"]).T.astype(np.float32)), 1.0, None)
    assert_recon_close(recon.cpu().numpy(), ref_recon)
    assert np.array_equal(dense.cpu().numpy(), O.densify(rv, ri, cfg["H"]))


def test_tsae_full_size_properties(cuda_device):
    """4096 x 32768 x 512 (BASELINE config 3 per GPU): spot rows against the fp32 CUDA-core encoder,
    fast decoder against the exact two-pass decoder, and linearity of the decoder."""
    B, H, D = 4096, 32768, 512
    g = torch.Generator(device=cuda_device).manual_seed(3)
    We = ((torch.rand((H, D), device=cuda_device, generator=g) * 2 - 1) * (6.0 / (H + D)) ** 0.5).bfloat16().float()
    be = 0.01 * torch.randn(H, device=cuda_device, generator=g)
    Wd = 0.4824 * torch.randn((D, H), device=cuda_device, generator=g)
    x = torch.randn((B, D), device=cuda_device, generator=g).bfloat16().float()
    t_bf16, _ = L.pack_ternary(Wd)
    h, recon = L.tsae_forward(x, (L.cast_bf16(We),), be, t_bf16, exact=False)
    rows = torch.tensor([0, 1, 127, 128, 2047, 4095], dtype=torch.int32, device=cuda_device)
    z = L.encode_dense(x, We, be, L.ACT_RELU, rows=rows)
    assert_vals_close(h[rows.long()].cpu().numpy(), z.cpu().numpy())
    assert float(h.min()) >= 0.0 and 0.4 < float((h > 0).float().mean()) < 0.6
    hi, lo = L.split_bf16(h)
    exact = L.decode_dense(hi, lo, t_bf16)
    assert_recon_close_bf16(recon.cpu().numpy(), exact.cpu().numpy())
    assert torch.equal(L.decode_dense(hi, None, t_bf16), recon)          # deterministic, same operand
    ref64 = (h[:64].double() @ t_bf16.double().T).float()
    assert_recon_close(exact[:64].cpu().numpy(), ref64.cpu().numpy())


# ------------------------------------------------------------------------------------------
# q_sae dense path (any activity level): level sums as tcgen05 GEMMs
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(cases.QSAE_CASES))
@pytest.mark.parametrize("exact", [True, False])
def test_qsae_dense_path_matches_reference(cuda_device, golden_dir, name, exact):
    cfg = cases.QSAE_CASES[name]
    if not exact and not cfg["bf16"]:
        pytest.skip("the tensor-core encoder needs bf16-representable inputs for sign-exact activity")
    g = np.load(golden_dir / f"{name}.npz")
    inp = cases.qsae_inputs(cfg)
    m = Q.QuantizedMatryoshkaSAE(cfg["D"], cfg["H"], 32, cfg["abs_range"], cfg["n_bits"], cfg["allow_bias"])
    m.load_state_dict({"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
                       "decoder.weight": torch.from_numpy(inp["W"]), "decoder.weight_mirror": torch.from_numpy(inp["Wm"]),
                       "decoder.bias": torch.from_numpy(inp["bd"])}, strict=True)
    m.to(cuda_device).eval()
    m.dense_mode, m.exact = "always", exact
    with torch.no_grad():
        groups, result = m(T(inp["x"], cuda_device))
    assert m.last_path == "dense"
    np.testing.assert_allclose(np.array([float(v) for v in groups]), g["latent_group"], rtol=1e-6, atol=1e-6)
    for i in range(cfg["n_bits"]):
        assert_recon_close(result[i].cpu().numpy(), g["result"][i])
    # T^T operand: bit exact against the oracle dictionary
    Tref, _, _, _ = O.qsae_dictionary(inp["W"], inp["Wm"], n_bits=cfg["n_bits"], abs_range=cfg["abs_range"])
    assert np.array_equal(m.decoder._t_bf16().float().cpu().numpy().astype(np.int8), Tref.T)


def test_qsae_untrained_model_falls_back_to_dense(cuda_device):
    """Random init, zero encoder bias: ~50 % of 32768 latents active per row (SURVEY 8d config 4, dense case).
    The sparse path overflows its survivor lists and the forward is redone on the dense path."""
    cfg = dict(D=512, H=32768, n_bits=4, abs_range=4.0, B=160, enc_bias=0.0, bf16=False, allow_bias=True, seed=92)
    inp = cases.qsae_inputs(cfg)
    m = Q.QuantizedMatryoshkaSAE(cfg["D"], cfg["H"], 32, cfg["abs_range"], cfg["n_bits"], True)
    m.load_state_dict({"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
                       "decoder.weight": torch.from_numpy(inp["W"]), "decoder.weight_mirror": torch.from_numpy(inp["Wm"]),
                       "decoder.bias": torch.from_numpy(inp["bd"])}, strict=True)
    m.to(cuda_device).eval()
    with torch.no_grad():
        groups, result = m(T(inp["x"], cuda_device))
    assert m.last_path == "dense"
    rg, rr, act = O.qsae_forward(inp["x"], inp["We"], inp["be"], inp["W"], inp["Wm"], inp["bd"],
                                 n_bits=4, abs_range=4.0, allow_bias=True)
    assert 15000 < act.sum(1).mean() < 18000
    np.testing.assert_allclose(np.array([float(v) for v in groups]), rg, rtol=1e-6, atol=1e-6)
    for i in range(4):
        assert_recon_close(result[i].cpu().numpy(), rr[i])
    m.dense_mode = "never"
    with pytest.raises(RuntimeError, match="more active latents"):
        m(T(inp["x"], cuda_device))


@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("B,H", [(160, 32768), (700, 4096), (40, 1024), (90, 832), (120, 2056)])
def test_qsae_dense_operand_from_the_encoder_epilogue(cuda_device, tuning, B, H, exact):
    """The dense path's A operand (active * scale as bf16 hi / lo) and the per-level activity counts written by the
    encoder epilogue itself (act = 2) against the first form: fp32 pre-activations to HBM + the streaming operand kernel.
    Same activity decisions, same operand bits: identical outputs. exact: the one-launch split-operand encoder."""
    cfg = dict(D=512, H=H, n_bits=4, abs_range=4.0, B=B, enc_bias=0.0, bf16=not exact, allow_bias=True, seed=B + H)
    inp = cases.qsae_inputs(cfg)
    m = Q.QuantizedMatryoshkaSAE(cfg["D"], H, 32, cfg["abs_range"], cfg["n_bits"], True)
    m.load_state_dict({"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
                       "decoder.weight": torch.from_numpy(inp["W"]), "decoder.weight_mirror": torch.from_numpy(inp["Wm"]),
                       "decoder.bias": torch.from_numpy(inp["bd"])}, strict=True)
    m.to(cuda_device).eval()
    m.dense_mode, m.exact = "always", exact
    x = T(inp["x"], cuda_device)
    with torch.no_grad():
        g1, r1 = m(x)
        tuning("QSAE_DENSE_STEP_FUSED", "0")
        g0, r0 = m(x)
    assert [float(v) for v in g1] == [float(v) for v in g0]
    assert all(torch.equal(a, b) for a, b in zip(r1, r0))
    rg, rr, _ = O.qsae_forward(inp["x"], inp["We"], inp["be"], inp["W"], inp["Wm"], inp["bd"], n_bits=4, abs_range=4.0,
                               allow_bias=True)
    # A pre-activation within fp32 accumulation noise of the threshold may fall on either side (of ~5 M decisions a
    # handful has |z| < 1e-7; the reference's own fp32 matmul decides them by its summation order), and one flipped
    # decision moves that row's reconstruction by 2 * scale: counts within 2e-5, all but a few rows within tolerance.
    np.testing.assert_allclose(np.array([float(v) for v in g1]), rg, rtol=2e-5, atol=1e-6)
    if exact:
        for i in range(4):
            got, ref = r1[i].cpu().numpy(), rr[i]
            rms = float(np.sqrt(np.mean(np.square(ref, dtype=np.float64)))) + 1e-30
            bad_rows = np.any(np.abs(got - ref) > 1e-4 * np.abs(ref) + 1e-4 * rms, axis=1)
            assert bad_rows.sum() <= max(1, B // 50)


def test_qsae_lazy_overflow_regime(cuda_device):
    """dense_mode = "auto" synchronises only on the first forward of a weight version. Sparse regime, then a batch whose
    activity overflows the survivor lists: that forward's outputs are NaN (never a silently wrong reconstruction), the
    flag is picked up lazily, a warning is issued and the module serves the dense path from then on. A second forward on
    the dense-regime model goes straight to the dense path (no wasted sparse sweep)."""
    import warnings

    D, H, B = 512, 32768, 256
    torch.manual_seed(5)
    with torch.device(cuda_device):
        m = Q.QuantizedMatryoshkaSAE(D, H, 32, abs_range=4.0, n_bits=4)
    with torch.no_grad():
        m.encoder[0].bias.fill_(-0.543)
    m.eval()
    x = torch.randn((B, D), device=cuda_device)
    with torch.no_grad():
        g0, r0 = m(x)                                   # first forward: synchronous check, regime = sparse
        assert m.last_path == "sparse" and m._regime[1] == "sparse" and not m.overflowed()
        g1, r1 = m(x)                                   # steady state: no host sync, flag copied lazily
        assert torch.equal(r0[3], r1[3])
        xbig = x * 40.0 + 30.0 * torch.sign(m.encoder[0].weight.detach()[:2000].sum(0))   # thousands of active latents per row
        g2, r2 = m(xbig)
        torch.cuda.synchronize()
        assert m.overflowed() and bool(torch.isnan(r2[3]).all())
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            g3, r3 = m(xbig)                            # picks the flag up, warns, switches to the dense regime
        assert any("overflowed" in str(i.message) for i in w)
        assert m.last_path == "dense" and not bool(torch.isnan(r3[3]).any())
        lg, res, act = O.qsae_forward(xbig[:8].cpu().numpy(), m.encoder[0].weight.detach().cpu().numpy(),
                                      m.encoder[0].bias.detach().cpu().numpy(), m.decoder.weight.detach().cpu().numpy(),
                                      m.decoder.weight_mirror.detach().cpu().numpy(), m.decoder.bias.detach().cpu().numpy(),
                                      n_bits=4, abs_range=4.0)
        assert act.sum(1).min() > 2100
        # thousands of active latents per row at |z| ~ 10: a latent within fp32 rounding of the threshold may flip
        # (one dictionary row, <= 0.5 per element), so compare robustly; the dense path itself is pinned bit-tight by
        # test_qsae_dense_path_matches_reference
        diff = np.abs(r3[3][:8].cpu().numpy() - res[3])
        rms = float(np.sqrt(np.mean(res[3].astype(np.float64) ** 2)))
        assert float(np.median(diff)) <= 1e-4 * rms and float(diff.max()) <= 1.0


@pytest.mark.parametrize("mcast", ["1", "2"])
def test_cluster_variants_are_bit_identical(cuda_device, tuning, mcast):
    """The cluster-of-two variants of the encoder -- 1: TMA multicast of the W stages, 2: cta_group::2
    MMA pairs -- with the sparse and the dense epilogue must give the same bits as the single-CTA
    variant; odd numbers of row blocks exercise the padding CTA. The dense epilogue has no multicast
    variant: under "1" it runs its default, the pair variant, so both parameters compare that with the
    single-CTA variant."""
    B, H, D, k = 300, 8192, 512, 32
    x, W, b = _enc_case(B, H, D, 55)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    tuning("QSAE_ENCODE_CLUSTER", mcast)
    vals, idx, _ = L.encode_topk(dx, wb, None, db, k, sample=L.prepare_sample(wb, db))
    assert_topk_matches(vals.cpu().numpy(), idx.cpu().numpy(), O.encode_pre(x, W, b), k)
    wd = (0.4824 * np.random.default_rng(1).standard_normal((D, H))).astype(np.float32)
    t_bf16, _ = L.pack_ternary(T(wd, cuda_device))
    h, recon = L.tsae_forward(dx, (wb,), db, t_bf16, exact=False)
    tuning("QSAE_ENCODE_CLUSTER", "0")
    v0, i0, _ = L.encode_topk(dx, wb, None, db, k, sample=L.prepare_sample(wb, db))
    h0, r0 = L.tsae_forward(dx, (wb,), db, t_bf16, exact=False)
    assert torch.equal(vals, v0) and torch.equal(idx, i0) and torch.equal(h, h0) and torch.equal(recon, r0)


# ------------------------------------------------------------------------------------------
# rq_sae (residual cascade of one-bit q_saes) vs the reference's own outputs
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(cases.RQSAE_CASES))
def test_rqsae_module_matches_reference(cuda_device, golden_dir, name):
    cfg = cases.RQSAE_CASES[name]
    g = np.load(golden_dir / f"{name}.npz")
    inp = cases.rqsae_inputs(cfg)
    m = Q.ResidualQuantizedSAE(cfg["D"], cfg["H"], 32, cfg["abs_range"], cfg["n_bits"])
    assert m.sae_hidden_dims == g["stage_sizes"].tolist()
    assert sorted(m.state_dict().keys()) == g["state_keys"].tolist()
    assert [str(tuple(v.shape)) for _, v in sorted(m.state_dict().items())] == g["state_shapes"].tolist()
    m.load_state_dict({k: torch.from_numpy(v) for k, v in cases.rqsae_state_dict(inp, cfg["n_bits"]).items()}, strict=True)
    m.to(cuda_device).eval()
    with torch.no_grad():
        groups, recons = m(T(inp["x"], cuda_device))
    assert len(groups) == len(recons) == cfg["n_bits"]
    np.testing.assert_allclose(np.array([float(v) for v in groups]), g["latent_group"], rtol=1e-6, atol=1e-6)
    for t in range(cfg["n_bits"]):
        assert_recon_close(recons[t].cpu().numpy(), g["recon"][t])


def test_inference_wrapper_on_gpu(cuda_device, golden_dir, tmp_path):
    """load_sae -> SAEWrapper on the B200 modules: output dictionaries of inference/framework.py:76-111 and
    the b_sae dictionary export (:114-124) against the reference fixture."""
    from quantizedsae_b200 import inference as I

    name = "bsae_polar_d64_h2048"
    cfg, g = cases.BSAE_CASES[name], np.load(golden_dir / f"{name}.npz")
    inp = cases.bsae_inputs(cfg)
    torch.save({"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
                "decoder.weight": torch.from_numpy(inp["logits"]), "decoder.bias": torch.from_numpy(inp["bd"])},
               tmp_path / "b.pth")
    w = I.load_sae("b_sae", device=cuda_device, checkpoint_path=tmp_path / "b.pth", input_dim=cfg["D"], hidden_dim=cfg["H"],
                   gamma=cfg["gamma"], n_bits=cfg["n_bits"])
    out = w([torch.from_numpy(inp["x"])])                       # DataLoader-style 1-list, host tensor
    assert set(out) == {"latent", "reconstruction", "aux"} and "polarize_loss" in out["aux"]
    assert_recon_close(out["reconstruction"].cpu().numpy(), g["recon"])
    assert tuple(out["latent"].shape) == (cfg["B"], cfg["H"])
    d = w.decoder_dictionary()
    ref = O.dequant_hard(inp["logits"], cfg["n_bits"]).astype(np.float32) * (cfg["gamma"] / 2 ** (cfg["n_bits"] - 1))
    assert np.array_equal(d["weight"].numpy(), ref) and not d["weight"].is_cuda
    recs = list(w.reconstruct_loader([torch.from_numpy(inp["x"][:8]), torch.from_numpy(inp["x"][8:])]))
    assert_recon_close(torch.cat(recs).cpu().numpy(), g["recon"])


@pytest.mark.parametrize("B,K,N", [(300, 4096, 512), (129, 1000, 64), (1024, 8192, 384)])
def test_decoder_gemm_pair_variant_is_bit_identical(cuda_device, tuning, B, K, N):
    """cta_group::2 pairs (default for more than one row block) against the single-CTA kernel."""
    rng = np.random.default_rng(B)
    a = np.maximum(rng.standard_normal((B, K)), 0).astype(np.float32)
    t = O.ternarize((0.4824 * rng.standard_normal((N, K))).astype(np.float32))
    hi, lo = L.split_bf16(T(a, cuda_device))
    tb = T(t.astype(np.float32), cuda_device).bfloat16().contiguous()
    tuning("QSAE_DECODE_PAIR", "1")
    one, two = L.decode_dense(hi, None, tb), L.decode_dense(hi, lo, tb)
    tuning("QSAE_DECODE_PAIR", "0")
    assert torch.equal(one, L.decode_dense(hi, None, tb)) and torch.equal(two, L.decode_dense(hi, lo, tb))
    assert_recon_close(two.cpu().numpy(), (a.astype(np.float64) @ t.T.astype(np.float64)).astype(np.float32))


@pytest.mark.parametrize("B,H,D", [(24, 4096, 512), (300, 8192, 512), (130, 1000, 72), (512, 32768, 512), (1024, 32768, 512),
                                   (1, 304, 8), (129, 264, 16), (257, 8, 8)])
def test_exact_dense_encoder_split_passes(cuda_device, B, H, D):
    """fp32-accurate dense encoder on the tensor cores (3 x 3 bf16 operand split: the six partial products
    above 2^-24 accumulate in one TMEM accumulator, one launch of the streamed-operand kernel on CTA pairs):
    arbitrary fp32 x and W, h within 1e-5 * max(1, |h|) of the fp64 value; split parts sum exactly."""
    x, W, b = _enc_case(B, H, D, seed=B + D, bf16=False)
    rng = np.random.default_rng(9)
    wd = (0.4824 * rng.standard_normal((D, H))).astype(np.float32)
    dW = T(W, cuda_device)
    parts = L.split_bf16x3(dW)
    total = parts[0].double() + parts[1].double() + parts[2].double()
    assert torch.equal(total.float(), dW) and torch.equal(total, dW.double())
    t_bf16, _ = L.pack_ternary(T(wd, cuda_device))
    h, recon = L.tsae_forward(T(x, cuda_device), parts, T(b, cuda_device), t_bf16, exact=True)
    h64 = np.maximum(x.astype(np.float64) @ W.astype(np.float64).T + b, 0)
    got = h.cpu().numpy()
    assert np.all(np.abs(got - h64) <= 1e-5 * np.maximum(1.0, np.abs(h64)))
    # tighter: the split passes are as good as an fp32 matmul (products exact, fp32 accumulation)
    assert np.max(np.abs(got - h64)) <= 4e-6 * max(1.0, np.max(np.abs(h64)))
    assert_recon_close(recon.cpu().numpy(), (h64 @ O.ternarize(wd).T.astype(np.float64)).astype(np.float32))


def test_stream_pipeline_matches_serial_forwards(cuda_device):
    """Two batches in flight on two streams (quantizedsae_b200/pipeline.py) give the bits of the serial loop."""
    from quantizedsae_b200.pipeline import StreamPipeline

    cfg = cases.BSAE_CASES["bsae_polar_d512_h4096"]
    inp = cases.bsae_inputs(cfg)
    m = Q.BinarySAE(cfg["D"], cfg["H"], cfg["gamma"], cfg["n_bits"]).to(cuda_device)
    m.load_state_dict({"encoder.0.weight": T(inp["We"], cuda_device), "encoder.0.bias": T(inp["be"], cuda_device),
                       "decoder.weight": T(inp["logits"], cuda_device), "decoder.bias": T(inp["bd"], cuda_device)}, strict=True)
    m.return_dense = False
    rng = np.random.default_rng(3)
    batches = [T(cases.round_bf16(rng.standard_normal((300 + 17 * i, cfg["D"])).astype(np.float32)), cuda_device) for i in range(7)]
    pipe = StreamPipeline(m, n_streams=2)
    got = list(pipe.map(batches))                      # the first batch also builds the prepared weights
    torch.cuda.synchronize()
    with torch.no_grad():
        want = [m(b) for b in batches]
    torch.cuda.synchronize()
    assert len(got) == len(want)
    for (gl, gr, gp), (wl, wr, wp) in zip(got, want):
        assert torch.equal(gl.indices, wl.indices) and torch.equal(gl.values, wl.values)
        assert torch.equal(gr, wr) and float(gp) == float(wp)
    # a q_sae model through the same pipeline, three streams
    qc = cases.QSAE_CASES["qsae_d512_h4096"]
    qi = cases.qsae_inputs(qc)
    q = Q.QuantizedMatryoshkaSAE(qc["D"], qc["H"], 32, qc["abs_range"], qc["n_bits"], qc["allow_bias"]).to(cuda_device)
    q.load_state_dict({"encoder.0.weight": T(qi["We"], cuda_device), "encoder.0.bias": T(qi["be"], cuda_device),
                       "decoder.weight": T(qi["W"], cuda_device), "decoder.weight_mirror": T(qi["Wm"], cuda_device),
                       "decoder.bias": T(qi["bd"], cuda_device)}, strict=True)
    qb = [T(cases.round_bf16(rng.standard_normal((200, qc["D"])).astype(np.float32)), cuda_device) for _ in range(5)]
    got = list(StreamPipeline(q, n_streams=3).map(qb))
    torch.cuda.synchronize()
    with torch.no_grad():
        want = [q(b) for b in qb]
    for (gg, gl), (wg, wl) in zip(got, want):
        assert all(torch.equal(a, b) for a, b in zip(gl, wl)) and all(float(a) == float(b) for a, b in zip(gg, wg))


@pytest.mark.parametrize("B,H", [(1, 5), (7, 130), (33, 2048), (5, 4099)])
def test_compact_dense_vs_numpy(cuda_device, B, H):
    rng = np.random.default_rng(B * 31 + H)
    a = rng.standard_normal((B, H)).astype(np.float32)
    a[rng.random((B, H)) < 0.9] = 0.0
    a[0, :] = 0.0                                                # an empty row
    idx, vals, cnt = L.compact_dense(T(a, cuda_device), 0, want_vals=True)
    idx, vals, cnt = idx.cpu().numpy(), vals.cpu().numpy(), cnt.cpu().numpy()
    assert np.array_equal(cnt, (a != 0).sum(1))
    assert idx.shape[1] == max(1, cnt.max())
    for b in range(B):
        nz = np.nonzero(a[b])[0]
        assert np.array_equal(idx[b, :len(nz)], nz) and np.all(idx[b, len(nz):] == -1)
        assert np.array_equal(vals[b, :len(nz)], a[b, nz]) and np.all(vals[b, len(nz):] == 0)
    pairs, _, cnt2 = L.compact_dense(T(a, cuda_device), 1, 0.5, want_pairs=True)
    pairs, cnt2 = pairs.cpu().numpy(), cnt2.cpu().numpy()
    assert np.array_equal(cnt2, (a > 0.5).sum(1))
    for b in range(B):
        hit = np.nonzero(a[b] > 0.5)[0]
        assert np.array_equal(pairs[b, :len(hit), 1], hit)
