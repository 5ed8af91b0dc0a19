"""Pin the CPU oracle (oracle/qsae_oracle.py) against outputs of the unmodified reference.

The fixtures under tests/golden/ were produced by tests/golden/make_golden.py, which runs the
reference's own nn.Modules. These tests need no GPU and no copy of the reference.
"""
import numpy as np
import pytest

from oracle import qsae_oracle as O
from tests.golden import cases

# float64 sparse accumulation vs the reference's dense float32 matmul
RECON_RTOL = 2e-5
RECON_ATOL_FRAC = 2e-6  # x rms(recon)


def _load(golden_dir, name):
    return np.load(golden_dir / f"{name}.npz")


def _close(a, b, rtol=RECON_RTOL):
    rms = float(np.sqrt(np.mean(np.square(b, dtype=np.float64)))) + 1e-30
    np.testing.assert_allclose(a, b, rtol=rtol, atol=RECON_ATOL_FRAC * rms + 1e-6)


def test_readme_known_answer(golden_dir):
    g = _load(golden_dir, "misc")
    # README.md:100 -- MSB-first [1,0,1,0] is LSB-first storage [0,1,0,1]
    logits = np.array([[-110.0, 110.0, -110.0, 110.0]], dtype=np.float32)
    iw = O.dequant_hard(logits, 4)
    assert iw[0, 0] == -6 == int(g["readme_int"])
    assert iw[0, 0] * (4.0 / 8) == -3.0 == float(g["readme_value"])


def test_all_sixteen_nibbles(golden_dir):
    g = _load(golden_dir, "misc")
    pat = np.array([[(v >> i) & 1 for i in range(4)] for v in range(16)], dtype=np.float32)
    logits = np.where(pat.reshape(1, 64) > 0, 110.0, -110.0).astype(np.float32)
    iw = O.dequant_hard(logits, 4)[0]
    assert iw.tolist() == g["nibble_ints"].tolist()
    assert iw.tolist() == [v if v < 8 else v - 16 for v in range(16)]
    # packed layout round trip
    packed = O.pack_nibbles(iw[None, :])
    assert O.unpack_nibbles(packed)[0].tolist() == iw.tolist()


@pytest.mark.parametrize("key", ["32768_4", "32768_8", "1048576_4", "2048_4", "32768_1", "1024_3", "4096_4"])
def test_matryoshka_level_sizes(golden_dir, key):
    g = _load(golden_dir, "misc")
    H, nb = (int(v) for v in key.split("_"))
    assert O.matryoshka_level_sizes(H, nb) == g[f"sizes_{key}"].tolist()


def test_level_sizes_headline():
    assert O.matryoshka_level_sizes(32768, 4) == [4096, 4096, 8192, 16384]


@pytest.mark.parametrize("name", list(cases.BSAE_CASES))
def test_bsae_matches_reference(golden_dir, name):
    cfg = cases.BSAE_CASES[name]
    g = _load(golden_dir, name)
    inp = cases.bsae_inputs(cfg)
    assert cases.checksum(inp) == str(g["input_sha"])
    k = O.bsae_k(cfg["H"])
    assert k == int(g["k"])
    # integer dictionary: bit exact
    iw = O.dequant_hard(inp["logits"], cfg["n_bits"])
    assert cases.int_weights_match(iw, g)
    # soft dictionary rows
    sw = O.dequant_soft(inp["logits"], cfg["n_bits"])
    np.testing.assert_allclose(sw[:4], g["soft_weights_row0"], rtol=1e-5, atol=1e-5)  # fp32 sum order
    # forward: reference uses soft bits; with polarised logits soft == hard exactly
    for mode in (["soft", "hard"] if cfg["polar"] else ["soft"]):
        vals, idx, recon, pol = O.bsae_forward(
            inp["x"], inp["We"], inp["be"], inp["logits"], inp["bd"],
            n_bits=cfg["n_bits"], gamma=cfg["gamma"], k=k, mode=mode)
        assert np.array_equal(idx, g["latent_idx"]), "top-k index sets/order differ"
        np.testing.assert_allclose(vals, g["latent_vals"], rtol=1e-5, atol=1e-6)
        _close(recon, g["recon"])
        assert pol == pytest.approx(float(g["polarize"]), rel=1e-5, abs=1e-9)
    if cfg["polar"]:
        assert float(g["polarize"]) == 0.0


@pytest.mark.parametrize("name", [n for n, c in cases.BSAE_CASES.items() if c["H"] <= 8192])
def test_timed_cpu_arm_matches_reference_fixture(golden_dir, name):
    """bench.py's CPU arm (`--impl reference`, `cpu_baseline`) times O.bsae_forward_dense_port_torch, the reference's own
    op sequence (sae/binary.py:91-103 + :24-47) on torch CPU tensors. Pin it to the outputs of the unmodified reference
    stored in the fixtures: the dense latent is bit-equal to the reference's (its k non-zeros at the reference's indices
    with the reference's values), reconstruction and polarize loss are equal up to fp32 summation order (the bits of
    a CPU matmul depend on the host's thread count and instruction set, so stored outputs can only pin them this far)."""
    import torch

    cfg = cases.BSAE_CASES[name]
    g = _load(golden_dir, name)
    inp = cases.bsae_inputs(cfg)
    k = int(g["k"])
    t = {n: torch.from_numpy(v) for n, v in inp.items()}
    lat, recon, pol = O.bsae_forward_dense_port_torch(t["x"], t["We"], t["be"], t["logits"], t["bd"], n_bits=cfg["n_bits"],
                                                      gamma=cfg["gamma"], k=k)
    ref_lat = np.zeros((cfg["B"], cfg["H"]), dtype=np.float32)
    np.put_along_axis(ref_lat, g["latent_idx"].astype(np.int64), g["latent_vals"], axis=1)
    assert np.array_equal(lat.numpy(), ref_lat)
    _close(recon.numpy(), g["recon"])
    assert float(pol) == pytest.approx(float(g["polarize"]), rel=1e-5, abs=1e-9)


def test_bsae_state_dict_layout(golden_dir):
    g = _load(golden_dir, "bsae_polar_d64_h2048")
    assert g["state_keys"].tolist() == ["decoder.bias", "decoder.weight", "encoder.0.bias", "encoder.0.weight"]
    assert g["state_shapes"].tolist() == ["(64,)", "(2048, 256)", "(2048,)", "(2048, 64)"]


@pytest.mark.parametrize("name", list(cases.BASELINE_CASES))
def test_baseline_matches_reference(golden_dir, name):
    cfg = cases.BASELINE_CASES[name]
    g = _load(golden_dir, name)
    inp = cases.baseline_inputs(cfg)
    assert cases.checksum(inp) == str(g["input_sha"])
    vals, idx, recon = O.baseline_forward(inp["x"], inp["We"], inp["be"], inp["Wd"], inp["bd"], k=int(g["k"]))
    assert np.array_equal(idx, g["latent_idx"])
    np.testing.assert_allclose(vals, g["latent_vals"], rtol=1e-5, atol=1e-6)
    _close(recon, g["recon"])


@pytest.mark.parametrize("name", list(cases.TSAE_CASES))
def test_tsae_matches_reference(golden_dir, name):
    cfg = cases.TSAE_CASES[name]
    g = _load(golden_dir, name)
    inp = cases.tsae_inputs(cfg)
    assert cases.checksum(inp) == str(g["input_sha"])
    h, recon = O.tsae_forward(inp["x"], inp["We"], inp["be"], inp["Wd"])
    np.testing.assert_allclose(h, g["h"], rtol=1e-5, atol=1e-6)
    _close(recon, g["recon"], rtol=1e-4)
    # the reference grows a buffer in its state_dict after the first forward (ternary.py:21-22)
    assert "decoder.input_activations" not in g["state_keys"].tolist()
    assert "decoder.input_activations" in g["state_keys_after_forward"].tolist()
    T = O.ternarize(inp["Wd"])
    assert set(np.unique(T).tolist()) <= {-1, 0, 1}
    assert 0.25 < (T != 0).mean() < 0.35


@pytest.mark.parametrize("name", list(cases.QSAE_CASES))
def test_qsae_matches_reference(golden_dir, name):
    cfg = cases.QSAE_CASES[name]
    g = _load(golden_dir, name)
    inp = cases.qsae_inputs(cfg)
    assert cases.checksum(inp) == str(g["input_sha"])
    groups, result, act = O.qsae_forward(
        inp["x"], inp["We"], inp["be"], inp["W"], inp["Wm"], inp["bd"],
        n_bits=cfg["n_bits"], abs_range=cfg["abs_range"], allow_bias=cfg["allow_bias"])
    assert O.matryoshka_level_sizes(cfg["H"], cfg["n_bits"]) == g["level_sizes"].tolist()
    assert np.array_equal(np.packbits(act, axis=1), g["active"])
    np.testing.assert_allclose(groups, g["latent_group"], rtol=1e-6, atol=1e-6)
    for i in range(cfg["n_bits"]):
        _close(result[i], g["result"][i])


def test_sigmoid_band_documented():
    """Outside |w| < 2.5e-7 the strict threshold is exactly w > 0; inside, it is implementation
    dependent (float32 logistic rounds to 0.5) -- parity inputs stay out of the band."""
    w = np.array([-1.0, -1e-6, -2.5e-7, 2.5e-7, 1e-6, 1.0, 0.0], dtype=np.float32)
    assert O.hard_bits(w).tolist() == [False, False, False, True, True, True, False]
    assert not O.hard_bits(np.array([1e-9], dtype=np.float32))[0]


def test_topk_tie_rule():
    z = np.array([[1, 3, 3, 3, 3, 0, 3]], dtype=np.float32)
    vals, idx = O.topk_rows(z, 2)
    assert idx.tolist() == [[1, 2]]            # lowest index among equals (stable sort order)
    z = np.zeros((1, 1024), dtype=np.float32)
    z[0, 512] = 1
    assert O.topk_rows(z, 4)[1].tolist() == [[512, 0, 1, 2]]
    with pytest.raises(RuntimeError):
        O.topk_rows(z, 2048)


@pytest.mark.parametrize("name", list(cases.RQSAE_CASES))
def test_rqsae_matches_reference(golden_dir, name):
    cfg = cases.RQSAE_CASES[name]
    g = np.load(golden_dir / f"{name}.npz")
    inp = cases.rqsae_inputs(cfg)
    assert cases.checksum(inp) == str(g["input_sha"])
    stages = [(inp[f"We{i}"], inp[f"be{i}"], inp[f"W{i}"], inp[f"Wm{i}"], inp[f"bd{i}"]) for i in range(cfg["n_bits"])]
    groups, recons = O.rqsae_forward(inp["x"], stages, abs_range=cfg["abs_range"])
    assert O.matryoshka_level_sizes(cfg["H"], cfg["n_bits"]) == g["stage_sizes"].tolist()
    np.testing.assert_allclose(groups, g["latent_group"], rtol=1e-6, atol=1e-6)
    for t in range(cfg["n_bits"]):
        rms = float(np.sqrt(np.mean(g["recon"][t].astype(np.float64) ** 2)))
        np.testing.assert_allclose(recons[t], g["recon"][t], rtol=2e-5, atol=2e-5 * rms)
