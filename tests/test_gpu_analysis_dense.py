"""GPU: the analysis consumers at dense activity -- the q_sae dense path's activity mask
(qsae_matryoshka_forward_dense_active) and the tensor-core co-activation product (qsae_coactivation_dense) -- against
float64 products on the GPU and the numpy restatement of the reference's analysis functions (oracle/analysis_oracle.py,
pinned to the reference by tests/golden/analysis_*.npz)."""
import numpy as np
import pytest
import torch

import quantizedsae_b200 as Q
from oracle import analysis_oracle as AO
from quantizedsae_b200 import _lib as L
from quantizedsae_b200 import analysis as AN
from quantizedsae_b200.inference import framework as FW
from quantizedsae_b200.sae.quantized_matryoshka import nested_sizes
from tests import analysis_common as AC
from tests.golden import cases

pytestmark = pytest.mark.gpu


def f64_product(mask):
    m = mask.double()
    return torch.matmul(m.t(), m).to(torch.int64)


def random_mask(K, H, density, gen, dev):
    m = (torch.rand((K, H), device=dev, generator=gen) < density).to(torch.bfloat16)
    if K > 2:
        m[0] = 0                        # an all-zero row
        m[-1] = 1                       # an all-one row
    return m.contiguous()


@pytest.mark.parametrize("H", [8, 832, 2056, 4096, 32768])
@pytest.mark.parametrize("K", [1, 127, 129, 4096])
def test_coactivation_dense_kernel(cuda_device, K, H):
    """cooc += M^T M bit for bit against a float64 product: densities 0, 1, 50, 100 %; two launches add; a non-zero
    starting matrix is read, modified and written once per element (no double count in the lower triangle); counts are
    the diagonal; two runs are bit-identical."""
    if H == 32768 and K == 4096:
        densities = [0.5]
    elif H == 32768:
        densities = [0.01, 0.5]
    else:
        densities = [0.0, 0.01, 0.5, 1.0]
    gen = torch.Generator(device=cuda_device).manual_seed(K * 7 + H)
    for d in densities:
        m1 = random_mask(K, H, d, gen, cuda_device)
        m2 = random_mask(K, H, d, gen, cuda_device)
        start = torch.randint(-1000, 1000, (H, H), device=cuda_device, generator=gen, dtype=torch.int32)
        start = start + start.t()                                   # symmetric, as an accumulator always is
        runs = []
        for _ in range(2):
            cooc = start.clone()
            counts = torch.arange(H, device=cuda_device, dtype=torch.int64)
            L.coactivation_dense(m1, cooc, counts)
            ref1 = start.to(torch.int64) + f64_product(m1)
            assert torch.equal(cooc.to(torch.int64), ref1), f"K={K} H={H} density={d}: one launch"
            assert torch.equal(counts, torch.arange(H, device=cuda_device) + m1.double().sum(0).to(torch.int64))
            L.coactivation_dense(m2, cooc, counts)
            assert torch.equal(cooc.to(torch.int64), ref1 + f64_product(m2)), f"K={K} H={H} density={d}: two launches"
            runs.append(cooc)
            del ref1
        assert torch.equal(runs[0], runs[1])
        del runs, start
        torch.cuda.empty_cache()


def test_coactivation_dense_rejects_bad_shapes(cuda_device):
    m = torch.zeros((4, 12), dtype=torch.bfloat16, device=cuda_device)
    with pytest.raises(L.QsaeError, match="multiple of 8"):
        L.coactivation_dense(m, torch.zeros((12, 12), dtype=torch.int32, device=cuda_device))


# ---- the analysis consumers on the dense route against the oracle

def qsae_model(cfg, inp, dev):
    m = Q.QuantizedMatryoshkaSAE(cfg["D"], cfg["H"], 32, cfg["abs_range"], cfg["n_bits"], cfg["allow_bias"])
    T = torch.from_numpy
    m.load_state_dict({"encoder.0.weight": T(inp["We"]), "encoder.0.bias": T(inp["be"]), "decoder.weight": T(inp["W"]),
                       "decoder.weight_mirror": T(inp["Wm"]), "decoder.bias": T(inp["bd"])}, strict=True)
    return m


def dense_case(name, exact, dev):
    """-> (kind, cfg, inp, SAEWrapper) with every q_sae of the model in the dense regime (dense_mode "always")."""
    if name == "rq_sae":
        cfg = dict(cases.RQSAE_CASES["rqsae_d64_h2048"], enc_bias=0.0)       # untrained stages: ~50 % active
        inp = AC.inputs("rq_sae", cfg)
        m = Q.ResidualQuantizedSAE(cfg["D"], cfg["H"], 32, cfg["abs_range"], cfg["n_bits"])
        m.load_state_dict({k: torch.from_numpy(v) for k, v in cases.rqsae_state_dict(inp, cfg["n_bits"]).items()}, strict=True)
        for s in m.saes:
            s.dense_mode, s.exact = "always", exact
        return "rq_sae", cfg, inp, FW.SAEWrapper(FW.SAE_REGISTRY["rq_sae"], m, dev)
    if name == "d64_h1024":
        cfg = dict(cases.QSAE_CASES["qsae_d64_h1024_dense_nobias"])
    else:
        cfg = dict(D=512, H=4096, n_bits=4, abs_range=4.0, B=48, enc_bias=0.0, allow_bias=True, seed=71)
    cfg["bf16"] = not exact          # fast mode: bf16-representable operands, so its products are exact as well
    inp = cases.qsae_inputs(cfg)
    m = qsae_model(cfg, inp, dev)
    m.dense_mode, m.exact = "always", exact
    return "q_sae", cfg, inp, FW.SAEWrapper(FW.SAE_REGISTRY["q_sae"], m, dev)


def last_paths(sae):
    model = sae.model
    return [s.last_path for s in model.saes] if isinstance(model, Q.ResidualQuantizedSAE) else [model.last_path]


@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("name", ["d64_h1024", "d512_h4096", "rq_sae"])
def test_dense_route_matches_oracle(cuda_device, name, exact):
    kind, cfg, inp, sae = dense_case(name, exact, cuda_device)
    H = cfg["H"]
    loader = [torch.from_numpy(b) for b in AC.batches(inp["x"])]
    rng = np.random.default_rng(5)
    tok = torch.from_numpy(rng.integers(0, 50000, size=(inp["x"].shape[0] // AC.TOKENS_PER_CONTEXT + 1,
                                                         AC.TOKENS_PER_CONTEXT)))
    st = AN.compute_activation_stats(sae, loader, token_ids=tok, tokens_per_context=AC.TOKENS_PER_CONTEXT, device="cuda")
    assert last_paths(sae) == ["dense"] * len(last_paths(sae))
    mse = AN.compute_reconstruction_error(sae, loader, device="cuda")
    mse_lv = AN.compute_reconstruction_error_by_level(sae, loader, device="cuda").numpy()
    l0 = AN.compute_l0_by_level(sae, loader, device="cuda").numpy()
    gpu_mask = torch.cat([AN._activation_mask(sae, b) for b in loader]).numpy()
    assert gpu_mask.shape == (inp["x"].shape[0], H)
    one = AN.analyze_dataset(sae, loader, token_ids=tok, tokens_per_context=AC.TOKENS_PER_CONTEXT, device="cuda")
    assert last_paths(sae) == ["dense"] * len(last_paths(sae))

    ref = AO.analyze(kind, cfg, inp, [b.numpy() for b in loader], tok.numpy(), AC.TOKENS_PER_CONTEXT)
    # the mask: the oracle's, except decisions within accumulation noise of the threshold (counted and bounded)
    flips = int((gpu_mask != ref["mask"]).sum())
    if kind == "q_sae" or exact:
        assert flips <= max(2, gpu_mask.size // 20000), f"{flips} activity decisions differ from the oracle"
        assert abs(mse - ref["mse"]) <= 2e-5 * ref["mse"]
        np.testing.assert_allclose(mse_lv, ref["mse_by_level"], rtol=2e-5)
    else:
        # fast mode casts each stage's fp32 residual to bf16: decisions near the threshold follow that rounding
        assert flips <= gpu_mask.size // 50
    # counts, co-activation, L0 and tokens per feature: exactly the oracle formulas on the GPU's own mask
    mi = gpu_mask.astype(np.int64)
    np.testing.assert_array_equal(st["activation_counts"].numpy(), mi.sum(0))
    np.testing.assert_array_equal(st["coactivation"].numpy().astype(np.int64), mi.T @ mi)
    if kind == "q_sae":
        edges = np.cumsum([0] + list(cases_sizes(cfg)))
    else:
        edges = np.cumsum([0] + list(sae.model.sae_hidden_dims))
    level_sums = np.array([mi[:, a:b].sum() for a, b in zip(edges[:-1], edges[1:])], dtype=np.float64)
    np.testing.assert_array_equal(np.rint(l0 * mi.shape[0]), level_sums)          # the active counts, exactly
    np.testing.assert_allclose(l0, level_sums / mi.shape[0], rtol=1e-15)         # / tokens on the device: last bit
    rows, feats = np.nonzero(gpu_mask)
    tpf = [[] for _ in range(H)]
    toks = tok.numpy()[rows // AC.TOKENS_PER_CONTEXT, rows % AC.TOKENS_PER_CONTEXT]
    for f, t in zip(feats.tolist(), toks.tolist()):
        tpf[f].append(int(t))
    assert st["tokens_per_feature"] == tpf
    assert one["tokens_per_feature"] == tpf
    assert torch.equal(one["activation_counts"], st["activation_counts"]) and torch.equal(one["coactivation"], st["coactivation"])
    assert abs(one["mse_final"] - mse) <= 1e-12 * mse


def cases_sizes(cfg):
    return nested_sizes(cfg["H"], cfg["n_bits"])


def test_forward_dense_active_rejects_unaligned_hidden_dim(cuda_device):
    m = Q.QuantizedMatryoshkaSAE(64, 1020, 32, n_bits=2).to(cuda_device)
    with pytest.raises(ValueError, match="multiple of 8"):
        m.forward_dense_active(torch.randn((4, 64), device=cuda_device))


def untrained_qsae(dev, seed=92):
    cfg = dict(D=512, H=32768, n_bits=4, abs_range=4.0, B=8, enc_bias=0.0, bf16=False, allow_bias=True, seed=seed)
    inp = cases.qsae_inputs(cfg)
    return qsae_model(cfg, inp, dev).to(dev).eval()


def test_baseline_shape_untrained_qsae(cuda_device):
    """q_sae 512 -> 32768, untrained (~16 k active per row), 2 x 4096 tokens through compute_activation_stats: the sparse
    lists overflow and the batches take the dense route. The 4.3 GB matrix equals a float64 product of the returned
    masks (row blocks); its diagonal equals the counts and its sum equals sum of (row activity)^2."""
    m = untrained_qsae(cuda_device)
    sae = FW.SAEWrapper(FW.SAE_REGISTRY["q_sae"], m, cuda_device)
    g = torch.Generator(device=cuda_device).manual_seed(11)
    xs = [torch.randn((4096, 512), device=cuda_device, generator=g) for _ in range(2)]
    masks = []
    for x in xs:
        r = AN.forward_with_active(sae, x)
        assert m.last_path == "dense" and r["active_idx"] is None
        masks.append(r["active_mask"].clone())
    m._regime = None
    acc = AN._StatsAccumulator(32768, cuda_device, None, 1)
    for x in xs:
        acc.add(AN.forward_with_active(sae, x))
    M = torch.cat(masks)
    act = M.double().sum(1)
    assert 14000 < float(act.mean()) < 19000
    assert torch.equal(acc.counts, M.double().sum(0).to(torch.int64))
    assert torch.equal(torch.diagonal(acc.cooc).to(torch.int64), acc.counts)
    assert int(acc.cooc.sum(dtype=torch.int64)) == int((act.to(torch.int64) ** 2).sum())
    Md = M.double()
    for r0 in range(0, 32768, 4096):
        blk = torch.matmul(Md[:, r0:r0 + 4096].t(), Md).to(torch.int64)
        assert torch.equal(acc.cooc[r0:r0 + 4096].to(torch.int64), blk), f"rows {r0}.."


def test_mixed_sparse_and_dense_batches(cuda_device):
    """One sparse-regime batch and one overflowing batch in one compute_activation_stats run equal the sum of the two
    single-batch runs (list route and mask route add into the same accumulators)."""
    D, H, B = 512, 32768, 256
    torch.manual_seed(5)
    with torch.device(cuda_device):
        m = Q.QuantizedMatryoshkaSAE(D, H, 32, abs_range=4.0, n_bits=4)
    with torch.no_grad():
        m.encoder[0].bias.fill_(-0.543)
    m.eval()
    sae = FW.SAEWrapper(FW.SAE_REGISTRY["q_sae"], m, cuda_device)
    x = torch.randn((B, D), device=cuda_device)
    xbig = x * 40.0 + 30.0 * torch.sign(m.encoder[0].weight.detach()[:2000].sum(0))
    tok = torch.arange(2 * B, dtype=torch.int64).reshape(-1, 4)

    def stats(batches, first_row=0):
        m._regime = None
        t = tok.reshape(-1)[first_row:].reshape(-1, 4)
        return AN.compute_activation_stats(sae, batches, token_ids=t, tokens_per_context=4, device="cuda")

    s_small = stats([x])
    assert m.last_path == "sparse"
    s_big = stats([xbig], B)
    assert m.last_path == "dense"
    both = stats([x, xbig])
    assert m.last_path == "dense"
    assert torch.equal(both["activation_counts"], s_small["activation_counts"] + s_big["activation_counts"])
    assert torch.equal(both["coactivation"], s_small["coactivation"] + s_big["coactivation"])
    assert both["tokens_per_feature"] == [a + b for a, b in zip(s_small["tokens_per_feature"], s_big["tokens_per_feature"])]


@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("H", [832, 2056, 32768])
def test_mask_from_both_operand_producers(cuda_device, tuning, H, exact):
    """The mask is bit-identical from the fused encoder epilogue (level boundaries on the 128-grid) and from the
    streaming operand kernel. It records activity, not A != 0: a latent whose decoder row is all zero (no effect on the
    reconstruction) is still active when its pre-activation is, as in the reference's `encoder(x) > 0.5`."""
    cfg = dict(D=512, H=H, n_bits=4, abs_range=4.0, B=300, enc_bias=0.0, bf16=not exact, allow_bias=True, seed=H + 1)
    inp = cases.qsae_inputs(cfg)
    # latent 5: S = -S_mirror everywhere, so its row of T = S + S_mirror is 0; latent 6: an encoder row that makes it
    # active on every row (z = 1)
    inp["Wm"][5] = -inp["W"][5]
    inp["We"][6] = 0.0
    inp["be"][6] = 1.0
    m = qsae_model(cfg, inp, cuda_device).to(cuda_device).eval()
    m.exact = exact
    x = torch.from_numpy(inp["x"]).to(cuda_device)
    with torch.no_grad():
        r1 = m.forward_dense_active(x)
        tuning("QSAE_DENSE_STEP_FUSED", "0")
        r0 = m.forward_dense_active(x)
    assert torch.equal(r1["active_mask"], r0["active_mask"])
    assert torch.equal(r1["level_counts"], r0["level_counts"])
    assert all(torch.equal(a, b) for a, b in zip(r1["reconstruction_levels"], r0["reconstruction_levels"]))
    mask = r1["active_mask"]
    assert set(torch.unique(mask.float()).tolist()) <= {0.0, 1.0}
    assert bool((mask[:, 6] == 1).all())                         # z = 1 >= threshold on every row
    assert int(mask.double().sum()) == int(r1["level_counts"].sum())
    # latent 5 is decided by its pre-activation alone, as in the reference (encoder(x) > 0.5)
    z5 = torch.from_numpy(inp["x"].astype(np.float64) @ inp["We"][5].astype(np.float64) + float(inp["be"][5]))
    agree = (mask[:, 5].cpu() == 1) == (z5 > 0)
    assert int((~agree).sum()) <= 1 and int(mask[:, 5].sum()) > 0
