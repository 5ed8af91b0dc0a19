"""Every input width the encoder keys on, against float64: each K-chunk count of encode_topk_kernel (KC = ceil(D / 64),
1 to 8), a partial last chunk (which TMA zero-fills) at every count, and the pair variants above D = 448 with a partial
chunk; then the sparse decoders at every (words per lane, full-width) pair and row-chunk count.

The rules are tests/test_gpu_large_batch.py's (the band (D + 1) 2^-23 S, the selection and swap rules, the decode
bounds, the prior-path counts). What is added here is the width axis, and a record of the kernels each case launched
(torch.profiler): every encoder case asserts the encode_topk_kernel<KC, DENSE, CL, SEL> instantiations it expects, so a
width that fell back to another kernel fails.

Widths. W8 (b_sae, baseline_sae, t_sae; D % 8 == 0): every chunk count, each with a partial last chunk, the full 6- and
7-chunk widths 384 and 448, and 456 / 504 above the pair threshold (D > 448). q_sae (D % 16 == 0) is covered by the
extra shapes of test_gpu_matryoshka_levels.py.

Schedules (csrc/encode_topk_sm100.cu, qsae_api.cu). Away from D = 256 and 512 the prior path runs a separate sample
pre-pass, which is the generic kernel (SEL = -1) on the (split, row block) grid, before the prior-threshold sweep (the
kernel compiled for mode 4 alone, SEL = 4, unless QSAE_ENCODE_SPECIALISED=0). The sweep's CL: 3 (pair range schedule)
at B = 4096 above D = 448, 0 on the single-CTA range schedule (B = 333) and on the grid below B = 16384, 1 (multicast
pair) at B >= 16384 above D = 448, 2 with QSAE_ENCODE_CLUSTER=2; the pre-pass follows the grid's choice. The b_sae
reconstruction runs through decode_int4_kernel (the fused merge-and-decode exists at D = 512 only).
"""
import re

import pytest
import torch

import quantizedsae_b200 as Q
from quantizedsae_b200 import _lib as L
from tests import test_gpu_bsae_train_det as DET
from tests.test_gpu_large_batch import (TopkStats, check_bsae_batch, check_decode, enc_case, int4_dictionary,
                                        make_bsae, prior_counts, prior_plan, reference_chunks, structure_errors,
                                        value_ratio)
from tests.test_gpu_sweep_specialised import assert_same_bits
from tests.test_gpu_tsae_train import TOL_EXACT, TOL_FAST

pytestmark = pytest.mark.gpu

W8 = [24, 72, 136, 200, 264, 328, 384, 392, 448, 456, 504]
PAIR = [456, 504]                               # above the pair threshold, with a partial last chunk
PARTIAL = [D for D in W8 if D % 64]
H_BIG = 32768


def report(msg):
    print(f"[widths] {msg}")


def kc(D):
    return -(-D // 64)


# ------------------------------------------------------------------------------------------
# launched kernels
# ------------------------------------------------------------------------------------------
_B = r"(true|false|0|1)"
ENC_RE = re.compile(r"encode_topk_kernel<(\d+),\s*" + _B + r",\s*(-?\d+),\s*(-?\d+)>")
DEC4_RE = re.compile(r"decode_int4_kernel<(\d+),\s*" + _B + r",\s*" + _B + r",\s*" + _B + ">")
ROWS_RE = re.compile(r"decode_rows_kernel<([^,<>]+),\s*(\d+)>")


def _flag(s):
    return s in ("true", "1")


def launched(fn):
    """fn() under torch.profiler (CUDA activity only) -> (fn's result, kernels) where kernels holds the sets "enc"
    (KC, DENSE, CL, SEL), "dec4" (WPL, FULL, RANGE, WIDE), "rows" (element type, NCH) and "names"."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        out = fn()
        torch.cuda.synchronize()
    names = {ev.key for ev in p.key_averages()}
    got = {"enc": set(), "dec4": set(), "rows": set(), "names": names}
    for n in names:
        for m in ENC_RE.finditer(n):
            got["enc"].add((int(m[1]), _flag(m[2]), int(m[3]), int(m[4])))
        for m in DEC4_RE.finditer(n):
            got["dec4"].add((int(m[1]), _flag(m[2]), _flag(m[3]), _flag(m[4])))
        for m in ROWS_RE.finditer(n):
            got["rows"].add((m[1].strip(), int(m[2])))
    return out, got


def fmt(enc):
    return ", ".join(f"<{a}, {'true' if b else 'false'}, {c}, {d}>" for a, b, c, d in sorted(enc))


def test_kernel_name_parser():
    """The parser reads both ways a bool template argument prints."""
    n = "void qsae::(anonymous namespace)::encode_topk_kernel<8, false, 3, 4>(CUtensorMap_st, CUtensorMap_st)"
    assert [(int(m[1]), _flag(m[2]), int(m[3]), int(m[4])) for m in ENC_RE.finditer(n)] == [(8, False, 3, 4)]
    n = "encode_topk_kernel<3, 1, 0, -1>"
    assert [(int(m[1]), _flag(m[2]), int(m[3]), int(m[4])) for m in ENC_RE.finditer(n)] == [(3, True, 0, -1)]
    n = "qsae::decode_int4_kernel<2, false, true, false>(float const*)"
    assert [(int(m[1]), _flag(m[2]), _flag(m[3]), _flag(m[4])) for m in DEC4_RE.finditer(n)] == [(2, False, True, False)]
    assert ROWS_RE.search("decode_rows_kernel<signed char, 4>(float const*)").groups() == ("signed char", "4")


# ------------------------------------------------------------------------------------------
# b_sae forward
# ------------------------------------------------------------------------------------------
def bsae_setup(dev, D, B, H=H_BIG, k=32, n_bits=4, exact=False, seed=0):
    x, W, b = enc_case(B, H, D, seed, exact, dev)
    m = make_bsae(W, b, D, H, n_bits, k, exact, dev, seed=seed + 1)
    return m, x, W, b


def bsae_call(m, x, W, b, k, exact, n_bits):
    dec = m.decoder
    return lambda: L.bsae_forward(x, m._w_bf16(), W if exact else None, b, k, dec._packed()[0], n_bits,
                                  dec.quantization_step, dec.bias.detach(), exact=exact, want_flags=True,
                                  sample=m._sample())


def wpl(D):
    return 1 if D <= 256 else (2 if D <= 512 else 4)


def nch(D):
    return 1 if D <= 128 else (2 if D <= 256 else (4 if D <= 512 else 8))


def run_bsae(m, x, W, b, k, exact, n_bits, capfd, cl_main, cl_pre=0, sel=4):
    """One profiled forward: the prior path ran with prior_plan's k_sel and m, through the expected encoder and decoder
    instantiations -> (outputs, encoder set)."""
    H, D = W.shape
    B = x.shape[0]
    capfd.readouterr()
    out, got = launched(bsae_call(m, x, W, b, k, exact, n_bits))
    c = prior_counts(capfd)
    k_sel, mm = prior_plan(H, k, exact, m._sample()[0].shape[0])
    assert mm > 0 and (c["B"], c["k_sel"], c["m"]) == (B, k_sel, mm), f"not the planned prior path: {c}"
    want = {(kc(D), False, cl_pre, -1), (kc(D), False, cl_main, sel)}
    assert got["enc"] == want, f"D={D} B={B}: launched {fmt(got['enc'])}, expected {fmt(want)}"
    if n_bits <= 4:
        assert got["dec4"] == {(wpl(D), D == 256, False, k > 128)}, f"D={D}: int4 decoders {got['dec4']}"
    else:
        assert {n for _, n in got["rows"]} == {nch(D)}, f"D={D}: row decoders {got['rows']}"
    return out, got["enc"]


BSAE_CASES = {   # name: (B, k, exact, QSAE_ENCODE_RANGE)
    "b4096-fast": (4096, 32, False, None),      # range schedule; the pair range schedule (CL = 3) above D = 448
    "b4096-exact": (4096, 32, True, None),
    "b333": (333, 32, False, None),             # single-CTA range schedule, a partial row block
    "b1000-grid": (1000, 32, False, 0),         # the (split, row block) grid
    "k65": (4096, 65, False, None),             # int(0.002 H) at H = 32768
}


@pytest.mark.parametrize("case", list(BSAE_CASES))
@pytest.mark.parametrize("D", W8)
def test_bsae_forward_every_row(cuda_device, tuning, capfd, D, case):
    B, k, exact, rng = BSAE_CASES[case]
    tuning("QSAE_DEBUG_LARGE", 1)
    if rng is not None:
        tuning("QSAE_ENCODE_RANGE", rng)
    m, x, W, b = bsae_setup(cuda_device, D, B, k=k, exact=exact, seed=D + B + k + exact)
    cl = 3 if (D > 448 and B == 4096) else 0
    out, enc = run_bsae(m, x, W, b, k, exact, 4, capfd, cl)
    what = f"b_sae D={D} {case} {fmt(enc)}"
    _, out2, vw, dw = check_bsae_batch(m, x, W, b, k, exact, 4, what, capfd)
    assert_same_bits(out, out2)
    report(f"{what}: value err/band {vw:.3g}, decode err/bound {dw:.3g}")


@pytest.mark.parametrize("D", W8)
def test_bsae_generic_sweep_same_bits(cuda_device, tuning, capfd, D):
    """QSAE_ENCODE_SPECIALISED=0: the prior-threshold sweep on the generic kernel gives the same bits."""
    tuning("QSAE_DEBUG_LARGE", 1)
    B, k = 4096, 32
    m, x, W, b = bsae_setup(cuda_device, D, B, seed=D + B + k)
    cl = 3 if D > 448 else 0
    spec, _ = run_bsae(m, x, W, b, k, False, 4, capfd, cl)
    tuning("QSAE_ENCODE_SPECIALISED", 0)
    gen, enc = run_bsae(m, x, W, b, k, False, 4, capfd, cl, sel=-1)
    assert_same_bits(spec, gen)
    report(f"b_sae D={D} generic sweep {fmt(enc)}: same bits as SEL = 4")


@pytest.mark.parametrize("D", PAIR)
def test_bsae_pair_variants_every_row_and_same_bits(cuda_device, tuning, capfd, D):
    """Above D = 448 with a partial last chunk: the multicast grid (B = 16384), the sparse cta_group::2 pair (range
    schedule off) and the pair range schedule (B = 4096), each against the single-CTA kernel's bits."""
    tuning("QSAE_DEBUG_LARGE", 1)
    k = 32
    # multicast pair, then the same batch on single CTAs
    m, x, W, b = bsae_setup(cuda_device, D, 16384, seed=D + 16384)
    mc, enc = run_bsae(m, x, W, b, k, False, 4, capfd, cl_main=1, cl_pre=1)
    _, out2, vw, dw = check_bsae_batch(m, x, W, b, k, False, 4, f"b_sae D={D} B=16384 {fmt(enc)}", capfd)
    assert_same_bits(mc, out2)
    tuning("QSAE_ENCODE_CLUSTER", 0)
    single, _ = run_bsae(m, x, W, b, k, False, 4, capfd, cl_main=0)
    assert_same_bits(mc, single)
    report(f"b_sae D={D} multicast {fmt(enc)}: value err/band {vw:.3g}, decode err/bound {dw:.3g}, same bits as CL = 0")
    # cta_group::2 pair on the grid
    tuning("QSAE_ENCODE_RANGE", 0)
    tuning("QSAE_ENCODE_CLUSTER", 2)
    m, x, W, b = bsae_setup(cuda_device, D, 1000, seed=D + 1000)
    pair, enc = run_bsae(m, x, W, b, k, False, 4, capfd, cl_main=2, cl_pre=2)
    _, out2, vw, dw = check_bsae_batch(m, x, W, b, k, False, 4, f"b_sae D={D} B=1000 {fmt(enc)}", capfd)
    assert_same_bits(pair, out2)
    tuning("QSAE_ENCODE_CLUSTER", 0)
    single, _ = run_bsae(m, x, W, b, k, False, 4, capfd, cl_main=0)
    assert_same_bits(pair, single)
    report(f"b_sae D={D} cta_group::2 {fmt(enc)}: value err/band {vw:.3g}, decode err/bound {dw:.3g}, same bits as CL = 0")
    # pair range schedule against the single-CTA range schedule
    tuning("QSAE_ENCODE_RANGE", 1)
    m, x, W, b = bsae_setup(cuda_device, D, 4096, seed=D + 4096 + k)
    rp, _ = run_bsae(m, x, W, b, k, False, 4, capfd, cl_main=3)
    tuning("QSAE_ENCODE_RANGE_PAIR", 0)
    single, _ = run_bsae(m, x, W, b, k, False, 4, capfd, cl_main=0)
    assert_same_bits(rp, single)
    report(f"b_sae D={D} pair range schedule: same bits as the single-CTA range schedule")


ODD_BSAE = {   # name: (H, n_bits)
    "h30000": (30000, 4),      # a partial last dictionary tile (no pair schedule either)
    "nb3": (H_BIG, 3),         # nibble packing at an odd bit count
    "nb8": (H_BIG, 8),         # int8 rows: the row decoder
}


@pytest.mark.parametrize("case", list(ODD_BSAE))
@pytest.mark.parametrize("D", [136, 392])
def test_bsae_partial_tile_and_bit_counts(cuda_device, tuning, capfd, D, case):
    H, nb = ODD_BSAE[case]
    tuning("QSAE_DEBUG_LARGE", 1)
    B, k = 4096, 32
    m, x, W, b = bsae_setup(cuda_device, D, B, H=H, n_bits=nb, seed=D + H + nb)
    out, enc = run_bsae(m, x, W, b, k, False, nb, capfd, cl_main=0)
    what = f"b_sae D={D} H={H} n_bits={nb} {fmt(enc)}"
    _, out2, vw, dw = check_bsae_batch(m, x, W, b, k, False, nb, what, capfd)
    assert_same_bits(out, out2)
    report(f"{what}: value err/band {vw:.3g}, decode err/bound {dw:.3g}")


@pytest.mark.parametrize("D", PARTIAL)
def test_band_catches_a_dropped_or_repeated_tail_chunk(cuda_device, tuning, capfd, D):
    """The float64 band has teeth at every partial-chunk width: the GPU's values break the band of a reference without
    the last K chunk, and of one that counts it twice, in most rows (and pass the true reference in every row)."""
    tuning("QSAE_DEBUG_LARGE", 1)
    B, k = 4096, 32
    m, x, W, b = bsae_setup(cuda_device, D, B, seed=D + B + k)
    (vals, idx, _, _), _ = run_bsae(m, x, W, b, k, False, 4, capfd, 3 if D > 448 else 0)
    c = 64 * (kc(D) - 1)
    shares = {}
    for name, xs, Ws in (("true", x, W), ("dropped", x[:, :c], W[:, :c]),
                         ("twice", torch.cat([x, x[:, c:]], 1), torch.cat([W, W[:, c:]], 1))):
        r = torch.cat([value_ratio(z, d, vals[r0:r0 + z.shape[0]], idx[r0:r0 + z.shape[0]])
                       for r0, z, d in reference_chunks(xs.contiguous(), Ws.contiguous(), b)])
        shares[name] = float((r > 1.0).double().mean())
    assert shares["true"] == 0.0
    assert shares["dropped"] > 0.5 and shares["twice"] > 0.5, shares
    report(f"D={D} (last chunk {D - c} wide): rows beyond the band without it {shares['dropped']:.3f}, "
           f"with it twice {shares['twice']:.3f}")


# ------------------------------------------------------------------------------------------
# baseline_sae forward
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact"])
@pytest.mark.parametrize("D", W8)
def test_baseline_forward_every_row(cuda_device, tuning, capfd, D, exact):
    B, H, k = 4096, H_BIG, 32
    tuning("QSAE_DEBUG_LARGE", 1)
    x, W, b = enc_case(B, H, D, 7 * D + exact, exact, cuda_device)
    torch.manual_seed(D)
    with torch.device(cuda_device):
        m = Q.BaselineSparseAutoencoder(D, H)
    with torch.no_grad():
        m.encoder[0].weight.copy_(W)
        m.encoder[0].bias.copy_(b)
    m.eval()
    m.return_dense, m.exact = False, exact
    capfd.readouterr()
    with torch.no_grad():
        (lat, recon), got = launched(lambda: m(x))
    c = prior_counts(capfd)
    k_sel, mm = prior_plan(H, k, exact, m._sample()[0].shape[0])
    assert mm > 0 and (c["B"], c["k_sel"], c["m"]) == (B, k_sel, mm)
    want = {(kc(D), False, 0, -1), (kc(D), False, 3 if D > 448 else 0, 4)}
    assert got["enc"] == want, f"launched {fmt(got['enc'])}, expected {fmt(want)}"
    assert got["rows"] == {("float", nch(D))}, got["rows"]
    vals, idx = lat.values, lat.indices
    what = f"baseline_sae D={D} {'exact' if exact else 'fast'} {fmt(got['enc'])}"
    assert structure_errors(vals, idx, H, m.last_flags, exact) == []
    rows = m.decoder.weight.detach().T.contiguous()
    st = TopkStats(what, k)
    dworst = 0.0
    for r0, z, delta in reference_chunks(x, W, b):
        r1 = r0 + z.shape[0]
        st.add(z, delta, vals[r0:r1], idx[r0:r1], r0=r0)
        for s0 in range(r0, r1, 2048):
            s1 = min(r1, s0 + 2048)
            dworst = max(dworst, check_decode(recon[s0:s1], vals[s0:s1], idx[s0:s1], rows, 1.0,
                                              m.decoder.bias.detach(), "rows", what, s0))
    vw = st.finish()
    report(f"{what}: value err/band {vw:.3g}, decode err/bound {dworst:.3g}")


@pytest.mark.parametrize("D", [136, 456])
def test_relu_flood_every_row(cuda_device, tuning, capfd, D):
    """ReLU with almost every pre-activation negative (bias -5, 20 latents raised): every row ends in a run of zeros,
    which the selection must order by index."""
    B, H, k = 150, 16384, 32
    tuning("QSAE_DEBUG_LARGE", 1)
    x, W, b = enc_case(B, H, D, 321 + D, False, cuda_device)
    b = b - 5.0
    b[torch.randperm(H, generator=torch.Generator().manual_seed(5))[:20].to(cuda_device)] += 10.0
    wb = L.cast_bf16(W)
    sample = L.prepare_sample(wb, b)
    capfd.readouterr()
    (vals, idx, flags), got = launched(lambda: L.encode_topk(x, wb, None, b, k, act=L.ACT_RELU, want_flags=True,
                                                             sample=sample))
    c = prior_counts(capfd)
    assert c["m"] > 0 and c["B"] == B
    want = {(kc(D), False, 0, -1), (kc(D), False, 0, 4)}
    assert got["enc"] == want, f"launched {fmt(got['enc'])}, expected {fmt(want)}"
    assert structure_errors(vals, idx, H) == []
    z, delta = next(reference_chunks(x, W, b, act=1, chunk=B))[1:]
    assert bool((torch.sort(z, 1, descending=True).values[:, k - 1] == 0).all()), "every row should end in zeros"
    st = TopkStats(f"relu flood D={D} {fmt(got['enc'])}", k)
    st.add(z, delta, vals, idx, stable=True)
    vw = st.finish(ties=True)
    report(f"relu flood D={D}: {c['block']} rows through the block select, value err/band {vw:.3g}")


# ------------------------------------------------------------------------------------------
# dense encoders
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("act", [0, 1], ids=["none", "relu"])
@pytest.mark.parametrize("D", W8)
def test_encode_dense_tc_every_entry(cuda_device, D, act):
    """The encoder's dense dump (the generic sparse kernel with debug_z) against the band, every entry."""
    B, H = 300, 4096
    x, W, b = enc_case(B, H, D, 11 * D + act, False, cuda_device)
    z, got = launched(lambda: L.encode_dense_tc(x, L.cast_bf16(W), b, act=act))
    want = {(kc(D), False, 0, -1)}
    assert got["enc"] == want, f"launched {fmt(got['enc'])}, expected {fmt(want)}"
    ref, delta = next(reference_chunks(x, W, b, act=act, chunk=B))[1:]
    ratio = float(((z.double() - ref).abs() / delta).max())
    assert ratio <= 1.0, f"D={D}: dense dump beyond the band, ratio {ratio:.3g}"
    report(f"encode_dense_tc D={D} act={act} {fmt(got['enc'])}: max err/band {ratio:.3g}")


TSAE_MODES = [(D, mode) for D in W8 for mode in ("fast", "exact")] + [(D, "fast-cl0") for D in PAIR]


@pytest.mark.parametrize("D,mode", TSAE_MODES, ids=[f"{D}-{m}" for D, m in TSAE_MODES])
def test_tsae_forward_every_entry(cuda_device, tuning, D, mode):
    """t_sae: the dense-epilogue kernel (fast; cta_group::2 pairs above D = 448 unless QSAE_ENCODE_CLUSTER=0) and the
    streamed-operand split kernel (exact, its chunk count a runtime argument). h against the float64 band: fast,
    (D + 1) 2^-23 S on bf16 operands; exact, six partial products of D terms each in one fp32 accumulator, plus the
    bias and the dropped cross terms (below 2^-26 S): (6 D + 3) 2^-23 S. recon against the float64 decode of the GPU's
    own h through the ternary dictionary, within test_gpu_tsae_train.py's fractions of S = |h| |T|^T."""
    B, H = 300, 4096
    exact = mode == "exact"
    if mode == "fast-cl0":
        tuning("QSAE_ENCODE_CLUSTER", 0)
    x, W, b = enc_case(B, H, D, 13 * D + exact, exact, cuda_device)
    g = torch.Generator(device=cuda_device).manual_seed(D)
    Wd = 0.4824 * torch.randn((D, H), device=cuda_device, generator=g)
    with torch.device(cuda_device):
        m = Q.TernarySparseAutoencoder(D, H)
    with torch.no_grad():
        m.encoder[0].weight.copy_(W)
        m.encoder[0].bias.copy_(b)
        m.decoder.weight.copy_(Wd)
    m.eval()
    m.exact = exact
    with torch.no_grad():
        (h, recon), got = launched(lambda: m(x))
    if exact:
        assert got["enc"] == set() and any("encode_dense_split_kernel" in n for n in got["names"]), got["names"]
        inst = "encode_dense_split_kernel"
    else:
        want = {(kc(D), True, 2 if (D > 448 and mode == "fast") else 0, -1)}
        assert got["enc"] == want, f"launched {fmt(got['enc'])}, expected {fmt(want)}"
        inst = fmt(want)
    ref, delta = next(reference_chunks(x, W, b, act=1, chunk=B))[1:]
    if exact:
        delta = delta * ((6 * D + 3) / (D + 1))
    hr = float(((h.double() - ref).abs() / delta).max())
    assert hr <= 1.0, f"D={D} {mode}: h beyond the band, ratio {hr:.3g}"
    T = torch.sign(Wd.double()) * (Wd.double().abs() >= 0.5)
    rref, S = h.double() @ T.T, h.double().abs() @ T.abs().T
    err = (recon.double() - rref).abs()
    assert not bool(((S == 0) & (err > 0)).any())
    frac = float((err / S.clamp_min(1e-300)).max())
    tol = TOL_EXACT if exact else TOL_FAST
    assert frac <= tol, f"D={D} {mode}: recon error {frac:.3g} S"
    report(f"t_sae D={D} {mode} {inst}: h err/band {hr:.3g}, recon err / S {frac:.3g} (allowed {tol:.3g})")


# ------------------------------------------------------------------------------------------
# the default (atomic) b_sae backward at the new widths, against the float64 bounds
# ------------------------------------------------------------------------------------------
ATOMIC_CASES = {name: DET.BOUND_CASES[name] for name in ("d136_h4096_3b_k32", "d456_h32768_4b_k32")}


@pytest.mark.parametrize("x_grad", [False, True])
@pytest.mark.parametrize("name", list(ATOMIC_CASES))
def test_atomic_backward_within_float64_bounds(cuda_device, name, x_grad):
    D, H, nb, k, B, gamma, skew = ATOMIC_CASES[name]
    m, x0 = DET._model(cuda_device, D, H, nb, k, B, seed=300 + list(ATOMIC_CASES).index(name), gamma=gamma, skew=skew)
    m.deterministic = False
    x = x0.clone().requires_grad_(x_grad)
    lat, g, gp = DET._step(m, x, 0.37)
    assert lat.indices.shape[1] == k
    DET._check(f"atomic {name} x_grad={x_grad}", m, x0, lat, g, gp, x.grad if x_grad else None)


# ------------------------------------------------------------------------------------------
# the sparse decoders alone
# ------------------------------------------------------------------------------------------
DEC_D = [8, 24, 200, 256, 264, 456, 512, 520, 776, 1000, 1024]
DEC_K = [1, 33, 128, 129, 4096]


def dec4_inst(D, aligned, rng, wide):
    full = D == 256 or (D in (512, 1024) and aligned)
    return (wpl(D), full, rng, wide)


@pytest.mark.parametrize("k", DEC_K)
@pytest.mark.parametrize("D", DEC_D)
def test_sparse_decoders(cuda_device, D, k):
    """decode_int4 / int8 / rows_f32 and their dictionary-shard variants against decode_bound, every row. The last
    value of a row is made 16 times the others so that dropping it breaks even the fp32 bound at k = 4096."""
    B, H = 37, 4096
    dev = cuda_device
    g = torch.Generator(device=dev).manual_seed(D * 7 + k)
    if k == H:
        idx = torch.stack([torch.randperm(H, device=dev, generator=g) for _ in range(B)]).int()
    else:
        idx = torch.randint(0, H, (B, k), device=dev, generator=g, dtype=torch.int32)
    vals = (0.25 + torch.rand((B, k), device=dev, generator=g)) * torch.where(
        torch.rand((B, k), device=dev, generator=g) < 0.5, -1.0, 1.0)
    vals[:, -1] *= 16.0
    bias = torch.randn(D, device=dev, generator=g)
    packed, ints4 = int4_dictionary(H, D, D + k, dev)
    rows8 = torch.randint(-128, 128, (H, D), device=dev, generator=g, dtype=torch.int8)
    rows32 = torch.randn((H, D), device=dev, generator=g)
    scale = 0.37
    wide = k > 128
    what = f"decoders D={D} k={k}"

    def rel(name, fn, dictionary, kind, want_dec4=None, want_rows=None, v=vals, i=idx):
        out, got = launched(fn)
        if want_dec4 is not None:
            assert got["dec4"] == {want_dec4}, f"{what} {name}: {got['dec4']}"
        if want_rows is not None:
            assert {n for _, n in got["rows"]} == {want_rows}, f"{what} {name}: {got['rows']}"
        return check_decode(out, v, i, dictionary, scale, bias, kind, f"{what} {name}")

    worst = {}
    worst["int4"] = rel("int4", lambda: L.decode_int4(vals, idx, packed, H, D, scale, bias), ints4, "int4",
                        want_dec4=dec4_inst(D, True, False, wide))
    worst["int8"] = rel("int8", lambda: L.decode_int8(vals, idx, rows8, H, D, scale, bias), rows8.float(), "rows",
                        want_rows=nch(D))
    worst["f32"] = rel("f32", lambda: L.decode_rows_f32(vals, idx, rows32, H, D, scale, bias), rows32, "rows",
                       want_rows=nch(D))
    if D in (512, 1024):   # the packed dictionary 4 bytes off a 16-byte boundary: the guarded branch
        raw = torch.empty(H * D // 2 + 16, dtype=torch.uint8, device=dev)
        off = (4 - raw.data_ptr()) % 16
        shifted = raw[off:off + H * D // 2].view(H, D // 2)
        shifted.copy_(packed)
        assert shifted.data_ptr() % 16 == 4
        worst["int4 unaligned"] = rel("int4 unaligned", lambda: L.decode_int4(vals, idx, shifted, H, D, scale, bias),
                                      ints4, "int4", want_dec4=dec4_inst(D, False, False, wide))
    # dictionary shards: the winners inside [begin, begin + n) of a shard that starts at a non-zero index
    begin, n = H // 4, H // 2
    own = (idx >= begin) & (idx < begin + n)
    vm = torch.where(own, vals, torch.zeros_like(vals))
    im = torch.where(own, idx - begin, torch.zeros_like(idx))
    assert bool(own.any()) and not bool(own.all())
    worst["int4 range"] = rel("int4 range", lambda: L.decode_range(vals, idx, packed[begin:begin + n], n, begin, D, scale,
                                                                  bias, 4),
                              ints4[begin:begin + n], "int4", want_dec4=dec4_inst(D, True, True, wide), v=vm, i=im)
    worst["int8 range"] = rel("int8 range", lambda: L.decode_range(vals, idx, rows8[begin:begin + n], n, begin, D, scale,
                                                                  bias, 8),
                              rows8[begin:begin + n].float(), "rows", want_rows=nch(D), v=vm, i=im)
    worst["f32 range"] = rel("f32 range", lambda: L.decode_rows_f32_range(vals, idx, rows32[begin:begin + n], begin,
                                                                         scale, bias),
                             rows32[begin:begin + n], "rows", want_rows=nch(D), v=vm, i=im)
    report(f"{what}: " + ", ".join(f"{n} {r:.3g}" for n, r in worst.items()) + " (err/bound)")
