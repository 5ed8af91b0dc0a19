"""Large batches (the launch plans of B >= 16384, which the benchmark's B = 65536 lines run) and every warp-merge tier,
against a float64 reference on every row.

Reference. z = x W^T + b and S = |x| |W|^T + |b| in float64 on the device (cuBLAS DGEMM), in row chunks, from exactly
the operands the kernel contracts: bf16-representable x and W in fast mode, arbitrary fp32 in exact mode.

Rules (u = 2^-24):
  band       delta = (D + 1) 2^-23 S per entry. An fp32 dot product of D exact products plus the bias is within
             2u of the running magnitude per addition, and the running magnitude never exceeds S. This covers the
             tensor cores (bf16 products are exact in fp32; accumulation may truncate: < 2u) and the fp32 re-scoring.
             ReLU is 1-Lipschitz, so the band of z bounds relu(z) as well.
  structure  bit exact, in every row: k distinct indices in [0, H), values non-increasing, equal values in ascending
             index order, flags == 0 in exact mode.
  values     every returned value is within delta of z at its index.
  selection  for the returned set G: max over i not in G of (z_i - delta_i) <= min over j in G of (z_j + delta_j).
             Rows whose float64 top-k set differs from G are counted; they are rows with a near-tie at the k-th value,
             and at most 1 % of a batch. The rule has teeth: with the k-th returned index replaced by the best unreturned
             one it rejects every row where those two are separated by more than their bands, and those rows are at
             least half of every batch (a third of the merge-tier batches at k_sel >= 100, D = 512).
  decode     the reference is the float64 decode of the kernel's own (values, indices): scale sum_j v_j w_j + bias,
             with the magnitude M = |scale| sum_j |v_j w_j| + |bias|. The bound follows the decoder's arithmetic:
               int4 (decode_common.cuh): each v_j is rounded to the fixed point 2^-S_row that begin() picks from the
                 row's max |v| (S = 25 - ceil(log2 k) - e2, or 29 - e2 with the 64-bit accumulators of k > 128, where
                 max |v| is in [2^e2, 2^(e2 + 1))): at most 2^-(S + 1) |scale| sum_j |w_j|; the integer sum is exact;
                 then three fp32 roundings (integer to float, times scale, plus bias): 2^-22 M.
               int8 and fp32 rows (decode_rows_kernel): fp32 fma accumulation over k terms and two roundings for
                 scale and bias: (k + 2) 2^-23 M.
             Dropping the last returned latent must break the bound in every row.
  q_sae      the activity, level-count and level / increment rules of tests/test_gpu_matryoshka_levels.py, with its
             own helpers, in row chunks.
Every section prints its largest error / band ratio.
"""
import math
import re

import numpy as np
import pytest
import torch

import quantizedsae_b200 as Q
from quantizedsae_b200 import _lib as L
from tests import test_gpu_matryoshka_levels as LV

gpu = pytest.mark.gpu
TIERS = (8, 12, 16, 32)


def report(msg):
    print(f"[large batch] {msg}")


# ------------------------------------------------------------------------------------------
# the rules (plain torch: they run on CPU tensors as well as on the device)
# ------------------------------------------------------------------------------------------
def reference_chunks(x, W, b, act=0, chunk=None):
    """-> (r0, z, delta) float64 chunks of the batch: z = x W^T + b (relu'd with act), delta = (D + 1) 2^-23 S."""
    H, D = W.shape
    chunk = chunk or max(256, min(4096, (1 << 28) // H))
    W64, b64 = W.double(), b.double()
    aW, ab = W64.abs(), b64.abs()
    for r0 in range(0, x.shape[0], chunk):
        xs = x[r0:r0 + chunk].double()
        z = torch.addmm(b64, xs, W64.T)
        if act:
            z.clamp_(min=0.0)
        delta = torch.addmm(ab, xs.abs(), aW.T).mul_((D + 1) * 2.0 ** -23)
        yield r0, z, delta


def structure_errors(vals, idx, H, flags=None, exact=False):
    """-> list of broken structure rules (empty: every row passes)."""
    bad = []
    i = idx.long()
    if not bool(((i >= 0) & (i < H)).all()):
        bad.append("index out of [0, H)")
    s = i.sort(1).values
    if i.shape[1] > 1 and not bool((s[:, 1:] != s[:, :-1]).all()):
        bad.append("duplicate indices")
    if not bool((vals[:, 1:] <= vals[:, :-1]).all()):
        bad.append("values not non-increasing")
    eq = vals[:, 1:] == vals[:, :-1]
    if not bool((i[:, 1:][eq] > i[:, :-1][eq]).all()):
        bad.append("equal values not in ascending index order")
    if exact and (flags is None or not bool((flags == 0).all())):
        bad.append("flags != 0 in exact mode")
    return bad


def selection_broken(z, delta, idx):
    """-> bool per row: max_{i not in G} (z_i - d_i) > min_{j in G} (z_j + d_j)."""
    g = idx.long()
    out = (z - delta).scatter_(1, g, float("-inf")).max(1).values
    inside = (z.gather(1, g) + delta.gather(1, g)).min(1).values
    return out > inside


def value_ratio(z, delta, vals, idx):
    """-> per-row max |v - z| / delta at the returned indices."""
    g = idx.long()
    return ((vals.double() - z.gather(1, g)).abs() / delta.gather(1, g)).max(1).values


def topk_set_differs(z, idx, k, stable=False):
    """-> bool per row: the float64 top-k set (ties by ascending index when stable) differs from the returned set."""
    ref = (torch.sort(z, dim=1, descending=True, stable=True).indices[:, :k] if stable else torch.topk(z, k, 1).indices)
    return (ref.sort(1).values != idx.long().sort(1).values).any(1)


def swap_kth_for_best_unreturned(z, delta, idx):
    """-> (swapped idx, separated rows): the k-th returned index replaced by the best unreturned one (float64 z);
    separated where z - delta of the dropped one is above z + delta of the one that came in."""
    g = idx.long()
    best = z.clone().scatter_(1, g, float("-inf")).argmax(1)
    out = g[:, -1]
    zk, dk = z.gather(1, out[:, None])[:, 0], delta.gather(1, out[:, None])[:, 0]
    zb, db = z.gather(1, best[:, None])[:, 0], delta.gather(1, best[:, None])[:, 0]
    swapped = g.clone()
    swapped[:, -1] = best
    return swapped, (zk - dk) > (zb + db)


class TopkStats:
    """Accumulates the rules over the chunks of one batch; finish() asserts the batch-level counts."""

    def __init__(self, what, k):
        self.what, self.k = what, k
        self.rows = self.differ = self.separated = 0
        self.worst = 0.0

    def add(self, z, delta, vals, idx, stable=False, r0=0):
        vr = value_ratio(z, delta, vals, idx)
        bad = vr > 1.0
        assert not bool(bad.any()), f"{self.what}: value beyond the band in row {r0 + int(bad.nonzero()[0])}, " \
                                    f"ratio {float(vr.max()):.3g}"
        broken = selection_broken(z, delta, idx)
        assert not bool(broken.any()), f"{self.what}: selection rule broken in {int(broken.sum())} rows, first " \
                                       f"{r0 + int(broken.nonzero()[0])}"
        swapped, sep = swap_kth_for_best_unreturned(z, delta, idx)
        caught = selection_broken(z, delta, swapped)
        assert bool(caught[sep].all()), f"{self.what}: a swapped selection passed the rule in a separated row"
        self.worst = max(self.worst, float(vr.max()))
        self.differ += int(topk_set_differs(z, idx, self.k, stable).sum())
        self.separated += int(sep.sum())
        self.rows += z.shape[0]

    def finish(self, ties=False, min_separated=0.5):
        """ties: rows end in runs of equal values (ReLU floods), where no swap can be separated. min_separated: the
        share of rows whose swap must be separated; at k_sel >= 100 and D = 512 the band spans about one gap between
        neighbouring order statistics, and a third is asked."""
        assert self.differ <= max(2, self.rows // 100), f"{self.what}: {self.differ} of {self.rows} rows differ " \
                                                        "from the float64 top-k set"
        assert ties or self.separated >= min_separated * self.rows, f"{self.what}: only {self.separated} of {self.rows} rows separate " \
                                                "the k-th value from the next by more than the bands"
        report(f"{self.what}: {self.rows} rows, max value err/band {self.worst:.3g}, {self.differ} rows differ from "
               f"the float64 top-k set, swap rejected in {self.separated} separated rows")
        return self.worst


def decode_bound(vals, idx, rows, scale, bias, kind):
    """float64 decode of (vals, idx) over the dictionary rows [H, D] -> (reference, bound, last-latent term), each
    [R, D]. kind: "int4" (fixed point) or "rows" (fp32 accumulation: int8 and fp32 rows)."""
    g = rows[idx.long()].double()                          # [R, k, D]
    v = vals.double()
    k = v.shape[1]
    ref = scale * torch.einsum("rk,rkd->rd", v, g)
    mag = abs(scale) * torch.einsum("rk,rkd->rd", v.abs(), g.abs())
    if bias is not None:
        ref = ref + bias.double()
        mag = mag + bias.double().abs()
    if kind == "int4":
        amax = vals.float().abs().max(1).values
        e2 = torch.where(amax > 0, torch.frexp(amax).exponent - 1, torch.full_like(amax, -100, dtype=torch.int32))
        e2 = e2.clamp(min=-100).double()
        klog = math.ceil(math.log2(k)) if k > 1 else 0
        S = torch.clamp((29.0 if k > 128 else 25.0 - klog) - e2, max=120.0)
        fixed = abs(scale) * torch.pow(2.0, -(S + 1))[:, None] * g.abs().sum(1)
        bnd = fixed + 2.0 ** -22 * (mag + fixed)
    else:
        bnd = (k + 2) * 2.0 ** -23 * mag
    last = scale * v[:, -1:] * g[:, -1]
    return ref, bnd, last


def check_decode(got, vals, idx, rows, scale, bias, kind, what, r0=0):
    """-> largest |got - ref| / bound; asserts the bound and that dropping the last latent breaks it in every row
    whose last value is not zero."""
    ref, bnd, last = decode_bound(vals, idx, rows, scale, bias, kind)
    err = (got.double() - ref).abs()
    bad = err > bnd
    assert not bool(bad.any()), f"{what}: reconstruction beyond the bound in row {r0 + int(bad.nonzero()[0, 0])}"
    live = vals[:, -1] != 0
    dropped = ((got.double() - (ref - last)).abs() > bnd).any(1)
    assert bool(dropped[live].all()), f"{what}: a reconstruction without its last latent passes the bound"
    return float((err / bnd.clamp(min=1e-300)).max())


# ------------------------------------------------------------------------------------------
# the planner, restated (qsae_api.cu: choose_prior_rank, plan_encode, the merge tier, the dense chunks)
# ------------------------------------------------------------------------------------------
def choose_prior_rank(k_sel, r):
    n = k_sel - 1
    if n <= 0:
        return 1
    pmf = (1.0 - r) ** n
    cdf = pmf
    for j in range(1, n + 1):
        if 1.0 - cdf < 1e-7:
            return j
        pmf *= (n - j + 1) / j * r / (1.0 - r)
        cdf += pmf
    return n + 1


def prior_plan(H, k, exact, n_sample):
    """k <= QSAE_MAX_K -> (k_sel, m); m = 0: no prior path."""
    k_sel = min(k + L.QSAE_RESCORE_MARGIN, L.QSAE_MAX_K, H) if exact else k
    if n_sample >= 256 and H >= 8 * n_sample:
        m = choose_prior_rank(k_sel, n_sample / H)
        if m <= 32 and m <= n_sample and (m + math.sqrt(m)) * H / n_sample <= 512.0:
            return k_sel, m
    return k_sel, 0


def auto_tier(B, H, k_sel, n_sample, m):
    tier = 16
    if n_sample > 0 and m > 0 and B > 8192:
        need = (m + 3.0 * math.sqrt(m)) * H / n_sample
        tier = 8 if need <= 256.0 else (12 if need <= 384.0 else 16)
    return 16 if 32 * tier < k_sel else tier


def dense_chunks(B, H):
    rows = (1 << 30) // (H * 4) // 128 * 128
    rows = min(max(rows, 128), B)
    return rows, -(-B // rows)


PRIOR_LINE = re.compile(r"\[qsae prior path\] B=(\d+) k_sel=(\d+) m=(\d+) nsub=\d+ cap=\d+: (\d+) rows recomputed "
                        r"exactly, (\d+) rows through the block select")
LARGE_LINE = re.compile(r"\[qsae large\] k=(\d+) k_sel=(\d+) m=(\d+) .*rescued rows (\d+), sweep overflow (\d+)")


def prior_counts(capfd):
    """The one `[qsae prior path]` line QSAE_DEBUG_LARGE printed since the last read -> dict."""
    lines = PRIOR_LINE.findall(capfd.readouterr().err)
    assert len(lines) == 1, f"expected one prior-path line, got {lines}"
    B, k_sel, m, rec, blk = (int(v) for v in lines[0])
    return dict(B=B, k_sel=k_sel, m=m, recomputed=rec, block=blk)


# ------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------
def enc_case(B, H, D, seed, exact, dev, row_scale=False, bias_std=0.01):
    """x ~ N(0, 1) (each row scaled by 2^U(-2, 2) with row_scale), xavier W, small bias; bf16-representable operands in
    fast mode."""
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn((B, D), device=dev, generator=g)
    if row_scale:
        x *= torch.pow(2.0, torch.rand((B, 1), device=dev, generator=g) * 4 - 2)
    W = (torch.rand((H, D), device=dev, generator=g) * 2 - 1) * (6.0 / (H + D)) ** 0.5
    b = bias_std * torch.randn(H, device=dev, generator=g)
    if not exact:
        x, W = x.bfloat16().float(), W.bfloat16().float()
    return x.contiguous(), W.contiguous(), b.contiguous()


def int4_dictionary(H, D, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    packed = torch.randint(0, 256, (H, D // 2), dtype=torch.uint8, device=dev, generator=g)
    lo, hi = (packed & 15).to(torch.int16), (packed >> 4).to(torch.int16)
    ints = torch.stack((lo, hi), -1).reshape(H, D)
    return packed, torch.where(ints >= 8, ints - 16, ints).float()


# ------------------------------------------------------------------------------------------
# 6. the rules on the CPU, with known-good and known-bad rows
# ------------------------------------------------------------------------------------------
def test_rules_on_synthetic_rows():
    gen = torch.Generator().manual_seed(0)
    R, H, k, D = 7, 64, 5, 16
    z = torch.randn((R, H), generator=gen).double()                 # fp32-representable: the fp32 values are exact
    z[3, :] = 0.0                                                   # a row of exact ties
    delta = torch.full_like(z, 1e-9)
    v, i = torch.sort(z, dim=1, descending=True, stable=True)
    vals, idx = v[:, :k].float(), i[:, :k].int()
    assert structure_errors(vals, idx, H) == []
    assert not bool(selection_broken(z, delta, idx).any())
    assert float(value_ratio(z, delta, vals.double(), idx).max()) == 0.0
    assert not bool(topk_set_differs(z, idx, k, stable=True).any())
    swapped, sep = swap_kth_for_best_unreturned(z, delta, idx)
    assert bool(sep[[0, 1, 2, 4, 5, 6]].all()) and not bool(sep[3])  # the tie row cannot be separated
    assert bool(selection_broken(z, delta, swapped)[sep].all())
    dup = idx.clone()
    dup[1, 2] = dup[1, 1]
    assert "duplicate indices" in structure_errors(vals, dup, H)
    assert "index out of [0, H)" in structure_errors(vals, idx - 100, H)
    assert "values not non-increasing" in structure_errors(vals.flip(1), idx.flip(1), H)
    tie = idx.clone()
    tie[3, :2] = tie[3, :2].flip(0)
    assert structure_errors(vals, tie, H) == ["equal values not in ascending index order"]
    assert structure_errors(vals, idx, H, flags=torch.tensor([0, 1] + [0] * (R - 2)), exact=True) == \
        ["flags != 0 in exact mode"]
    st = TopkStats("synthetic", k)
    st.add(z, delta, vals, idx, stable=True)
    assert st.differ == 0 and st.separated == R - 1
    with pytest.raises(AssertionError, match="selection rule broken"):
        TopkStats("synthetic", k).add(z, delta, z.gather(1, swapped).float(), swapped.int(), stable=True)
    off = vals.clone()
    off[0, 0] += 1e-3
    with pytest.raises(AssertionError, match="value beyond the band"):
        TopkStats("synthetic", k).add(z, delta, off, idx, stable=True)
    # reconstructions: the exact float64 decode passes either bound, one latent less fails both
    vals = vals.abs() + 0.25
    ints = torch.randint(-8, 8, (H, D), generator=gen).float()
    bias = torch.randn(D, generator=gen)
    for kind in ("int4", "rows"):
        ref, bnd, last = decode_bound(vals, idx, ints, 0.5, bias, kind)
        assert float(check_decode(ref, vals, idx, ints, 0.5, bias, kind, kind)) == 0.0
        assert float(check_decode(ref + 0.5 * bnd, vals, idx, ints, 0.5, bias, kind, kind)) == pytest.approx(0.5)
        with pytest.raises(AssertionError, match="beyond the bound"):
            check_decode(ref - last, vals, idx, ints, 0.5, bias, kind, kind)
    # the int4 fixed point: S = 25 - ceil(log2 5) - e2 with max |v| in [2^e2, 2^(e2 + 1))
    one = torch.tensor([[1.5, 0.75, 0.25, 0.25, 0.25]])
    _, bnd, _ = decode_bound(one, torch.zeros((1, 5), dtype=torch.int32), torch.ones((1, 1)), 1.0, None, "int4")
    assert float(bnd[0, 0]) == pytest.approx(2.0 ** -(25 - 3 + 1) * 5 * (1 + 2.0 ** -22) + 2.0 ** -22 * 3.0)


# ------------------------------------------------------------------------------------------
# 1. the device reference against numpy float64
# ------------------------------------------------------------------------------------------
@gpu
def test_device_reference_matches_numpy(cuda_device):
    x, W, b = enc_case(4096 + 5, 32768, 512, 1, True, cuda_device)
    rows = [0, 1, 4095, 4096, 4100]
    xn, Wn, bn = (t.cpu().numpy().astype(np.float64) for t in (x, W, b))
    for r0, z, d in reference_chunks(x, W, b):
        for r in rows:
            if r0 <= r < r0 + z.shape[0]:
                zr = xn[r] @ Wn.T + bn
                sr = np.abs(xn[r]) @ np.abs(Wn).T + np.abs(bn)
                np.testing.assert_allclose(z[r - r0].cpu().numpy(), zr, rtol=1e-12, atol=1e-12)
                np.testing.assert_allclose(d[r - r0].cpu().numpy(), 513 * 2.0 ** -23 * sr, rtol=1e-12)


# ------------------------------------------------------------------------------------------
# 2. every merge tier, forced, at small batches
# ------------------------------------------------------------------------------------------
# (k, exact, QSAE_SAMPLE_DIV): every sort_and_emit width on the prior path. 32 keys: k_sel 8, 16 + 16, 32; 64: 33, 64;
# TAIL (k_sel 65): 65, 49 + 16; 128: 100, 128, 112 + 16; 256: k_sel 144, which needs a sample of H / 13 (2560 rows):
# the largest prior rank is 32 and the survivors must fit the warp merge, so k_sel <= 129 at H / 16 and <= 147 at H / 13.
TIER_KS = [(8, False, 16), (32, False, 16), (33, False, 16), (64, False, 16), (65, False, 16), (100, False, 16),
           (128, False, 16), (16, True, 16), (49, True, 16), (112, True, 16), (144, False, 13), (128, True, 13)]
TIER_SHAPES = [(1000, 512), (333, 512), (1000, 256), (333, 256)]


def fit_tiers(k_sel):
    """Tiers that hold every survivor of some rows: 32 T > 2 k_sel. Below that (tier 8 at k_sel >= 128) the prior's
    survivors (16 m on average, 416 at k_sel = 128) overflow the registers in every row; those rows take the
    prefilter and, since the first 32 T survivors give a weak k_sel-th value, the block select."""
    return [T for T in TIERS if 32 * T > 2 * k_sel]


def pick_shift(z, prior, k_sel):
    """The sample-bias shift (prior lowered by it; negative: raised) that best splits the rows into ones that fit the
    registers and ones that take the two-pass prefilter, at every tier of fit_tiers; 0 when the unshifted prior does."""
    zs = torch.sort(z, 1, descending=True).values
    a = {T: (prior.double() - zs[:, 32 * T]) for T in fit_tiers(k_sel)}   # survivors > 32 T  <=>  shift > a
    def score(s):
        return min(min(float((a[T] > s).double().mean()), float((a[T] < s).double().mean())) for T in a)
    if score(0.0) >= 0.1:
        return 0.0
    cand = torch.cat(list(a.values()))
    qs = torch.quantile(cand.float().cpu(), torch.linspace(0.0, 1.0, 201)).tolist()
    return max(qs, key=score)


@gpu
@pytest.mark.parametrize("B,D", TIER_SHAPES, ids=[f"b{B}-d{D}" for B, D in TIER_SHAPES])
@pytest.mark.parametrize("k,exact,div", TIER_KS, ids=[f"{'exact' if e else 'fast'}-k{k}-div{d}" for k, e, d in TIER_KS])
def test_every_merge_tier(cuda_device, tuning, capfd, B, D, k, exact, div):
    H = 32768
    tuning("QSAE_SAMPLE_DIV", div)
    tuning("QSAE_DEBUG_LARGE", 1)
    x, W, b = enc_case(B, H, D, 7 * k + B + D + div, exact, cuda_device, row_scale=True)
    wb = L.cast_bf16(W)
    ws, bs = L.prepare_sample(wb, b)
    n_sample = ws.shape[0]
    k_sel, m = prior_plan(H, k, exact, n_sample)
    assert m > 0, "this case must take the prior path"
    z, delta = next(reference_chunks(x, W, b, chunk=B))[1:]
    # the sweep and the prior see the bf16 operands (in exact mode too: only the merge re-scores in fp32)
    zb, db = next(reference_chunks(x.bfloat16().float(), wb.float(), b, chunk=B))[1:]
    prior = L.prior_prep(x, (ws, bs), m)[1]
    shift = pick_shift(zb, prior, k_sel)
    sample = (ws, (bs - shift).contiguous())
    prior = L.prior_prep(x, sample, m)[1].double()[:, None]
    surv_lo = ((zb - db) > prior).sum(1)                            # the sweep keeps the values at or above the prior
    surv_hi = ((zb + db) >= prior).sum(1)
    del zb, db
    packed, ints = int4_dictionary(H, D, k, cuda_device)
    bd = torch.randn(D, device=cuda_device, generator=torch.Generator(device=cuda_device).manual_seed(k))
    capfd.readouterr()
    outs, worst = [], [0.0, 0.0]
    for T in TIERS:
        assert 32 * T >= k_sel                                      # the forced tier is the tier that runs
        tuning("QSAE_MERGE_TIER", T)
        o = L.bsae_forward(x, wb, W if exact else None, b, k, packed, 4, 0.5, bd, exact=exact, want_flags=True,
                           sample=sample)
        c = prior_counts(capfd)
        assert (c["B"], c["k_sel"], c["m"]) == (B, k_sel, m)
        fit, pre = int((surv_hi <= 32 * T).sum()), int((surv_lo > 32 * T).sum())
        what = f"tier {T} {'exact' if exact else 'fast'} k={k} B={B} D={D}"
        if T in fit_tiers(k_sel):
            assert fit > 0 and pre > 0, f"{what}: {fit} rows fit the registers, {pre} take the two-pass prefilter"
        else:
            assert pre > 0 and c["block"] > 0, f"{what}: {pre} rows prefiltered, {c['block']} in the block select"
        vals, idx, flags, recon = o
        assert structure_errors(vals, idx, H, flags, exact) == []
        st = TopkStats(what, k)
        st.add(z, delta, vals, idx)
        worst[0] = max(worst[0], st.finish(min_separated=1 / 3 if k_sel >= 100 and D == 512 else 0.5))
        worst[1] = max(worst[1], check_decode(recon, vals, idx, ints, 0.5, bd, "int4", what))
        report(f"{what}: shift {shift:.4g}, {fit} rows fit, {pre} prefiltered, {c['block']} block select, "
               f"{c['recomputed']} recomputed")
        outs.append(o)
    for o in outs[1:]:
        assert all(torch.equal(a, c) for a, c in zip(outs[0], o)), "the tiers differ"
    report(f"merge tiers {'exact' if exact else 'fast'} k={k} B={B} D={D}: max value err/band {worst[0]:.3g}, "
           f"decode err/bound {worst[1]:.3g}")


@gpu
@pytest.mark.parametrize("tier", TIERS)
def test_merge_tier_relu_flood_and_failed_prior(cuda_device, tuning, capfd, tier):
    """ReLU with almost every pre-activation negative: the prior is 0 and every list fills with equal zeros, which the
    warp merge hands to the block select of the tail kernel (at 32 keys per lane the filled lists fit the registers). Then a prior far too high (sampled rows with a bias the
    real rows lack): every row fails the count check and is recomputed exactly."""
    B, H, D, k = 150, 16384, 512, 32
    tuning("QSAE_DEBUG_LARGE", 1)
    tuning("QSAE_MERGE_TIER", tier)
    x, W, b = enc_case(B, H, D, 321, False, cuda_device)
    b = b - 5.0
    b[torch.randperm(H, generator=torch.Generator().manual_seed(5))[:20].to(cuda_device)] += 10.0
    wb = L.cast_bf16(W)
    sample = L.prepare_sample(wb, b)
    capfd.readouterr()
    vals, idx, flags = L.encode_topk(x, wb, None, b, k, act=L.ACT_RELU, want_flags=True, sample=sample)
    c = prior_counts(capfd)
    if tier < 32:
        assert c["block"] == B, f"tier {tier}: {c['block']} of {B} flooded rows reached the block select"
    else:   # 1024 keys hold the rows' full survivor lists: the ties are ordered in the registers
        assert c["block"] == 0, f"tier {tier}: {c['block']} flooded rows reached the block select"
    assert structure_errors(vals, idx, H) == []
    z, delta = next(reference_chunks(x, W, b, act=1, chunk=B))[1:]
    assert bool((torch.sort(z, 1, descending=True).values[:, k - 1] == 0).all()), "every row should end in zeros"
    st = TopkStats(f"relu flood tier {tier}", k)
    st.add(z, delta, vals, idx, stable=True)
    w0 = st.finish(ties=True)
    n_block = c["block"]
    packed, ints = int4_dictionary(H, D, 3, cuda_device)
    bd = torch.randn(D, device=cuda_device)
    worst = 0.0
    for exact in (False, True):
        ws, bs = sample
        o = L.bsae_forward(x, wb, W if exact else None, b, k, packed, 4, 0.5, bd, exact=exact, want_flags=True,
                           sample=(ws, bs + 100.0))
        c = prior_counts(capfd)
        assert c["recomputed"] == B, f"tier {tier}: {c['recomputed']} of {B} rows recomputed"
        what = f"failed prior tier {tier} {'exact' if exact else 'fast'}"
        assert structure_errors(o[0], o[1], H, o[2], exact) == []
        z, delta = next(reference_chunks(x, W, b, chunk=B))[1:]
        st = TopkStats(what, k)
        st.add(z, delta, o[0], o[1])
        worst = max(worst, st.finish(), w0)
        check_decode(o[3], o[0], o[1], ints, 0.5, bd, "int4", what)
    report(f"relu flood / failed prior tier {tier}: {n_block} block-select rows; max value err/band {worst:.3g}")


# ------------------------------------------------------------------------------------------
# 3. the automatic plan at large batches, every row
# ------------------------------------------------------------------------------------------
def make_bsae(W, b, D, H, n_bits, k, exact, dev, seed):
    with torch.device(dev):
        m = Q.BinarySAE(D, H, 4.0, n_bits)
    g = torch.Generator(device=dev).manual_seed(seed)
    with torch.no_grad():
        m.encoder[0].weight.copy_(W)
        m.encoder[0].bias.copy_(b)
        m.decoder.weight.copy_(torch.where(torch.rand(m.decoder.weight.shape, device=dev, generator=g) < 0.5, 110.0, -110.0))
        m.decoder.bias.copy_(torch.randn(D, device=dev, generator=g))
    m.eval()
    m.k = (k + 0.5) / H                                             # int(H * m.k) == k
    m.return_dense, m.exact = False, exact
    assert int(H * m.k) == k and m.decoder.resolved_mode() == "int"
    return m


def check_bsae_batch(m, x, W, b, k, exact, n_bits, what, capfd):
    """BinarySAE forward vs L.bsae_forward (same bits), then every row against the rules."""
    H, D = W.shape
    dec = m.decoder
    wb = m._w_bf16()
    sample = m._sample()
    capfd.readouterr()
    vals, idx, flags, recon = L.bsae_forward(x, wb, W if exact else None, b, k, dec._packed()[0], n_bits,
                                             dec.quantization_step, dec.bias.detach(), exact=exact, want_flags=True,
                                             sample=sample)
    c = prior_counts(capfd)
    with torch.no_grad():
        lat, rec2, _ = m(x)
    capfd.readouterr()
    assert torch.equal(lat.values, vals) and torch.equal(lat.indices, idx) and torch.equal(rec2, recon)
    if exact:
        assert torch.equal(m.last_flags, flags)
    assert structure_errors(vals, idx, H, flags, exact) == []
    ints = dec.quantized_int_weights().detach()
    kind = "int4" if n_bits <= 4 else "rows"
    st = TopkStats(what, k)
    dworst = 0.0
    for r0, z, delta in reference_chunks(x, W, b):
        r1 = r0 + z.shape[0]
        st.add(z, delta, vals[r0:r1], idx[r0:r1], r0=r0)
        for s0 in range(r0, r1, 2048):
            s1 = min(r1, s0 + 2048)
            dworst = max(dworst, check_decode(recon[s0:s1], vals[s0:s1], idx[s0:s1], ints, dec.quantization_step,
                                              dec.bias.detach(), kind, what, s0))
    vworst = st.finish()
    report(f"{what}: {c['recomputed']} rows recomputed, {c['block']} block select; decode err/bound {dworst:.3g}")
    return c, (vals, idx, flags, recon), vworst, dworst


BSAE_CASES = [   # (B, H, D, k, n_bits, exact, expected tier)
    (65536, 32768, 512, 32, 4, False, 12), (65536, 32768, 512, 32, 4, True, 16),
    (65536, 32768, 512, 65, 4, False, 16), (65536, 32768, 512, 65, 4, True, 16),
    (16384, 32768, 512, 8, 4, False, 8),
    (16513, 30000, 512, 32, 4, False, 12), (16513, 30000, 512, 32, 4, True, 16),
    (16384, 32768, 256, 32, 2, False, 12), (16384, 32768, 256, 32, 8, True, 16),
]


@gpu
@pytest.mark.parametrize("B,H,D,k,n_bits,exact,tier", BSAE_CASES,
                         ids=[f"b{c[0]}-h{c[1]}-d{c[2]}-k{c[3]}-nb{c[4]}-{'exact' if c[5] else 'fast'}" for c in BSAE_CASES])
def test_bsae_automatic_plan_every_row(cuda_device, tuning, capfd, B, H, D, k, n_bits, exact, tier):
    """B >= 16384: the (split, row block) grid sweep (multicast clusters at D > 448), separate prior launches, and the
    merge tier from the survivor statistics. B = 16513 at H = 30000 leaves a partial last row block, an odd number of
    row blocks and a partial last dictionary tile."""
    tuning("QSAE_DEBUG_LARGE", 1)
    x, W, b = enc_case(B, H, D, B + k + D, exact, cuda_device)
    m = make_bsae(W, b, D, H, n_bits, k, exact, cuda_device, seed=k)
    n_sample = m._sample()[0].shape[0]
    k_sel, mm = prior_plan(H, k, exact, n_sample)
    assert mm > 0 and auto_tier(B, H, k_sel, n_sample, mm) == tier
    what = f"b_sae B={B} H={H} D={D} k={k} n_bits={n_bits} {'exact' if exact else 'fast'} (tier {tier})"
    c, out, _, _ = check_bsae_batch(m, x, W, b, k, exact, n_bits, what, capfd)
    assert (c["B"], c["k_sel"], c["m"]) == (B, k_sel, mm)
    if B == 16384 and D == 512:
        tuning("QSAE_ENCODE_CLUSTER", 0)
        o2 = L.bsae_forward(x, m._w_bf16(), W if exact else None, b, k, m.decoder._packed()[0], n_bits,
                            m.decoder.quantization_step, m.decoder.bias.detach(), exact=exact, want_flags=True,
                            sample=m._sample())
        assert all(torch.equal(a, c2) for a, c2 in zip(out, o2)), "the sweep without clusters differs"


@gpu
@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact"])
def test_baseline_sae_bench_batch_every_row(cuda_device, capfd, tuning, exact):
    """baseline_sae at B = 65536 (bench config 2): fused encoder + top-32, fp32 row-gather decode."""
    B, H, D, k = 65536, 32768, 512, 32
    tuning("QSAE_DEBUG_LARGE", 1)
    x, W, b = enc_case(B, H, D, 2, exact, cuda_device)
    with torch.device(cuda_device):
        m = Q.BaselineSparseAutoencoder(D, H)
    with torch.no_grad():
        m.encoder[0].weight.copy_(W)
        m.encoder[0].bias.copy_(b)
    m.eval()
    m.return_dense, m.exact = False, exact
    capfd.readouterr()
    with torch.no_grad():
        lat, recon = m(x)
    c = prior_counts(capfd)
    k_sel, mm = prior_plan(H, k, exact, m._sample()[0].shape[0])
    assert (c["B"], c["k_sel"], c["m"]) == (B, k_sel, mm)
    vals, idx = lat.values, lat.indices
    what = f"baseline_sae B={B} {'exact' if exact else 'fast'}"
    assert structure_errors(vals, idx, H, m.last_flags, exact) == []
    rows = m.decoder.weight.detach().T.contiguous()
    st = TopkStats(what, k)
    dworst = 0.0
    for r0, z, delta in reference_chunks(x, W, b):
        r1 = r0 + z.shape[0]
        st.add(z, delta, vals[r0:r1], idx[r0:r1], r0=r0)
        dworst = max(dworst, check_decode(recon[r0:r1], vals[r0:r1], idx[r0:r1], rows, 1.0,
                                          m.decoder.bias.detach(), "rows", what, r0))
    st.finish()
    report(f"{what}: decode err/bound {dworst:.3g}")


# ------------------------------------------------------------------------------------------
# 4. large k at large batches
# ------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact"])
def test_large_k_prior_path_large_batch(cuda_device, tuning, capfd, exact):
    """BinarySAE at H = 2^17 keeps int(0.002 H) = 262 latents: the sampled prior, the block-level radix merge and the
    64-bit int4 decoder (k > 128), at B = 16384."""
    B, H, D, k = 16384, 2 ** 17, 64, 262
    tuning("QSAE_DEBUG_LARGE", 1)
    x, W, b = enc_case(B, H, D, 262, exact, cuda_device)
    m = make_bsae(W, b, D, H, 4, k, exact, cuda_device, seed=5)
    m.k = 0.002
    assert int(H * m.k) == k
    capfd.readouterr()
    with torch.no_grad():
        lat, recon, _ = m(x)
    lines = LARGE_LINE.findall(capfd.readouterr().err)
    assert len(lines) == 1 and int(lines[0][0]) == k and int(lines[0][2]) > 0, f"not the prior path: {lines}"
    vals, idx = lat.values, lat.indices
    what = f"large k prior path B={B} H={H} k={k} {'exact' if exact else 'fast'}"
    assert structure_errors(vals, idx, H, m.last_flags, exact) == []
    ints = m.decoder.quantized_int_weights().detach()
    st = TopkStats(what, k)
    dworst = 0.0
    for r0, z, delta in reference_chunks(x, W, b):
        r1 = r0 + z.shape[0]
        st.add(z, delta, vals[r0:r1], idx[r0:r1], r0=r0)
        dworst = max(dworst, check_decode(recon[r0:r1], vals[r0:r1], idx[r0:r1], ints, m.decoder.quantization_step,
                                          m.decoder.bias.detach(), "int4", what, r0))
    st.finish()
    report(f"{what}: {lines[0][3]} rows rescued; decode err/bound {dworst:.3g}")


@gpu
@pytest.mark.parametrize("B,n_chunks", [(20000, 3), (16384, 2)])
@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact"])
def test_large_k_dense_fallback_chunks(cuda_device, tuning, capfd, B, n_chunks, exact):
    """No sample: pre-activations in row chunks of at most 1 GB (8192 rows at H = 32768), a dense radix select per
    chunk. A bias spread of 2 keeps the k-th value separated from the next by more than the band in most rows."""
    H, D, k = 32768, 512, 500
    tuning("QSAE_DEBUG_LARGE", 1)
    assert dense_chunks(B, H) == (8192, n_chunks)
    x, W, b = enc_case(B, H, D, B + 500, exact, cuda_device, bias_std=2.0)
    capfd.readouterr()
    vals, idx, flags = L.encode_topk(x, L.cast_bf16(W), W if exact else None, b, k, exact=exact, want_flags=True)
    assert not LARGE_LINE.search(capfd.readouterr().err), "the dense path prints no prior-path statistics"
    what = f"large k dense B={B} ({n_chunks} chunks) k={k} {'exact' if exact else 'fast'}"
    assert structure_errors(vals, idx, H, flags, exact) == []
    st = TopkStats(what, k)
    for r0, z, delta in reference_chunks(x, W, b):
        st.add(z, delta, vals[r0:r0 + z.shape[0]], idx[r0:r0 + z.shape[0]], r0=r0)
    st.finish()


# ------------------------------------------------------------------------------------------
# 5. q_sae at large batches
# ------------------------------------------------------------------------------------------
def level_grid(B, num_sms, warps=4):
    """decode_matryoshka_launch: resident blocks of `warps` warps, 6 to 8 per SM -> rows per warp (ceil)."""
    bps = 6
    if num_sms * 6 * warps < B <= num_sms * 7 * warps:
        bps = 7
    elif num_sms * 6 * warps < B <= num_sms * 8 * warps:
        bps = 8
    blocks = min(-(-B // warps), num_sms * bps)
    return -(-B // (blocks * warps))


@gpu
@pytest.mark.parametrize("B", [4737, 65536])
@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact"])
@pytest.mark.parametrize("nb", [4, 8])
def test_qsae_large_batch_levels(cuda_device, B, exact, nb):
    """q_sae at 512 -> 32768 (bench config 4): B = 4737 is the first batch whose level decoder warps loop over rows."""
    H, D = 32768, 512
    sms = torch.cuda.get_device_properties(cuda_device).multi_processor_count
    assert level_grid(B, sms) > 1 and (sms != 148 or level_grid(4736, sms) == 1)
    cfg = LV.qsae_cfg(nb, H, D, B, bf16=not exact)
    inp = LV.qsae_case(cfg)
    m = LV.make_qsae(inp, cfg, cuda_device)
    m.exact = exact
    x = torch.from_numpy(inp["x"]).to(cuda_device)
    with torch.no_grad():
        out = m.forward_active(x)
        groups, result = m(x)
    assert m.last_path == "sparse"
    for a, c in zip(result, out["reconstruction_levels"]):
        assert torch.equal(a, c)
    starts = LV.starts_of(cfg)
    Tm, scale = LV.dictionary(inp, cfg)
    We = torch.from_numpy(inp["We"]).to(cuda_device)
    be = torch.from_numpy(inp["be"]).to(cuda_device)
    a_idx, a_cnt = out["active_idx"], out["active_cnt"]
    cap = a_idx.shape[1]
    slot = torch.arange(cap, device=cuda_device)[None, :]
    assert bool((a_cnt <= cap).all()) and bool(((a_idx >= 0) == (slot < a_cnt[:, None])).all())
    assert bool((a_idx < H).all())
    srt = torch.sort(a_idx, 1).values
    assert bool(((srt[:, 1:] != srt[:, :-1]) | (srt[:, 1:] < 0)).all()), "duplicate active latents"
    got_all = torch.stack(result)
    what = f"q_sae {'exact' if exact else 'fast'} nb={nb} B={B}"
    totals = np.zeros(len(starts) - 1, dtype=np.int64)
    worst, n_band = 0.0, 0
    chunk = 2048
    for r0, z, delta in reference_chunks(x, We, be, chunk=chunk):
        r1 = r0 + z.shape[0]
        d = delta * 0.5                                              # the levels file's band: (D + 1) u S
        band = ((z - LV.THR).abs() <= d)
        forced = ((z >= LV.THR) & ~band).cpu().numpy()
        band = band.cpu().numpy()
        act = torch.zeros((r1 - r0, H + 1), dtype=torch.bool, device=cuda_device)
        ai = a_idx[r0:r1].long()
        act.scatter_(1, torch.where(ai >= 0, ai, H), True)           # empty slots land in the extra column H
        act = act[:, :H].cpu().numpy()
        n_band += LV.check_decisions(act, forced, band, f"{what} rows {r0}:{r1}")
        totals += LV.level_sums(act, starts)
        worst = max(worst, LV.check_levels(got_all[:, r0:r1].cpu().numpy(), act, Tm, scale, starts, inp["bd"], False,
                                           f"{what} rows {r0}:{r1}"))
    assert np.array_equal(out["level_counts"].cpu().numpy(), totals)
    assert np.array_equal(LV.group_counts(groups, B), totals)
    report(f"{what}: {int(totals.sum()) / B:.1f} active per row, {n_band} band entries, level err/bound {worst:.3g}")


@gpu
def test_qsae_chunked_band_matches_the_levels_file(cuda_device):
    """The device-side activity band used above is the levels file's activity_band."""
    cfg = LV.qsae_cfg(4, 32768, 512, 64)
    inp = LV.qsae_case(cfg)
    forced, band = LV.activity_band(inp["x"], inp["We"], inp["be"])
    x, We, be = (torch.from_numpy(inp[n]).to(cuda_device) for n in ("x", "We", "be"))
    _, z, delta = next(reference_chunks(x, We, be))
    b2 = ((z - LV.THR).abs() <= delta * 0.5)
    assert np.array_equal(b2.cpu().numpy(), band)
    assert np.array_equal(((z >= LV.THR) & ~b2).cpu().numpy(), forced)
