"""The prior-threshold sweep compiled for that selection mode alone (QSAE_ENCODE_SPECIALISED=1, the default: pipelined
TMEM drain, no other modes in the kernel) against the generic kernel (=0). Every output must be the same bits: survivor
lists, bounds and counts are identical by construction, so values, indices, flags, reconstructions, level counts and
overflow flags are too. Covers every launch shape of the mode-4 sweep: the pair range schedule, the single-CTA range
schedule, the multicast grid, narrower inputs, the exact mode, baseline_sae, q_sae's threshold-only sweep (with and
without an overflow), a ReLU flood that filters full survivor lists in place, and a failed prior."""
import numpy as np
import pytest
import torch

import quantizedsae_b200 as Q
from quantizedsae_b200 import _lib as L
from tests.golden import cases

pytestmark = pytest.mark.gpu

SWITCH = "QSAE_ENCODE_SPECIALISED"


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def enc_case(B, H, D, seed, bf16=True):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((B, D)).astype(np.float32)
    W = cases.xavier_uniform(rng, H, D)
    if bf16:
        x, W = cases.round_bf16(x), cases.round_bf16(W)
    b = (0.01 * rng.standard_normal(H)).astype(np.float32)
    return x, W, b


def assert_same_bits(a, b):
    """Bitwise equality of two output tuples (NaN outputs of an overflowed forward compare equal to themselves)."""
    assert len(a) == len(b)
    for u, v in zip(a, b):
        if u is None or v is None:
            assert u is None and v is None
            continue
        assert u.dtype == v.dtype and u.shape == v.shape
        if u.dtype == torch.float32:
            u, v = u.view(torch.int32), v.view(torch.int32)
        assert torch.equal(u, v)


def both(tuning, fn):
    """fn() on the specialised kernel, then on the generic kernel"""
    outs = []
    for flag in ("1", "0"):
        tuning(SWITCH, flag)
        outs.append(fn())
        torch.cuda.synchronize()
    return outs


@pytest.mark.parametrize("B,H,D,k,exact", [
    (4096, 32768, 512, 32, False),      # the headline: pair range schedule
    (4096, 32768, 512, 32, True),       # exact mode (k_sel = k + 16)
    (4096, 32768, 512, 65, False),
    (333, 32768, 512, 32, False),       # not a multiple of 256: single-CTA range schedule
    (65536, 32768, 512, 32, False),     # multicast grid
    (700, 16384, 256, 32, False),       # D = 256
])
def test_bsae_forward_specialised_sweep_is_bit_identical(cuda_device, tuning, B, H, D, k, exact):
    x, W, b = enc_case(B, H, D, 1000 + B + k, bf16=not exact)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    sample = L.prepare_sample(wb, db)
    packed = torch.randint(0, 256, (H, D // 2), dtype=torch.uint8, device=cuda_device)
    bd = torch.randn(D, device=cuda_device)
    spec, gen = both(tuning, lambda: L.bsae_forward(dx, wb, dW if exact else None, db, k, packed, 4, 0.5, bd, exact=exact,
                                                    want_flags=True, sample=sample))
    assert_same_bits(spec, gen)
    assert int((spec[2] != 0).sum()) == 0


def test_baseline_sae_specialised_sweep_is_bit_identical(cuda_device, tuning):
    D, H, B = 512, 32768, 4096
    torch.manual_seed(3)
    with torch.device(cuda_device):
        m = Q.BaselineSparseAutoencoder(D, H)
    with torch.no_grad():
        m.encoder[0].weight.copy_(m.encoder[0].weight.bfloat16().float())
    m.eval()
    m.return_dense, m.exact = False, False
    x = torch.randn((B, D), device=cuda_device)

    def run():
        with torch.no_grad():
            lat, recon = m(x)
        return lat.values, lat.indices, recon

    spec, gen = both(tuning, run)
    assert_same_bits(spec, gen)


def test_qsae_threshold_sweep_specialised_is_bit_identical(cuda_device, tuning):
    """q_sae's sparse path sweeps with k_sel <= 0 (every value above the threshold is kept): a normal batch, then one
    whose activity overflows the survivor lists (overflow flag set, NaN outputs) -- same bits on both kernels."""
    D, H, B = 512, 32768, 4096
    torch.manual_seed(5)
    with torch.device(cuda_device):
        m = Q.QuantizedMatryoshkaSAE(D, H, 32, abs_range=4.0, n_bits=4)
    with torch.no_grad():
        m.encoder[0].bias.fill_(-0.543)
    m.eval()
    x = torch.randn((B, D), device=cuda_device)
    xbig = x[:256] * 40.0 + 30.0 * torch.sign(m.encoder[0].weight.detach()[:2000].sum(0))
    with torch.no_grad():
        spec, gen = both(tuning, lambda: m._forward_sparse(x))
        assert_same_bits(spec, gen)
        assert int(spec[2].item()) == 0
        spec, gen = both(tuning, lambda: m._forward_sparse(xbig))
        assert_same_bits(spec, gen)
        assert int(spec[2].item()) == 1


def test_relu_flood_relieves_full_lists_identically(cuda_device, tuning):
    """ReLU with almost every pre-activation negative: the prior is 0, every survivor list fills with zeros and is
    filtered / cut in place (relieve_warp_buffers) during the sweep, and the rows end in the tail kernel."""
    B, H, D, k = 150, 16384, 512, 32
    x, W, b = enc_case(B, H, D, 321)
    b = (b - 5.0).astype(np.float32)
    b[np.random.default_rng(5).choice(H, 20, replace=False)] += 10.0
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    sample = L.prepare_sample(wb, db)
    spec, gen = both(tuning, lambda: L.encode_topk(dx, wb, None, db, k, act=L.ACT_RELU, want_flags=True, sample=sample))
    assert_same_bits(spec, gen)
    assert bool((spec[0] == 0).any(1).all())


@pytest.mark.parametrize("exact", [False, True])
def test_failed_prior_goes_through_the_tail_kernel_identically(cuda_device, tuning, exact):
    """A prior far above every row's k-th value (sampled rows carry a bias the real rows do not have): every row fails
    the count check and is recomputed by the tail kernel."""
    B, H, D, k = 70, 16384, 256, 32
    x, W, b = enc_case(B, H, D, 77, bf16=not exact)
    dx, dW, db = T(x, cuda_device), T(W, cuda_device), T(b, cuda_device)
    wb = L.cast_bf16(dW)
    ws, bs = L.prepare_sample(wb, db, 512)
    packed = torch.randint(0, 256, (H, D // 2), dtype=torch.uint8, device=cuda_device)
    bd = torch.randn(D, device=cuda_device)
    spec, gen = both(tuning, lambda: L.bsae_forward(dx, wb, dW if exact else None, db, k, packed, 4, 0.5, bd, exact=exact,
                                                    want_flags=True, sample=(ws, bs + 100.0)))
    assert_same_bits(spec, gen)
    assert int((spec[2] != 0).sum()) == 0
