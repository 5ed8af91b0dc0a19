"""Shared pieces of the dictionary-sharded baseline_sae tests: seeded inputs, the full state_dict, and a numpy `ops`
backend (built on the oracle's baseline_forward pieces) that runs the sharded choreography on CPU under gloo."""
from __future__ import annotations

import numpy as np
import torch

from oracle import qsae_oracle as O
from tests.golden import cases
from tests.sharded_common import NumpyShardOps


def baseline_case(D=64, H=2048, B=37, seed=321, skew=False):
    """skew: every latent of the first half of the dictionary gets a large encoder bias, so shard 0 of a 2-way split
    owns ALL winners (the truncated candidate exchange must notice and fall back to the full one)."""
    cfg = dict(D=D, H=H, B=B, bf16=True, seed=seed)
    inp = cases.baseline_inputs(cfg)
    if skew:
        inp["be"] = inp["be"].copy()
        inp["be"][: H // 2] += np.float32(8.0)
    return cfg, inp


def exact_grid_case(D, H, B, seed):
    """Inputs whose pre-activations every summation order computes exactly: x integers in [-31, 31], encoder weights
    and biases integers times 2^-12 (|x w| <= 3937 * 2^-12, so every partial sum of D <= 1024 terms is an integer
    multiple of 2^-12 below 2^24 of them), all bf16-representable. The GPU's z then equals the oracle's bit for bit in
    fast and exact mode, there are no near-ties, and exact ties follow the (value desc, index asc) rule on both
    sides, so the selected indices must match exactly."""
    rng = np.random.default_rng(seed)
    step = np.float32(2.0 ** -12)
    x = rng.integers(-31, 32, size=(B, D)).astype(np.float32)
    We = rng.integers(-127, 128, size=(H, D)).astype(np.float32) * step
    be = rng.integers(-4096, 4097, size=H).astype(np.float32) * step
    Wd = cases.xavier_uniform(rng, D, H)
    bd = rng.standard_normal(D).astype(np.float32)
    return dict(D=D, H=H, B=B), dict(x=x, We=We, be=be, Wd=Wd, bd=bd)


def full_baseline_state_dict(inp):
    return {"encoder.0.weight": torch.from_numpy(inp["We"]), "encoder.0.bias": torch.from_numpy(inp["be"]),
            "decoder.weight": torch.from_numpy(inp["Wd"]), "decoder.bias": torch.from_numpy(inp["bd"])}


class NumpyBaselineShardOps(NumpyShardOps):
    """CPU restatement of CudaBaselineShardOps (test infrastructure only): the encoder, top-k and merge steps are the
    b_sae backend's (they do not depend on the decoder); the decode uses this shard's decoder columns."""

    def decode_partial(self, vals, idx, plan, with_bias):
        rows = np.ascontiguousarray(self.m.decoder.weight.detach().numpy().T)        # [H/G, D]
        a, b = plan.latent_range()
        i = idx.numpy().astype(np.int64)
        mine = (i >= a) & (i < b)
        v = np.where(mine, vals.numpy(), np.float32(0))
        li = np.where(mine, i - a, 0)
        bias = self.m.decoder.bias.detach().numpy() if with_bias else None
        return torch.from_numpy(O.decode_rows(v, li, rows, 1.0, bias))
