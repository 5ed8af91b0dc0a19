"""TEST INFRASTRUCTURE ONLY -- CPU restatement (numpy, float64) of one baseline_sae training step's gradients, the oracle
of the baseline backward (quantizedsae_b200/training.py, csrc/train.cu). The product package never imports it.

Reference lines are cited as in oracle/train_oracle.py (paths relative to the reference's src/quantized_sae/). No
stored reference outputs exist for this step; tests/test_baseline_train_oracle.py pins the closed form against torch
float64 autograd on a restatement of the reference forward (SURVEY A.2: Linear -> topk -> zeros_like + scatter_ ->
Linear), and that restatement against the stored forward fixtures tests/golden/baseline_*.npz.
"""
from __future__ import annotations

import numpy as np

F64 = np.float64


def baseline_training_grads(x, We, be, Wd, bd, g_recon, g_h=None, *, k: int = 32, idx=None):
    """Gradients of a loss L(h, recon) through BaselineSparseAutoencoder.forward (sae/baseline.py:17-40), given
    g = dL/drecon [B, D] and g_h = dL/dh dense [B, H] (None: 0). Forward: z = x We^T + be (no ReLU), the top-k of z per
    row (idx given: those selections), h = z on the kept entries and 0 elsewhere, recon = h Wd^T + bd.
      gv[b, j] = g[b] . Wd[:, idx[b, j]] + g_h[b, idx[b, j]]        (top-k passes the gradient at the kept entries)
      dWe[h] = sum gv x[b],  dbe[h] = sum gv,  dWd[:, h] = sum v g[b]  (over the rows b that kept h)
      dbd = sum_b g,  dx = sum_j gv[b, j] We[idx[b, j]]
    float64 throughout. -> dict(h, recon, vals, idx, gv, grad_we, grad_be, grad_wd, grad_bd, grad_x)"""
    x, We, be, Wd, bd, g = (np.asarray(a, dtype=F64) for a in (x, We, be, Wd, bd, g_recon))
    B = x.shape[0]
    H = We.shape[0]
    z = x @ We.T + be
    if idx is None:
        idx = np.argsort(-z, axis=1, kind="stable")[:, :k]
    idx = np.asarray(idx, dtype=np.int64)
    rows = np.arange(B)[:, None]
    vals = z[rows, idx]
    h = np.zeros((B, H))
    h[rows, idx] = vals
    recon = h @ Wd.T + bd
    gv = np.einsum("bd,bjd->bj", g, Wd.T[idx])
    if g_h is not None:
        gv = gv + np.asarray(g_h, dtype=F64)[rows, idx]
    G = np.zeros((B, H))                  # dL/dz: gv on the kept entries
    G[rows, idx] = gv
    return {"h": h, "recon": recon, "vals": vals, "idx": idx, "gv": gv, "grad_we": G.T @ x, "grad_be": G.sum(0),
            "grad_wd": g.T @ h, "grad_bd": g.sum(0), "grad_x": G @ We}
