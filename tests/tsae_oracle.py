"""TEST INFRASTRUCTURE ONLY -- CPU restatement (numpy, float64) of one t_sae training step's gradients, the oracle of
the t_sae backward (quantizedsae_b200/training.py, csrc/wgrad_sm100.cu). The product package never imports it.

Reference lines are cited as in oracle/train_oracle.py (paths relative to the reference's src/quantized_sae/). No
stored reference outputs exist for this step; tests/test_tsae_train_oracle.py pins the closed form against torch
float64 autograd on a restatement of the reference forward.
"""
from __future__ import annotations

import numpy as np

F64 = np.float64


# --------------------------------------------------------------------------------------
# t_sae: one training step's gradients                        (sae/ternary.py:41-52, :95-122)
# --------------------------------------------------------------------------------------

def tsae_training_grads(x, We, be, Wd, mask, g_recon, g_h=None, *, threshold: float = 0.5):
    """Gradients of a loss L(h, recon) through TernarySparseAutoencoder.forward, given g = dL/drecon [B, D] and
    g_h = dL/dh [B, H] (None: 0). Forward: h = relu(x We^T + be) (encoder = Linear + ReLU, :95-98, :116-118);
    recon = F.linear(h, ste) with ste = (T - Wd*mask).detach() + Wd*mask, T = sign(Wd) * (|Wd| >= threshold)
    (STEWeights.forward, :41-52; its value is T, the mask only gates gradients).
      gz = (g T + g_h) * 1[h > 0]        (torch's ReLU backward masks on the returned h)
      dWe = gz^T x,  dbe = sum_b gz,  dWd = mask * (g^T h),  dx = gz We
    float64 throughout. -> dict(h, recon, gz, grad_we, grad_be, grad_wd, grad_x)"""
    x, We, be, Wd, mask, g = (np.asarray(a, dtype=F64) for a in (x, We, be, Wd, mask, g_recon))
    T = np.sign(Wd) * (np.abs(Wd) >= threshold)
    h = np.maximum(x @ We.T + be, 0.0)
    recon = h @ T.T
    gz = g @ T
    if g_h is not None:
        gz = gz + np.asarray(g_h, dtype=F64)
    gz = np.where(h > 0, gz, 0.0)
    return {"h": h, "recon": recon, "gz": gz, "grad_we": gz.T @ x, "grad_be": gz.sum(0), "grad_wd": mask * (g.T @ h),
            "grad_x": gz @ We}
