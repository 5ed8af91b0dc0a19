"""t_sae training step on the GPU (TernarySparseAutoencoder with autograd = True), fast and exact mode:

  * forward, loss.backward() and the whole trainer step (training/trainer.py:152-173: forward, loss, backward,
    mask_grad, SGD step, update_mask) from CUDA events, mean over --iters steps after warm-up, for the loss 0.5 mse
    and for 0.5 mse + 1e-3 |h|.mean() (whose own backward is eager torch over [B, H]);
  * the plain no-grad forward in the same run, for scale;
  * each backward kernel's time (torch.profiler, a separate pass) and its TFLOP/s computed from the shapes;
  * the card's name and power limit, read in the same run.

    python tools/prof_tsae_train.py [--B 4096] [--D 512] [--H 32768] [--iters 20] [--out DIR]

Writes DIR/prof_tsae_train.json when --out is given. Inputs are seeded; x and encoder.0.weight are bf16-representable
(the benchmark's precondition for the fast mode)."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import quantizedsae_b200 as Q  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + ", power limit unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=4096)
    ap.add_argument("--D", type=int, default=512)
    ap.add_argument("--H", type=int, default=32768)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_tsae_train needs a CUDA device")
    B, D, H = a.B, a.D, a.H
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    m = Q.TernarySparseAutoencoder(D, H)
    with torch.no_grad():
        m.encoder[0].weight.copy_(m.encoder[0].weight.bfloat16().float())
        m.decoder.weight.normal_(0.0, 0.4824)
    m.to(dev)
    m.autograd = True
    m.decoder.init_mask(0.7)
    x = torch.randn((B, D), device=dev).bfloat16().float()
    opt = torch.optim.SGD(m.parameters(), lr=1e-3)
    flop = 2.0 * B * H * D
    res = {"card": card(), "B": B, "D": D, "H": H, "iters": a.iters, "modes": {}}

    def loss_of(h, recon, lam):
        loss = 0.5 * F.mse_loss(recon, x)
        return loss + lam * h.abs().mean() if lam > 0 else loss

    def step(lam, ev=None):
        opt.zero_grad(set_to_none=True)
        if ev: ev[0].record()
        h, recon = m(x)
        if ev: ev[1].record()
        loss = loss_of(h, recon, lam)
        if ev: ev[2].record()
        loss.backward()
        if ev: ev[3].record()
        m.decoder.mask_grad()
        opt.step()
        m.decoder.update_mask(0.1)
        if ev: ev[4].record()

    for exact in (False, True):
        m.exact = exact
        mode = "exact" if exact else "fast"
        res["modes"][mode] = {}
        for lam, loss_name in ((0.0, "0.5 mse"), (1e-3, "0.5 mse + 1e-3 |h|.mean()")):
            for _ in range(3):
                step(lam)
            torch.cuda.synchronize()
            evs = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(a.iters)]
            for ev in evs:
                step(lam, ev)
            torch.cuda.synchronize()
            fwd = sum(e[0].elapsed_time(e[1]) for e in evs) / a.iters
            bwd = sum(e[2].elapsed_time(e[3]) for e in evs) / a.iters
            tot = sum(e[0].elapsed_time(e[4]) for e in evs) / a.iters
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.no_grad():
                m(x)
                p0.record()
                for _ in range(a.iters):
                    m(x)
                p1.record()
            torch.cuda.synchronize()
            plain = p0.elapsed_time(p1) / a.iters
            # per-kernel breakdown of one backward, in a pass of its own
            opt.zero_grad(set_to_none=True)
            h, recon = m(x)
            loss = loss_of(h, recon, lam)
            torch.cuda.synchronize()
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                loss.backward()
                torch.cuda.synchronize()
            kernels = []
            wgrad_seen = 0
            for e in prof.events():
                if e.device_type != torch.autograd.DeviceType.CUDA or e.device_time <= 0:
                    continue
                name = e.name
                us = e.device_time
                f = None
                if "encode_dense_split_kernel" in name:
                    name, f = "gz = (g T + g_h) 1[h > 0], bias grad (encode_dense_split_kernel)", flop * (3 if exact else 1)
                elif "wgrad_kernel" in name:
                    name = ("grad W_enc = gz^T x", "grad W_dec = g^T h", "grad x")[min(wgrad_seen, 2)] + " (wgrad_kernel)"
                    wgrad_seen += 1
                    f = flop * (6 if exact else 1)
                kernels.append({"kernel": name, "us": round(us, 1), "tflops": round(f / us / 1e6, 1) if f else None})
            res["modes"][mode][loss_name] = {"forward_ms": round(fwd, 4), "backward_ms": round(bwd, 4),
                                             "trainer_step_ms": round(tot, 4), "plain_forward_ms": round(plain, 4),
                                             "backward_kernels": kernels}
            print(f"{mode}, loss {loss_name}: forward {fwd:.3f} ms (no-grad forward {plain:.3f}), loss.backward() "
                  f"{bwd:.3f} ms, trainer step {tot:.3f} ms  [{res['card']}]")
            for k in kernels:
                tf = "" if k["tflops"] is None else f"{k['tflops']:7.1f} TFLOP/s"
                print(f"    {k['us']:9.1f} us  {tf:15s}  {k['kernel'][:100]}")
    if a.out:
        Path(a.out).mkdir(parents=True, exist_ok=True)
        (Path(a.out) / "prof_tsae_train.json").write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
