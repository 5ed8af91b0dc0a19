"""Outputs of the encoder paths on seeded inputs, saved or compared bit for bit: a change to the encoder's launch code
must leave the results of every default launch exactly as they were.

    python tools/cmp_outputs.py save DIR            # on a B200: DIR/outputs.npz
    python tools/cmp_outputs.py compare DIR_A DIR_B

Covered (512 -> 32768): t_sae h and recon at B = 4096 in fast and exact mode (dense encoder: resident-x kernel and
the one-launch split-operand kernel), the q_sae dense path of an untrained model (dense_mode = "always") in both
modes, and the b_sae forward at B = 65536 in both modes (separate cast / sample pre-pass / prior kernels).
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
D, H = 512, 32768


def _flatten(prefix, obj, out):
    import torch

    if isinstance(obj, torch.Tensor):
        out[prefix] = obj.detach().cpu().numpy()
    elif hasattr(obj, "values") and hasattr(obj, "indices"):
        _flatten(prefix + ".values", obj.values, out)
        _flatten(prefix + ".indices", obj.indices, out)
    elif isinstance(obj, (list, tuple)):
        for i, o in enumerate(obj):
            _flatten(f"{prefix}.{i}", o, out)
    else:
        out[prefix] = np.asarray(obj)


def outputs():
    import torch

    import quantizedsae_b200 as Q

    dev = torch.device("cuda:0")

    def x_of(batch, seed):
        return torch.randn((batch, D), device=dev, generator=torch.Generator(device=dev).manual_seed(seed))

    out = {}
    torch.manual_seed(0)
    with torch.device(dev):
        t = Q.TernarySparseAutoencoder(D, H)
        q = Q.QuantizedMatryoshkaSAE(D, H, 32, abs_range=4.0, n_bits=4)
        b = Q.BinarySAE(D, H, 4.0, 4)
    with torch.no_grad():
        b.encoder[0].bias.normal_(0.0, 0.1)
    q.dense_mode = "always"
    b.k = 32 / H
    b.return_dense = False
    x4, x64 = x_of(4096, 1), x_of(65536, 2).bfloat16().float()
    with torch.no_grad():
        for m in (t, q, b):
            m.eval()
            for exact in (False, True):
                m.exact = exact
                name = f"{type(m).__name__}_{'exact' if exact else 'fast'}"
                _flatten(name, m(x64 if m is b else x4), out)
    torch.cuda.synchronize()
    return out


def main():
    if len(sys.argv) == 3 and sys.argv[1] == "save":
        os.makedirs(sys.argv[2], exist_ok=True)
        out = outputs()
        np.savez(os.path.join(sys.argv[2], "outputs.npz"), **out)
        print(f"saved {len(out)} arrays to {sys.argv[2]}/outputs.npz")
    elif len(sys.argv) == 4 and sys.argv[1] == "compare":
        a, b = (np.load(os.path.join(d, "outputs.npz")) for d in sys.argv[2:])
        bad = sorted(set(a.files) ^ set(b.files))
        for k in sorted(set(a.files) & set(b.files)):
            same = a[k].dtype == b[k].dtype and a[k].shape == b[k].shape and a[k].tobytes() == b[k].tobytes()
            print(f"{k:40s} {str(a[k].shape):18s} {'identical' if same else 'DIFFERENT'}")
            if not same:
                bad.append(k)
        print("all outputs bit-identical" if not bad else f"differences: {bad}")
        sys.exit(1 if bad else 0)
    else:
        sys.exit(__doc__)


if __name__ == "__main__":
    main()
