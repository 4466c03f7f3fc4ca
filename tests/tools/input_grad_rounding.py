"""How much of the 16-bit mode's d loss / d mean_stress error the node encoder's own fp16 rounding explains (CPU only).

The 16-bit node-encoder backward rounds two things to fp16: the tile of dy (the gradient at the second layer's
pre-activation, formed in fp32 from d loss / d x_0) and the W2 weight image.  This script takes the exact fp64 dy of the
oracle, applies those two roundings, forms dfeat = relu'(h0) * (dy W2) . W0 in fp64 and compares it with the exact
d loss / d features.  Everything else the GPU result carries comes from upstream of the encoder.

    python tests/tools/input_grad_rounding.py"""
import os
import sys

R = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, R)
sys.path.insert(0, os.path.join(R, "tests"))
from types import SimpleNamespace  # noqa: E402

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import pdg_helpers as H  # noqa: E402
from oracle import pdg_oracle as O  # noqa: E402


def case(name):
    if name == "synthetic":
        samples, graphs, batch, stats = H.synthetic_batch(3, 600, seed0=123, stress_scale=3.0)
        return batch, stats, O.init_state_dict(seed=7), True, 10.0
    g = H.load_golden(name)
    graphs, batch, stats = H.oracle_batch_from_samples(H.golden_samples(g), bool(g["periodic"]))
    return batch, stats, H.golden_params(), bool(g["divergence"]), float(g["penalty"])


def main():
    for name in ("train2_div", "train2_nodiv", "train3_noperiodic", "train2_quad", "synthetic"):
        batch, stats, sd, div, pen = case(name)
        cap = {}
        orig = O._mlp_ln

        def mlp(x, s, p):
            if p != "node_encoder":
                return orig(x, s, p)
            x.retain_grad()
            h = F.relu(F.linear(x, s[p + ".0.weight"], s[p + ".0.bias"]))
            z2 = F.linear(h, s[p + ".2.weight"], s[p + ".2.bias"])
            z2.retain_grad()
            cap.update(feat=x, h=h, z2=z2)
            return O.graph_layer_norm(F.relu(z2), s[p + ".4.weight"], s[p + ".4.bias"])

        O._mlp_ln = mlp
        try:
            b = SimpleNamespace(**vars(batch))
            for k in ("mean_stress", "pos", "edge_attr"):
                setattr(b, k, getattr(batch, k).detach().double().requires_grad_(True))
            O.train_loss(sd, b, stats, 10, div, pen, torch.float64)[0].backward()
        finally:
            O._mlp_ln = orig
        dy, h = cap["z2"].grad, cap["h"]
        W0, W2 = sd["node_encoder.0.weight"].double()[:, :5], sd["node_encoder.2.weight"].double()
        exact = cap["feat"].grad[:, :5]
        approx = ((dy.half().double() @ W2.half().double()) * (h > 0)) @ W0
        ms, pos = H.rel_err(approx[:, :3], exact[:, :3]), H.rel_err(approx[:, 3:], exact[:, 3:])
        print(f"{name}: encoder-local fp16 rounding -> d/d mean_stress {ms[0]:.1e} / {ms[1]:.1e}, "
              f"d/d pos {pos[0]:.1e} / {pos[1]:.1e} (L-inf / L2 vs fp64)")


if __name__ == "__main__":
    main()
