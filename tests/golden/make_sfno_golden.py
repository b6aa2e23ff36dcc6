#!/usr/bin/env python
"""Golden vectors for the SFNO network restatement (makani_b200/sfno.py, SURVEY rows A8/A9), produced by the REFERENCE's own
network class: /root/reference/makani/models/networks/sfnonet.py (SphericalFourierNeuralOperatorNet, NeuralOperatorBlock, unmodified)
with the reference's own SpectralConv / MLP / EncoderDecoder, run on the CPU oracle posed as `torch_harmonics`
(tests/reference_suites/run_reference_tests.py::install_environment).  Stored per case: the full state dict, the input, the output,
d(loss)/d(input) and the gradients of a few parameters for loss = sum(out * g).

    MAKANI_REFERENCE=<makani checkout> python tests/golden/make_sfno_golden.py   -> tests/golden/sfno_golden_<case>.npz (one file per case)
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "reference_suites"))

SFNO_GOLDEN_CASES = {
    # two resolutions (scale_factor 2), SpectralConv bias, learned "frequency" position embedding, 3 blocks
    "sc2_freq": dict(inp_shape=(33, 64), out_shape=(33, 64), inp_chans=5, out_chans=3, embed_dim=8, num_layers=3, scale_factor=2,
                     model_grid_type="equiangular", sht_grid_type="legendre-gauss", bias=True, pos_embed="frequency"),
    # the shipped configuration's structure (config/sfnonet.yaml: instance norm, gelu, mlp_ratio 2, dhconv, big skip), scaled down; scale_factor 3
    "sc3_base": dict(inp_shape=(49, 96), out_shape=(49, 96), inp_chans=7, out_chans=4, embed_dim=12, num_layers=4, scale_factor=3,
                     model_grid_type="equiangular", sht_grid_type="legendre-gauss", mlp_ratio=2, normalization_layer="instance_norm",
                     hard_thresholding_fraction=1.0, use_mlp=True, operator_type="dhconv", activation_function="gelu", pos_embed="none"),
    # no norm / relu / direct position embedding / no big skip / two encoder layers
    "plain": dict(inp_shape=(32, 64), out_shape=(32, 64), inp_chans=3, out_chans=3, embed_dim=6, num_layers=2, scale_factor=2,
                  model_grid_type="legendre-gauss", sht_grid_type="legendre-gauss", normalization_layer="none", activation_function="relu",
                  pos_embed="direct", big_skip=False, encoder_layers=2),
}
GRAD_KEYS = ["blocks.0.filter.filter.weight", "blocks.1.outer_skip.weight", "encoder.fwd.0.weight"]


def main():
    import run_reference_tests as R
    from build_reference_sfno import stub_physicsnemo

    R.install_environment()
    stub_physicsnemo()
    from makani.models.networks import sfnonet

    out = {}
    for name, cfg in SFNO_GOLDEN_CASES.items():
        torch.manual_seed(333)
        net = sfnonet.SphericalFourierNeuralOperatorNet(**cfg)
        with torch.no_grad():   # non-trivial values where the reference initialises with zeros / ones
            for k, p in net.named_parameters():
                if k.endswith(".bias") or "norm" in k:
                    p.add_(0.1 * torch.randn_like(p))
        x = torch.randn(2, cfg["inp_chans"], *cfg["inp_shape"], requires_grad=True)
        y = net(x)
        g = torch.randn_like(y)
        (y * g).sum().backward()
        for k, v in net.state_dict().items():
            v = v.detach()
            out[f"{name}/sd/{k}"] = torch.view_as_real(v).numpy() if v.is_complex() else v.numpy()
        out[f"{name}/x"], out[f"{name}/y"], out[f"{name}/g"], out[f"{name}/dx"] = x.detach().numpy(), y.detach().numpy(), g.numpy(), x.grad.numpy()
        params = dict(net.named_parameters())
        for k in GRAD_KEYS:
            gr = params[k].grad
            out[f"{name}/grad/{k}"] = torch.view_as_real(gr).numpy() if gr.is_complex() else gr.numpy()
        print(name, "params", sum(p.numel() for p in net.parameters()), "y", tuple(y.shape), "|y|", float(y.abs().mean()))
    for name in SFNO_GOLDEN_CASES:
        path = os.path.join(HERE, f"sfno_golden_{name}.npz")
        np.savez_compressed(path, **{k: v for k, v in out.items() if k.startswith(name + "/")})
        print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
