"""makani_b200/sfno.py (NeuralOperatorBlock + SphericalFourierNeuralOperatorNet restated, SURVEY rows A8/A9) against golden vectors produced
by the REFERENCE's own network class (tests/golden/make_sfno_golden.py: /root/reference/makani/models/networks/sfnonet.py on the oracle).
CPU: the network logic on the oracle backend (same arithmetic as the golden run) and the parameter surface of the CUDA-backed network."""
import os
import sys

import numpy as np
import pytest
import torch

from makani_b200.sfno import SphericalFourierNeuralOperatorNet
from oracle.sfno_backend import OracleBackend

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from make_sfno_golden import GRAD_KEYS, SFNO_GOLDEN_CASES  # noqa: E402

GOLDEN_DIR = os.path.join(os.path.dirname(__file__), "golden")


def load_golden(name):
    """the arrays of one case (keys `<name>/...`), one file per case to keep each file small"""
    return np.load(os.path.join(GOLDEN_DIR, f"sfno_golden_{name}.npz"))


def golden_state_dict(g, name):
    sd = {}
    for k in g.files:
        if k.startswith(f"{name}/sd/"):
            v = torch.from_numpy(g[k])
            key = k[len(f"{name}/sd/"):]
            sd[key] = torch.view_as_complex(v.contiguous()) if (key.endswith("filter.filter.weight") and v.shape[-1] == 2 and v.dtype == torch.float32) else v
    return sd


@pytest.mark.parametrize("name", sorted(SFNO_GOLDEN_CASES))
def test_network_on_oracle_backend_matches_reference_network(name):
    g = load_golden(name)
    torch.manual_seed(0)
    net = SphericalFourierNeuralOperatorNet(**SFNO_GOLDEN_CASES[name], backend=OracleBackend())
    sd = golden_state_dict(g, name)
    assert sorted(net.state_dict().keys()) == sorted(sd.keys())
    net.load_state_dict(sd, strict=True)
    x = torch.from_numpy(g[f"{name}/x"]).requires_grad_(True)
    y = net(x)
    assert torch.allclose(y, torch.from_numpy(g[f"{name}/y"]), rtol=1e-4, atol=1e-5), (y - torch.from_numpy(g[f"{name}/y"])).abs().max()
    (y * torch.from_numpy(g[f"{name}/g"])).sum().backward()
    assert torch.allclose(x.grad, torch.from_numpy(g[f"{name}/dx"]), rtol=1e-3, atol=1e-4)
    params = dict(net.named_parameters())
    for k in GRAD_KEYS:
        ref = torch.from_numpy(g[f"{name}/grad/{k}"])
        got = params[k].grad
        got = torch.view_as_real(got) if got.is_complex() else got
        assert torch.allclose(got, ref, rtol=1e-3, atol=1e-4 * ref.abs().max().item() + 1e-6), k


@pytest.mark.parametrize("name", sorted(SFNO_GOLDEN_CASES))
def test_cuda_backed_network_has_the_reference_parameter_surface(name):
    """constructed on CPU (plans are created lazily on the device): names, shapes, dtypes of every state-dict entry, and the checkpoint loads"""
    g = load_golden(name)
    net = SphericalFourierNeuralOperatorNet(**SFNO_GOLDEN_CASES[name], precision="fp32")
    sd = golden_state_dict(g, name)
    mine = net.state_dict()
    assert sorted(mine.keys()) == sorted(sd.keys())
    for k, v in sd.items():
        assert tuple(mine[k].shape) == tuple(v.shape) and mine[k].dtype == v.dtype, k
    net.load_state_dict(sd, strict=True)
