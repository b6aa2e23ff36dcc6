"""SURVEY rows A8 / A9 on the GPU: the SFNO network (makani_b200/sfno.py: NeuralOperatorBlock, SphericalFourierNeuralOperatorNet) running on the
CUDA spherical-harmonic kernels, loaded with the REFERENCE network's state dict and compared with the REFERENCE network's output and gradients
(tests/golden/sfno_golden_<case>.npz, produced by makani's makani/models/networks/sfnonet.py on the CPU oracle, tests/golden/make_sfno_golden.py)."""
import os
import sys

import numpy as np
import pytest
import torch

from makani_b200.sfno import SphericalFourierNeuralOperatorNet
from test_gpu_parity import close

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from make_sfno_golden import GRAD_KEYS, SFNO_GOLDEN_CASES  # noqa: E402
from test_sfno_cpu import golden_state_dict, load_golden  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture
def torch_tf32(request):
    """PyTorch's own 1x1 convolutions (encoder / MLP / skips) follow torch.backends.*.allow_tf32; the strict-fp32 comparison switches it off,
    as the reference's tests do (tests/testutils.py:55-66 disable_tf32)."""
    prev = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev


@pytest.mark.parametrize("name", sorted(SFNO_GOLDEN_CASES))
@pytest.mark.parametrize("precision,rtol,grtol", [("fp32", 2e-4, 5e-4), ("tf32", 4e-3, 1.5e-2)])
def test_sfno_network_matches_reference_network(name, precision, rtol, grtol, torch_tf32):
    """fp32: the golden run is itself fp32 (oracle einsums), so the bound is a few fp32 roundings through 2-4 blocks; tf32: five TF32 stages per
    transform pair and block (+ cuDNN TF32 convolutions), amplified through the instance norms in the gradients (grtol).  The ReLU network
    ("plain") is compared in its output only at TF32: a 1e-3 perturbation flips ReLU gates, its gradient is not a continuous function."""
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = (precision == "tf32")
    g = load_golden(name)
    net = SphericalFourierNeuralOperatorNet(**SFNO_GOLDEN_CASES[name], precision=precision)
    net.load_state_dict(golden_state_dict(g, name), strict=True)
    net = net.to(DEV)
    x = torch.from_numpy(g[f"{name}/x"]).to(DEV).requires_grad_(True)
    y = net(x)
    close(y, torch.from_numpy(g[f"{name}/y"]), rtol, f"SFNO[{name},{precision}] y")
    (y * torch.from_numpy(g[f"{name}/g"]).to(DEV)).sum().backward()
    if precision == "tf32" and SFNO_GOLDEN_CASES[name].get("activation_function") == "relu":
        assert torch.isfinite(x.grad).all()
        return
    close(x.grad, torch.from_numpy(g[f"{name}/dx"]), grtol, f"SFNO[{name},{precision}] dx")
    params = dict(net.named_parameters())
    for k in GRAD_KEYS:
        ref = torch.from_numpy(g[f"{name}/grad/{k}"])
        got = params[k].grad
        got = torch.view_as_real(got) if got.is_complex() else got
        close(got, ref, grtol, f"SFNO[{name},{precision}] d{k}")


def test_sfno_network_bf16_autocast_runs_and_is_close():
    """the way the reference trains (bf16 autocast around the network; the transforms stay fp32/TF32): loose agreement with the fp32 golden output"""
    name = "sc3_base"
    g = load_golden(name)
    net = SphericalFourierNeuralOperatorNet(**SFNO_GOLDEN_CASES[name], precision="tf32")
    net.load_state_dict(golden_state_dict(g, name), strict=True)
    net = net.to(DEV)
    x = torch.from_numpy(g[f"{name}/x"]).to(DEV).requires_grad_(True)
    with torch.autocast(device_type="cuda", dtype=torch.bfloat16):
        y = net(x)
    yref = torch.from_numpy(g[f"{name}/y"])
    rel = ((y.float().cpu() - yref).norm() / yref.norm()).item()
    print(f"[parity] SFNO[{name}] bf16 autocast rel_l2={rel:.3e}")
    assert torch.isfinite(y).all() and rel < 5e-2
    y.float().square().mean().backward()
    assert torch.isfinite(x.grad).all()
