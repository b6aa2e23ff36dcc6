#!/usr/bin/env python
"""Golden data for tests/test_reference_suites.py, produced by the REFERENCE's own code (a makani checkout at $MAKANI_REFERENCE) so that
those tests run without it:

  reference_sht_boundary.npz          the calls the reference's loss / grid / noise suites make into torch_harmonics (the oracle's
                                      transforms, makani_b200.quadrature), recorded by run_reference_tests.py --record
  reference_sfno_surface.json         parameter names / shapes / dtypes / model-parallel tags, state-dict keys and output shape of the
                                      reference's SphericalFourierNeuralOperatorNet on the oracle (build_reference_sfno.py a)
  reference_dist_conv_inputs.npz      one case of the reference's distributed SpectralConv test (91 x 180 -> 91 x 180, B = 1, C = 4):
  reference_dist_conv_outputs.npz     the serial reference SpectralConv (operator dhconv, bias) on the oracle transforms, its input,
                                      weight, bias and output gradient, and its output and gradients (two files: each stays under 1 MB)

    MAKANI_REFERENCE=<makani checkout> python tests/golden/make_reference_suite_golden.py
"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
SUITES = os.path.join(HERE, "..", "reference_suites")
sys.path.insert(0, SUITES)

DIST_CASE = dict(nlat_in=91, nlon_in=180, nlat_out=91, nlon_out=180, batch_size=1, num_chan=4, tol=1e-4)


def sfno_surface():
    out = {}
    for variant in ("linear", "nonlinear"):
        r = subprocess.run([sys.executable, os.path.join(SUITES, "build_reference_sfno.py"), "a", variant], capture_output=True, text=True, check=True)
        out[variant] = json.loads(r.stdout.strip().splitlines()[-1])
    with open(os.path.join(HERE, "reference_sfno_surface.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)


def dist_conv_case():
    """the serial half of the reference's test_distributed_spectral_conv for DIST_CASE (same construction, seed and draws)"""
    import run_reference_tests as R
    from build_reference_sfno import stub_physicsnemo

    R.install_environment()
    stub_physicsnemo()
    import torch_harmonics as th
    from makani.models.common import SpectralConv

    c = DIST_CASE
    B, C = c["batch_size"], c["num_chan"]
    fwd = th.RealSHT(nlat=c["nlat_in"], nlon=c["nlon_in"])
    inv = th.InverseRealSHT(nlat=c["nlat_out"], nlon=c["nlon_out"], lmax=fwd.lmax, mmax=fwd.mmax)
    torch.manual_seed(333)
    conv = SpectralConv(fwd, inv, C, C, operator_type="dhconv", num_groups=1, bias=True, gain=1.0)
    x = torch.randn((B, C, c["nlat_in"], c["nlon_in"]), dtype=torch.float32, requires_grad=True)
    y, _ = conv(x)
    gy = torch.randn_like(y)
    y.backward(gy)
    real = lambda t: (torch.view_as_real(t) if t.is_complex() else t).detach().numpy()
    np.savez_compressed(os.path.join(HERE, "reference_dist_conv_inputs.npz"), case=np.array(json.dumps(c)), x=real(x), gy=real(gy),
                        weight=real(conv.weight), bias=real(conv.bias))
    np.savez_compressed(os.path.join(HERE, "reference_dist_conv_outputs.npz"), y=real(y), dx=real(x.grad), dweight=real(conv.weight.grad),
                        dbias=real(conv.bias.grad))


def main():
    if not os.path.isdir(os.environ.get("MAKANI_REFERENCE", "")):
        raise SystemExit("set MAKANI_REFERENCE to a makani checkout")
    subprocess.run([sys.executable, os.path.join(SUITES, "run_reference_tests.py"), "--record", os.path.join(HERE, "reference_sht_boundary.npz")],
                   check=True)
    sfno_surface()
    # own process: install_environment() replaces sys.modules entries
    subprocess.run([sys.executable, os.path.abspath(__file__), "--dist-conv"], check=True)


if __name__ == "__main__":
    if "--dist-conv" in sys.argv:
        dist_conv_case()
    else:
        main()
