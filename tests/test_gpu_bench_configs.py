"""Parity of the exact objects bench.py times, at the benched sizes (VERDICT r1 "what's weak" 2): SpectralConv(dhconv) through the
one-call C path (b200sht_spectral_conv_forward / _backward), bf16 activations + precision tf32 -- and the strict fp32 mode -- against
the CPU oracle in fp64 (oracle/makani_oracle.py, restating makani/models/common/spectral_convolution.py:213-264 on
torch-harmonics semantics).  y, residual, dx, dweight: element bound |a-b| <= rtol max|b| + rtol |b| AND relative L2."""
import pytest
import torch

from test_gpu_parity import _run_conv_case

pytestmark = pytest.mark.gpu

#            nlat_i nlon_i grid_i         nlat_o nlon_o grid_o           lmax mmax B Cin Cout G op        sep    bias
CFG_2C = (721, 1440, "equiangular", 721, 1440, "equiangular", 240, 241, 1, 73, 73, 1, "dhconv", False, False)        # bench default: sfno_block_721x1440x73
CFG_2A = (240, 480, "legendre-gauss", 240, 480, "legendre-gauss", 240, 241, 1, 384, 384, 1, "dhconv", False, False)  # sfno_block_240x480x384
CFG_2B = (721, 1440, "equiangular", 240, 480, "legendre-gauss", 240, 241, 1, 384, 384, 1, "dhconv", False, False)    # sfno_block_721to240x384 (+ residual)


@pytest.mark.parametrize("name,case", [("sfno_block_721x1440x73", CFG_2C), ("sfno_block_240x480x384", CFG_2A), ("sfno_block_721to240x384", CFG_2B)])
def test_benched_block_bf16_tf32(name, case):
    """rtol 1e-3 on the TF32 contractions (weight gradient, fp32 output), + one bf16 rounding on bf16 outputs (4e-3 element bound)."""
    rel = _run_conv_case(case, "tf32", 1e-3, act_dtype=torch.bfloat16)
    print(f"[benched] {name} bf16+tf32 rel_l2: {rel}")
    assert rel["dweight"] < 1.5e-3, rel
    for k in ("y", "dx", "residual"):
        if k in rel:
            assert rel[k] < 3e-3, (k, rel)     # bf16 output rounding alone is ~1.7e-3 rel. L2 (uniform 8-bit mantissa)


def test_benched_block_fp32_activations_tf32():
    """same object with fp32 activations: isolates the TF32 arithmetic (five TF32 stages per direction) from the bf16 output rounding"""
    rel = _run_conv_case(CFG_2C, "tf32", 1e-3, act_dtype=torch.float32)
    print(f"[benched] sfno_block_721x1440x73 fp32+tf32 rel_l2: {rel}")
    for k, v in rel.items():
        assert v < 1e-3, (k, rel)


def test_benched_block_strict_fp32():
    """precision="fp32" (the mode the reference's tests run in, TF32 disabled): rtol 1e-5"""
    rel = _run_conv_case(CFG_2C, "fp32", 1e-5, act_dtype=torch.float32)
    print(f"[benched] sfno_block_721x1440x73 fp32 rel_l2: {rel}")
    for k, v in rel.items():
        assert v < 5e-6, (k, rel)


@pytest.mark.parametrize("chunks,act_dtype", [pytest.param(2, torch.float32, id="2"), pytest.param(3, torch.float32, id="3"),
                                              pytest.param(2, torch.bfloat16, id="2-bf16"), pytest.param(3, torch.bfloat16, id="3-bf16")])
def test_benched_block_latitude_chunked_analysis(chunks, act_dtype):
    """The latitude-chunked (longitude analysis -> Legendre analysis) pair (b200sht_debug_set_lat_chunks; DESIGN.md section 10): same
    tolerances against the oracle as the unchunked path, and agreement with it up to the summation order of the Legendre sums.  bf16
    activations run the DFT's bf16 loader from a latitude offset."""
    from makani_b200 import _lib

    lib = _lib.load()
    old = lib.b200sht_debug_set_lat_chunks(1)
    try:
        ref = _run_conv_case(CFG_2C, "tf32", 1e-3, act_dtype=act_dtype, return_outputs=True)
        lib.b200sht_debug_set_lat_chunks(chunks)
        got = _run_conv_case(CFG_2C, "tf32", 1e-3, act_dtype=act_dtype, return_outputs=True)
    finally:
        lib.b200sht_debug_set_lat_chunks(old)
    bf16 = act_dtype == torch.bfloat16
    for k in ref[1]:
        a, b = got[1][k].double(), ref[1][k].double()
        d = float((a - b).norm() / b.norm())
        print(f"[chunked x{chunks} {act_dtype}] {k}: rel_l2 vs unchunked {d:.2e}, vs oracle {got[0][k]:.2e} (unchunked {ref[0][k]:.2e})")
        if bf16 and k != "dweight":
            # bf16 outputs: the fp32 differences above flip a few percent of the bf16 roundings (one bf16 unit is 2^-8 relative)
            assert d < 2e-3, (k, d)
            assert got[0][k] < 3e-3, (k, got[0])
        else:
            assert d < 5e-4, (k, d)      # measured 1.5e-4: different summation order + TF32 rounding flips of the coefficients, below the 7e-4 error against the oracle
            assert got[0][k] < (1.5e-3 if bf16 else 1e-3), (k, got[0])
