"""GPU tests of the tensor-core longitude DFT (csrc/dft.cu) through the C ABI: b200sht_fft_analysis / _synthesis with the TF32
precision bit (scale_mode | 2) against torch.fft in fp64 -- the semantics of torch_harmonics.RealSHT / InverseRealSHT along
longitude (2 pi rfft(norm="forward")[..., :mmax], irfft(norm="forward"); SURVEY App. A).  Tolerance: TF32 contraction, rtol 1e-3
(BASELINE north_star "1e-3 bf16"); rel-L2 printed and asserted as well."""
import math

import pytest
import torch

import makani_b200 as mb
from makani_b200 import _lib
from oracle import makani_oracle as O
from test_gpu_dispatch import kernels_run, ran
from test_gpu_parity import close

pytestmark = pytest.mark.gpu
DEV = "cuda"

# (nlat, nlon, mmax, C, dtype): N2/2+1 <= 32 (4 replicas), <= 64 (2 replicas), <= 96; odd N2; Nyquist order present; ragged nlat
CASES = [
    (64, 128, 65, 8, torch.float32),       # BASELINE cfg 1 grid, all orders incl. Nyquist
    (33, 72, 30, 5, torch.float32),        # N2 = 9 (odd)
    (721, 1440, 241, 3, torch.bfloat16),   # headline grid
    (721, 1440, 241, 2, torch.float32),
    (240, 480, 241, 6, torch.float32),     # interior SFNO grid, all orders
    (240, 480, 241, 5, torch.bfloat16),
    (45, 360, 100, 2, torch.bfloat16),     # N2 = 45 (odd)
    (181, 720, 121, 3, torch.float32),     # N2 = 90: two lane quadrants
    (7, 1512, 256, 2, torch.float32),      # largest supported length class (N2 = 189, odd)
    (19, 16, 9, 3, torch.float32),         # smallest
]
# The analysis kernel reads fp32 rows only when nlon % 32 == 0 (16-byte TMA boxes; otherwise fft_analysis runs the Stockham FFT):
# test_dft_analysis_gpu runs the other fp32 entries of CASES as bf16.  Its further cases cover the analysis variants of dft.cu --
# bf16 box groups gs = 1 / 4 / 8 (dft_box_group), one / two / three K-blocks (N2/2 + 1 <= 32 / 64 / 96), the N2 = 90 specialisation --
# at ragged nlat, with mmax truncated or up to the Nyquist order.
ANALYSIS_CASES = [
    (7, 16, 9, 3, torch.bfloat16),         # N2 = 2, gs 4, Nyquist
    (45, 16, 5, 2, torch.bfloat16),
    (19, 72, 37, 3, torch.bfloat16),       # N2 = 9 (odd), gs 8, 4 replicas, Nyquist
    (181, 72, 20, 2, torch.bfloat16),
    (45, 128, 65, 2, torch.bfloat16),      # gs 1, Nyquist
    (7, 128, 30, 3, torch.bfloat16),
    (181, 720, 241, 2, torch.bfloat16),    # N2 = 90 template, gs 4, two K-blocks: the 360 x 720 inner grid of SFNO scale_factor 2
    (19, 720, 256, 3, torch.bfloat16),
    (7, 1024, 256, 2, torch.bfloat16),     # gs 1, three K-blocks
    (45, 1024, 100, 3, torch.bfloat16),
    (19, 1512, 256, 2, torch.bfloat16),    # N2 = 189 (odd, largest), gs 8, three K-blocks
    (181, 1512, 121, 2, torch.bfloat16),
    (45, 256, 129, 3, torch.float32),      # Nyquist
    (181, 256, 60, 2, torch.float32),
    (19, 1024, 256, 2, torch.float32),     # three K-blocks
    (7, 1024, 33, 3, torch.float32),
]


def _latview(lat, plan, B, C, mmax):
    return lat[: mmax * 2 * B * C * plan.kp].view(mmax, 2, B * C, plan.kp)


def _analysis_vs_rfft(lat, x, plan, mode, rtol, name):
    """latspec written by b200sht_fft_analysis (scale mode 0 or 1) against 2 pi rfft in fp64 (mode 0: times the quadrature weights)"""
    B, C, nlat, nlon = x.shape
    mmax = plan.mmax
    X = _latview(lat, plan, B, C, mmax)
    got = torch.complex(X[:, 0, :, :nlat], X[:, 1, :, :nlat]).permute(1, 2, 0).reshape(B, C, nlat, mmax)
    assert (X[..., nlat:] == 0).all(), "latitude padding must hold exact zeros"
    ref = torch.fft.rfft(x.double().cpu(), dim=-1)[..., :mmax]
    if mode == 0:
        _, w = O.precompute_latitudes(nlat, "equiangular")
        ref = ref * (torch.from_numpy(w) * 2 * math.pi / nlon)[:, None]
    else:
        ms = torch.full((mmax,), 2.0, dtype=torch.float64)
        ms[0] = 1
        if mmax - 1 == nlon // 2:
            ms[-1] = 1
        ref = ref * ms
    return close(got, ref, rtol, name)


def to_tiled(Z, plan):
    """standard latspec [mmax][2][R][kp] -> the tiled layout [R][kp/8][2][M2][8][8] (orders zero-padded to 8 * M2) that
    b200sht_legendre_synthesis_tiled writes and b200sht_fft_synthesis(scale_mode | 2) reads (include/b200sht.h)"""
    mmax, _, R, kp = Z.shape
    M2 = (mmax + 7) // 8
    Zp = torch.zeros(8 * M2, 2, R, kp, device=Z.device, dtype=Z.dtype)
    Zp[:mmax] = Z
    # (m2, c, p, r, kt, k8) -> (r, kt, p, m2, c, k8)
    return Zp.view(M2, 8, 2, R, kp // 8, 8).permute(3, 4, 2, 0, 1, 5).contiguous().reshape(-1)


@pytest.mark.parametrize("nlat,nlon,mmax,C,dtype", CASES + ANALYSIS_CASES)
def test_dft_analysis_gpu(nlat, nlon, mmax, C, dtype):
    if dtype == torch.float32 and nlon % 32:
        dtype = torch.bfloat16
    torch.manual_seed(333)
    plan = mb.get_plan(nlat, nlon, min(nlat, 16), mmax, "equiangular", True, torch.device(DEV))
    B = 2
    x = torch.randn(B, C, nlat, nlon, device=DEV).to(dtype)
    st = mb.sht._stream(x.device)
    N2 = nlon // 8
    for mode in (0, 1):
        lat = torch.full((plan.latspec_elems(B, C),), float("nan"), device=DEV)
        _, names = kernels_run(lambda: _lib.call("b200sht_fft_analysis", plan.handle, mb.sht._ptr(x), mb.sht._dtype_code(dtype), B, C, mb.sht._ptr(lat),
                                                 mode | 2, st))
        assert ran(names, "dft_analysis_kernel<", f", {N2 if N2 in (60, 90, 180) else 0}>"), names
        rel = _analysis_vs_rfft(lat, x, plan, mode, 1e-3, f"dft_analysis mode{mode} {nlat}x{nlon} mmax={mmax} {dtype}")
        assert rel < 6e-4, rel


def test_fp32_input_at_nlon_720_runs_stockham_rounded_to_tf32():
    """fp32 rows of 720 samples cannot be read by the DFT's TMA boxes: with the TF32 bit the Stockham FFT runs and rounds its output to
    TF32 (it feeds the tcgen05 Legendre GEMM)"""
    torch.manual_seed(335)
    nlat, nlon, mmax, B, C = 45, 720, 241, 2, 3
    plan = mb.get_plan(nlat, nlon, 16, mmax, "equiangular", True, torch.device(DEV))
    assert plan.query(8) == 1
    x = torch.randn(B, C, nlat, nlon, device=DEV)
    st = mb.sht._stream(x.device)
    for mode in (0, 1):
        lat = torch.full((plan.latspec_elems(B, C),), float("nan"), device=DEV)
        _, names = kernels_run(lambda: _lib.call("b200sht_fft_analysis", plan.handle, mb.sht._ptr(x), 0, B, C, mb.sht._ptr(lat), mode | 2, st))
        assert ran(names, "fft_analysis_") and not ran(names, "dft_analysis_kernel"), names
        X = _latview(lat, plan, B, C, mmax)
        assert (X.view(torch.int32) & 0x1FFF == 0).all(), "output not rounded to TF32"
        rel = _analysis_vs_rfft(lat, x, plan, mode, 1e-3, f"stockham+tf32 mode{mode} {nlat}x{nlon} fp32")
        assert rel < 6e-4, rel


def test_misaligned_bf16_input_runs_stockham():
    """bf16 721 x 1440 samples 2 bytes off a 16-byte boundary: TMA cannot address them, the Stockham FFT runs -- through the C ABI and
    through RealSHT(precision="tf32") on a contiguous view with a storage offset"""
    torch.manual_seed(336)
    nlat, nlon, lmax, mmax, B, C = 721, 1440, 240, 241, 1, 2
    plan = mb.get_plan(nlat, nlon, lmax, mmax, "equiangular", True, torch.device(DEV))
    assert plan.query(8) == 1
    buf = torch.randn(B * C * nlat * nlon + 1, device=DEV).to(torch.bfloat16)
    x = buf[1:].view(B, C, nlat, nlon)
    assert x.is_contiguous() and x.data_ptr() % 16 == 2
    st = mb.sht._stream(x.device)
    lat = torch.full((plan.latspec_elems(B, C),), float("nan"), device=DEV)
    _, names = kernels_run(lambda: _lib.call("b200sht_fft_analysis", plan.handle, mb.sht._ptr(x), _lib.BF16, B, C, mb.sht._ptr(lat), 0 | 2, st))
    assert ran(names, "fft_analysis_") and not ran(names, "dft_analysis_kernel"), names
    rel = _analysis_vs_rfft(lat, x, plan, 0, 1e-3, f"misaligned bf16 fft_analysis {nlat}x{nlon}")
    assert rel < 6e-4, rel
    sht = mb.RealSHT(nlat, nlon, lmax, mmax, "equiangular", precision="tf32")
    c, names = kernels_run(lambda: sht(x))
    assert ran(names, "fft_analysis_") and not ran(names, "dft_analysis_kernel"), names
    assert ran(names, "umma_kernel", "AnaTraits"), names
    rel = close(c, O.RealSHT(nlat, nlon, lmax, mmax, "equiangular", dtype=torch.float64)(x.double().cpu()), 1e-3, "misaligned bf16 RealSHT tf32")
    assert rel < 1e-3, rel


@pytest.mark.parametrize("nlat,nlon,mmax,C,dtype", CASES)
def test_dft_synthesis_gpu(nlat, nlon, mmax, C, dtype):
    torch.manual_seed(334)
    plan = mb.get_plan(nlat, nlon, min(nlat, 16), mmax, "equiangular", True, torch.device(DEV))
    assert plan.query(8) == 1
    B = 2
    st = mb.sht._stream(torch.device(DEV))
    Z = torch.randn(mmax, 2, B * C, plan.kp, device=DEV)
    # operands of the kind::tf32 GEMM are TF32 values in the product path (the Legendre epilogue rounds): do the same here
    Z = (Z.view(torch.int32) + 0x1000).bitwise_and(~0x1FFF).view(torch.float32)
    lat = to_tiled(Z, plan)
    assert lat.numel() == plan.latspec_elems(B, C)
    bias = torch.randn(C, device=DEV)
    Zc = torch.complex(Z[:, 0, :, :nlat], Z[:, 1, :, :nlat]).permute(1, 2, 0).reshape(B, C, nlat, mmax).to(torch.complex128).cpu()
    y = torch.full((B, C, nlat, nlon), float("nan"), device=DEV, dtype=dtype)
    _, names = kernels_run(lambda: _lib.call("b200sht_fft_synthesis", plan.handle, mb.sht._ptr(lat), mb.sht._ptr(y), mb.sht._dtype_code(dtype), B, C,
                                             mb.sht._ptr(bias), 0 | 2, st))
    assert ran(names, "dft_synthesis_kernel<"), names
    ref = torch.fft.irfft(Zc, n=nlon, dim=-1, norm="forward") + bias.double().cpu()[None, :, None, None]
    rel = close(y, ref, 1e-3 if dtype == torch.float32 else 4e-3, f"dft_synthesis mode0 {nlat}x{nlon} mmax={mmax} {dtype}")
    assert rel < (6e-4 if dtype == torch.float32 else 3e-3), rel
    # mode 1 = adjoint of the mode-0 analysis: y = rowscale[k] * sum_m Re(Z[m] exp(i m phi))
    y1 = torch.full((B, C, nlat, nlon), float("nan"), device=DEV, dtype=dtype)
    _lib.call("b200sht_fft_synthesis", plan.handle, mb.sht._ptr(lat), mb.sht._ptr(y1), mb.sht._dtype_code(dtype), B, C, mb.sht._VP(0), 1 | 2, st)
    _, w = O.precompute_latitudes(nlat, "equiangular")
    half = Zc.clone()
    half[..., 1:] *= 0.5
    if mmax - 1 == nlon // 2:
        half[..., -1] *= 2.0
    ref1 = torch.fft.irfft(half, n=nlon, dim=-1, norm="forward") * (torch.from_numpy(w) * 2 * math.pi / nlon)[:, None]
    rel = close(y1, ref1, 1e-3 if dtype == torch.float32 else 4e-3, f"dft_synthesis mode1 {nlat}x{nlon} mmax={mmax} {dtype}")
    assert rel < (6e-4 if dtype == torch.float32 else 3e-3), rel


def test_dft_adjoint_pair_full_size():
    """<A x, Z> = <x, A^T Z> at the headline size (size-independent property): mode-0 analysis against mode-1 synthesis."""
    torch.manual_seed(5)
    nlat, nlon, mmax, B, C = 721, 1440, 241, 1, 4
    plan = mb.get_plan(nlat, nlon, 16, mmax, "equiangular", True, torch.device(DEV))
    st = mb.sht._stream(torch.device(DEV))
    x = torch.randn(B, C, nlat, nlon, device=DEV)
    lat = torch.zeros(plan.latspec_elems(B, C), device=DEV)
    _lib.call("b200sht_fft_analysis", plan.handle, mb.sht._ptr(x), 0, B, C, mb.sht._ptr(lat), 0 | 2, st)
    Ax = _latview(lat, plan, B, C, mmax).clone()
    Z = torch.randn(mmax, 2, B * C, plan.kp, device=DEV)
    lat2 = to_tiled(Z, plan)
    y = torch.empty(B, C, nlat, nlon, device=DEV)
    _lib.call("b200sht_fft_synthesis", plan.handle, mb.sht._ptr(lat2), mb.sht._ptr(y), 0, B, C, mb.sht._VP(0), 1 | 2, st)
    lhs = (Ax[..., :nlat].double() * Z[..., :nlat].double()).sum().item()
    rhs = (x.double() * y.double()).sum().item()
    assert abs(lhs - rhs) <= 2e-3 * max(abs(lhs), abs(rhs), 1.0), (lhs, rhs)


@pytest.mark.parametrize("grid,nlat,nlon,lmax,mmax,B,C", [("equiangular", 64, 128, 64, 65, 1, 8), ("legendre-gauss", 48, 96, 32, 33, 2, 5), ("equiangular", 721, 1440, 240, 241, 1, 3)])
def test_legendre_synthesis_tiled_is_a_relayout(grid, nlat, nlon, lmax, mmax, B, C):
    """b200sht_legendre_synthesis_tiled writes exactly the values of b200sht_legendre_synthesis(TF32) in the tiled layout, with exact
    zeros in the padding orders -- bit-identical (same kernel, different epilogue addressing)."""
    torch.manual_seed(7)
    plan = mb.get_plan(nlat, nlon, lmax, mmax, grid, True, torch.device(DEV))
    assert plan.query(8) == 1
    st = mb.sht._stream(torch.device(DEV))
    sp = torch.randn(plan.spec_elems(B, C), device=DEV)
    std = torch.full((plan.latspec_elems(B, C),), float("nan"), device=DEV)
    til = torch.full((plan.latspec_elems(B, C),), float("nan"), device=DEV)
    _lib.call("b200sht_legendre_synthesis", plan.handle, mb.sht._ptr(sp), mb.sht._ptr(std), B, C, _lib.PREC_TF32, st)
    _lib.call("b200sht_legendre_synthesis_tiled", plan.handle, mb.sht._ptr(sp), mb.sht._ptr(til), B, C, st)
    ref = to_tiled(_latview(std, plan, B, C, mmax), plan)
    assert torch.isfinite(til).all()
    assert torch.equal(til, ref)
