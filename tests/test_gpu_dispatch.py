"""Which kernel computed a result.  Every stage has several kernels -- the tensor-core DFT or the Stockham FFT, tcgen05 or CUDA-core
Legendre and mix, and tile / loader variants inside each -- chosen at run time from dtype, pointer alignment, nlon, batch and groups.
The tests here compare each variant with the fp64 oracle AND assert, from the CUDA kernels the profiler saw, that the intended kernel
ran, so that a change of the dispatch conditions cannot quietly turn a test into a test of another kernel.  (The longitude-transform
variants are in test_gpu_dft.py, which uses `kernels_run` from here.)"""
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest
import torch
from torch.autograd import DeviceType
from torch.profiler import ProfilerActivity, profile

import makani_b200 as mb
from makani_b200 import _lib
from test_gpu_bench_configs import CFG_2C
from test_gpu_parity import CONV_CASES, _run_conv_case, close, oracle_pair

pytestmark = pytest.mark.gpu
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def kernels_run(fn):
    """(fn(), names of the CUDA kernels it launched, one entry per launch in launch order), recorded by torch.profiler (CUPTI)"""
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    events = sorted((e for e in prof.events() if e.device_type == DeviceType.CUDA), key=lambda e: e.time_range.start)
    return out, [e.name for e in events]


def ran(names, *parts):
    """a launched kernel whose (demangled) name contains every part, e.g. ran(names, "umma_kernel", "AnaTraits")"""
    return any(all(p in n for p in parts) for n in names)


def _mix_fallback_warnings(rec):
    return [w for w in rec if issubclass(w.category, RuntimeWarning) and "tensor-core channel mix" in str(w.message)]


def test_profiler_records_library_kernels():
    """self-check of kernels_run: kernels launched by libb200sht.so (ctypes, cudaLaunchKernelEx with the PDL attribute) are recorded"""
    torch.manual_seed(333)
    x = torch.randn(1, 4, 33, 64, device=DEV)
    for precision, kernel in (("fp32", ("legendre_analysis_simt_kernel",)), ("tf32", ("umma_kernel", "AnaTraits"))):
        sht = mb.RealSHT(33, 64, 16, 17, "equiangular", precision=precision)
        _, names = kernels_run(lambda: sht(x))
        print(f"[kernels] RealSHT {precision}: {names}")
        assert ran(names, *kernel), (precision, names)


# ------------------------------------------------------------------------------------------------ SpectralConv on the tcgen05 mix
#        nlat_i nlon_i grid_i   nlat_o nlon_o grid_o   lmax mmax B Cin Cout G  op       sep    bias
_SMALL = (24, 48, "legendre-gauss", 24, 48, "legendre-gauss", 16, 17)
TC_CONV_CASES = {
    # Mt = 128 / B orders per m-tile: 32 (one ragged tile of 17), 16 (16 + 1), 4 (four full tiles + 1)
    "B4": _SMALL + (4, 8, 8, 1, "dhconv", False, True),
    "B8": _SMALL + (8, 8, 8, 1, "dhconv", False, True),
    "B32": _SMALL + (32, 8, 8, 1, "dhconv", False, True),
    # group slices of 8 -> 12 and 8 -> 8 channels on the tensor cores
    "G2": _SMALL + (1, 16, 24, 2, "dhconv", False, True),
    "G4": _SMALL + (2, 32, 32, 4, "dhconv", False, True),
    "B4G2": _SMALL + (4, 16, 24, 2, "dhconv", False, True),
    # Legendre batch tiles: analysis PBc = 3 of PB = 4 (ragged second tile), synthesis JP = 304 columns = 256 + 48
    "B2C73": (48, 96, "legendre-gauss", 48, 96, "legendre-gauss", 32, 33, 2, 73, 73, 1, "dhconv", False, True),
}


@pytest.mark.parametrize("name", list(TC_CONV_CASES))
def test_spectral_conv_tensor_core_mix(name):
    case = TC_CONV_CASES[name]
    B, Ci, Co, G = case[8:12]
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        rel, names = kernels_run(lambda: _run_conv_case(case, "tf32", 1e-3))
    print(f"[dispatch] SpectralConv {name} tf32 rel_l2: {rel}")
    for traits in ("AnaTraits", "SynTraits", "MixFwdTraits", "MixDgradTraits", "MixWgradTraits"):
        assert ran(names, "umma_kernel", traits), (traits, sorted(set(names)))
    assert not ran(names, "mix_dense_kernel") and not ran(names, "mix_wgrad_kernel"), sorted(set(names))
    assert _lib.load().b200sht_mix_uses_tensor_cores(_lib.OP_DHCONV, B, G, Ci, Co, _lib.PREC_TF32) == 1
    assert not _mix_fallback_warnings(rec), [str(w.message) for w in rec]
    for k, v in rel.items():
        assert v < 1e-3, (k, rel)


def test_spectral_conv_mix_fallback_batch_3():
    """a batch that does not divide 32: the fp32 CUDA-core mix, one RuntimeWarning (once per shape and process: channels 9 -> 11 are
    used by no other test), the same tolerances"""
    case = _SMALL + (3, 9, 11, 1, "dhconv", False, True)
    assert _lib.load().b200sht_mix_uses_tensor_cores(_lib.OP_DHCONV, 3, 1, 9, 11, _lib.PREC_TF32) == 0
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        rel, names = kernels_run(lambda: _run_conv_case(case, "tf32", 1e-3))
    print(f"[dispatch] SpectralConv B=3 tf32 (CUDA-core mix) rel_l2: {rel}")
    assert ran(names, "mix_dense_kernel"), sorted(set(names))
    assert not ran(names, "umma_kernel", "Mix"), sorted(set(names))
    assert ran(names, "umma_kernel", "AnaTraits") and ran(names, "umma_kernel", "SynTraits"), sorted(set(names))
    assert len(_mix_fallback_warnings(rec)) == 1, [str(w.message) for w in rec]
    for k, v in rel.items():
        assert v < 1e-3, (k, rel)


# ------------------------------------------------------------------------------------------------ Legendre batch / channel tiles
# analysis (umma.cu legendre_analysis_umma): batch planes in tiles of PBc when 2B > 256 / cp -- (2, 73): 3 + 1 planes; (4, 40): 6 + 2;
# (3, 200): two channel tiles of 100 x three tiles of 2 planes.  synthesis: JP = 2B cp columns in tiles of 256: 304, 320, 1200.
@pytest.mark.parametrize("precision", ["tf32", "fp32x3"])
@pytest.mark.parametrize("B,C", [(2, 73), (4, 40), (3, 200)])
def test_legendre_batch_tiles(B, C, precision):
    grid, nlat, nlon, lmax, mmax = "legendre-gauss", 48, 96, 32, 33
    torch.manual_seed(333)
    sht = mb.RealSHT(nlat, nlon, lmax, mmax, grid, precision=precision)
    isht = mb.InverseRealSHT(nlat, nlon, lmax, mmax, grid, precision=precision)
    osht, oisht = oracle_pair(nlat, nlon, nlat, nlon, lmax, mmax, grid, grid)
    x = torch.randn(B, C, nlat, nlon)
    gc = torch.randn(B, C, lmax, mmax, dtype=torch.complex64)
    cin = torch.randn(B, C, lmax, mmax, dtype=torch.complex64)
    gy = torch.randn(B, C, nlat, nlon)

    def run():
        xd = x.to(DEV).requires_grad_(True)
        c = sht(xd)
        c.backward(gc.to(DEV))
        cd = cin.to(DEV).requires_grad_(True)
        y = isht(cd)
        y.backward(gy.to(DEV))
        return c, xd.grad, y, cd.grad

    (c, gx, y, gcin), names = kernels_run(run)
    assert ran(names, "umma_kernel", "AnaTraits") and ran(names, "umma_kernel", "SynTraits"), sorted(set(names))
    assert not ran(names, "legendre_analysis_simt") and not ran(names, "legendre_synthesis_simt"), sorted(set(names))
    xr = x.double().requires_grad_(True)
    cr = osht(xr)
    cr.backward(gc.to(torch.complex128))
    cinr = cin.to(torch.complex128).requires_grad_(True)
    yr = oisht(cinr)
    yr.backward(gy.double())
    keep = torch.tril(torch.ones(lmax, mmax)).bool()   # the oracle's gradient for l < m is exactly zero as well (P = 0)
    rtol, bound = (1e-3, {"analysis": 6e-4, "synthesis": 1e-3}) if precision == "tf32" else (1e-5, {"analysis": 6e-6, "synthesis": 6e-6})
    tag = f"B={B} C={C} {precision}"
    for what, a, b, kind in (("RealSHT", c, cr, "analysis"), ("dRealSHT/dx", gx, xr.grad, "synthesis"), ("InverseRealSHT", y, yr, "synthesis"),
                             ("dInverseRealSHT/dc", gcin * keep.to(DEV), cinr.grad * keep, "analysis")):
        rel = close(a, b, rtol, f"legendre tiles {tag} {what}")
        assert rel < bound[kind], (what, rel)


# ------------------------------------------------------------------------------------------------ overlapped backward schedule
def _conv_grads(case, act_dtype, event):
    (nlat_i, nlon_i, grid_i, nlat_o, nlon_o, grid_o, lmax, mmax, B, Cin, Cout, G, op, sep, bias) = case
    torch.manual_seed(333)
    f = mb.RealSHT(nlat_i, nlon_i, lmax, mmax, grid_i, precision="tf32")
    i = mb.InverseRealSHT(nlat_o, nlon_o, lmax, mmax, grid_o, precision="tf32")
    conv = mb.SpectralConv(f, i, Cin, Cout, num_groups=G, operator_type=op, separable=sep, bias=bias, precision="tf32").to(DEV)
    if bias:
        with torch.no_grad():
            conv.bias.copy_(torch.randn_like(conv.bias))
    if event is not None:
        conv.wgrad_ready_event = event
    xd = torch.randn(B, Cin, nlat_i, nlon_i).to(act_dtype).to(DEV).requires_grad_(True)
    y, _ = conv(xd)
    y.backward(torch.randn(y.shape).to(act_dtype).to(DEV))
    torch.cuda.synchronize()
    return {"dx": xd.grad, "dweight": conv.weight.grad, **({"dbias": conv.bias.grad} if bias else {})}


@pytest.mark.parametrize("name,case,act_dtype", [("cfg2c_bf16", CFG_2C, torch.bfloat16), ("small_fp32_bias", CONV_CASES[0], torch.float32)])
def test_backward_with_wgrad_event_is_bit_identical(name, case, act_dtype):
    """b200sht_spectral_conv_backward_ex with an event: the weight gradient first, the mix input gradient split off, SMs reserved for a
    collective (fewer persistent CTAs) and PDL off.  Fewer CTAs change which CTA computes a tile, not its arithmetic: same bits."""
    plain = _conv_grads(case, act_dtype, None)
    ev = torch.cuda.Event()
    overlapped = _conv_grads(case, act_dtype, ev)
    assert ev.cuda_event != 0, "the event was never handed to the library (it has no CUDA event behind it)"
    assert ev.query(), "the weight-gradient event has not completed after a synchronise"
    for k in plain:
        assert torch.isfinite(plain[k].abs()).all(), k
        assert torch.equal(overlapped[k], plain[k]), (name, k, float((overlapped[k] - plain[k]).abs().max()))


# ------------------------------------------------------------------------------------------------ latitude-chunked synthesis
_CHILD = """
import os, sys
import numpy as np, torch
sys.path[:0] = [{root!r}, {tests!r}]
from test_gpu_bench_configs import CFG_2C
from test_gpu_dispatch import kernels_run
from test_gpu_parity import _run_conv_case
(rel, out), names = kernels_run(lambda: _run_conv_case(CFG_2C, "tf32", 1e-3, act_dtype=torch.float32, return_outputs=True))
print("[chunked syn] rel_l2 vs oracle", rel, "dft_synthesis launches", sum("dft_synthesis_kernel" in n for n in names))
assert all(v < 1e-3 for v in rel.values()), rel
for k, v in out.items():
    np.save(os.path.join({dst!r}, k + ".npy"), v.numpy())
np.save(os.path.join({dst!r}, "syn_launches.npy"), np.array(sum("dft_synthesis_kernel" in n for n in names)))
"""


def test_latitude_chunked_synthesis_is_bit_identical(tmp_path):
    """B200SHT_LAT_CHUNKS_SYN (read once per process: each setting in its own process): the chunks are 128-row multiples of the same
    tiles, so y, dx and dweight equal the unchunked ones bit for bit (and stay within the oracle tolerance)."""
    out = {}
    for n in (None, 2, 3):
        env = dict(os.environ)
        env.pop("B200SHT_LAT_CHUNKS_SYN", None)
        if n is not None:
            env["B200SHT_LAT_CHUNKS_SYN"] = str(n)
        dst = tmp_path / f"chunks{n or 1}"
        dst.mkdir()
        code = _CHILD.format(root=ROOT, tests=os.path.join(ROOT, "tests"), dst=str(dst))
        r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
        print(r.stdout[-2000:])
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
        out[n or 1] = {k: np.load(dst / f"{k}.npy") for k in ("y", "dx", "dweight", "syn_launches")}
    # one synthesis pair for y and one for dx, each split into n latitude chunks
    for n in (1, 2, 3):
        assert int(out[n]["syn_launches"]) == 2 * n, (n, out[n]["syn_launches"])
    for n in (2, 3):
        for k in ("y", "dx", "dweight"):
            assert np.array_equal(out[n][k], out[1][k]), (n, k, float(np.abs(out[n][k] - out[1][k]).max()))
