#!/usr/bin/env python
"""Kernel-by-kernel check of the tcgen05 path against the fp32 CUDA-core kernels (same C ABI, precision flag only).

    python scripts/umma_diag.py all            # every (kernel, case) in its own subprocess (a trap cannot poison the rest)
    python scripts/umma_diag.py <kernel> <case>

Unstored entries of the packed spectra (l < 32*floor(m/32)) are filled with NaN to prove no kernel reads them.
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = {
    # name: (nlat, nlon, L, M, grid, B, Ci, Co, G)
    "small": (33, 64, 16, 17, "equiangular", 1, 8, 8, 1),
    "odd": (91, 180, 91, 91, "equiangular", 2, 5, 7, 1),
    "tiles": (181, 360, 181, 181, "legendre-gauss", 1, 16, 24, 2),     # two groups of 8 -> 12 channels
    "cfg2c": (721, 1440, 240, 241, "equiangular", 1, 73, 73, 1),
    "wide": (64, 128, 64, 65, "legendre-gauss", 1, 200, 136, 1),
    "cfg2a": (240, 480, 240, 241, "legendre-gauss", 1, 384, 384, 1),
    "wide3": (64, 128, 64, 65, "legendre-gauss", 1, 300, 330, 1),     # three ragged column tiles
}
KERNELS = ["analysis", "synthesis", "mix_fwd", "mix_dgrad", "mix_wgrad"]


def run_one(kernel, case):
    import torch

    import makani_b200 as mb
    from makani_b200 import _lib
    from makani_b200.sht import _ptr, _stream

    nlat, nlon, L, M, grid, B, Ci, Co, G = CASES[case]
    dev = torch.device("cuda", 0)
    torch.manual_seed(333)
    plan = mb.get_plan(nlat, nlon, L, M, grid, True, dev)
    st = _stream(dev)
    lib = _lib.load()

    def spec_rand(C):
        cp = (C + 3) // 4 * 4
        t = torch.randn(L, M, 2 * B, cp, device=dev)
        t[..., C:] = 0
        l = torch.arange(L, device=dev)[:, None]
        m = torch.arange(M, device=dev)[None, :]
        unstored = l < (m // 32) * 32
        t[unstored] = float("nan")
        return t, unstored

    def report(name, a, b, mask=None):
        if mask is not None:
            a = a[~mask]
            b = b[~mask]
        fin = bool(torch.isfinite(a).all())
        rel = ((a - b).double().norm() / b.double().norm().clamp_min(1e-30)).item()
        mx = (a - b).abs().max().item()
        print(json.dumps({"kernel": kernel, "case": case, "what": name, "finite": fin, "rel_l2": rel, "max_abs": mx, "ref_max": b.abs().max().item()}), flush=True)
        return fin and rel < 3e-3

    ok = True
    if kernel == "analysis":
        X = torch.randn(M, 2 * B * Ci, plan.kp, device=dev)
        X[..., nlat:] = 0
        outs = []
        for prec in (0, 1):
            sp = torch.zeros(plan.spec_elems(B, Ci), device=dev)
            _lib.call("b200sht_legendre_analysis", plan.handle, _ptr(X), _ptr(sp), B, Ci, prec, st)
            torch.cuda.synchronize()
            outs.append(sp.view(L, M, 2 * B, -1))
        _, unstored = spec_rand(Ci)
        ok = report("spec", outs[1], outs[0], unstored)
    elif kernel == "synthesis":
        sp, _ = spec_rand(Ci)
        outs = []
        for prec in (0, 1):
            Z = torch.full((plan.latspec_elems(B, Ci),), float("nan"), device=dev)
            _lib.call("b200sht_legendre_synthesis", plan.handle, _ptr(sp), _ptr(Z), B, Ci, prec, st)
            torch.cuda.synchronize()
            outs.append(Z[: M * 2 * B * Ci * plan.kp].view(M, 2 * B * Ci, plan.kp))   # the buffer is padded to round_up(M, 8) orders
        ok = report("latspec", outs[1], outs[0])
    else:
        op = _lib.OP_DHCONV
        if not lib.b200sht_mix_uses_tensor_cores(op, B, G, Ci, Co, _lib.PREC_TF32):   # precision 1 would run the CUDA-core kernel as well
            print(json.dumps({"kernel": kernel, "case": case, "ok": False, "error": "this shape does not run the tcgen05 mix"}), flush=True)
            return 1
        wn = torch.randn(G, Ci // G, Co // G, L, dtype=torch.complex64, device=dev)
        wp = torch.empty(int(lib.b200sht_mix_weight_elems(op, L, M, G, Ci, Co)), device=dev)
        _lib.call("b200sht_mix_weight_pack", op, _ptr(wn), _ptr(wp), L, G, Ci, Co, 0, st)
        x, un = spec_rand(Ci)
        gy, _ = spec_rand(Co)
        outs = []
        for prec in (0, 1):
            if kernel == "mix_fwd":
                y = torch.zeros(L, M, 2 * B, (Co + 3) // 4 * 4, device=dev)
                _lib.call("b200sht_mix_forward", L, M, op, _ptr(x), _ptr(wp), mb.sht._VP(0), _ptr(y), B, G, Ci, Co, prec, st)
                outs.append(y)
            elif kernel == "mix_dgrad":
                gx = torch.zeros(L, M, 2 * B, (Ci + 3) // 4 * 4, device=dev)
                _lib.call("b200sht_mix_backward", L, M, op, mb.sht._VP(0), _ptr(wp), _ptr(gy), _ptr(gx), mb.sht._VP(0), mb.sht._VP(0), B, G, Ci, Co, prec, st)
                outs.append(gx)
            else:
                gw = torch.full_like(wp, float("nan"))
                _lib.call("b200sht_mix_backward", L, M, op, _ptr(x), _ptr(wp), _ptr(gy), mb.sht._VP(0), _ptr(gw), mb.sht._VP(0), B, G, Ci, Co, prec, st)
                outs.append(gw)
            torch.cuda.synchronize()
        ok = report(kernel, outs[1], outs[0], un if kernel != "mix_wgrad" else None)
    print(json.dumps({"kernel": kernel, "case": case, "ok": ok}), flush=True)
    return 0 if ok else 1


def main():
    if len(sys.argv) >= 2 and sys.argv[1] == "all":
        cases = sys.argv[2:] or list(CASES)
        bad = 0
        for case in cases:
            for k in KERNELS:
                try:
                    r = subprocess.run([sys.executable, os.path.abspath(__file__), k, case], capture_output=True, text=True, timeout=300)
                    out = (r.stdout + r.stderr).strip().splitlines()
                    tail = [ln for ln in out if ln.startswith("{")] or out[-6:]
                    print(f"--- {k}/{case}: rc={r.returncode}")
                    for ln in tail[-4:]:
                        print("   ", ln[:400])
                    if r.returncode != 0:
                        for ln in out[-8:]:
                            if not ln.startswith("{"):
                                print("    !", ln[:300])
                    bad += r.returncode != 0
                except subprocess.TimeoutExpired:
                    print(f"--- {k}/{case}: TIMEOUT")
                    bad += 1
        print("umma_diag: failures =", bad)
        return 1 if bad else 0
    return run_one(sys.argv[1], sys.argv[2])


if __name__ == "__main__":
    sys.exit(main())
