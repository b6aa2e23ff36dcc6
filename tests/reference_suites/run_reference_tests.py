#!/usr/bin/env python
"""Run the REFERENCE's own test classes that exercise torch-harmonics' RealSHT / InverseRealSHT / quadrature against the oracle.

torch-harmonics is not installable in this environment, and `import makani` needs physicsnemo / h5py / zarr / ruamel.  This script
poses `oracle/makani_oracle.py` as the `torch_harmonics` package (RealSHT, InverseRealSHT), the product module `makani_b200.quadrature`
as `torch_harmonics.quadrature` (REFTESTS_ORACLE_QUADRATURE=1: the oracle's), `makani_b200.distributed` as `torch_harmonics.distributed`
(primitives, split helpers), stubs the packages the reference imports but these tests never call
(h5py, zarr, properscoring, parameterized, makani.utils.comm / YParams, the heavy `makani/__init__` files) and then imports the test
modules from /root/reference/tests unmodified and runs the listed unittest classes.  Nothing is copied: the reference's loss / grid /
noise code and its test expectations (Parseval, H1 = l(l+1) L2, quadrature sums to 4 pi, GRF variance, spectral CRPS identities ...)
execute from where they lie.  These are the known-answer tests the reference holds at the SHT boundary (SURVEY section 4, 8c).

    python tests/reference_suites/run_reference_tests.py            # prints one line per class, exit code 1 on any failure
    python tests/reference_suites/run_reference_tests.py --report   # also rewrites tests/reference_suites/report.txt

    python tests/reference_suites/run_reference_tests.py --record tests/golden/reference_sht_boundary.npz
                                                                    # also stores the calls the suites make into the stand-ins

The reference tree is taken from $MAKANI_REFERENCE (a checkout of makani).  The recorded calls are replayed without it by
tests/test_reference_suites.py.
"""
import importlib
import inspect
import os
import sys
import types
import unittest

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF = os.environ.get("MAKANI_REFERENCE", "")

# reference test classes that go through torch_harmonics.{RealSHT, InverseRealSHT, quadrature}
SUITES = {
    "tests.test_losses": ["TestSpectralLpLoss", "TestSpectralH1Loss", "TestSpectralAMSELoss", "TestSpectralCRPSLoss", "TestSpectralCoherenceLoss",
                          "TestSpectralL2EnergyScoreLoss", "TestCorrectedSpectralL2EnergyScoreLoss", "TestSobolevEnergyScoreLoss",
                          "TestSpectralLossWeighted", "TestSpectralRegularization", "TestSpectralRelativeLoss", "TestGeometricLpLoss"],
    "tests.test_grids": ["TestGridQuadrature", "TestGridToQuadratureRule", "TestGridConverter"],
    "tests.test_noise": ["TestIsotropicGRF", "TestDiffusionNoiseS2"],
}


def install_environment():
    sys.path.insert(0, ROOT)
    from oracle import makani_oracle as O
    import makani_b200.distributed as thd
    import makani_b200.distributed.primitives as thdp

    def as_torch(f):
        def g(*a, **k):
            r = f(*a, **k)
            if isinstance(r, tuple):
                return tuple(torch.from_numpy(x) if hasattr(x, "dtype") and not isinstance(x, torch.Tensor) else x for x in r)
            return r
        return g

    th = types.ModuleType("torch_harmonics")
    th.RealSHT, th.InverseRealSHT = O.RealSHT, O.InverseRealSHT
    quad = types.ModuleType("torch_harmonics.quadrature")
    quad.legendre_gauss_weights = as_torch(O.legendre_gauss_weights)
    quad.clenshaw_curtiss_weights = as_torch(O.clenshaw_curtiss_weights)
    quad.precompute_latitudes = as_torch(O.precompute_latitudes)
    if os.environ.get("REFTESTS_ORACLE_QUADRATURE"):
        th.quadrature = quad                      # the oracle's quadrature functions
    else:
        import makani_b200.quadrature as mbq      # PRODUCT code (pure torch / numpy, runs without a GPU): what the shim installs

        th.quadrature = quad = mbq
    th.distributed = thd
    sys.modules.update({"torch_harmonics": th, "torch_harmonics.quadrature": quad, "torch_harmonics.distributed": thd,
                        "torch_harmonics.distributed.primitives": thdp})

    # namespace packages: the reference's sub-modules are importable, its heavy package __init__ files are not executed
    def ns(name, path):
        m = types.ModuleType(name)
        m.__path__ = [path]
        sys.modules[name] = m
        return m

    mk = ns("makani", f"{REF}/makani")
    mu = ns("makani.utils", f"{REF}/makani/utils")
    mk.utils, mk.models, mk.mpu = mu, ns("makani.models", f"{REF}/makani/models"), ns("makani.mpu", f"{REF}/makani/mpu")
    ns("tests", f"{REF}/tests")
    comm = types.ModuleType("makani.utils.comm")   # single-process answers
    comm.get_rank = lambda n=None: 0
    comm.get_size = lambda n=None: 1
    comm.get_world_rank = lambda: 0
    comm.get_world_size = lambda: 1
    comm.is_distributed = lambda n=None: False
    comm.get_group = lambda n=None: None
    comm.get_names = lambda *a, **k: []
    mu.comm, mu.LossHandler = comm, object
    sys.modules["makani.utils.comm"] = comm
    yp = types.ModuleType("makani.utils.YParams")

    class ParamsBase:
        def __init__(self):
            self.params = {}

        def __getitem__(self, k):
            return self.params[k]

        def __setitem__(self, k, v):
            self.params[k] = v
            setattr(self, k, v)

        def __contains__(self, k):
            return k in self.params

        def get(self, k, d=None):
            return self.params.get(k, d)

    yp.ParamsBase = ParamsBase
    sys.modules["makani.utils.YParams"] = yp
    for name in ("h5py", "zarr"):
        sys.modules.setdefault(name, types.ModuleType(name))
    ps = types.ModuleType("properscoring")
    ps.crps_ensemble = ps.crps_gaussian = lambda *a, **k: None
    sys.modules.setdefault("properscoring", ps)

    # minimal `parameterized` (absent here): expand() generates one method per case, parameterized_class keeps the first (CPU) set
    par = types.ModuleType("parameterized")

    class parameterized:
        @staticmethod
        def expand(cases, **kw):
            cases = list(cases)

            def deco(f):
                loc = inspect.currentframe().f_back.f_locals
                for i, c in enumerate(cases):
                    args = tuple(c) if isinstance(c, (list, tuple)) else (c,)
                    loc[f"{f.__name__}_{i}"] = (lambda a: (lambda self: f(self, *a)))(args)
                loc[f"_orig_{f.__name__}"] = f      # the undecorated method, for debugging a single case by hand
                return None
            return deco

    def parameterized_class(names, values):
        names = (names,) if isinstance(names, str) else tuple(names)

        def deco(cls):
            for k, v in zip(names, values[0]):
                setattr(cls, k, v)
            return cls
        return deco

    par.parameterized, par.parameterized_class = parameterized, parameterized_class
    sys.modules.setdefault("parameterized", par)


MAX_CALLS_PER_KEY = 2          # recorded calls per distinct transform / quadrature call
MAX_SLICE_ELEMS = 1 << 14      # larger transform slices are not recorded (file size)
QUADRATURE_FNS = ("legendre_gauss_weights", "clenshaw_curtiss_weights", "precompute_latitudes", "precompute_longitudes")


def install_recorder(transforms, quadrature):
    """Wrap the stand-ins installed as torch_harmonics: per distinct transform (constructor arguments, table and input dtype) the first
    MAX_CALLS_PER_KEY inputs and outputs are kept, reduced to the leading [0, ..., 0] slice (the transforms act on the last two
    dimensions only); per distinct quadrature call its outputs."""
    import json

    from oracle import makani_oracle as O

    th = sys.modules["torch_harmonics"]

    def wrap(base, kind, table):
        class Recording(base):
            def forward(self, x):
                y = super().forward(x)
                key = json.dumps([kind, self.nlat, self.nlon, self.lmax, self.mmax, self.grid, self.csphase,
                                  str(getattr(self, table).dtype), str(x.dtype)])
                xs, ys = x.detach().reshape(-1, *x.shape[-2:])[0], y.detach().reshape(-1, *y.shape[-2:])[0]
                calls = transforms.setdefault(key, [])
                if len(calls) < MAX_CALLS_PER_KEY and xs.numel() <= MAX_SLICE_ELEMS and ys.numel() <= MAX_SLICE_ELEMS:
                    calls.append((xs.clone(), ys.clone()))
                return y

        Recording.__name__ = base.__name__
        return Recording

    th.RealSHT = wrap(O.RealSHT, "RealSHT", "weights")
    th.InverseRealSHT = wrap(O.InverseRealSHT, "InverseRealSHT", "pct")
    quad = types.ModuleType("torch_harmonics.quadrature")
    quad.__dict__.update({k: v for k, v in vars(th.quadrature).items() if not k.startswith("__")})

    def wrap_fn(name, fn):
        def g(*a, **k):
            r = fn(*a, **k)
            key = json.dumps([name, list(a), sorted(k.items())])
            if key not in quadrature:
                quadrature[key] = [t.clone() for t in (r if isinstance(r, tuple) else (r,))]
            return r
        return g

    for name in QUADRATURE_FNS:
        if hasattr(quad, name):
            setattr(quad, name, wrap_fn(name, getattr(quad, name)))
    th.quadrature = quad
    sys.modules["torch_harmonics.quadrature"] = quad


def save_recording(path, transforms, quadrature):
    """npz: `meta` (JSON: one [key, n_calls] per transform, one [key, n_outputs] per quadrature call) and the arrays
    t{i}/{j}/x, t{i}/{j}/y, q{i}/{j}; complex arrays are stored as (..., 2) real views."""
    import json

    import numpy as np

    def arr(t):
        return (torch.view_as_real(t) if t.is_complex() else t).numpy()

    data, meta = {}, {"transforms": [], "quadrature": []}
    for i, (key, calls) in enumerate(sorted(transforms.items())):
        meta["transforms"].append([key, len(calls)])
        for j, (x, y) in enumerate(calls):
            data[f"t{i}/{j}/x"], data[f"t{i}/{j}/y"] = arr(x), arr(y)
    for i, (key, outs) in enumerate(sorted(quadrature.items())):
        meta["quadrature"].append([key, len(outs)])
        for j, t in enumerate(outs):
            data[f"q{i}/{j}"] = arr(t)
    data["meta"] = np.array(json.dumps(meta))
    np.savez_compressed(path, **data)


def run(record=None):
    """-> list of (module, class, ran, failures, errors, [messages]); record: (transforms, quadrature) dicts filled by install_recorder"""
    install_environment()
    if record is not None:
        install_recorder(*record)
    results = []
    for modname, classes in SUITES.items():
        M = importlib.import_module(modname)
        for name in classes:
            suite = unittest.defaultTestLoader.loadTestsFromTestCase(getattr(M, name))
            r = unittest.TextTestRunner(verbosity=0, stream=open(os.devnull, "w")).run(suite)
            msgs = [t.id().split(".")[-1] + ": " + tb.strip().splitlines()[-1][:160] for t, tb in r.failures + r.errors]
            results.append((modname, name, r.testsRun, len(r.failures), len(r.errors), msgs))
    return results


def main():
    if not os.path.isdir(REF):
        print("reference tree not found (set MAKANI_REFERENCE): nothing to run")
        return 0
    record = ({}, {}) if "--record" in sys.argv else None
    results = run(record)
    if record is not None:
        save_recording(sys.argv[sys.argv.index("--record") + 1], *record)
    lines = []
    for modname, name, ran, nf, ne, msgs in results:
        lines.append(f"{modname}.{name}: ran {ran}  failures {nf}  errors {ne}")
        lines += ["    " + m for m in msgs]
    total = sum(r[2] for r in results)
    bad = sum(r[3] + r[4] for r in results)
    lines.append(f"TOTAL: {total} reference tests against the oracle as torch_harmonics, {bad} failing")
    print("\n".join(lines))
    if "--report" in sys.argv:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "report.txt"), "w") as f:
            f.write("python tests/reference_suites/run_reference_tests.py --report   (reference tree at $MAKANI_REFERENCE)\n" + "\n".join(lines) + "\n")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
