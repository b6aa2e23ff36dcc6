"""Checks at the boundary with the reference (makani), run from golden data under tests/golden/ that tests/golden/make_reference_suite_golden.py
produces from a makani checkout (through tests/reference_suites/*.py), so that no makani sources are needed here:

* the reference's loss / grid / noise suites, run against the oracle posing as `torch_harmonics`: a regression pin of the calls they made
  into the stand-ins (per distinct call at most MAX_CALLS_PER_KEY recorded, leading slice only), replayed on the same stand-ins;
* the reference's SphericalFourierNeuralOperatorNet: its stored parameter surface and state-dict keys against makani_b200.sfno's network;
* one case of the reference's distributed SpectralConv test: makani_b200.distributed on 2 gloo ranks against the serial reference.

Not checked without a makani checkout: makani's own network class built on makani_b200 through makani_b200.compat (the torch_harmonics shim)."""
import json
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
sys.path.insert(0, os.path.join(HERE, "reference_suites"))


def test_reference_sht_suite_calls_replay_on_the_oracle():
    """The 193 tests of the reference's loss / grid / noise suites passed with the oracle's RealSHT / InverseRealSHT and
    makani_b200.quadrature posed as torch_harmonics (reference_suites/report.txt).  This pins what those stand-ins returned there: the
    calls recorded by run_reference_tests.py --record (every distinct transform configuration and quadrature call the suites made: 3
    transforms on the 32 x 64 equiangular grid, 2 quadrature rules; per transform at most MAX_CALLS_PER_KEY calls, the leading
    (nlat, nlon) / (lmax, mmax) slice of each) must give the recorded outputs again.  It is not a comparison with the reference's code."""
    from oracle import makani_oracle as O
    import makani_b200.quadrature as mbq

    g = np.load(os.path.join(GOLDEN, "reference_sht_boundary.npz"))
    meta = json.loads(str(g["meta"]))
    assert len(meta["transforms"]) >= 3 and len(meta["quadrature"]) >= 2, meta
    for i, (key, n) in enumerate(meta["transforms"]):
        kind, nlat, nlon, lmax, mmax, grid, csphase, table_dtype, x_dtype = json.loads(key)
        cls = O.RealSHT if kind == "RealSHT" else O.InverseRealSHT
        t = cls(nlat, nlon, lmax, mmax, grid, csphase=csphase, dtype=getattr(torch, table_dtype.split(".")[1]))
        assert n >= 1, key
        for j in range(n):
            x = torch.from_numpy(g[f"t{i}/{j}/x"])
            x = torch.view_as_complex(x) if x_dtype.startswith("torch.complex") else x
            y = t(x)
            y = torch.view_as_real(y) if y.is_complex() else y
            ref = torch.from_numpy(g[f"t{i}/{j}/y"])
            assert y.shape == ref.shape and y.dtype == ref.dtype, key
            tol = 1e-5 if ref.dtype == torch.float32 else 1e-12
            assert (y - ref).abs().max().item() <= tol * ref.abs().max().item(), key
    for i, (key, n) in enumerate(meta["quadrature"]):
        name, args, kwargs = json.loads(key)
        out = getattr(mbq, name)(*args, **dict(kwargs))
        out = out if isinstance(out, tuple) else (out,)
        assert len(out) == n, key
        for j, o in enumerate(out):
            np.testing.assert_allclose(o.numpy(), g[f"q{i}/{j}"], rtol=1e-13, atol=1e-15, err_msg=key)


def test_committed_report_is_green():
    rep = open(os.path.join(HERE, "reference_suites", "report.txt")).read()
    total = [ln for ln in rep.splitlines() if ln.startswith("TOTAL:")]
    assert total and total[0].rstrip().endswith(" 0 failing"), total


@pytest.mark.parametrize("variant", ["linear", "nonlinear"])
def test_sfno_network_has_the_reference_network_surface(variant):
    """SURVEY rows A8/A9: makani_b200.sfno's SphericalFourierNeuralOperatorNet (the restated class), constructed on its CUDA-backed transforms
    and spectral layers, exposes the same parameters (names, shapes, dtypes, model-parallel tags) and state-dict keys as the reference's
    network class on the reference semantics (oracle), stored in golden/reference_sfno_surface.json by reference_suites/build_reference_sfno.py."""
    from build_reference_sfno import CFG, CFG_NONLINEAR, describe
    from makani_b200.sfno import SphericalFourierNeuralOperatorNet

    with open(os.path.join(GOLDEN, "reference_sfno_surface.json")) as f:
        ref = json.load(f)[variant]
    cfg = CFG if variant == "linear" else CFG_NONLINEAR
    torch.manual_seed(333)
    net = SphericalFourierNeuralOperatorNet(**cfg, precision="fp32")
    mine = describe(net)
    assert mine["state_dict_keys"] == ref["state_dict_keys"]
    assert not any("weights" in k or "pct" in k for k in mine["state_dict_keys"])      # SHT tables are not checkpointed
    assert mine["params"].keys() == ref["params"].keys()
    for name in ref["params"]:
        assert mine["params"][name] == ref["params"][name], (name, ref["params"][name], mine["params"][name])
    classes = sorted({type(m).__module__ + "." + type(m).__name__ for m in net.modules()
                      if type(m).__name__ in ("SpectralConv", "SpectralAttention", "RealSHT", "InverseRealSHT")})
    assert all(c.startswith("makani_b200.") for c in classes), classes
    assert any(c.endswith("SpectralConv" if variant == "linear" else "SpectralAttention") for c in classes)
    if variant == "linear":      # the reference's SpectralAttention.forward raises (SURVEY F3): construction only for "nonlinear"
        from oracle.sfno_backend import OracleBackend

        y = SphericalFourierNeuralOperatorNet(**cfg, backend=OracleBackend())(torch.randn(1, cfg["inp_chans"], *cfg["inp_shape"]))
        assert list(y.shape) == ref["forward_shape"] == [1, 3, 33, 64]


def _dist_conv_worker(rank, world, port, q):
    """rank of an h = world, w = 1 grid: the dhconv SpectralConv of the golden case on makani_b200.distributed's transforms"""
    import torch.distributed as dist

    import makani_b200.distributed as mbd
    from test_distributed_cpu import OracleLocalOps

    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("gloo", rank=rank, world_size=world)
        mbd.init(dist.new_group(list(range(world))), None)
        mbd.set_local_ops(OracleLocalOps)
        g = np.load(os.path.join(GOLDEN, "reference_dist_conv_inputs.npz"))
        c = json.loads(str(g["case"]))
        fwd = mbd.DistributedRealSHT(nlat=c["nlat_in"], nlon=c["nlon_in"])
        inv = mbd.DistributedInverseRealSHT(nlat=c["nlat_out"], nlon=c["nlon_out"], lmax=fwd.lmax, mmax=fwd.mmax)
        lat = lambda t, shapes: torch.split(t, shapes, dim=-2)[rank].contiguous()
        x = lat(torch.from_numpy(g["x"]).double(), fwd.lat_shapes).requires_grad_(True)
        w = torch.view_as_complex(torch.from_numpy(g["weight"])).to(torch.complex128)
        w = torch.split(w, fwd.l_shapes, dim=-1)[rank].contiguous().requires_grad_(True)     # the weight is sharded along l over h
        b = torch.from_numpy(g["bias"]).double().requires_grad_(True)
        y = inv(torch.einsum("bixy,iox->boxy", fwd(x), w[0]), dtype=torch.float64) + b
        y.backward(lat(torch.from_numpy(g["gy"]).double(), inv.lat_shapes))
        dist.all_reduce(b.grad)      # the bias is shared by every rank (the reference's gradient-reduction hooks sum it)
        # plain numpy arrays: a torch tensor on this queue is handed over through a handshake with the sending process, which may have exited
        res = {"y": y.detach(), "dx": x.grad, "dweight": torch.view_as_real(w.grad), "dbias": b.grad}
        q.put((rank, {k: v.detach().numpy().copy() for k, v in res.items()}, None))
        dist.destroy_process_group()
    except Exception:  # pragma: no cover
        import traceback

        q.put((rank, None, traceback.format_exc()))


def test_reference_distributed_spectral_conv_case_on_gloo():
    """One (odd-size, uneven 46/45 split) case of the reference's own distributed SpectralConv test on 2 gloo ranks: output, input, weight and
    bias gradients of makani_b200.distributed's transforms, gathered, against the serial reference SpectralConv stored by
    make_reference_suite_golden.py; the reference test's criterion (allclose, atol = rtol = its tol)."""
    import torch.multiprocessing as mp
    from test_distributed_cpu import _free_port

    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dist_conv_worker, args=(r, world, port, q)) for r in range(world)]
    try:
        for p in procs:
            p.start()
        out = sorted((q.get(timeout=600) for _ in range(world)), key=lambda r: r[0])
        for p in procs:
            p.join(timeout=60)
    finally:
        for p in procs:     # a rank that failed or hangs must not outlive the test
            if p.is_alive():
                p.kill()
                p.join()
    for rank, _, err in out:
        assert err is None, f"rank {rank}:\n{err}"
    ref = np.load(os.path.join(GOLDEN, "reference_dist_conv_outputs.npz"))
    tol = json.loads(str(np.load(os.path.join(GOLDEN, "reference_dist_conv_inputs.npz"))["case"]))["tol"]
    got = {k: torch.cat([torch.from_numpy(r[k]) for _, r, _ in out], dim=-2) for k in ("y", "dx", "dweight")}
    for name, t in got.items():
        want = torch.from_numpy(ref[name]).double()
        assert t.shape == want.shape and torch.allclose(t, want, atol=tol, rtol=tol), (name, (t - want).abs().max().item())
    for rank, r, _ in out:
        assert np.allclose(r["dbias"], ref["dbias"], atol=tol, rtol=tol), (rank, r["dbias"].flatten())
