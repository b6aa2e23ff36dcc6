#!/usr/bin/env python
"""bench.py -- one SFNO SpectralConv block, forward + backward, on synthetic ERA5-shaped input.

Contract: `python bench.py --gpus N --steps K --warmup W` (N > 1 under torchrun) prints ONE JSON line on rank 0.
  metric    SFNO-block fwd+bwd samples/sec (BASELINE.json), workload = configs[1]: 721x1440x73ch, bf16, batch 1 per GPU
  value     device-resident input, CUDA-event timed, max over ranks
  e2e       same step through the public nn.Module with the input in pinned HOST memory (H2D of x and D2H of the weight
            gradient inside the timed region)
  roofline  dominant kernel (largest share of the step), algorithmic bytes / CUDA-event time vs MEASURED_PEAKS.json
  cpu_baseline  the CPU oracle (restatement of torch-harmonics + makani einsums) on this box's host cores (bounded sample)
`--dump-outputs DIR` writes the outputs of the last timed step (the inputs are seeded: two builds can be compared output for output).
`--impl reference` times that CPU implementation alone (the reference has no other implementation of this path that can run
here: torch-harmonics is not installable, see DESIGN.md).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (nlat_in, nlon_in, grid_in, nlat_out, nlon_out, grid_out, lmax, mmax, C)
    "sfno_block_721x1440x73": (721, 1440, "equiangular", 721, 1440, "equiangular", 240, 241, 73),       # BASELINE configs[1] (SURVEY cfg 2c)
    "sfno_block_240x480x384": (240, 480, "legendre-gauss", 240, 480, "legendre-gauss", 240, 241, 384),  # interior SFNO block (cfg 2a)
    "sfno_block_721to240x384": (721, 1440, "equiangular", 240, 480, "legendre-gauss", 240, 241, 384),  # first SFNO block (cfg 2b)
    "tiny": (33, 64, "equiangular", 33, 64, "equiangular", 16, 17, 8),
}


def nnz_modes(L, M):
    return sum(max(0, L - m) for m in range(M))


def stage_bytes(wl, act_bytes):
    """Algorithmic HBM bytes per launch of each stage (DESIGN.md section 5), B = 1."""
    nlat_i, nlon_i, _, nlat_o, nlon_o, _, L, M, C = WORKLOADS[wl]
    nnz = nnz_modes(L, M)
    spec = C * nnz * 8  # complex fp32 coefficients, l >= m only
    w = C * C * L * 8
    return {
        "fft_analysis_in": C * nlat_i * nlon_i * act_bytes + C * nlat_i * M * 8,
        "legendre_analysis_in": C * nlat_i * M * 8 + nnz * nlat_i * 4 + spec,
        "mix_forward": 2 * spec + w,
        "legendre_synthesis_out": spec + nnz * nlat_o * 4 + C * nlat_o * M * 8,
        "fft_synthesis_out": C * nlat_o * M * 8 + C * nlat_o * nlon_o * act_bytes,
        "fft_analysis_out": C * nlat_o * nlon_o * act_bytes + C * nlat_o * M * 8,
        "legendre_analysis_out": C * nlat_o * M * 8 + nnz * nlat_o * 4 + spec,
        "mix_backward": 3 * spec + 2 * w,
        "legendre_synthesis_in": spec + nnz * nlat_i * 4 + C * nlat_i * M * 8,
        "fft_synthesis_in": C * nlat_i * M * 8 + C * nlat_i * nlon_i * act_bytes,
    }


def stage_flops(wl):
    """Algorithmic flops per launch of the contraction stages (SURVEY section 8d: structurally non-zero l >= m pairs only), B = 1."""
    nlat_i, _, _, nlat_o, _, _, L, M, C = WORKLOADS[wl]
    nnz = nnz_modes(L, M)
    mix = 8 * C * C * nnz
    return {"legendre_analysis_in": 4 * C * nlat_i * nnz, "legendre_synthesis_out": 4 * C * nlat_o * nnz, "legendre_analysis_out": 4 * C * nlat_o * nnz,
            "legendre_synthesis_in": 4 * C * nlat_i * nnz, "mix_forward": mix, "mix_backward": 2 * mix}


def add_stage_tflops(stages, wl):
    """annotate the per-stage records of the contraction kernels with their algorithmic TFLOP/s (metric (ii) of SURVEY section 8d)"""
    fl = stage_flops(wl)
    for name, rec in stages.items():
        if name in fl and rec.get("ms"):
            rec["alg_GFLOP"] = round(fl[name] / 1e9, 3)
            rec["TFLOPs"] = round(fl[name] / (rec["ms"] * 1e-3) / 1e12, 2)
    return stages


def flops_fwd_bwd(wl):
    nlat_i, _, _, nlat_o, _, _, L, M, C = WORKLOADS[wl]
    nnz = nnz_modes(L, M)
    leg = lambda nlat: 4 * C * nlat * nnz
    return 2 * (leg(nlat_i) + leg(nlat_o)) + 3 * 8 * C * C * nnz


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------- CPU arm
def build_oracle_block(wl, dtype=torch.float32):
    from oracle import makani_oracle as O

    nlat_i, nlon_i, grid_i, nlat_o, nlon_o, grid_o, L, M, C = WORKLOADS[wl]
    sht = O.RealSHT(nlat_i, nlon_i, L, M, grid_i, dtype=dtype)
    isht = O.InverseRealSHT(nlat_o, nlon_o, L, M, grid_o, dtype=dtype)
    return O, sht, isht


def pick_cpu_threads():
    """Host threads for the CPU arm: the cores this process may use, calibrated -- torch's bmm/fft scale poorly past a point
    and a container may expose more logical CPUs than its quota, so time a small forward at a few thread counts and keep the best."""
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    from oracle import makani_oracle as O

    sht = O.RealSHT(240, 480, 120, 121, "legendre-gauss")
    x = torch.randn(1, 16, 240, 480)
    best, best_t = 1, float("inf")
    cands = sorted({n for n in (4, 8, 16, 32, 64, avail) if n <= avail} | {min(avail, 8)})
    for n in cands:
        torch.set_num_threads(n)
        sht(x)
        t0 = time.perf_counter()
        for _ in range(3):
            sht(x)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best, avail


def cpu_reference_steps(wl, steps, warmup, act_dtype=torch.bfloat16):
    """fwd+bwd of the block through the CPU oracle (restated torch-harmonics + makani SpectralConv)."""
    O, sht, isht = build_oracle_block(wl)
    nlat_i, nlon_i, _, nlat_o, nlon_o, _, L, M, C = WORKLOADS[wl]
    torch.manual_seed(333)
    w = (math.sqrt(1.0 / C) * torch.randn(1, C, C, L, dtype=torch.complex64)).requires_grad_(True)
    x = torch.randn(1, C, nlat_i, nlon_i).to(act_dtype).requires_grad_(True)
    gy = torch.randn(1, C, nlat_o, nlon_o).to(act_dtype)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        y, _ = O.spectral_conv_forward(x, w, sht, isht, operator_type="dhconv")
        y.backward(gy)
        x.grad = None
        w.grad = None
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return sum(times) / len(times)


def gpu_library_baseline(wl, act_dtype, dev, flush, steps=5):
    """fwd+bwd of the block through torch.fft + torch.einsum ON THE GPU (what torch-harmonics + makani dispatch to: cuFFT, cuBLAS)."""
    O, sht, isht = build_oracle_block(wl)
    sht, isht = sht.to(dev), isht.to(dev)
    nlat_i, nlon_i, _, nlat_o, nlon_o, _, L, M, C = WORKLOADS[wl]
    torch.manual_seed(333)
    w = (math.sqrt(1.0 / C) * torch.randn(1, C, C, L, dtype=torch.complex64, device=dev)).requires_grad_(True)
    x = torch.randn(1, C, nlat_i, nlon_i, device=dev).to(act_dtype).requires_grad_(True)
    gy = torch.randn(1, C, nlat_o, nlon_o, device=dev).to(act_dtype)
    prev = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    try:
        def step():
            x.grad = None
            w.grad = None
            y, _ = O.spectral_conv_forward(x, w, sht, isht, operator_type="dhconv")
            y.backward(gy)
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        ms = 0.0
        for _ in range(steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step()
            e1.record()
            torch.cuda.synchronize()
            ms += e0.elapsed_time(e1)
        ms /= steps
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev
    return {"value": 1e3 / ms, "unit": "samples/s", "ms_per_step": ms,
            "what": "same block through torch.fft + torch.einsum on this GPU (cuFFT + cuBLAS, allow_tf32=True, dense einsums incl. l<m zeros)"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload in MODEL_WORKLOADS:
        return run_reference_model_arm(args)
    wl = args.workload
    cores, avail = pick_cpu_threads()
    steps = args.steps   # each step is a full fwd+bwd of the workload (~10 s of CPU work at the default workload)
    t = cpu_reference_steps(wl, steps, args.warmup)
    val = 1.0 / t
    line = {
        "impl": "reference", "metric": "SFNO-block fwd+bwd samples/sec", "value": val, "unit": "samples/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": wl, "batch_per_gpu": 1, "activations": "bf16", "parallelism": "cpu"},
        "cpu_baseline": {"value": val, "unit": "samples/s", "cores": cores, "kind": "port",
                         "sample": f"{steps} full fwd+bwd steps of the workload through oracle/makani_oracle.py (torch.fft + torch.einsum, fp32, {cores} threads chosen by calibration of {avail} available)"},
        "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def run_reference_model_arm(args):
    """CPU arm of the full-model workloads: the same network (makani_b200.sfno, pinned against the reference's network class by
    tests/golden/sfno_golden_<case>.npz) on the oracle transforms / SpectralConv, bf16 autocast off (CPU), --warmup + --steps steps."""
    from makani_b200.sfno import SphericalFourierNeuralOperatorNet
    from oracle.sfno_backend import OracleBackend

    cfg = MODEL_WORKLOADS[args.workload]
    cores, avail = pick_cpu_threads()
    torch.manual_seed(333)
    net = SphericalFourierNeuralOperatorNet(**cfg, backend=OracleBackend())
    x = torch.randn(1, cfg["inp_chans"], *cfg["inp_shape"])
    times = []
    for it in range(args.warmup + args.steps):
        net.zero_grad(set_to_none=True)
        t0 = time.perf_counter()
        out = net(x)
        out.float().square().mean().backward()
        if it >= args.warmup:
            times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    val = 1.0 / t
    print(json.dumps({
        "impl": "reference", "metric": "SFNO model fwd+bwd samples/sec", "value": val, "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "batch_per_gpu": 1, "parallelism": "cpu"},
        "cpu_baseline": {"value": val, "unit": "samples/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} full fwd+bwd steps of the network on oracle/ (torch.fft + torch.einsum, fp32, {cores} threads of {avail})"},
        "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


DUMP_SAMPLE = 1 << 22    # --dump-outputs: elements kept of a larger output (a fixed, seeded sample)
DUMP_GRAD_SAMPLE = 4096  # --dump-outputs, model workloads: elements kept of each parameter gradient


def sample_flat(t, k, seed=0):
    """t flattened to float32 on the host; when it has more than k elements, the same k of them on every run (seeded, sorted indices)"""
    t = torch.view_as_real(t) if t.is_complex() else t
    flat = t.detach().reshape(-1)
    if flat.numel() <= k:
        return t.detach().float().cpu()
    idx = torch.randint(0, flat.numel(), (k,), generator=torch.Generator().manual_seed(seed)).sort().values
    return flat[idx.to(flat.device)].float().cpu()


def dump_outputs(out_dir, arrays):
    """arrays: name -> tensor, each written as out_dir/<name>.npy (float32)"""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.numpy().astype(np.float32, copy=False))


HXW_GRID = {2: (1, 2), 4: (2, 2), 8: (4, 2)}   # h x w spatial model-parallel grids (cfg 4 of BASELINE.json is h = 4, w = 2)


def hxw_measure(wl, world, rank, dev, act_dtype, precision, steps, warmup):
    """The SAME block with ONE sample split over all ranks (h x w spatial model parallelism, makani_b200.distributed: latitude over h, longitude
    over w, l over h, m over w; 4 all-to-all transposes per distributed transform, makani/mpu/mappings.py:38-67).  Strong scaling: global batch 1.
    Returns a dict for the JSON line (never raises: an h x w failure must not lose the data-parallel line)."""
    import torch.distributed as dist

    try:
        import makani_b200 as mb
        import makani_b200.distributed as mbd

        h, w = HXW_GRID[world]
        nlat_i, nlon_i, grid_i, nlat_o, nlon_o, grid_o, L, M, C = WORKLOADS[wl]
        h_groups = [dist.new_group([ih * w + iw for ih in range(h)]) for iw in range(w)]
        w_groups = [dist.new_group([ih * w + iw for iw in range(w)]) for ih in range(h)]
        ih, iw = rank // w, rank % w
        mbd.init(h_groups[iw] if h > 1 else None, w_groups[ih] if w > 1 else None)
        fd = mbd.DistributedRealSHT(nlat_i, nlon_i, L, M, grid_i, precision=precision)
        idd = mbd.DistributedInverseRealSHT(nlat_o, nlon_o, L, M, grid_o, precision=precision)
        torch.manual_seed(333)
        conv = mb.SpectralConv(fd, idd, C, C, operator_type="dhconv", precision=precision).to(dev)
        conv._wcache.enabled = False
        x = torch.randn(1, C, fd.lat_shapes[ih], fd.lon_shapes[iw], device=dev).to(act_dtype)
        gy = torch.randn(1, C, idd.lat_shapes[ih], idd.lon_shapes[iw], device=dev).to(act_dtype)
        wg = w_groups[ih] if w > 1 else None

        def step():
            x.requires_grad_(True)
            conv.weight.grad = None
            y, _ = conv(x)
            y.backward(gy)
            x.grad = None
            x.requires_grad_(False)
            if wg is not None:   # the dhconv weight shard is shared over w (spectral_convolution.py:195-198)
                dist.all_reduce(torch.view_as_real(conv.weight.grad), group=wg)

        for _ in range(max(3, warmup)):
            step()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        dist.barrier()
        t = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
        mbd.finalize() if hasattr(mbd, "finalize") else None
        return {"h": h, "w": w, "ms_per_step": ms, "value": 1e3 / ms, "unit": "samples/s", "scaling": "strong", "global_batch": 1,
                "local_input": [1, C, fd.lat_shapes[ih], fd.lon_shapes[iw]], "lat_shapes": list(fd.lat_shapes), "m_shapes": list(fd.m_shapes),
                "what": "one sample of the same block split over all ranks (latitude over h, longitude over w); NCCL all-to-all transposes + "
                        "weight-gradient all-reduce over w inside the timed step; max over ranks"}
    except Exception as e:  # noqa: BLE001
        return {"error": f"{type(e).__name__}: {str(e)[:300]}"}


# ----------------------------------------------------------------------------------------------------- GPU arm
def run_gpu_arm(args):
    import torch.distributed as dist

    import makani_b200 as mb
    from makani_b200 import _lib
    from makani_b200.sht import _ptr, _stream, _dtype_code

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dp_group = None
    dp_mode = args.dp_mode
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        if dp_mode == "overlap":
            # the gradient all-reduce runs beside persistent kernels that leave it B200SHT_OVERLAP_SMS (8) SMs: a communicator of its own, capped at as
            # many CTAs.  (Measured slower than the trailing all-reduce on the default communicator, DESIGN.md section 7: not the default.)
            try:
                opts = dist.ProcessGroupNCCL.Options()
                opts.config.max_ctas = int(os.environ.get("B200SHT_DP_MAXCTAS", os.environ.get("B200SHT_OVERLAP_SMS", "8"))) or 8
                opts.config.min_ctas = 1
                dp_group = dist.new_group(list(range(world)), pg_options=opts)
            except Exception as e:   # older torch / NCCL: default communicator
                sys.stderr.write(f"bench: NCCL communicator with max_ctas unavailable ({e}); using the default one\n")
                dp_group = None
    wl = args.workload
    nlat_i, nlon_i, grid_i, nlat_o, nlon_o, grid_o, L, M, C = WORKLOADS[wl]
    act_dtype = torch.bfloat16 if args.act == "bf16" else torch.float32
    act_bytes = 2 if act_dtype == torch.bfloat16 else 4

    f = mb.RealSHT(nlat_i, nlon_i, L, M, grid_i)
    i = mb.InverseRealSHT(nlat_o, nlon_o, L, M, grid_o)
    plan_f, plan_i = f.plan(dev), i.plan(dev)
    precision = args.precision
    if precision == "best":
        precision = "tf32" if plan_f.umma_ok else "fp32"
    f.precision = i.precision = precision
    torch.manual_seed(333 + rank)
    conv = mb.SpectralConv(f, i, C, C, operator_type="dhconv", precision=precision).to(dev)
    conv._wcache.enabled = False  # weights change every optimizer step in training: re-layout inside the timed step
    x_host = torch.randn(1, C, nlat_i, nlon_i).to(act_dtype).pin_memory()
    x_dev = x_host.to(dev)
    gy = torch.randn(1, C, nlat_o, nlon_o, device=dev).to(act_dtype)
    gw_host = torch.empty(conv.weight.shape, dtype=torch.complex64).pin_memory()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step(xin, keep=None):
        xin.requires_grad_(True)
        conv.weight.grad = None
        y, _ = conv(xin)
        y.backward(gy)
        g = xin.grad
        xin.grad = None
        xin.requires_grad_(False)
        if keep is not None:   # --dump-outputs: what a caller of the step receives
            keep.update(y=y.detach(), dx=g)
        return g

    def step_e2e():
        xd = x_host.to(dev, non_blocking=True)
        step(xd)
        if world > 1:
            dist.all_reduce(torch.view_as_real(conv.weight.grad))
        gw_host.copy_(conv.weight.grad, non_blocking=True)

    feed = mb.HostFeed(x_host.shape, act_dtype, dev)

    def e2e_pipelined(steps):
        """K steps through HostFeed: the H2D copy of step i+1 and the read-back of step i-1 overlap the kernels of step i.
        Returns ms per step (device clock, first push .. last read-back)."""
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        feed.h2d.wait_event(e0)          # the first copy starts inside the timed region
        feed.push(x_host)
        for i in range(steps):
            xd = feed.pop()
            if i + 1 < steps:
                feed.push(x_host)
            step(xd)
            feed.release(xd)
            if world > 1:
                dist.all_reduce(torch.view_as_real(conv.weight.grad))
            feed.read_back(conv.weight.grad, gw_host)
        feed.drain()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1) / steps
        if world > 1:
            tt = torch.tensor([ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = tt.item()
        return ms

    graph_info = None

    def try_cuda_graph():
        """Capture one fwd+bwd step (weight re-layout included) into a CUDA graph and time its replay.  Returns a dict for the JSON
        line; any failure is reported there and never affects the eager numbers."""
        try:
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(3):
                    step(x_dev)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize()
            step(x_dev)
            ref_gw = conv.weight.grad.detach().clone()
            conv.weight.grad = None
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                static_gx = step(x_dev)
            g.replay()
            torch.cuda.synchronize()
            same = torch.allclose(torch.view_as_real(conv.weight.grad), torch.view_as_real(ref_gw), rtol=1e-5, atol=1e-6) and bool(torch.isfinite(static_gx.float()).all())
            if not same:
                return {"ok": False, "why": "replay does not reproduce the eager weight gradient"}
            ms = timed(g.replay, args.steps, args.warmup)
            return {"ok": True, "ms_per_step": ms, "value": 1e3 / ms}
        except Exception as e:  # noqa: BLE001
            return {"ok": False, "why": str(e)[:300]}

    host_enqueue = {}

    def timed(fn, steps, warmup, use_flush=True):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        evs = []
        t_host = time.perf_counter()
        for _ in range(steps):
            if use_flush:
                flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        host_enqueue["ms_per_step"] = (time.perf_counter() - t_host) * 1e3 / steps   # host time to ENQUEUE a step (no synchronisation inside the loop)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs) / steps
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    # data parallel: the weight-gradient all-reduce is launched on a side stream as soon as the gradient is final (event recorded inside
    # b200sht_spectral_conv_backward_ex, before the two input-gradient stages), so it overlaps legendre_synthesis + fft_synthesis
    side = torch.cuda.Stream(dev) if (world > 1 and dp_mode == "overlap") else None
    if world > 1 and dp_mode == "overlap":
        conv.wgrad_ready_event = torch.cuda.Event()

    last = {} if args.dump_outputs else None   # outputs of the latest timed step

    def dp_step():
        step(x_dev, last)
        if world > 1 and dp_mode != "overlap":   # the all-reduce trails the backward pass on the compute stream (default communicator)
            dist.all_reduce(torch.view_as_real(conv.weight.grad))
        elif world > 1:
            side.wait_event(conv.wgrad_ready_event)
            with torch.cuda.stream(side):
                dist.all_reduce(torch.view_as_real(conv.weight.grad), group=dp_group)
            conv.weight.grad.record_stream(side)
            torch.cuda.current_stream(dev).wait_stream(side)
        if last is not None:
            last["dweight"] = conv.weight.grad

    # kernel launches of OUR library inside one step (counted by the ctypes call wrapper)
    counter = {"n": 0}
    kernels_per_call = {"b200sht_fft_analysis": 1, "b200sht_fft_synthesis": 1, "b200sht_legendre_analysis": 1, "b200sht_legendre_synthesis": 1, "b200sht_legendre_synthesis_tiled": 1,
                        "b200sht_mix_forward": 1, "b200sht_mix_backward": 2, "b200sht_mix_weight_pack": 1, "b200sht_mix_weight_unpack": 1,
                        "b200sht_bias_grad": 1, "b200sht_spec_pack": 1, "b200sht_spec_unpack": 1,
                        # one-call entry points: fft + legendre + mix + legendre + fft / fft + legendre + dgrad + wgrad + legendre + fft
                        "b200sht_spectral_conv_forward": 5, "b200sht_spectral_conv_backward": 6,
                        "b200sht_spectral_conv_backward_ex": 7,   # + the weight-gradient re-layout, now inside the call
                        "b200sht_legendre_synthesis_tiled": 1}
    if precision == "fp32x3":   # + one operand-residual kernel per Legendre stage
        for k, extra in (("b200sht_legendre_analysis", 1), ("b200sht_legendre_synthesis", 1), ("b200sht_spectral_conv_forward", 2),
                         ("b200sht_spectral_conv_backward", 2), ("b200sht_spectral_conv_backward_ex", 2)):
            kernels_per_call[k] += extra
    orig_call = _lib.call

    def counting_call(name, *a):
        counter["n"] += kernels_per_call.get(name, 0)
        return orig_call(name, *a)

    sampler = ClockSampler(local) if rank == 0 else None
    ms_dev = None
    host_ms = None
    try:
        dp_step()  # first call builds plans / tables
        torch.cuda.synchronize()
        _lib.call = counting_call
        counter["n"] = 0
        dp_step()
        launches_per_step = counter["n"]
        _lib.call = orig_call
        if sampler:
            # nvidia-smi needs ~1 s to start sampling and the timed region may be shorter than its period: keep the GPU under
            # the same load (untimed extra steps) until the first sample arrives, then warm up + time as specified
            sampler.start()
            t_wait = time.perf_counter()
            while not sampler.lines and time.perf_counter() - t_wait < 5.0:
                step(x_dev)  # local load only: no collective here, the other ranks are waiting at the next barrier
                torch.cuda.synchronize()
        ms_dev = timed(dp_step, args.steps, args.warmup)
        host_ms = host_enqueue.get("ms_per_step")
        dumped = {k: sample_flat(v, DUMP_SAMPLE) for k, v in last.items()} if (last is not None and rank == 0) else None
        last = None
        # the same step replayed from a CUDA graph, reported separately (`value` stays the eager step: it is what N > 1 and e2e run)
        if args.graph and world == 1:
            graph_info = try_cuda_graph()
        if sampler:
            n_before = len(sampler.lines)
            t_wait = time.perf_counter()
            while len(sampler.lines) < n_before + 2 and time.perf_counter() - t_wait < 1.0:  # one more sample under the same load
                step(x_dev)
                torch.cuda.synchronize()
        clocks = sampler.stop() if sampler else None
        ms_e2e_serial = timed(step_e2e, args.steps, max(1, args.warmup // 2), use_flush=True)
        e2e_pipelined(max(2, args.warmup))      # warm-up of the pipelined loop (allocator, streams)
        ms_e2e = e2e_pipelined(args.steps)
    finally:
        _lib.call = orig_call

    hxw = None
    if world in HXW_GRID and not args.no_hxw:
        hxw = hxw_measure(wl, world, rank, dev, act_dtype, precision, max(3, min(args.steps, 10)), args.warmup)

    # ---- per-stage kernel timings (CUDA events, L2 flushed before each launch) -> roofline
    stages = {}
    if rank == 0 and not args.no_stages:
        st = _stream(dev)
        prec = mb.resolve_precision(precision)
        B = 1
        lat_i = torch.empty(plan_f.latspec_elems(B, C), device=dev)
        lat_o = torch.empty(plan_i.latspec_elems(B, C), device=dev)
        sp_a = torch.zeros(plan_f.spec_elems(B, C), device=dev)
        sp_b = torch.zeros(plan_f.spec_elems(B, C), device=dev)
        sp_c = torch.zeros(plan_f.spec_elems(B, C), device=dev)
        wpk = conv._wcache.get(conv.weight, _lib.OP_DHCONV, L, M, 1, C, C, prec)
        gwpk = torch.empty_like(wpk)
        y_dev = torch.empty(1, C, nlat_o, nlon_o, device=dev, dtype=act_dtype)
        gx_dev = torch.empty_like(x_dev)
        dt = _dtype_code(act_dtype)
        VP0 = mb.sht._VP(0)
        tfb = 2 if prec == _lib.PREC_TF32 else 0   # TF32 precision bit of the longitude-transform entry points (tensor-core DFT)

        def syn_bit(plan):   # tiled latspec + tensor-core DFT when the plan has it (what SpectralConv's one-call path does)
            return 2 if (tfb and plan.dft_ok) else 0

        def leg_syn(plan, sp, lat):
            if syn_bit(plan):
                return _lib.call("b200sht_legendre_synthesis_tiled", plan.handle, _ptr(sp), _ptr(lat), B, C, st)
            return _lib.call("b200sht_legendre_synthesis", plan.handle, _ptr(sp), _ptr(lat), B, C, prec, st)

        calls = {
            "fft_analysis_in": lambda: _lib.call("b200sht_fft_analysis", plan_f.handle, _ptr(x_dev), dt, B, C, _ptr(lat_i), 0 | tfb, st),
            "legendre_analysis_in": lambda: _lib.call("b200sht_legendre_analysis", plan_f.handle, _ptr(lat_i), _ptr(sp_a), B, C, prec, st),
            "mix_forward": lambda: _lib.call("b200sht_mix_forward", L, M, _lib.OP_DHCONV, _ptr(sp_a), _ptr(wpk), VP0, _ptr(sp_b), B, 1, C, C, prec, st),
            "legendre_synthesis_out": lambda: leg_syn(plan_i, sp_b, lat_o),
            "fft_synthesis_out": lambda: _lib.call("b200sht_fft_synthesis", plan_i.handle, _ptr(lat_o), _ptr(y_dev), dt, B, C, VP0, 0 | syn_bit(plan_i), st),
            "fft_analysis_out": lambda: _lib.call("b200sht_fft_analysis", plan_i.handle, _ptr(gy), dt, B, C, _ptr(lat_o), 1 | tfb, st),
            "legendre_analysis_out": lambda: _lib.call("b200sht_legendre_analysis", plan_i.handle, _ptr(lat_o), _ptr(sp_b), B, C, prec, st),
            "mix_backward": lambda: _lib.call("b200sht_mix_backward", L, M, _lib.OP_DHCONV, _ptr(sp_a), _ptr(wpk), _ptr(sp_b), _ptr(sp_c), _ptr(gwpk), VP0, B, 1, C, C, prec, st),
            "legendre_synthesis_in": lambda: leg_syn(plan_f, sp_c, lat_i),
            "fft_synthesis_in": lambda: _lib.call("b200sht_fft_synthesis", plan_f.handle, _ptr(lat_i), _ptr(gx_dev), dt, B, C, VP0, 1 | syn_bit(plan_f), st),
        }
        sb = stage_bytes(wl, act_bytes)
        for name, fn in calls.items():
            for _ in range(3):
                fn()
            ts = []
            for _ in range(max(3, min(args.steps, 10))):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            ms = sum(ts) / len(ts)
            stages[name] = {"ms": round(ms, 4), "alg_MB": round(sb[name] / 1e6, 2), "GBps": round(sb[name] / ms / 1e6, 1)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    try:
        add_stage_tflops(stages, wl)
    except Exception:  # never lose the line over an annotation
        pass
    peak, peak_src = measured_peaks()
    roof = None
    if stages:
        top = max(stages, key=lambda k: stages[k]["ms"])
        # DRAM bytes per launch of that kernel from the last committed ncu --set full capture (profiles/traffic.json)
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tj = json.load(f)
            fam = {"fft_analysis": ("dft_analysis_kernel", "fft_analysis_ct_kernel"), "fft_synthesis": ("dft_synthesis_kernel", "fft_synthesis_ct_kernel"),
                   "legendre_analysis": ("umma_kernel<AnaTraits>",), "legendre_synthesis": ("umma_kernel<SynTraits>",),
                   "mix_forward": ("umma_kernel<MixFwdTraits>",), "mix_backward": ("umma_kernel<MixDgradTraits>",)}
            keys = next((v for k, v in fam.items() if top.startswith(k)), ())
            for key in keys:   # only a capture of THIS workload says anything about this launch's traffic
                for name, rec in tj.items():
                    if key in name and rec.get("workload") == wl:
                        traffic = rec["dram_bytes_per_launch"]
                        break
                if traffic is not None:
                    break
        except Exception:
            traffic = None
        roof = {"bound": "hbm", "kernel": top, "achieved": stages[top]["GBps"], "peak": peak, "unit": "GB/s", "frac": round(stages[top]["GBps"] / peak, 4),
                "traffic": traffic, "peak_source": peak_src, "kernel_ms": stages[top]["ms"], "sum_stage_ms": round(sum(s["ms"] for s in stages.values()), 3)}

    # CPU baseline beside it (bounded sample: 1 warm-up + 2 timed steps of the same workload)
    cpu = None
    if not args.no_cpu and world == 1:   # reported at N = 1 only (the other ranks have left; the scaling runs need not wait for it)
        cores, avail = pick_cpu_threads()
        t = cpu_reference_steps(wl, 1, 1, act_dtype)
        cpu = {"value": 1.0 / t, "unit": "samples/s", "cores": cores, "kind": "port",
               "sample": f"1 warm-up + 1 timed full fwd+bwd step of {wl} through oracle/makani_oracle.py (torch.fft + torch.einsum fp32, {cores} threads "
                         f"chosen by calibration of {avail} available), {t:.2f} s/step"}

    # The library path the reference runs on a GPU (cuFFT + cuBLAS einsum, allow_tf32=True as makani/train.py:87), timed on this
    # B200 with the same restated modules (the real torch-harmonics is not installable): informational, never the product path.
    lib = None
    if not args.no_cpu and world == 1:
        try:
            lib = gpu_library_baseline(wl, act_dtype, dev, flush)
        except Exception as e:  # pragma: no cover
            lib = {"error": str(e)[:200]}

    x_bytes = x_host.numel() * x_host.element_size()
    line = {
        "metric": "SFNO-block fwd+bwd samples/sec", "value": world * 1e3 / ms_dev, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "tf32" if precision == "tf32" else ("f32 (3 x tf32 Legendre)" if precision == "fp32x3" else "f32"),
        "data": "synthetic",
        "config": {"workload": wl, "shape": [1, C, nlat_i, nlon_i], "activations": args.act, "contraction": {"tf32": "tcgen05 kind::tf32, fp32 accumulate", "fp32x3": "Legendre: 3 x TF32 on tcgen05 (fp32 operands); mix, FFT: fp32 FMA"}.get(precision, "fp32 FMA (CUDA cores)"),
                   "batch_per_gpu": 1, "global_batch": world, "parallelism": f"dp{world}" if world > 1 else "single", "dp_allreduce": dp_mode if world > 1 else None, "operator": "dhconv", "lmax": L, "mmax": M,
                   "l2": f"256 MiB buffer written between timed iterations (L2 flush); input {x_host.numel() * x_host.element_size() / 1e6:.0f} MB",
                   "weight_relayout_in_step": True, "flops_fwd_bwd_nnz": flops_fwd_bwd(wl)},
        "clocks": clocks,
        "e2e": {"value": world * 1e3 / ms_e2e, "unit": "samples/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": x_bytes, "d2h_bytes_per_step": gw_host.numel() * 8,
                "how": f"makani_b200.HostFeed: every step copies its {x_bytes / 1e6:.0f} MB input from pinned host memory and reads its weight gradient back; the "
                       "copy of step i+1 (side stream, second device buffer) and the read-back of step i-1 overlap the kernels of step i; K steps timed "
                       "from the first copy to the last read-back; two input buffers + gradients exceed the 126 MB L2",
                "serial_value": world * 1e3 / ms_e2e_serial, "serial_ms_per_step": ms_e2e_serial,
                "serial_how": "copy -> fwd+bwd -> read-back in one stream, L2 flushed between steps"},
        "gpu_launches": launches_per_step,
        # host time to enqueue one step (Python + ctypes + tensor-map encodes + launches), measured around the timed loop: when it is not well
        # below ms_per_step the step is launch-bound on this host and cuda_graph_replay (--graph) is the device-bound number
        "host_enqueue_ms_per_step": host_ms,
        "roofline": roof,
        "roofline_stages": stages,
        "cpu_baseline": cpu,
        "gpu_library_baseline": lib,
        "tflops_nnz": flops_fwd_bwd(wl) / (ms_dev * 1e-3) / 1e12,
    }
    if graph_info is not None:
        line["cuda_graph_replay"] = graph_info
    if hxw is not None:
        line["hxw"] = hxw
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------- full-model workloads
MODEL_WORKLOADS = {
    # BASELINE configs[2]: config/sfnonet.yaml sfno_sc3_layers8_edim384 (inp_chans 77 = 73 + zenith + orography + 2 land masks, driver.py:180-257)
    "sfno_sc3_layers8_edim384": dict(inp_shape=(721, 1440), out_shape=(721, 1440), inp_chans=77, out_chans=73, embed_dim=384, num_layers=8, scale_factor=3,
                                     model_grid_type="equiangular", sht_grid_type="legendre-gauss", filter_type="linear", operator_type="dhconv", use_mlp=True,
                                     mlp_ratio=2, activation_function="gelu", normalization_layer="instance_norm", hard_thresholding_fraction=1.0,
                                     pos_embed="none", complex_activation="real", separable=False),
    "sfno_tiny_model": dict(inp_shape=(49, 96), out_shape=(49, 96), inp_chans=7, out_chans=4, embed_dim=16, num_layers=3, scale_factor=3,
                            model_grid_type="equiangular", sht_grid_type="legendre-gauss"),
}


def run_model_arm(args):
    """fwd+bwd of the whole SFNO network (makani_b200.sfno on the CUDA kernels), bf16 autocast, loss = out.float().square().mean() (SURVEY cfg 3).
    One rank per GPU, data parallel replicas when WORLD_SIZE > 1 (no gradient exchange timed here: the block bench covers that)."""
    import makani_b200 as mb
    from makani_b200 import _lib
    from makani_b200.sfno import SphericalFourierNeuralOperatorNet

    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    cfg = MODEL_WORKLOADS[args.workload]
    precision = "tf32" if args.precision in ("best", "tf32") else "fp32"
    prev = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = True     # makani/train.py:87
    torch.manual_seed(333 + rank)
    net = SphericalFourierNeuralOperatorNet(**cfg, precision=precision).to(dev)
    act_dtype = torch.bfloat16 if args.act == "bf16" else torch.float32
    x_host = torch.randn(1, cfg["inp_chans"], *cfg["inp_shape"]).pin_memory()
    x_dev = x_host.to(dev)
    loss_host = torch.zeros(1).pin_memory()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def step(xd, keep=None):
        for p_ in net.parameters():
            p_.grad = None
        with torch.autocast(device_type="cuda", dtype=act_dtype, enabled=(act_dtype == torch.bfloat16)):
            out = net(xd)
        loss = out.float().square().mean()
        loss.backward()
        if keep is not None:   # --dump-outputs: what a caller of the step receives (the parameter gradients are read after the timed loop)
            keep.update(out=out.detach(), loss=loss.detach().reshape(1))
        return loss

    last = {} if args.dump_outputs else None   # outputs of the latest timed step

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        evs = []
        for _ in range(steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs) / steps
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    def step_e2e():
        xd = x_host.to(dev, non_blocking=True)
        loss_host.copy_(step(xd).detach().reshape(1), non_blocking=True)

    counter = {"n": 0}
    per_call = {"b200sht_spectral_conv_forward": 5, "b200sht_spectral_conv_backward": 6, "b200sht_spectral_conv_backward_ex": 7, "b200sht_mix_weight_pack": 1, "b200sht_mix_weight_unpack": 1,
                "b200sht_fft_analysis": 1, "b200sht_fft_synthesis": 1, "b200sht_legendre_analysis": 1, "b200sht_legendre_synthesis": 1,
                "b200sht_legendre_synthesis_tiled": 1, "b200sht_spec_pack": 1, "b200sht_spec_unpack": 1, "b200sht_bias_grad": 1}
    orig = _lib.call

    def counting(name, *a):
        counter["n"] += per_call.get(name, 0)
        return orig(name, *a)

    sampler = ClockSampler(local) if rank == 0 else None
    try:
        step(x_dev)
        torch.cuda.synchronize()
        _lib.call = counting
        step(x_dev)
        launches = counter["n"]
        _lib.call = orig
        if sampler:
            sampler.start()
            t_wait = time.perf_counter()
            while not sampler.lines and time.perf_counter() - t_wait < 5.0:
                step(x_dev)
                torch.cuda.synchronize()
        ms = timed(lambda: step(x_dev, last), args.steps, args.warmup)
        dumped = None
        if last is not None and rank == 0:
            grads = [sample_flat(p_.grad, DUMP_GRAD_SAMPLE, seed=i).reshape(-1) for i, (_, p_) in enumerate(net.named_parameters()) if p_.grad is not None]
            dumped = {"out": sample_flat(last["out"], DUMP_SAMPLE), "loss": last["loss"].float().cpu(), "param_grads": torch.cat(grads)}
        last = None
        clocks = sampler.stop() if sampler else None
        ms_e2e = timed(step_e2e, args.steps, max(1, args.warmup // 2))
    finally:
        _lib.call = orig
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    lib = None
    if not args.no_cpu and world == 1:
        # the same network on this GPU through torch.fft + torch.einsum (cuFFT / cuBLAS): what torch-harmonics + makani dispatch to
        try:
            from oracle.sfno_backend import OracleBackend

            del net
            torch.cuda.empty_cache()
            torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = True
            ref = SphericalFourierNeuralOperatorNet(**cfg, backend=OracleBackend()).to(dev)

            def ref_step():
                for p_ in ref.parameters():
                    p_.grad = None
                with torch.autocast(device_type="cuda", dtype=act_dtype, enabled=(act_dtype == torch.bfloat16)):
                    out = ref(x_dev)
                out.float().square().mean().backward()

            ms_lib = timed(ref_step, max(2, min(args.steps, 5)), 2)
            lib = {"value": 1e3 / ms_lib, "unit": "samples/s", "ms_per_step": ms_lib,
                   "what": "same network (makani_b200.sfno) with the spectral layers through torch.fft + torch.einsum on this GPU (cuFFT + cuBLAS, allow_tf32=True)"}
        except Exception as e:  # noqa: BLE001
            lib = {"error": str(e)[:300]}
        finally:
            torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev
    x_bytes = x_host.numel() * x_host.element_size()
    line = {
        "metric": "SFNO model fwd+bwd samples/sec", "value": world * 1e3 / ms, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16 autocast + " + precision, "data": "synthetic",
        "config": {"workload": args.workload, "shape": [1, cfg["inp_chans"], *cfg["inp_shape"]], "activations": args.act, "batch_per_gpu": 1, "global_batch": world,
                   "parallelism": f"dp{world} replicas" if world > 1 else "single", "embed_dim": cfg["embed_dim"], "num_layers": cfg["num_layers"],
                   "l2": "256 MiB buffer written between timed iterations (L2 flush)", "loss": "out.float().square().mean()"},
        "clocks": clocks,
        "e2e": {"value": world * 1e3 / ms_e2e, "unit": "samples/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": x_bytes, "d2h_bytes_per_step": 4,
                "how": "copy of the fp32 input from pinned host memory -> fwd+bwd -> read-back of the loss, one stream"},
        "gpu_launches": launches,
        "cpu_baseline": None,
        "gpu_library_baseline": lib,
    }
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the measured step (`value`, also with --impl reference); the side measurements (roofline_stages, hxw, "
                         "cpu_baseline, gpu_library_baseline) use their own small bounded counts")
    ap.add_argument("--warmup", type=int, default=5, help="untimed steps before the timed ones")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="sfno_block_721x1440x73", choices=sorted(WORKLOADS) + sorted(MODEL_WORKLOADS))
    ap.add_argument("--precision", default="best", choices=["best", "fp32", "tf32", "fp32x3"])
    ap.add_argument("--act", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-stages", action="store_true", help="skip per-stage kernel timing")
    ap.add_argument("--no-hxw", action="store_true", help="N > 1: skip the additional h x w spatial-model-parallel measurement of the same block")
    ap.add_argument("--graph", action="store_true", default=True, help="also time the step replayed from a CUDA graph (N = 1; reported as cuda_graph_replay, never as `value`)")
    ap.add_argument("--no-graph", dest="graph", action="store_false")
    ap.add_argument("--dp-mode", default=os.environ.get("B200SHT_DP_MODE", "trailing"), choices=["overlap", "trailing"],
                    help="N > 1: weight-gradient all-reduce after the backward pass on the compute stream (trailing, default: measured faster, DESIGN.md section 7) or on a "
                         "side stream behind the wgrad event with reserved SMs (overlap)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float32): block workloads y, dx, dweight; model workloads "
                         f"out, loss, param_grads; outputs over {DUMP_SAMPLE} elements as a fixed seeded sample of that many")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA path (--impl b200)")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback); use --impl reference for the CPU arm")
        if args.workload in MODEL_WORKLOADS:
            run_model_arm(args)
        else:
            run_gpu_arm(args)


if __name__ == "__main__":
    main()
