#!/usr/bin/env python
"""Benchmark of the gadfly GP hot path on B200 (contract: see the task's bench.py section).

Workload (BASELINE.json configs[2], the one the metric "solar kernel" is quoted on):
solar kernel ``Hyperparameters.for_sun()`` (86 SHO terms, J = 172), 1-min cadence light curves
of ``--n-points`` points (default 2^20 ~ 1M, SOHO/VIRGO-like), ``--batch`` light curves per GPU
(default: one per SM).  One *step* = one fused log-likelihood pass (K1) + one fused sampling
pass with in-kernel Philox normals (K2) over the whole batch.

  value   N*J^2-updates/s, device-timed, inputs resident in HBM          (whole job, all GPUs)
  e2e     same metric through the public Python API with HOST buffers (pinned), H2D/D2H
          copies inside the timed region
  roofline  FP64-FMA bound: algorithmic 4 J^2 flop per time step / kernel time vs the DFMA
          peak measured in this run by the library's microbenchmark (MEASURED_PEAKS.json has
          no FP64 figure); the HBM view (24 B per step) is reported beside it
  cpu_baseline  the oracle (celerite2-equivalent restatement, -O3 -march=native, OpenMP, one
          light curve per core) on a bounded sample of the same workload

``--impl reference`` times only that CPU path (celerite2 itself is not installable here:
DESIGN.md) and prints the same line with "impl": "reference".
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "GP loglike+sample N*J^2-updates/s (FP64), solar kernel"
UNIT = "N*J^2-updates/s"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--n-points", type=int, default=1 << 20)
    p.add_argument("--batch", type=int, default=0, help="light curves per GPU (0: one per SM)")
    p.add_argument("--cpu-points", type=int, default=1 << 16,
                   help="points per light curve of the bounded CPU sample")
    p.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--legs", default="cfg4,cfg5",
                   help="extra legs after the headline workload (cfg3): BASELINE configs[3] / [4], sharded over "
                        "the ranks with the NCCL gather inside the timed region; '' for none")
    p.add_argument("--grid", type=int, default=100000, help="cfg4: hyper-parameter grid points (whole job)")
    p.add_argument("--psd-stars", type=int, default=10000, help="cfg5: stars (whole job)")
    return p.parse_args()


def solar_kernel():
    import gadfly_b200 as g
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return g.SolarOscillatorKernel(texp=1 * g.units.min, bandpass="SOHO VIRGO")


# ---- CPU reference arm --------------------------------------------------------------------
def host_cores():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_reference(kernel, n_points, steps, warmup):
    """The celerite2-equivalent CPU path on all host cores: one light curve per core,
    loglike + sample per step.  Returns dict(value, cores, sample, ms_per_step)."""
    import oracle
    # the cores this process may run on -- NOT omp_get_max_threads(): torch.distributed.run exports
    # OMP_NUM_THREADS=1, which made the round-1 reference arm time one core at N > 1
    cores = host_cores()
    J = kernel.J
    scan = kernel.scan_coefficients()
    B = cores
    t = np.arange(n_points) * 6e-5
    rng = np.random.default_rng(42)
    y = rng.standard_normal(B * n_points) * 300.0
    n_off = np.arange(B + 1) * n_points
    t_off = np.zeros(B, dtype=np.int64)
    j_off = np.arange(B + 1) * len(scan[2])
    coef = [np.tile(scan[i], B) for i in (2, 3, 4, 5)]
    ddiag = np.full(B, scan[6])

    def step():
        oracle.stream_batch(0, n_off, t_off, j_off, t, y, ddiag, *coef, nthreads=cores, fast=True)
        oracle.stream_batch(1, n_off, t_off, j_off, t, y, ddiag, *coef, nthreads=cores, fast=True)

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    updates = 2.0 * B * n_points * J * J
    return dict(value=updates / dt, unit=UNIT, cores=cores, kind="port",
                sample=f"{B} light curves x {n_points} points, solar J={J}, loglike+sample per step, "
                       f"{steps} steps after {warmup} warm-up; oracle/celerite_oracle.c "
                       f"-O3 -march=native, OpenMP one light curve per core",
                ms_per_step=dt * 1e3, light_curves_per_s=2.0 * B / dt)


# ---- clocks -------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        with open(self.path) as fh:
            for line in fh:
                parts = [x.strip() for x in line.split(",")]
                if len(parts) < 7:
                    continue
                try:
                    sm.append(float(parts[0])); mx.append(float(parts[1])); pw.append(float(parts[2]))
                except ValueError:
                    continue
                for nm, v in zip(names, parts[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        os.unlink(self.path)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(np.max(mx)),
                    power_w_max=float(np.max(pw)), samples=len(sm), reasons=sorted(reasons))



# ---- sharded legs: BASELINE configs[3] and [4] ---------------------------------------------
def _timed(dev, world, fn):
    """Device time [s] of fn() on torch's current stream, barrier + synchronize on both sides,
    maximum over ranks."""
    import torch
    import torch.distributed as dist
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    v = torch.tensor([e0.elapsed_time(e1) * 1e-3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        dist.barrier()
    return float(v.item()), out


def leg_cfg4(args, solver, dev, rank, world, peak):
    """Hyper-parameter grid x one 100 000-point light curve (GF_FLAG_SHARED_Y: passed once), strong
    scaling: the grid is cut into contiguous blocks (batch.shard_bounds), every rank scans its block,
    and log L + status of the WHOLE grid are all-gathered by NCCL inside the timed region."""
    import torch
    from gadfly_b200 import batch, solver as S, workloads
    from gadfly_b200.solver import Geometry
    G, N = args.grid, 100000
    bounds = batch.shard_bounds(np.ones(G), world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    _, host_feeder_s = workloads.lattice_batch(G, 3, lo, hi)               # host feeder, for the record
    workloads.lattice_batch(G, 3, lo, min(hi, lo + 8), solver=solver)      # warm-up of the device feeder
    kb, feeder_s = workloads.lattice_batch(G, 3, lo, hi, solver=solver)
    J = kb.J.astype(np.float64)
    gen = torch.Generator(device=dev)
    gen.manual_seed(3)                                   # the same light curve on every rank
    t = torch.arange(N, dtype=torch.float64, device=dev) * 6e-5
    y = torch.randn(N, dtype=torch.float64, device=dev, generator=gen) * 285.0
    B = kb.B
    logdet = torch.empty(B, dtype=torch.float64, device=dev)
    quad = torch.empty(B, dtype=torch.float64, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    geom = Geometry.shared_t(B, N)

    def run():
        solver.loglike(kb, geom, t, y, logdet=logdet, quad=quad, status=status,
                       flags=S.FLAG_SHARED_Y | S.FLAG_ASYNC)
        ll = -0.5 * (quad + logdet + N * float(np.log(2 * np.pi)))
        return batch.gather_concat(ll, bounds), batch.gather_concat(status, bounds)

    # warm-up on a few grid points (allocations, NCCL channels), then ONE timed pass over the grid
    kw = kb.take(np.arange(min(B, 8)))
    solver.loglike(kw, Geometry.shared_t(kw.B, N), t, y, flags=S.FLAG_SHARED_Y)
    if world > 1:
        batch.gather_concat(torch.zeros(B, dtype=torch.float64, device=dev), bounds)
    seconds, (ll_all, st_all) = _timed(dev, world, run)
    assert ll_all.numel() == G and int(st_all.abs().sum().item()) == 0
    # the gathered vector against a recomputation, on THIS rank's GPU, of a slice that another rank owns
    other = (rank + 1) % world
    s_lo = int(bounds[other])
    s_n = min(8, int(bounds[other + 1]) - s_lo)
    ks, _ = workloads.lattice_batch(G, 3, s_lo, s_lo + s_n, solver=solver)
    ll_s = batch.log_likelihood(ks, t, y, solver=solver, flags=S.FLAG_SHARED_Y)
    got = ll_all[s_lo:s_lo + s_n].cpu().numpy()
    assert np.array_equal(got, ll_s), (got, ll_s)
    flops_local = 4.0 * float(np.sum(J * J)) * N
    return dict(workload=f"BASELINE configs[3]: {G} hyper-parameter sets (solar kernel, S0/w0/Q lattice +-10 %) x "
                         f"one {N}-point light curve, log-likelihood; grid sharded over {world} rank(s)",
                grid_points=G, n_points=N, J=int(J.max()), seconds=seconds, scaling="strong",
                grid_points_per_s=G / seconds, updates_per_s=float(np.mean(J * J)) * G * N / seconds,
                fp64_frac_per_gpu=flops_local / seconds / peak if peak else None,
                gather=dict(collective="all_gather_into_tensor (NCCL)" if world > 1 else "none (1 rank)",
                            in_timed_region=True, bytes_per_rank=int(B * 12), verified=f"{s_n} grid points of rank "
                            f"{other} recomputed on rank {rank}: bit-identical"),
                host_feeder_s=host_feeder_s, device_feeder_s=feeder_s)


def leg_cfg5(args, solver, dev, rank, world, peak):
    """Kernel PSD of Kepler-like stars on a 10^6-bin grid: stars sharded over the ranks; the rows
    stay on the rank that made them (10^4 x 10^6 doubles are 80 GB), a per-star checksum (sum over
    the bins) is all-gathered by NCCL inside the timed region."""
    import torch
    from gadfly_b200 import batch, solver as S, workloads
    n_stars, F, chunk = args.psd_stars, 1000000, 256
    _, host_feeder_s = workloads.kepler_like_batch(n_stars, 4)            # host feeder, for the record
    workloads.kepler_like_batch(8, 4, solver=solver)                       # warm-up of the device feeder
    kb_all, feeder_s = workloads.kepler_like_batch(n_stars, 4, solver=solver)
    nterm = np.diff(kb_all.j_off).astype(np.float64)
    bounds = batch.shard_bounds(nterm, world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    omega = torch.as_tensor(2 * np.pi * np.linspace(0.01, 8333.0, F), device=dev)
    out = torch.empty(chunk * F, dtype=torch.float64, device=dev)
    chunks = [kb_all.take(np.arange(a, min(a + chunk, hi))) for a in range(lo, hi, chunk)]
    sums = torch.empty(hi - lo, dtype=torch.float64, device=dev)

    def run():
        pos = 0
        for kc in chunks:
            solver.psd(kc, omega, out=out[:kc.B * F], flags=S.FLAG_ASYNC)
            sums[pos:pos + kc.B] = out[:kc.B * F].view(kc.B, F).sum(dim=1)
            pos += kc.B
        return batch.gather_concat(sums, bounds)

    solver.psd(chunks[0], omega, out=out[:chunks[0].B * F])
    if world > 1:
        batch.gather_concat(sums, bounds)
    seconds, all_sums = _timed(dev, world, run)
    assert all_sums.numel() == n_stars and bool(torch.isfinite(all_sums).all())
    # one star against the closed form of the reference (gadfly/core.py:33-41) x sinc^2, every bin
    kc = chunks[-1]
    solver.psd(kc, omega, out=out[:kc.B * F])
    row = out[(kc.B - 1) * F:kc.B * F].cpu().numpy()
    w = omega.cpu().numpy()
    ref = np.zeros(F)
    for a, b, c, d in kc.base[kc.j_off[kc.B - 1]:kc.j_off[kc.B]]:
        w0 = np.sqrt(c * c + d * d)
        Q = w0 / (2 * c)
        ref += np.sqrt(2 / np.pi) * (a / (w0 * Q)) * w0 ** 4 / ((w ** 2 - w0 ** 2) ** 2 + (w ** 2 * w0 ** 2 / Q ** 2))
    arg = 0.5 * kc.delta[kc.B - 1] * w
    ref *= (np.sin(arg) / arg) ** 2
    rel = float(np.max(np.abs(row / ref - 1)))
    # (the (a, b, c, d) form of the PSD, A.5, cancels by ~Q^2 next to a p-mode resonance: up to ~1e-7 there; parity with
    # the oracle, which evaluates the same form, is 1e-12 in tests/)
    assert rel < 1e-6, rel
    assert abs(float(all_sums[hi - 1].item()) / float(np.sum(row)) - 1) < 1e-12
    flops_local = 12.0 * float(np.sum(nterm[lo:hi])) * F
    return dict(workload=f"BASELINE configs[4]: kernel PSD of {n_stars} Kepler-like stars on a {F}-bin grid "
                         f"(to the Nyquist frequency of the 1-min cadence); stars sharded over {world} rank(s)",
                stars=n_stars, bins=F, seconds=seconds, scaling="strong",
                star_bins_per_s=n_stars * float(F) / seconds,
                fp64_frac_per_gpu=flops_local / seconds / peak if peak else None,
                hbm_write_GBps_per_gpu=(hi - lo) * F * 8 / seconds / 1e9,
                gather=dict(collective="all_gather_into_tensor (NCCL)" if world > 1 else "none (1 rank)",
                            in_timed_region=True, payload="per-star sum over the bins (rows stay sharded)",
                            bytes_per_rank=int((hi - lo) * 8)),
                max_rel_vs_closed_form=rel, host_feeder_s=host_feeder_s, device_feeder_s=feeder_s)

# ---- the B200 arm -------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    import gadfly_b200 as g
    from gadfly_b200 import batch, solver as S
    from gadfly_b200.solver import Geometry, KernelBatch, Solver

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run for --gpus > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    kernel = solar_kernel()
    J = kernel.J
    solver = Solver(local)
    info = solver.device_info(measure=True)
    B = args.batch or info["sm_count"]
    N = args.n_points
    kb = KernelBatch([kernel] * B)
    geom = Geometry.shared_t(B, N)

    # synthetic data, resident in HBM: white N(0, k(0)) draws (the scan's cost is data-independent)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    k0 = float(np.sum(kb.coef[:len(kernel.term.terms), 0]) + kb.ddiag[0])
    t_dev = torch.arange(N, dtype=torch.float64, device=dev) * 6e-5
    y_dev = torch.randn(B * N, dtype=torch.float64, device=dev, generator=gen) * k0 ** 0.5
    x_dev = torch.empty(B * N, dtype=torch.float64, device=dev)
    logdet = torch.empty(B, dtype=torch.float64, device=dev)
    quad = torch.empty(B, dtype=torch.float64, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    stream = torch.cuda.ExternalStream(solver.stream, device=dev)

    kernel_ms = {"loglike": [], "sample": []}

    def step(i, record=False):
        solver.loglike(kb, geom, t_dev, y_dev, logdet=logdet, quad=quad, status=status,
                       flags=S.FLAG_ASYNC)
        if record:
            kernel_ms["loglike"].append(solver.last_kernel_ms)
        solver.sample(kb, geom, t_dev, seed=1000 + i, seq0=rank * B, out=x_dev, logdet=logdet,
                      status=status, flags=S.FLAG_ASYNC)
        if record:
            kernel_ms["sample"].append(solver.last_kernel_ms)

    def sync_all():
        solver.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    torch.cuda.synchronize()      # the synthetic inputs above were produced on torch's stream
    for i in range(args.warmup):
        step(i)
    sync_all()

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    launches0 = solver.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record(stream)
    for i in range(args.steps):
        step(args.warmup + i)
    e1.record(stream)
    sync_all()
    ms_total = e0.elapsed_time(e1)
    launches = solver.launch_count - launches0
    clk = clocks.stop() if rank == 0 else None
    assert int(status.abs().sum().item()) == 0, "non-positive pivot in the benchmark batch"

    # per-kernel device times: re-run the timed steps synchronously (same launches)
    for i in range(args.steps):
        step(args.warmup + i, record=True)
    sync_all()

    # ---- e2e: public API, pinned host buffers, copies inside the timed region ------------
    e2e = None
    if not args.no_e2e:
        t_host = torch.empty(N, dtype=torch.float64).pin_memory()
        t_host.copy_(t_dev)
        y_host = torch.empty(B * N, dtype=torch.float64).pin_memory()
        y_host.copy_(y_dev)
        x_host = torch.empty(B * N, dtype=torch.float64).pin_memory()
        t_np, y_np, x_np = t_host.numpy(), y_host.numpy(), x_host.numpy()

        def e2e_issue(i):
            # One step = sample + log-likelihood of the whole batch from / to pinned host buffers.  The
            # sample call needs only t: issued first, its kernel runs beside the H2D copy of y (copy-in
            # stream); the log-likelihood kernel then runs beside the D2H copy of x (copy-out stream).
            # Nothing blocks the host here: the step's result is read one step later (result() waits
            # for THAT step's ticket), so the next step's copies and kernels are queued behind the
            # running ones.  (The small outputs -- log det, status: ordinary numpy arrays -- reach the
            # host through the handle's pinned ring; copied straight into pageable memory they held
            # the host until the kernel had finished, which is what kept H2D(y) from overlapping in
            # round 1 and early round 2: tools/overlap_probe2.cu, overlap_probe3.py, e2e_probe.py.)
            solver.sample(kb, geom, t_np, seed=2000 + i, seq0=rank * B, out=x_np, flags=S.FLAG_ASYNC)
            return batch.log_likelihood(kb, t_np, y_np, solver=solver, wait=False)

        e2e_issue(0).result()
        sync_all()
        t0 = time.perf_counter()
        n_e2e = max(1, args.steps)
        pending = None
        for i in range(n_e2e):
            nxt = e2e_issue(1 + i)
            if pending is not None:
                assert np.all(np.isfinite(pending.result()))       # the previous step's log-likelihoods
            pending = nxt
        ll = pending.result()
        assert np.all(np.isfinite(ll))
        sync_all()
        dt = time.perf_counter() - t0
        e2e = dict(seconds=dt / n_e2e,
                   h2d=(2 * N + B * N) * 8 + 2 * (4 * len(kb.coef) + B) * 8,
                   d2h=B * N * 8 + 2 * B * (8 + 8 + 4))
        del t_host, y_host, x_host

    # ---- reduce over ranks ------------------------------------------------------------------
    vals = torch.tensor([ms_total, e2e["seconds"] if e2e else 0.0,
                         float(np.mean(kernel_ms["loglike"])), float(np.mean(kernel_ms["sample"]))],
                        dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    ms_total, e2e_s, ll_ms, sm_ms = [float(v) for v in vals.cpu()]
    units_per_step = 2.0 * world * B * N * J * J
    ms_per_step = ms_total / args.steps
    value = units_per_step / (ms_per_step * 1e-3)

    # free the headline workload's buffers, then the sharded legs (every rank takes part)
    del y_dev, x_dev
    torch.cuda.empty_cache()
    extra = {}
    for leg in [x for x in args.legs.split(",") if x]:
        fn = {"cfg4": leg_cfg4, "cfg5": leg_cfg5}[leg]
        extra[leg] = fn(args, solver, dev, rank, world, info["fp64_flops"])

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:      # reported baseline: rank 0 at N = 1 only
        cpu = cpu_reference(kernel, args.cpu_points, 1, 1)

    if rank == 0:
        flops_per_launch = 4.0 * J * J * B * N
        dom = "loglike" if ll_ms >= sm_ms else "sample"
        dom_ms = max(ll_ms, sm_ms)
        achieved = flops_per_launch / (dom_ms * 1e-3) / 1e12
        peak = info["fp64_flops"] / 1e12
        hbm_peak = 6553.6
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                hbm_peak = float(json.load(fh)["hbm_gbs"])
        except Exception:
            pass
        hbm_achieved = 24.0 * B * N / (dom_ms * 1e-3) / 1e9
        # DRAM traffic of one launch of the dominant kernel: only from an ncu capture of THIS launch
        # geometry (profiles/r2_traffic.json, same B x N), never extrapolated from a smaller one
        # whose output still fits in L2; otherwise null
        traffic, traffic_src = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as fh:
                tj = json.load(fh)
            ent = tj.get(f"scan ({dom})")
            if ent and int(ent["points_per_launch"]) == B * N:
                traffic = float(ent["dram_bytes_read"] + ent["dram_bytes_write"])
                traffic_src = (f"ncu --set full of scan ({dom}) at {B} x {N} points "
                               f"(profiles/r2_traffic.json): dram__bytes_read.sum + dram__bytes_write.sum")
        except Exception:
            pass
        nominal = 148 * 64 * 2 * 1.965e9 / 1e12
        # executed work: the kernel stores the upper triangle only and spends 3 DFMA per stored
        # element (8x8 register tiles, 253 of them at J <= 176): 6 flop x 253 x 64 per step
        nt = ((J + 7) // 8) * ((J + 7) // 8 + 1) // 2
        executed = 6.0 * 64 * nt * B * N / (dom_ms * 1e-3) / 1e12
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": f"BASELINE configs[2]: solar kernel Hyperparameters.for_sun() "
                            f"(86 SHO terms, J={J}), {B} light curves/GPU x {N} points at 1-min "
                            f"cadence; step = fused log_likelihood + fused Philox sample over the batch",
                "light_curves_per_gpu": B, "n_points": N, "J": J,
                "l2": "inputs larger than L2 (t,y,x: %.1f GB per step)" % (3 * B * N * 8 / 1e9),
                "sharding": "independent light curves per rank, no data-path collective",
            },
            "light_curves_per_s": 2.0 * world * B / (ms_per_step * 1e-3),
            "roofline": {
                "bound": "fp64", "kernel": f"scan ({dom})", "achieved": achieved, "peak": peak,
                "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                "frac_nominal": achieved / nominal, "peak_nominal": nominal,
                "executed": {"tflops": executed, "frac": executed / peak if peak else None,
                             "note": "DFMA actually issued by the matrix warps (3 per stored element of "
                                     "the upper triangle, padded to 8x8 tiles); `achieved` counts the "
                                     "algorithmic 4 J^2 of SURVEY 8d"},
                "peak_source": "DFMA microbenchmark measured in this run (gf_device_info); "
                               "MEASURED_PEAKS.json has no FP64 figure; nominal 148 SM x 64 FMA/clk "
                               "x 2 x 1.965 GHz = 37.2",
                "algorithmic": "4 J^2 flop per time step (SURVEY 8d) x B x N per launch",
                "kernel_ms": {"loglike": ll_ms, "sample": sm_ms},
                "hbm": {"achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s",
                        "frac": hbm_achieved / hbm_peak, "bytes_per_step": 24},
                "traffic": traffic, "traffic_source": traffic_src,
            },
            "gpu_launches": int(launches),
            "clocks": clk,
        }
        if e2e:
            line["e2e"] = {"value": units_per_step / e2e_s, "unit": UNIT,
                           "h2d_bytes_per_step": int(e2e["h2d"]), "d2h_bytes_per_step": int(e2e["d2h"]),
                           "ms_per_step": e2e_s * 1e3,
                           "api": "Solver.sample(FLAG_ASYNC) + gadfly_b200.batch.log_likelihood(wait=False) on pinned host "
                                  "arrays, result() of each step read while the next one runs"}
        if cpu:
            line["cpu_baseline"] = cpu
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kernel = solar_kernel()
    cpu = cpu_reference(kernel, args.cpu_points, args.steps, max(args.warmup, 1))
    J = kernel.J
    line = {
        "impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": cpu["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"BASELINE configs[2]: solar kernel (J={J}), bounded sample: "
                               f"{cpu['cores']} light curves x {args.cpu_points} points on the host "
                               f"cores; step = log_likelihood + sample"},
        "light_curves_per_s": cpu["light_curves_per_s"],
        "cpu_baseline": {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cpu["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "celerite2 is not installable here (no wheel, no Eigen, no network): the CPU arm is "
                "the validated restatement in oracle/ (DESIGN.md)",
    }
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
