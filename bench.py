#!/usr/bin/env python
"""bench.py -- geodesics/sec of the B200 hot path on BASELINE.json's headline configuration.

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference ...                     (the reference algorithm on the host cores: CPU oracle)
  python bench.py ... --dump-outputs bench_outputs         (also write the last timed step's images to bench_outputs/<name>.npy)

A "step" is one full render of the workload: Kerr a=0.998, observer r=1000 theta=60deg, ThinDisc(0,50),
2048 x 2048 image plane per GPU, two fused point functions (redshift + disc radius), Tsit5 abstol=reltol=1e-9
(BASELINE.json configs[1]).  Rays shard across ranks with no data-path collective (weak scaling: the
image is 2048 x (2048*N) over the same field of view and rank r integrates every N-th strip of 4 image columns).
Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H_IMG = 2048
W_IMG_PER_GPU = 2048
F_RHS = {0: 118.0, 1: 163.0}  # algorithmic flops per RHS evaluation (Kerr: SURVEY 8d; JP: the Euler-Lagrange closed form, FMA = 2; round 1 counted 222 for the generated Jacobian + contraction)
F_STAGE, F_EVENT, F_IC, F_END = 566.0, 280.0, 60.0, 150.0


def flops_per_attempt(metric_kind, has_disc):
    return 6.0 * F_RHS[metric_kind] + F_STAGE + (F_EVENT if has_disc else 0.0)


def build_workload(world, ensemble=None):
    import gradus_b200 as gb
    from gradus_b200.api import RenderGrid, tracing_configuration

    m = gb.KerrMetric(M=1.0, a=0.998)
    x = [0.0, 1000.0, math.radians(60.0), 0.0]
    d = gb.ThinDisc(0.0, 50.0)
    w, h = W_IMG_PER_GPU * world, H_IMG
    cfg = tracing_configuration(m, x, RenderGrid(w, h, (-60, 60), (-40, 40)), d, 2000.0, ensemble=ensemble, trajectories=w * h)
    return cfg, w, h


_JSON_FD = None


def claim_stdout():
    """Keep the process's stdout for the single JSON line: fd 1 is pointed at stderr for everything else (NCCL prints its
    version banner to stdout from C, whatever NCCL_DEBUG the box sets)."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(out):
    line = (json.dumps(out) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, line)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.rows, self.proc, self.device = [], None, device

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


REF_SAMPLE_RAYS = 262144  # rays per step of the CPU arm: the same bounded sample at every N


def host_threads():
    """Every host core of the box: torchrun exports OMP_NUM_THREADS=1 to its workers, which would otherwise pin the CPU
    arm to one thread at N > 1."""
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args, rank, world):
    """The reference's CPU algorithm (EnsembleEndpointThreads work decomposition) on this box's host cores.
    Julia cannot run here, so this is the C++ oracle port (kind = "port"), all host threads, bounded sample per step:
    every k-th ray of the SAME image the GPU arm renders, k chosen so that a step is REF_SAMPLE_RAYS rays at every N."""
    if rank != 0:
        return
    from gradus_b200 import _cabi as cabi
    from oracle import oracle

    cfg, w, h = build_workload(world)
    p, ic = cfg.to_c(validate=False)
    stride = args.ref_stride if args.ref_stride > 0 else max(1, ic.n // REF_SAMPLE_RAYS)
    rng = cabi.Range(0, (ic.n + stride - 1) // stride, stride)
    pfs = [cabi.PF_REDSHIFT, cabi.PF_DISC_RADIUS]
    threads = host_threads()
    # The arm the driver's ratio is taken against is the OPTIMISED build of the port (-O3, FMA, closed-form Kerr right-hand
    # side: ~10x the checker build, and per thread what the reference documents for itself, docs/src/getting-started.md:437);
    # the checker build (dual-number Jacobian, -O2, no contraction) is timed once beside it.
    for _ in range(args.warmup):
        oracle.render_fast(p, ic, pfs, rng=rng, nthreads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        imgs = oracle.render_fast(p, ic, pfs, rng=rng, nthreads=threads)
    dt = (time.perf_counter() - t0) / args.steps
    val = rng.count / dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"redshift": imgs[0], "disc_radius": imgs[1]})
    t0 = time.perf_counter()
    oracle.render(p, ic, pfs, rng=cabi.Range(0, max(1, rng.count // 4), stride * 4), nthreads=threads)
    checker = max(1, rng.count // 4) / (time.perf_counter() - t0)
    sample = f"every {stride}th ray of the {w}x{h} image ({rng.count} rays per step)"
    out = {
        "impl": "reference", "metric": "geodesics/sec", "value": val, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": workload_config(world, w, h),
        "cpu_baseline": {"value": val, "unit": "rays/s", "cores": threads, "kind": "port", "sample": sample,
                         "build": "port_optimised: g++ -O3 -march=x86-64-v3 -ffp-contract=fast, closed-form Kerr right-hand side (oracle/liboracle_fast.so)",
                         "checker_build": {"value": checker, "unit": "rays/s", "kind": "port", "build": "-O2 -ffp-contract=off, dual-number metric Jacobian (oracle/liboracle.so)"}},
        "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(out)


def workload_config(world, w, h):
    return {"workload": f"C2: KerrMetric a=0.998, observer r=1000 theta=60deg, ThinDisc(0,50), {w}x{h} image plane "
                        f"({W_IMG_PER_GPU}x{H_IMG} per GPU), redshift + disc-radius point functions, Tsit5 abstol=reltol=1e-9, lambda_max=2000",
            "rays_per_gpu": W_IMG_PER_GPU * H_IMG, "parallelism": f"ray-sharded x{world} (strips of 4 image columns interleaved over ranks, no collective)",
            "l2": "flushed between timed steps (256 MiB write); the kernel reads no input arrays"}


def run_ours(args, rank, world, local):
    import torch

    import gradus_b200 as gb
    from gradus_b200 import _cabi as cabi
    from gradus_b200 import distributed as gd

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the host baseline)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    lib = cabi.load()
    ens = gb.EnsembleB200(devices=(local,))
    ctx = ens.ctx(local)
    cfg, w, h = build_workload(world, ensemble=ens)
    p, ic = cfg.to_c()
    rng = gd.strip_interleaved_range(ic, rank, world)
    n_local = rng.count
    pfs = np.array([cabi.PF_REDSHIFT, cabi.PF_DISC_RADIUS], np.int32)
    stream = torch.cuda.Stream(device=dev)  # explicit non-default stream: the library launches on it, the events time it
    torch.cuda.set_stream(stream)
    sptr = C.c_void_p(stream.cuda_stream)

    # ---- device-resident arm: outputs stay in HBM
    d_imgs = [torch.empty(n_local, dtype=torch.float64, device=dev) for _ in pfs]
    d_ptrs = (C.c_void_p * len(pfs))(*[C.c_void_p(t.data_ptr()) for t in d_imgs])
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def step_device(async_=1):
        cabi.check(lib.gb200_render_device(ctx, C.byref(p), C.byref(ic), C.byref(rng), cabi.iptr(pfs), len(pfs), None, d_ptrs, sptr, async_), ctx)

    peak = C.c_double()
    cabi.check(lib.gb200_fp64_peak(ctx, C.byref(peak)), ctx)
    peak3 = C.c_double()  # the same stream with three distinct register operands per DFMA (register-file bound)
    cabi.check(lib.gb200_fp64_issue_probe(ctx, 3, C.byref(peak3)), ctx)
    step_device(0)  # synchronous once: per-call counters for the algorithmic flop count
    st = ens.stats(local)
    attempts = st.steps_accepted + st.steps_rejected
    for _ in range(args.warmup):
        step_device()
    torch.cuda.synchronize()
    gd.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    torch.cuda.synchronize()
    for a, b in evs:
        flush.fill_(1.0)  # L2 flush, outside the event pair
        a.record(stream)
        step_device()
        b.record(stream)
    torch.cuda.synchronize()
    gd.barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms_local = sum(a.elapsed_time(b) for a, b in evs) / args.steps
    ms = gd.max_over_ranks(ms_local, dev)
    ms_ranks = gd.gather_floats(ms_local, dev)
    total_rays = gd.sum_over_ranks(float(n_local), dev)
    total_attempts = gd.sum_over_ranks(float(attempts), dev)
    value = total_rays / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"redshift": d_imgs[0].cpu().numpy(), "disc_radius": d_imgs[1].cpu().numpy()})

    # ---- end-to-end arm: the reference-facing C-ABI call with HOST buffers (D2H inside the timed region)
    h_imgs = [torch.empty(n_local, dtype=torch.float64, pin_memory=True) for _ in pfs]
    h_ptrs = (cabi._dp * len(pfs))(*[C.cast(t.data_ptr(), cabi._dp) for t in h_imgs])

    def step_e2e():
        cabi.check(lib.gb200_render(ctx, C.byref(p), C.byref(ic), C.byref(rng), cabi.iptr(pfs), len(pfs), None, h_ptrs), ctx)

    for _ in range(args.warmup):
        step_e2e()
    torch.cuda.synchronize()
    gd.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_local = (time.perf_counter() - t0) / args.steps
    gd.barrier()
    e2e_s = gd.max_over_ranks(e2e_local, dev)
    e2e_value = total_rays / e2e_s
    checksum = float(np.nansum(h_imgs[0].numpy()))

    # ---- which parity tolerance covers which share of this workload's rays (tests/test_gpu_parity.py::check_parity)
    d_status = torch.empty(n_local, dtype=torch.float64, device=dev)
    spf = np.array([cabi.PF_STATUS], np.int32)
    cabi.check(lib.gb200_render_device(ctx, C.byref(p), C.byref(ic), C.byref(rng), cabi.iptr(spf), 1, None, (C.c_void_p * 1)(C.c_void_p(d_status.data_ptr())), sptr, 0), ctx)
    frac = torch.bincount(d_status.to(torch.int64), minlength=4).double().cpu().numpy() / n_local
    parity = {
        "protocol": "GPU vs CPU oracle on identical inputs; identical termination class for every ray outside the grazing band (0.42 % of C1/C2 rays)",
        "intersected_with_geometry": {"fraction": float(frac[2]), "tolerance": "end point and momentum 1e-6 relative, redshift 1e-6 absolute (root-found on the dense output)"},
        "no_status": {"fraction": float(frac[3]), "tolerance": "end point 1e-6 relative at lambda_max"},
        "within_inner_boundary": {"fraction": float(frac[1]), "tolerance": "class identical; state on the oracle's geodesic at the same affine parameter to 2e-4 "
                                  "(the chart callback r <= 1.01 r_h has no root find, charts.jl:8-24: the stored point is wherever the last step landed)"},
        "out_of_domain": {"fraction": float(frac[0]), "tolerance": "class identical; state on the oracle's geodesic to 1e-5"},
    }

    # ---- secondary: binned line profile with the histogram all-reduced over NCCL (BASELINE.json configs[2])
    lp = None
    if not args.no_lineprofile:
        lp = run_lineprofile(args, rank, world, local, ens, dev, stream, sptr)

    strong = None
    if not args.no_strong:
        strong = run_strong(args, rank, world, local, ens, dev, stream, sptr)

    if rank != 0:
        return
    # ---- roofline (FP64 CUDA-core pipe; DESIGN.md states the per-attempt algorithmic flop count)
    fpa = flops_per_attempt(p.metric_kind, p.geometry_kind != 0)
    flops_per_launch_local = attempts * fpa + n_local * (F_IC + F_END)
    achieved = flops_per_launch_local / (ms_local * 1e-3) / 1e12
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    nominal_fp64 = 148 * 64 * 2 * (peaks.get("sm_max_mhz", 1965.0) * 1e6) / 1e12
    traffic = None
    try:  # dram bytes per launch of the same kernel from the committed `ncu --set full` capture
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
    except Exception:
        pass
    roofline = {
        "bound": "fp64", "achieved": achieved, "peak": peak.value, "unit": "TFLOP/s", "frac": achieved / peak.value if peak.value else None,
        "traffic": traffic,
        "traffic_note": "bytes per launch (dram read + write) from profiles/r02_traffic.json; algorithmic bytes per launch = 16 B x rays",
        "peak_source": "measured in this run: dependent-free DFMA micro-benchmark (gb200_fp64_peak); MEASURED_PEAKS.json has no FP64 entry",
        "peak_nominal": nominal_fp64,
        "peak_three_register_dfma": peak3.value,
        "peak_note": "peak = DFMAs with one constant operand; DFMAs whose three operands are distinct registers sustain only "
                     "peak_three_register_dfma on this chip (register-file read bandwidth), and 22 % of this kernel's FP64 instructions are such",
        "flops_per_step_attempt": fpa, "step_attempts_per_ray": attempts / max(n_local, 1),
        "hbm": {"algorithmic_bytes_per_ray": 16, "achieved_GBs": 16.0 * n_local / (ms_local * 1e-3) / 1e9, "peak_GBs": peaks.get("hbm_gbs")},
    }
    # ---- CPU baseline: the oracle port on a bounded sample of the same workload (rank 0, N = 1 only)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import oracle

        threads = host_threads()
        stride = args.cpu_stride if args.cpu_stride > 0 else max(1, ic.n // (4 * REF_SAMPLE_RAYS))
        crng = cabi.Range(0, (ic.n + stride - 1) // stride, stride)
        t0 = time.perf_counter()
        oracle.render_fast(p, ic, [cabi.PF_REDSHIFT, cabi.PF_DISC_RADIUS], rng=crng, nthreads=threads)
        fdt = time.perf_counter() - t0
        srng = cabi.Range(0, (ic.n + 4 * stride - 1) // (4 * stride), 4 * stride)
        t0 = time.perf_counter()
        oracle.render(p, ic, [cabi.PF_REDSHIFT, cabi.PF_DISC_RADIUS], rng=srng, nthreads=threads)
        cdt = time.perf_counter() - t0
        cpu = {"value": crng.count / fdt, "unit": "rays/s", "cores": threads, "kind": "port",
               "sample": f"every {stride}th ray of the {w}x{h} image ({crng.count} rays, {fdt:.1f} s)",
               "build": "port_optimised: g++ -O3 -march=x86-64-v3 -ffp-contract=fast, closed-form Kerr right-hand side (oracle/liboracle_fast.so)",
               "checker_build": {"value": srng.count / cdt, "unit": "rays/s", "kind": "port", "sample": f"{srng.count} rays, {cdt:.1f} s",
                                 "build": "-O2 -ffp-contract=off, dual-number metric Jacobian (oracle/liboracle.so): the build every parity test uses"},
               "note": "C++ restatement of the reference algorithm (no Julia in this image). The reference documents ~3.3e4 rays/s for itself on a "
                       "2021 M1 laptop (docs/src/getting-started.md:437); per thread that is what the optimised build reaches"}
    out = {
        "metric": "geodesics/sec", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(world, w, h),
        "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": C.sizeof(cabi.Problem) + C.sizeof(cabi.IC) + C.sizeof(cabi.Range),
                "d2h_bytes_per_step": 8 * len(pfs) * n_local, "ms_per_step": e2e_s * 1e3, "timing": "wall clock around the blocking C-ABI call, max over ranks"},
        "gpu_launches": int(args.steps * 1),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "clocks": clocks,
        "ms_per_step_per_rank": ms_ranks,
        "total_rays_per_step": total_rays, "step_attempts_per_step": total_attempts, "image_checksum": checksum,
    }
    out["parity"] = parity
    if strong is not None:
        out["strong"] = strong
    if lp is not None:
        out["lineprofile"] = lp
    if world == 1 and not args.no_callers:
        out["callers"] = run_callers(ens)
    emit(out)


DUMP_RAYS = 1 << 21  # rays kept per dumped image: 2 images x (16 MiB of float64 + 8 MiB of float32 mask)


def dump_outputs(path, images):
    """Write each image of the last timed step as float64 `path/<name>.npy`, with `path/<name>_finite.npy` (float32, 1 where
    the ray has a value): a ray that a filter drops (NaN, e.g. one that misses the disc) is stored as 0 and 0 in the mask, so
    every stored number is finite.  An image of more than DUMP_RAYS rays is cut to the same seeded sample of rays (in ray
    order) every run, so the dumps of two builds compare ray for ray."""
    os.makedirs(path, exist_ok=True)
    n = len(next(iter(images.values())))
    keep = np.arange(n) if n <= DUMP_RAYS else np.sort(np.random.default_rng(0).choice(n, DUMP_RAYS, replace=False))
    for name, img in images.items():
        img = np.asarray(img, np.float64)[keep]
        finite = np.isfinite(img)
        np.save(os.path.join(path, f"{name}.npy"), np.where(finite, img, 0.0))
        np.save(os.path.join(path, f"{name}_finite.npy"), finite.astype(np.float32))


def run_callers(ens):
    """Secondary, N = 1 only: the two callers of the path built on host orchestration + device traces (SURVEY 8 f1/f2).
    Wall clock through the public API (host buffers both ways); the device share is launch-latency bound."""
    import math

    import gradus_b200 as gb
    from gradus_b200 import corona
    from gradus_b200 import transfer_functions as tf

    m = gb.KerrMetric(1.0, 0.998)
    x = [0.0, 1e5, math.radians(30), 0.0]
    d = gb.ThinDisc(0.0, float("inf"))
    pr = gb.DeviceProber(m, x, d, chart=gb.chart_for_metric(m, 2e5, closest_approach=1.005), ensemble=ens)
    radii = np.geomspace(gb.isco(m) + 1e-2, 1000.0, 150)
    tf.cunningham_transfer_functions(m, x, d, radii[::10], prober=pr)
    out = {}
    # "exact": the reference's own iteration (every offset search from max(20, r_e), all max_iter trials at the noise floor);
    # "fast": golden-section probes warm-started, noise-floor pairs stopped after 6 trials without progress (same roots to
    # zero_atol / the same acceptance rule; fewer sequential launches)
    for mode, kw in (("transfer_functions", {}), ("transfer_functions_fast", {"warm_start": True, "stall_exit": 6})):
        pr.launches = pr.rays = 0
        t0 = time.perf_counter()
        tf.cunningham_transfer_functions(m, x, d, radii, prober=pr, **kw)
        dt = time.perf_counter() - t0
        out[mode] = {"workload": "Kerr a=0.998, observer r=1e5 at 30deg, 150 emission radii x 114 samples (N=80 + 2x17), forward-mode traces at 1e-9",
                     "seconds": dt, "radii_per_s": len(radii) / dt, "launches": pr.launches, "rays": pr.rays, "options": kw}
    # BASELINE config 4, transfer-function half: an (a, theta) table, all cells in lock step (gb200_render_batch)
    cells = [(a, th) for a in np.linspace(0.0, 0.998, 8) for th in np.linspace(10.0, 80.0, 8)]
    metrics = [gb.KerrMetric(1.0, a) for a, _ in cells]
    observers = [[0.0, 10_000.0, math.radians(th), 0.0] for _, th in cells]
    radii_of = lambda mm: 1.0 / np.linspace(1.0 / 500.0, 1.0 / (gb.isco(mm) + 1e-2), 50)[::-1]
    fast = tf.TransferFunctionSetup(warm_start=True, stall_exit=6)
    tf.transfer_function_table(metrics[:2], observers[:2], d, radii_of, ensemble=ens, setup=fast)
    t0 = time.perf_counter()
    table = tf.transfer_function_table(metrics, observers, d, radii_of, ensemble=ens, setup=fast)
    dt = time.perf_counter() - t0
    nctf = sum(len(row) for row in table)
    out["transfer_function_table"] = {"workload": "Kerr, 8 spins x 8 inclinations, observer r=1e4, 50 emission radii x 114 samples per cell, "
                                                  "every probe round of all cells in one gb200_trace_dual_batch call (warm_start, stall_exit = 6)",
                                      "seconds": dt, "transfer_functions": nctf, "transfer_functions_per_s": nctf / dt}
    disc = gb.ThinDisc(0.0, 1000.0)
    grid = [(gb.KerrMetric(1.0, a), disc, corona.LampPostModel(h=h)) for a in np.linspace(0.0, 0.998, 10) for h in np.geomspace(2.5, 50.0, 10)]
    corona.emissivity_profiles(grid[:4], n_samples=1000, ensemble=ens)
    t0 = time.perf_counter()
    corona.emissivity_profiles(grid, n_samples=1000, ensemble=ens)
    dt = time.perf_counter() - t0
    out["emissivity_profiles"] = {"workload": "lamp post, 10 spins x 10 heights, 1000 rays each, one gb200_trace_batch",
                                  "seconds": dt, "profiles_per_s": len(grid) / dt, "rays": 1000 * len(grid)}
    # the target solver (optimize_for_target through gb200_trace_target): the reference's own test target
    from gradus_b200 import api
    mt, xt, target = gb.KerrMetric(1.0, 1.0), [0.0, 1000.0, math.pi / 2, 0.0], (10.0, math.radians(40), -math.pi / 4)
    api.optimize_for_target(target, mt, xt, ensemble=ens)
    t0 = time.perf_counter()
    a_, b_, _, acc = api.optimize_for_target(target, mt, xt, ensemble=ens)
    out["target_solver"] = {"workload": "optimize_for_target, Kerr a=1, observer r=1000 at 90deg, target (10, 40deg, -45deg), d_tol=1e-2: "
                                        "33 x 33 impact parameters per launch, re-centred and shrunk until the best ray is within d_tol",
                            "seconds": time.perf_counter() - t0, "alpha": a_, "beta": b_, "closest_approach": acc}
    return out


def run_strong(args, rank, world, local, ens, dev, stream, sptr):
    """Strong scaling of the STATED configurations: the same 2048 x 2048 image (BASELINE.json configs[1]) and the same
    4096 x 4096 line-profile plane (configs[2]) split over the ranks by whole strips, strip r, r + N, ... for rank r.
      * N > 1 (torchrun): every rank times its shard (CUDA events, max over ranks); rank 0 then renders the whole
        image alone for the N = 1 time of the same box, so efficiency = t_1 / (N t_N) comes from one run.  The line-profile
        histogram of the N shards (NCCL all-reduce) is compared bin by bin with the single-GPU histogram.
      * N = 1: there is nothing to split, but rank r's shard of an N-way split is the same launch whichever GPU runs it and
        the shards never talk, so the one GPU runs shard 0 of N = 2, 4, 8 as a PREDICTION of the multi-GPU line
        ("emulated": true); the driver's SCALE run measures it for real."""
    import torch

    import gradus_b200 as gb
    from gradus_b200 import _cabi as cabi
    from gradus_b200 import distributed as gd
    from gradus_b200.api import tracing_configuration

    lib = cabi.load()
    ctx = ens.ctx(local)
    cfg, w, h = build_workload(1, ensemble=ens)
    p, ic = cfg.to_c()
    pfs = np.array([cabi.PF_REDSHIFT, cabi.PF_DISC_RADIUS], np.int32)
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)
    def time_shard(r, n):
        rng = gd.strip_interleaved_range(ic, r, n)
        imgs = [torch.empty(rng.count, dtype=torch.float64, device=dev) for _ in pfs]
        ptrs = (C.c_void_p * len(pfs))(*[C.c_void_p(t.data_ptr()) for t in imgs])
        call = lambda: cabi.check(lib.gb200_render_device(ctx, C.byref(p), C.byref(ic), C.byref(rng), cabi.iptr(pfs), len(pfs), None, ptrs, sptr, 1), ctx)
        for _ in range(2):
            call()
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for a, b in evs:
            flush.fill_(1.0)
            a.record(stream); call(); b.record(stream)
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs) / args.steps, rng.count, float(torch.nansum(imgs[0]).item())

    out = {"workload": f"the same {w}x{h} C2 image split over N GPUs (strips of 4 columns, strip r, r+N, ... on rank r)"}
    if world > 1:
        gd.barrier()
        ms_local, n_local, cs = time_shard(rank, world)
        ms = gd.max_over_ranks(ms_local, dev)
        checksum = gd.sum_over_ranks(cs, dev)
        gd.barrier()
        ms1, n1, cs1 = time_shard(0, 1) if rank == 0 else (0.0, 0, 0.0)
        gd.barrier()
        out.update({"n_gpus": world, "ms_per_step": ms, "ms_per_step_per_rank": gd.gather_floats(ms_local, dev), "rays_per_s": w * h / (ms * 1e-3),
                    "ms_single_gpu": ms1, "efficiency_vs_1": (ms1 / (world * ms)) if ms1 else None,
                    "redshift_checksum_split": checksum, "redshift_checksum_single": cs1, "emulated": False})
    else:
        ms1, n1, cs1 = time_shard(0, 1)
        pred = {}
        for n in (2, 4, 8):
            worst = max(time_shard(r, n)[0] for r in ((0, n - 1) if n > 2 else (0, 1)))
            pred[str(n)] = {"ms_per_step": worst, "rays_per_s": w * h / (worst * 1e-3), "efficiency_vs_1": ms1 / (n * worst)}
        out.update({"n_gpus": 1, "ms_per_step": ms1, "rays_per_s": w * h / (ms1 * 1e-3), "predicted": pred, "emulated": True,
                    "what_limits_it": "each rank's launch is one persistent wave: with 1/N of the rays the tail (the last, longest rays finishing "
                                      "on a draining grid) and the fixed launch + refill cost are a larger share"})
    # ---- the 4096^2 line profile split the same way; histogram of the split vs the single-GPU histogram
    m = gb.KerrMetric(1.0, 0.998)
    x = [0.0, 1000.0, math.radians(40.0), 0.0]
    plane = gb.PolarPlane(gb.GeometricGrid(), Nr=args.lp_n, Ntheta=args.lp_n, r_min=1.0, r_max=250.0)
    cfg = tracing_configuration(m, x, plane, gb.ThinDisc(0.0, 400.0), (0.0, 2000.0), callback=gb.domain_upper_hemisphere(), ensemble=ens)
    lp_p, lp_ic = cfg.to_c()
    bins = np.ascontiguousarray(np.linspace(0.1, 1.5, 180))
    emis = cabi.Emissivity(cabi.EMISSIVITY_POWERLAW, 0, 3.0, None, None)
    opts = cabi.LineProfileOpts(gb.isco(m), 50.0, 0, 0)

    def lp_shard(r, n):
        rng = gd.strip_interleaved_range(lp_ic, r, n)
        d_flux = torch.zeros(len(bins), dtype=torch.float64, device=dev)
        call = lambda: cabi.check(lib.gb200_lineprofile_device(ctx, C.byref(lp_p), C.byref(lp_ic), C.byref(rng), C.byref(emis), None, cabi.dptr(bins),
                                                               len(bins), C.byref(opts), C.c_void_p(d_flux.data_ptr()), sptr, 1), ctx)
        call()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream); call(); b.record(stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b), d_flux

    lp = {"workload": f"the same PolarPlane {args.lp_n}x{args.lp_n} line profile (C3) split over N GPUs, raw histograms all-reduced"}
    if world > 1:
        import torch.distributed as dist

        gd.barrier()
        ms_local, part = lp_shard(rank, world)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        dist.all_reduce(part, op=dist.ReduceOp.SUM)
        b.record(stream)
        torch.cuda.synchronize()
        ms = gd.max_over_ranks(ms_local, dev)
        gd.barrier()
        if rank == 0:
            ms1, single = lp_shard(0, 1)
            hs, h1 = part.cpu().numpy(), single.cpu().numpy()
            lp.update({"n_gpus": world, "ms_per_step": ms, "allreduce_ms": a.elapsed_time(b), "ms_single_gpu": ms1, "efficiency_vs_1": ms1 / (world * ms),
                       "rays_per_s": lp_ic.n / (ms * 1e-3), "L1_split_minus_single_over_peak": float(np.abs(hs - h1).sum() / h1.max()),
                       "max_bin_rel_diff": float(np.max(np.abs(hs - h1) / h1.max()))})
        gd.barrier()
    else:
        ms1, single = lp_shard(0, 1)
        h1 = single.cpu().numpy()
        hs = np.zeros_like(h1)
        worst = 0.0
        for r in range(4):  # the four shards of a 4-way split, summed in rank order like the all-reduce
            msr, part = lp_shard(r, 4)
            hs += part.cpu().numpy()
            worst = max(worst, msr)
        lp.update({"n_gpus": 1, "ms_per_step": ms1, "rays_per_s": lp_ic.n / (ms1 * 1e-3), "emulated": True,
                   "predicted": {"4": {"ms_per_step": worst, "efficiency_vs_1": ms1 / (4 * worst)}},
                   "L1_split_minus_single_over_peak": float(np.abs(hs - h1).sum() / h1.max()),
                   "max_bin_rel_diff": float(np.max(np.abs(hs - h1) / h1.max()))})
    out["lineprofile"] = lp
    return out


def run_lineprofile(args, rank, world, local, ens, dev, stream, sptr):
    """C3: lineprofile(BinningMethod) for Kerr a=0.998 theta=40deg, PolarPlane 4096 x 4096 per GPU, eps(r) = r^-3,
    histogram partial sums all-reduced with NCCL, then normalised."""
    import torch

    import gradus_b200 as gb
    from gradus_b200 import _cabi as cabi
    from gradus_b200 import distributed as gd
    from gradus_b200.api import tracing_configuration

    lib = cabi.load()
    ctx = ens.ctx(local)
    m = gb.KerrMetric(1.0, 0.998)
    x = [0.0, 1000.0, math.radians(40.0), 0.0]
    plane = gb.PolarPlane(gb.GeometricGrid(), Nr=args.lp_n, Ntheta=args.lp_n * world, r_min=1.0, r_max=250.0)
    cfg = tracing_configuration(m, x, plane, gb.ThinDisc(0.0, 400.0), (0.0, 2000.0), callback=gb.domain_upper_hemisphere(), ensemble=ens)
    p, ic = cfg.to_c()
    rng = gd.strip_interleaved_range(ic, rank, world)
    bins = np.ascontiguousarray(np.linspace(0.1, 1.5, 180))
    emis = cabi.Emissivity(cabi.EMISSIVITY_POWERLAW, 0, 3.0, None, None)
    opts = cabi.LineProfileOpts(gb.isco(m), 50.0, 0, 0)
    d_flux = torch.zeros(len(bins), dtype=torch.float64, device=dev)

    def step():
        cabi.check(lib.gb200_lineprofile_device(ctx, C.byref(p), C.byref(ic), C.byref(rng), C.byref(emis), None, cabi.dptr(bins), len(bins),
                                                C.byref(opts), C.c_void_p(d_flux.data_ptr()), sptr, 1), ctx)
        return gd.allreduce_histogram(d_flux)

    step()
    torch.cuda.synchronize()
    gd.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(args.lp_steps):
        flux = step()
    b.record(stream)
    torch.cuda.synchronize()
    gd.barrier()
    ms = gd.max_over_ranks(a.elapsed_time(b) / args.lp_steps, dev)
    total = gd.sum_over_ranks(float(rng.count), dev)
    fl = flux.cpu().numpy()
    # end to end through the blocking C-ABI call: host bins in, host flux out (this rank's shard), wall clock
    h_flux = np.zeros(len(bins))
    e2e_call = lambda: cabi.check(lib.gb200_lineprofile(ctx, C.byref(p), C.byref(ic), C.byref(rng), C.byref(emis), None, cabi.dptr(bins), len(bins),
                                                        C.byref(opts), cabi.dptr(h_flux)), ctx)
    e2e_call()
    gd.barrier()
    t0 = time.perf_counter()
    for _ in range(args.lp_steps):
        e2e_call()
    e2e_s = gd.max_over_ranks((time.perf_counter() - t0) / args.lp_steps, dev)
    return {"metric": "geodesics/sec (binned line profile, NCCL-reduced histogram)", "value": total / (ms * 1e-3), "unit": "rays/s",
            "ms_per_step": ms, "rays_per_step": total, "plane": f"PolarPlane geometric {args.lp_n}x{args.lp_n * world}", "nbins": 180,
            "histogram": "fused into the trace kernel: per-CTA shared-memory bins, exact 128-bit fixed-point sums, 0 B/ray through HBM",
            "e2e": {"value": total / e2e_s, "unit": "rays/s", "ms_per_step": e2e_s * 1e3, "h2d_bytes_per_step": 8 * len(bins) + C.sizeof(cabi.Problem),
                    "d2h_bytes_per_step": 8 * len(bins), "timing": "wall clock around the blocking gb200_lineprofile call (host bins in, host flux out)"},
            "flux_sum": float(fl.sum()), "flux_argmax_g": float(bins[int(np.argmax(fl))])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-stride", type=int, default=0, help="cpu_baseline sample: every n-th ray (0: 262144 rays)")
    ap.add_argument("--ref-stride", type=int, default=0, help="--impl reference sample per step: every n-th ray (0: 65536 rays per step at every N)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-lineprofile", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling section (the same image / plane split over the ranks)")
    ap.add_argument("--no-callers", action="store_true", help="skip the transfer-function / emissivity-profile timings")
    ap.add_argument("--lp-n", type=int, default=4096)
    ap.add_argument("--lp-steps", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the images of the last timed step (rank 0's rays, a fixed seeded "
                                                          f"sample of {DUMP_RAYS} per image) to DIR/<name>.npy as float64, "
                                                          "NaN stored as 0 with DIR/<name>_finite.npy marking the rays that have a value")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    claim_stdout()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        from gradus_b200 import distributed as gd

        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"  # keep stdout to the single JSON line (NCCL prints its version banner there)
        gd.init_from_env("nccl")
    run_ours(args, rank, world, local)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
