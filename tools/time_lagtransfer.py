"""Wall time of the binned lag-energy transfer function: the host composition binflux(lagtransfer(...)) against
binned_lagtransfer(...), which bins on the device.

Configuration: Kerr a = 0.998, theta_obs = 30 deg, ThinDisc(isco, 500), lamp post at h = 10 (10 000 coronal rays),
300 x 300 bins, GeometricGrid PolarPlane(r_max = 50) of 800^2 (lagtransfer's default) and 2048^2 rays.  Both routes
trace the corona too.  Per route: median wall time of the blocking call (after warm-up) and the trace kernel's CUDA-event
time (gb200_stats.kernel_ms, the largest over the devices; the multi-device composition, gb200_comm_render, does not time
its kernels), so the non-trace part of each route is visible.  Repeated over 1, 2 and up to 8 devices where present.
Prints the card's name and power limit with the numbers.

    python tools/time_lagtransfer.py [--reps 10] [--warmup 2] [--sizes 800 2048]
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import gradus_b200 as gb  # noqa: E402
from gradus_b200 import _cabi as cabi  # noqa: E402
from gradus_b200 import corona  # noqa: E402
from gradus_b200 import reverberation as rv  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def trace_ms(ens):
    lib = cabi.load()
    comm = ens.comm()
    ctxs = [C.c_void_p(lib.gb200_comm_context(comm, i)) for i in range(len(ens.devices))] if comm is not None else [ens.ctx(ens.devices[0])]
    out = []
    for ctx in ctxs:
        s = cabi.Stats()
        cabi.check(lib.gb200_get_stats(ctx, C.byref(s)))
        out.append(s.kernel_ms)
    return max(out)


def timed(fn, ens, reps, warmup):
    for _ in range(warmup):
        fn()
    wall, kern = [], []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        wall.append(1e3 * (time.perf_counter() - t))
        kern.append(trace_ms(ens))
    return float(np.median(wall)), float(np.median(kern))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--sizes", type=int, nargs="+", default=[800, 2048])
    args = ap.parse_args()
    print("device:", card(), flush=True)
    m = gb.KerrMetric(1.0, 0.998)
    x = [0.0, 1e6, math.radians(30), 0.0]
    d, model = gb.ThinDisc(gb.isco(m), 500.0), corona.LampPostModel(h=10.0)
    ndev_all = torch.cuda.device_count()
    for ndev in [k for k in (1, 2, 8) if k <= ndev_all] or [1]:
        ens = gb.EnsembleB200(tuple(range(ndev)))
        for size in args.sizes:
            plane = gb.PolarPlane(gb.GeometricGrid(), Nr=size, Ntheta=size, r_max=50.0)
            kw = dict(plane=plane, ensemble=ens)
            comp = lambda: rv.binflux(rv.lagtransfer(m, x, d, model, **kw), N_E=300, N_t=300)  # noqa: E731
            dev = lambda: rv.binned_lagtransfer(m, x, d, model, N_E=300, N_t=300, **kw)  # noqa: E731
            c_wall, c_kern = timed(comp, ens, args.reps, args.warmup)
            d_wall, d_kern = timed(dev, ens, args.reps, args.warmup)
            print(json.dumps(dict(devices=ndev, plane=f"{size}^2", bins="300x300", reps=args.reps,
                                  composition_wall_ms=round(c_wall, 2), composition_trace_ms=round(c_kern, 2) if ndev == 1 else None,
                                  device_wall_ms=round(d_wall, 2), device_trace_ms=round(d_kern, 2),
                                  speedup=round(c_wall / d_wall, 2))), flush=True)
        ens.close()


if __name__ == "__main__":
    main()
