"""Time of the quadrature of Cunningham transfer functions: the host functions integrate_lineprofile / integrate_lagtransfer
against the device's integrate_lineprofiles / integrate_lagtransfers (gb200_tf_lineprofile / gb200_tf_lagtransfer).

Tables: synthetic, 100 radii on the inverse grid of (1.3, 50), 114 samples per radius (the size of a table a user computes
with the default numrₑ and N), split and interpolated as interpolate_branches does.  Line profile: 1000 annuli, 180 bins of
(0.1, 1.5); lag: 1000 annuli, 100 x 100 cells of (0, 1.5) x (0, 150); 7 Gauss points, g_grid_upscale 1.
  1. one model: host (one thread of the host CPU) against the device, with the largest difference relative to the peak;
  2. the device for 1000 models over 4 tables in one call (model k: table k % 4, ε = r^-(2 + k / 1000)).
Device numbers are the median over --reps calls after a warm-up: the wall time of the blocking call and the kernels'
CUDA-event time (gb200_stats.kernel_ms).  Prints the card's name and power limit with the numbers.

    python tools/time_tf_quadrature.py [--reps 5]
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

import gradus_b200 as gb  # noqa: E402
from gradus_b200 import _cabi as cabi  # noqa: E402
from gradus_b200 import api  # noqa: E402
from gradus_b200 import reverberation as rv  # noqa: E402
from gradus_b200 import tf_integration as ti  # noqa: E402
from gradus_b200 import transfer_functions as tf  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def synthetic_table(seed):
    rng = np.random.default_rng(seed)
    brs = []
    for r in ti.inverse_grid(1.3, 50.0, 100):
        th = np.sort(rng.uniform(0, 2 * math.pi, 114))
        gs = (1 - np.cos(th)) / 2
        ctf = tf.CunninghamTransferData(1.0 + 0.3 * np.sin(th), (gs - gs.min()) / (gs.max() - gs.min()), r * (1 + 0.1 * np.sin(th)),
                                        0.5 - 0.1 / r**0.5, 1.0 + 0.3 / r**0.5, r, th)
        brs.append(ti.interpolate_branches(ctf))
    return ti.InterpolatingTransferBranches(brs)


def kernel_ms():
    ens = api.default_ensemble()
    s = cabi.Stats()
    cabi.check(cabi.load().gb200_get_stats(ens.ctx(ens.devices[0]), C.byref(s)))
    return s.kernel_ms, int(s.launches)


def device(fn, reps):
    fn()
    wall, kern = [], []
    for _ in range(reps):
        t = time.perf_counter()
        out = fn()
        wall.append(1e3 * (time.perf_counter() - t))
        kern.append(kernel_ms()[0])
    return out, float(np.median(wall)), float(np.median(kern))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    print("card:", card())
    tables = [synthetic_table(s) for s in range(4)]
    g_line, g_lag, t_lag = np.linspace(0.1, 1.5, 180), np.linspace(0.0, 1.5, 100), np.linspace(0.0, 150.0, 100)
    time_of = ti.NaNLinearInterpolator(np.linspace(1.0, 60.0, 50), 0.1 * np.linspace(1.0, 60.0, 50))
    eps = gb.PowerLawEmissivity(3.0)
    prof = rv.AnalyticRadialDiscProfile(eps, time_of)
    rows = []

    t = time.perf_counter()
    host = ti.integrate_lineprofile(eps, tables[0], g_line, n_radii=1000)
    host_ms = 1e3 * (time.perf_counter() - t)
    dev, wall, kern = device(lambda: ti.integrate_lineprofiles(eps, tables[0], g_line, n_radii=1000), a.reps)
    rows.append(dict(call="lineprofile", models=1, host_ms=host_ms, device_wall_ms=wall, device_kernel_ms=kern,
                     max_diff_over_peak=float(np.abs(dev[0] - host).max() / host.max())))
    t = time.perf_counter()
    host = ti.integrate_lagtransfer(prof, tables[0], g_lag, t_lag, n_radii=1000)
    host_ms = 1e3 * (time.perf_counter() - t)
    dev, wall, kern = device(lambda: ti.integrate_lagtransfers(prof, tables[0], g_lag, t_lag, n_radii=1000), a.reps)
    rows.append(dict(call="lagtransfer", models=1, host_ms=host_ms, device_wall_ms=wall, device_kernel_ms=kern,
                     max_diff_over_peak=float(np.abs(dev[0] - host).max() / host.max()),
                     same_nonzero_cells=bool(np.array_equal(dev[0] != 0, host != 0))))

    n = 1000
    emis = [gb.PowerLawEmissivity(2.0 + k / n) for k in range(n)]
    profs = [rv.AnalyticRadialDiscProfile(e, time_of) for e in emis]
    table_of = np.arange(n) % 4
    line, wall, kern = device(lambda: ti.integrate_lineprofiles(emis, tables, g_line, table_of=table_of, n_radii=1000), a.reps)
    rows.append(dict(call="lineprofile", models=n, tables=4, device_wall_ms=wall, device_kernel_ms=kern, launches=kernel_ms()[1]))
    lag, wall, kern = device(lambda: ti.integrate_lagtransfers(profs, tables, g_lag, t_lag, table_of=table_of, n_radii=1000), a.reps)
    rows.append(dict(call="lagtransfer", models=n, tables=4, device_wall_ms=wall, device_kernel_ms=kern, launches=kernel_ms()[1]))
    # spot check of the batch against the host: model 999
    k = n - 1
    rows.append(dict(check="model 999 of the batch against the host",
                     line=float(np.abs(line[k] - ti.integrate_lineprofile(emis[k], tables[k % 4], g_line, n_radii=1000)).max() / line[k].max()),
                     lag=float(np.abs(lag[k] - ti.integrate_lagtransfer(profs[k], tables[k % 4], g_lag, t_lag, n_radii=1000)).max()
                               / lag[k].max())))
    for r in rows:
        print(json.dumps(r))


if __name__ == "__main__":
    main()
