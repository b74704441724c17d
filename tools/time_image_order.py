"""What the equatorial-crossing counter and the photon-ring image orders cost on one B200.

Variants, alternated within each round and repeated over several rounds (other work shares the host):
  c2          BASELINE configs[1] (2048 x 2048, Kerr a = 0.998, 60 deg, ThinDisc(0, 50)): redshift + radius, as bench.py
  c2+count    the same plus equatorial_crossings (the counting instantiation of the kernel)
  order0..2   ImageOrder(ThinDisc(0, 50), n), redshift + radius
  lp_order0/1 BASELINE configs[2]'s line profile (4096 x 4096 polar plane, a = 0.998, 40 deg, ThinDisc(0, 400), r^-3)
              with ImageOrder(., n), fused histogram.  Without configs[2]'s hemisphere callback: r cos(theta) < delta ends
              every ray at its first equatorial crossing, so no order >= 1 image survives it
  lp          the same line profile on the plain disc (also without the callback), for reference
Device-resident outputs, CUDA events around each call on the call's own stream, a 256 MiB L2 flush before each call (as
bench.py).  Prints the card's name and power limit with the numbers.

    python tools/time_image_order.py [--rounds 5] [--reps 3] [--warmup 2]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import gradus_b200 as gb  # noqa: E402
from gradus_b200 import _cabi as cabi  # noqa: E402

import common  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3, help="timed calls per variant per round")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--size", type=int, default=2048, help="image side of the render variants")
    ap.add_argument("--lp-size", type=int, default=4096, help="plane side of the line-profile variants")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    ens = gb.EnsembleB200(devices=(0,))
    lib = cabi.load()
    ctx = ens.ctx(0)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sptr = C.c_void_p(stream.cuda_stream)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    m, x, d, _ = common.c1(8, 8)
    n = args.size * args.size
    imgs = [torch.empty(n, dtype=torch.float64, device=dev) for _ in range(3)]
    ptrs = (C.c_void_p * 3)(*[C.c_void_p(t.data_ptr()) for t in imgs])

    def render(geometry, kinds):
        cfg = common.render_config(m, x, geometry, 2000.0, args.size, args.size, ensemble=ens)
        p, ic = cfg.to_c()
        rng = cabi.Range(0, ic.n, 1)
        pfs = np.array(kinds, np.int32)

        def call():
            cabi.check(lib.gb200_render_device(ctx, C.byref(p), C.byref(ic), C.byref(rng), cabi.iptr(pfs), len(pfs), None, ptrs, sptr, 1), ctx)

        def checksum():
            return [float(torch.nansum(imgs[k]).item()) for k in range(len(pfs))]
        return call, checksum, (p, ic, pfs)

    lm, lx, ld, lplane, _ = common.c3(8, 8)
    bins = np.linspace(0.1, 1.5, 180)
    flux = torch.zeros(len(bins), dtype=torch.float64, device=dev)
    emis = cabi.Emissivity(cabi.EMISSIVITY_POWERLAW, 0, 3.0, None, None)
    opts = cabi.LineProfileOpts(gb.isco(lm), 50.0, 0, 0)

    def lineprofile(geometry):
        plane = gb.PolarPlane(gb.GeometricGrid(), Nr=args.lp_size, Ntheta=args.lp_size, r_min=1.0, r_max=250.0)
        cfg = gb.tracing_configuration(lm, lx, plane, geometry, (0.0, 2000.0), ensemble=ens)
        p, ic = cfg.to_c()
        rng = cabi.Range(0, ic.n, 1)

        def call():
            cabi.check(lib.gb200_lineprofile_device(ctx, C.byref(p), C.byref(ic), C.byref(rng), C.byref(emis), None, cabi.dptr(bins),
                                                    len(bins), C.byref(opts), C.c_void_p(flux.data_ptr()), sptr, 1), ctx)

        def checksum():
            return [float(flux.sum().item())]
        return call, checksum, (p, ic, None)

    R, Z = cabi.PF_REDSHIFT, cabi.PF_DISC_RADIUS
    variants = {
        "c2": render(d, [R, Z]),
        "c2+count": render(d, [R, Z, cabi.PF_EQUATORIAL_CROSSINGS]),
        "order0": render(gb.ImageOrder(d, 0), [R, Z]),
        "order1": render(gb.ImageOrder(d, 1), [R, Z]),
        "order2": render(gb.ImageOrder(d, 2), [R, Z]),
        "lp": lineprofile(ld),
        "lp_order0": lineprofile(gb.ImageOrder(ld, 0)),
        "lp_order1": lineprofile(gb.ImageOrder(ld, 1)),
    }
    info = {"card": card(), "torch": torch.__version__, "size": args.size, "lp_size": args.lp_size, "rounds": args.rounds,
            "reps": args.reps, "l2": "256 MiB write before every timed call, outside the event pair"}
    print("# " + json.dumps(info), flush=True)
    extra = {}
    for name, (call, checksum, _) in variants.items():  # warm-up; checksums and hit counts of the last call
        for _ in range(args.warmup):
            call()
        torch.cuda.synchronize()
        extra[name] = {"checksum": checksum()}
        if not name.startswith("lp"):
            extra[name]["hits"] = int((~torch.isnan(imgs[1])).sum().item())
    times = {k: [] for k in variants}
    for rnd in range(args.rounds):
        order = list(variants) if rnd % 2 == 0 else list(reversed(variants))
        for name in order:
            call = variants[name][0]
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.reps)]
            for a, b in evs:
                flush.fill_(1.0)
                a.record(stream)
                call()
                b.record(stream)
            torch.cuda.synchronize()
            times[name] += [a.elapsed_time(b) for a, b in evs]
    base = float(np.median(times["c2"]))
    lp_base = float(np.median(times["lp"]))
    for name, ts in times.items():
        med = float(np.median(ts))
        ref = lp_base if name.startswith("lp") else base
        row = {"variant": name, "median_ms": round(med, 3), "min_ms": round(float(np.min(ts)), 3), "max_ms": round(float(np.max(ts)), 3),
               "vs_ref": round(med / ref, 4), "n": len(ts)}
        row.update(extra[name])
        print(json.dumps(row), flush=True)
    print("# " + json.dumps({"card_after": card()}), flush=True)
    ens.close()


if __name__ == "__main__":
    main()
