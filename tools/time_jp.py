#!/usr/bin/env python
"""Kernel time of the C5 (Johannsen-Psaltis), Kerr Shakura-Sunyaev and Kerr no-disc renders."""
import math, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import gradus_b200 as gb
ens = gb.EnsembleB200(devices=(0,))
cpf = gb.ConstPointFunctions
pf = [cpf.redshift() @ cpf.filter_intersected(), cpf.radius() @ cpf.filter_intersected()]
x = [0.0, 1000.0, math.radians(60), 0.0]
for name, m, d in [("JP", gb.JohannsenPsaltisMetric(1.0, 0.6, 2.0), None), ("KerrSS", gb.KerrMetric(1.0, 0.998), "ss"), ("KerrNoDisc", gb.KerrMetric(1.0, 0.998), "none")]:
    if d is None: d = gb.ThinDisc(gb.isco(m), 50.0)
    best = 1e9
    for _ in range(3):
        if d == "none": gb.rendergeodesics(m, x, 2000.0, image_width=2048, image_height=2048, ensemble=ens)
        else: gb.rendergeodesics(m, x, gb.ShakuraSunyaev(m) if d == "ss" else d, 2000.0, pf=pf, image_width=2048, image_height=2048, ensemble=ens)
        best = min(best, ens.stats().kernel_ms)
    print(f"{name:10s} kernel {best:.2f} ms")
