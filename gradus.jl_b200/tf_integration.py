"""Line profiles by integrating Cunningham transfer functions (SURVEY 8 row f3): the reference's
`lineprofile(bins, ε, m, x, d, TransferFunctionMethod())` (src/line-profiles.jl:121-150).

    splitbranches, interpolate_branches       src/transfer-functions/cunningham-transfer-functions.jl:64-186
    NaNLinearInterpolator                      src/interpolations.jl:1-30
    InterpolatingTransferBranches (radial)     src/transfer-functions/transfer-functions-2d.jl:1-88
    integrate_bin / integrate_edge / quadrature, _integrate_transfer_problem!, _normalize!
                                               src/transfer-functions/integration.jl:5-19, 158-207, 322-357,
                                               src/transfer-functions/utils.jl:121-133

The transfer functions themselves (all radii in lock step) come from `transfer_functions.py`, i.e. from device traces;
the quadrature below is the reference's host-side arithmetic, vectorised over the energy bins of one annulus."""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Callable, Optional, Sequence

import numpy as np

from . import _cabi as cabi
from . import api
from . import transfer_functions as tf


class NaNLinearInterpolator:
    """interpolations.jl:1-30: piecewise linear, linear extrapolation beyond the ends, NaN knots fall back to the
    nearer finite neighbour (else `default`)."""

    def __init__(self, t, u, default=0.0):
        self.t = np.asarray(t, np.float64)
        self.u = np.asarray(u, np.float64)
        self.default = default

    def __call__(self, x):
        x = np.asarray(x, np.float64)
        n = self.t.size
        idx = np.clip(np.searchsorted(self.t, x, side="right") - 1, 0, n - 2)
        x1, x2 = self.t[idx], self.t[idx + 1]
        y1, y2 = self.u[idx], self.u[idx + 1]
        with np.errstate(invalid="ignore", divide="ignore"):
            w = (x - x1) / (x2 - x1)
            y = (1 - w) * y1 + w * y2
        bad = np.isnan(y)
        if bad.any():
            near = np.where(w < 0.5, y1, y2)
            y = np.where(bad, np.where(np.isnan(near), self.default, near), y)
        return y


@dataclass
class TransferBranches:
    """transfer-functions/types.jl `TransferBranches`: f and t on the upper / lower branch as functions of g✶."""

    upper_f: Callable
    lower_f: Callable
    upper_t: Callable
    lower_t: Callable
    gmin: float
    gmax: float
    r_e: float


def splitbranches(ctf: tf.CunninghamTransferData):
    """cunningham-transfer-functions.jl:104-154 → (lower g✶, f, t, upper g✶, f, t)."""
    gs, f, t = ctf.g_star, ctf.f, ctf.t
    imin, imax = int(np.argmin(gs)), int(np.argmax(gs))
    i1, i2 = (imin, imax) if imax > imin else (imax, imin)
    if i1 == i2:
        raise RuntimeError(f"Resolved same min/max for rₑ = {ctf.r_e}")
    n = len(f)
    b1 = slice(i1, i2 + 1)
    j2 = np.concatenate([np.arange(0, i1 + 1), np.arange(i2, n)])
    b1g, b1f, b1t = gs[b1].copy(), f[b1].copy(), t[b1].copy()
    b2g, b2f, b2t = gs[j2].copy(), f[j2].copy(), t[j2].copy()
    if b1f[1] > b1f[0]:
        return b2g, b2f, b2t, b1g, b1f, b1t
    return b1g, b1f, b1t, b2g, b2f, b2t


def _sorted_with_adjustments(g1, f1, t1, g2, f2, t2, h):
    """cunningham-transfer-functions.jl:66-102"""
    I1, I2 = np.argsort(g1, kind="stable"), np.argsort(g2, kind="stable")
    g1, f1, t1 = g1[I1], f1[I1], t1[I1]
    g2, f2, t2 = g2[I2], f2[I2], t2[I2]
    J1 = (g1 < 1 - h) & (g1 > h)
    J2 = (g2 < 1 - h) & (g2 > h)
    t_lo = (t1[0] + t2[0]) / 2
    t_hi = (t1[-1] + t2[-1]) / 2
    g1, f1, t1 = g1[J1], f1[J1], t1[J1]
    g2, f2, t2 = g2[J2], f2[J2], t2[J2]
    for tt in (t1, t2):
        tt[0], tt[-1] = t_lo, t_hi
    for gg in (g1, g2):
        gg[0], gg[-1] = 0.0, 1.0
    return g1, f1, t1, g2, f2, t2


def interpolate_branches(ctf: tf.CunninghamTransferData, h=1e-6) -> TransferBranches:
    """cunningham-transfer-functions.jl:156-186"""
    lg, lf, lt, ug, uf, ut = _sorted_with_adjustments(*splitbranches(ctf), h)
    return TransferBranches(NaNLinearInterpolator(ug, uf), NaNLinearInterpolator(lg, lf), NaNLinearInterpolator(ug, ut),
                            NaNLinearInterpolator(lg, lt), ctf.gmin, ctf.gmax, ctf.r_e)


class InterpolatingTransferBranches:
    """transfer-functions-2d.jl:1-88: branches tabulated on sorted radii, linearly blended between neighbours."""

    def __init__(self, branches: Sequence[TransferBranches]):
        order = np.argsort([b.r_e for b in branches], kind="stable")
        self.branches = [branches[i] for i in order]
        self.radii = np.array([b.r_e for b in self.branches])
        self.gmin = np.array([b.gmin for b in self.branches])
        self.gmax = np.array([b.gmax for b in self.branches])

    def inner_radius(self):
        return float(self.radii[0])

    def outer_radius(self):
        return float(self.radii[-1])

    def __call__(self, r) -> TransferBranches:
        idx = int(np.clip(np.searchsorted(self.radii, r, side="right") - 1, 0, len(self.radii) - 2))
        r1, r2 = self.radii[idx], self.radii[idx + 1]
        th = (r - r1) / (r2 - r1)
        b1, b2 = self.branches[idx], self.branches[idx + 1]

        def lazy(f1, f2):
            return lambda x: (1 - th) * f1(x) + th * f2(x)

        return TransferBranches(lazy(b1.upper_f, b2.upper_f), lazy(b1.lower_f, b2.lower_f), lazy(b1.upper_t, b2.upper_t),
                                lazy(b1.lower_t, b2.lower_t), (1 - th) * self.gmin[idx] + th * self.gmin[idx + 1],
                                (1 - th) * self.gmax[idx] + th * self.gmax[idx + 1], float(r))


def inverse_grid(lo, hi, n):
    """Grids._inverse_grid (src/image-planes/grids.jl:26-28): ascending, dense at small radii."""
    return (1.0 / np.linspace(1.0 / hi, 1.0 / lo, n))[::-1]


def transferfunctions(m, x, d, *, min_re=None, max_re=50.0, num_re=100, radii=None, h=1e-6, **kwargs):
    """`transferfunctions(m, x, d; minrₑ, maxrₑ, numrₑ, radii)` (cunningham-transfer-functions.jl:548-558):
    all radii are computed in one lock-step batch on the device."""
    if radii is None:
        if min_re is None:
            min_re = api.isco(m) + 1e-2
        radii = inverse_grid(min_re, max_re, num_re)
    ctfs = tf.cunningham_transfer_functions(m, x, d, radii, **kwargs)
    return InterpolatingTransferBranches([interpolate_branches(c, h=h) for c in ctfs])


def _gauss(n):
    return np.polynomial.legendre.leggauss(n)


def _integrate_bins(S, lo, hi, gmin, gmax, h, rule):
    """`integrate_bin` (integration.jl:167-203) for all bins [lo_j, hi_j] of one annulus at once."""
    X, W = rule
    span = gmax - gmin
    glo = np.clip(lo, gmin, gmax)
    ghi = np.clip(hi, gmin, gmax)
    lum = np.zeros_like(lo)
    live = glo != ghi
    gs_lo = (lo - gmin) / span
    gs_hi = (hi - gmin) / span

    def edge(mask, lim, lim_gs):
        gh = span * lim_gs + gmin
        with np.errstate(invalid="ignore", divide="ignore"):  # masked-out lanes may sit outside [gmin, gmax]
            return np.where(mask, S(gh) * np.abs(np.sqrt(gh) - np.sqrt(lim)) * math.sqrt(h), 0.0)

    near_lo = live & (gs_lo < h)
    only_lo = near_lo & ~(gs_hi > h)  # the whole bin lies inside the lower edge zone
    part_lo = near_lo & (gs_hi > h)
    lum += edge(part_lo, glo, np.full_like(lo, h))
    glo = np.where(part_lo, span * h + gmin, glo)
    lum = np.where(only_lo, edge(only_lo, glo, gs_hi), lum)
    live = live & ~only_lo

    near_hi = live & (gs_hi > 1 - h)
    only_hi = near_hi & ~(gs_lo < 1 - h)
    part_hi = near_hi & (gs_lo < 1 - h)
    lum += edge(part_hi, ghi, np.full_like(lo, 1 - h))
    ghi = np.where(part_hi, span * (1 - h) + gmin, ghi)
    lum = np.where(only_hi, edge(only_hi, ghi, gs_lo), lum)
    live = live & ~only_hi

    q = (ghi - glo) / 2
    u = (X[None, :] + 1) * q[:, None] + glo[:, None]
    with np.errstate(invalid="ignore", divide="ignore"):
        quad = (W[None, :] * S(u)).sum(axis=1) * q
    return lum + np.where(live, quad, 0.0)


def integrate_lineprofile(emissivity: Callable, itb: InterpolatingTransferBranches, g_grid, *, rmin=None, rmax=None,
                          g_scale=1.0, h=1e-8, n_radii=1000, g_grid_upscale=1, quadrature_points=7):
    """`integrate_lineprofile(ε, tfs, g_grid; rmin, rmax, h, n_radii, ...)` (integration.jl:233-254, 322-357)."""
    g_grid = np.asarray(g_grid, np.float64)
    rmin = itb.inner_radius() if rmin is None else rmin
    rmax = itb.outer_radius() if rmax is None else rmax
    rule = _gauss(quadrature_points)
    out = np.zeros(g_grid.size)
    radii = inverse_grid(rmin, rmax, n_radii)
    r_prev = rmin - (radii[1] - rmin)
    lo_all = g_grid[:-1] / g_scale
    hi_all = g_grid[1:] / g_scale
    for r_e in radii:
        br = itb(r_e)
        span = br.gmax - br.gmin

        def S(g, br=br, span=span):
            gs = (g - br.gmin) / span
            fu, fl = br.upper_f(gs), br.lower_f(gs)
            f = np.where(np.isnan(fu), 0.0, fu) + np.where(np.isnan(fl), 0.0, fl)
            with np.errstate(invalid="ignore", divide="ignore"):
                return g * g * f * g / np.sqrt(gs * (1 - gs))

        weight = (r_e - r_prev) * r_e * emissivity(r_e) * math.pi / span
        contrib = np.zeros(lo_all.size)
        dg = (hi_all - lo_all) / g_grid_upscale
        for i in range(g_grid_upscale):
            flo = lo_all + i * dg
            contrib += _integrate_bins(S, flo, flo + dg, br.gmin, br.gmax, h, rule)
        out[:-1] += contrib * weight
        r_prev = r_e
    # _normalize!, transfer-functions/utils.jl:121-133
    out[:-1] = out[:-1] / (g_grid[1:] + g_grid[:-1])
    total = out[:-1].sum()
    if total > 0:
        out = out / total
    return out


def lineprofile_transfer_functions(bins, emissivity: Callable, m, x, d, *, min_re=None, max_re=50.0, num_re=100, h=2e-8,
                                   n_radii=1000, **kwargs):
    """`lineprofile(bins, ε, m, u, d, ::TransferFunctionMethod; minrₑ, maxrₑ, numrₑ, h, n_radii, ...)`
    (src/line-profiles.jl:121-150).  Returns (bins, flux)."""
    bins = np.asarray(bins, np.float64)
    itb = transferfunctions(m, x, d, min_re=min_re, max_re=max_re, num_re=num_re, **kwargs)
    return bins, integrate_lineprofile(emissivity, itb, bins, h=h, n_radii=n_radii)


# --------------------------------------------------------------------------- lag (2-D) transfer functions
def _time_interpolate(t0, f1, f2, gs, h):
    """integration.jl:73-84: near the ends of the g✶ range blend the two branches' times."""
    lo, hi = gs < h, gs > 1 - h
    if not (lo.any() or hi.any()):
        return t0
    w = np.where(lo, gs / h, 1 - (1 - gs) / h)
    t1 = np.where(lo, f1(np.full_like(gs, h)), f1(np.full_like(gs, 1 - h)))
    t2 = np.where(lo, f2(np.full_like(gs, h)), f2(np.full_like(gs, 1 - h)))
    return np.where(lo | hi, t1 * w + (1 - w) * t2, t0)


def _time_gstar(br: TransferBranches, gs, h):
    tl, tu = br.lower_t(gs), br.upper_t(gs)
    return _time_interpolate(tl, br.lower_t, br.upper_t, gs, h), _time_interpolate(tu, br.upper_t, br.lower_t, gs, h)


def geometric_grid(lo, hi, n):
    """Grids._geometric_grid (src/image-planes/grids.jl:16-19)"""
    return lo * (hi / lo) ** (np.arange(n) / (n - 1))


def integrate_lagtransfer(profile, itb: InterpolatingTransferBranches, g_grid, t_grid, *, rmin=None, rmax=None, g_scale=1.0,
                          h=1e-8, n_radii=1000, g_grid_upscale=1, quadrature_points=7, t0=0.0):
    """`integrate_lagtransfer(prof, tfs, g_grid, t_grid; t0, n_radii, rmin, rmax)` (integration.jl:256-279, 359-442):
    flux[energy bin, time bin]; `profile` gives emissivity_at(r) and coordtime_at(r)."""
    g_grid = np.asarray(g_grid, np.float64)
    t_grid = np.asarray(t_grid, np.float64)
    rmin = itb.inner_radius() if rmin is None else rmin
    rmax = itb.outer_radius() if rmax is None else rmax
    rule = _gauss(quadrature_points)
    out = np.zeros((g_grid.size, t_grid.size))
    radii = geometric_grid(rmin, rmax, n_radii)
    r_prev = rmin - (radii[1] - rmin)
    nt = t_grid.size
    rows = np.arange(g_grid.size - 1)
    for r_e in radii:
        br = itb(r_e)
        span = br.gmax - br.gmin

        def branch(fn, br=br, span=span):
            def S(g):
                gs = (g - br.gmin) / span
                f = fn(gs)
                with np.errstate(invalid="ignore", divide="ignore"):
                    return g * g * np.where(np.isnan(f), 0.0, f) * g / np.sqrt(gs * (1 - gs))
            return S

        S_lower, S_upper = branch(br.lower_f), branch(br.upper_f)
        weight = (r_e - r_prev) * r_e * float(profile.emissivity_at(r_e)) * math.pi / span
        t_sd = float(profile.coordtime_at(r_e)) - t0
        glo = np.clip(g_grid[:-1] / g_scale, br.gmin, br.gmax)
        ghi = np.clip(g_grid[1:] / g_scale, br.gmin, br.gmax)
        live = glo != ghi
        dg = (ghi - glo) / g_grid_upscale
        for i in range(g_grid_upscale):
            flo = glo + i * dg
            fhi = flo + dg
            k1 = _integrate_bins(S_lower, flo, fhi, br.gmin, br.gmax, h, rule)
            k2 = _integrate_bins(S_upper, flo, fhi, br.gmin, br.gmax, h, rule)
            gs_lo = np.clip((flo - br.gmin) / span, 0, 1)
            gs_hi = np.clip((fhi - br.gmin) / span, 0, 1)
            tl1, tu1 = _time_gstar(br, gs_lo, h)
            tl2, tu2 = _time_gstar(br, gs_hi, h)
            i1 = np.searchsorted(t_grid, (tl1 + tl2) / 2 + t_sd, side="left")
            i2 = np.searchsorted(t_grid, (tu1 + tu2) / 2 + t_sd, side="left")
            ok1, ok2 = live & (i1 < nt), live & (i2 < nt)
            np.add.at(out, (rows[ok1], i1[ok1]), k1[ok1] * weight)
            np.add.at(out, (rows[ok2], i2[ok2]), k2[ok2] * weight)
        r_prev = r_e
    # _normalize! (matrix form), transfer-functions/utils.jl:135-147 — the caller receives the Σ = 1 array
    out[:-1] = out[:-1] / (g_grid[1:] + g_grid[:-1])[:, None]
    total = out[:-1].sum()
    if total > 0:
        out = out / total
    return out


# --------------------------------------------------------------------------- many models on the device
@dataclass
class PackedBranches:
    """An InterpolatingTransferBranches as the flat arrays of `gb200_tf_branches`: branch 2k is the lower, 2k+1 the upper
    branch of radius k, with knots gs[off[b]:off[b+1]] and values f, t there."""

    r_e: np.ndarray
    gmin: np.ndarray
    gmax: np.ndarray
    off: np.ndarray
    gs: np.ndarray
    f: np.ndarray
    t: np.ndarray

    def to_c(self):
        return cabi.TfBranches(len(self.r_e), 0, cabi.dptr(self.r_e), cabi.dptr(self.gmin), cabi.dptr(self.gmax),
                               self.off.ctypes.data_as(C.POINTER(C.c_int64)), cabi.dptr(self.gs), cabi.dptr(self.f), cabi.dptr(self.t))


def pack_branches(itb: InterpolatingTransferBranches) -> PackedBranches:
    """Flatten `itb` for the device.  Every branch must be a `NaNLinearInterpolator` with the default fallback 0 (what
    `interpolate_branches` makes), and f and t of a branch must share their knots."""
    gs, f, t, off = [], [], [], [0]
    for br in itb.branches:
        for fb, tb in ((br.lower_f, br.lower_t), (br.upper_f, br.upper_t)):
            for fn in (fb, tb):
                if not isinstance(fn, NaNLinearInterpolator) or fn.default != 0.0:
                    raise TypeError("only NaNLinearInterpolator branches with default 0 can be integrated on the device: "
                                    "use integrate_lineprofile / integrate_lagtransfer")
            if not np.array_equal(fb.t, tb.t):
                raise ValueError(f"the f and t branches at r_e = {br.r_e} do not share their knots")
            gs.append(fb.t)
            f.append(fb.u)
            t.append(tb.u)
            off.append(off[-1] + fb.t.size)
    cat = lambda parts: np.ascontiguousarray(np.concatenate(parts), np.float64)  # noqa: E731
    return PackedBranches(np.ascontiguousarray(itb.radii, np.float64), np.ascontiguousarray(itb.gmin, np.float64),
                          np.ascontiguousarray(itb.gmax, np.float64), np.array(off, np.int64), cat(gs), cat(f), cat(t))


def _per_model(values: dict):
    """Broadcast the per-model arguments (a scalar, or a sequence of one or of n values) to one list per argument."""
    lists = {k: list(v) if isinstance(v, (list, tuple, np.ndarray)) else [v] for k, v in values.items()}
    n = max(len(v) for v in lists.values())
    for k, v in lists.items():
        if len(v) not in (1, n):
            raise ValueError(f"{k}: {len(v)} values for {n} models")
    return n, {k: v * n if len(v) == 1 else v for k, v in lists.items()}


def _ascending(name, a):
    a = np.ascontiguousarray(a, np.float64)
    if a.ndim != 1 or a.size < 1 or not np.all(np.isfinite(a)) or not np.all(np.diff(a) > 0):
        raise ValueError(f"{name} must be a finite, strictly ascending 1-D grid")
    return a


def _device_quadrature(lag, profiles, itbs, g_grid, t_grid, *, table_of, rmin, rmax, g_scale, h, n_radii, g_grid_upscale,
                       quadrature_points, t0, ensemble):
    from .reverberation import _disc_profile_to_c, _emissivity_to_c

    itbs = [itbs] if isinstance(itbs, InterpolatingTransferBranches) else list(itbs)
    packed = [pack_branches(itb) for itb in itbs]
    if isinstance(profiles, (list, tuple)) and len(profiles) == 0:
        raise ValueError("no emission models")
    n, per = _per_model({"profiles": profiles if isinstance(profiles, (list, tuple)) else [profiles],
                         "table_of": list(range(len(itbs))) if table_of is None else table_of,
                         "rmin": rmin, "rmax": rmax, "g_scale": g_scale, "n_radii": n_radii})
    host = "integrate_lagtransfer" if lag else "integrate_lineprofile"
    g_grid = _ascending("g_grid", g_grid)
    if g_grid.size < 2:
        raise ValueError("g_grid needs at least two edges")
    if lag:
        t_grid = _ascending("t_grid", t_grid)
    if not 1 <= int(quadrature_points) <= 32:
        raise ValueError(f"quadrature_points must be in 1..32 (got {quadrature_points})")
    if int(g_grid_upscale) < 1:
        raise ValueError(f"g_grid_upscale must be >= 1 (got {g_grid_upscale})")
    if not 0 < h < 0.5:
        raise ValueError(f"h must lie in (0, 0.5) (got {h})")
    models, keep = (cabi.TfModel * n)(), []
    for k in range(n):
        tab = per["table_of"][k]
        if int(tab) != tab or not 0 <= tab < len(itbs):
            raise ValueError(f"model {k}: table index {tab} out of range for {len(itbs)} tables")
        nr = per["n_radii"][k]
        if int(nr) != nr or nr < 2:
            raise ValueError(f"model {k}: n_radii must be an integer >= 2 (got {nr})")
        itb = itbs[int(tab)]
        lo = itb.inner_radius() if per["rmin"][k] is None else float(per["rmin"][k])
        hi = itb.outer_radius() if per["rmax"][k] is None else float(per["rmax"][k])
        if not lo < hi:
            raise ValueError(f"model {k}: need rmin < rmax (got {lo}, {hi})")
        radii = np.ascontiguousarray((geometric_grid if lag else inverse_grid)(lo, hi, int(nr)), np.float64)
        if lag:
            prof, pk = _disc_profile_to_c(per["profiles"][k], host)
        else:
            prof, pk = cabi.DiscProfile(), []
            _emissivity_to_c(per["profiles"][k], prof, pk, host)
        keep += [radii, pk]
        models[k] = cabi.TfModel(int(tab), int(nr), cabi.dptr(radii), lo, float(per["g_scale"][k]), prof)
    X, W = (np.ascontiguousarray(a, np.float64) for a in _gauss(int(quadrature_points)))
    opts = cabi.TfQuadOpts(float(h), float(t0), int(g_grid_upscale), int(quadrature_points), cabi.dptr(X), cabi.dptr(W), 1, 0)
    tables = (cabi.TfBranches * len(packed))(*[p.to_c() for p in packed])
    ens = ensemble if ensemble is not None else api.default_ensemble()
    ctx = ens.ctx(ens.devices[0])
    lib = cabi.load()
    if lag:
        out = np.zeros((n, g_grid.size, t_grid.size))
        cabi.check(lib.gb200_tf_lagtransfer(ctx, len(packed), tables, n, models, cabi.dptr(g_grid), g_grid.size, cabi.dptr(t_grid),
                                            t_grid.size, C.byref(opts), cabi.dptr(out.reshape(-1))), ctx)
    else:
        out = np.zeros((n, g_grid.size))
        cabi.check(lib.gb200_tf_lineprofile(ctx, len(packed), tables, n, models, cabi.dptr(g_grid), g_grid.size, C.byref(opts),
                                            cabi.dptr(out.reshape(-1))), ctx)
    return out


def integrate_lineprofiles(emissivities, itbs, g_grid, *, table_of=None, rmin=None, rmax=None, g_scale=1.0, h=1e-8,
                           n_radii=1000, g_grid_upscale=1, quadrature_points=7, ensemble=None):
    """`integrate_lineprofile` for many emission models in one device call (`gb200_tf_lineprofile`): row k of the returned
    (nmodels, len(g_grid)) array is `integrate_lineprofile(emissivities[k], itbs[table_of[k]], g_grid, rmin=rmin[k], ...)`.
    `emissivities`, `table_of` (default: model k uses table k), `rmin`, `rmax`, `g_scale` and `n_radii` are per model and
    broadcast; an emissivity is a `PowerLawEmissivity` or a `TabulatedEmissivity`."""
    return _device_quadrature(False, emissivities, itbs, g_grid, None, table_of=table_of, rmin=rmin, rmax=rmax, g_scale=g_scale,
                              h=h, n_radii=n_radii, g_grid_upscale=g_grid_upscale, quadrature_points=quadrature_points, t0=0.0,
                              ensemble=ensemble)


def integrate_lagtransfers(profiles, itbs, g_grid, t_grid, *, t0=0.0, table_of=None, rmin=None, rmax=None, g_scale=1.0, h=1e-8,
                           n_radii=1000, g_grid_upscale=1, quadrature_points=7, ensemble=None):
    """`integrate_lagtransfer` for many emission models in one device call (`gb200_tf_lagtransfer`): returns an
    (nmodels, len(g_grid), len(t_grid)) array.  Profiles are `AnalyticRadialDiscProfile`s with a `PowerLawEmissivity` or
    `TabulatedEmissivity` ε, or `RadialDiscProfile`s; per-model arguments broadcast as in `integrate_lineprofiles`."""
    return _device_quadrature(True, profiles, itbs, g_grid, t_grid, table_of=table_of, rmin=rmin, rmax=rmax, g_scale=g_scale, h=h,
                              n_radii=n_radii, g_grid_upscale=g_grid_upscale, quadrature_points=quadrature_points, t0=t0,
                              ensemble=ensemble)
