"""Coronal illumination of the disc (SURVEY 8 row f1): arbitrary-initial-condition ensembles traced on the device,
post-processing on the host exactly where the reference has it.

    LampPostModel, BeamedPointSource       src/corona/models/lamp-post.jl:1-44
    samplers, sky_angles_to_velocity       src/corona/samplers.jl:1-97
    sample_position_direction_velocity     src/corona/corona-models.jl:1-33
    tracecorona                            src/corona/corona-models.jl:164-190
    emissivity_profile (point source)      src/corona/models/lamp-post.jl:77-164
    emissivity_profile (sampled sky)       src/corona/emissivity.jl:139-168, src/corona/radial.jl:41-132
    energy_ratio, lorentz_factor           src/corona/flux-calculations.jl:32-36, 98-113

Every geodesic is an explicit-IC endpoint trace through `gb200_trace`; many (metric, source) models can be fused into
one launch with `emissivity_profiles` (a 1000-ray launch is far too small for a B200)."""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _cabi as cabi
from . import api, hostmath


# --------------------------------------------------------------------------- models, spectra, samplers
@dataclass(frozen=True)
class LampPostModel:
    h: float = 5.0
    theta: float = 0.01
    phi: float = 0.0


@dataclass(frozen=True)
class BeamedPointSource:
    r: float
    beta: float


@dataclass(frozen=True)
class RingCorona:
    """`RingCorona(vf, r, h)` (src/corona/models/extended.jl:56-80): a ring of radius r at height h above the disc; `vf` is
    one of `SourceVelocities` ("co_rotating", "stationary").  Position and four-velocity of the source point are built here;
    sky-sampled ray fans (`tracecorona`) run on the device like any other explicit-IC ensemble.  The reference's
    time-dependent ring emissivity (its longitudinal-arm sampling, ring.jl) is not built."""

    r: float = 5.0
    h: float = 5.0
    vf: str = "co_rotating"


@dataclass(frozen=True)
class PowerLawSpectrum:
    """`coronal_spectrum(spec, g) = g^-Γ`, src/corona/spectra.jl:11-25"""

    gamma: float = 2.0

    def __call__(self, g):
        return np.asarray(g) ** (-self.gamma)


def sample_position_velocity(m, model):
    """Source position and four-velocity (lamp-post.jl:8-13, 36-42)."""
    if isinstance(model, LampPostModel):
        x = np.array([0.0, model.h, model.theta, model.phi])
        g = hostmath.metric_components(m, x[1], x[2])
        return x, np.array([1.0 / math.sqrt(-g[0]), 0.0, 0.0, 0.0])
    if isinstance(model, BeamedPointSource):
        x = np.array([0.0, model.r, 1e-4, 0.0])
        g = hostmath.metric_components(m, x[1], x[2])
        drdt = model.beta * math.sqrt(-g[0] / g[1])
        # constrain_normalize(m, x, (1, drdt, 0, 0); μ = 1): scale to g(v, v) = −1
        v = np.array([1.0, drdt, 0.0, 0.0])
        return x, v / math.sqrt(-hostmath.dot(g, v, v))
    if isinstance(model, RingCorona):
        x = np.array([0.0, math.hypot(model.r, model.h), math.atan2(model.r, model.h), 0.0])
        g = hostmath.metric_components(m, x[1], x[2])
        if model.vf == "stationary":  # SourceVelocities.stationary (extended.jl:27-41)
            return x, np.array([1.0 / math.sqrt(-g[0]), 0.0, 0.0, 0.0])
        if model.vf != "co_rotating":
            raise ValueError("RingCorona.vf must be 'co_rotating' or 'stationary'")
        # SourceVelocities.co_rotating (extended.jl:13-25): the Keplerian four-velocity of the disc below, scaled by sin θ,
        # normalised at x, then constrain_all for a unit-mass particle
        s = math.sin(x[2])
        v = np.asarray(hostmath.circular_fourvelocity(m, max(api.isco(m), x[1] * s)), np.float64) * s
        v = v / math.sqrt(abs(hostmath.dot(g, v, v)))
        disc = -g[0] * g[1] * v[1] ** 2 - g[0] * g[2] * v[2] ** 2 - g[0] - (g[0] * g[3] - g[4] ** 2) * v[3] ** 2
        v[0] = -(g[4] * v[3] + math.sqrt(disc)) / g[0]
        return x, v
    raise ValueError(f"corona model {type(model).__name__} has no position/velocity sampler here")


def _radial_angles(generator, n_samples):
    idx = np.arange(1, n_samples + 1, dtype=np.float64)
    if generator == "golden":
        return idx, math.pi * (1 + math.sqrt(5.0)) * idx
    if generator == "even":
        return idx / n_samples, 2 * math.pi * (idx / n_samples)
    raise ValueError("generator must be 'golden' or 'even'")


@dataclass(frozen=True)
class EvenSampler:
    """`EvenSampler(domain, generator)` (samplers.jl:8-16): domain "lower" | "both", generator "golden" | "even".
    (The reference's RandomGenerator draws from Julia's RNG and has no reproducible counterpart.)"""

    domain: str = "lower"
    generator: str = "golden"

    def angles(self, n_samples):
        i, radial = _radial_angles(self.generator, n_samples)
        u = i / n_samples
        if self.domain == "both":
            elev = np.arccos(np.clip(1 - 2 * u, -1.0, 1.0))
        elif self.domain == "lower":
            elev = np.arccos(np.clip(1 - u, -1.0, 1.0))
        else:
            raise ValueError("domain must be 'lower' or 'both'")
        return elev, np.mod(radial, 2 * math.pi)


@dataclass(frozen=True)
class WeierstrassSampler:
    """`WeierstrassSampler(res, domain, generator)` (samplers.jl:17-28, 42-54): elevations 2 atan(√(res / i)) -- the inverse
    stereographic projection of a spiral in the plane --, alternating between the hemispheres for domain "both"."""

    res: float = 100.0
    domain: str = "lower"
    generator: str = "golden"

    def angles(self, n_samples):
        i, radial = _radial_angles(self.generator, n_samples)
        elev = 2.0 * np.arctan(np.sqrt(self.res / i))
        if self.domain == "both":
            # `iseven(i)` of the generator's index: the ray counter for the golden spiral, i / N (never an even integer) otherwise
            even = (np.arange(1, n_samples + 1) % 2 == 0) if self.generator == "golden" else np.zeros(n_samples, bool)
            elev = np.where(even, elev, math.pi - elev)
        elif self.domain != "lower":
            raise ValueError("domain must be 'lower' or 'both'")
        return elev, np.mod(radial, 2 * math.pi)


def sky_angles_to_velocity(m, x, v_source, theta, phi, E0=1.0):
    """Local sky direction (θ, φ) of a source at x moving with v_source → coordinate velocity (samplers.jl:79-97).
    θ, φ may be arrays; returns (4, n)."""
    theta = np.atleast_1d(np.asarray(theta, np.float64))
    phi = np.broadcast_to(np.asarray(phi, np.float64), theta.shape)
    hat = -np.stack([np.sin(theta) * np.cos(phi), np.sin(theta) * np.sin(phi), np.cos(theta)])
    th, ph = x[2], x[3]
    J = np.array([[math.sin(th) * math.cos(ph), math.sin(th) * math.sin(ph), math.cos(th)],
                  [math.cos(th) * math.cos(ph), math.cos(th) * math.sin(ph), -math.sin(th)],
                  [-math.sin(ph), math.cos(ph), 0.0]])
    k = J @ hat
    p = np.vstack([np.full((1, theta.size), E0), E0 * k])
    return hostmath.tetradframe_matrix(m, x, v_source) @ p


# --------------------------------------------------------------------------- disc-side quantities
class _KeplerianProjector:
    """`_keplerian_velocity_projector` (circular-orbits.jl:155-170): circular outside the ISCO, plunging inside."""

    def __init__(self, m, ensemble=None):
        self.m = m
        self.r_isco = api.isco(m)
        self.ensemble = ensemble
        self._table = None

    def __call__(self, rho):
        rho = np.atleast_1d(np.asarray(rho, np.float64))
        v = hostmath.circular_fourvelocity(self.m, np.maximum(rho, self.r_isco))
        inside = rho < self.r_isco
        if inside.any():
            if self._table is None:
                self._table = api.interpolate_plunging_velocities(self.m, self.ensemble)
            ut, ur, uph = self._table(rho[inside])
            v[0, inside], v[1, inside], v[3, inside] = ut, -ur, uph
        return v


def energy_ratio(m, x_init, v_init, x, v, v_src, v_disc):
    """e_src / e_disc (flux-calculations.jl:100-113); all vectors (4, n) or (4,)."""
    gs = hostmath.metric_components(m, x_init[1], x_init[2])
    gd = hostmath.metric_components(m, x[1], x[2])
    return hostmath.dot(gs, v_init, v_src) / hostmath.dot(gd, v, v_disc)


@dataclass
class RadialDiscProfile:
    """src/corona/radial.jl:1-37: radii, emissivity and coordinate arrival time with linear interpolation."""

    radii: np.ndarray
    eps: np.ndarray
    t: np.ndarray

    def emissivity_at(self, r):
        return np.interp(np.clip(r, self.radii[0], self.radii[-1]), self.radii, self.eps)

    def coordtime_at(self, r):
        return np.interp(np.clip(r, self.radii[0], self.radii[-1]), self.radii, self.t)

    def as_tabulated_emissivity(self):
        """For `lineprofile(bins, ε, ...)`: the profile as a device-side emissivity table."""
        return api.TabulatedEmissivity(self.radii, self.eps)


@dataclass
class CoronaGeodesics:
    """corona-models.jl:155-162 (only intersecting rays are kept)."""

    metric: object
    geometry: object
    model: object
    geodesic_points: dict  # x_init, v_init, x, v each (4, n)
    source_velocity: np.ndarray  # (4, n)


# --------------------------------------------------------------------------- tracing
def _device_solver(configs):
    """The product tracer: one `gb200_trace` for a single ensemble, `gb200_trace_batch` (one stream per ensemble,
    one host synchronisation) for several."""
    if len(configs) == 1:
        return [api.solve_tracing_problem(configs[0])]
    return api.tracegeodesics_batch(configs)


def _trace_many(jobs, ensemble=None, solver=None):
    """jobs: list of (m, xs(4,n), vs(4,n), d, lam_max, kwargs) → list of GeodesicPoints, one fused launch.
    `solver` maps a list of TracingConfigurations to a list of GeodesicPoints (tests inject the oracle here)."""
    configs = [api.tracing_configuration(m, xs.T, vs.T, d, lam, ensemble=ensemble, **kw) for (m, xs, vs, d, lam, kw) in jobs]
    return (solver or _device_solver)(configs)


def _intersected(gps):
    return np.asarray(gps.status) == cabi.STATUS_INTERSECTED


def tracecorona(m, d, model, *, lambda_max=10_000.0, n_samples=1024, sampler=None, callback="default", ensemble=None,
                solver=None, **kwargs) -> CoronaGeodesics:
    """`tracecorona(m, g, model; λmax, n_samples, sampler, callback)` (corona-models.jl:164-190)."""
    if isinstance(d, api.ImageOrder):
        raise ValueError("geometry ImageOrder is outside the corona models' scope: they trace to the whole disc")
    if sampler is None:
        sampler = EvenSampler("both", "golden")
    if callback == "default":
        callback = api.domain_upper_hemisphere()
    x, v_src = sample_position_velocity(m, model)
    r_min = api.inner_radius(m)
    if x[1] < 1.9 * r_min:
        raise ValueError("source position is inside 1.9 r_inner (corona-models.jl:13-15 would resample forever)")
    x = x.copy()
    x[2] = min(max(x[2], 1e-3), math.pi - 1e-3)  # corona-models.jl:18-24
    elev, azim = sampler.angles(n_samples)
    vs = sky_angles_to_velocity(m, x, v_src, elev, azim)
    xs = np.repeat(x[:, None], n_samples, axis=1)
    gps = _trace_many([(m, xs, vs, d, lambda_max, dict(callback=callback, **kwargs))], ensemble, solver)[0]
    I = _intersected(gps)
    pts = dict(x_init=gps.x_init[:, I], v_init=gps.v_init[:, I], x=gps.x[:, I], v=gps.v[:, I])
    return CoronaGeodesics(m, d, model, pts, np.repeat(v_src[:, None], int(I.sum()), axis=1))


# --------------------------------------------------------------------------- emissivity profiles
def _point_source_emissivity(m, spec, v_src, r, deltas, pts, disc_velocity):
    """lamp-post.jl:117-152: ε_i = w_i |sin δ_i| g_i^-Γ / (A_i γ_i) on the sorted intersection radii."""
    n = len(r)
    v_disc = disc_velocity(r)
    gs = energy_ratio(m, pts["x_init"], pts["v_init"], pts["x"], pts["v"], v_src[:, None], v_disc)
    gam = hostmath.lorentz_factor(m, pts["x"][1], pts["x"][2], v_disc)
    i = np.arange(n)
    i2 = np.where(i == 0, 1, np.where(i != n - 1, i + 1, i - 1))
    i4 = np.where(i == 0, 1, i - 1)
    dr = (np.abs(r[i] - r[i2]) + np.abs(r[i] - r[i4])) / 2
    w = (np.abs(deltas[i] - deltas[i2]) + np.abs(deltas[i] - deltas[i4])) / 4
    A = hostmath.proper_area(m, pts["x"][1], pts["x"][2]) * dr
    eps = w * np.abs(np.sin(deltas)) * spec(gs) / (A * gam)
    return eps, gs


def _point_source_postprocess(m, spec, v_src, deltas, gps, ensemble):
    I = _intersected(gps)
    pts = dict(x_init=gps.x_init[:, I], v_init=gps.v_init[:, I], x=gps.x[:, I], v=gps.v[:, I])
    deltas = deltas[I]
    rs = pts["x"][1] * np.sin(pts["x"][2])
    J = np.argsort(rs, kind="stable")
    rs, deltas = rs[J], deltas[J]
    pts = {k: a[:, J] for k, a in pts.items()}
    if len(rs) < 2:
        raise RuntimeError("fewer than two rays of the point source reached the disc")
    eps, _ = _point_source_emissivity(m, spec, v_src, rs, deltas, pts, _KeplerianProjector(m, ensemble))
    return RadialDiscProfile(rs, eps, pts["x"][0].copy())


def _point_source_job(m, d, model, delta_min, delta_max, n_samples, lambda_max, callback, kwargs):
    deltas = np.deg2rad(np.linspace(delta_min, delta_max, n_samples))
    x, v_src = sample_position_velocity(m, model)
    vs = sky_angles_to_velocity(m, x, v_src, deltas, 0.0)  # polar_angle_to_velfunc, emissivity.jl:177-181
    xs = np.repeat(x[:, None], n_samples, axis=1)
    return deltas, v_src, (m, xs, vs, d, lambda_max, dict(callback=callback, **kwargs))


def _build_radial_profile(m, spec, radii, times, v_src, pts, N, ensemble, grid="geometric"):
    """radial.jl:41-100: bin the sorted intersection radii, mean energy ratio per bin, photon count → emissivity."""
    disc_velocity = _KeplerianProjector(m, ensemble)
    lo, hi = radii[0], radii[-1]
    if grid == "geometric":
        bins = lo * (hi / lo) ** (np.arange(N) / (N - 1))
    elif grid == "linear":
        bins = np.linspace(lo, hi, N)
    else:
        raise ValueError("grid must be 'geometric' or 'linear'")
    idx = np.clip(np.searchsorted(bins, radii, side="right") - 1, 0, N - 1)  # Buckets.Simple: last edge ≤ value, clamped
    g_each = energy_ratio(m, pts["x_init"], pts["v_init"], pts["x"], pts["v"], v_src, disc_velocity(radii))
    counts = np.bincount(idx, minlength=N).astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        g_mean = np.bincount(idx, weights=g_each, minlength=N) / counts
        t_mean = np.bincount(idx, weights=times, minlength=N) / counts
    inner = np.concatenate([[0.0], bins[:-1]])
    A = (bins - inner) * hostmath.proper_area(m, bins, math.pi / 2)
    gam = hostmath.lorentz_factor(m, bins, math.pi / 2, disc_velocity(bins))
    eps = counts * spec(g_mean) / (A * gam)  # source_to_disc_emissivity, emissivity.jl:62-78
    return bins, t_mean, eps


def radial_disc_profile(cg: CoronaGeodesics, spectrum=PowerLawSpectrum(2.0), *, N=100, grid="geometric", ensemble=None):
    """`RadialDiscProfile(cg::CoronaGeodesics, spec; grid, N)` (radial.jl:136-147)."""
    pts = cg.geodesic_points
    rho = pts["x"][1] * np.sin(pts["x"][2])
    J = np.argsort(rho, kind="stable")
    pts = {k: a[:, J] for k, a in pts.items()}
    r, t, eps = _build_radial_profile(cg.metric, spectrum, rho[J], pts["x"][0], cg.source_velocity[:, J], pts, N, ensemble, grid)
    return RadialDiscProfile(r, eps, t)


def emissivity_profiles(models: Sequence, spectrum=PowerLawSpectrum(2.0), *, n_samples=1000, delta_min=0.01,
                        delta_max=179.99, lambda_max=10_000.0, callback="default", ensemble=None, solver=None, **kwargs):
    """Point-source emissivity profiles for many (metric, disc, model) triples in ONE fused launch: the loop a
    parameter study (e.g. 20×20 spins × heights) runs around `emissivity_profile`."""
    if callback == "default":
        callback = api.domain_upper_hemisphere()
    prepared = [_point_source_job(m, d, model, delta_min, delta_max, n_samples, lambda_max, callback, kwargs)
                for (m, d, model) in models]
    results = _trace_many([p[2] for p in prepared], ensemble, solver)
    return [_point_source_postprocess(models[k][0], spectrum, prepared[k][1], prepared[k][0], gps, ensemble)
            for k, gps in enumerate(results)]


def emissivity_profile(m, d, model, spectrum=PowerLawSpectrum(2.0), *, sampler=None, n_samples=1000, N=100,
                       grid="geometric", ensemble=None, solver=None, **kwargs) -> RadialDiscProfile:
    """`emissivity_profile(m, d, model, spectrum; n_samples, sampler, ...)` (emissivity.jl:139-168).  Without a
    sampler, point sources on the axis use the polar-angle scheme (lamp-post.jl:156-164); with one, the sky is
    sampled and photon counts are binned."""
    if sampler is None and isinstance(model, (LampPostModel, BeamedPointSource)):
        return emissivity_profiles([(m, d, model)], spectrum, n_samples=n_samples, ensemble=ensemble, solver=solver,
                                   **kwargs)[0]
    lam = kwargs.pop("lambda_max", kwargs.pop("λmax", 10_000.0))
    cg = tracecorona(m, d, model, sampler=sampler, lambda_max=lam, n_samples=n_samples, ensemble=ensemble, solver=solver)
    return radial_disc_profile(cg, spectrum, N=N, grid=grid, ensemble=ensemble)
