"""Lag (2-D) transfer functions (rest of SURVEY 8 row f3): `lagtransfer` / `binflux`
(src/transfer-functions/transfer-functions-2d.jl:100-242) and `AnalyticRadialDiscProfile` (src/corona/analytic.jl:1-40).

Both legs are endpoint traces on the device: source → disc through `tracecorona` (explicit ICs), observer → disc through
one fused `gb200_render` over the image plane that returns (status, g, ρ, t) per ray, so no endpoint arrays cross the
bus.  Binning is the reference's `Buckets.Simple` in two dimensions (slot i takes bins[i] ≤ v < bins[i+1], clamped).
`binned_lagtransfer` returns what `binflux(lagtransfer(...))` returns with the binning on the device as well
(`gb200_lagtransfer`), so no per-ray data reaches the host."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Callable, Optional

import numpy as np

from . import _cabi as cabi
from . import api, corona
from .tf_integration import NaNLinearInterpolator


@dataclass
class AnalyticRadialDiscProfile:
    """ε(r) given as a function, arrival time interpolated from the coronal geodesics (corona/analytic.jl:1-40)."""

    eps: Callable
    t: NaNLinearInterpolator

    @classmethod
    def from_corona(cls, emissivity, cg: corona.CoronaGeodesics):
        x = cg.geodesic_points["x"]
        rho = x[1] * np.sin(x[2])
        J = np.argsort(rho, kind="stable")
        return cls(emissivity, NaNLinearInterpolator(rho[J], x[0][J]))

    def emissivity_at(self, r):
        return self.eps(np.asarray(r))

    def coordtime_at(self, r):
        return self.t(np.clip(r, self.t.t[0], self.t.t[-1]))


@dataclass
class LagTransferFunction:
    """transfer-functions/types.jl `LagTransferFunction`; the observer→disc leg is kept as the per-ray quantities
    `binflux` needs (g, ρ, t) instead of full geodesic points."""

    max_t: float
    x: np.ndarray
    image_plane_areas: np.ndarray
    coronal_geodesics: corona.CoronaGeodesics
    g: np.ndarray
    rho: np.ndarray
    t: np.ndarray

    @property
    def observer_to_disc_count(self):
        return len(self.g)


def unnormalized_areas(plane: api.PolarPlane):
    """image-planes/planes.jl:108-115: r² per ray, r the fastest index."""
    if not isinstance(plane, api.PolarPlane):
        raise ValueError("lagtransfer is implemented for PolarPlane image planes")
    if isinstance(plane.grid, api.GeometricGrid):
        rs = plane.r_min * (plane.r_max / plane.r_min) ** (np.arange(plane.Nr) / (plane.Nr - 1))
    elif isinstance(plane.grid, api.InverseGrid):
        rs = (1.0 / np.linspace(1.0 / plane.r_max, 1.0 / plane.r_min, plane.Nr))[::-1]
    else:
        rs = np.linspace(plane.r_min, plane.r_max, plane.Nr)
    return np.tile(rs**2, plane.Ntheta)


def _device_evaluator(config, pfs):
    return api.apply_point_functions(config, pfs)


def lagtransfer(m, x, d, model, *, plane=None, max_t=None, n_samples=10_000, sampler=None, callback="default",
                ensemble=None, solver=None, evaluator=None, **solver_opts) -> LagTransferFunction:
    """`lagtransfer(m, u, d, model; plane, max_t, n_samples, sampler, ...)` (transfer-functions-2d.jl:163-218).
    `solver` / `evaluator` replace the device tracer in the CPU tests (oracle)."""
    x = np.asarray(x, np.float64)
    if plane is None:
        plane = api.PolarPlane(api.GeometricGrid(), Nr=800, Ntheta=800, r_max=50.0)
    if max_t is None:
        max_t = 2 * x[1]
    if sampler is None:
        sampler = corona.EvenSampler("both", "golden")  # the reference's default draws from its RNG
    if callback == "default":
        callback = api.domain_upper_hemisphere()
    ce = corona.tracecorona(m, d, model, lambda_max=max_t, n_samples=n_samples, sampler=sampler, callback=callback,
                            ensemble=ensemble, solver=solver, **solver_opts)
    config = api.tracing_configuration(m, x, plane, d, (0.0, max_t), chart=api.chart_for_metric(m, 1.1 * x[1]),
                                       callback=callback, ensemble=ensemble, **solver_opts)
    C = api.ConstPointFunctions
    pfs = [api.PointFunction("status"), C.redshift(m, x) @ C.filter_intersected(), C.radius() @ C.filter_intersected(),
           C.coordinate_time() @ C.filter_intersected()]
    status, g, rho, t = (evaluator or _device_evaluator)(config, pfs)
    I = status == cabi.STATUS_INTERSECTED
    return LagTransferFunction(float(max_t), x, unnormalized_areas(plane)[I], ce, g[I], rho[I], t[I])


def _simple_bucket_index(bins, v):
    return np.clip(np.searchsorted(bins, v, side="right") - 1, 0, len(bins) - 1)


def bucket2d(x, y, w, xbins, ybins, ensemble=None):
    """`bucket(x, y, w, xbins, ybins; reduction = sum)` (Buckets.Simple in both axes).  With an `ensemble` the histogram is
    accumulated on the device (`gb200_bucket2d`, order-independent fixed-point sums); without, on the host."""
    xbins = np.ascontiguousarray(xbins, np.float64)
    ybins = np.ascontiguousarray(ybins, np.float64)
    if ensemble is None:
        out = np.zeros((len(xbins), len(ybins)))
        np.add.at(out, (_simple_bucket_index(xbins, x), _simple_bucket_index(ybins, y)), w)
        return out
    import ctypes as C

    x, y, w = (np.ascontiguousarray(a, np.float64) for a in (x, y, w))
    out = np.zeros((len(xbins), len(ybins)))
    ctx = ensemble.ctx(ensemble.devices[0])
    cabi.check(cabi.load().gb200_bucket2d(ctx, len(x), cabi.dptr(x), cabi.dptr(y), cabi.dptr(w), cabi.dptr(xbins), len(xbins), cabi.dptr(ybins),
                                          len(ybins), cabi.dptr(out.reshape(-1))), ctx)
    return out


def bin_transfer_function(time_delays, energy, flux, *, N_E=300, N_t=300, energy_lims=None, time_lims=None, ensemble=None):
    """transfer-functions-2d.jl:100-122 → (time_bins, energy_bins, tf[N_E, N_t]) with empty cells NaN."""
    energy_lims = (np.min(energy), np.max(energy)) if energy_lims is None else energy_lims
    time_lims = (np.min(time_delays), np.max(time_delays)) if time_lims is None else time_lims
    eb = np.linspace(energy_lims[0], energy_lims[1], N_E)
    tb = np.linspace(time_lims[0], time_lims[1], N_t)
    de, dt = eb[1] - eb[0], tb[1] - tb[0]
    out = bucket2d(energy, time_delays, flux, eb, tb, ensemble)
    out /= de * dt
    out[out == 0.0] = np.nan
    return tb, eb, out


def binflux(tf: LagTransferFunction, profile=None, *, E0=6.4, t0=None, **kwargs):
    """`binflux(tf, profile; E₀, t0, N_E, N_t, ...)` (transfer-functions-2d.jl:220-242)."""
    if profile is None:
        profile = AnalyticRadialDiscProfile.from_corona(lambda r: r**-3.0, tf.coronal_geodesics)
    if t0 is None:
        t0 = tf.x[1]
    t = profile.coordtime_at(tf.rho) + tf.t
    eps = profile.emissivity_at(tf.rho)
    f = tf.g**3 * eps * tf.image_plane_areas
    F = f / f.sum()
    tb, eb, td = bin_transfer_function(t, tf.g * E0, F, **kwargs)
    return tb - t0, eb, td


def _emissivity_to_c(eps, c: cabi.DiscProfile, keep: list, host="binflux(lagtransfer(...), profile)"):
    """Fill c.emissivity from a PowerLawEmissivity or TabulatedEmissivity (its arrays appended to `keep`); anything else
    raises TypeError naming the host function that evaluates it instead."""
    if isinstance(eps, api.PowerLawEmissivity):
        c.emissivity.kind, c.emissivity.index = cabi.EMISSIVITY_POWERLAW, float(eps.index)
    elif isinstance(eps, api.TabulatedEmissivity):
        r, e = np.ascontiguousarray(eps.r, np.float64), np.ascontiguousarray(eps.eps, np.float64)
        keep += [r, e]
        c.emissivity.kind, c.emissivity.n = cabi.EMISSIVITY_TABLE, len(r)
        c.emissivity.r, c.emissivity.eps = cabi.dptr(r), cabi.dptr(e)
    else:
        raise TypeError("an emissivity given as a Python callable cannot cross the C ABI: pass PowerLawEmissivity or "
                        f"TabulatedEmissivity, or use {host}")


def _disc_profile_to_c(profile, host="binflux(lagtransfer(...), profile)"):
    """-> (gb200_disc_profile, arrays it points into).  Raises TypeError for an ε the device cannot evaluate, naming `host`,
    the host function that can."""
    if isinstance(profile, AnalyticRadialDiscProfile):
        eps, r, t, kind = profile.eps, profile.t.t, profile.t.u, cabi.PROFILE_TIME_NAN_LINEAR
        if profile.t.default != 0.0:
            raise TypeError("the device supports NaNLinearInterpolator's default fallback value 0 only")
    elif isinstance(profile, corona.RadialDiscProfile):
        eps, r, t, kind = api.TabulatedEmissivity(profile.radii, profile.eps), profile.radii, profile.t, cabi.PROFILE_TIME_LINEAR
    else:
        raise TypeError(f"profile {type(profile).__name__} cannot be evaluated on the device: use {host}")
    keep = [np.ascontiguousarray(r, np.float64), np.ascontiguousarray(t, np.float64)]
    c = cabi.DiscProfile()
    _emissivity_to_c(eps, c, keep, host)
    c.time_kind, c.n, c.r, c.t = kind, len(keep[0]), cabi.dptr(keep[0]), cabi.dptr(keep[1])
    return c, keep


def binned_lagtransfer(m, x, d, model, profile=None, *, plane=None, max_t=None, n_samples=10_000, sampler=None, callback="default",
                       E0=6.4, t0=None, N_E=300, N_t=300, energy_lims=None, time_lims=None, ensemble=None, **solver_opts):
    """`binflux(lagtransfer(m, x, d, model; ...), profile; E0, t0, N_E, N_t, energy_lims, time_lims)` with the observer→disc
    leg binned on the device (`gb200_lagtransfer`, or `gb200_comm_lagtransfer` over several devices): no per-ray data
    reaches the host, and the histogram is summed in fixed point, so it is the same bits on any number of devices.
    Returns (time edges - t0, energy edges, tf[N_E, N_t], number of observer→disc hits).  `profile=None` is ε = r⁻³ with the
    coronal arrival times; an `AnalyticRadialDiscProfile` needs a `PowerLawEmissivity` or `TabulatedEmissivity` ε."""
    x = np.asarray(x, np.float64)
    if plane is None:
        plane = api.PolarPlane(api.GeometricGrid(), Nr=800, Ntheta=800, r_max=50.0)
    if not isinstance(plane, api.PolarPlane):
        raise ValueError("lagtransfer is implemented for PolarPlane image planes")
    if profile is not None:
        _disc_profile_to_c(profile)  # reject what cannot cross the ABI before tracing
    if max_t is None:
        max_t = 2 * x[1]
    if sampler is None:
        sampler = corona.EvenSampler("both", "golden")
    if callback == "default":
        callback = api.domain_upper_hemisphere()
    if t0 is None:
        t0 = x[1]
    ce = corona.tracecorona(m, d, model, lambda_max=max_t, n_samples=n_samples, sampler=sampler, callback=callback,
                            ensemble=ensemble, **solver_opts)
    if profile is None:
        profile = AnalyticRadialDiscProfile.from_corona(api.PowerLawEmissivity(3.0), ce)
    config = api.tracing_configuration(m, x, plane, d, (0.0, max_t), chart=api.chart_for_metric(m, 1.1 * x[1]),
                                       callback=callback, ensemble=ensemble, **solver_opts)
    p, ic = config.to_c()
    prof, _keep = _disc_profile_to_c(profile)
    nan = float("nan")
    opts = cabi.LagTransferOpts(float(E0), float(t0), tuple(energy_lims) if energy_lims is not None else (nan, nan),
                                tuple(time_lims) if time_lims is not None else (nan, nan), int(N_E), int(N_t))
    plunging = api._auto_plunging(m, d, config.ensemble, True, None)
    pl_ref = C.byref(plunging.c) if plunging is not None else None
    tb, eb, tf, hits = np.zeros(int(N_t)), np.zeros(int(N_E)), np.zeros((int(N_E), int(N_t))), C.c_int64()
    args = (C.byref(p), C.byref(ic), C.byref(prof), pl_ref, C.byref(opts), cabi.dptr(tb), cabi.dptr(eb), cabi.dptr(tf.reshape(-1)), C.byref(hits))
    lib = cabi.load()
    comm = config.ensemble.comm()
    if comm is not None:
        api._install_on_comm(comm, config.geometry)
        cabi.check(lib.gb200_comm_lagtransfer(comm, *args))
    else:
        ctx = config.ensemble.ctx(config.ensemble.devices[0])
        if hasattr(config.geometry, "install"):
            config.geometry.install(ctx)
        cabi.check(lib.gb200_lagtransfer(ctx, *args), ctx)
    return tb, eb, tf, int(hits.value)


def continuum_time(m, x, model, **kwargs):
    """`continuum_time(m, x, model)` (src/reverberation.jl:81-93): coordinate time of the direct corona-to-observer light
    path, found backwards as the geodesic from the observer that reaches the corona's position (`optimize_for_target`
    with the upper-hemisphere callback and a chart of twice the observer's radius)."""
    pos, _ = corona.sample_position_velocity(m, model)
    kwargs.setdefault("chart", api.chart_for_metric(m, 2.0 * float(x[1])))
    kwargs.setdefault("callback", api.domain_upper_hemisphere())
    _, _, gp, _ = api.optimize_for_target(pos[1:], m, x, **kwargs)
    return float(gp["x"][0])



def lag_frequency(t, f, *, flo=5e-5, R=1.0):
    """`lag_frequency(t, f::AbstractMatrix; flo)` (src/reverberation.jl:29-49): the impulse response ψ(t) = Σ_E f[E, t] (NaNs as
    zeros) is padded with zeros out to 1 / flo on the same time step, Fourier transformed, and the phase
    atan(Im ψ̂ / (1 + Re ψ̂)) of the positive frequencies becomes a time lag φ / (2π ν).  Returns (frequencies, −lag); the
    zero-frequency entry is 0 / 0 as in the reference.  Host FFT of a ~20 000-point array."""
    t = np.asarray(t, np.float64)
    f = np.asarray(f, np.float64)
    psi = np.nansum(f, axis=0) if f.ndim == 2 else np.where(np.isnan(f), 0.0, f)
    dt = t[1] - t[0]
    t_ext = np.arange(t.min(), 1.0 / flo + 0.5 * dt * 1e-9, dt)  # range(minimum(t), 1 / flo, step = Δt)
    psi_ext = np.zeros(t_ext.size)
    psi_ext[: psi.size] = psi
    freq = np.fft.fftfreq(t_ext.size, dt)
    F = R * np.fft.fft(psi_ext)
    n = t_ext.size // 2
    phase = np.arctan(F[:n].imag / (1.0 + F[:n].real))
    with np.errstate(divide="ignore", invalid="ignore"):
        lag = phase / (2.0 * np.pi * freq[:n])
    return freq[:n], -lag
