"""Host-side mirror of the reference's tracing front-end for the in-scope path.

Everything here is argument plumbing: it flattens the reference's configuration objects
(`TracingConfiguration`, src/tracing/configuration.jl:3-125) into the POD structs of
include/gradus_b200.h and calls the C ABI.  The Julia extension described in
INTEGRATION.md does exactly the same with `ccall`."""
from __future__ import annotations

import ctypes as C
import math
import threading
from dataclasses import dataclass, field
from typing import Any, Callable, Optional, Sequence

import numpy as np

from . import _cabi as cabi

DEFAULT_TOLERANCE = 1e-9  # src/tracing/configuration.jl:1


class StatusCodes:
    """src/Gradus.jl:59-64 (declaration order = integer value)."""

    OutOfDomain = 0
    WithinInnerBoundary = 1
    IntersectedWithGeometry = 2
    NoStatus = 3


# --------------------------------------------------------------------------- metrics
@dataclass(frozen=True)
class KerrMetric:
    """src/metrics/kerr-metric.jl:62-68"""

    M: float = 1.0
    a: float = 0.0
    kind = cabi.METRIC_KERR

    def params(self):
        return _pad8(self.M, self.a)


@dataclass(frozen=True)
class JohannsenPsaltisMetric:
    """src/metrics/johannsen-psaltis-ad.jl:38-46 (`eps3` is the reference's `ϵ3`)."""

    M: float = 1.0
    a: float = 0.0
    eps3: float = 0.0
    kind = cabi.METRIC_JP

    def params(self):
        return _pad8(self.M, self.a, self.eps3)


@dataclass(frozen=True)
class JohannsenMetric:
    """src/metrics/johannsen-ad.jl:40-62 (`alpha13, alpha22, alpha52, eps3` are the reference's α13, α22, α52, ϵ3)."""

    M: float = 1.0
    a: float = 0.0
    alpha13: float = 0.0
    alpha22: float = 0.0
    alpha52: float = 0.0
    eps3: float = 0.0
    kind = cabi.METRIC_JOHANNSEN

    def params(self):
        return _pad8(self.M, self.a, self.alpha13, self.alpha22, self.alpha52, self.eps3)


@dataclass(frozen=True)
class BumblebeeMetric:
    """src/metrics/bumblebee-ad.jl:26-46: slow-rotation metric with Lorentz-symmetry-breaking parameter l."""

    M: float = 1.0
    a: float = 0.0
    l: float = 0.0  # noqa: E741
    kind = cabi.METRIC_BUMBLEBEE

    def __post_init__(self):
        if self.l <= -1.0:
            raise ValueError("l must be >-1")
        if abs(self.a) > 0.3:
            raise ValueError("This metric is for the slow rotation approximation only, and requires |a| < 0.3.")

    def params(self):
        return _pad8(self.M, self.a, self.l)


@dataclass(frozen=True)
class KerrNewmanMetric:
    """src/metrics/kerr-newman-ad.jl:41-58.  Charged test particles: pass `q=` to the tracing call (Lorentz force,
    kerr-newman-ad.jl:66-102)."""

    M: float = 1.0
    a: float = 0.0
    Q: float = 0.0
    kind = cabi.METRIC_KERR_NEWMAN

    def __post_init__(self):
        if self.a**2 + self.Q**2 > self.M**2:
            raise ValueError("Value error: `a^2 + Q^2` must be `<= M^2`")

    def params(self):
        return _pad8(self.M, self.a, self.Q)


@dataclass(frozen=True)
class MorrisThorneWormhole:
    """src/metrics/morris-thorne-ad.jl:28-40: wormhole with throat size b; the radial coordinate is the proper distance l
    (negative on the far side of the throat), `inner_radius` = 0, no horizon and no ISCO."""

    b: float = 1.0
    kind = cabi.METRIC_MORRIS_THORNE

    def params(self):
        return _pad8(self.b)


@dataclass(frozen=True)
class DilatonAxion:
    """src/metrics/dilaton-axion-ad.jl:48-72: Einstein-Maxwell-Dilaton-Axion metric (Garcia et al. 1995); `beta` is the
    reference's β (dilaton coupling), `b` the axion coupling.  The ratios β/b, β/a, β/(a b) follow the reference's rule
    (0 where β == 0, :24-26) and travel as parameters 4..6."""

    M: float = 1.0
    a: float = 0.5
    beta: float = 0.0
    b: float = 1.0
    kind = cabi.METRIC_DILATON_AXION

    def ratios(self):
        if self.beta == 0.0:
            return 0.0, 0.0, 0.0
        if self.a == 0.0 or self.b == 0.0:
            raise ValueError("DilatonAxion with β ≠ 0 needs a ≠ 0 and b ≠ 0")
        return self.beta / self.b, self.beta / self.a, self.beta / (self.a * self.b)

    def params(self):
        return _pad8(self.M, self.a, self.beta, self.b, *self.ratios())


def _pad8(*vals):
    return tuple(float(v) for v in vals) + (0.0,) * (8 - len(vals))


_SUPPORTED_METRICS = (KerrMetric, JohannsenPsaltisMetric, JohannsenMetric, BumblebeeMetric, KerrNewmanMetric, MorrisThorneWormhole, DilatonAxion)


def _check_metric(m):
    if not isinstance(m, _SUPPORTED_METRICS):
        raise ValueError("EnsembleB200 supports " + ", ".join(c.__name__ for c in _SUPPORTED_METRICS)
                         + f" only, got {type(m).__name__} (no CPU fallback)")


def inner_radius(m) -> float:
    """kerr-metric.jl:72, johannsen-psaltis-ad.jl:50, johannsen-ad.jl:66, bumblebee-ad.jl:51, kerr-newman-ad.jl:65"""
    _check_metric(m)
    if isinstance(m, MorrisThorneWormhole):
        return 0.0  # morris-thorne-ad.jl:40
    if isinstance(m, DilatonAxion):  # dilaton-axion-ad.jl:69-72
        bb = m.ratios()[0]
        return m.M + m.b + math.sqrt((m.M + m.b) ** 2 - m.a**2 + m.beta**2 - (m.M - 2 * m.b) * m.M * bb**2)
    q2 = m.Q**2 if isinstance(m, KerrNewmanMetric) else 0.0
    return m.M + math.sqrt(m.M**2 - m.a**2 - q2)


def _metric_params_array(m):
    return (C.c_double * 8)(*m.params())


def isco(m) -> float:
    """Innermost stable circular orbit (kerr-metric.jl:91; src/special-radii.jl:14-60). Host arithmetic in the library."""
    _check_metric(m)
    out = C.c_double()
    cabi.check(cabi.load().gb200_isco(m.kind, _metric_params_array(m), C.byref(out)))
    return out.value


# --------------------------------------------------------------------------- geometry
@dataclass(frozen=True)
class ThinDisc:
    """src/geometry/discs/thin-disc.jl:9-14"""

    inner_radius: float = 0.0
    outer_radius: float = 500.0

    def to_c(self):
        return cabi.GEOMETRY_THIN_DISC, (float(self.inner_radius), float(self.outer_radius), 0.0, 0.0)


@dataclass(frozen=True)
class DatumPlane:
    """src/geometry/discs/datum-plane.jl:1-10"""

    height: float = 0.0

    def to_c(self):
        return cabi.GEOMETRY_DATUM_PLANE, (float(self.height), 0.0, 0.0, 0.0)


class ShakuraSunyaev:
    """src/geometry/discs/shakura-sunyaev.jl:22-52.  `ShakuraSunyaev(m; eddington_ratio, η)`."""

    def __init__(self, m, eddington_ratio=0.3, eta=None):
        _check_metric(m)
        self.inner_radius = isco(m)
        if eta is None:
            out = C.c_double()
            cabi.check(cabi.load().gb200_radiative_efficiency(m.kind, _metric_params_array(m), C.byref(out)))
            eta = out.value
        self.Mdot_Medd = float(eddington_ratio)
        self.inv_eta = 1.0 / eta

    def to_c(self):
        return cabi.GEOMETRY_SHAKURA_SUNYAEV, (self.Mdot_Medd, self.inv_eta, self.inner_radius, 0.0)

    def cross_section(self, rho):
        """`cross_section(d::ShakuraSunyaev, ρ)`, shakura-sunyaev.jl:28-33 (vectorised)."""
        rho = np.asarray(rho, np.float64)
        with np.errstate(all="ignore"):
            h = 3.0 * self.inv_eta * self.Mdot_Medd * (1.0 - np.sqrt(self.inner_radius / rho))
        return np.where(rho < self.inner_radius, -0.0, h)


def cartesian_tangent_vector(d, rho):
    """`_cartesian_tangent_vector(d, ρ)` (src/geometry/discs/thick-disc.jl:65-72): the unit tangent of the disc surface
    (ρ, 0, cross_section(ρ)) in the x-z plane; the derivative the reference takes by ForwardDiff is a complex step here for
    the Shakura-Sunyaev height and a central difference for closures."""
    rho = float(rho)
    if isinstance(d, ShakuraSunyaev):
        dh = 0.0 if rho < d.inner_radius else 3.0 * d.inv_eta * d.Mdot_Medd * 0.5 * math.sqrt(d.inner_radius / rho) / rho
    else:
        h = 1e-6 * max(1.0, abs(rho))
        dh = float(d.cross_section(rho + h) - d.cross_section(rho - h)) / (2 * h)
    v = np.array([1.0, 0.0, dh])
    return v / np.linalg.norm(v)


def cartesian_surface_normal(d, rho):
    """`_cartesian_surface_normal(d, ρ)` (thick-disc.jl:74-78): the tangent rotated by 90° about φ̂."""
    t = cartesian_tangent_vector(d, rho)
    return np.array([-t[2], t[1], t[0]])


class ThickDisc:
    """`ThickDisc(f; inner_radius, outer_radius)` (src/geometry/discs/thick-disc.jl:32-52): a disc whose height above the
    equatorial plane is the closure `f(ρ)` (non-positive where there is no disc).  A closure cannot cross the C ABI, so it is
    tabulated once: `n` Chebyshev nodes over `support = (ρ_lo, ρ_hi)` -- they crowd towards the ends as 1/n², which resolves
    the square-root edges of tori -- and the device interpolates linearly (GB200_GEOMETRY_THICK_TABLE); outside the support
    there is no disc."""

    def __init__(self, f, support, n=4097, inner_radius=0.0, outer_radius=float("inf")):
        lo, hi = float(support[0]), float(support[1])
        if not (hi > lo) or n < 2:
            raise ValueError("ThickDisc needs support = (lo, hi) with hi > lo and n >= 2")
        k = np.arange(n)
        self.rho = np.ascontiguousarray(0.5 * (lo + hi) - 0.5 * (hi - lo) * np.cos(math.pi * k / (n - 1)))
        self.rho[0], self.rho[-1] = lo, hi
        self.height = np.ascontiguousarray([float(f(r)) for r in self.rho])
        self.f, self.inner_radius, self.outer_radius = f, float(inner_radius), float(outer_radius)

    def to_c(self):
        return cabi.GEOMETRY_THICK_TABLE, (float(self.height.max()), float(self.rho[0]), float(self.rho[-1]), 0.0)

    def cross_section(self, rho):
        return np.interp(rho, self.rho, self.height, left=-1.0, right=-1.0)

    def install(self, ctx):
        cabi.check(cabi.load().gb200_set_cross_section(ctx, cabi.dptr(self.rho), cabi.dptr(self.height), len(self.rho)), ctx)


class PolishDoughnut(ThickDisc):
    """`PolishDoughnut(m; rₖ = 12, n = 0.21, init_r = 5)` (src/geometry/discs/polish-doughnut.jl): a pressure-supported torus
    (Fuerst & Wu 2004; Younsi et al. 2012) whose surface is an isobar through the innermost radius.  As in the reference the
    set-up runs on the host -- innermost radius = the root of dE/dr of the sub-Keplerian orbital energy, the isobar as a
    2-D ODE in (r, θ) integrated with Tsit5 (dtmax = 5e-2, OrdinaryDiffEq's default tolerances, every step saved) -- and the
    cross-section is the linear interpolation of height over the saved radii; that table is what the device receives
    (GB200_GEOMETRY_THICK_TABLE), so it interpolates the same nodes the reference does.  Kerr only, as in the reference."""

    def __init__(self, m, rk=12.0, n=0.21, init_r=5.0, lambda_max=40.0, dtmax=5e-2):
        from . import hostmath
        if not isinstance(m, KerrMetric):
            raise ValueError("PolishDoughnut: the isobar differential is defined for KerrMetric only (polish-doughnut.jl:39)")
        M, a = m.M, m.a

        def omega(r, th):  # Ω of the circular orbit at the cylindrical radius, scaled by (rₖ / r sinθ)^n (:17-21)
            rs = r * np.sin(th)
            kep = math.sqrt(M) / (rs**1.5 + a * math.sqrt(M))  # CircularOrbits.Ω of Kerr in closed form (prograde)
            return kep * (rk / rs) ** n

        def energy(r):  # orbital_energy at θ = π/2 (:23-31); complex r for the complex-step derivative
            g = hostmath.metric_components(m, r, math.pi / 2)
            w = omega(r, math.pi / 2)
            return -(g[0] + g[4] * w) / np.sqrt(-g[0] - 2 * g[4] * w - g[3] * w * w)

        dE = lambda r: float(np.imag(energy(r + 1e-30j)) / 1e-30)  # noqa: E731
        r0 = float(init_r)
        for _ in range(100):  # Newton on dE/dr with a central second difference (Roots.find_zero((df, d2f), init_r))
            h = 1e-5 * max(1.0, abs(r0))
            step = dE(r0) / ((dE(r0 + h) - dE(r0 - h)) / (2 * h))
            r0 -= step
            if abs(step) < 1e-14 * max(1.0, abs(r0)):
                break
        self.rk, self.n = float(rk), float(n)

        def rhs(u):  # isobar_differential (:39-52), Younsi et al. (2012) eqs. (30), (31)
            r, th = u
            inv_w = 1.0 / float(omega(r, th))
            s, c = math.sin(th), math.cos(th)
            sig, dlt = r * r + a * a * c * c, r * r - 2 * M * r + a * a
            p1 = M * ((sig - 2 * r * r) / sig**2) * (inv_w - a * s) ** 2 + r * s * s
            p2 = math.sin(2 * th) * ((M * r / sig**2) * (a * inv_w - (r * r + a * a)) ** 2 + dlt / 2)
            d = 1.0 / (math.sqrt(dlt * p1 * p1 + p2 * p2) * math.sqrt(1.0 / (dlt / sig)))
            return np.array([p2 * d, -p1 * d])

        sol = hostmath.tsit5_solve(rhs, [r0, math.pi / 2], float(lambda_max), dtmax=float(dtmax), terminate=lambda u: u[0] * math.cos(u[1]) < 0)
        r = np.array([u[0] for u in sol])
        z = np.array([math.cos(u[1]) * u[0] for u in sol])
        keep = z > 0
        self.rho, self.height = np.ascontiguousarray(r[keep]), np.ascontiguousarray(z[keep])
        if np.any(np.diff(self.rho) <= 0):
            raise ValueError("PolishDoughnut: the isobar does not run monotonically outwards for these parameters")
        self.inner_radius, self.outer_radius = r0, float(r.max())
        self.f = self.cross_section

    def cross_section(self, rho):
        """`cross_section(d, ρ)` (:123-129): the interpolated height inside [inner_radius, outer_radius], zero outside."""
        rho = np.asarray(rho, np.float64)
        return np.where((rho >= self.inner_radius) & (rho <= self.rho[-1]), np.interp(rho, self.rho, self.height), 0.0)


@dataclass(frozen=True)
class ImageOrder:
    """`ImageOrder(disc, n)`: the order-n image of a thin disc (n = 0 the direct image, 1 and 2 the first subrings).
    A ray hits it at its first entry into the disc's wedge in a step that starts with n equatorial crossings (see
    `ConstPointFunctions.equatorial_crossings`); entries before that pass through, and once the count exceeds n the disc
    is inert.  A ray that hits `disc` with c crossings gives the same end point under `ImageOrder(disc, c)`.  Not a type
    of the reference: GB200_GEOMETRY_THIN_DISC_ORDER of include/gradus_b200.h."""

    disc: ThinDisc
    n: int

    def __post_init__(self):
        if type(self.disc) is not ThinDisc:
            raise ValueError("ImageOrder is defined for a ThinDisc only")
        if isinstance(self.n, bool) or not isinstance(self.n, (int, np.integer)) or self.n < 0:
            raise ValueError("ImageOrder needs a non-negative integer order n")

    @property
    def inner_radius(self):
        return self.disc.inner_radius

    @property
    def outer_radius(self):
        return self.disc.outer_radius

    def to_c(self):
        return cabi.GEOMETRY_THIN_DISC_ORDER, (float(self.disc.inner_radius), float(self.disc.outer_radius), float(self.n), 0.0)


_SUPPORTED_GEOMETRY = (ThinDisc, ShakuraSunyaev, DatumPlane, ThickDisc, ImageOrder)


# --------------------------------------------------------------------------- charts and callbacks
@dataclass(frozen=True)
class PolarChart:
    """src/tracing/charts.jl:3-6"""

    inner_radius: float
    outer_radius: float


def chart_for_metric(m, outer_radius=12000.0, closest_approach=1.01):
    """src/tracing/charts.jl:51-58"""
    return PolarChart(inner_radius(m) * closest_approach, float(outer_radius))


@dataclass(frozen=True)
class UpperHemisphereCallback:
    delta: float = 1e-4


def domain_upper_hemisphere(delta=1e-4):
    """src/tracing/callbacks.jl:31-39"""
    return UpperHemisphereCallback(float(delta))


# --------------------------------------------------------------------------- image planes
@dataclass(frozen=True)
class LinearGrid:
    kind = cabi.GRID_LINEAR


@dataclass(frozen=True)
class GeometricGrid:
    kind = cabi.GRID_GEOMETRIC


@dataclass(frozen=True)
class InverseGrid:
    kind = cabi.GRID_INVERSE


@dataclass(frozen=True)
class PolarPlane:
    """src/image-planes/planes.jl:70-91"""

    grid: Any = field(default_factory=GeometricGrid)
    Nr: int = 400
    Ntheta: int = 100
    r_min: float = 1.0
    r_max: float = 250.0
    theta_min: float = 0.0
    theta_max: float = 2 * math.pi

    def trajectory_count(self):
        return self.Nr * self.Ntheta


@dataclass(frozen=True)
class CartesianPlane:
    """src/image-planes/planes.jl:130-163"""

    grid: Any = field(default_factory=LinearGrid)
    Nx: int = 150
    Ny: int = 150
    x_min: float = 0.0
    x_max: float = 150.0
    y_min: float = 0.0
    y_max: float = 150.0

    def trajectory_count(self):
        return (2 * (self.Ny // 2) - 1) * (2 * (self.Nx // 2) - 1)


@dataclass(frozen=True, eq=False)
class ImpactParameters:
    """`map_impact_parameters(m, x, αs, βs)` (src/tracing/utility.jl:70-87) as data: one ray per (α, β) pair."""

    alpha: Any
    beta: Any
    height: Any = None  # optional per-ray datum-plane heights (`datumplane(d, rₑ)` of many radii in one launch)

    def trajectory_count(self):
        return len(self.alpha)


@dataclass(frozen=True)
class RenderGrid:
    """The closure returned by `_render_velocity_function` (src/rendering/rendering.jl:140-163) as data."""

    image_width: int
    image_height: int
    alpha_lims: tuple
    beta_lims: tuple

    def trajectory_count(self):
        return self.image_width * self.image_height


# --------------------------------------------------------------------------- ensembles
class EnsembleB200:
    """New ensemble type (next to `EnsembleEndpointThreads`, src/Gradus.jl:412): rays are
    integrated on the listed CUDA devices by libgradus_b200.  One context per device."""

    def __init__(self, devices: Sequence[int] = (0,)):
        self.devices = tuple(int(d) for d in devices)
        if not self.devices:
            raise ValueError("EnsembleB200 needs at least one device")
        self._ctx = {}
        self._comm = None

    def ctx(self, device, slot=0):
        """Context for `device`; `slot` distinguishes several contexts on the same device (one per host thread)."""
        key = (device, slot)
        if key not in self._ctx:
            h = C.c_void_p()
            cabi.check(cabi.load().gb200_init(device, C.byref(h)))
            self._ctx[key] = h
        return self._ctx[key]

    def comm(self):
        """The library's own multi-device communicator over `devices` (`gb200_comm_init`: one context per device plus an
        NCCL communicator, all in this process) -- what a Julia caller uses.  None for a single device or a list that
        names a device twice (those run through per-device contexts on host threads)."""
        if len(self.devices) < 2 or len(set(self.devices)) != len(self.devices):
            return None
        if self._comm is None:
            h = C.c_void_p()
            devs = np.array(self.devices, np.int32)
            cabi.check(cabi.load().gb200_comm_init(cabi.iptr(devs), len(devs), C.byref(h)))
            self._comm = h
        return self._comm

    def close(self):
        for h in self._ctx.values():
            cabi.load().gb200_destroy(h)
        self._ctx = {}
        if self._comm is not None:
            cabi.load().gb200_comm_destroy(self._comm)
            self._comm = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def stats(self, device=None):
        s = cabi.Stats()
        cabi.check(cabi.load().gb200_get_stats(self.ctx(self.devices[0] if device is None else device), C.byref(s)))
        return s


_DEFAULT_ENSEMBLE = None


def default_ensemble() -> EnsembleB200:
    """The ensemble used when a call passes none: one shared `EnsembleB200` on device 0, so repeated calls reuse one CUDA
    context, stream pool and device-buffer pool instead of creating one each (contexts are created lazily: building a
    configuration on a box without a GPU does not fail, running it does)."""
    global _DEFAULT_ENSEMBLE
    if _DEFAULT_ENSEMBLE is None:
        _DEFAULT_ENSEMBLE = EnsembleB200()
    return _DEFAULT_ENSEMBLE


class EnsembleEndpointThreads:
    """The reference's CPU ensemble.  Not available here by design: there is no CPU fallback."""


class BinningMethod:
    """src/Gradus.jl:447"""


class TransferFunctionMethod:
    """src/Gradus.jl:448: `lineprofile` by integrating Cunningham transfer functions (src/line-profiles.jl:121-150).  Carries
    that method's keywords -- `minrₑ` / `min_re`, `maxrₑ` / `max_re`, `numrₑ` / `num_re`, `h` (the quadrature's edge zone
    in g✶), `n_radii` -- and any keyword of the transfer-function set-up (`N`, `β₀` / `beta0`, `chart`, ...).  The defaults
    are those of `tf_integration.lineprofile_transfer_functions`."""

    def __init__(self, *, min_re=None, max_re=50.0, num_re=100, h=2e-8, n_radii=1000, **setup):
        # Python folds a keyword written minrₑ=... to "minre" (NFKC); a dict can still carry "minrₑ"
        self.min_re = _pop_alias(setup, ("minrₑ", "minre"), min_re)
        self.max_re = _pop_alias(setup, ("maxrₑ", "maxre"), max_re)
        self.num_re = _pop_alias(setup, ("numrₑ", "numre"), num_re)
        self.h, self.n_radii, self.setup = h, n_radii, setup


# --------------------------------------------------------------------------- configuration
@dataclass
class TracingConfiguration:
    """src/tracing/configuration.jl:3-88, restricted to what the device path supports."""

    metric: Any
    position: Any
    velocity: Any
    geometry: Any
    chart: PolarChart
    callback: Any
    solver: str
    ensemble: Any
    trajectories: Optional[int]
    lambda_domain: tuple
    abstol: float
    reltol: float
    gtol: float = 1e-2
    mu: float = 0.0
    q: float = 0.0  # charge of the test particle (TraceGeodesic(μ, q), src/tracing/tracing.jl; Kerr-Newman only)
    pow_mode: int = cabi.POW_EXACT
    maxiters: int = 0
    dtmax: float = 0.0
    _keep: list = field(default_factory=list, repr=False)

    def to_c(self, validate=True):
        """-> (gb200_problem, gb200_ic).  Raises ValueError for anything outside the hot-path scope.  `validate=False` skips
        the library's own `gb200_validate` (callers that must not load libgradus_b200: the CPU reference arm of bench.py)."""
        m = self.metric
        _check_metric(m)
        p = cabi.Problem()
        p.metric_kind = m.kind
        p.metric_params[:] = m.params()
        if self.q != 0.0:
            if not isinstance(m, KerrNewmanMetric):
                raise ValueError("charged test particles need a metric with an electromagnetic potential (KerrNewmanMetric)")
            # geodesic_ode_problem(::KerrNewmanMetric), kerr-newman-ad.jl:74-78: q for photons, q / μ otherwise
            p.metric_params[3] = self.q if abs(self.mu) < 1e-8 else self.q / self.mu
        if self.geometry is None:
            p.geometry_kind = cabi.GEOMETRY_NONE
        elif isinstance(self.geometry, _SUPPORTED_GEOMETRY):
            p.geometry_kind, gp = self.geometry.to_c()
            p.geometry_params[:] = gp
        else:
            raise ValueError(f"geometry {type(self.geometry).__name__} is outside the EnsembleB200 scope")
        if self.callback is None:
            p.callback_kind = cabi.CALLBACK_NONE
        elif isinstance(self.callback, UpperHemisphereCallback):
            p.callback_kind = cabi.CALLBACK_UPPER_HEMISPHERE
            p.callback_delta = self.callback.delta
        else:
            raise ValueError("only `domain_upper_hemisphere` user callbacks can run on the device")
        if not isinstance(self.chart, PolarChart):
            raise ValueError("only PolarChart is supported")
        if self.solver != "Tsit5":
            raise ValueError("EnsembleB200 integrates with Tsit5 only")
        p.pow_mode = self.pow_mode
        p.gtol = self.gtol
        p.chart_inner, p.chart_outer = self.chart.inner_radius, self.chart.outer_radius
        p.lambda_min, p.lambda_max = float(self.lambda_domain[0]), float(self.lambda_domain[1])
        p.abstol, p.reltol = float(self.abstol), float(self.reltol)
        p.dtmax = float(self.dtmax)
        p.mu = float(self.mu)
        p.maxiters = int(self.maxiters)

        ic = cabi.IC()
        v = self.velocity
        pos = np.asarray(self.position, np.float64)
        if isinstance(v, RenderGrid):
            if not (v.alpha_lims[0] <= v.alpha_lims[1] and v.beta_lims[0] <= v.beta_lims[1]):
                raise AssertionError("α/β limits must be sorted")  # rendering.jl:148-149
            p.observer[:] = pos
            ic.kind = cabi.IC_RENDER_GRID
            ic.width, ic.height = v.image_width, v.image_height
            ic.lo0, ic.hi0 = map(float, v.alpha_lims)
            ic.lo1, ic.hi1 = map(float, v.beta_lims)
            ic.n = v.trajectory_count()
        elif isinstance(v, PolarPlane):
            p.observer[:] = pos
            ic.kind = cabi.IC_POLAR_PLANE
            ic.grid_kind = v.grid.kind
            ic.width, ic.height = v.Nr, v.Ntheta
            ic.lo0, ic.hi0 = float(v.r_min), float(v.r_max)
            ic.lo1, ic.hi1 = float(v.theta_min), float(v.theta_max)
            ic.n = v.trajectory_count()
        elif isinstance(v, ImpactParameters):
            al = np.ascontiguousarray(v.alpha, np.float64)
            be = np.ascontiguousarray(v.beta, np.float64)
            if al.shape != be.shape or al.ndim != 1:
                raise ValueError("alpha and beta must be 1-D arrays of equal length")
            self._keep = [al, be]
            p.observer[:] = pos
            ic.kind = cabi.IC_IMPACT_PARAMETERS
            ic.x[0], ic.x[1] = cabi.dptr(al), cabi.dptr(be)
            if v.height is not None:
                hg = np.ascontiguousarray(np.broadcast_to(np.asarray(v.height, np.float64), al.shape))
                if not isinstance(self.geometry, DatumPlane):
                    raise ValueError("per-ray heights need a DatumPlane geometry")
                self._keep.append(hg)
                ic.x[2] = cabi.dptr(hg)
            ic.n = len(al)
        elif isinstance(v, CartesianPlane):
            p.observer[:] = pos
            ic.kind = cabi.IC_CARTESIAN_PLANE
            ic.grid_kind = v.grid.kind
            ic.width, ic.height = v.Nx, v.Ny
            ic.lo0, ic.hi0 = float(v.x_min), float(v.x_max)
            ic.lo1, ic.hi1 = float(v.y_min), float(v.y_max)
            ic.n = v.trajectory_count()
        else:
            # explicit SoA: what the Julia shim builds by evaluating prob_func on host threads
            if callable(v):
                if self.trajectories is None:
                    raise ValueError("When velocity is a function, trajectories must be defined.")  # configuration.jl:47-49
                vs = np.array([np.asarray(v(i + 1), np.float64) for i in range(self.trajectories)])
            else:
                vs = np.atleast_2d(np.asarray(v, np.float64))
                if self.trajectories is not None and vs.shape[0] == 1 and pos.ndim == 1:
                    raise ValueError("Trajectories should be `nothing` when solving only a single geodesic problem.")
            n = vs.shape[0]
            xs = np.broadcast_to(pos, (n, 4)) if pos.ndim == 1 else pos
            if xs.shape != (n, 4) or vs.shape != (n, 4):
                raise ValueError("positions and velocities must be (n, 4)")
            xs_soa = np.ascontiguousarray(xs.T)
            vs_soa = np.ascontiguousarray(vs.T)
            self._keep = [xs_soa, vs_soa]
            p.observer[:] = xs[0]
            ic.kind = cabi.IC_EXPLICIT
            for k in range(4):
                ic.x[k] = cabi.dptr(xs_soa[k])
                ic.v[k] = cabi.dptr(vs_soa[k])
            ic.n = n
        if validate:
            cabi.check(cabi.load().gb200_validate(C.byref(p), C.byref(ic)))
        return p, ic


_CONFIG_KWARGS = {"chart", "callback", "solver", "ensemble", "trajectories", "abstol", "reltol", "gtol", "mu", "μ",
                  "q", "pow_mode", "maxiters", "dtmax", "save_on", "verbose", "progress_bar", "integrator_verbose"}


def tracing_configuration(m, position, velocity, *args, **kwargs):
    """`tracing_configuration` (src/geometry/bootstrap.jl:1-22, src/tracing/configuration.jl:90-138).

    args = ([geometry], λ) with λ a number (λ_max) or a (λ_min, λ_max) pair."""
    if len(args) == 1:
        geometry, lam = None, args[0]
    elif len(args) == 2:
        geometry, lam = args
    else:
        raise TypeError("expected tracing_configuration(m, x, v, [geometry], λ)")
    unknown = set(kwargs) - _CONFIG_KWARGS
    if unknown:
        # solver_opts reach `solve` with kwargshandle = KeywordArgError (tracing.jl:106,146,215); the device
        # integrator has no further options, so every unknown keyword is an error.
        raise TypeError(f"unrecognised keyword arguments for the B200 integrator: {sorted(unknown)}")
    if kwargs.get("save_on", False):
        raise ValueError("Cannot use `EnsembleB200` with `save_on`")  # tracing.jl:159-161
    lam_dom = (0.0, float(lam)) if np.isscalar(lam) else (float(lam[0]), float(lam[1]))
    ensemble = kwargs.get("ensemble", None)
    if ensemble is None:
        ensemble = default_ensemble()
    if not isinstance(ensemble, EnsembleB200):
        raise ValueError("this build integrates on the GPU only: pass ensemble=EnsembleB200(...) (no CPU fallback)")
    return TracingConfiguration(
        metric=m,
        position=position,
        velocity=velocity,
        geometry=geometry,
        chart=kwargs.get("chart") or chart_for_metric(m),
        callback=kwargs.get("callback"),
        solver=kwargs.get("solver", "Tsit5"),
        ensemble=ensemble,
        trajectories=kwargs.get("trajectories"),
        lambda_domain=lam_dom,
        abstol=kwargs.get("abstol", DEFAULT_TOLERANCE),
        reltol=kwargs.get("reltol", DEFAULT_TOLERANCE),
        gtol=kwargs.get("gtol", 1e-2),
        mu=kwargs.get("mu", kwargs.get("μ", 0.0)),
        q=float(kwargs.get("q", 0.0)),
        pow_mode=kwargs.get("pow_mode", cabi.POW_EXACT),
        maxiters=kwargs.get("maxiters", 0),
        dtmax=kwargs.get("dtmax", 0.0),
    )


# --------------------------------------------------------------------------- results
class GeodesicPoints:
    """SoA of `GeodesicPoint`s (src/solution-processing.jl:15-32); `gps[i]` gives one point."""

    def __init__(self, arrays: cabi.EndpointArrays, lambda_min: float):
        self.status = arrays.status
        self.lambda_min = lambda_min
        self.lambda_max = arrays.lambda_max
        self.x_init, self.v_init = arrays.x_init, arrays.v_init
        self.x, self.v = arrays.x, arrays.v
        self.naccept, self.nreject, self.flags = arrays.naccept, arrays.nreject, arrays.flags

    def __len__(self):
        return len(self.status)

    def __getitem__(self, i):
        return dict(status=int(self.status[i]), lambda_min=self.lambda_min, lambda_max=float(self.lambda_max[i]),
                    x_init=self.x_init[:, i].copy(), x=self.x[:, i].copy(), v_init=self.v_init[:, i].copy(),
                    v=self.v[:, i].copy(), aux=None)


def _shards(n, ndev):
    """Contiguous ray blocks, one per device (SURVEY 8e)."""
    base, rem = divmod(n, ndev)
    out, first = [], 0
    for d in range(ndev):
        cnt = base + (1 if d < rem else 0)
        out.append((first, cnt))
        first += cnt
    return out


def _run_sharded(ensemble, n, fn, geometry=None):
    """Call fn(ctx, first, count, slot) for each device concurrently (ctypes drops the GIL)."""
    devs = ensemble.devices
    shards = [(i, d, f, c) for i, (d, (f, c)) in enumerate(zip(devs, _shards(n, len(devs)))) if c > 0]
    errs = []

    def work(i, dev, first, count):
        try:
            # a device listed twice gets two contexts: a context is used by one thread at a time
            ctx = ensemble.ctx(dev, devs[:i].count(dev))
            if geometry is not None and hasattr(geometry, "install"):
                geometry.install(ctx)
            fn(ctx, first, count, i)
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    if len(shards) <= 1:
        for sh in shards:
            work(*sh)
    else:
        ths = [threading.Thread(target=work, args=sh) for sh in shards]
        [t.start() for t in ths]
        [t.join() for t in ths]
    if errs:
        raise errs[0]
    return shards


def _install_on_comm(comm, geometry):
    if geometry is not None and hasattr(geometry, "install"):
        lib = cabi.load()
        for i in range(lib.gb200_comm_size(comm)):
            geometry.install(C.c_void_p(lib.gb200_comm_context(comm, i)))


def solve_tracing_problem(config: TracingConfiguration) -> GeodesicPoints:
    """`ensemble_solve_tracing_problem(::EnsembleB200, ...)`: the seam of src/tracing/tracing.jl:151-196."""
    p, ic = config.to_c()
    n = ic.n
    out = cabi.EndpointArrays(n)
    lib = cabi.load()

    def fn(ctx, first, count, slot):
        view = cabi.Endpoints()
        off = first
        view.status = C.cast(C.addressof(out.c.status.contents) + 4 * off, cabi._ip)
        view.lambda_max = C.cast(C.addressof(out.c.lambda_max.contents) + 8 * off, cabi._dp)
        for k in range(4):
            for name in ("x", "v", "x_init", "v_init"):
                src = getattr(out.c, name)[k]
                getattr(view, name)[k] = C.cast(C.addressof(src.contents) + 8 * off, cabi._dp)
        for name in ("naccept", "nreject", "flags"):
            setattr(view, name, C.cast(C.addressof(getattr(out.c, name).contents) + 4 * off, cabi._ip))
        rng = cabi.Range(first, count, 1)
        cabi.check(lib.gb200_trace(ctx, C.byref(p), C.byref(ic), C.byref(rng), C.byref(view)), ctx)

    _run_sharded(config.ensemble, n, fn, config.geometry)
    return GeodesicPoints(out, config.lambda_domain[0])


def trace_target(config: TracingConfiguration, target, d_tol=1e-2):
    """The objective of `optimize_for_target` (src/tracing/precision-solvers.jl:452-510) for every ray of `config` in one
    launch (`gb200_trace_target`): returns (closest approach to `target` = (r, θ, φ) per ray, GeodesicPoints).  Rays end
    where they first come within `d_tol` of the target (status IntersectedWithGeometry), like the reference's
    `distance_callback`."""
    p, ic = config.to_c()
    n = ic.n
    out = cabi.EndpointArrays(n)
    closest = np.zeros(n)
    tgt = np.ascontiguousarray(target, np.float64)
    if tgt.shape != (3,):
        raise ValueError("target must be (r, θ, φ)")
    ens = config.ensemble
    ctx = ens.ctx(ens.devices[0])
    rng = cabi.Range(0, n, 1)
    cabi.check(cabi.load().gb200_trace_target(ctx, C.byref(p), C.byref(ic), C.byref(rng), cabi.dptr(tgt), float(d_tol),
                                              C.byref(out.c), cabi.dptr(closest)), ctx)
    return closest, GeodesicPoints(out, config.lambda_domain[0])


def optimize_for_target(target, m, x0, *, d_tol=1e-2, max_time=None, p0=(0.0, 0.0), window=None, grid=33, max_rounds=10,
                        tracer=trace_target, **kwargs):
    """`optimize_for_target(target, m, x0; ...)` (src/tracing/precision-solvers.jl:512-531): impact parameters (α, β) of a
    geodesic from `x0` that passes within `d_tol` of `target` = (r, θ, φ).  Returns (α, β, geodesic point, accuracy) with
    accuracy = the closest approach reached.

    The reference minimises the closest approach one trace at a time (Optim.NelderMead from `p0`, a local search).  A
    device traces a thousand rays in the time of one, so the search here is a `grid` × `grid` patch of impact parameters
    per launch, centred on the best ray so far and shrunk to two cells of the previous patch each round, until the best
    ray is within `d_tol` (three to five launches).  The first patch spans ±`window` around `p0` (default: 1.5 r_target +
    10, which contains the direct image of the target for any viewing angle).  `tracer` exists for the tests (the CPU
    oracle in place of the device)."""
    x0 = [float(v) for v in x0]
    lam = 2.0 * x0[1] if max_time is None else float(max_time)
    half = float(window) if window is not None else 1.5 * float(target[0]) + 10.0
    ca, cb = float(p0[0]), float(p0[1])
    best = (np.inf, ca, cb, None)
    for _ in range(max_rounds):
        a1 = ca + np.linspace(-half, half, grid)
        b1 = cb + np.linspace(-half, half, grid)
        aa, bb = np.meshgrid(a1, b1, indexing="ij")
        cfg = tracing_configuration(m, x0, ImpactParameters(aa.ravel(), bb.ravel()), lam, trajectories=aa.size, **kwargs)
        closest, gps = tracer(cfg, target, d_tol)
        i = int(np.nanargmin(closest))
        if closest[i] < best[0]:
            best = (float(closest[i]), float(aa.ravel()[i]), float(bb.ravel()[i]), gps[i])
        if best[0] < d_tol:
            break
        ca, cb = best[1], best[2]
        half = 2.0 * (2.0 * half / (grid - 1))
    return best[1], best[2], best[3], best[0]


def impact_parameters_for_target(target, m, x0, **kwargs):
    """`impact_parameters_for_target` (src/tracing/precision-solvers.jl:533-543): (α, β, accuracy)."""
    a, b, _, acc = optimize_for_target(target, m, x0, **kwargs)
    return a, b, acc


def tracegeodesics_batch(configs: Sequence[TracingConfiguration]) -> list:
    """Many (short) ensembles in one call: every configuration is traced on its own stream of the first device's
    stream pool and the host synchronises once (SURVEY 8f-1; the reference calls `tracegeodesics` once per corona
    model, src/corona/models/lamp-post.jl:89-100).  Returns one `GeodesicPoints` per configuration."""
    if not configs:
        return []
    ens = configs[0].ensemble
    nb = len(configs)
    pcs = [c.to_c() for c in configs]
    problems = (cabi.Problem * nb)(*[pc[0] for pc in pcs])
    ics = (cabi.IC * nb)(*[pc[1] for pc in pcs])
    ranges = (cabi.Range * nb)(*[cabi.Range(0, pc[1].n, 1) for pc in pcs])
    arrays = [cabi.EndpointArrays(pc[1].n) for pc in pcs]
    outs = (cabi.Endpoints * nb)(*[a.c for a in arrays])
    ctx = ens.ctx(ens.devices[0])
    cabi.check(cabi.load().gb200_trace_batch(ctx, nb, problems, ics, ranges, outs), ctx)
    return [GeodesicPoints(a, c.lambda_domain[0]) for a, c in zip(arrays, configs)]


def trace_dual(config: TracingConfiguration, arrays: "cabi.DualArrays", norm_mode=cabi.DUAL_NORM_WITH_PARTIALS, plunging=None):
    """Forward-mode trace (`gb200_trace_dual`): the rays of `arrays` (impact parameters with seeded partials) through the
    problem `config` describes (metric, observer, geometry, chart, tolerances; its own velocity source is ignored).  What
    the reference does by pushing ForwardDiff duals through `_solve_reinit!` / `tracegeodesics`
    (src/tracing/precision-solvers.jl:73-131, 401-451).  Fills and returns `arrays`."""
    p, _ = config.to_c()
    ens = config.ensemble
    ctx = ens.ctx(ens.devices[0])
    pl_ref = C.byref(plunging.c) if plunging is not None else None
    cabi.check(cabi.load().gb200_trace_dual(ctx, C.byref(p), C.byref(arrays.ic), norm_mode, pl_ref, C.byref(arrays.out)), ctx)
    return arrays


def trace_dual_batch(configs: Sequence[TracingConfiguration], arrays: Sequence["cabi.DualArrays"], norm_mode=cabi.DUAL_NORM_WITH_PARTIALS,
                     plungings=None):
    """`trace_dual` for many (configuration, rays) pairs in one `gb200_trace_dual_batch` call (one launch per pair on the
    first device's stream pool, one staged copy each way)."""
    nb = len(configs)
    if nb == 0:
        return arrays
    ens = configs[0].ensemble
    problems = (cabi.Problem * nb)(*[c.to_c()[0] for c in configs])
    ics = (cabi.DualIC * nb)(*[a.ic for a in arrays])
    outs = (cabi.DualOut * nb)(*[a.out for a in arrays])
    pl_ptrs = None
    if plungings is not None and any(pl is not None for pl in plungings):
        PT = C.POINTER(cabi.PlungingTable)
        pl_ptrs = (PT * nb)(*[C.pointer(pl.c) if pl is not None else PT() for pl in plungings])
    ctx = ens.ctx(ens.devices[0])
    cabi.check(cabi.load().gb200_trace_dual_batch(ctx, nb, problems, ics, norm_mode, pl_ptrs, outs), ctx)
    return arrays


def tracegeodesics(m, position, velocity, *args, **kwargs) -> GeodesicPoints:
    """`tracegeodesics(m, x, v | plane | velfunc, [geometry], λ; kwargs...)` (src/tracing/tracing.jl:66-80)."""
    config = tracing_configuration(m, position, velocity, *args, **kwargs)
    return solve_tracing_problem(config)


# --------------------------------------------------------------------------- plunging region (non-Kerr redshift)
class PlungingInterpolation:
    """`PlungingInterpolation` (src/orbits/orbit-solving.jl:99-135) as data: r (ascending) -> (u^t, u^r, u^phi)."""

    def __init__(self, r, ut, ur, uphi):
        self.r, self.ut, self.ur, self.uphi = (np.ascontiguousarray(a, np.float64) for a in (r, ut, ur, uphi))
        self.c = cabi.PlungingTable(len(self.r), cabi.dptr(self.r), cabi.dptr(self.ut), cabi.dptr(self.ur), cabi.dptr(self.uphi))

    def __call__(self, r):
        x = np.clip(r, self.r[0], self.r[-1])  # _enforce_interpolation_bounds
        return np.interp(x, self.r, self.ut), np.interp(x, self.r, self.ur), np.interp(x, self.r, self.uphi)


_PLUNGING_CACHE = {}


def interpolate_plunging_velocities(m, ensemble=None, cap=1 << 17) -> PlungingInterpolation:
    """`interpolate_plunging_velocities(m)` (orbit-solving.jl:137-167): the massive plunging geodesic from the ISCO is
    integrated on the device (gb200_trace_path) and tabulated."""
    _check_metric(m)
    key = (type(m).__name__, m.params())
    if key in _PLUNGING_CACHE:
        return _PLUNGING_CACHE[key]
    ens = ensemble or default_ensemble()
    ctx = ens.ctx(ens.devices[0])
    arrs = [np.zeros(cap) for _ in range(4)]
    n = C.c_int32()
    cabi.check(cabi.load().gb200_build_plunging_table(ctx, m.kind, _metric_params_array(m), cap, *[cabi.dptr(a) for a in arrs], C.byref(n)), ctx)
    tab = PlungingInterpolation(*[a[: n.value] for a in arrs])
    _PLUNGING_CACHE[key] = tab
    return tab


def _auto_plunging(m, geometry, ensemble, want_redshift, plunging):
    """The reference's `redshift(m::AbstractMetric, u)` builds the plunging interpolation for every non-Kerr metric
    (const-point-functions.jl:79); here it is only needed when the disc reaches inside the ISCO."""
    if plunging is not None or not want_redshift or isinstance(m, KerrMetric):
        return plunging
    inner = getattr(geometry, "inner_radius", 0.0)
    try:
        if inner >= isco(m):
            return None
    except cabi.GradusB200Error:
        return None  # no ISCO (e.g. near-naked-singularity JP): redshift is undefined inside, NaN like a missing table
    return interpolate_plunging_velocities(m, ensemble)


# --------------------------------------------------------------------------- point functions
@dataclass(frozen=True)
class PointFunction:
    """A point function the device can evaluate at the ray endpoint (src/point-functions.jl:81-125)."""

    name: str
    filter: Optional[str] = None

    def __matmul__(self, other):  # pf ∘ filter
        if not isinstance(other, FilterPointFunction):
            raise TypeError("only composition with a FilterPointFunction is supported")
        return PointFunction(self.name, other.name)

    def kind(self):
        table = {
            ("affine_time", "early_term"): cabi.PF_SHADOW,
            ("redshift", "intersected"): cabi.PF_REDSHIFT,
            ("radius", "intersected"): cabi.PF_DISC_RADIUS,
            ("coordinate_time", "intersected"): cabi.PF_COORDINATE_TIME,
            ("status", None): cabi.PF_STATUS,
            ("affine_time", None): cabi.PF_AFFINE_TIME,
            ("radius", None): cabi.PF_RADIUS,
            ("equatorial_crossings", None): cabi.PF_EQUATORIAL_CROSSINGS,
            ("equatorial_crossings", "intersected"): cabi.PF_EQUATORIAL_CROSSINGS,  # filtered on the host, see apply_point_functions
        }
        key = (self.name, self.filter)
        if key not in table:
            raise ValueError(f"point function {key} has no device implementation")
        return table[key]


@dataclass(frozen=True)
class FilterPointFunction:
    name: str


class ConstPointFunctions:
    """src/const-point-functions.jl"""

    @staticmethod
    def filter_early_term():
        return FilterPointFunction("early_term")

    @staticmethod
    def filter_intersected():
        return FilterPointFunction("intersected")

    @staticmethod
    def affine_time():
        return PointFunction("affine_time")

    @staticmethod
    def shadow():
        return PointFunction("affine_time") @ FilterPointFunction("early_term")

    @staticmethod
    def redshift(m=None, u=None):
        return PointFunction("redshift")

    @staticmethod
    def radius():
        return PointFunction("radius")

    @staticmethod
    def coordinate_time():
        return PointFunction("coordinate_time")

    @staticmethod
    def equatorial_crossings():
        """The number of accepted integrator steps whose start and end differ in the sign of cos θ (GB200_PF_EQUATORIAL_
        CROSSINGS), unfiltered.  A disc hit reports the count at the start of its event step, so
        `equatorial_crossings() @ filter_intersected()` is the image order of each hit.  ThinDisc, ImageOrder or no
        geometry only."""
        return PointFunction("equatorial_crossings")


def _filter_on_host(pfs, kinds):
    """Point functions with no device filter of their own (the crossing count composed with `filter_intersected`):
    the status joins the device's list and the host masks the rays that did not hit.  Returns (device kinds, mask)."""
    masked = [k for k, f in enumerate(pfs) if (f.name, f.filter) == ("equatorial_crossings", "intersected")]
    if not masked:
        return kinds, None
    if len(kinds) >= 4:  # GB_MAX_PF
        raise ValueError("equatorial_crossings() @ filter_intersected() needs a free point-function slot (at most 3 others)")
    return np.append(kinds, np.int32(cabi.PF_STATUS)), masked


def _apply_host_filter(images, masked):
    if masked is None:
        return images
    miss = images[-1] != cabi.STATUS_INTERSECTED
    out = images[:-1].copy()
    for k in masked:
        out[k][miss] = np.nan
    return out


def impact_axes(width, height, alpha_lims, beta_lims):
    """src/rendering/utility.jl:43-47"""
    return np.linspace(alpha_lims[0], alpha_lims[1], width), np.linspace(beta_lims[0], beta_lims[1], height)


def _pop_alias(kwargs, names, default):
    for nme in names:
        if nme in kwargs:
            return kwargs.pop(nme)
    return default


def apply_point_functions(config, pfs, plunging=None):
    """Trace every ray of `config` and evaluate the point functions `pfs` at its endpoint in the same kernel
    (the fused form of `apply(pf, rendergeodesics(...))`, src/rendering/rendering.jl:64-107, for any velocity source
    including `ImpactParameters`).  Returns an array of shape (len(pfs), n_rays)."""
    kinds, masked = _filter_on_host(pfs, np.array([f.kind() for f in pfs], np.int32))
    p, ic = config.to_c()
    n = ic.n
    images = np.zeros((len(kinds), n))
    lib = cabi.load()
    plunging = _auto_plunging(config.metric, config.geometry, config.ensemble, cabi.PF_REDSHIFT in kinds, plunging)
    pl_ref = C.byref(plunging.c) if plunging is not None else None

    comm = config.ensemble.comm()
    if comm is not None:  # several GPUs: strips interleaved over the devices inside the library
        _install_on_comm(comm, config.geometry)
        ptrs = (cabi._dp * len(kinds))(*[cabi.dptr(images[k]) for k in range(len(kinds))])
        cabi.check(lib.gb200_comm_render(comm, C.byref(p), C.byref(ic), cabi.iptr(kinds), len(kinds), pl_ref, ptrs))
        return _apply_host_filter(images, masked)

    def fn(ctx, first, count, slot):
        ptrs = (cabi._dp * len(kinds))(*[C.cast(images[k].ctypes.data + 8 * first, cabi._dp) for k in range(len(kinds))])
        rng = cabi.Range(first, count, 1)
        cabi.check(lib.gb200_render(ctx, C.byref(p), C.byref(ic), C.byref(rng), cabi.iptr(kinds), len(kinds), pl_ref, ptrs), ctx)

    _run_sharded(config.ensemble, n, fn, config.geometry)
    return _apply_host_filter(images, masked)


def apply_point_functions_batch(configs: Sequence[TracingConfiguration], pfs, plungings=None) -> list:
    """`apply_point_functions` for many configurations in one `gb200_render_batch` call (one launch per configuration
    on the first device's stream pool, one staged copy each way).  Returns one (len(pfs), n_rays) array per
    configuration.  Used by the transfer-function table, where every probe round spans all (a, θ) cells."""
    if not configs:
        return []
    kinds, masked = _filter_on_host(pfs, np.array([f.kind() for f in pfs], np.int32))
    npf, nb = len(kinds), len(configs)
    ens = configs[0].ensemble
    pcs = [c.to_c() for c in configs]
    problems = (cabi.Problem * nb)(*[pc[0] for pc in pcs])
    ics = (cabi.IC * nb)(*[pc[1] for pc in pcs])
    ranges = (cabi.Range * nb)(*[cabi.Range(0, pc[1].n, 1) for pc in pcs])
    images = [np.zeros((npf, pc[1].n)) for pc in pcs]
    ptrs = (cabi._dp * (nb * npf))(*[C.cast(images[b][k].ctypes.data, cabi._dp) for b in range(nb) for k in range(npf)])
    pl_ptrs = None
    if plungings is not None and any(p is not None for p in plungings):
        PT = C.POINTER(cabi.PlungingTable)
        pl_ptrs = (PT * nb)(*[C.pointer(p.c) if p is not None else PT() for p in plungings])
    ctx = ens.ctx(ens.devices[0])
    cabi.check(cabi.load().gb200_render_batch(ctx, nb, problems, ics, ranges, cabi.iptr(kinds), npf, pl_ptrs, ptrs), ctx)
    return [_apply_host_filter(im, masked) for im in images]


def rendergeodesics(m, position, *args, pf=None, image_width=375, image_height=250, ensemble=None, plunging=None, **kwargs):
    """`rendergeodesics(m, x, [d], λ_max; pf, image_width, image_height, αlims, βlims, ensemble, ...)`
    (src/rendering/rendering.jl:28-54).  Returns (α, β, image) with image of shape (H, W).

    `pf` may also be a sequence of point functions: one fused trace, several images."""
    alpha_lims = _pop_alias(kwargs, ("αlims", "alpha_lims"), (-60, 60))
    beta_lims = _pop_alias(kwargs, ("βlims", "beta_lims"), (-40, 40))
    velocity = RenderGrid(int(image_width), int(image_height), tuple(alpha_lims), tuple(beta_lims))
    config = tracing_configuration(m, position, velocity, *args, ensemble=ensemble,
                                   trajectories=image_width * image_height, **kwargs)
    pfs = [ConstPointFunctions.shadow()] if pf is None else (list(pf) if isinstance(pf, (list, tuple)) else [pf])
    images = apply_point_functions(config, pfs, plunging=plunging)
    alpha, beta = impact_axes(image_width, image_height, alpha_lims, beta_lims)
    imgs = [images[k].reshape(image_width, image_height).T for k in range(len(pfs))]  # column-major (H, W)
    return (alpha, beta, imgs[0]) if not isinstance(pf, (list, tuple)) else (alpha, beta, imgs)


# --------------------------------------------------------------------------- endpoint caches
@dataclass
class EndpointCache:
    """`EndpointCache` (src/rendering/cache.jl): the `GeodesicPoint`s of an image, kept so that any number of point
    functions can be applied afterwards without tracing again."""

    metric: Any
    max_time: float
    height: int
    width: int
    points: GeodesicPoints


class HostPointFunction:
    """`PointFunction(f)` / `FilterPointFunction(f, default)` with user callables (src/point-functions.jl:81-125),
    evaluated on the host over a cache: `f(m, gps, max_time)` receives the whole `GeodesicPoints` SoA and returns one
    value (or one boolean, for a filter) per point.  `pf @ filt` is `pf ∘ filt`."""

    def __init__(self, f, default=None):
        self.f, self.default, self.inner = f, default, None

    def __matmul__(self, other):
        out = HostPointFunction(self.f, self.default)
        out.inner = other
        return out

    def __call__(self, m, gps, max_time):
        if self.default is not None:  # a filter on its own: pass mask
            return np.asarray(self.f(m, gps, max_time), bool)
        val = np.asarray(self.f(m, gps, max_time), np.float64)
        if self.inner is not None:
            keep = np.asarray(self.inner.f(m, gps, max_time), bool)
            val = np.where(keep, val, self.inner.default)
        return val


_HOST_FIELDS = {"affine_time": lambda m, g, t: g.lambda_max, "coordinate_time": lambda m, g, t: g.x[0],
                "radius": lambda m, g, t: g.x[1] * np.abs(np.sin(g.x[2])), "status": lambda m, g, t: g.status.astype(np.float64)}
_HOST_FILTERS = {"early_term": lambda m, g, t: g.lambda_max < t, "intersected": lambda m, g, t: g.status == StatusCodes.IntersectedWithGeometry}


def prerendergeodesics(m, position, *args, image_width=375, image_height=250, ensemble=None, **kwargs):
    """`prerendergeodesics(m, x, [d], λ_max; image_width, image_height, αlims, βlims, ...)` (src/rendering/rendering.jl:56-87).
    Returns (α, β, cache)."""
    alpha_lims = _pop_alias(kwargs, ("αlims", "alpha_lims"), (-60, 60))
    beta_lims = _pop_alias(kwargs, ("βlims", "beta_lims"), (-40, 40))
    velocity = RenderGrid(int(image_width), int(image_height), tuple(alpha_lims), tuple(beta_lims))
    config = tracing_configuration(m, position, velocity, *args, ensemble=ensemble, trajectories=image_width * image_height, **kwargs)
    gps = solve_tracing_problem(config)
    alpha, beta = impact_axes(image_width, image_height, alpha_lims, beta_lims)
    return alpha, beta, EndpointCache(m, config.lambda_domain[1], int(image_height), int(image_width), gps)


def apply(pf, cache: EndpointCache):
    """`apply(pf, cache)` (src/rendering/cache.jl): the (H, W) image of a point function over cached endpoints.  Accepts
    `HostPointFunction`s (user callables) and the built-in endpoint fields of `ConstPointFunctions`; the redshift needs the
    disc velocity field and is evaluated by the fused device path (`rendergeodesics(..., pf=redshift ∘ filter)`)."""
    gps = cache.points
    if isinstance(pf, HostPointFunction):
        vals = pf(cache.metric, gps, cache.max_time)
    elif isinstance(pf, PointFunction):
        if pf.name not in _HOST_FIELDS:
            raise ValueError(f"point function {pf.name!r} is evaluated on the device: use rendergeodesics(..., pf=...)")
        vals = np.asarray(_HOST_FIELDS[pf.name](cache.metric, gps, cache.max_time), np.float64)
        if pf.filter is not None:
            vals = np.where(_HOST_FILTERS[pf.filter](cache.metric, gps, cache.max_time), vals, np.nan)
    else:
        raise TypeError("apply expects a PointFunction or a HostPointFunction")
    return np.asarray(vals, np.float64).reshape(cache.width, cache.height).T  # column-major (H, W), rendering.jl:50


# --------------------------------------------------------------------------- line profiles
@dataclass(frozen=True)
class PowerLawEmissivity:
    """ε(r) = r^-index"""

    index: float = 3.0

    def __call__(self, r):
        return np.asarray(r, np.float64) ** -float(self.index)


@dataclass(frozen=True)
class TabulatedEmissivity:
    """ε(r) by linear interpolation in (r, eps), clamped to the ends"""

    r: Any
    eps: Any

    def __call__(self, r):
        rs = np.asarray(self.r, np.float64)
        return np.interp(np.clip(r, rs[0], rs[-1]), rs, np.asarray(self.eps, np.float64))


def _lineprofile_transfer_functions(bins, emissivity, m, position, d, method, min_re, max_re, ensemble, setup):
    """Transfer functions on the device (`tf_integration.transferfunctions`), integrated on the device
    (`gb200_tf_lineprofile`).  `min_re` / `max_re` given to `lineprofile` replace the method's."""
    from . import tf_integration as ti

    if not isinstance(emissivity, (PowerLawEmissivity, TabulatedEmissivity)):
        raise TypeError("an emissivity given as a Python callable cannot cross the C ABI: pass PowerLawEmissivity or "
                        "TabulatedEmissivity, or use tf_integration.lineprofile_transfer_functions")
    itb = ti.transferfunctions(m, position, d, min_re=method.min_re if min_re is None else min_re,
                               max_re=method.max_re if max_re is None else max_re, num_re=method.num_re, ensemble=ensemble,
                               **{**method.setup, **setup})
    return ti.integrate_lineprofiles(emissivity, itb, bins, h=method.h, n_radii=method.n_radii, ensemble=ensemble)[0]


def lineprofile(bins, emissivity, m, position, d, method=None, *, lambda_max=None, min_re=None, max_re=None,
                plane=None, callback="default", ensemble=None, bin_right_closed=False, plunging=None, **solver_args):
    """`lineprofile(bins, ε, m, u, d, ::BinningMethod; λ_max, minrₑ, maxrₑ, plane, callback, ...)`
    (src/line-profiles.jl:152-198), or with `TransferFunctionMethod(...)` (src/line-profiles.jl:121-150).  Returns
    (bins, flux ./ sum(flux))."""
    if method is not None and not isinstance(method, (BinningMethod, TransferFunctionMethod)):
        raise ValueError("method must be BinningMethod() or TransferFunctionMethod()")
    lambda_max = _pop_alias(solver_args, ("λ_max",), lambda_max)
    min_re = _pop_alias(solver_args, ("minrₑ",), min_re)
    max_re = _pop_alias(solver_args, ("maxrₑ",), max_re)
    bins = np.ascontiguousarray(bins, np.float64)
    if isinstance(method, TransferFunctionMethod):
        if lambda_max is not None or plane is not None or callback != "default" or bin_right_closed or plunging is not None:
            raise ValueError("λ_max, plane, callback, bin_right_closed and plunging belong to BinningMethod")
        return bins, _lineprofile_transfer_functions(bins, emissivity, m, position, d, method, min_re, max_re, ensemble, solver_args)
    if max_re is None:
        max_re = 50.0
    if lambda_max is None:
        lambda_max = 2 * position[1]
    if min_re is None:
        min_re = isco(m)
    if plane is None:
        plane = PolarPlane(GeometricGrid(), Nr=450, Ntheta=1300, r_max=5 * max_re)
    if callback == "default":
        callback = domain_upper_hemisphere()
    config = tracing_configuration(m, position, plane, d, (0.0, lambda_max), callback=callback, ensemble=ensemble,
                                   **solver_args)
    p, ic = config.to_c()
    n = ic.n
    lib = cabi.load()
    emis = cabi.Emissivity()
    keep = []
    if isinstance(emissivity, PowerLawEmissivity):
        emis.kind, emis.index = cabi.EMISSIVITY_POWERLAW, float(emissivity.index)
    elif isinstance(emissivity, TabulatedEmissivity):
        r = np.ascontiguousarray(emissivity.r, np.float64)
        e = np.ascontiguousarray(emissivity.eps, np.float64)
        keep += [r, e]
        emis.kind, emis.n, emis.r, emis.eps = cabi.EMISSIVITY_TABLE, len(r), cabi.dptr(r), cabi.dptr(e)
    else:
        raise ValueError("emissivity must be PowerLawEmissivity or TabulatedEmissivity (a closure cannot cross the C ABI)")
    opts = cabi.LineProfileOpts(float(min_re), float(max_re), 0, 1 if bin_right_closed else 0)
    plunging = _auto_plunging(m, d, config.ensemble, min_re < (isco(m) if not isinstance(m, KerrMetric) else 0.0), plunging)
    pl_ref = C.byref(plunging.c) if plunging is not None else None
    comm = config.ensemble.comm()
    if comm is not None:  # several GPUs: sharded inside the library, histograms summed with one NCCL all-reduce
        _install_on_comm(comm, config.geometry)
        flux = np.zeros(len(bins))
        opts.normalise = 1
        cabi.check(lib.gb200_comm_lineprofile(comm, C.byref(p), C.byref(ic), C.byref(emis), pl_ref, cabi.dptr(bins), len(bins), C.byref(opts),
                                              cabi.dptr(flux)))
        return bins, flux
    ndev = len(config.ensemble.devices)
    partial = np.zeros((ndev, len(bins)))

    def fn(ctx, first, count, slot):
        rng = cabi.Range(first, count, 1)
        cabi.check(lib.gb200_lineprofile(ctx, C.byref(p), C.byref(ic), C.byref(rng), C.byref(emis), pl_ref,
                                         cabi.dptr(bins), len(bins), C.byref(opts), cabi.dptr(partial[slot])), ctx)

    _run_sharded(config.ensemble, n, fn, config.geometry)
    flux = partial.sum(axis=0)  # fixed device order: deterministic
    return bins, flux / flux.sum()
