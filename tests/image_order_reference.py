"""CPU reference for equatorial crossings and photon-ring image orders (test infrastructure).

The definitions of include/gradus_b200.h (GB200_PF_EQUATORIAL_CROSSINGS, GB200_GEOMETRY_THIN_DISC_ORDER) restated on top
of the CPU oracle's own pieces: the oracle integrates each ray with no geometry and records every accepted step
(`oracle.trace_path`), which is the step sequence of the ray under any disc too (a disc only ends a ray, it never changes
its steps).  This module then
  * counts the sign changes of cos(theta) between consecutive step ends (cos >= 0 counting as positive);
  * replays the oracle's ContinuousCallback on those steps: the Tsit5 stages are recomputed from the recorded u_prev and
    dt with the oracle's right-hand side (`oracle.rhs`) in the oracle's order of operations -- the recomputed step end is
    checked bitwise against the recorded one --, then the sign test at the step end, the interior samples at
    Theta = 1/7 .. 6/7 and the left-biased bisection on the dense output, exactly as `trace_ray` does them.
With `order = None` the replay is the oracle's ThinDisc (every sign change of the condition is an event), which the tests
hold bitwise against `oracle.trace` of the same ThinDisc problem; with `order = n` only a wedge entry in a step that starts
with n crossings is one.  Double precision throughout; `precision = 1` replays the long-double oracle's step sequence (its
states rounded to double), the rounding-perturbed run that defines the band."""
import math
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from gradus_b200 import _cabi as cabi
from oracle import oracle

A21 = 0.161
A31, A32 = -0.008480655492356989, 0.335480655492357
A41, A42, A43 = 2.8971530571054935, -6.359448489975075, 4.3622954328695815
A51, A52, A53, A54 = 5.325864828439257, -11.748883564062828, 7.4955393428898365, -0.09249506636175525
A61, A62, A63, A64, A65 = 5.86145544294642, -12.92096931784711, 8.159367898576159, -0.071584973281401, -0.028269050394068383
A71, A72, A73, A74, A75, A76 = 0.09646076681806523, 0.01, 0.4798896504144996, 1.379008574103742, -3.290069515436081, 2.324710524099774
R11, R12, R13, R14 = 1.0, -2.763706197274826, 2.9132554618219126, -1.0530884977290216
R22, R23, R24 = 0.13169999999999998, -0.2234, 0.1017
R32, R33, R34 = 3.9302962368947516, -5.941033872131505, 2.490627285651253
R42, R43, R44 = -12.411077166933676, 30.33818863028232, -16.548102889244902
R52, R53, R54 = 37.50931341651104, -88.1789048947664, 47.37952196281928
R62, R63, R64 = -27.896526289197286, 65.09189467479366, -34.87065786149661
R72, R73, R74 = 1.5, -4.0, 2.5


def _copy(p):
    return cabi.Problem.from_buffer_copy(p)


class _Ray:
    """One ray's transparent trajectory: u[0] = initial state, u[i] = end of the i-th accepted step (t[i], dt[i])."""

    def __init__(self, p_none, u0, precision):
        cap = 4096
        while True:
            t, dt, _, u = oracle.trace_path(p_none, u0, precision=precision, cap=cap)
            if len(t) < cap:
                break
            cap *= 4
        self.u = np.vstack([u0[None, :], u])
        self.dt = dt
        # integrator.t after each step (fixed_t_for_floatingpoint_error!: a step that lands within 100 eps of tstop is tstop)
        tstop = p_none.lambda_max
        ts = [p_none.lambda_min]
        for d in dt:
            tt = ts[-1] + d
            big = max(ts[-1], tstop)
            epsb = np.nextafter(abs(big), np.inf) - abs(big)
            ts.append(tstop if abs(tt - tstop) < 100.0 * epsb else tt)
        self.t = np.array(ts)
        self.cpos = np.cos(self.u[:, 2]) >= 0.0
        # a step whose ends are both further than 4 gtol from the equator, by more than the step moves theta, cannot
        # reach the wedge |cos theta| <= gtol at an interior sample (the oracle's own band_ratio skips these steps)
        c = np.abs(np.cos(self.u[:, 2]))
        self.far = (self.cpos[1:] == self.cpos[:-1]) & (np.minimum(c[1:], c[:-1]) - np.abs(np.diff(self.u[:, 2])) > 0.0)
        self.exact = precision == 0


def _rhs(p, u):
    return oracle.rhs(p.metric_kind, list(p.metric_params), u)


def _stages(p, uprev, dt):
    k0 = _rhs(p, uprev)
    k1 = _rhs(p, uprev + (dt * A21) * k0)
    k2 = _rhs(p, uprev + dt * (A31 * k0 + A32 * k1))
    k3 = _rhs(p, uprev + dt * (A41 * k0 + A42 * k1 + A43 * k2))
    k4 = _rhs(p, uprev + dt * (A51 * k0 + A52 * k1 + A53 * k2 + A54 * k3))
    k5 = _rhs(p, uprev + dt * (A61 * k0 + A62 * k1 + A63 * k2 + A64 * k3 + A65 * k4))
    u = uprev + dt * (A71 * k0 + A72 * k1 + A73 * k2 + A74 * k3 + A75 * k4 + A76 * k5)
    k6 = _rhs(p, u)
    return (k0, k1, k2, k3, k4, k5, k6), u


def _interp(Th, dt, y0, k):
    Th2 = Th * Th
    b1 = Th * (R11 + Th * (R12 + Th * (R13 + Th * R14)))
    b2 = Th2 * (R22 + Th * (R23 + Th * R24))
    b3 = Th2 * (R32 + Th * (R33 + Th * R34))
    b4 = Th2 * (R42 + Th * (R43 + Th * R44))
    b5 = Th2 * (R52 + Th * (R53 + Th * R54))
    b6 = Th2 * (R62 + Th * (R63 + Th * R64))
    b7 = Th2 * (R72 + Th * (R73 + Th * R74))
    return y0 + dt * (k[0] * b1 + k[1] * b2 + k[2] * b3 + k[3] * b4 + k[4] * b5 + k[5] * b6 + k[6] * b7)


def _cond(p, y):
    """distance_to_disc of the thin disc (thin-disc.jl:20-26, the oracle's disc_condition)."""
    r, th = float(y[1]), float(y[2])
    rho = r * abs(math.sin(th))
    if rho < p.geometry_params[0] or rho > p.geometry_params[1]:
        return 1.0
    return r * abs(math.cos(th)) - p.gtol * abs(r)


def _sgn(x):
    return int(x > 0) - int(x < 0)


def _event_in_step(p, ray, i):
    """The oracle's ContinuousCallback on step i (u[i-1] -> u[i]) given that its sign test is armed: (event, state)."""
    uprev, u, dt, tprev, t = ray.u[i - 1], ray.u[i], ray.dt[i - 1], ray.t[i - 1], ray.t[i]
    cprev, cnext = _cond(p, uprev), _cond(p, u)
    sprev, snext = _sgn(cprev), _sgn(cnext)
    k = None
    bottom, top = tprev, t
    if sprev * snext <= 0:
        event = True
    else:
        event = False
        if ray.far[i - 1] and np.min(np.abs(np.cos(ray.u[i - 1:i + 1, 2]))) - abs(ray.u[i, 2] - ray.u[i - 1, 2]) > 4.0 * p.gtol:
            return False, None, None
        k, ue = _stages(p, uprev, dt)
        assert not ray.exact or np.array_equal(ue, u), "the recomputed step end differs from the oracle's"
        last = tprev
        for j in range(2, 9):
            abst = t if j == 8 else tprev + ((j - 1) * (t - tprev)) / 7.0
            cnew = cnext if j == 8 else _cond(p, _interp((abst - tprev) / dt, dt, uprev, k))
            if sprev * cnew < 0:
                event, bottom, top = True, last, abst
                break
            last = abst
    if not event:
        return False, None, None
    if k is None:
        k, ue = _stages(p, uprev, dt)
        assert not ray.exact or np.array_equal(ue, u), "the recomputed step end differs from the oracle's"

    def zf(abst):
        if abst == t:
            return _cond(p, u)
        if abst == tprev:
            return cprev
        return _cond(p, _interp((abst - tprev) / dt, dt, uprev, k))

    if zf(top) == 0.0:
        tev = top
    else:
        lo, hi = bottom, top
        for _ in range(200):
            mid = lo + (hi - lo) / 2.0
            if not (lo < mid < hi):
                break
            cm = zf(mid)
            if cm == 0.0:
                hi = mid
                continue
            if (cm > 0) == (sprev > 0):
                lo = mid
            else:
                hi = mid
        tev = lo
    ue = u.copy() if tev == t else _interp((tev - tprev) / dt, dt, uprev, k)
    return True, ue, tev


def _discrete_status(p, u):
    status = cabi.STATUS_INTERSECTED
    if p.callback_kind == cabi.CALLBACK_UPPER_HEMISPHERE and u[1] * math.cos(u[2]) < p.callback_delta:
        status = cabi.STATUS_OUT_OF_DOMAIN
    if u[1] <= p.chart_inner:
        status = cabi.STATUS_WITHIN_INNER_BOUNDARY
    elif u[1] > p.chart_outer:
        status = cabi.STATUS_OUT_OF_DOMAIN
    return status


def _one(p, ray, none_status, order, thin):
    """(status, lambda, u_end[8], crossings) of one ray; thin: the disc is present (ThinDisc or its order)."""
    n = len(ray.dt)
    crossings = 0
    for i in range(1, n + 1):
        if thin:
            sprev = _sgn(_cond(p, ray.u[i - 1]))
            armed = (sprev > 0 and crossings == order) if order is not None else sprev != 0
            if armed:
                hit, ue, tev = _event_in_step(p, ray, i)
                if hit:
                    return _discrete_status(p, ue), tev, ue, crossings
        crossings += int(ray.cpos[i] != ray.cpos[i - 1])
    return none_status, ray.t[-1], ray.u[-1], crossings


def trace_orders(p, ic, orders, precision=0, threads=16):
    """Per entry of `orders` (None = the plain ThinDisc, n = the order-n image; p's geometry kind NONE: counts only), a dict
    of per-ray status, lam, x (4, N), v (4, N), x_init, v_init, crossings.  One transparent trajectory serves them all."""
    thin = p.geometry_kind in (cabi.GEOMETRY_THIN_DISC, cabi.GEOMETRY_THIN_DISC_ORDER)
    q = _copy(p)
    q.geometry_kind = cabi.GEOMETRY_NONE
    q.geometry_params[2] = 0.0
    ep = oracle.trace(q, ic, precision=0)  # initial states and the transparent terminations
    ep_l = oracle.trace(q, ic, precision=1) if precision == 1 else ep
    N = ep.x.shape[1]
    outs = [dict(status=np.zeros(N, np.int32), lam=np.zeros(N), x=np.zeros((4, N)), v=np.zeros((4, N)),
                 crossings=np.zeros(N, int), x_init=ep.x_init.copy(), v_init=ep.v_init.copy()) for _ in orders]

    def work(i):
        u0 = np.concatenate([ep.x_init[:, i], ep.v_init[:, i]])
        ray = _Ray(q, u0, precision)
        for order, out in zip(orders, outs):
            st, lam, ue, c = _one(p, ray, int(ep_l.status[i]), order, thin)
            out["status"][i], out["lam"][i], out["crossings"][i] = st, lam, c
            out["x"][:, i], out["v"][:, i] = ue[:4], ue[4:]

    with ThreadPoolExecutor(threads) as pool:
        list(pool.map(work, range(N)))
    return outs


def trace(p, ic, order=None, precision=0):
    """`trace_orders` for one entry; a THIN_DISC_ORDER problem brings its own order."""
    if p.geometry_kind == cabi.GEOMETRY_THIN_DISC_ORDER and order is None:
        order = int(p.geometry_params[2])
    return trace_orders(p, ic, [order], precision)[0]


def kerr_redshift(p, ref):
    """redshift_function(::KerrMetric, gp) (src/redshift.jl:93-220) as the oracle's redshift_of states it; NaN off the disc."""
    assert p.metric_kind == cabi.METRIC_KERR
    M, a = p.metric_params[0], p.metric_params[1]
    mp = [M, a]
    risco = oracle.isco(cabi.METRIC_KERR, mp)
    g = np.full(ref["x"].shape[1], np.nan)
    for i in np.where(ref["status"] == cabi.STATUS_INTERSECTED)[0]:
        x, v, x0, v0 = ref["x"][:, i], ref["v"][:, i], ref["x_init"][:, i], ref["v_init"][:, i]
        rho = x[1] * abs(math.sin(x[2]))
        if rho < risco:
            rms, r = risco, rho
            sM = math.sqrt(M)
            Le = sM * (rms * rms - 2 * a * math.sqrt(M * rms) + a * a) / (rms * math.sqrt(rms) - 2 * M * math.sqrt(rms) + a * sM)
            Delta = r * r - 2 * M * r + a * a
            H = (2 * M * r - a * Le) / Delta
            ge = math.sqrt(1 - (2 * M) / (3 * rms))
            qq = rms / r - 1
            ur = -math.sqrt((2 * M) / (3 * rms)) * (qq * math.sqrt(qq))
            vd = [ge * (1 + 2 * M * (1 + H) / r), -ur, 0.0, ge / (r * r) * (Le + a * H)]
        else:
            vd = oracle.circular_fourvelocity(cabi.METRIC_KERR, mp, rho)
        gd = oracle.metric(cabi.METRIC_KERR, mp, x[1], x[2])[0]
        go = oracle.metric(cabi.METRIC_KERR, mp, x0[1], x0[2])[0]
        Ed = (gd[0] * v[0] + gd[4] * v[3]) * vd[0] + (gd[1] * v[1]) * vd[1] + (gd[2] * v[2]) * vd[2] + (gd[4] * v[0] + gd[3] * v[3]) * vd[3]
        Eo = go[0] * v0[0] + go[4] * v0[3]
        g[i] = Eo / Ed
    return g


def disc_radius(ref):
    hit = ref["status"] == cabi.STATUS_INTERSECTED
    return np.where(hit, ref["x"][1] * np.abs(np.sin(ref["x"][2])), np.nan)


def band(ref, alt):
    """Rounding-sensitive rays: status, crossing count or hit state (beyond 3e-7) differ between the replays of the double
    (`ref`) and of the long-double (`alt`, precision = 1) oracle's step sequences."""
    moved = (alt["status"] != ref["status"]) | (alt["crossings"] != ref["crossings"])
    both = (alt["status"] == cabi.STATUS_INTERSECTED) & (ref["status"] == cabi.STATUS_INTERSECTED)
    dx = np.abs(alt["x"][1:3] - ref["x"][1:3]) / np.maximum(np.abs(ref["x"][1:3]), 1.0)
    return moved | (both & (dx.max(axis=0) > 3e-7))


def polar_plane_area(ic):
    """The image-plane area weight r^2 of each ray of a PolarPlane (planes.jl:93-115, the oracle's ic_for_ray)."""
    Nr, Nt = ic.width, ic.height
    k = np.arange(ic.n) % Nr
    lo, hi = ic.lo0, ic.hi0
    if ic.grid_kind == cabi.GRID_GEOMETRIC:
        K = math.pow(hi / lo, 1.0 / (Nr - 1))
        r = np.array([lo * math.pow(K, float(kk)) for kk in k])
    else:
        raise ValueError("only the geometric grid is restated here")
    return r * r


def lineprofile(p, ic, ref, bins, index, min_re, max_re):
    """lineprofile(::BinningMethod) (line-profiles.jl:186-197) of the replayed end points: r^-index emissivity, Buckets.Simple
    bins (searchsortedlast, clamped), summed in ray order and normalised."""
    g = kerr_redshift(p, ref)
    rho = disc_radius(ref)
    area = polar_plane_area(ic)
    flux = np.zeros(len(bins))
    for i in range(len(g)):
        if not (g[i] == g[i]) or not (min_re <= rho[i] <= max_re):
            continue
        b = min(max(int(np.searchsorted(bins, g[i], side="right")) - 1, 0), len(bins) - 1)
        flux[b] += rho[i] ** -index * g[i] * g[i] * g[i] * area[i]
    return flux / flux.sum()
