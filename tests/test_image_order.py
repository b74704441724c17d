"""Equatorial crossings (GB200_PF_EQUATORIAL_CROSSINGS) and photon-ring image orders (GB200_GEOMETRY_THIN_DISC_ORDER,
`gb.ImageOrder(ThinDisc, n)`).

Pins.  (1) An independent closed form: in Schwarzschild every ray stays in the plane through the hole, its observer and its
initial momentum; the in-plane angle swept between the observer and the end radius follows from the orbit equation
(du/dpsi)^2 = 1/b^2 - u^2 + 2 M u^3 alone, and cos(theta) along the orbit is cos(theta_o) cos(psi) - sin(theta_o) sin(psi)
k^theta / k_perp, so the count is the number of its zeros.  (2) The definitions themselves: a ray that hits ThinDisc with
count c takes the same steps and the same event step under ImageOrder(., c), so both give the same end point.  (3) Device
against the oracle outside the grazing band, which here also holds the rays whose count moves between the double and
long-double runs.  The CPU side of (2) and (3) is `image_order_reference`: the definitions replayed on the oracle's own
recorded step sequences, itself held bitwise to the oracle's ThinDisc."""
import ctypes as C
import math

import numpy as np
import pytest

import gradus_b200 as gb
from gradus_b200 import _cabi as cabi
from gradus_b200 import api
from oracle import oracle

import common
import image_order_reference as reference

M = 1.0
THETAS = (17.0, 60.0)


# --------------------------------------------------------------------------- the closed form (Schwarzschild)
def _schwarzschild_rays(theta_deg, n=300, seed=0):
    rng = np.random.default_rng(seed + int(theta_deg))
    alpha = rng.uniform(-12.0, 12.0, n)
    beta = rng.uniform(-12.0, 12.0, n)
    m = gb.KerrMetric(M, 0.0)
    x = [0.0, 1000.0, math.radians(theta_deg), 0.0]
    return m, x, api.tracing_configuration(m, x, api.ImpactParameters(alpha, beta), 2000.0, trajectories=n)


def _psi_between(u_obs, u_end, b, outgoing_end):
    """In-plane angle swept from u_obs to u_end along (du/dpsi)^2 = f(u) = 2M u^3 - u^2 + 1/b^2, through the periapsis u_p
    (the smallest positive root of f) when there is one.  Near u_p, u = u_p - s^2 turns the integrand into the smooth
    2 / sqrt(2M (u_p - s^2 - u_neg)(u_3 - u_p + s^2))."""
    from scipy.integrate import quad

    roots = np.roots([2.0 * M, -1.0, 0.0, 1.0 / b**2])
    real = np.sort(roots[np.abs(roots.imag) < 1e-12].real)
    pos = real[real > 0]
    if len(pos) == 0 or pos[0] < u_end:  # no turning point before the end radius: plunges (or ends on the way in)
        val, _ = quad(lambda u: 1.0 / math.sqrt(2.0 * M * u**3 - u**2 + 1.0 / b**2), u_obs, u_end, epsabs=1e-13, epsrel=1e-12, limit=400)
        return val
    u_neg, u_p = real[0], pos[0]
    u_3 = pos[1] if len(pos) > 1 else np.inf

    def tail(u):  # integral from u to u_p
        g = lambda s: 2.0 / math.sqrt(2.0 * M * (u_p - s * s - u_neg) * (u_3 - u_p + s * s))
        val, _ = quad(g, 0.0, math.sqrt(max(u_p - u, 0.0)), epsabs=1e-13, epsrel=1e-12, limit=400)
        return val

    return tail(u_obs) + tail(u_end) if outgoing_end else tail(u_obs) - tail(u_end)


def _closed_form_counts(ep, theta_o):
    """(count, excluded) per ray from the ray's own initial state and end radius."""
    counts = np.zeros(ep.x.shape[1], int)
    excluded = np.zeros(ep.x.shape[1], bool)
    for i in range(ep.x.shape[1]):
        r0, th0 = ep.x_init[1, i], ep.x_init[2, i]
        vt, vth, vph = ep.v_init[0, i], ep.v_init[2, i], ep.v_init[3, i]
        kperp = math.sqrt(vth**2 + math.sin(th0) ** 2 * vph**2)
        L, E = r0 * r0 * kperp, (1.0 - 2.0 * M / r0) * vt
        b = L / E
        psi_end = _psi_between(1.0 / r0, 1.0 / ep.x[1, i], b, ep.v[1, i] > 0)
        A, B = math.cos(theta_o), math.sin(theta_o) * vth / kperp  # cos(theta) = A cos(psi) - B sin(psi) = R cos(psi + delta)
        delta = math.atan2(B, A)
        ks = np.arange(math.floor((delta - math.pi / 2) / math.pi) - 1, math.ceil((psi_end + delta) / math.pi) + 2)
        zeros = math.pi / 2 + ks * math.pi - delta
        counts[i] = int(np.sum((zeros > 0) & (zeros < psi_end)))
        excluded[i] = bool(np.any(np.abs(zeros) < 1e-5) or np.any(np.abs(zeros - psi_end) < 1e-5))
    return counts, excluded


def _check_closed_form(theta_deg, render):
    m, x, cfg = _schwarzschild_rays(theta_deg)
    p, ic = cfg.to_c()
    ep = oracle.trace(p, ic)
    got = render(cfg, p, ic)
    want, excluded = _closed_form_counts(ep, math.radians(theta_deg))
    ok = ~excluded
    print(f"theta_o = {theta_deg} deg: {excluded.sum()} of {len(ok)} rays excluded (a zero within 1e-5 rad of an end); "
          f"counts {np.bincount(want[ok])}")
    assert excluded.sum() < 0.05 * len(ok)
    assert np.array_equal(got[ok], want[ok]), np.where(got[ok] != want[ok])[0][:10]
    assert want[ok].max() >= 2  # rays that wind around the hole are part of the sample


@pytest.mark.parametrize("theta_deg", THETAS)
def test_oracle_count_against_the_schwarzschild_orbit_equation(theta_deg):
    _check_closed_form(theta_deg, lambda cfg, p, ic: reference.trace(p, ic)["crossings"])


# --------------------------------------------------------------------------- the definitions, on the oracle
SUBRING_WINDOW = dict(alims=(-3.2, -2.0), blims=(-1.5, 1.5))  # across the critical curve left of the hole (C1 observer)


def _order_config(n, w, h, **window):
    m, x, d, _ = common.c1(8, 8)
    return common.render_config(m, x, gb.ImageOrder(d, n), 2000.0, w, h, **window)


def _fields(ref, p):
    return np.stack([ref["status"], ref["lam"], *ref["x"], *ref["v"], ref["crossings"], reference.kerr_redshift(p, ref)])


def test_reference_replays_the_oracle_thin_disc_and_its_orders():
    """The replay with every sign change an event is the oracle's ThinDisc bit for bit; each ThinDisc hit with count c is
    bit for bit its order-c hit; an order-n hit always reports count n."""
    m, x, d, cfg = common.c1(48, 48)
    p, ic = cfg.to_c()
    ep = oracle.trace(p, ic)
    thin, *orders = reference.trace_orders(p, ic, [None, 0, 1, 2])
    assert np.array_equal(thin["status"], ep.status) and np.array_equal(thin["lam"], ep.lambda_max)
    assert np.array_equal(thin["x"], ep.x) and np.array_equal(thin["v"], ep.v)
    assert np.array_equal(reference.kerr_redshift(p, thin), oracle.render(p, ic, [cabi.PF_REDSHIFT])[0], equal_nan=True)
    hit = thin["status"] == cabi.STATUS_INTERSECTED
    assert hit.sum() > 500
    for c, ref_c in enumerate(orders):
        sel = hit & (thin["crossings"] == c)
        assert np.array_equal(_fields(ref_c, p)[:, sel], _fields(thin, p)[:, sel])
    pw, icw = _order_config(0, 32, 32, **SUBRING_WINDOW).to_c()
    for n, ref_n in enumerate(reference.trace_orders(pw, icw, [0, 1, 2])):
        h = ref_n["status"] == cabi.STATUS_INTERSECTED
        assert h.sum() > 0 and np.all(ref_n["crossings"][h] == n)


# --------------------------------------------------------------------------- validation (no device needed)
def _validate(p, ic):
    return cabi.load().gb200_validate(C.byref(p), C.byref(ic))


def test_validation_of_the_order_and_of_the_crossings_point_function():
    lib = cabi.load()
    cfg = _order_config(1, 8, 8)
    p, ic = cfg.to_c()
    assert _validate(p, ic) == cabi.OK
    for bad in (-1.0, 0.5, float("nan"), float("inf"), 2.0**31):
        p.geometry_params[2] = bad
        assert _validate(p, ic) == cabi.ERR_INVALID_ARGUMENT, bad
    p.geometry_params[2] = 2.0
    p.geometry_params[0], p.geometry_params[1] = 50.0, 10.0
    assert _validate(p, ic) == cabi.ERR_INVALID_ARGUMENT
    p.geometry_params[0], p.geometry_params[1] = 0.0, 50.0
    # the generic integrator has no order rule: the forward-mode, target and path entry points refuse the kind
    dic = cabi.DualIC()
    assert lib.gb200_trace_dual(None, C.byref(p), C.byref(dic), 0, None, None) == cabi.ERR_UNSUPPORTED
    tgt = np.array([10.0, 1.0, 0.0])
    assert lib.gb200_trace_target(None, C.byref(p), C.byref(ic), None, cabi.dptr(tgt), 1e-2, None, None) == cabi.ERR_UNSUPPORTED
    u0, lam, u = np.zeros(8), np.zeros(4), np.zeros(32)
    nrows, status = C.c_int32(), C.c_int32()
    assert lib.gb200_trace_path(None, C.byref(p), cabi.dptr(u0), 4, cabi.dptr(lam), cabi.dptr(u), C.byref(nrows), C.byref(status)) == cabi.ERR_UNSUPPORTED
    # the crossings point function: no geometry, ThinDisc and ImageOrder only
    pfs = np.array([cabi.PF_EQUATORIAL_CROSSINGS], np.int32)
    img = np.zeros(64)
    ptrs = (cabi._dp * 1)(cabi.dptr(img))
    rng = cabi.Range(0, 64, 1)
    m = gb.KerrMetric(1.0, 0.9)
    x = [0.0, 1000.0, math.radians(60.0), 0.0]
    rough = gb.ThickDisc(lambda rho: np.where((rho > 9) & (rho < 11), np.sqrt(np.maximum(1 - (rho - 10) ** 2, 0)), 0.0), (9.0, 11.0), n=64)
    for d in (gb.ShakuraSunyaev(m), gb.DatumPlane(1.0), rough):
        pd, icd = common.render_config(m, x, d, 2000.0, 8, 8).to_c()
        assert _validate(pd, icd) == cabi.OK
        assert lib.gb200_render(None, C.byref(pd), C.byref(icd), C.byref(rng), cabi.iptr(pfs), 1, None, ptrs) == cabi.ERR_UNSUPPORTED
        dptrs = (C.c_void_p * 1)(img.ctypes.data)
        assert lib.gb200_render_device(None, C.byref(pd), C.byref(icd), C.byref(rng), cabi.iptr(pfs), 1, None, dptrs, None, 0) == cabi.ERR_UNSUPPORTED
        assert lib.gb200_render_batch(None, 1, C.byref(pd), C.byref(icd), C.byref(rng), cabi.iptr(pfs), 1, None, ptrs) == cabi.ERR_UNSUPPORTED
    for d in (None, gb.ThinDisc(0.0, 50.0), gb.ImageOrder(gb.ThinDisc(0.0, 50.0), 1)):
        pd, icd = common.render_config(m, x, d, 2000.0, 8, 8).to_c()
        assert lib.gb200_render(None, C.byref(pd), C.byref(icd), C.byref(rng), cabi.iptr(pfs), 1, None, ptrs) == cabi.ERR_INVALID_ARGUMENT  # null context


def test_python_mirror():
    d = gb.ThinDisc(0.0, 50.0)
    assert gb.ImageOrder(d, 2).to_c() == (cabi.GEOMETRY_THIN_DISC_ORDER, (0.0, 50.0, 2.0, 0.0))
    for bad in (-1, 1.0, 0.5, True, "1"):
        with pytest.raises(ValueError):
            gb.ImageOrder(d, bad)
    with pytest.raises(ValueError):
        gb.ImageOrder(gb.DatumPlane(0.0), 0)
    pf = gb.ConstPointFunctions.equatorial_crossings()
    assert pf.kind() == cabi.PF_EQUATORIAL_CROSSINGS
    assert (pf @ gb.ConstPointFunctions.filter_intersected()).kind() == cabi.PF_EQUATORIAL_CROSSINGS
    m, x = gb.KerrMetric(1.0, 0.998), [0.0, 1000.0, math.radians(60.0), 0.0]
    with pytest.raises(ValueError):  # transfer functions: the same error as for any other unsupported geometry
        gb.DeviceProber(m, x, gb.ImageOrder(d, 1))
    from gradus_b200 import corona
    with pytest.raises(ValueError):
        corona.tracecorona(m, gb.ImageOrder(d, 1), corona.LampPostModel(h=10.0))


# --------------------------------------------------------------------------- on the device
def _device_counts(cfg, p, ic):
    return api.apply_point_functions(cfg, [gb.ConstPointFunctions.equatorial_crossings()])[0].astype(int)


def _count_band(p, ic):
    """Rays whose crossing count or end state is rounding-sensitive: the count or status moves between the replays of the
    oracle's double and long-double step sequences."""
    ref = reference.trace(p, ic)
    return ref, reference.band(ref, reference.trace(p, ic, precision=1))


@pytest.mark.gpu
@pytest.mark.parametrize("theta_deg", THETAS)
def test_device_count_against_the_schwarzschild_orbit_equation(theta_deg):
    _check_closed_form(theta_deg, _device_counts)


@pytest.mark.gpu
# the band may hold at most 1.5 x the rays measured in it on a B200 run (C1 window 0 of 16384, the critical-curve window 2 of
# 4096, Johannsen-Psaltis 0 of 9216), and never less than one ray
@pytest.mark.parametrize("name, max_band", [("c1", 1), ("critical", 3), ("jp", 1)])
def test_device_count_against_the_oracle(name, max_band):
    if name == "c1":
        m, x, _, cfg = common.c1(128, 128)
        cfg = common.render_config(m, x, None, 2000.0, 128, 128)
    elif name == "critical":
        m, x, _, _ = common.c1(8, 8)
        cfg = common.render_config(m, x, None, 2000.0, 64, 64, alims=(-3.0, -2.2), blims=(-0.4, 0.4))
    else:
        m, x, d, cfg = common.c5(96, 96)
        cfg = common.render_config(m, x, None, 2000.0, 96, 96)
    p, ic = cfg.to_c()
    want, band = _count_band(p, ic)
    got = _device_counts(cfg, p, ic)
    ok = ~band
    print(f"{name}: band {band.mean():.3%} ({band.sum()} rays), counts {np.bincount(want['crossings'][ok])}")
    assert band.sum() <= max_band
    assert np.array_equal(got[ok], want["crossings"][ok]), np.where(got[ok] != want["crossings"][ok])[0][:10]
    if name == "critical":
        assert want["crossings"][ok].max() >= 3


@pytest.mark.gpu
def test_device_thin_disc_hits_equal_their_image_order():
    m, x, d, cfg = common.c1(128, 128)
    pfs = [gb.ConstPointFunctions.equatorial_crossings(), gb.ConstPointFunctions.redshift(m, x) @ gb.ConstPointFunctions.filter_intersected(),
           gb.ConstPointFunctions.radius() @ gb.ConstPointFunctions.filter_intersected(), gb.ConstPointFunctions.radius()]
    ref = api.apply_point_functions(cfg, pfs)
    hit = ~np.isnan(ref[2])
    assert hit.sum() > 5000
    filtered = api.apply_point_functions(cfg, [gb.ConstPointFunctions.equatorial_crossings() @ gb.ConstPointFunctions.filter_intersected()])
    assert np.array_equal(filtered[0], np.where(hit, ref[0], np.nan), equal_nan=True)  # the order of each hit
    bitwise = []
    for c in np.unique(ref[0][hit]).astype(int):
        got = api.apply_point_functions(_order_config(c, 128, 128), pfs)
        sel = hit & (ref[0] == c)
        assert np.all(~np.isnan(got[1][sel]))
        assert np.max(np.abs(got[1:, sel] - ref[1:, sel]) / np.abs(ref[1:, sel])) <= 1e-12
        bitwise.append((c, int(sel.sum()), bool(np.array_equal(got[:, sel], ref[:, sel]))))
    print("count, rays, bitwise:", bitwise)


@pytest.fixture(scope="module")
def subring_reference():
    """The order-0, 1, 2 replays on a 64^2 window across the critical curve, and their bands."""
    p, ic = _order_config(0, 64, 64, **SUBRING_WINDOW).to_c()
    refs = reference.trace_orders(p, ic, [0, 1, 2])
    alts = reference.trace_orders(p, ic, [0, 1, 2], precision=1)
    return [(ref, reference.band(ref, alt)) for ref, alt in zip(refs, alts)]


# measured on the 64^2 window: 4096, 3099 and 735 hits outside bands of 0, 0 and 0 rays; the band may hold at most 1.5 x
# that, and never less than one ray
ORDER_LIMITS = [(0, 4000, 1), (1, 3000, 1), (2, 700, 1)]
@pytest.mark.gpu
@pytest.mark.parametrize("n, min_hits, max_band", ORDER_LIMITS)
def test_device_image_order_against_the_reference(n, min_hits, max_band, subring_reference):
    cfg = _order_config(n, 64, 64, **SUBRING_WINDOW)
    p, ic = cfg.to_c()
    ref, band = subring_reference[n]
    m, x = cfg.metric, cfg.position
    pfs = [gb.ConstPointFunctions.redshift(m, x) @ gb.ConstPointFunctions.filter_intersected(),
           gb.ConstPointFunctions.radius() @ gb.ConstPointFunctions.filter_intersected(),
           gb.ConstPointFunctions.equatorial_crossings()]
    got = api.apply_point_functions(cfg, pfs)
    want = [reference.kerr_redshift(p, ref), reference.disc_radius(ref), ref["crossings"]]
    gps = api.solve_tracing_problem(cfg)
    ok = ~band
    hit = ok & (ref["status"] == cabi.STATUS_INTERSECTED)
    print(f"order {n}: {hit.sum()} hits outside the band, band {band.mean():.3%} ({band.sum()} rays)")
    assert band.sum() <= max_band
    assert np.array_equal(gps.status[ok], ref["status"][ok])
    assert hit.sum() >= min_hits
    assert np.all(want[2][hit] == n) and np.all(got[2][hit] == n)
    for k in range(2):
        assert np.array_equal(np.isnan(got[k][ok]), np.isnan(want[k][ok]))
        assert np.max(np.abs(got[k][hit] - want[k][hit]) / (1.0 if k == 0 else 50.0)) < 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1])
def test_device_line_profile_per_order(n):
    """BASELINE configs[2]'s line profile per image order, without its hemisphere callback: r cos(theta) < delta ends every
    ray at its first equatorial crossing, so no order >= 1 image would survive it."""
    m, x, d, plane, _ = common.c3(64, 64)
    bins = np.linspace(0.1, 1.5, 180)
    dn = gb.ImageOrder(d, n)
    _, flux = gb.lineprofile(bins, gb.PowerLawEmissivity(3.0), m, x, dn, gb.BinningMethod(), plane=plane, lambda_max=2000.0, callback=None)
    _, flux2 = gb.lineprofile(bins, gb.PowerLawEmissivity(3.0), m, x, dn, gb.BinningMethod(), plane=plane, lambda_max=2000.0, callback=None)
    assert np.array_equal(flux, flux2)  # fixed-point histogram: bitwise reproducible
    cfg_n = api.tracing_configuration(m, x, plane, dn, (0.0, 2000.0))
    p, ic = cfg_n.to_c()
    want = reference.lineprofile(p, ic, reference.trace(p, ic), bins, 3.0, gb.isco(m), 50.0)
    print(f"order {n}: L1 {np.abs(flux - want).sum():.2e}, {np.count_nonzero(want)} non-empty bins")
    assert flux.sum() == pytest.approx(1.0, abs=1e-12)
    assert np.count_nonzero(want) > 20
    assert np.abs(flux - want).sum() < 1e-4


@pytest.mark.gpu
def test_comm_render_of_the_crossings_equals_one_context():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two devices")
    m, x, d, _ = common.c1(8, 8)
    pf = [gb.ConstPointFunctions.equatorial_crossings(), gb.ConstPointFunctions.redshift(m, x) @ gb.ConstPointFunctions.filter_intersected()]
    ens2 = gb.EnsembleB200(devices=(0, 1))
    try:
        _, _, one = gb.rendergeodesics(m, x, gb.ImageOrder(d, 1), 2000.0, pf=pf, image_width=64, image_height=48)
        _, _, two = gb.rendergeodesics(m, x, gb.ImageOrder(d, 1), 2000.0, pf=pf, image_width=64, image_height=48, ensemble=ens2)
        assert all(np.array_equal(a, b, equal_nan=True) for a, b in zip(one, two))
        _, _, one = gb.rendergeodesics(m, x, d, 2000.0, pf=pf, image_width=64, image_height=48)
        _, _, two = gb.rendergeodesics(m, x, d, 2000.0, pf=pf, image_width=64, image_height=48, ensemble=ens2)
        assert all(np.array_equal(a, b, equal_nan=True) for a, b in zip(one, two))
    finally:
        ens2.close()
