"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on identical inputs.

Protocol (DESIGN.md "What parity means here"):
  * termination class identical for every ray outside the grazing band.  The band is defined by the oracle alone:
    (a) rays whose transparent trajectory crosses the disc region for less than 1.3x the event sampler's spacing
    dt/7 (oracle.band_ratio), plus (b) rays whose status, or whose disc-hit state beyond 3e-7, changes when the
    oracle itself runs in long double (rounding-sensitive: photon-ring windings, disc hits next to the horizon);
  * disc hits and lambda_max-terminated rays: endpoint x and v within 1e-6 relative (vector norm);
  * rays ended by a DiscreteCallback (horizon chart, hemisphere): the stored endpoint is wherever the last step
    landed, which is rounding-noise dependent in the reference itself, so the GPU state is compared with the
    oracle's solution of the same ray evaluated at the same affine parameter;
  * redshift images within 1e-6 absolute, identical NaN mask outside the band; line profiles within 1e-4 L1.
"""
import ctypes as C
import math

import numpy as np
import pytest

import gradus_b200 as gb
from gradus_b200 import _cabi as cabi
from gradus_b200.api import solve_tracing_problem, tracing_configuration
from oracle import oracle

import common

pytestmark = pytest.mark.gpu

TOL = 1e-6


def _vec_rel(a, b, floor=1.0):
    """max-norm relative difference of 4-vectors stored as (4, n)."""
    return np.max(np.abs(a - b), axis=0) / np.maximum(np.max(np.abs(b), axis=0), floor)


def _x_rel(a, b):
    """component-wise relative difference of positions (t, r, theta, phi), each against max(|ref|, 1)."""
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1.0), axis=0)


def grazing_band(p, ic, ref, rng=None):
    ratio = oracle.band_ratio(p, ic, rng=rng)
    band = (ratio > 0) & (ratio < 1.3)
    # rounding-sensitive rays: the same oracle in x87 long double (64-bit mantissa) takes a different step sequence
    # (the first steps' error estimates are rounding noise), exactly as any other correct implementation does
    alt = oracle.trace(p, ic, rng=rng, precision=1)
    hit = (ref.status == cabi.STATUS_INTERSECTED) & (alt.status == cabi.STATUS_INTERSECTED)
    moved = np.zeros(len(band), bool)
    moved[hit] = (_x_rel(alt.x[:, hit], ref.x[:, hit]) > 3e-7) | (_vec_rel(alt.v[:, hit], ref.v[:, hit], 1e-12) > 3e-7)
    return band | (alt.status != ref.status) | moved


def check_parity(cfg, name, max_band, discrete_tol=1e-5):
    """`max_band`: the grazing band of this configuration may not be larger (1.5 x what was measured: C1 0.42 %, C3 0.06 %,
    Johannsen-Psaltis 0.41 %; none at all in the Shakura-Sunyaev, datum-plane, no-geometry and lamp-post fixtures)."""
    p, ic = cfg.to_c()
    ref = oracle.trace(p, ic)
    band = grazing_band(p, ic, ref)
    gps = solve_tracing_problem(cfg)
    st = cfg.ensemble.stats()
    ok = ~band
    # (1) termination classes
    mism = (gps.status != ref.status) & ok
    assert not mism.any(), f"{name}: {mism.sum()} status mismatches outside the grazing band at rays {np.where(mism)[0][:10]}"
    assert band.mean() < max_band, f"{name}: grazing band {band.mean():.3%}"
    # (2) well-defined endpoints
    same = (gps.status == ref.status) & ok
    for code in (cabi.STATUS_INTERSECTED, cabi.STATUS_NO_STATUS):
        sel = same & (ref.status == code)
        if not sel.any():
            continue
        # hemisphere/chart callbacks can override a disc event's status but the state is still root-found
        ex, ev = _x_rel(gps.x[:, sel], ref.x[:, sel]), _vec_rel(gps.v[:, sel], ref.v[:, sel], 1e-12)
        el = np.abs(gps.lambda_max[sel] - ref.lambda_max[sel]) / np.maximum(np.abs(ref.lambda_max[sel]), 1.0)
        assert ex.max() < TOL and ev.max() < TOL and el.max() < TOL, f"{name}: status {code}: x {ex.max():.2e} v {ev.max():.2e} lam {el.max():.2e}"
    # (3) DiscreteCallback-terminated rays: same geodesic at the same affine parameter.  At the horizon chart
    # (r = 1.01 r_h) phi, v^t and v^phi diverge logarithmically: the oracle's own double vs long-double spread of this
    # very check is 2.3e-5 there, so the inner-boundary tolerance is 2e-4; escaping / hemisphere rays get 1e-5.
    for code, tol in ((cabi.STATUS_WITHIN_INNER_BOUNDARY, 20 * discrete_tol), (cabi.STATUS_OUT_OF_DOMAIN, discrete_tol)):
        idx = np.where(same & (ref.status == code))[0]
        if not len(idx):
            continue
        idx = idx[:: max(1, len(idx) // 400)]
        u0 = np.concatenate([gps.x_init[:, idx], gps.v_init[:, idx]]).T
        want = oracle.trace_to(p, u0, gps.lambda_max[idx])
        got = np.concatenate([gps.x[:, idx], gps.v[:, idx]]).T
        ex = np.max(np.abs(got[:, :4] - want[:, :4]) / np.maximum(np.abs(want[:, :4]), 1.0), axis=1)
        ev = np.max(np.abs(got[:, 4:] - want[:, 4:]), axis=1) / np.maximum(np.max(np.abs(want[:, 4:]), axis=1), 1e-12)
        assert ex.max() < tol and ev.max() < tol, f"{name}: same-geodesic check (status {code}) x {ex.max():.2e} v {ev.max():.2e}"
    # (4) initial conditions (closed-form LNRF vs the oracle's Gram-Schmidt tetrad) and counters
    assert _vec_rel(gps.v_init, ref.v_init, 1e-12).max() < 1e-11
    assert np.array_equal(gps.x_init, ref.x_init)
    assert int(gps.naccept.sum()) == st.steps_accepted and int(gps.nreject.sum()) == st.steps_rejected
    assert st.flagged == 0 and not gps.flags.any()
    return p, ic, ref, gps, band


def check_sampled_parity(p, ic, rng, got_g, got_rho, got_status, name, max_band):
    """A strided sample (>= 65 536 rays) of a full-size launch against the oracle, by the protocol of `check_parity`:
    identical termination class for EVERY sampled ray outside the grazing band (band-ratio rays plus the rays the
    oracle itself moves between double and long double), redshift within 1e-6 absolute, radius within 1e-6 relative."""
    want, ref = oracle.render(p, ic, [cabi.PF_REDSHIFT, cabi.PF_DISC_RADIUS], rng=rng, endpoints=True)
    band = grazing_band(p, ic, ref, rng=rng)
    assert band.mean() < max_band, f"{name}: grazing band {band.mean():.3%}"
    ok = ~band
    mism = (got_status.astype(np.int32) != ref.status) & ok
    assert not mism.any(), f"{name}: {mism.sum()} of {ok.sum()} sampled rays outside the band differ in status (sample indices {np.where(mism)[0][:10]})"
    hit = ok & (ref.status == cabi.STATUS_INTERSECTED)
    assert hit.sum() > 0.25 * rng.count
    assert np.array_equal(np.isnan(got_g[ok]), np.isnan(want[0][ok]))
    assert np.abs(got_g[hit] - want[0][hit]).max() < 1e-6 and np.abs(got_rho[hit] / want[1][hit] - 1).max() < 1e-6
    counts = np.bincount(ref.status, minlength=4) / rng.count
    print(f"{name}: {rng.count} sampled rays, band {band.mean():.3%}; status fractions out-of-domain {counts[0]:.3f} inner-boundary {counts[1]:.3f} "
          f"intersected {counts[2]:.3f} no-status {counts[3]:.3f}")
    return band


def test_c1_kerr_thin_disc_128(ensemble):
    """BASELINE configs[0]: Kerr a=0.998, r=1000, theta=60deg, 128x128, ThinDisc(0,50), Tsit5 1e-9."""
    m, x, d, cfg = common.c1(128, 128, ensemble=ensemble)
    p, ic, ref, gps, band = check_parity(cfg, "C1", 6e-3)
    # redshift + disc-radius images through the fused render path
    pfs = [gb.ConstPointFunctions.redshift(m, x) @ gb.ConstPointFunctions.filter_intersected(),
           gb.ConstPointFunctions.radius() @ gb.ConstPointFunctions.filter_intersected()]
    _, _, imgs = gb.rendergeodesics(m, x, d, 2000.0, pf=pfs, image_width=128, image_height=128, ensemble=ensemble)
    want = oracle.render(p, ic, [cabi.PF_REDSHIFT, cabi.PF_DISC_RADIUS])
    okimg = (~band).reshape(128, 128).T
    for k in range(2):
        ref_img = want[k].reshape(128, 128).T
        assert np.array_equal(np.isnan(imgs[k])[okimg], np.isnan(ref_img)[okimg])
        both = okimg & ~np.isnan(imgs[k]) & ~np.isnan(ref_img)
        assert both.sum() > 5000
        tol = 1e-6 if k == 0 else 1e-6 * 50.0  # radius is O(50): 1e-6 relative
        assert np.abs(imgs[k][both] - ref_img[both]).max() < tol


def test_c3_line_profile_plane(ensemble):
    """BASELINE configs[2] at reduced size: PolarPlane(GeometricGrid) + hemisphere callback + binned line profile."""
    m, x, d, plane, cfg = common.c3(128, 128, ensemble=ensemble)
    p, ic, ref, gps, band = check_parity(cfg, "C3", 2e-3)
    bins = np.linspace(0.1, 1.5, 180)
    _, flux = gb.lineprofile(bins, gb.PowerLawEmissivity(3.0), m, x, d, gb.BinningMethod(), plane=plane, lambda_max=2000.0, ensemble=ensemble)
    emis = cabi.Emissivity(cabi.EMISSIVITY_POWERLAW, 0, 3.0, None, None)
    want = oracle.lineprofile(p, ic, emis, bins, cabi.LineProfileOpts(gb.isco(m), 50.0, 1, 0))
    assert flux.sum() == pytest.approx(1.0, abs=1e-12)
    assert np.abs(flux - want).sum() < 1e-4  # L1, north_star tolerance
    # coarse features the reference's own test pins (test/line-profiles/test-binning.jl:24-29 analogue)
    assert bins[np.argmax(flux)] > 0.9
    # tabulated emissivity takes the same path
    rr = np.geomspace(1.0, 60.0, 200)
    _, flux_t = gb.lineprofile(bins, gb.TabulatedEmissivity(rr, rr**-3.0), m, x, d, gb.BinningMethod(), plane=plane, lambda_max=2000.0, ensemble=ensemble)
    assert np.abs(flux_t - flux).sum() < 2e-3  # linear interpolation of r^-3 on a 200-point grid


@pytest.mark.parametrize("a,eps3", [(0.6, 2.0), (0.8831, 0.4)])
def test_c5_johannsen_psaltis(ensemble, a, eps3):
    """BASELINE configs[4]: closed-form non-Kerr RHS (the reference's JP test points)."""
    inner = None if a == 0.6 else 2.0  # the near-naked-singularity point has no ISCO
    m, x, d, cfg = common.c5(96, 96, a=a, eps3=eps3, ensemble=ensemble, inner=inner)
    p, ic, ref, gps, band = check_parity(cfg, f"C5 a={a}", 6e-3)
    if a == 0.6:
        pf = gb.ConstPointFunctions.redshift(m, x) @ gb.ConstPointFunctions.filter_intersected()
        _, _, img = gb.rendergeodesics(m, x, d, 2000.0, pf=pf, image_width=96, image_height=96, ensemble=ensemble)
        want = oracle.render(p, ic, [cabi.PF_REDSHIFT])[0].reshape(96, 96).T
        ok = (~band).reshape(96, 96).T & ~np.isnan(img) & ~np.isnan(want)
        assert ok.sum() > 2000 and np.abs(img[ok] - want[ok]).max() < 1e-6


def test_shakura_sunyaev_and_datum_plane(ensemble):
    m = gb.KerrMetric(1.0, 0.9)
    x = [0.0, 1000.0, math.radians(70.0), 0.0]
    cfg = common.render_config(m, x, gb.ShakuraSunyaev(m, eddington_ratio=0.3), 2000.0, 64, 64, (-40, 40), (-30, 30), ensemble=ensemble)
    check_parity(cfg, "ShakuraSunyaev", 1e-3)
    cfg = common.render_config(m, x, gb.DatumPlane(0.5), 2000.0, 48, 48, (-30, 30), (-20, 20), ensemble=ensemble)
    check_parity(cfg, "DatumPlane", 1e-3)
    cfg = common.render_config(m, x, None, 2000.0, 48, 48, (-12, 12), (-12, 12), ensemble=ensemble)
    check_parity(cfg, "no geometry", 1e-3)


def test_explicit_initial_conditions_lamp_post_like(ensemble):
    """The arbitrary-IC path (corona ensembles, src/corona/models/lamp-post.jl:89-100): rays fanned from a source on the axis."""
    m = gb.KerrMetric(1.0, 0.998)
    xs = [0.0, 10.0, 0.01, 0.0]
    delta = np.radians(np.linspace(0.01, 179.99, 300))
    # unnormalised directions in the (r, theta) plane; v^t is re-constrained by the library like constrain_all does
    vs = np.stack([np.zeros_like(delta), -np.cos(delta), np.sin(delta) / 10.0, np.zeros_like(delta)], axis=1)
    cfg = tracing_configuration(m, xs, vs, gb.ThinDisc(0.0, 1000.0), 10000.0, callback=gb.domain_upper_hemisphere(), ensemble=ensemble)
    p, ic, ref, gps, band = check_parity(cfg, "explicit IC", 1e-3)
    assert (gps.status == cabi.STATUS_INTERSECTED).sum() > 50


def test_reference_golden_values_on_gpu(ensemble):
    """The reference's own golden literals, now produced by the CUDA path (tests/golden/reference_literals.json)."""
    x = [0.0, 100.0, math.radians(85), 0.0]
    kw = dict(image_width=20, image_height=20, αlims=(-9.5, 9.5), βlims=(-9.5, 9.5), ensemble=ensemble)
    _, _, img = gb.rendergeodesics(gb.KerrMetric(), x, 200.0, **kw)
    assert np.nansum(img) == pytest.approx(9009.452876609641, rel=1e-6)  # test/smoke-tests/rendergeodesics.jl:44
    _, _, img = gb.rendergeodesics(gb.KerrMetric(), x, gb.ThinDisc(0.0, 40.0), 200.0, **kw)
    assert np.nansum(img) == pytest.approx(38412.08347901267, rel=1e-6)  # :59
    m = gb.JohannsenPsaltisMetric(M=1.0, a=0.8831, eps3=0.4)
    _, _, img = gb.rendergeodesics(m, [0.0, 1000.0, math.pi / 2, 0.0], 2000.0, image_width=100, image_height=100, αlims=(-8, 8), βlims=(-8, 8),
                                   ensemble=ensemble)
    assert np.nansum(img) == pytest.approx(2.9619136946153212e6, rel=1e-6)  # test/integration/test-charts.jl:18 (reference rtol 1e-4)
    for grid, count in [(gb.LinearGrid(), 10), (gb.GeometricGrid(), 30), (gb.InverseGrid(), 80)]:  # test-polar-grids.jl:13-21
        gps = gb.tracegeodesics(gb.KerrMetric(), [1.0, 1e3, math.pi / 2, 0.0], gb.PolarPlane(grid, Nr=10, Ntheta=10), (0.0, 2000.0), ensemble=ensemble)
        assert int((gps.status == cabi.STATUS_WITHIN_INNER_BOUNDARY).sum()) == count
    for grid, count in [(gb.LinearGrid(), 1), (gb.GeometricGrid(), 25), (gb.InverseGrid(), 81)]:  # test-cartesian-grids.jl:13-21
        plane = gb.CartesianPlane(grid, x_min=0.1, y_min=0.1, Nx=12, Ny=12)
        gps = gb.tracegeodesics(gb.KerrMetric(), [1.0, 1e3, math.pi / 2, 0.0], plane, (0.0, 2000.0), ensemble=ensemble)
        assert len(gps) == 121 and int((gps.status == cabi.STATUS_WITHIN_INNER_BOUNDARY).sum()) == count
    m = gb.KerrMetric(1.0, 0.998)  # test/transfer-functions/test-2d.jl:25
    x = [0.0, 1e6, math.radians(30), 0.0]
    gps = gb.tracegeodesics(m, x, gb.PolarPlane(gb.GeometricGrid(), Nr=20, Ntheta=20), gb.ThinDisc(gb.isco(m), 500.0), (0.0, 2e6),
                            chart=gb.chart_for_metric(m, 1.1e6), callback=gb.domain_upper_hemisphere(), ensemble=ensemble)
    assert int((gps.status == cabi.STATUS_INTERSECTED).sum()) == 337


@pytest.mark.parametrize("m,g_low_ref", [(gb.KerrMetric(1.0, 0.6), 0.355), (gb.JohannsenPsaltisMetric(1.0, 0.6, 2.0), 0.27)])
def test_reference_line_profile_edges_on_gpu(ensemble, m, g_low_ref):
    """test/line-profiles/test-binning.jl:5-57 through the GPU `lineprofile`, and L1 parity with the oracle on the same fixture."""
    u = [0.0, 1000.0, math.radians(60), 0.0]
    d = gb.ThinDisc(gb.isco(m), 250.0)
    plane = gb.PolarPlane(gb.GeometricGrid(), Nr=100, Ntheta=400)
    bins = np.linspace(0.1, 1.3, 100)
    x, y = gb.lineprofile(bins, gb.PowerLawEmissivity(3.0), m, u, d, gb.BinningMethod(), plane=plane, callback=gb.domain_upper_hemisphere(), ensemble=ensemble)
    nzi = np.nonzero(y > 0)[0]
    assert x[nzi[0]] == pytest.approx(g_low_ref, abs=0.05) and x[nzi[-1] - 1] == pytest.approx(1.2, abs=0.05)
    assert y.sum() == pytest.approx(1.0, abs=1e-12)
    cfg = tracing_configuration(m, u, plane, d, (0.0, 2000.0), callback=gb.domain_upper_hemisphere(), ensemble=ensemble)
    p, ic = cfg.to_c()
    want = oracle.lineprofile(p, ic, cabi.Emissivity(cabi.EMISSIVITY_POWERLAW, 0, 3.0, None, None), bins, cabi.LineProfileOpts(gb.isco(m), 50.0, 1, 0))
    # In this fixture the disc's inner edge IS the ISCO, so the handful of rays that graze that edge (grazing band, DESIGN.md)
    # carry the largest r^-3 g^3 weights of a 40 000-ray plane: L1 is band-limited here (the band-free C3 test requires 1e-4).
    assert np.abs(y - want).sum() < 5e-3


def test_full_size_render_properties(ensemble):
    """BASELINE configs[1] at full 2048x2048 size: size-independent properties + a strided oracle sample."""
    m, x, d, cfg = common.c1(2048, 2048, ensemble=ensemble)
    p, ic = cfg.to_c()
    lib = cabi.load()
    ctx = ensemble.ctx(ensemble.devices[0])
    pfs = np.array([cabi.PF_REDSHIFT, cabi.PF_DISC_RADIUS, cabi.PF_STATUS], np.int32)

    def render(rng):
        imgs = np.zeros((3, rng.count))
        ptrs = (cabi._dp * 3)(*[cabi.dptr(imgs[k]) for k in range(3)])
        cabi.check(lib.gb200_render(ctx, C.byref(p), C.byref(ic), C.byref(rng), cabi.iptr(pfs), 3, None, ptrs), ctx)
        return imgs

    full = render(cabi.Range(0, ic.n, 1))
    again = render(cabi.Range(0, ic.n, 1))
    assert np.array_equal(full, again, equal_nan=True)  # deterministic: no dependence on work-queue timing
    # sharding invariance: an interleaved shard reproduces exactly the same pixels (what the multi-GPU path relies on)
    shard = render(cabi.Range(3, ic.n // 8, 8))
    assert np.array_equal(shard, full[:, 3::8][:, : ic.n // 8], equal_nan=True)
    # strips of 4 image columns interleaved over 8 ranks (bench.py's decomposition; 2-D tiled work order inside)
    from gradus_b200 import distributed as gd

    for rank in (0, 5):
        rng = gd.strip_interleaved_range(ic, rank, 8)
        assert rng.block == 4 * 2048 and rng.count == ic.n // 8
        assert np.array_equal(render(rng), full[:, rng.indices()], equal_nan=True)
    # physics: redshift range of a a=0.998 disc seen at 60 degrees, radii inside the disc, NaN masks consistent
    g, rho, status = full
    hit = status == cabi.STATUS_INTERSECTED
    assert np.array_equal(np.isnan(g), ~hit) and np.array_equal(np.isnan(rho), ~hit)
    assert 0.4 < hit.mean() < 0.5
    assert 0.0 < np.nanmin(g) < 0.3 and 1.2 < np.nanmax(g) < 1.5 and np.nanmax(rho) <= 50.0 * (1 + 1e-12)
    # strided oracle sample of the full-size image: every 64th ray, 65 536 rays
    rng = cabi.Range(17, 65536, 64)
    got = full[:, 17::64][:, :65536]
    check_sampled_parity(p, ic, rng, got[0], got[1], got[2], "C2 2048x2048", 6e-3)


def test_full_size_trace_conservation_laws(ensemble):
    """2048x2048 endpoints straight from gb200_trace: E, L_z and the null condition hold for every ray."""
    m, x, d, cfg = common.c1(2048, 2048, ensemble=ensemble)
    gps = solve_tracing_problem(cfg)
    st = ensemble.stats()
    assert int(gps.naccept.sum(dtype=np.int64)) == st.steps_accepted
    M, a = 1.0, 0.998

    def metric(r, th):
        s2, c2 = np.sin(th) ** 2, np.cos(th) ** 2
        S = r * r + a * a * c2
        D = r * r - 2 * M * r + a * a
        return -(1 - 2 * M * r / S), S / D, S, s2 * (r * r + a * a + 2 * M * r * a * a * s2 / S), -2 * M * r * a * s2 / S

    def invariants(xx, vv):
        tt, rr, thth, phph, tph = metric(xx[1], xx[2])
        E = -(tt * vv[0] + tph * vv[3])
        L = phph * vv[3] + tph * vv[0]
        n = tt * vv[0] ** 2 + rr * vv[1] ** 2 + thth * vv[2] ** 2 + phph * vv[3] ** 2 + 2 * tph * vv[0] * vv[3]
        return E, L, n

    E0, L0, n0 = invariants(gps.x_init, gps.v_init)
    E1, L1, n1 = invariants(gps.x, gps.v)
    scale = 1.0 + np.abs(gps.v[0])  # v^t diverges towards the horizon: errors are measured against it
    far = scale < 10.0
    assert far.mean() > 0.95
    assert np.abs(n0).max() < 1e-12
    assert np.abs(E1 - E0)[far].max() < 1e-6 and np.abs(L1 - L0)[far].max() < 1e-5 and np.abs(n1)[far].max() < 1e-6
    assert (np.abs(E1 - E0) / scale).max() < 1e-6 and (np.abs(n1) / scale**2).max() < 1e-6
    assert np.bincount(gps.status, minlength=4)[cabi.STATUS_OUT_OF_DOMAIN] == 0  # nothing escapes past r=12000 by lambda=2000


def test_device_resident_entry_points_and_fp64_peak(ensemble):
    import torch

    m, x, d, cfg = common.c1(96, 96, ensemble=ensemble)
    p, ic = cfg.to_c()
    lib = cabi.load()
    dev = ensemble.devices[0]
    ctx = ensemble.ctx(dev)
    stream = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(stream):
        d_img = torch.empty(ic.n, dtype=torch.float64, device=f"cuda:{dev}")
        ptrs = (C.c_void_p * 1)(C.c_void_p(d_img.data_ptr()))
        pfs = np.array([cabi.PF_REDSHIFT], np.int32)
        rng = cabi.Range(0, ic.n, 1)
        cabi.check(lib.gb200_render_device(ctx, C.byref(p), C.byref(ic), C.byref(rng), cabi.iptr(pfs), 1, None, ptrs, C.c_void_p(stream.cuda_stream), 1), ctx)
        stream.synchronize()
    host = np.zeros(ic.n)
    hp = (cabi._dp * 1)(cabi.dptr(host))
    cabi.check(lib.gb200_render(ctx, C.byref(p), C.byref(ic), C.byref(rng), cabi.iptr(pfs), 1, None, hp), ctx)
    assert np.array_equal(d_img.cpu().numpy(), host, equal_nan=True)
    peak = C.c_double()
    cabi.check(lib.gb200_fp64_peak(ctx, C.byref(peak)), ctx)
    assert 20.0 < peak.value < 45.0  # B200 FP64 CUDA-core peak is ~37 TFLOP/s


def test_invalid_calls_fail_loudly(ensemble):
    m, x, d, cfg = common.c1(8, 8, ensemble=ensemble)
    p, ic = cfg.to_c()
    lib = cabi.load()
    ctx = ensemble.ctx(ensemble.devices[0])
    out = cabi.EndpointArrays(4)
    rng = cabi.Range(60, 8, 1)  # exceeds 64 rays
    assert lib.gb200_trace(ctx, C.byref(p), C.byref(ic), C.byref(rng), C.byref(out.c)) == cabi.ERR_INVALID_ARGUMENT
    assert b"range" in lib.gb200_last_error(ctx)
    p.geometry_kind = 9
    rng = cabi.Range(0, 4, 1)
    assert lib.gb200_trace(ctx, C.byref(p), C.byref(ic), C.byref(rng), C.byref(out.c)) == cabi.ERR_UNSUPPORTED


def test_batched_short_ensembles_match_individual_calls(ensemble):
    """SURVEY 8f-1 / BASELINE configs[3]: lamp-post-like 1000-ray fans over a spin grid, one batched call."""
    from gradus_b200 import tracegeodesics_batch

    xs = [0.0, 10.0, 0.01, 0.0]
    delta = np.radians(np.linspace(0.01, 179.99, 1000))
    vs = np.stack([np.zeros_like(delta), -np.cos(delta), np.sin(delta) / 10.0, np.zeros_like(delta)], axis=1)
    spins = [0.0, 0.3, 0.6, 0.9, 0.998]
    cfgs = [tracing_configuration(gb.KerrMetric(1.0, a), xs, vs, gb.ThinDisc(0.0, 1000.0), 10000.0, callback=gb.domain_upper_hemisphere(),
                                  ensemble=ensemble) for a in spins]
    cfgs.append(common.c1(40, 40, ensemble=ensemble)[3])  # a structured-IC ensemble mixed into the same batch
    batch = tracegeodesics_batch(cfgs)
    st = ensemble.stats()
    assert st.launches == len(cfgs) and st.rays == 5 * 1000 + 1600
    for cfg, got in zip(cfgs, batch):
        want = solve_tracing_problem(cfg)
        assert np.array_equal(got.status, want.status)
        assert np.array_equal(got.x, want.x) and np.array_equal(got.v, want.v) and np.array_equal(got.lambda_max, want.lambda_max)
        assert np.array_equal(got.x_init, want.x_init) and np.array_equal(got.naccept, want.naccept)
    assert sum(int(g.naccept.sum()) for g in batch) == st.steps_accepted


def test_edge_cases(ensemble):
    """Empty and single-ray ranges, strided sub-ranges, non-default tolerances and lambda domain, iteration cap."""
    m, x, d, cfg = common.c1(32, 32, ensemble=ensemble)
    p, ic = cfg.to_c()
    lib = cabi.load()
    ctx = ensemble.ctx(ensemble.devices[0])
    out = cabi.EndpointArrays(1)
    assert lib.gb200_trace(ctx, C.byref(p), C.byref(ic), C.byref(cabi.Range(5, 0, 1)), C.byref(out.c)) == cabi.OK  # empty: no launch
    assert ensemble.stats().launches == 0 and ensemble.stats().rays == 0
    full = solve_tracing_problem(cfg)
    for first, count, stride, block in [(777, 1, 1, 1), (3, 100, 7, 1), (1023, 1, 1, 1), (0, 1024, 1, 1), (32, 96, 3, 32), (128, 256, 2, 128), (5, 70, 4, 10)]:
        sub = cabi.EndpointArrays(count)
        rng = cabi.Range(first, count, stride, block)
        cabi.check(lib.gb200_trace(ctx, C.byref(p), C.byref(ic), C.byref(rng), C.byref(sub.c)), ctx)
        idx = rng.indices()
        assert np.array_equal(sub.status, full.status[idx]) and np.array_equal(sub.x, full.x[:, idx]) and np.array_equal(sub.v, full.v[:, idx])
    # looser and tighter tolerances, shifted affine domain: still matches the oracle
    for tol in (1e-6, 1e-11):
        c2 = common.render_config(m, x, d, (5.0, 2005.0), 24, 24, ensemble=ensemble, abstol=tol, reltol=tol)
        p2, ic2 = c2.to_c()
        ref = oracle.trace(p2, ic2)
        got = solve_tracing_problem(c2)
        agree = got.status == ref.status
        assert agree.mean() > 0.99
        hit = agree & (ref.status == cabi.STATUS_INTERSECTED)
        assert _x_rel(got.x[:, hit], ref.x[:, hit]).max() < max(1e-6, 300 * tol)
        assert got.lambda_max.min() > 5.0 and np.all(got.lambda_max[ref.status == cabi.STATUS_NO_STATUS] == 2005.0)
    # iteration cap: the ray keeps NoStatus and raises the MAXITERS flag (SciML retcode MaxIters is invisible in GeodesicPoint)
    c3 = common.render_config(m, x, d, 2000.0, 8, 8, ensemble=ensemble, maxiters=20)
    got = solve_tracing_problem(c3)
    assert np.all(got.status == cabi.STATUS_NO_STATUS) and np.all(got.flags == cabi.FLAG_MAXITERS) and np.all(got.naccept + got.nreject == 20)
    assert ensemble.stats().flagged == 64


def test_fast32_controller_and_massive_geodesics(ensemble):
    m, x, d, _ = common.c1(8, 8, ensemble=ensemble)
    # Float32 controller power (FastPower.jl-style): same classes and hits as the oracle's fast32 mode
    cfg = common.render_config(m, x, d, 2000.0, 48, 48, ensemble=ensemble, pow_mode=cabi.POW_FAST32)
    p, ic = cfg.to_c()
    ref = oracle.trace(p, ic)
    got = solve_tracing_problem(cfg)
    agree = got.status == ref.status
    assert agree.mean() > 0.995
    hit = agree & (ref.status == cabi.STATUS_INTERSECTED)
    assert _x_rel(got.x[:, hit], ref.x[:, hit]).max() < 1e-6
    # massive particles (mu = 1, explicit ICs): the plunging-orbit set-up of orbit-solving.jl:137-167 uses this path
    mk = gb.KerrMetric(1.0, 0.5)
    vs = np.array([[0.0, -0.05 * k, 0.0, 0.02] for k in range(1, 33)])
    cfg = tracing_configuration(mk, [0.0, 8.0, math.pi / 2 - 0.05, 0.0], vs, 5.0, mu=1.0, ensemble=ensemble)
    p, ic = cfg.to_c()
    ref = oracle.trace(p, ic)
    got = solve_tracing_problem(cfg)
    assert np.array_equal(got.status, ref.status)
    assert np.all(got.v_init[0] > 0) and _vec_rel(got.v_init, ref.v_init, 1e-12).max() < 1e-11
    done = ref.status == cabi.STATUS_NO_STATUS
    assert done.sum() >= 16 and _x_rel(got.x[:, done], ref.x[:, done]).max() < 1e-6
    # timelike normalisation g(v, v) = -mu^2 is kept along the orbit
    r_, th_ = got.x[1, done], got.x[2, done]
    S = r_**2 + 0.25 * np.cos(th_) ** 2
    D = r_**2 - 2 * r_ + 0.25
    s2 = np.sin(th_) ** 2
    vv = got.v[:, done]
    norm = (-(1 - 2 * r_ / S) * vv[0] ** 2 + S / D * vv[1] ** 2 + S * vv[2] ** 2 + s2 * (r_**2 + 0.25 + 2 * r_ * 0.25 * s2 / S) * vv[3] ** 2
            - 2 * (2 * r_ * 0.5 * s2 / S) * vv[0] * vv[3])
    assert np.abs(norm + 1.0).max() < 1e-6
    # mu = NaN: states that arrive already constrained (an ensemble's prob_func output, what the Julia extension uploads)
    # keep their v^t -- the very same rays again, bit for bit
    cfg2 = tracing_configuration(mk, [0.0, 8.0, math.pi / 2 - 0.05, 0.0], got.v_init.T.copy(), 5.0, mu=float("nan"), ensemble=ensemble)
    again = solve_tracing_problem(cfg2)
    assert np.array_equal(again.v_init, got.v_init) and np.array_equal(again.x, got.x) and np.array_equal(again.status, got.status)
    ref2 = oracle.trace(*cfg2.to_c())
    assert np.array_equal(ref2.v_init, ref.v_init) and np.array_equal(ref2.x, ref.x)


def test_in_process_sharding_over_contexts(ensemble):
    """EnsembleB200 with several contexts (here: the same GPU listed twice) = the Julia ext's multi-GPU path."""
    ens2 = gb.EnsembleB200(devices=(ensemble.devices[0], ensemble.devices[0]))
    try:
        m, x, d, plane, cfg1 = common.c3(48, 48, ensemble=ensemble)
        _, _, _, _, cfg2 = common.c3(48, 48, ensemble=ens2)
        a, b = solve_tracing_problem(cfg1), solve_tracing_problem(cfg2)
        assert np.array_equal(a.status, b.status) and np.array_equal(a.x, b.x) and np.array_equal(a.naccept, b.naccept)
        bins = np.linspace(0.1, 1.5, 60)
        _, f1 = gb.lineprofile(bins, gb.PowerLawEmissivity(3.0), m, x, d, gb.BinningMethod(), plane=plane, lambda_max=2000.0, ensemble=ensemble)
        _, f2 = gb.lineprofile(bins, gb.PowerLawEmissivity(3.0), m, x, d, gb.BinningMethod(), plane=plane, lambda_max=2000.0, ensemble=ens2)
        assert np.abs(f1 - f2).max() < 1e-12  # invariant to the device count up to summation order
        pf = gb.ConstPointFunctions.redshift() @ gb.ConstPointFunctions.filter_intersected()
        mm, xx, dd, _ = common.c1(8, 8)
        _, _, i1 = gb.rendergeodesics(mm, xx, dd, 2000.0, pf=pf, image_width=33, image_height=17, ensemble=ensemble)
        _, _, i2 = gb.rendergeodesics(mm, xx, dd, 2000.0, pf=pf, image_width=33, image_height=17, ensemble=ens2)
        assert i1.shape == (17, 33) and np.array_equal(i1, i2, equal_nan=True)
    finally:
        ens2.close()


def test_plunging_table_and_redshift_inside_isco(ensemble):
    """Non-Kerr redshift inside the ISCO (src/redshift.jl:246-276): table built on the device vs the oracle's."""
    m = gb.JohannsenPsaltisMetric(1.0, 0.6, 2.0)
    mp = (1.0, 0.6, 2.0)
    tab = gb.interpolate_plunging_velocities(m, ensemble)
    r_o, ut_o, ur_o, uph_o = common.oracle_plunging_table(cabi.METRIC_JP, mp)
    risco = gb.isco(m)
    assert tab.r[0] == pytest.approx(r_o[0], rel=2e-2) and tab.r[-1] == pytest.approx(risco, abs=1e-6)
    # Two correct integrations sample the plunge at different radii, and the reference interpolates LINEARLY between
    # samples: near the horizon (u^t ~ 9, steep, sparsely sampled) that alone is worth ~3e-3 (u^r -> 0 at the ISCO inflates its relative error there).
    rr = np.linspace(max(tab.r[0], r_o[0]) * 1.001, risco * 0.9999, 200)
    for got, want in zip(tab(rr), (np.interp(rr, r_o, ut_o), np.interp(rr, r_o, ur_o), np.interp(rr, r_o, uph_o))):
        rel = np.abs(got - want) / np.maximum(np.abs(want), 1e-3)
        assert rel.max() < 1e-2 and np.median(rel) < 1e-4
    # Kerr limit of the machinery: the table reproduces Cunningham's analytic plunging flow (src/redshift.jl:93-164) to table accuracy
    mk = gb.JohannsenPsaltisMetric(1.0, 0.6, 0.0)
    tk = gb.interpolate_plunging_velocities(mk, ensemble)
    rk = np.linspace(tk.r[0] * 1.05, gb.isco(mk) * 0.98, 50)
    rms = gb.isco(mk)
    ur_analytic = -np.sqrt(2.0 / (3.0 * rms)) * (rms / rk - 1.0) ** 1.5
    assert np.max(np.abs(tk(rk)[1] - ur_analytic)) < 2e-4
    # end to end: JP disc reaching inside the ISCO, redshift image vs oracle with the oracle's own table
    x = [0.0, 1000.0, math.radians(60.0), 0.0]
    d = gb.ThinDisc(0.0, 30.0)
    pf = gb.ConstPointFunctions.redshift(m, x) @ gb.ConstPointFunctions.filter_intersected()
    _, _, img = gb.rendergeodesics(m, x, d, 2000.0, pf=pf, image_width=64, image_height=64, αlims=(-30, 30), βlims=(-20, 20), ensemble=ensemble)
    cfg = common.render_config(m, x, d, 2000.0, 64, 64, (-30, 30), (-20, 20), ensemble=ensemble)
    p, ic = cfg.to_c()
    otab = cabi.PlungingTable(len(r_o), cabi.dptr(np.ascontiguousarray(r_o)), cabi.dptr(np.ascontiguousarray(ut_o)),
                              cabi.dptr(np.ascontiguousarray(ur_o)), cabi.dptr(np.ascontiguousarray(uph_o)))
    want, ep = oracle.render(p, ic, [cabi.PF_REDSHIFT, cabi.PF_DISC_RADIUS], plunging=otab, endpoints=True)
    want_g = want[0].reshape(64, 64).T
    rho = want[1].reshape(64, 64).T
    both = ~np.isnan(img) & ~np.isnan(want_g)
    inside = both & (rho < risco)
    assert inside.sum() > 20 and (both & ~inside).sum() > 500
    assert np.abs(img[both & ~inside] - want_g[both & ~inside]).max() < 1e-6
    assert np.abs(img[inside] - want_g[inside]).max() < 2e-3  # two independently integrated tables, linearly interpolated


def test_device_math_against_oracle(ensemble):
    """Function-level check of the closed forms: device RHS vs the oracle's dual-number RHS, sincos and reciprocal."""
    lib = cabi.load()
    ctx = ensemble.ctx(ensemble.devices[0])
    rs = np.random.RandomState(7)
    n = 4000
    for kind, mp in [(cabi.METRIC_KERR, (1.0, 0.998)), (cabi.METRIC_KERR, (1.3, -0.4)), (cabi.METRIC_JP, (1.0, 0.6, 2.0)), (cabi.METRIC_JP, (1.0, 0.8831, 0.4))]:
        rh = mp[0] + math.sqrt(mp[0] ** 2 - mp[1] ** 2)
        u = np.zeros((n, 8))
        u[:, 1] = rh * 1.02 * np.exp(rs.uniform(0, 7, n))  # 1.02 r_h .. 1e3 r_h
        u[:, 2] = rs.uniform(0.05, math.pi - 0.05, n)
        u[:, 3] = rs.uniform(-3, 3, n)
        u[:, 4:] = rs.normal(size=(n, 4)) * np.array([1.5, 1.0, 0.3, 0.3])
        du = np.zeros_like(u)
        mpa = np.array(list(mp) + [0.0] * (4 - len(mp)))
        cabi.check(lib.gb200_debug_rhs(ctx, kind, cabi.dptr(mpa), n, cabi.dptr(u.reshape(-1)), cabi.dptr(du.reshape(-1))), ctx)
        want = np.array([oracle.rhs(kind, mp, u[i]) for i in range(n)])
        scale = np.max(np.abs(want[:, 4:]), axis=1, keepdims=True)
        # the oracle's generic inverse g_tt g_phph - g_tph^2 cancels near the horizon (condition number ~1e4): 1e-10 there
        err = np.abs(du[:, 4:] - want[:, 4:]) / scale
        assert np.array_equal(du[:, :4], u[:, 4:])
        assert err.max() < 1e-10 and np.median(err) < 1e-14, (kind, mp, err.max(), np.median(err))
    x = np.concatenate([rs.uniform(-60, 60, 20000), np.array([0.0, 1e-300, math.pi / 2, math.pi, -math.pi / 4, 40.0, 1e-9])])
    nsc = len(x)  # sin / cos are checked on the polar-angle range only
    x = np.concatenate([x, 10.0 ** rs.uniform(-12, 6, 4000), rs.uniform(-8, 8, 4000)])
    out = np.zeros((len(x), 5))
    cabi.check(lib.gb200_debug_math(ctx, len(x), cabi.dptr(x), cabi.dptr(out.reshape(-1))), ctx)
    assert np.abs(out[:nsc, 0] - np.sin(x[:nsc])).max() < 2.5e-16 and np.abs(out[:nsc, 1] - np.cos(x[:nsc])).max() < 2.5e-16
    nz = x != 0
    assert np.max(np.abs(out[nz, 2] * x[nz] - 1.0)) < 4.5e-16
    # the step controller's log / exp: a few ulp of libm (the controller only needs ~1e-10)
    lg = np.log(np.abs(x[nz]))
    assert np.max(np.abs(out[nz, 3] - lg) / np.maximum(np.abs(lg), 1.0)) < 4.5e-16
    assert out[~nz, 3].max() < -700.0  # log 0: very negative instead of -inf, clamped by the controller all the same
    ex = np.exp(np.clip(x, -8.0, 8.0))
    assert np.max(np.abs(out[:, 4] - ex) / ex) < 1e-15
    # the pair the controller actually uses (gb_log_pos_lo / gb_exp_small_lo): evaluated to the accuracy of the error estimate it acts on
    lo = np.zeros((len(x), 2))
    cabi.check(lib.gb200_debug_math_lo(ctx, len(x), cabi.dptr(x), cabi.dptr(lo.reshape(-1))), ctx)
    assert np.max(np.abs(lo[nz, 0] - lg) / np.maximum(np.abs(lg), 1.0)) < 3e-7
    assert np.max(np.abs(lo[:, 1] - ex) / ex) < 1e-7


def test_gpu_against_committed_golden_fixtures(ensemble):
    """CUDA path vs the frozen vectors of tests/golden/oracle_small.npz (no oracle run involved)."""
    import os

    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "oracle_small.npz"))
    for name, cfg in [("c1_24x24", common.c1(24, 24, ensemble=ensemble)[3]), ("c3_20x20", common.c3(20, 20, ensemble=ensemble)[4]),
                      ("c5_20x20", common.c5(20, 20, ensemble=ensemble)[3])]:
        got = solve_tracing_problem(cfg)
        same = got.status == gold[name + "_status"]
        assert same.mean() > 0.99  # grazing-band rays may differ (these tiny fixtures carry no band analysis)
        hit = same & (got.status == cabi.STATUS_INTERSECTED)
        assert hit.sum() > 50
        assert _x_rel(got.x[:, hit], gold[name + "_x"][:, hit]).max() < 1e-6
        assert _vec_rel(got.v[:, hit], gold[name + "_v"][:, hit], 1e-12).max() < 2e-6


def test_pipelined_host_output_calls_equal_single_launches(ensemble, monkeypatch):
    """Calls with >= 2^20 rays and host output run as four chunks on two streams with overlapped copies
    (run_pipelined): endpoints, images and step counters must equal the single-launch path bit for bit, for a plain and
    for a strided (multi-GPU style) range."""
    m, x, d, cfg = common.c1(1024, 1152, ensemble=ensemble)
    pfs = [gb.ConstPointFunctions.redshift(m, x) @ gb.ConstPointFunctions.filter_intersected(),
           gb.ConstPointFunctions.radius() @ gb.ConstPointFunctions.filter_intersected()]
    got = solve_tracing_problem(cfg)
    st_p = ensemble.stats()
    imgs_p = gb.api.apply_point_functions(cfg, pfs)
    assert st_p.launches == 4
    monkeypatch.setenv("GB200_NO_PIPELINE", "1")
    ref = solve_tracing_problem(cfg)
    st_1 = ensemble.stats()
    imgs_1 = gb.api.apply_point_functions(cfg, pfs)
    assert st_1.launches == 1
    assert (st_p.steps_accepted, st_p.steps_rejected) == (st_1.steps_accepted, st_1.steps_rejected)
    for name in ("status", "lambda_max", "x", "v", "x_init", "v_init", "naccept", "nreject"):
        assert np.array_equal(getattr(got, name), getattr(ref, name), equal_nan=True), name
    assert np.array_equal(imgs_p, imgs_1, equal_nan=True)


def test_full_size_lineprofile_properties(ensemble):
    """BASELINE configs[2] at full size (PolarPlane 4096 x 4096 = 1.7e7 rays, 180 bins): determinism, the raw histogram
    of 8 strip-interleaved shards sums to the single-launch histogram (what the NCCL all-reduce relies on), unit area,
    and a strided oracle sample of the (g, f) pairs behind the histogram."""
    from gradus_b200 import distributed as gd

    m, x, d, plane, cfg = common.c3(4096, 4096, ensemble=ensemble)
    p, ic = cfg.to_c()
    lib = cabi.load()
    ctx = ensemble.ctx(ensemble.devices[0])
    bins = np.linspace(0.1, 1.5, 180)
    emis = cabi.Emissivity(cabi.EMISSIVITY_POWERLAW, 0, 3.0, None, None)
    opts = cabi.LineProfileOpts(gb.isco(m), 50.0, 0, 0)  # raw partial sums

    def hist(rng):
        flux = np.zeros(len(bins))
        cabi.check(lib.gb200_lineprofile(ctx, C.byref(p), C.byref(ic), C.byref(rng), C.byref(emis), None, cabi.dptr(bins), len(bins),
                                         C.byref(opts), cabi.dptr(flux)), ctx)
        return flux

    full = hist(cabi.Range(0, ic.n, 1))
    assert np.array_equal(full, hist(cabi.Range(0, ic.n, 1)))  # exact fixed-point sums in the kernel: bitwise reproducible
    parts = sum(hist(gd.strip_interleaved_range(ic, r, 8)) for r in range(8))
    assert np.max(np.abs(parts - full)) <= 1e-14 * full.max()  # each shard is an exact sum; only the 8-term host sum rounds
    # the histogram fused into the trace kernel against the two-pass form ((g, f) per ray through HBM, then the binning kernels)
    import os

    os.environ["GB200_HIST_TWO_PASS"] = "1"
    try:
        two_pass = hist(cabi.Range(0, ic.n, 1))
    finally:
        del os.environ["GB200_HIST_TWO_PASS"]
    assert np.max(np.abs(two_pass - full)) <= 1e-12 * full.max()
    flux = full / full.sum()
    assert flux.sum() == pytest.approx(1.0) and flux[0] < 1e-3 and flux[-1] == 0.0  # g < 0.1 is clamped into the first bin (Buckets.Simple)
    g_peak = bins[np.argmax(flux)]
    assert 1.0 < g_peak < 1.15  # blue horn of an a = 0.998 disc seen at 40 degrees
    # strided oracle sample: every 255th ray (65 536 rays) through the oracle's line-profile path, compared as a histogram,
    # and ray by ray through the fused render of the same rays
    rng = cabi.Range(29, 65536, 255)
    want = oracle.lineprofile(p, ic, emis, bins, opts, rng=rng)
    got = hist(rng)
    assert np.abs(got - want).sum() <= 1e-4 * np.abs(want).sum()
    pfs = np.array([cabi.PF_REDSHIFT, cabi.PF_DISC_RADIUS, cabi.PF_STATUS], np.int32)
    imgs = np.zeros((3, rng.count))
    cabi.check(lib.gb200_render(ctx, C.byref(p), C.byref(ic), C.byref(rng), cabi.iptr(pfs), 3, None, (cabi._dp * 3)(*[cabi.dptr(imgs[k]) for k in range(3)])), ctx)
    check_sampled_parity(p, ic, rng, imgs[0], imgs[1], imgs[2], "C3 4096x4096", 2e-3)


def test_full_size_johannsen_psaltis_properties(ensemble):
    """BASELINE configs[4] at full size (JP a = 0.6, eps3 = 2, 2048 x 2048): determinism, shard invariance, physical ranges
    and a strided oracle sample (the generated closed-form Jacobian against the oracle's dual numbers)."""
    m, x, d, cfg = common.c5(2048, 2048, ensemble=ensemble)
    p, ic = cfg.to_c()
    lib = cabi.load()
    ctx = ensemble.ctx(ensemble.devices[0])
    pfs = np.array([cabi.PF_REDSHIFT, cabi.PF_DISC_RADIUS, cabi.PF_STATUS], np.int32)

    def render(rng):
        imgs = np.zeros((3, rng.count))
        ptrs = (cabi._dp * 3)(*[cabi.dptr(imgs[k]) for k in range(3)])
        cabi.check(lib.gb200_render(ctx, C.byref(p), C.byref(ic), C.byref(rng), cabi.iptr(pfs), 3, None, ptrs), ctx)
        return imgs

    full = render(cabi.Range(0, ic.n, 1))
    assert np.array_equal(full, render(cabi.Range(0, ic.n, 1)), equal_nan=True)
    shard = render(cabi.Range(5, ic.n // 8, 8))
    assert np.array_equal(shard, full[:, 5::8][:, : ic.n // 8], equal_nan=True)
    g, rho, status = full
    hit = status == cabi.STATUS_INTERSECTED
    assert np.array_equal(np.isnan(g), ~hit) and 0.3 < hit.mean() < 0.5
    assert np.nanmin(rho) >= gb.isco(m) * (1 - 1e-12) and np.nanmax(rho) <= 50.0 * (1 + 1e-12)
    assert 0.1 < np.nanmin(g) < 0.5 and 1.1 < np.nanmax(g) < 1.5
    rng = cabi.Range(23, 65536, 63)  # every 63rd ray: 65 536 rays
    got = full[:, 23::63][:, :65536]
    check_sampled_parity(p, ic, rng, got[0], got[1], got[2], "C5 2048x2048", 6e-3)


# --------------------------------------------------------------------------- the library's own multi-device path
def _comm(devices):
    h = C.c_void_p()
    devs = np.array(devices, np.int32)
    cabi.check(cabi.load().gb200_comm_init(cabi.iptr(devs), len(devs), C.byref(h)))
    return h


@pytest.mark.gpu
def test_comm_entry_points_on_one_device_equal_the_single_context_calls(ensemble):
    """`gb200_comm_render` / `gb200_comm_lineprofile` (one process, NCCL inside the library) with a single device: the same
    numbers as `gb200_render` / `gb200_lineprofile`; a device listed twice is refused."""
    lib = cabi.load()
    m, x, d, cfg = common.c1(96, 64, ensemble=ensemble)
    p, ic = cfg.to_c()
    pfs = np.array([cabi.PF_REDSHIFT, cabi.PF_DISC_RADIUS], np.int32)
    a, b = np.zeros((2, ic.n)), np.zeros((2, ic.n))
    rng = cabi.Range(0, ic.n, 1)
    cabi.check(lib.gb200_render(ensemble.ctx(0), C.byref(p), C.byref(ic), C.byref(rng), cabi.iptr(pfs), 2, None,
                                (cabi._dp * 2)(cabi.dptr(a[0]), cabi.dptr(a[1]))), ensemble.ctx(0))
    comm = _comm([0])
    try:
        assert lib.gb200_comm_size(comm) == 1 and lib.gb200_comm_context(comm, 0)
        cabi.check(lib.gb200_comm_render(comm, C.byref(p), C.byref(ic), cabi.iptr(pfs), 2, None, (cabi._dp * 2)(cabi.dptr(b[0]), cabi.dptr(b[1]))))
        assert np.array_equal(a, b, equal_nan=True)
        m, x, d, plane, cfg = common.c3(64, 64, ensemble=ensemble)
        p, ic = cfg.to_c()
        bins = np.ascontiguousarray(np.linspace(0.1, 1.5, 180))
        emis = cabi.Emissivity(cabi.EMISSIVITY_POWERLAW, 0, 3.0, None, None)
        opts = cabi.LineProfileOpts(gb.isco(m), 50.0, 1, 0)
        f1, f2 = np.zeros(180), np.zeros(180)
        rng = cabi.Range(0, ic.n, 1)
        cabi.check(lib.gb200_lineprofile(ensemble.ctx(0), C.byref(p), C.byref(ic), C.byref(rng), C.byref(emis), None, cabi.dptr(bins), 180,
                                         C.byref(opts), cabi.dptr(f1)), ensemble.ctx(0))
        cabi.check(lib.gb200_comm_lineprofile(comm, C.byref(p), C.byref(ic), C.byref(emis), None, cabi.dptr(bins), 180, C.byref(opts), cabi.dptr(f2)))
        assert np.array_equal(f1, f2)
    finally:
        lib.gb200_comm_destroy(comm)
    h = C.c_void_p()
    devs = np.array([0, 0], np.int32)
    assert lib.gb200_comm_init(cabi.iptr(devs), 2, C.byref(h)) == cabi.ERR_INVALID_ARGUMENT


@pytest.mark.gpu
def test_comm_entry_points_over_two_devices(ensemble):
    """Real distinct GPUs in one process (run under `gpurun --gpus 2`): the image equals the single-GPU image bit for bit
    (a ray's result does not depend on who traces it) and the NCCL-reduced histogram equals the single-GPU one to the
    order of summation."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    lib = cabi.load()
    ens2 = gb.EnsembleB200(devices=(0, 1))
    m, x, d, cfg = common.c1(256, 128, ensemble=ensemble)
    pf = [gb.ConstPointFunctions.redshift(m, x) @ gb.ConstPointFunctions.filter_intersected()]
    one = gb.api.apply_point_functions(cfg, pf)
    cfg2 = common.c1(256, 128, ensemble=ens2)[3]
    two = gb.api.apply_point_functions(cfg2, pf)
    assert np.array_equal(one, two, equal_nan=True)
    bins = np.linspace(0.1, 1.5, 180)
    plane = gb.PolarPlane(gb.GeometricGrid(), Nr=256, Ntheta=256, r_min=1.0, r_max=250.0)
    m = gb.KerrMetric(1.0, 0.998)
    x = [0.0, 1000.0, math.radians(40.0), 0.0]
    _, f1 = gb.lineprofile(bins, gb.PowerLawEmissivity(3.0), m, x, gb.ThinDisc(0.0, 400.0), gb.BinningMethod(), plane=plane, lambda_max=2000.0, ensemble=ensemble)
    _, f2 = gb.lineprofile(bins, gb.PowerLawEmissivity(3.0), m, x, gb.ThinDisc(0.0, 400.0), gb.BinningMethod(), plane=plane, lambda_max=2000.0, ensemble=ens2)
    assert np.abs(f1 - f2).sum() <= 1e-12 * f1.max() * len(bins)
    ens2.close()


# --------------------------------------------------------------------------- seeded random configurations
def _random_config(seed, ensemble):
    """Metric, spin, deformation, observer radius and inclination, disc extent and field of view drawn from a seeded
    generator: the main parity protocol away from the hand-picked fixtures."""
    rng = np.random.default_rng(4200 + seed)
    if seed % 2 == 0:
        m = gb.KerrMetric(1.0, float(rng.uniform(-0.95, 0.998)))
    else:
        m = gb.JohannsenPsaltisMetric(1.0, float(rng.uniform(-0.9, 0.9)), float(rng.uniform(-0.3, 1.0)))
    r_obs = float(10.0 ** rng.uniform(2.3, 3.3))
    x = [0.0, r_obs, math.radians(float(rng.uniform(15.0, 88.0))), 0.0]
    outer = float(rng.uniform(15.0, 60.0))
    inner = 0.0 if rng.uniform() < 0.5 else gb.isco(m)
    d = gb.ThinDisc(inner, outer)
    cfg = common.render_config(m, x, d, 2.0 * r_obs + 200.0, 64, 64, (-1.2 * outer, 1.2 * outer), (-0.9 * outer, 0.9 * outer), ensemble=ensemble)
    return m, x, d, cfg


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(8))
def test_seeded_random_configurations(ensemble, seed):
    m, x, d, cfg = _random_config(seed, ensemble)
    p, ic, ref, gps, band = check_parity(cfg, f"random configuration {seed}", max_band=0.01)  # measured 0.15 - 0.54 %
    hit = ~band & (ref.status == cabi.STATUS_INTERSECTED)
    assert hit.sum() > 100
    print(f"random configuration {seed}: {type(m).__name__} {m.params()[:3]} r_obs {x[1]:.0f} theta {math.degrees(x[2]):.1f} disc ({d.inner_radius:.2f}, {d.outer_radius:.1f}): "
          f"band {band.mean():.3%}, {int(hit.sum())} disc hits")


def _random_config_other_metrics(seed, ensemble):
    """The generated-Jacobian metrics and the other geometries under the same protocol."""
    rng = np.random.default_rng(9100 + seed)
    k = seed % 3
    if k == 0:
        m = gb.JohannsenMetric(1.0, float(rng.uniform(-0.8, 0.8)), *(float(v) for v in rng.uniform(-0.3, 0.3, 4)))
    elif k == 1:
        m = gb.BumblebeeMetric(1.0, float(rng.uniform(-0.1, 0.1)), float(rng.uniform(-0.3, 0.5)))
    else:
        a, q = float(rng.uniform(-0.7, 0.7)), float(rng.uniform(0.0, 0.5))
        m = gb.KerrNewmanMetric(1.0, a, q)
    r_obs = float(10.0 ** rng.uniform(2.3, 3.0))
    x = [0.0, r_obs, math.radians(float(rng.uniform(20.0, 85.0))), 0.0]
    outer = float(rng.uniform(20.0, 50.0))
    g = seed % 4
    d = gb.ThinDisc(gb.isco(m), outer) if g in (0, 1) else (gb.ShakuraSunyaev(m, eddington_ratio=float(rng.uniform(0.1, 0.4))) if g == 2 else None)
    cfg = common.render_config(m, x, d, 2.0 * r_obs + 200.0, 64, 64, (-1.2 * outer, 1.2 * outer), (-0.9 * outer, 0.9 * outer), ensemble=ensemble)
    return m, x, d, cfg


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(9))
def test_seeded_random_configurations_other_metrics(ensemble, seed):
    m, x, d, cfg = _random_config_other_metrics(seed, ensemble)
    p, ic, ref, gps, band = check_parity(cfg, f"random configuration (other metrics) {seed}", max_band=0.01)
    print(f"random configuration (other metrics) {seed}: {type(m).__name__} {tuple(round(v, 3) for v in m.params()[:6])} r_obs {x[1]:.0f} theta {math.degrees(x[2]):.1f} "
          f"{type(d).__name__}: band {band.mean():.3%}, status counts {np.bincount(ref.status, minlength=4)}")


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(4))
def test_seeded_random_line_profiles(ensemble, seed):
    """PolarPlane + hemisphere callback + fused binned line profile at random spin, inclination, emissivity index, radial
    range and bin grid: L1(flux) against the oracle at the north-star tolerance."""
    rng = np.random.default_rng(7700 + seed)
    m = gb.KerrMetric(1.0, float(rng.uniform(-0.9, 0.998))) if seed % 2 == 0 else gb.JohannsenPsaltisMetric(1.0, float(rng.uniform(0.0, 0.8)), float(rng.uniform(0.0, 0.8)))
    x = [0.0, 1000.0, math.radians(float(rng.uniform(10.0, 80.0))), 0.0]
    max_re = float(rng.uniform(20.0, 80.0))
    d = gb.ThinDisc(0.0, 400.0)
    grid = (gb.GeometricGrid(), gb.LinearGrid(), gb.InverseGrid())[seed % 3]
    plane = gb.PolarPlane(grid, Nr=96, Ntheta=96, r_min=1.0, r_max=5.0 * max_re)
    nb = int(rng.integers(60, 300))
    bins = np.linspace(0.05, 1.6, nb)
    index = float(rng.uniform(2.0, 4.0))
    cfg = tracing_configuration(m, x, plane, d, (0.0, 2000.0), callback=gb.domain_upper_hemisphere(), ensemble=ensemble)
    p, ic = cfg.to_c()
    _, flux = gb.lineprofile(bins, gb.PowerLawEmissivity(index), m, x, d, gb.BinningMethod(), plane=plane, lambda_max=2000.0, max_re=max_re, ensemble=ensemble)
    emis = cabi.Emissivity(cabi.EMISSIVITY_POWERLAW, 0, index, None, None)
    want = oracle.lineprofile(p, ic, emis, bins, cabi.LineProfileOpts(gb.isco(m), max_re, 1, 0))
    l1 = np.abs(flux - want).sum()
    print(f"random line profile {seed}: {type(m).__name__} {tuple(round(v, 3) for v in m.params()[:3])} theta {math.degrees(x[2]):.1f} index {index:.2f} max_re {max_re:.1f} {nb} bins "
          f"{type(grid).__name__}: L1 = {l1:.2e}")
    assert flux.sum() == pytest.approx(1.0, abs=1e-12) and l1 < 1e-4


def _random_config_planes_and_fans(seed, ensemble):
    """Image planes (polar / Cartesian, every grid kind) with the hemisphere callback, and explicit-IC fans from an off-axis
    source with random directions: the remaining initial-condition kinds under the main protocol."""
    rng = np.random.default_rng(5300 + seed)
    m = gb.KerrMetric(1.0, float(rng.uniform(-0.9, 0.998)))
    d = gb.ThinDisc(0.0 if seed % 2 else gb.isco(m), float(rng.uniform(30.0, 120.0)))
    grid = (gb.LinearGrid(), gb.GeometricGrid(), gb.InverseGrid())[seed % 3]
    x = [0.0, 1000.0, math.radians(float(rng.uniform(20.0, 80.0))), 0.0]
    if seed < 3:
        plane = gb.PolarPlane(grid, Nr=48, Ntheta=64, r_min=1.0, r_max=float(rng.uniform(60.0, 150.0)))
        return tracing_configuration(m, x, plane, d, (0.0, 2200.0), callback=gb.domain_upper_hemisphere(), ensemble=ensemble)
    if seed < 6:
        plane = gb.CartesianPlane(grid, x_min=0.1, y_min=0.1, x_max=float(rng.uniform(40.0, 100.0)), y_max=float(rng.uniform(30.0, 80.0)), Nx=40, Ny=40)
        return tracing_configuration(m, x, plane, d, (0.0, 2200.0), callback=gb.domain_upper_hemisphere(), ensemble=ensemble)
    # a source off the axis, rays in random directions (unnormalised: the library constrains v^t like constrain_all)
    n = 2000
    src = [0.0, float(rng.uniform(4.0, 30.0)), float(rng.uniform(0.2, 1.2)), float(rng.uniform(0.0, 6.0))]
    dirs = rng.normal(size=(n, 3))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    vs = np.stack([np.zeros(n), dirs[:, 0], dirs[:, 1] / src[1], dirs[:, 2] / (src[1] * math.sin(src[2]))], axis=1)
    return tracing_configuration(m, src, vs, d, 5000.0, callback=gb.domain_upper_hemisphere(), ensemble=ensemble)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(9))
def test_seeded_random_planes_and_fans(ensemble, seed):
    cfg = _random_config_planes_and_fans(seed, ensemble)
    p, ic, ref, gps, band = check_parity(cfg, f"random plane / fan {seed}", max_band=0.01)
    print(f"random plane / fan {seed}: ic kind {ic.kind}, {ic.n} rays, band {band.mean():.3%}, status counts {np.bincount(ref.status, minlength=4)}")
    assert (ref.status == cabi.STATUS_INTERSECTED).sum() > 50
