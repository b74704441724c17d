"""Line profiles and lag-energy transfer functions integrated from Cunningham transfer functions on the device
(`integrate_lineprofiles`, `integrate_lagtransfers`, `gb200_tf_lineprofile`, `gb200_tf_lagtransfer`,
`lineprofile(..., TransferFunctionMethod())`) against the host quadrature they restate, `integrate_lineprofile` and
`integrate_lagtransfer` (src/transfer-functions/integration.jl), bin for bin."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

import gradus_b200 as gb
from gradus_b200 import _cabi as cabi
from gradus_b200 import api, corona
from gradus_b200 import reverberation as rv
from gradus_b200 import tf_integration as ti
from gradus_b200 import transfer_functions as tf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

REF_LAG_ROW_40 = 0.021759503160585468  # test-2d.jl:65
REF_FREQ_SUM = 2449.8787687490535      # reverberation.jl:44
REF_TAU_132 = 9.322742661315855        # reverberation.jl:45


def synthetic_itb(n_radii=6, nan_knots=False, seed=0):
    """Closed (g✶, f) curves per radius, split and interpolated as the host does; optionally with NaN knots in f and t."""
    rng = np.random.default_rng(seed)
    brs = []
    for r in ti.inverse_grid(2.0, 40.0, n_radii):
        th = np.sort(rng.uniform(0, 2 * math.pi, 60))
        gs = (1 - np.cos(th)) / 2
        f = 1.0 + 0.3 * np.sin(th)
        t = r * (1 + 0.1 * np.sin(th))
        if nan_knots:
            f[rng.integers(0, 60, 4)] = np.nan
            t[rng.integers(0, 60, 4)] = np.nan
        ctf = tf.CunninghamTransferData(f, (gs - gs.min()) / (gs.max() - gs.min()), t, 0.5 - 0.1 / r**0.5, 1.0 + 0.3 / r**0.5, r, th)
        brs.append(ti.interpolate_branches(ctf))
    return ti.InterpolatingTransferBranches(brs)


def unpack_branches(p: ti.PackedBranches) -> ti.InterpolatingTransferBranches:
    brs = []
    for k, r in enumerate(p.r_e):
        sl = [slice(p.off[2 * k + b], p.off[2 * k + b + 1]) for b in (0, 1)]
        lo = (ti.NaNLinearInterpolator(p.gs[sl[0]], p.f[sl[0]]), ti.NaNLinearInterpolator(p.gs[sl[0]], p.t[sl[0]]))
        up = (ti.NaNLinearInterpolator(p.gs[sl[1]], p.f[sl[1]]), ti.NaNLinearInterpolator(p.gs[sl[1]], p.t[sl[1]]))
        brs.append(ti.TransferBranches(up[0], lo[0], up[1], lo[1], p.gmin[k], p.gmax[k], r))
    return ti.InterpolatingTransferBranches(brs)


def flat_itb():
    """The flat table of test_tf_integration.test_quadrature_of_a_flat_transfer_function_is_analytic."""
    flat = ti.NaNLinearInterpolator([0.0, 1.0], [1.0, 1.0])
    zero_t = ti.NaNLinearInterpolator([0.0, 1.0], [0.0, 0.0])
    return ti.InterpolatingTransferBranches([ti.TransferBranches(flat, flat, zero_t, zero_t, 0.5, 1.0, r) for r in (5.0, 6.0)])


# --------------------------------------------------------------------------- no device needed
def test_ctypes_layout_of_the_quadrature_structs_matches_header():
    fields = {"gb200_tf_branches": (cabi.TfBranches, ["n_radii", "reserved", "r_e", "gmin", "gmax", "off", "gs", "f", "t"]),
              "gb200_tf_model": (cabi.TfModel, ["table", "n_radii", "radii", "rmin", "g_scale", "profile"]),
              "gb200_tf_quad_opts": (cabi.TfQuadOpts, ["h", "t0", "upscale", "npoints", "nodes", "weights", "normalise", "reserved"])}
    body = "".join(f'  printf("%zu\\n", sizeof({s}));\n' + "".join(f'  printf("%zu\\n", offsetof({s}, {f}));\n' for f in fs)
                   for s, (_, fs) in fields.items())
    src = f"#include <stdio.h>\n#include <stddef.h>\n#include \"gradus_b200.h\"\nint main(void) {{\n{body}  return 0; }}\n"
    with tempfile.TemporaryDirectory() as d:
        cfile, exe = os.path.join(d, "q.c"), os.path.join(d, "q")
        open(cfile, "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), cfile, "-o", exe])
        got = [int(v) for v in subprocess.check_output([exe], text=True).split()]
    want = []
    for S, fs in fields.values():
        want += [C.sizeof(S)] + [getattr(S, f).offset for f in fs]
    assert got == want


@pytest.mark.parametrize("nan_knots", [False, True])
def test_packed_branches_reproduce_the_table(nan_knots):
    itb = synthetic_itb(nan_knots=nan_knots)
    p = ti.pack_branches(itb)
    assert p.off[0] == 0 and p.off.size == 2 * itb.radii.size + 1 and p.gs.size == p.off[-1] == p.f.size == p.t.size
    back = unpack_branches(p)
    x = np.concatenate([np.linspace(-0.2, 1.2, 57), [0.0, 1.0, 1e-8, 1 - 1e-8]])
    radii = np.concatenate([itb.radii, 0.5 * (itb.radii[1:] + itb.radii[:-1]), [1.5, 45.0]])
    for r in radii:
        a, b = itb(r), back(r)
        assert (a.gmin, a.gmax, a.r_e) == (b.gmin, b.gmax, b.r_e)
        for fn in ("upper_f", "lower_f", "upper_t", "lower_t"):
            assert np.array_equal(getattr(a, fn)(x), getattr(b, fn)(x), equal_nan=True), (r, fn)


@pytest.fixture
def no_library(monkeypatch):
    def refuse():
        raise AssertionError("the library was called")

    monkeypatch.setattr(cabi, "load", refuse)


def test_argument_errors_raise_before_any_library_call(no_library):
    itb, g = synthetic_itb(), np.linspace(0.3, 1.4, 20)
    pl = gb.PowerLawEmissivity(3.0)
    with pytest.raises(TypeError, match="integrate_lineprofile"):
        ti.integrate_lineprofiles(lambda r: r**-3.0, itb, g)
    prof = rv.AnalyticRadialDiscProfile(lambda r: r**-3.0, ti.NaNLinearInterpolator([1.0, 50.0], [0.0, 49.0]))
    with pytest.raises(TypeError, match="integrate_lagtransfer"):
        ti.integrate_lagtransfers(prof, itb, g, np.linspace(0, 100, 10))
    odd = ti.InterpolatingTransferBranches([ti.TransferBranches(lambda x: x, b.lower_f, b.upper_t, b.lower_t, b.gmin, b.gmax, b.r_e)
                                            for b in itb.branches])
    with pytest.raises(TypeError, match="NaNLinearInterpolator"):
        ti.integrate_lineprofiles(pl, odd, g)
    with pytest.raises(ValueError, match="table index"):
        ti.integrate_lineprofiles(pl, [itb, itb], g, table_of=[0, 2])
    with pytest.raises(ValueError, match="n_radii"):
        ti.integrate_lineprofiles(pl, itb, g, n_radii=1)
    with pytest.raises(ValueError, match="ascending"):
        ti.integrate_lineprofiles(pl, itb, g[::-1])
    with pytest.raises(ValueError, match="ascending"):
        ti.integrate_lagtransfers(rv.AnalyticRadialDiscProfile(pl, prof.t), itb, g, [0.0, 2.0, 1.0])
    with pytest.raises(ValueError, match="quadrature_points"):
        ti.integrate_lineprofiles(pl, itb, g, quadrature_points=33)
    with pytest.raises(ValueError, match="2 values for 3 models"):
        ti.integrate_lineprofiles([pl, pl], itb, g, g_scale=[1.0, 1.1, 1.2])
    with pytest.raises(TypeError, match="PowerLawEmissivity"):
        gb.lineprofile(g, lambda r: r**-3.0, gb.KerrMetric(1.0, 0.6), [0.0, 1000.0, 1.0, 0.0], gb.ThinDisc(0.0, 50.0),
                       gb.TransferFunctionMethod())


# --------------------------------------------------------------------------- device
def assert_same_bins(dev, host, tol):
    assert dev.shape == host.shape
    assert np.array_equal(dev == 0, host == 0)
    assert np.abs(dev - host).max() <= tol * np.abs(host).max(), np.abs(dev - host).max() / np.abs(host).max()


def raw_call(lag, tables, models, g, opts, t_grid=None):
    """The C ABI directly (no Python checks): (return code, output, stats)."""
    ens = api.default_ensemble()
    ctx = ens.ctx(ens.devices[0])
    lib = cabi.load()
    T, M = (cabi.TfBranches * len(tables))(*tables), (cabi.TfModel * len(models))(*models)
    if lag:
        out = np.zeros(len(models) * g.size * t_grid.size)
        rc = lib.gb200_tf_lagtransfer(ctx, len(tables), T, len(models), M, cabi.dptr(g), g.size, cabi.dptr(t_grid), t_grid.size,
                                      C.byref(opts), cabi.dptr(out))
    else:
        out = np.zeros(len(models) * g.size)
        rc = lib.gb200_tf_lineprofile(ctx, len(tables), T, len(models), M, cabi.dptr(g), g.size, C.byref(opts), cabi.dptr(out))
    return rc, out, ens.stats()


@pytest.mark.gpu
def test_flat_transfer_function_matches_the_host_and_the_closed_form():
    itb, grid = flat_itb(), np.linspace(0.4, 1.1, 141)
    eps = gb.PowerLawEmissivity(0.0)  # ε ≡ 1
    host = ti.integrate_lineprofile(eps, itb, grid, n_radii=4)
    dev = ti.integrate_lineprofiles(eps, itb, grid, n_radii=4)[0]
    assert_same_bins(dev, host, 1e-13)
    assert dev.sum() == pytest.approx(1.0) and dev[-1] == 0.0
    # raw sums: every annulus integrates the same flat function, so Σ bins = closed form × Σ annulus weights
    gmin, gmax = 0.5, 1.0
    phi = np.linspace(0, math.pi / 2, 200001)
    exact = np.trapezoid(4 * (gmax - gmin) * (gmin + (gmax - gmin) * np.sin(phi) ** 2) ** 3, phi)
    radii = np.ascontiguousarray(ti.inverse_grid(5.0, 6.0, 4))
    r_prev = np.concatenate([[5.0 - (radii[1] - 5.0)], radii[:-1]])
    weights = (radii - r_prev) * radii * math.pi / (gmax - gmin)
    pk = ti.pack_branches(itb)
    X, W = (np.ascontiguousarray(a) for a in ti._gauss(7))
    model = cabi.TfModel(0, 4, cabi.dptr(radii), 5.0, 1.0, cabi.DiscProfile())
    model.profile.emissivity.kind = cabi.EMISSIVITY_POWERLAW
    rc, raw, _ = raw_call(False, [pk.to_c()], [model], grid, cabi.TfQuadOpts(1e-8, 0.0, 1, 7, cabi.dptr(X), cabi.dptr(W), 0, 0))
    assert rc == cabi.OK
    assert abs(raw.sum() / (exact * weights.sum()) - 1) < 2e-2
    norm = raw[:-1] / (grid[1:] + grid[:-1])
    assert np.abs(np.append(norm / norm.sum(), 0.0) - dev).max() <= 1e-13 * dev.max()


X60 = [0.0, 1000.0, math.radians(60), 0.0]


@pytest.fixture(scope="module")
def line_tables():
    """Kerr and Johannsen-Psaltis thin discs (test_transfer_function_line_profile_on_the_device) and the Shakura-Sunyaev
    disc of test_thick_disc_line_profile_on_the_device, computed on the device."""
    kerr, jp = gb.KerrMetric(1.0, 0.6), gb.JohannsenPsaltisMetric(1.0, 0.6, 2.0)
    thin = gb.ThinDisc(0.0, 250.0)
    return {"kerr": ti.transferfunctions(kerr, X60, thin, N=40, num_re=30),
            "johannsen_psaltis": ti.transferfunctions(jp, X60, thin, N=40, num_re=30),
            "shakura_sunyaev": ti.transferfunctions(kerr, X60, gb.ShakuraSunyaev(kerr, eddington_ratio=0.3), N=40, num_re=30,
                                                    min_re=gb.isco(kerr) + 1e-2)}


@pytest.mark.gpu
@pytest.mark.parametrize("table", ["kerr", "johannsen_psaltis", "shakura_sunyaev"])
def test_line_profiles_match_the_host_quadrature(line_tables, table):
    itb = line_tables[table]
    bins = np.linspace(0.1, 1.3, 100)
    r_in, r_out = itb.inner_radius(), itb.outer_radius()
    tab = gb.TabulatedEmissivity(np.geomspace(r_in, r_out, 40), np.geomspace(r_in, r_out, 40) ** -2.5 * (1 + 0.2 * np.sin(np.arange(40))))
    emis = [gb.PowerLawEmissivity(3.0), tab, gb.PowerLawEmissivity(2.2), tab]
    g_scale = [1.0, 1.25, 1.0, 0.9]
    rmin = [None, None, r_in + 0.7, r_in + 0.3]
    rmax = [None, None, 0.6 * r_out, 30.0]
    n_radii = [1000, 1000, 400, 400]
    for up in (1, 3):
        dev = ti.integrate_lineprofiles(emis, itb, bins, rmin=rmin, rmax=rmax, g_scale=g_scale, n_radii=n_radii, g_grid_upscale=up)
        for k in range(len(emis)):
            host = ti.integrate_lineprofile(emis[k], itb, bins, rmin=rmin[k], rmax=rmax[k], g_scale=g_scale[k], n_radii=n_radii[k],
                                            g_grid_upscale=up)
            assert_same_bins(dev[k], host, 1e-12)


def reference_lag_setup():
    """run_reference_test of test_reverberation.py: sampled-sky emissivity profile and five transfer functions."""
    m = gb.KerrMetric(1.0, 0.998)
    x = [0.0, 1e6, math.radians(30), 0.0]
    d = gb.ThinDisc(gb.isco(m), 500.0)
    model = corona.LampPostModel(h=10.0, theta=math.radians(0.0001))
    prof = corona.emissivity_profile(m, d, model, n_samples=5000, sampler=corona.EvenSampler("both", "golden"))
    radii = ti.inverse_grid(gb.isco(m), 100.0, 5)
    itb = ti.transferfunctions(m, x, gb.ThinDisc(0.0, 500.0), radii=radii)
    return x, prof, radii, itb


@pytest.mark.gpu
def test_lag_transfer_matches_the_host_and_the_reference_literal():
    x, prof, radii, itb = reference_lag_setup()
    g, t = np.linspace(0.0, 1.5, 100), np.linspace(0.0, 150.0, 100)
    kw = dict(t0=x[1], n_radii=1000, rmin=radii.min(), rmax=radii.max())
    # the sampled profile (np.interp times) and the same table as an AnalyticRadialDiscProfile (NaNLinearInterpolator times)
    analytic = rv.AnalyticRadialDiscProfile(gb.PowerLawEmissivity(3.0), ti.NaNLinearInterpolator(prof.radii, prof.t))
    dev = ti.integrate_lagtransfers([prof, analytic], itb, g, t, **kw)
    for k, p in enumerate((prof, analytic)):
        host = ti.integrate_lagtransfer(p, itb, g, t, **kw)
        assert_same_bins(dev[k], host, 1e-12)
    assert dev[0].sum() == pytest.approx(1.0) and np.all(dev[0][-1] == 0)
    assert abs(dev[0][39].sum() - REF_LAG_ROW_40) < 1e-5
    up = ti.integrate_lagtransfers(prof, itb, g, t, g_grid_upscale=3, g_scale=1.1, **kw)[0]
    assert_same_bins(up, ti.integrate_lagtransfer(prof, itb, g, t, g_grid_upscale=3, g_scale=1.1, **kw), 1e-12)


@pytest.mark.gpu
def test_lag_frequency_smoke_through_the_device_quadrature():
    """run_lag_frequency_smoke of test_reverberation.py with the quadrature on the device."""
    m = gb.KerrMetric(1.0, 0.998)
    x = [0.0, 10_000.0, math.radians(45), 0.0]
    d = gb.ThinDisc(0.0, float("inf"))
    model = corona.LampPostModel()
    radii = ti.inverse_grid(gb.isco(m), 100.0, 10)
    itb = ti.transferfunctions(m, x, d, radii=radii, beta0=2.0)
    prof = corona.emissivity_profile(m, d, model, n_samples=500)
    t0 = rv.continuum_time(m, x, model)
    bins, tbins = np.linspace(0.0, 1.5, 100), np.linspace(0.0, 100.0, 100)
    kw = dict(t0=t0, n_radii=100, h=1e-8, rmin=radii.min(), rmax=radii.max())
    flux = ti.integrate_lagtransfers(prof, itb, bins, tbins, **kw)[0]
    assert_same_bins(flux, ti.integrate_lagtransfer(prof, itb, bins, tbins, **kw), 1e-12)
    flux[flux == 0] = np.nan
    freq, tau = rv.lag_frequency(tbins, flux)
    assert freq.sum() == pytest.approx(REF_FREQ_SUM, rel=1e-2)
    assert tau[131] == pytest.approx(REF_TAU_132, rel=1e-2)


@pytest.mark.gpu
def test_batches_are_bit_identical_to_single_calls_and_ignore_the_order(line_tables):
    itbs = list(line_tables.values())
    rng = np.random.default_rng(7)
    n = 64
    table_of = rng.integers(0, 3, n)
    emis = [gb.PowerLawEmissivity(float(rng.uniform(2, 4))) if k % 2 else
            gb.TabulatedEmissivity(np.linspace(1.0, 60.0, 30), rng.uniform(0.5, 1.5, 30)) for k in range(n)]
    g_scale = rng.uniform(0.9, 1.2, n)
    rmin = [itbs[t].inner_radius() + rng.uniform(0, 0.5) for t in table_of]
    bins, tb = np.linspace(0.1, 1.3, 60), np.linspace(0.0, 80.0, 40)
    kw = dict(table_of=table_of, g_scale=g_scale, rmin=rmin, n_radii=150)
    times = [rv.AnalyticRadialDiscProfile(e, ti.NaNLinearInterpolator(np.linspace(1.0, 60.0, 20), np.linspace(5.0, 60.0, 20)))
             for e in emis]
    perm = rng.permutation(n)
    shuffled = dict(table_of=table_of[perm], g_scale=g_scale[perm], rmin=[rmin[i] for i in perm], n_radii=150)
    line = ti.integrate_lineprofiles(emis, itbs, bins, **kw)
    lag = ti.integrate_lagtransfers(times, itbs, bins, tb, t0=3.0, **kw)
    assert np.array_equal(ti.integrate_lineprofiles([emis[i] for i in perm], itbs, bins, **shuffled), line[perm])
    assert np.array_equal(ti.integrate_lagtransfers([times[i] for i in perm], itbs, bins, tb, t0=3.0, **shuffled), lag[perm])
    for k in range(n):
        one = dict(table_of=int(table_of[k]), g_scale=g_scale[k], rmin=rmin[k], n_radii=150)
        assert np.array_equal(ti.integrate_lineprofiles(emis[k], itbs, bins, **one)[0], line[k])
        assert np.array_equal(ti.integrate_lagtransfers(times[k], itbs, bins, tb, t0=3.0, **one)[0], lag[k])


@pytest.mark.gpu
@pytest.mark.parametrize("m, g_low_ref", [(gb.KerrMetric(1.0, 0.6), 0.355), (gb.JohannsenPsaltisMetric(1.0, 0.6, 2.0), 0.27)],
                         ids=["kerr", "johannsen_psaltis"])
def test_lineprofile_with_the_transfer_function_method(m, g_low_ref):
    """test/line-profiles/test-cunningham.jl through `lineprofile(..., TransferFunctionMethod())`, and the cross-check against
    the device's binned line profile that test_tf_integration makes for the host quadrature."""
    d = gb.ThinDisc(0.0, 250.0)
    bins = np.linspace(0.1, 1.3, 100)
    _, y = gb.lineprofile(bins, gb.PowerLawEmissivity(3.0), m, X60, d, gb.TransferFunctionMethod(N=40, num_re=30))
    nz = np.nonzero(y > 0)[0]
    assert abs(bins[nz[0]] - g_low_ref) < 0.05 and abs(bins[nz[-1]] - 1.2) < 0.05 and y.sum() == pytest.approx(1.0)
    _, yb = gb.lineprofile(bins, gb.PowerLawEmissivity(3.0), m, X60, d, gb.BinningMethod(), min_re=gb.isco(m) + 1e-2, max_re=50.0)
    assert np.abs(y - yb).sum() < 0.03


@pytest.mark.gpu
def test_device_validation_rejects_bad_tables_and_models_without_a_launch():
    itb = synthetic_itb()
    g = np.linspace(0.3, 1.4, 20)
    X, W = (np.ascontiguousarray(a) for a in ti._gauss(7))
    opts = cabi.TfQuadOpts(1e-8, 0.0, 1, 7, cabi.dptr(X), cabi.dptr(W), 1, 0)
    radii = np.ascontiguousarray(ti.inverse_grid(2.0, 40.0, 50))

    def model(table=0, n=50, r=radii):
        mo = cabi.TfModel(table, n, cabi.dptr(r), float(r[0]), 1.0, cabi.DiscProfile())
        mo.profile.emissivity.kind, mo.profile.emissivity.index = cabi.EMISSIVITY_POWERLAW, 3.0
        return mo

    good = ti.pack_branches(itb)
    rc, _, st = raw_call(False, [good.to_c()], [model()], g, opts)
    assert rc == cabi.OK and st.launches == 2

    descending = np.ascontiguousarray(radii[::-1])
    alive = []  # the packed arrays must outlive the calls that read them through pointers

    def bad_table(edit):
        p = ti.pack_branches(itb)
        p = ti.PackedBranches(*(np.array(a) for a in (p.r_e, p.gmin, p.gmax, p.off, p.gs, p.f, p.t)))
        edit(p)
        alive.append(p)
        return p

    cases = {
        "table index": ([good.to_c()], [model(table=1)], opts),
        "n_radii": ([good.to_c()], [model(n=1)], opts),
        "radii must be": ([good.to_c()], [model(r=descending)], opts),
        "2 knots": ([bad_table(lambda p: p.off.__setitem__(slice(1, None), p.off[1:] - p.off[1] + 1)).to_c()], [model()], opts),
        "gmin < gmax": ([bad_table(lambda p: p.gmax.__setitem__(2, p.gmin[2])).to_c()], [model()], opts),
        "r_e must be": ([bad_table(lambda p: p.r_e.__setitem__(1, p.r_e[0])).to_c()], [model()], opts),
        "Gauss points": ([good.to_c()], [model()], cabi.TfQuadOpts(1e-8, 0.0, 1, 33, cabi.dptr(X), cabi.dptr(W), 1, 0)),
        "h <": ([good.to_c()], [model()], cabi.TfQuadOpts(0.5, 0.0, 1, 7, cabi.dptr(X), cabi.dptr(W), 1, 0)),
    }
    lib = cabi.load()
    for what, (tables, models, o) in cases.items():
        rc, out, st = raw_call(False, tables, models, g, o)
        assert rc == cabi.ERR_INVALID_ARGUMENT, what
        assert what in lib.gb200_last_error(None).decode(), (what, lib.gb200_last_error(None))
        assert st.launches == 0 and not out.any(), what
    rc, _, st = raw_call(True, [good.to_c()], [model()], g, opts, t_grid=np.array([0.0, 5.0, 5.0]))
    assert rc == cabi.ERR_INVALID_ARGUMENT and st.launches == 0
