"""The binned lag-energy transfer function on the device (`binned_lagtransfer`, `gb200_lagtransfer`,
`gb200_comm_lagtransfer`) against the host composition `binflux(lagtransfer(...))` it replaces
(src/transfer-functions/transfer-functions-2d.jl:100-122,163-242)."""
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

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

REF_OBSERVER_TO_DISC = 337            # test-2d.jl:25
REF_BINFLUX_SUM = 3.9126785201177956  # test-2d.jl:32


def reference_fixture():
    """test/transfer-functions/test-2d.jl, as in test_reverberation.py"""
    m = gb.KerrMetric(1.0, 0.998)
    x = [0.0, 1e6, math.radians(30), 0.0]
    plane = gb.PolarPlane(gb.GeometricGrid(), Nr=20, Ntheta=20)
    d = gb.ThinDisc(gb.isco(m), 500.0)
    model = corona.LampPostModel(h=10.0, theta=math.radians(0.0001))
    return m, x, plane, d, model


def user_fixture():
    """The reference's default 800 x 800 plane (lagtransfer's default)."""
    m = gb.KerrMetric(1.0, 0.998)
    x = [0.0, 1e6, math.radians(30), 0.0]
    return m, x, gb.ThinDisc(gb.isco(m), 500.0), corona.LampPostModel(h=10.0)


# --------------------------------------------------------------------------- no device needed
def test_ctypes_layout_of_the_lag_structs_matches_header():
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "gradus_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(gb200_disc_profile), offsetof(gb200_disc_profile, time_kind),
         offsetof(gb200_disc_profile, n), offsetof(gb200_disc_profile, r), offsetof(gb200_disc_profile, t),
         sizeof(gb200_lagtransfer_opts), offsetof(gb200_lagtransfer_opts, t0), offsetof(gb200_lagtransfer_opts, energy_lims),
         offsetof(gb200_lagtransfer_opts, time_lims), offsetof(gb200_lagtransfer_opts, N_t));
  return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        cfile = os.path.join(d, "l.c")
        open(cfile, "w").write(src)
        exe = os.path.join(d, "l")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), cfile, "-o", exe])
        got = [int(v) for v in subprocess.check_output([exe], text=True).split()]
    P, O = cabi.DiscProfile, cabi.LagTransferOpts
    assert got == [C.sizeof(P), P.time_kind.offset, P.n.offset, P.r.offset, P.t.offset,
                   C.sizeof(O), O.t0.offset, O.energy_lims.offset, O.time_lims.offset, O.N_t.offset]


@pytest.mark.parametrize("plane", [gb.CartesianPlane(), api.RenderGrid(8, 8, (-10, 10), (-10, 10))])
def test_planes_without_an_area_weight_are_refused_before_tracing(plane):
    m, x, d, model = user_fixture()
    with pytest.raises(ValueError, match="PolarPlane"):
        rv.binned_lagtransfer(m, x, d, model, plane=plane)


def test_a_python_emissivity_is_refused_before_tracing():
    m, x, d, model = user_fixture()
    prof = rv.AnalyticRadialDiscProfile(lambda r: r ** -3.0, rv.NaNLinearInterpolator([1.0, 2.0], [0.0, 1.0]))
    with pytest.raises(TypeError, match="binflux"):
        rv.binned_lagtransfer(m, x, d, model, prof)


def test_emissivity_descriptors_evaluate_like_the_host_profiles():
    r = np.array([0.5, 1.0, 3.7, 12.0, 900.0])
    assert np.array_equal(api.PowerLawEmissivity(3.0)(r), r ** -3.0)
    tab = api.TabulatedEmissivity([1.0, 10.0, 100.0], [1.0, 0.1, 0.01])
    prof = corona.RadialDiscProfile(np.array([1.0, 10.0, 100.0]), np.array([1.0, 0.1, 0.01]), np.zeros(3))
    assert np.array_equal(tab(r), prof.emissivity_at(r))


# --------------------------------------------------------------------------- against the composition
def _scale(H, fmax):
    """The documented rule: the largest power of two with scale * H * max|f| <= 2^62."""
    mant, e = math.frexp(H * fmax)
    return math.ldexp(1.0, (63 if mant == 0.5 else 62) - e)


def _bucket(bins, v):
    return np.clip(np.searchsorted(bins, v, side="right") - 1, 0, len(bins) - 1)


def assert_equals_composition(got, lt, profile=None, E0=6.4, energy_lims=None, time_lims=None, N_E=300, N_t=300):
    """Same hits and NaN mask, edges within 1 ulp, and every cell within its quantisation bound: each of the cell's
    contributing samples is rounded by at most half a unit of 1 / scale, and so is each of the H terms of the total."""
    tb, eb, tf, hits = got
    kw = dict(E0=E0, N_E=N_E, N_t=N_t, energy_lims=energy_lims, time_lims=time_lims)
    tbh, ebh, tfh = rv.binflux(lt, profile, **kw)
    assert hits == lt.observer_to_disc_count
    assert tf.shape == tfh.shape == (N_E, N_t)
    assert np.all(np.abs(eb - ebh) <= np.spacing(np.abs(ebh)))
    assert np.all(np.abs(tb - tbh) <= np.spacing(np.abs(tbh)))
    assert np.array_equal(np.isnan(tf), np.isnan(tfh))
    prof = profile or rv.AnalyticRadialDiscProfile.from_corona(lambda r: r ** -3.0, lt.coronal_geodesics)
    f = lt.g ** 3 * prof.emissivity_at(lt.rho) * lt.image_plane_areas
    E, T = lt.g * E0, prof.coordtime_at(lt.rho) + lt.t
    elims = (E.min(), E.max()) if energy_lims is None else energy_lims
    tlims = (T.min(), T.max()) if time_lims is None else time_lims
    e_edges, t_edges = np.linspace(*elims, N_E), np.linspace(*tlims, N_t)
    count = np.zeros((N_E, N_t))
    np.add.at(count, (_bucket(e_edges, E), _bucket(t_edges, T)), f != 0)
    H, S = len(f), f.sum()
    scale = _scale(H, np.abs(f).max())
    dedt = (e_edges[1] - e_edges[0]) * (t_edges[1] - t_edges[0])
    ok = ~np.isnan(tfh)
    bound = count[ok] * 0.5 / (scale * S * dedt) + tfh[ok] * H * 0.5 / (scale * S) + 1e-13 * tfh[ok].max()
    assert np.all(np.abs(tf[ok] - tfh[ok]) <= bound)


@pytest.mark.gpu
def test_reference_literals_through_the_device_binning():
    m, x, plane, d, model = reference_fixture()
    sampler = corona.EvenSampler("both", "golden")
    got = rv.binned_lagtransfer(m, x, d, model, plane=plane, n_samples=100, sampler=sampler, N_E=100, N_t=100)
    assert got[3] == REF_OBSERVER_TO_DISC
    assert abs(np.nansum(got[2]) - REF_BINFLUX_SUM) < 1e-4
    lt = rv.lagtransfer(m, x, d, model, plane=plane, n_samples=100, sampler=sampler)
    assert_equals_composition(got, lt, N_E=100, N_t=100)


@pytest.fixture(scope="module")
def user_case():
    m, x, d, model = user_fixture()
    return m, x, d, model, rv.lagtransfer(m, x, d, model)


@pytest.mark.gpu
def test_default_profile_with_automatic_limits_equals_the_composition(user_case):
    m, x, d, model, lt = user_case
    got = rv.binned_lagtransfer(m, x, d, model)
    assert got[3] > 100_000
    assert_equals_composition(got, lt)


@pytest.mark.gpu
def test_radial_disc_profile_equals_the_composition(user_case):
    m, x, d, model, lt = user_case
    prof = corona.emissivity_profile(m, d, model, n_samples=2000, sampler=corona.EvenSampler("both", "golden"))
    assert_equals_composition(rv.binned_lagtransfer(m, x, d, model, prof), lt, prof)


@pytest.mark.gpu
def test_limits_narrower_than_the_data_clamp_into_the_edge_cells(user_case):
    m, x, d, model, lt = user_case
    _, eb, _ = rv.binflux(lt)
    tb = rv.binflux(lt)[0] + x[1]
    elims = (eb[60], eb[240])
    tlims = (tb[30], tb[150])
    prof = rv.AnalyticRadialDiscProfile.from_corona(api.TabulatedEmissivity([1.0, 10.0, 600.0], [1.0, 0.02, 1e-6]), lt.coronal_geodesics)
    got = rv.binned_lagtransfer(m, x, d, model, prof, energy_lims=elims, time_lims=tlims, E0=6.0, N_E=200, N_t=250)
    assert not np.isnan(got[2][0]).all() and not np.isnan(got[2][-1]).all()
    assert_equals_composition(got, lt, prof, E0=6.0, energy_lims=elims, time_lims=tlims, N_E=200, N_t=250)


@pytest.mark.gpu
def test_johannsen_psaltis_with_its_plunging_table_equals_the_composition():
    m = gb.JohannsenPsaltisMetric(1.0, 0.6, 2.0)
    x = [0.0, 1e4, math.radians(40), 0.0]
    d, model = gb.ThinDisc(0.0, 500.0), corona.LampPostModel(h=8.0)
    plane = gb.PolarPlane(gb.GeometricGrid(), Nr=120, Ntheta=120, r_max=50.0)
    lt = rv.lagtransfer(m, x, d, model, plane=plane, n_samples=2000)
    got = rv.binned_lagtransfer(m, x, d, model, plane=plane, n_samples=2000, N_E=120, N_t=120)
    assert_equals_composition(got, lt, N_E=120, N_t=120)


# --------------------------------------------------------------------------- determinism and devices
def _small_call(ensemble=None, **kw):
    m, x, plane, d, model = reference_fixture()
    plane = gb.PolarPlane(gb.GeometricGrid(), Nr=200, Ntheta=200, r_max=50.0)
    return rv.binned_lagtransfer(m, x, d, model, plane=plane, n_samples=1000, N_E=150, N_t=150, ensemble=ensemble, **kw)


def _bitwise_equal(a, b):
    return a[3] == b[3] and all(np.array_equal(u.view(np.int64), v.view(np.int64)) for u, v in zip(a[:3], b[:3]))


@pytest.mark.gpu
def test_repeated_calls_and_a_one_device_communicator_are_bitwise_identical():
    first, second = _small_call(), _small_call()
    assert _bitwise_equal(first, second)
    ens = gb.EnsembleB200((0,))
    h = C.c_void_p()
    cabi.check(cabi.load().gb200_comm_init(cabi.iptr(np.array([0], np.int32)), 1, C.byref(h)))
    ens._comm = h
    ens.comm = lambda: h  # EnsembleB200 uses per-device contexts for one device; force gb200_comm_lagtransfer
    try:
        assert _bitwise_equal(_small_call(ens), first)
    finally:
        ens.close()


@pytest.mark.gpu
def test_two_devices_give_the_one_device_bits():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two devices")
    ens = gb.EnsembleB200((0, 1))
    try:
        assert _bitwise_equal(_small_call(ens), _small_call())
    finally:
        ens.close()


# --------------------------------------------------------------------------- validation on the device
class _Call:
    """Direct gb200_lagtransfer calls on one context with a synthetic RadialDiscProfile-like table."""

    def __init__(self, ctx, m=None, plane=None, disc=None):
        m = m or gb.KerrMetric(1.0, 0.998)
        x = [0.0, 1e6, math.radians(30), 0.0]
        plane = plane or gb.PolarPlane(gb.GeometricGrid(), Nr=20, Ntheta=20)
        d = disc or gb.ThinDisc(gb.isco(m), 500.0)
        self.config = api.tracing_configuration(m, x, plane, d, (0.0, 2e6), chart=api.chart_for_metric(m, 1.1e6),
                                                callback=api.domain_upper_hemisphere())
        self.p, self.ic = self.config.to_c()
        self.ctx = ctx
        self.r = np.geomspace(1.0, 1000.0, 40)
        self.t = np.sqrt(self.r ** 2 + 100.0)

    def __call__(self, p=None, ic=None, r=None, eps_r=None, **opt):
        r = self.r if r is None else np.ascontiguousarray(r, np.float64)
        eps_r = self.r if eps_r is None else np.ascontiguousarray(eps_r, np.float64)
        eps = eps_r ** -3.0
        prof = cabi.DiscProfile()
        prof.emissivity.kind, prof.emissivity.n = cabi.EMISSIVITY_TABLE, len(eps_r)
        prof.emissivity.r, prof.emissivity.eps = cabi.dptr(eps_r), cabi.dptr(eps)
        prof.time_kind, prof.n, prof.r, prof.t = cabi.PROFILE_TIME_LINEAR, len(r), cabi.dptr(r), cabi.dptr(self.t)
        nan = float("nan")
        o = dict(E0=6.4, t0=1e6, energy_lims=(nan, nan), time_lims=(nan, nan), N_E=50, N_t=40)
        o.update(opt)
        opts = cabi.LagTransferOpts(o["E0"], o["t0"], tuple(o["energy_lims"]), tuple(o["time_lims"]), o["N_E"], o["N_t"])
        self.tb, self.eb = np.zeros(max(o["N_t"], 1)), np.zeros(max(o["N_E"], 1))
        ncell = o["N_E"] * o["N_t"]
        self.tf, self.hits = np.zeros(ncell if 0 < ncell <= 1 << 26 else 1), C.c_int64()
        return cabi.load().gb200_lagtransfer(self.ctx, C.byref(p or self.p), C.byref(ic or self.ic), C.byref(prof), None, C.byref(opts),
                                             cabi.dptr(self.tb), cabi.dptr(self.eb), cabi.dptr(self.tf), C.byref(self.hits))

    def launches(self):
        s = cabi.Stats()
        cabi.check(cabi.load().gb200_get_stats(self.ctx, C.byref(s)))
        return s.launches


@pytest.mark.gpu
def test_rejected_arguments_launch_nothing(ensemble):
    ctx = ensemble.ctx(ensemble.devices[0])
    call = _Call(ctx)
    assert call() == cabi.OK and call.hits.value == REF_OBSERVER_TO_DISC and call.launches() > 0
    cart = _Call(ctx, plane=gb.CartesianPlane(Nx=8, Ny=8))
    nan, inf = float("nan"), float("inf")
    cases = [
        (cabi.ERR_UNSUPPORTED, dict(p=cart.p, ic=cart.ic)),
        (cabi.ERR_INVALID_ARGUMENT, dict(N_E=1)),
        (cabi.ERR_INVALID_ARGUMENT, dict(N_t=1)),
        (cabi.ERR_INVALID_ARGUMENT, dict(N_E=1 << 13, N_t=(1 << 13) + 1)),
        (cabi.ERR_INVALID_ARGUMENT, dict(energy_lims=(2.0, 2.0))),
        (cabi.ERR_INVALID_ARGUMENT, dict(energy_lims=(3.0, 2.0))),
        (cabi.ERR_INVALID_ARGUMENT, dict(time_lims=(nan, 2e6))),
        (cabi.ERR_INVALID_ARGUMENT, dict(time_lims=(0.0, inf))),
        (cabi.ERR_INVALID_ARGUMENT, dict(r=call.r[::-1].copy())),
        (cabi.ERR_INVALID_ARGUMENT, dict(r=np.r_[call.r[:20], call.r[19:39]])),
        (cabi.ERR_INVALID_ARGUMENT, dict(eps_r=np.r_[call.r[:20], call.r[19:39]])),
        (cabi.ERR_INVALID_ARGUMENT, dict(E0=0.0)),
        (cabi.ERR_INVALID_ARGUMENT, dict(E0=-6.4)),
        (cabi.ERR_INVALID_ARGUMENT, dict(E0=inf)),
    ]
    for code, kw in cases:
        assert call(**kw) == code, kw
        assert call.launches() == 0, kw
    assert call() == cabi.OK and call.hits.value == REF_OBSERVER_TO_DISC


@pytest.mark.gpu
def test_findings_after_the_trace_are_reported(ensemble):
    ctx = ensemble.ctx(ensemble.devices[0])
    # every ray of a plane inside the shadow falls into the hole: automatic limits have nothing to take min / max of,
    # explicit limits give an all-NaN table
    miss = _Call(ctx, plane=gb.PolarPlane(gb.GeometricGrid(), Nr=8, Ntheta=8, r_min=0.5, r_max=1.5))
    assert miss() == cabi.ERR_INVALID_ARGUMENT and b"need hits" in cabi.load().gb200_last_error(ctx)
    assert miss(energy_lims=(1.0, 8.0), time_lims=(1e6, 1.1e6)) == cabi.OK and miss.hits.value == 0
    assert np.isnan(miss.tf).all()
    # a non-Kerr disc reaching inside the ISCO without a plunging table has hits with no redshift: reported, not dropped
    jp = gb.JohannsenPsaltisMetric(1.0, 0.6, 2.0)
    bad = _Call(ctx, m=jp, disc=gb.ThinDisc(0.0, 500.0), plane=gb.PolarPlane(gb.GeometricGrid(), Nr=40, Ntheta=40, r_max=20.0))
    assert bad() == cabi.ERR_INVALID_ARGUMENT and b"non-finite" in cabi.load().gb200_last_error(ctx)
    assert bad(energy_lims=(1.0, 8.0), time_lims=(1e6, 1.1e6)) == cabi.ERR_INVALID_ARGUMENT
