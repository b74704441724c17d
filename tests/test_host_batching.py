"""The batch entry points against single calls of the same items, bit for bit, for the cases their shared host plumbing
(one arena per batch, laid out per item, with plunging tables shared between consecutive items) has to get right: partial
outputs, empty items, mixed initial conditions, shared tables and per-ray heights; and the pipelined single call with
partial outputs against the one-launch path.  A batch that fails returns with nothing of it running, and fails before its
first launch where the host can tell."""
import ctypes as C
import math

import numpy as np
import pytest

import gradus_b200 as gb
from gradus_b200 import _cabi as cabi
from gradus_b200 import api

import common

pytestmark = pytest.mark.gpu

ENDPOINT_FIELDS = ("status", "lambda_max", "x", "v", "x_init", "v_init", "naccept", "nreject", "flags")
DUAL_FIELDS = ("status", "lambda_max", "x", "v", "g", "dg", "rho", "drho", "naccept", "nreject", "flags")


def _same_arrays(got, want, fields):
    for name in fields:
        a, b = getattr(got, name), getattr(want, name)
        assert (a is None) == (b is None), name
        if a is not None:
            assert np.array_equal(a, b, equal_nan=True), name


def _lamp_post(ensemble, n, a=0.9):
    delta = np.radians(np.linspace(0.01, 179.99, n))
    vs = np.stack([np.zeros_like(delta), -np.cos(delta), np.sin(delta) / 10.0, np.zeros_like(delta)], axis=1)
    return api.tracing_configuration(gb.KerrMetric(1.0, a), [0.0, 10.0, 0.01, 0.0], vs, gb.ThinDisc(0.0, 1000.0), 10000.0,
                                     callback=gb.domain_upper_hemisphere(), ensemble=ensemble)


def test_trace_batch_partial_outputs_empty_ranges_and_mixed_ics(ensemble):
    lib = cabi.load()
    ctx = ensemble.ctx(ensemble.devices[0])
    grid = common.c1(24, 24, ensemble=ensemble)[3]
    # (configuration, range, which outputs the caller asks for)
    items = [(_lamp_post(ensemble, 300), lambda n: cabi.Range(0, n, 1), dict(init=False, stats=False)),
             (grid, lambda n: cabi.Range(0, n, 1), dict(init=True, stats=False)),
             (_lamp_post(ensemble, 200, 0.5), lambda n: cabi.Range(0, 0, 1), dict()),  # empty: no launch, nothing written
             (grid, lambda n: cabi.Range(5, 70, 3), dict(init=False, stats=True)),  # strided structured range
             (_lamp_post(ensemble, 250, 0.998), lambda n: cabi.Range(10, 200, 1), dict())]
    pcs = [cfg.to_c() for cfg, _, _ in items]
    ranges = [mk(ic.n) for (_, mk, _), (_, ic) in zip(items, pcs)]
    singles, launches, rays, accepted = [], 0, 0, 0
    for (p, ic), rng, (_, _, kw) in zip(pcs, ranges, items):
        out = cabi.EndpointArrays(rng.count, **kw)
        cabi.check(lib.gb200_trace(ctx, C.byref(p), C.byref(ic), C.byref(rng), C.byref(out.c)), ctx)
        st = ensemble.stats()
        singles.append(out)
        launches, rays, accepted = launches + st.launches, rays + st.rays, accepted + st.steps_accepted
    nb = len(items)
    batch = [cabi.EndpointArrays(rng.count, **kw) for rng, (_, _, kw) in zip(ranges, items)]
    cabi.check(lib.gb200_trace_batch(ctx, nb, (cabi.Problem * nb)(*[p for p, _ in pcs]), (cabi.IC * nb)(*[ic for _, ic in pcs]),
                                     (cabi.Range * nb)(*ranges), (cabi.Endpoints * nb)(*[b.c for b in batch])), ctx)
    st = ensemble.stats()
    for got, want in zip(batch, singles):
        _same_arrays(got, want, ENDPOINT_FIELDS)
    assert batch[2].status.size == 0 and launches == nb - 1
    assert (st.launches, st.rays, st.steps_accepted) == (launches, rays, accepted)


def test_render_batch_shares_plunging_tables_and_skips_empty_items(ensemble):
    lib = cabi.load()
    ctx = ensemble.ctx(ensemble.devices[0])
    m = gb.JohannsenPsaltisMetric(1.0, 0.6, 2.0)
    table = api.interpolate_plunging_velocities(m, ensemble)  # the disc reaches inside the ISCO: the table is read
    disc = gb.ThinDisc(0.0, 50.0)
    cfgs = [common.render_config(m, [0.0, 1000.0, math.radians(inc), 0.0], disc, 2000.0, 20, 16, ensemble=ensemble) for inc in (60.0, 75.0)]
    rng = np.random.default_rng(9)
    al, be = rng.uniform(-20, 20, 150), rng.uniform(-20, 20, 150)
    cfgs.append(cfgs[0])  # empty item between two items with the same table
    cfgs.append(api.tracing_configuration(m, [0.0, 1000.0, math.radians(45.0), 0.0], api.ImpactParameters(al, be), disc, 2000.0,
                                          ensemble=ensemble))
    cfgs.append(common.c1(16, 16, ensemble=ensemble)[3])  # Kerr, no table
    tabs = [table, table, table, table, None]
    pcs = [c.to_c() for c in cfgs]
    counts = [ic.n for _, ic in pcs]
    counts[2] = 0
    pfs = np.array([cabi.PF_REDSHIFT, cabi.PF_STATUS], np.int32)
    npf, nb = len(pfs), len(cfgs)

    def pl(t):
        return C.byref(t.c) if t is not None else None

    singles = []
    for (p, ic), n, t in zip(pcs, counts, tabs):
        img = np.zeros((npf, n))
        ptrs = (cabi._dp * npf)(*[cabi.dptr(img[k]) for k in range(npf)])
        cabi.check(lib.gb200_render(ctx, C.byref(p), C.byref(ic), C.byref(cabi.Range(0, n, 1)), cabi.iptr(pfs), npf, pl(t), ptrs), ctx)
        singles.append(img)
    images = [np.zeros((npf, n)) for n in counts]
    ptrs = (cabi._dp * (nb * npf))(*[cabi.dptr(images[b][k]) if counts[b] else cabi.dptr(None) for b in range(nb) for k in range(npf)])
    PT = C.POINTER(cabi.PlungingTable)
    pl_ptrs = (PT * nb)(*[C.pointer(t.c) if t is not None else PT() for t in tabs])
    cabi.check(lib.gb200_render_batch(ctx, nb, (cabi.Problem * nb)(*[p for p, _ in pcs]), (cabi.IC * nb)(*[ic for _, ic in pcs]),
                                      (cabi.Range * nb)(*[cabi.Range(0, n, 1) for n in counts]), cabi.iptr(pfs), npf, pl_ptrs, ptrs), ctx)
    assert ensemble.stats().launches == nb - 1
    for got, want in zip(images, singles):
        assert np.array_equal(got, want, equal_nan=True)
    hit = singles[0][1] == cabi.STATUS_INTERSECTED
    assert hit.sum() > 50 and np.isfinite(singles[0][0][hit]).any()


def test_dual_batch_shares_plunging_tables_and_takes_heights(ensemble):
    m = gb.JohannsenPsaltisMetric(1.0, 0.6, 2.0)
    table = api.interpolate_plunging_velocities(m, ensemble)
    rng = np.random.default_rng(13)

    def item(inc, n, nd=1, height=None, metric=m):
        rr, th = rng.uniform(2.5, 25.0, n), rng.uniform(0, 2 * math.pi, n)
        al, be = rr * np.cos(th), rr * np.sin(th)
        x = [0.0, 1e4, math.radians(inc), 0.0]
        rays = api.ImpactParameters(al, be) if n else api.ImpactParameters(np.ones(1), np.ones(1))  # the dual trace reads only the problem
        cfg = api.tracing_configuration(metric, x, rays, gb.DatumPlane(0.0), 2e4,
                                        chart=gb.chart_for_metric(metric, 2e4), ensemble=ensemble)
        da, db = (np.cos(th)[None, :], np.sin(th)[None, :]) if nd == 1 else (np.stack([np.ones(n), np.zeros(n)]), np.stack([np.zeros(n), np.ones(n)]))
        return cfg, (al, be, da, db, height)

    heights = rng.uniform(0.0, 2.0, 60)
    items = [item(30.0, 70), item(60.0, 50, nd=2), item(45.0, 0), item(50.0, 60, height=heights), item(40.0, 40, metric=gb.KerrMetric(1.0, 0.9))]
    tabs = [table, table, table, table, None]

    def arrays(args, partial):
        arr = cabi.DualArrays(*args)
        if partial:  # outputs the caller does not ask for stay NULL
            for k in range(4):
                arr.out.x[k] = cabi.dptr(None)
            arr.out.drho, arr.out.nreject = cabi.dptr(None), cabi.iptr(None)
        return arr

    partial = [False, True, False, False, True]
    singles = [api.trace_dual(cfg, arrays(args, pt), plunging=t) if args[0].size else None
               for (cfg, args), t, pt in zip(items, tabs, partial)]
    batch = [arrays(args, pt) for (_, args), pt in zip(items, partial)]
    api.trace_dual_batch([cfg for cfg, _ in items], batch, plungings=tabs)
    st = ensemble.stats()
    assert st.launches == len(items) - 1 and st.rays == sum(args[0].size for _, args in items)
    for got, want, pt in zip(batch, singles, partial):
        if want is None:
            assert got.n == 0
            continue
        _same_arrays(got, want, DUAL_FIELDS)
        if pt:
            assert not got.x.any() and not got.drho.any() and not got.nreject.any()
    assert (batch[3].status == cabi.STATUS_INTERSECTED).sum() > 10


def test_pipelined_trace_with_partial_outputs_equals_one_launch(ensemble, monkeypatch):
    lib = cabi.load()
    ctx = ensemble.ctx(ensemble.devices[0])
    cfg = common.c1(1024, 1152, ensemble=ensemble)[3]
    p, ic = cfg.to_c()
    rng = cabi.Range(0, ic.n, 1)
    kinds = [dict(init=False, stats=False), dict(init=True, stats=False), dict(init=False, stats=True)]

    def run():
        outs, stats = [], []
        for kw in kinds:
            out = cabi.EndpointArrays(ic.n, **kw)
            cabi.check(lib.gb200_trace(ctx, C.byref(p), C.byref(ic), C.byref(rng), C.byref(out.c)), ctx)
            outs.append(out)
            st = ensemble.stats()
            stats.append((st.launches, st.rays, st.steps_accepted, st.steps_rejected, st.flagged))
        return outs, stats

    piped, st_p = run()
    monkeypatch.setenv("GB200_NO_PIPELINE", "1")
    single, st_1 = run()
    assert all(s[0] == 4 for s in st_p) and all(s[0] == 1 for s in st_1)
    assert [s[1:] for s in st_p] == [s[1:] for s in st_1]
    for got, want in zip(piped, single):
        _same_arrays(got, want, ENDPOINT_FIELDS)


def _dual_item(ensemble, n):
    m = gb.KerrMetric(1.0, 0.9)
    rng = np.random.default_rng(n)
    cfg = api.tracing_configuration(m, [0.0, 1e4, math.radians(40.0), 0.0], api.ImpactParameters(np.ones(1), np.ones(1)), gb.DatumPlane(0.0),
                                    2e4, chart=gb.chart_for_metric(m, 2e4), ensemble=ensemble)
    return cfg.to_c()[0], None, cabi.DualArrays(rng.uniform(-10, 10, n), rng.uniform(-10, 10, n), np.ones((1, n)), np.zeros((1, n)))


def _batch(lib, ctx, call, items):
    """`items`, [(problem, ic, rays)], as one gb200_<call>_batch; its return code.  rays: a count, or trace_dual's DualArrays."""
    nb = len(items)
    problems = (cabi.Problem * nb)(*[p for p, _, _ in items])
    if call == "trace_dual":
        return lib.gb200_trace_dual_batch(ctx, nb, problems, (cabi.DualIC * nb)(*[a.ic for _, _, a in items]), cabi.DUAL_NORM_WITH_PARTIALS,
                                          None, (cabi.DualOut * nb)(*[a.out for _, _, a in items]))
    ics = (cabi.IC * nb)(*[ic for _, ic, _ in items])
    ranges = (cabi.Range * nb)(*[cabi.Range(0, n, 1) for _, _, n in items])
    if call == "trace":
        outs = [cabi.EndpointArrays(n) for _, _, n in items]
        return lib.gb200_trace_batch(ctx, nb, problems, ics, ranges, (cabi.Endpoints * nb)(*[o.c for o in outs]))
    images = [np.zeros(n) for _, _, n in items]
    return lib.gb200_render_batch(ctx, nb, problems, ics, ranges, cabi.iptr(np.array([cabi.PF_STATUS], np.int32)), 1, None,
                                  (cabi._dp * nb)(*[cabi.dptr(img) for img in images]))


@pytest.mark.parametrize("call, check", [("trace", "table"), ("render", "table"), ("trace_dual", "table"), ("trace_dual", "dg")])
def test_batch_whose_later_item_fails_a_host_check_launches_nothing(ensemble, call, check):
    """GB200_GEOMETRY_THICK_TABLE without a cross-section table, or a dual item asking for dg but not g, fails the batch before
    its first item launches: the stats keep the launch count of the last successful call."""
    lib = cabi.load()
    ctx = ensemble.ctx(ensemble.devices[0])
    cabi.check(lib.gb200_set_cross_section(ctx, None, None, 0), ctx)
    if call == "trace_dual":
        good, empty, bad = _dual_item(ensemble, 50), _dual_item(ensemble, 0), _dual_item(ensemble, 40)
    else:
        p, ic = (_lamp_post(ensemble, 64) if call == "trace" else common.c1(16, 16, ensemble=ensemble)[3]).to_c()
        good, empty, bad = (p, ic, ic.n), (p, ic, 0), (cabi.Problem.from_buffer_copy(p), ic, ic.n)
    if check == "table":
        bad[0].geometry_kind = cabi.GEOMETRY_THICK_TABLE
    else:
        bad[2].out.g = cabi.dptr(None)
    cabi.check(_batch(lib, ctx, call, [empty]), ctx)
    assert ensemble.stats().launches == 0
    assert _batch(lib, ctx, call, [good, bad]) == cabi.ERR_INVALID_ARGUMENT
    assert (b"GB200_GEOMETRY_THICK_TABLE needs a table" if check == "table" else b"dg needs g") in lib.gb200_last_error(ctx)
    assert ensemble.stats().launches == 0


def test_render_batch_failing_after_a_launch_leaves_nothing_running(ensemble):
    """A metric without an ISCO is found on the host only when its item's turn comes, after the items before it launched:
    the batch returns the error once those have finished, so the next batch on the context has its arena to itself."""
    lib = cabi.load()
    ctx = ensemble.ctx(ensemble.devices[0])
    kerr = common.c1(1024, 1024, ensemble=ensemble)[3].to_c()
    jp = common.render_config(gb.JohannsenPsaltisMetric(1.0, 0.8831, 0.4), [0.0, 1000.0, math.radians(60.0), 0.0], gb.ThinDisc(0.0, 50.0),
                              2000.0, 16, 16, ensemble=ensemble).to_c()
    pfs = np.array([cabi.PF_REDSHIFT], np.int32)

    def render(items):
        nb = len(items)
        images = [np.zeros(ic.n) for _, ic in items]
        rc = lib.gb200_render_batch(ctx, nb, (cabi.Problem * nb)(*[p for p, _ in items]), (cabi.IC * nb)(*[ic for _, ic in items]),
                                    (cabi.Range * nb)(*[cabi.Range(0, ic.n, 1) for _, ic in items]), cabi.iptr(pfs), 1, None,
                                    (cabi._dp * nb)(*[cabi.dptr(img) for img in images]))
        return rc, images[0]

    rc, before = render([kerr])
    cabi.check(rc, ctx)
    assert render([kerr, jp])[0] == cabi.ERR_INVALID_ARGUMENT and b"no ISCO" in lib.gb200_last_error(ctx)
    rc, after = render([kerr])
    cabi.check(rc, ctx)
    assert np.isfinite(before).any() and np.array_equal(after, before, equal_nan=True)
