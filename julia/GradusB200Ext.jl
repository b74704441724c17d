# GradusB200Ext.jl -- reference-side binding for libgradus_b200 (the `ccall` shim a Gradus.jl maintainer adds).
#
# NOT EXECUTED IN THIS REPOSITORY'S CI: the build image has no Julia toolchain (DESIGN.md section 1).  Every entry point
# used below is exercised through the very same C ABI from Python (gradus.jl_b200/_cabi.py, tests/) and from plain C
# (tests/c/cabi_render.c).  Struct layouts mirror include/gradus_b200.h field for field
# (tests/test_host_api.py::test_ctypes_struct_layout_matches_header checks the sizes and offsets used here).
#
# What it adds, next to the stock ensembles (`EnsembleEndpointThreads`, src/Gradus.jl:412):
#   * `EnsembleB200(devices)`                                 -- a new ensemble type;
#   * a method of `Gradus.ensemble_solve_tracing_problem`     -- the seam of src/tracing/tracing.jl:113-196; it replaces
#     ext/GradusDiffEqGPUExt/GradusDiffEqGPUExt.jl:10-31.  With it `tracegeodesics`, `rendergeodesics`,
#     `prerendergeodesics`, `lineprofile(...; ensemble = EnsembleB200())` (the keyword reaches `tracegeodesics` through
#     `solver_args...`, src/line-profiles.jl:172-184), `tracecorona`, ... run their rays on the GPU with no other change;
#   * fused methods that skip the 152 B/ray `GeodesicPoint` round trip: `render_into_image!` for device point
#     functions (src/rendering/rendering.jl:89-107) and `lineprofile_b200` (src/line-profiles.jl:152-198).
# It overrides NO existing Gradus method: stock ensembles keep working with the extension loaded.  The initial
# conditions are recognised from the closures the reference builds (their captured variables are read as fields and the
# reading is verified against the closure itself on two rays); anything unrecognised takes the generic path, which
# evaluates `prob_func` on host threads exactly as the reference's ensembles do.
module GradusB200Ext

using Gradus
using Gradus: TracingConfiguration, GeodesicPoint, StatusCodes, KerrMetric, JohannsenPsaltisMetric, JohannsenMetric,
    BumblebeeMetric, KerrNewmanMetric, MorrisThorneWormhole, ThinDisc, ShakuraSunyaev, DatumPlane, PolarChart, PolarPlane, GeometricGrid,
    LinearGrid, InverseGrid, AbstractTrace, BinningMethod
using StaticArrays
import SciMLBase

const libgradus_b200 = get(ENV, "GRADUS_B200_LIB", "libgradus_b200")

# ---------------------------------------------------------------------------------------------------------------------
# ensemble type: one library context per device, created on first use and kept for the life of the ensemble
"""
    EnsembleB200(devices = [0])

Integrate every ray of an ensemble on the listed CUDA devices (B200, sm_100a) with libgradus_b200.  There is no CPU
fallback: configurations outside the library's scope raise `ArgumentError`.
"""
mutable struct EnsembleB200
    devices::Vector{Int}
    contexts::Vector{Ptr{Cvoid}}
    function EnsembleB200(devices::AbstractVector{<:Integer} = [0])
        isempty(devices) && throw(ArgumentError("EnsembleB200 needs at least one device"))
        e = new(collect(Int, devices), fill(C_NULL, length(devices)))
        finalizer(e) do x
            for c in x.contexts
                c == C_NULL || ccall((:gb200_destroy, libgradus_b200), Cvoid, (Ptr{Cvoid},), c)
            end
        end
        e
    end
end
Gradus.restrict_ensemble(::Gradus.AbstractMetric, e::EnsembleB200) = e

function _context(e::EnsembleB200, d::Int)
    if e.contexts[d] == C_NULL
        ctx = Ref{Ptr{Cvoid}}(C_NULL)
        _check(ccall((:gb200_init, libgradus_b200), Cint, (Cint, Ref{Ptr{Cvoid}}), e.devices[d], ctx), C_NULL)
        e.contexts[d] = ctx[]
    end
    e.contexts[d]
end

function _check(rc, ctx)
    rc == 0 && return
    msg = unsafe_string(ccall((:gb200_last_error, libgradus_b200), Cstring, (Ptr{Cvoid},), ctx))
    (rc == -1 || rc == -4) ? throw(ArgumentError(msg)) : error("libgradus_b200 ($rc): $msg")
end

# ---------------------------------------------------------------------------------------------------------------------
# POD mirrors of include/gradus_b200.h
struct CProblem
    metric_kind::Int32; geometry_kind::Int32; callback_kind::Int32; pow_mode::Int32
    metric_params::NTuple{8,Float64}; observer::NTuple{4,Float64}; geometry_params::NTuple{4,Float64}
    gtol::Float64; chart_inner::Float64; chart_outer::Float64; callback_delta::Float64
    lambda_min::Float64; lambda_max::Float64; abstol::Float64; reltol::Float64
    dtmax::Float64; mu::Float64; maxiters::Int64
end
struct CIC
    kind::Int32; grid_kind::Int32; width::Int64; height::Int64
    lo0::Float64; hi0::Float64; lo1::Float64; hi1::Float64
    x::NTuple{4,Ptr{Float64}}; v::NTuple{4,Ptr{Float64}}; n::Int64
end
struct CRange
    first::Int64; count::Int64; stride::Int64; block::Int64
end
struct CEndpoints
    status::Ptr{Int32}; lambda_max::Ptr{Float64}
    x::NTuple{4,Ptr{Float64}}; v::NTuple{4,Ptr{Float64}}; x_init::NTuple{4,Ptr{Float64}}; v_init::NTuple{4,Ptr{Float64}}
    naccept::Ptr{Int32}; nreject::Ptr{Int32}; flags::Ptr{Int32}
end
struct CEmissivity
    kind::Int32; n::Int32; index::Float64; r::Ptr{Float64}; eps::Ptr{Float64}
end
struct CLineProfileOpts
    min_re::Float64; max_re::Float64; normalise::Int32; bin_right_closed::Int32
end
struct CDiscProfile
    emissivity::CEmissivity; time_kind::Int32; n::Int32; r::Ptr{Float64}; t::Ptr{Float64}
end
struct CLagTransferOpts
    E0::Float64; t0::Float64; energy_lims::NTuple{2,Float64}; time_lims::NTuple{2,Float64}; N_E::Int32; N_t::Int32
end
struct CTfBranches
    n_radii::Int32; reserved::Int32; r_e::Ptr{Float64}; gmin::Ptr{Float64}; gmax::Ptr{Float64}; off::Ptr{Int64}
    gs::Ptr{Float64}; f::Ptr{Float64}; t::Ptr{Float64}
end
struct CTfModel
    table::Int32; n_radii::Int32; radii::Ptr{Float64}; rmin::Float64; g_scale::Float64; profile::CDiscProfile
end
struct CTfQuadOpts
    h::Float64; t0::Float64; upscale::Int32; npoints::Int32; nodes::Ptr{Float64}; weights::Ptr{Float64}; normalise::Int32
    reserved::Int32
end
const NULL4 = ntuple(_ -> Ptr{Float64}(C_NULL), 4)

# ---------------------------------------------------------------------------------------------------------------------
# configuration -> POD
_mp8(v...) = ntuple(i -> i <= length(v) ? Float64(v[i]) : 0.0, 8)
_metric(m::KerrMetric, qμ) = (Int32(0), _mp8(m.M, m.a))
_metric(m::JohannsenPsaltisMetric, qμ) = (Int32(1), _mp8(m.M, m.a, m.ϵ3))
_metric(m::JohannsenMetric, qμ) = (Int32(2), _mp8(m.M, m.a, m.α13, m.α22, m.α52, m.ϵ3))
_metric(m::BumblebeeMetric, qμ) = (Int32(3), _mp8(m.M, m.a, m.l))
_metric(m::MorrisThorneWormhole, qμ) = (Int32(5), _mp8(m.b))
_metric(m::Gradus.DilatonAxion, qμ) = begin   # the ratios as src/metrics/dilaton-axion-ad.jl:24-26 forms them
    z = iszero(m.β)
    (Int32(6), _mp8(m.M, m.a, m.β, m.b, z ? 0.0 : m.β / m.b, z ? 0.0 : m.β / m.a, z ? 0.0 : m.β / (m.a * m.b)))
end
# slot 4 (metric_params[3]) carries q for photons and q/μ otherwise (geodesic_ode_problem(::KerrNewmanMetric),
# src/metrics/kerr-newman-ad.jl:74-78)
_metric(m::KerrNewmanMetric, qμ) = (Int32(4), _mp8(m.M, m.a, m.Q, qμ))
_metric(m, qμ) = throw(ArgumentError("EnsembleB200 has no closed-form right-hand side for $(typeof(m)); there is no CPU fallback"))

_geometry(::Nothing) = (Int32(0), (0.0, 0.0, 0.0, 0.0))
_geometry(d::ThinDisc) = (Int32(1), (Float64(d.inner_radius), Float64(d.outer_radius), 0.0, 0.0))
_geometry(d::ShakuraSunyaev) = (Int32(2), (Float64(d.Ṁ_Ṁedd), Float64(d.inv_η), Float64(d.inner_radius), 0.0))
_geometry(d::DatumPlane) = (Int32(3), (Float64(d.height), 0.0, 0.0, 0.0))

"""
    ImageOrder(d::ThinDisc, n)

The order-n image of a thin disc (n = 0 the direct image, 1 and 2 the first photon-ring subrings): a ray hits it at its
first entry into the disc's wedge in a step that starts with n equatorial crossings (`equatorial_crossings()`); earlier
entries pass through and once the count exceeds n the disc is inert (GB200_GEOMETRY_THIN_DISC_ORDER, include/gradus_b200.h).
Not a type of the reference: it lives in this extension and goes wherever `EnsembleB200` takes a geometry
(`tracegeodesics`, `rendergeodesics`, `lineprofile_b200`); the transfer-function and target paths refuse it.
"""
struct ImageOrder{D}
    disc::D
    n::Int
    function ImageOrder(d::D, n::Integer) where {D<:ThinDisc}
        n >= 0 || throw(ArgumentError("ImageOrder needs a non-negative order"))
        new{D}(d, Int(n))
    end
end
_geometry(d::ImageOrder) = (Int32(6), (Float64(d.disc.inner_radius), Float64(d.disc.outer_radius), Float64(d.n), 0.0))
# thick discs whose height is a closure (`ThickDisc(f)`, `PolishDoughnut`: src/geometry/discs/thick-disc.jl:32-63,
# polish-doughnut.jl:102-129) cross the ABI as a table (GB200_GEOMETRY_THICK_TABLE); `_install_geometry` uploads it
_geometry(d::Gradus.AbstractThickAccretionDisc) = begin
    ρ, h = _cross_section_table(d)
    (Int32(4), (maximum(h), first(ρ), last(ρ), 0.0))
end
_geometry(d) = throw(ArgumentError("geometry $(typeof(d)) is outside the EnsembleB200 scope"))

const _THICK_TABLES = IdDict{Any,Tuple{Vector{Float64},Vector{Float64}}}()
function _cross_section_table(d::Gradus.AbstractThickAccretionDisc; n = 4097)
    get!(_THICK_TABLES, d) do
        if d isa Gradus.PolishDoughnut        # `d.f` is a linear interpolation already: its own nodes
            return (collect(Float64, d.f.t), collect(Float64, d.f.u))
        end
        lo, hi = Float64(d.inner_radius), Float64(d.outer_radius)
        (isfinite(lo) && isfinite(hi) && hi > lo) ||
            throw(ArgumentError("EnsembleB200 tabulates cross_section(d, ρ) over [inner_radius, outer_radius]: give the disc finite radii"))
        # Chebyshev nodes crowd towards the ends as 1/n^2, which resolves the square-root edges of tori
        ρ = [0.5 * (lo + hi) - 0.5 * (hi - lo) * cospi((k - 1) / (n - 1)) for k = 1:n]
        ρ[1], ρ[end] = lo, hi
        (ρ, Float64[Gradus.cross_section(d, r) for r in ρ])
    end
end
_install_geometry(ctx, d) = nothing
function _install_geometry(ctx, d::Gradus.AbstractThickAccretionDisc)
    d isa ShakuraSunyaev && return nothing
    ρ, h = _cross_section_table(d)
    _check(ccall((:gb200_set_cross_section, libgradus_b200), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int32), ctx, ρ, h, length(ρ)), ctx)
end

# Julia names a closure type "#name#NN": recognise the reference's closures by the stem of that name.
_closure_is(f, stem::AbstractString) = startswith(string(nameof(typeof(f))), "#" * stem)

_flatten_callbacks(::Nothing) = ()
_flatten_callbacks(cb::SciMLBase.CallbackSet) = (cb.continuous_callbacks..., cb.discrete_callbacks...)
_flatten_callbacks(cb) = (cb,)

"""
`config.callback` is what `tracing_configuration` stored: `merge_callbacks(user_callback, geometry_callback)`
(src/geometry/bootstrap.jl:12-19, src/tracing/callbacks.jl:13-23), i.e. a `CallbackSet` holding the geometry's
`ContinuousCallback` (condition closure `_distance_to_disc_wrapper`, capturing `g` and `gtol`, bootstrap.jl:56-60) and the
user's callbacks.  Returns (callback_kind, δ, gtol); the geometry itself is taken from `config.geometry`.
"""
function _callbacks(config)
    kind, δ, gtol, seen_geometry = Int32(0), 0.0, 1e-2, false
    for cb in _flatten_callbacks(config.callback)
        isnothing(cb) && continue
        cond = cb.condition
        if cb isa SciMLBase.ContinuousCallback && _closure_is(cond, "_distance_to_disc_wrapper")
            cond.g === config.geometry || throw(ArgumentError("the geometry callback does not belong to config.geometry"))
            gtol = Float64(cond.gtol)
            seen_geometry = true
        elseif cb isa SciMLBase.DiscreteCallback && _closure_is(cond, "_domain_upper_hemisphere_check")
            kind == 0 || throw(ArgumentError("only one `domain_upper_hemisphere` callback can run on the device"))
            kind, δ = Int32(1), Float64(cond.δ)          # src/tracing/callbacks.jl:31-39
        else
            throw(ArgumentError("callback $(typeof(cond)) cannot run on the device: only the disc intersection and `domain_upper_hemisphere` do"))
        end
    end
    isnothing(config.geometry) || seen_geometry || throw(ArgumentError("config.geometry has no intersection callback in config.callback"))
    kind, δ, gtol
end

# mass of the traced particle: not stored in `config` (it lives in `trace`); recover it from the norm of the first,
# already constrained, initial state (constrain_all, src/tracing/constraints.jl:14-15)
function _mass(m, u0)
    x, v = SVector{4}(u0[1:4]), SVector{4}(u0[5:8])
    μ2 = -Gradus.dotproduct(Gradus.metric(m, x), v, v)
    μ2 < 1e-10 ? 0.0 : sqrt(μ2)
end
# q/μ of a charged particle: captured by the Kerr-Newman ODE function (kerr-newman-ad.jl:73-92)
_charge(prob) = hasproperty(prob.f.f, :q_μ) ? Float64(prob.f.f.q_μ) : 0.0

function _problem(config::TracingConfiguration, prob::SciMLBase.ODEProblem; mu = _mass(config.metric, prob.u0), solver_opts...)
    config.solver isa Gradus.Tsit5 || throw(ArgumentError("EnsembleB200 integrates with Tsit5 only"))
    config.chart isa PolarChart || throw(ArgumentError("EnsembleB200 supports PolarChart only"))
    # the device integrator has two further options; everything else errors like `kwargshandle = KeywordArgError`
    # (src/tracing/tracing.jl:106,146)
    dtmax, maxiters = 0.0, 0
    for (k, v) in pairs(solver_opts)
        k === :dtmax ? (dtmax = Float64(v)) : k === :maxiters ? (maxiters = Int(v)) :
        throw(ArgumentError("unrecognised keyword argument $k for the B200 integrator"))
    end
    mk, mp = _metric(config.metric, _charge(prob))
    gk, gp = _geometry(config.geometry)
    ck, cδ, gtol = _callbacks(config)
    CProblem(mk, gk, ck, 0, mp, Tuple(Float64.(prob.u0[1:4])), gp, gtol, config.chart.inner_radius, config.chart.outer_radius, cδ,
             config.λ_domain[1], config.λ_domain[2], config.abstol, config.reltol, dtmax, mu, maxiters)
end

# ---------------------------------------------------------------------------------------------------------------------
# initial conditions
"""
Structured initial conditions read off the reference's velocity closures, or `nothing`.
  * `_render_velocity_function` (src/rendering/rendering.jl:140-163) returns `velfunc` capturing the ranges `αs`, `βs` and
    `image_height`: -> GB200_IC_RENDER_GRID (rays generated on the device from six scalars).
  * `promote_velfunc(m, x, plane)` (src/image-planes/planes.jl:180-184) returns `velfunc` capturing the materialised `αs`, `βs`
    arrays of any image plane: -> GB200_IC_IMPACT_PARAMETERS (two host arrays, 16 B/ray); `lineprofile_b200` below passes a
    `PolarPlane` as data instead (GB200_IC_POLAR_PLANE, nothing uploaded).
The reading is checked against the closure itself on the first and last ray.
"""
function _structured_ic(config, keep)
    v = config.velocity
    (v isa Function && _closure_is(v, "velfunc") && hasproperty(v, :αs) && hasproperty(v, :βs)) || return nothing
    m, x, n = config.metric, config.position, config.trajectories
    if v.αs isa AbstractRange && v.βs isa AbstractRange && hasproperty(v, :image_height)
        w, h = length(v.αs), Int(v.image_height)
        (length(v.βs) == h && w * h == n) || return nothing
        for i in (1, n)
            col, row = (i - 1) ÷ h + 1, mod1(i, h)
            Gradus.map_impact_parameters(m, x, v.αs[col] + 1e-6, v.βs[row] + 1e-6) == v(i) || return nothing
        end
        return CIC(0, 0, w, h, first(v.αs), last(v.αs), first(v.βs), last(v.βs), NULL4, NULL4, n)
    elseif v.αs isa AbstractArray{Float64} && length(v.αs) == n == length(v.βs)
        for i in (1, n)
            Gradus.map_impact_parameters(m, x, v.αs[i], v.βs[i]) == v(i) || return nothing
        end
        αs, βs = vec(collect(v.αs)), vec(collect(v.βs))
        push!(keep, αs, βs)
        return CIC(4, 0, 0, 0, 0.0, 0.0, 0.0, 0.0, (pointer(αs), pointer(βs), Ptr{Float64}(C_NULL), Ptr{Float64}(C_NULL)), NULL4, n)
    end
    nothing
end

# generic path: evaluate prob_func on host threads into SoA, as the reference's ensembles do per ray
# (corona fans, src/corona/models/lamp-post.jl:89-100; arrays of positions and velocities)
function _explicit_ic(problem, n, keep)
    xs = [Vector{Float64}(undef, n) for _ = 1:4]
    vs = [Vector{Float64}(undef, n) for _ = 1:4]
    Threads.@threads for i = 1:n
        u0 = problem.prob_func(problem.prob, i, 0).u0
        for k = 1:4
            xs[k][i] = u0[k]
            vs[k][i] = u0[4+k]
        end
    end
    append!(keep, xs)
    append!(keep, vs)
    CIC(2, 0, 0, 0, 0.0, 0.0, 0.0, 0.0, Tuple(pointer.(xs)), Tuple(pointer.(vs)), n)
end

_grid_kind(::LinearGrid) = Int32(0)
_grid_kind(::GeometricGrid) = Int32(1)
_grid_kind(::InverseGrid) = Int32(2)
_grid_kind(g) = throw(ArgumentError("grid $(typeof(g)) is outside the EnsembleB200 scope"))
_plane_ic(p::PolarPlane) = CIC(1, _grid_kind(p.grid), p.Nr, p.Nθ, p.r_min, p.r_max, p.θ_min, p.θ_max, NULL4, NULL4, p.Nr * p.Nθ)

# ---------------------------------------------------------------------------------------------------------------------
# sharding: whole strips of four image columns (render grid) / θ-rows (polar plane), strip d, d + ndev, ... on device d:
# balances the expensive photon-ring region and keeps neighbouring rays in one warp (15 % of kernel time at 8 devices,
# DESIGN.md section 6).  Output slot s of a range holds ray first + (s ÷ block) * stride * block + s % block (0-based).
function _ranges(ic::CIC, ndev)
    h = ic.kind == 0 ? ic.height : ic.kind == 1 ? ic.width : 0
    strip = 4h
    if ndev == 1
        return [CRange(0, ic.n, 1, 1)]
    elseif strip > 0 && ic.n % strip == 0
        nstrips = ic.n ÷ strip
        return [CRange(d * strip, (d < nstrips ? (nstrips - d + ndev - 1) ÷ ndev : 0) * strip, ndev, strip) for d = 0:ndev-1]
    end
    [CRange(d, ic.n > d ? (ic.n - d + ndev - 1) ÷ ndev : 0, ndev, 1) for d = 0:ndev-1]
end
_ray_of_slot(r::CRange, s) = r.first + (s ÷ r.block) * r.stride * r.block + s % r.block   # 0-based

# run f(device_index, context, range) for every device on its own task (the library call blocks; contexts are
# independent, one thread at a time per context)
function _foreach_device(f, e::EnsembleB200, ranges)
    tasks = map(1:length(e.devices)) do d
        Threads.@spawn ranges[d].count > 0 && f(d, _context(e, d), ranges[d])
    end
    foreach(fetch, tasks)
end

# ---------------------------------------------------------------------------------------------------------------------
# the seam: ensemble_solve_tracing_problem(::EnsembleB200, ...) -> Vector{GeodesicPoint}
function Gradus.ensemble_solve_tracing_problem(
    ensemble::EnsembleB200,
    problem::SciMLBase.EnsembleProblem,
    config::TracingConfiguration{T};
    progress_bar = nothing,
    save_on = false,
    solver_opts...,
) where {T}
    save_on && error("Cannot use `EnsembleB200` with `save_on`")                      # tracing.jl:159-161
    isnothing(progress_bar) || @warn "Progress bar not supported with EnsembleB200" maxlog = 1
    keep = Any[]
    n = config.trajectories
    ic = _structured_ic(config, keep)
    # explicit states arrive constrained for the trace's own μ: mu = NaN tells the library to keep v^t as given
    p = isnothing(ic) ? _problem(config, problem.prob; mu = NaN, solver_opts...) : _problem(config, problem.prob; solver_opts...)
    isnothing(ic) && (ic = _explicit_ic(problem, n, keep))
    ranges = _ranges(ic, length(ensemble.devices))
    outs = map(ranges) do r
        (status = Vector{Int32}(undef, r.count), λ = Vector{Float64}(undef, r.count),
         x = [Vector{Float64}(undef, r.count) for _ = 1:4], v = [Vector{Float64}(undef, r.count) for _ = 1:4],
         x0 = [Vector{Float64}(undef, r.count) for _ = 1:4], v0 = [Vector{Float64}(undef, r.count) for _ = 1:4])
    end
    GC.@preserve keep outs begin
        _foreach_device(ensemble, ranges) do d, ctx, r
            _install_geometry(ctx, config.geometry)
            o = outs[d]
            ep = CEndpoints(pointer(o.status), pointer(o.λ), Tuple(pointer.(o.x)), Tuple(pointer.(o.v)), Tuple(pointer.(o.x0)),
                            Tuple(pointer.(o.v0)), C_NULL, C_NULL, C_NULL)
            _check(ccall((:gb200_trace, libgradus_b200), Cint, (Ptr{Cvoid}, Ref{CProblem}, Ref{CIC}, Ref{CRange}, Ref{CEndpoints}),
                         ctx, p, ic, r, ep), ctx)
        end
    end
    # return contract of tracing.jl:179-189: a concretely typed Vector{GeodesicPoint{T,Nothing}} in ray order
    points = Vector{GeodesicPoint{T,Nothing}}(undef, n)
    λ0 = T(config.λ_domain[1])
    for (r, o) in zip(ranges, outs)
        Threads.@threads for s = 0:r.count-1
            j = s + 1
            points[_ray_of_slot(r, s)+1] = GeodesicPoint(
                StatusCodes.T(o.status[j]), λ0, T(o.λ[j]),
                SVector{4,T}(o.x0[1][j], o.x0[2][j], o.x0[3][j], o.x0[4][j]), SVector{4,T}(o.x[1][j], o.x[2][j], o.x[3][j], o.x[4][j]),
                SVector{4,T}(o.v0[1][j], o.v0[2][j], o.v0[3][j], o.v0[4][j]), SVector{4,T}(o.v[1][j], o.v[2][j], o.v[3][j], o.v[4][j]),
                nothing)
        end
    end
    points
end

# ---------------------------------------------------------------------------------------------------------------------
# fused paths
"""
    B200PointFunction(:redshift | :radius | :shadow | :coordinate_time | :status | :affine_time | :end_radius | :equatorial_crossings)

A point function the device evaluates at the ray end point inside the trace kernel (include/gradus_b200.h, GB200_PF_*):
`:redshift` = `ConstPointFunctions.redshift(m, x) ∘ ConstPointFunctions.filter_intersected()`, `:radius` =
`PointFunction((m, gp, λ) -> gp.x[2] * sin(gp.x[3])) ∘ filter_intersected()`, `:shadow` = the default `pf` of
`render_into_image!` (affine time of rays that ended early), ...  Pass it as `pf = ...` to `rendergeodesics`.
"""
struct B200PointFunction
    kind::Int32
end
const _PF_KINDS = Dict(:shadow => 0, :redshift => 1, :radius => 2, :coordinate_time => 3, :status => 4, :affine_time => 5, :end_radius => 6,
                       :equatorial_crossings => 7)
B200PointFunction(s::Symbol) = B200PointFunction(Int32(_PF_KINDS[s]))

"""
    equatorial_crossings()

The number of accepted integrator steps whose start and end differ in the sign of cos θ, unfiltered
(GB200_PF_EQUATORIAL_CROSSINGS); a disc hit reports the count at the start of its event step, i.e. its image order.
`ThinDisc`, `ImageOrder` or no geometry.  Not a point function of the reference.
"""
equatorial_crossings() = B200PointFunction(:equatorial_crossings)

const _B200Config{T} = TracingConfiguration{T,M,P,V,G,C,Ch,S,<:EnsembleB200} where {M,P,V,G,C,Ch,S}

"""
`render_into_image!` (src/rendering/rendering.jl:89-102) for an `EnsembleB200` configuration and a device point function:
one fused launch per device writes the (H, W) column-major image; no `GeodesicPoint` is materialised.  Any other `pf`
takes the stock method (trace on the GPU through `ensemble_solve_tracing_problem`, point function on the host).
"""
function Gradus.render_into_image!(image, trace::AbstractTrace, config::_B200Config{T}; pf = B200PointFunction(:shadow), solver_opts...) where {T}
    if !(pf isa B200PointFunction)
        return invoke(Gradus.render_into_image!, Tuple{Any,AbstractTrace,TracingConfiguration{T}}, image, trace, config; pf = pf, solver_opts...)
    end
    problem = Gradus.assemble_tracing_problem(trace, config)
    keep = Any[]
    ic = _structured_ic(config, keep)
    isnothing(ic) && throw(ArgumentError("render_into_image! needs the render-grid velocity function"))
    p = _problem(config, problem.prob; mu = Float64(trace.μ), solver_opts...)
    ensemble = config.ensemble
    ranges = _ranges(ic, length(ensemble.devices))
    pfs = Int32[pf.kind]
    if length(ranges) == 1          # the whole image in ray order: write straight into `image`
        _install_geometry(_context(ensemble, 1), config.geometry)
        GC.@preserve keep image pfs begin
            imgs = [pointer(image)]
            _check(ccall((:gb200_render, libgradus_b200), Cint,
                         (Ptr{Cvoid}, Ref{CProblem}, Ref{CIC}, Ref{CRange}, Ptr{Int32}, Int32, Ptr{Cvoid}, Ptr{Ptr{Float64}}),
                         _context(ensemble, 1), p, ic, ranges[1], pfs, 1, C_NULL, imgs), _context(ensemble, 1))
        end
    else
        parts = [Vector{T}(undef, r.count) for r in ranges]
        GC.@preserve keep parts pfs begin
            _foreach_device(ensemble, ranges) do d, ctx, r
                _install_geometry(ctx, config.geometry)
                imgs = [pointer(parts[d])]
                _check(ccall((:gb200_render, libgradus_b200), Cint,
                             (Ptr{Cvoid}, Ref{CProblem}, Ref{CIC}, Ref{CRange}, Ptr{Int32}, Int32, Ptr{Cvoid}, Ptr{Ptr{Float64}}),
                             ctx, p, ic, r, pfs, 1, C_NULL, imgs), ctx)
            end
        end
        for (r, part) in zip(ranges, parts), b = 0:(r.count ÷ r.block)-1     # whole strips are contiguous in the image
            dst = r.first + b * r.stride * r.block
            copyto!(image, dst + 1, part, b * r.block + 1, r.block)
        end
    end
    image
end

"""
    lineprofile_b200(bins, ε, m, u, d; ensemble = EnsembleB200(), λ_max, minrₑ, maxrₑ, plane, callback, power_law_index, solver_args...)

`lineprofile(bins, ε, m, u, d, BinningMethod(); ...)` (src/line-profiles.jl:152-198) fused on the device: trace, redshift,
`ε(rₑ) g³ area`, and the `Buckets.Simple` histogram in shared memory; with several devices the raw histograms are summed
with one NCCL all-reduce inside the library (`gb200_comm_lineprofile`).  `ε` crosses the ABI as a power-law index when
`power_law_index` is given (`ε(r) = r^-index`), otherwise as a 4096-point table of `ε` on a geometric grid over
[minrₑ, maxrₑ] (linear interpolation: 1e-6 relative for power laws).  Returns `(bins, flux ./ sum(flux))`.
"""
function lineprofile_b200(bins, ε, m::Gradus.AbstractMetric{T}, u, d;
                          ensemble::EnsembleB200 = EnsembleB200(), λ_max = 2 * u[2], minrₑ = Gradus.isco(m), maxrₑ = T(50),
                          plane::PolarPlane = PolarPlane(GeometricGrid(); Nr = 450, Nθ = 1300, r_max = 5maxrₑ),
                          callback = Gradus.domain_upper_hemisphere(), power_law_index = nothing, solver_args...) where {T}
    trace = Gradus.TraceGeodesic()
    config, solver_opts = Gradus.tracing_configuration(trace, m, u, plane, d, (0.0, λ_max); callback = callback, ensemble = ensemble, solver_args...)
    problem = Gradus.assemble_tracing_problem(trace, config)
    p = _problem(config, problem.prob; mu = 0.0, solver_opts...)
    ic = _plane_ic(plane)
    binsv = collect(Float64, bins)
    rs = isnothing(power_law_index) ? collect(exp.(range(log(minrₑ), log(maxrₑ), 4096))) : Float64[]
    es = isnothing(power_law_index) ? Float64.(ε.(rs)) : Float64[]
    flux = zeros(Float64, length(binsv))
    GC.@preserve binsv rs es flux begin
        emis = isnothing(power_law_index) ? CEmissivity(1, length(rs), 0.0, pointer(rs), pointer(es)) :
               CEmissivity(0, 0, Float64(power_law_index), C_NULL, C_NULL)
        opts = CLineProfileOpts(minrₑ, maxrₑ, 1, 0)
        if length(ensemble.devices) == 1
            ctx = _context(ensemble, 1)
            _install_geometry(ctx, d)
            _check(ccall((:gb200_lineprofile, libgradus_b200), Cint,
                         (Ptr{Cvoid}, Ref{CProblem}, Ref{CIC}, Ref{CRange}, Ref{CEmissivity}, Ptr{Cvoid}, Ptr{Float64}, Int32, Ref{CLineProfileOpts}, Ptr{Float64}),
                         ctx, p, ic, CRange(0, ic.n, 1, 1), emis, C_NULL, binsv, length(binsv), opts, flux), ctx)
        else
            comm = Ref{Ptr{Cvoid}}(C_NULL)
            devs = Int32.(ensemble.devices)
            _check(ccall((:gb200_comm_init, libgradus_b200), Cint, (Ptr{Int32}, Int32, Ref{Ptr{Cvoid}}), devs, length(devs), comm), C_NULL)
            try
                for i = 0:length(devs)-1   # a thick disc's table goes to every context of the communicator
                    _install_geometry(ccall((:gb200_comm_context, libgradus_b200), Ptr{Cvoid}, (Ptr{Cvoid}, Int32), comm[], i), d)
                end
                _check(ccall((:gb200_comm_lineprofile, libgradus_b200), Cint,
                             (Ptr{Cvoid}, Ref{CProblem}, Ref{CIC}, Ref{CEmissivity}, Ptr{Cvoid}, Ptr{Float64}, Int32, Ref{CLineProfileOpts}, Ptr{Float64}),
                             comm[], p, ic, emis, C_NULL, binsv, length(binsv), opts, flux), C_NULL)
            finally
                ccall((:gb200_comm_destroy, libgradus_b200), Cvoid, (Ptr{Cvoid},), comm[])
            end
        end
    end
    bins, flux
end

"""
    lagtransfer_b200(m, u, d, r, t; linear_time = false, power_law_index = 3.0, ε = nothing, ensemble = EnsembleB200(),
                     plane, max_t, E₀ = 6.4, t0 = u[2], N_E = 300, N_t = 300, energy_lims = nothing, time_lims = nothing,
                     callback, solver_args...)

`binflux(lagtransfer(m, u, d, model; plane, max_t, ...), profile; E₀, t0, N_E, N_t, energy_lims, time_lims)`
(src/transfer-functions/transfer-functions-2d.jl:100-122,163-242) with the observer→disc leg traced and binned on the
device (`gb200_lagtransfer`; `gb200_comm_lagtransfer` over several devices, bit-identical).  The profile crosses the ABI
as data: `r`, `t` are its arrival-time knots (for `AnalyticRadialDiscProfile` the coronal geodesics' ρ sorted ascending and
their coordinate times, interpolated as its NaN-linear interpolator; `linear_time = true` for `RadialDiscProfile`), `ε`
a power law (`power_law_index`) or, when `ε = (radii, values)`, a clamped linear table.  Returns
`(time_edges .- t0, energy_edges, tf, hits)`.  Not run: there is no Julia toolchain where this binding was written; the
Python mirror `binned_lagtransfer` is the tested form.
"""
function lagtransfer_b200(m::Gradus.AbstractMetric{T}, u, d, r, t; linear_time = false, power_law_index = 3.0, ε = nothing,
                          ensemble::EnsembleB200 = EnsembleB200(), max_t = 2 * u[2],
                          plane::PolarPlane = PolarPlane(GeometricGrid(); Nr = 800, Nθ = 800, r_max = 50.0),
                          E₀ = 6.4, t0 = u[2], N_E = 300, N_t = 300, energy_lims = nothing, time_lims = nothing,
                          callback = Gradus.domain_upper_hemisphere(), solver_args...) where {T}
    trace = Gradus.TraceGeodesic()
    chart = Gradus.chart_for_metric(m, 1.1 * u[2])
    config, solver_opts = Gradus.tracing_configuration(trace, m, u, plane, d, (0.0, max_t); chart = chart, callback = callback,
                                                       ensemble = ensemble, solver_args...)
    problem = Gradus.assemble_tracing_problem(trace, config)
    p = _problem(config, problem.prob; mu = 0.0, solver_opts...)
    ic = _plane_ic(plane)
    rv, tv = collect(Float64, r), collect(Float64, t)
    er = isnothing(ε) ? Float64[] : collect(Float64, ε[1])
    ev = isnothing(ε) ? Float64[] : collect(Float64, ε[2])
    tb, eb, tf = zeros(Float64, N_t), zeros(Float64, N_E), zeros(Float64, N_t, N_E) # column-major: tf[j, i] = cell (i, j)
    hits = Ref{Int64}(0)
    lims(l) = isnothing(l) ? (NaN, NaN) : (Float64(l[1]), Float64(l[2]))
    opts = CLagTransferOpts(E₀, t0, lims(energy_lims), lims(time_lims), N_E, N_t)
    GC.@preserve rv tv er ev tb eb tf begin
        emis = isnothing(ε) ? CEmissivity(0, 0, Float64(power_law_index), C_NULL, C_NULL) :
               CEmissivity(1, length(er), 0.0, pointer(er), pointer(ev))
        prof = CDiscProfile(emis, linear_time ? 1 : 0, length(rv), pointer(rv), pointer(tv))
        if length(ensemble.devices) == 1
            ctx = _context(ensemble, 1)
            _install_geometry(ctx, d)
            _check(ccall((:gb200_lagtransfer, libgradus_b200), Cint,
                         (Ptr{Cvoid}, Ref{CProblem}, Ref{CIC}, Ref{CDiscProfile}, Ptr{Cvoid}, Ref{CLagTransferOpts}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ref{Int64}),
                         ctx, p, ic, prof, C_NULL, opts, tb, eb, tf, hits), ctx)
        else
            comm = Ref{Ptr{Cvoid}}(C_NULL)
            devs = Int32.(ensemble.devices)
            _check(ccall((:gb200_comm_init, libgradus_b200), Cint, (Ptr{Int32}, Int32, Ref{Ptr{Cvoid}}), devs, length(devs), comm), C_NULL)
            try
                for i = 0:length(devs)-1
                    _install_geometry(ccall((:gb200_comm_context, libgradus_b200), Ptr{Cvoid}, (Ptr{Cvoid}, Int32), comm[], i), d)
                end
                _check(ccall((:gb200_comm_lagtransfer, libgradus_b200), Cint,
                             (Ptr{Cvoid}, Ref{CProblem}, Ref{CIC}, Ref{CDiscProfile}, Ptr{Cvoid}, Ref{CLagTransferOpts}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ref{Int64}),
                             comm[], p, ic, prof, C_NULL, opts, tb, eb, tf, hits), C_NULL)
            finally
                ccall((:gb200_comm_destroy, libgradus_b200), Cvoid, (Ptr{Cvoid},), comm[])
            end
        end
    end
    tb, eb, permutedims(tf), hits[]
end

# ---------------------------------------------------------------------------------------------------------------------
# quadrature of Cunningham transfer functions, many emission models per call

# An InterpolatingTransferBranches as the flat arrays of gb200_tf_branches: branch 2k is the lower, 2k+1 the upper branch
# of radius k; every branch a NaNLinearInterpolator (fields t, u) with default 0, f and t on the same knots.
function _pack_branches(itb)
    rs, gmin, gmax, off, gs, f, t = Float64[], Float64[], Float64[], Int64[0], Float64[], Float64[], Float64[]
    for br in sort(collect(itb.branches); by = b -> b.rₑ)
        push!(rs, br.rₑ); push!(gmin, br.gmin); push!(gmax, br.gmax)
        for (fb, tb) in ((br.lower_f, br.lower_t), (br.upper_f, br.upper_t))
            all(x -> x isa Gradus.NaNLinearInterpolator && iszero(x.default), (fb, tb)) ||
                throw(ArgumentError("only NaNLinearInterpolator branches with default 0 can be integrated on the device"))
            fb.t == tb.t || throw(ArgumentError("the f and t branches at rₑ = $(br.rₑ) do not share their knots"))
            append!(gs, fb.t); append!(f, fb.u); append!(t, tb.u); push!(off, length(gs))
        end
    end
    (rs, gmin, gmax, off, gs, f, t)
end

_per_model(v, n) = v isa AbstractVector ? (length(v) == n ? v : throw(ArgumentError("$(length(v)) values for $n models"))) : fill(v, n)

# ε: a power-law index (a Number) or a clamped linear table (radii, values); profile time: (r, t) knots, NaN-linear
# (AnalyticRadialDiscProfile) or linear (`linear_time`, RadialDiscProfile)
function _c_disc_profile(ε, r, t, linear_time, keep)
    emis = if ε isa Number
        CEmissivity(0, 0, Float64(ε), C_NULL, C_NULL)
    else
        er, ev = collect(Float64, ε[1]), collect(Float64, ε[2])
        push!(keep, er, ev)
        CEmissivity(1, length(er), 0.0, pointer(er), pointer(ev))
    end
    rv, tv = collect(Float64, r), collect(Float64, t)
    push!(keep, rv, tv)
    CDiscProfile(emis, linear_time ? 1 : 0, length(rv), isempty(rv) ? C_NULL : pointer(rv), isempty(tv) ? C_NULL : pointer(tv))
end

function _tf_quadrature(lag, itbs, g_grid, t_grid, profiles, n; table_of, rmin, rmax, g_scale, h, n_radii, g_grid_upscale,
                        quadrature_points, t0, ensemble)
    itbs = itbs isa AbstractVector ? itbs : [itbs]
    packed = [_pack_branches(itb) for itb in itbs]
    table_of = isnothing(table_of) ? _per_model(collect(1:length(itbs)), n) : _per_model(table_of, n)
    rmin, rmax, g_scale, n_radii = _per_model(rmin, n), _per_model(rmax, n), _per_model(g_scale, n), _per_model(n_radii, n)
    X, W = Gradus.FastGaussQuadrature.gausslegendre(quadrature_points)
    g, tg = collect(Float64, g_grid), collect(Float64, t_grid)
    keep = Any[]
    out = lag ? zeros(Float64, length(tg), length(g), n) : zeros(Float64, length(g), n) # column-major of the C layout
    GC.@preserve packed keep X W g tg begin
        tables = [CTfBranches(length(p[1]), 0, pointer(p[1]), pointer(p[2]), pointer(p[3]), pointer(p[4]), pointer(p[5]),
                              pointer(p[6]), pointer(p[7])) for p in packed]
        models = map(1:n) do k
            itb = itbs[table_of[k]]
            lo = isnothing(rmin[k]) ? minimum(b.rₑ for b in itb.branches) : Float64(rmin[k])
            hi = isnothing(rmax[k]) ? maximum(b.rₑ for b in itb.branches) : Float64(rmax[k])
            radii = collect(Float64, lag ? Gradus._geometric_grid(lo, hi, n_radii[k]) : Gradus._inverse_grid(lo, hi, n_radii[k]))
            push!(keep, radii)
            CTfModel(table_of[k] - 1, n_radii[k], pointer(radii), lo, g_scale[k], profiles(k, keep))
        end
        opts = CTfQuadOpts(h, t0, g_grid_upscale, quadrature_points, pointer(X), pointer(W), 1, 0)
        ctx = _context(ensemble, 1)
        if lag
            _check(ccall((:gb200_tf_lagtransfer, libgradus_b200), Cint,
                         (Ptr{Cvoid}, Int32, Ptr{CTfBranches}, Int32, Ptr{CTfModel}, Ptr{Float64}, Int32, Ptr{Float64}, Int32,
                          Ref{CTfQuadOpts}, Ptr{Float64}),
                         ctx, length(tables), tables, n, models, g, length(g), tg, length(tg), opts, out), ctx)
        else
            _check(ccall((:gb200_tf_lineprofile, libgradus_b200), Cint,
                         (Ptr{Cvoid}, Int32, Ptr{CTfBranches}, Int32, Ptr{CTfModel}, Ptr{Float64}, Int32, Ref{CTfQuadOpts}, Ptr{Float64}),
                         ctx, length(tables), tables, n, models, g, length(g), opts, out), ctx)
        end
    end
    lag ? permutedims(out, (2, 1, 3)) : out
end

"""
    integrate_lineprofile_b200(itbs, g_grid; ε = 3.0, table_of = nothing, rmin = nothing, rmax = nothing, g_scale = 1.0,
                               h = 1e-8, n_radii = 1000, g_grid_upscale = 1, quadrature_points = 7, ensemble = EnsembleB200())

`integrate_lineprofile(ε, itb, g_grid; rmin, rmax, h, n_radii, g_grid_upscale, ...)`
(src/transfer-functions/integration.jl:233-254, 322-357) for many emission models in one device call
(`gb200_tf_lineprofile`).  `itbs`: one `InterpolatingTransferBranches` or a vector of them; `ε` (a power-law index or a
`(radii, values)` table), `table_of` (1-based; default model k uses table k), `rmin`, `rmax`, `g_scale` and `n_radii` are
per model, a vector with one entry per model or one value for all.  Returns a `length(g_grid)` × nmodels matrix of
normalised profiles.  Not run: there is no Julia toolchain where this binding was written; the Python mirror
`integrate_lineprofiles` is the tested form.
"""
function integrate_lineprofile_b200(itbs, g_grid; ε = 3.0, table_of = nothing, rmin = nothing, rmax = nothing, g_scale = 1.0,
                                    h = 1e-8, n_radii = 1000, g_grid_upscale = 1, quadrature_points = 7,
                                    ensemble::EnsembleB200 = EnsembleB200())
    n = maximum(v -> v isa AbstractVector ? length(v) : 1, (table_of, rmin, rmax, g_scale, n_radii,
                                                            ε isa AbstractVector ? ε : nothing))
    isnothing(table_of) && itbs isa AbstractVector && (n = max(n, length(itbs)))
    εs = _per_model(ε isa AbstractVector ? ε : [ε for _ = 1:n], n)
    _tf_quadrature(false, itbs, g_grid, Float64[], (k, keep) -> _c_disc_profile(εs[k], Float64[], Float64[], false, keep), n;
                   table_of, rmin, rmax, g_scale, h, n_radii, g_grid_upscale, quadrature_points, t0 = 0.0, ensemble)
end

"""
    integrate_lagtransfer_b200(itbs, g_grid, t_grid, profiles; t0 = 0.0, table_of = nothing, rmin = nothing, rmax = nothing,
                               g_scale = 1.0, h = 1e-8, n_radii = 1000, g_grid_upscale = 1, quadrature_points = 7,
                               ensemble = EnsembleB200())

`integrate_lagtransfer(profile, itb, g_grid, t_grid; t0, n_radii, rmin, rmax, ...)`
(src/transfer-functions/integration.jl:256-279, 359-442) for many emission models in one device call
(`gb200_tf_lagtransfer`).  `profiles`: a vector of named tuples `(r, t, linear_time = false, ε = 3.0)`, the profile's
arrival-time knots as in `lagtransfer_b200`; the other per-model keywords as in `integrate_lineprofile_b200`.  Returns a
`length(g_grid)` × `length(t_grid)` × nmodels array.  Not run: there is no Julia toolchain where this binding was written;
the Python mirror `integrate_lagtransfers` is the tested form.
"""
function integrate_lagtransfer_b200(itbs, g_grid, t_grid, profiles::AbstractVector; t0 = 0.0, table_of = nothing, rmin = nothing,
                                    rmax = nothing, g_scale = 1.0, h = 1e-8, n_radii = 1000, g_grid_upscale = 1,
                                    quadrature_points = 7, ensemble::EnsembleB200 = EnsembleB200())
    n = length(profiles)
    prof(k, keep) = (p = profiles[k]; _c_disc_profile(get(p, :ε, 3.0), p.r, p.t, get(p, :linear_time, false), keep))
    _tf_quadrature(true, itbs, g_grid, t_grid, prof, n; table_of, rmin, rmax, g_scale, h, n_radii, g_grid_upscale,
                   quadrature_points, t0, ensemble)
end

"""
    optimize_for_target_b200(target, m, x0; ensemble, d_tol = 1e-2, max_time = 2x0[2], p0 = (0.0, 0.0), window, grid = 33, kwargs...)

`Gradus.optimize_for_target` (src/tracing/precision-solvers.jl:512-531) with the device under it: instead of one trace per
Nelder-Mead evaluation, every round traces a `grid` x `grid` patch of impact parameters in one `gb200_trace_target` call
(the reference's distance callback, closest approach per ray), re-centres on the best ray and shrinks the patch to two of
its cells, until the best ray passes within `d_tol` of `target` = (r, θ, ϕ).  Returns `(α, β, gp, accuracy)` like the
reference (`gp` is a named tuple of the end point: status, λ, x, v).
"""
function optimize_for_target_b200(target, m::Gradus.AbstractMetric{T}, x0; ensemble::EnsembleB200 = EnsembleB200(), d_tol = 1e-2,
                                  max_time = 2 * x0[2], p0 = (0.0, 0.0), window = 1.5 * target[1] + 10, grid = 33, max_rounds = 10,
                                  callback = nothing, solver_args...) where {T}
    trace = Gradus.TraceGeodesic()
    ctx = _context(ensemble, 1)
    tgt = collect(Float64, target)
    half, ca, cb = Float64(window), Float64(p0[1]), Float64(p0[2])
    best = (Inf, ca, cb, nothing)
    n = grid * grid
    αs, βs, closest = Vector{Float64}(undef, n), Vector{Float64}(undef, n), Vector{Float64}(undef, n)
    status, λs = Vector{Int32}(undef, n), Vector{Float64}(undef, n)
    xs, vs = [Vector{Float64}(undef, n) for _ = 1:4], [Vector{Float64}(undef, n) for _ = 1:4]
    for _ = 1:max_rounds
        for i = 1:grid, j = 1:grid
            αs[(i-1)*grid+j] = ca - half + 2half * (i - 1) / (grid - 1)
            βs[(i-1)*grid+j] = cb - half + 2half * (j - 1) / (grid - 1)
        end
        velfunc = i -> Gradus.map_impact_parameters(m, x0, αs[i], βs[i])
        config, solver_opts = Gradus.tracing_configuration(trace, m, x0, velfunc, (0.0, max_time); callback = callback,
                                                           ensemble = ensemble, trajectories = n, solver_args...)
        problem = Gradus.assemble_tracing_problem(trace, config)
        p = _problem(config, problem.prob; mu = 0.0, solver_opts...)
        GC.@preserve αs βs closest status λs xs vs tgt begin
            ic = CIC(4, 0, 0, 0, 0.0, 0.0, 0.0, 0.0, (pointer(αs), pointer(βs), Ptr{Float64}(C_NULL), Ptr{Float64}(C_NULL)), NULL4, n)
            out = CEndpoints(pointer(status), pointer(λs), Tuple(pointer.(xs)), Tuple(pointer.(vs)), NULL4, NULL4, C_NULL, C_NULL, C_NULL)
            _check(ccall((:gb200_trace_target, libgradus_b200), Cint,
                         (Ptr{Cvoid}, Ref{CProblem}, Ref{CIC}, Ref{CRange}, Ptr{Float64}, Float64, Ref{CEndpoints}, Ptr{Float64}),
                         ctx, p, ic, CRange(0, n, 1, 1), tgt, Float64(d_tol), out, closest), ctx)
        end
        i = argmin(closest)
        if closest[i] < best[1]
            gp = (status = Gradus.StatusCodes.T(status[i]), λ_max = λs[i], x = SVector{4}(ntuple(k -> xs[k][i], 4)), v = SVector{4}(ntuple(k -> vs[k][i], 4)))
            best = (closest[i], αs[i], βs[i], gp)
        end
        best[1] < d_tol && break
        ca, cb = best[2], best[3]
        half = 2 * (2half / (grid - 1))
    end
    best[2], best[3], best[4], best[1]
end

export EnsembleB200, B200PointFunction, ImageOrder, equatorial_crossings, lineprofile_b200, lagtransfer_b200, optimize_for_target_b200,
       integrate_lineprofile_b200, integrate_lagtransfer_b200
end # module
