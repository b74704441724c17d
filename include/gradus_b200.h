/*
 * gradus_b200.h -- C ABI of libgradus_b200.so: the B200-native (sm_100a, FP64)
 * implementation of Gradus.jl's per-ray geodesic integration hot path.
 *
 * This is the drop-in boundary for the reference's ensemble seam
 *     Gradus.ensemble_solve_tracing_problem(ensemble, problem, config; ...)
 *         reference: src/tracing/tracing.jl:113-196
 *         (GPU specialisation it replaces: ext/GradusDiffEqGPUExt/GradusDiffEqGPUExt.jl:10-31)
 * A Julia extension adds `struct EnsembleB200` plus one method of that function
 * which fills the POD structs below from `TracingConfiguration` fields
 * (src/tracing/configuration.jl:16-29) and `ccall`s into this library; see
 * INTEGRATION.md for the binding.  Plain C only: pointers, sizes, PODs.
 *
 * Ownership: the caller owns every host buffer passed in; the library owns all
 * device memory, streams and events inside `gb200_ctx`.  All calls are blocking.
 * A context may be used from one thread at a time.  Every entry point returns
 * GB200_OK (0) or a negative error code; the message is available through
 * gb200_last_error().  Nothing here ever falls back to a CPU implementation:
 * without a usable CUDA device gb200_init fails with GB200_ERR_NO_DEVICE.
 */
#ifndef GRADUS_B200_H
#define GRADUS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GB200_VERSION 100 /* 0.1.0 */

/* ---- error codes ------------------------------------------------------- */
#define GB200_OK 0
#define GB200_ERR_INVALID_ARGUMENT (-1) /* mirrors Julia ArgumentError / KeywordArgError */
#define GB200_ERR_NO_DEVICE (-2)        /* no CUDA device: there is no CPU fallback */
#define GB200_ERR_CUDA (-3)
#define GB200_ERR_UNSUPPORTED (-4) /* configuration outside the hot-path scope */
#define GB200_ERR_NOMEM (-5)

/* ---- StatusCodes.T, declaration order of src/Gradus.jl:59-64 ----------- */
#define GB200_STATUS_OUT_OF_DOMAIN 0
#define GB200_STATUS_WITHIN_INNER_BOUNDARY 1
#define GB200_STATUS_INTERSECTED_WITH_GEOMETRY 2
#define GB200_STATUS_NO_STATUS 3

/* ---- metrics: src/metrics/kerr-metric.jl:62-68, johannsen-psaltis-ad.jl:38-46 */
#define GB200_METRIC_KERR 0              /* params: M, a          */
#define GB200_METRIC_JOHANNSEN_PSALTIS 1 /* params: M, a, eps3    */
#define GB200_METRIC_JOHANNSEN 2         /* src/metrics/johannsen-ad.jl:40-62     params: M, a, alpha13, alpha22, alpha52, eps3 */
#define GB200_METRIC_BUMBLEBEE 3         /* src/metrics/bumblebee-ad.jl:26-46     params: M, a, l  (l > -1, |a| <= 0.3)        */
#define GB200_METRIC_KERR_NEWMAN 4       /* src/metrics/kerr-newman-ad.jl:41-58   params: M, a, Q, q/mu (charge of the test particle:
                                            Lorentz force q/mu F v of geodesic_ode_problem(::KerrNewmanMetric), :66-102; 0 = neutral) */
#define GB200_METRIC_MORRIS_THORNE 5     /* src/metrics/morris-thorne-ad.jl:4-15  params: b (throat size, metric_params[0]); r is the proper
                                            radial coordinate l, inner_radius = 0 (:40), no ISCO */
#define GB200_METRIC_DILATON_AXION 6     /* src/metrics/dilaton-axion-ad.jl:8-46  params: M, a, beta, b, beta/b, beta/a, beta/(a b) -- the three
                                            ratios as the reference forms them (0 where beta == 0, :24-26) */
#define GB200_METRIC_COUNT 7

/* ---- accretion geometry: src/geometry/discs/ --------------------------- */
#define GB200_GEOMETRY_NONE 0
#define GB200_GEOMETRY_THIN_DISC 1       /* thin-disc.jl:9-26       params: inner_radius, outer_radius */
#define GB200_GEOMETRY_SHAKURA_SUNYAEV 2 /* shakura-sunyaev.jl:22-33 params: Mdot/Mdot_edd, inv_eta, inner_radius(isco) */
#define GB200_GEOMETRY_DATUM_PLANE 3     /* datum-plane.jl:1-10     params: height */
#define GB200_GEOMETRY_THICK_TABLE 4     /* thick-disc.jl:32-63: `ThickDisc(f)` with its closure f(rho) tabulated -- a closure cannot
                                            cross the ABI.  cross_section(rho) = linear interpolation in the table installed with
                                            gb200_set_cross_section, -1 (no disc) outside its range; distance_to_disc = |r cos theta| - h,
                                            1 where h <= 0.  params: max of the table (filled in by the library) */

#define GB200_GEOMETRY_TARGET_POINT 5    /* gb200_trace_target only: the distance ContinuousCallback of _make_target_objective,
                                            src/tracing/precision-solvers.jl:473-488 */
#define GB200_GEOMETRY_THIN_DISC_ORDER 6 /* ImageOrder(ThinDisc(r_in, r_out), n): the order-n image of the thin disc.
                                            params: inner_radius, outer_radius, n (a non-negative integer stored as a double,
                                            at most 2^31 - 1; anything else is GB200_ERR_INVALID_ARGUMENT).  The wedge, its
                                            condition and gtol are GB200_GEOMETRY_THIN_DISC's; only the events differ:
                                              - an entry into the wedge (condition positive -> non-positive) in a step that starts
                                                with n equatorial crossings (GB200_PF_EQUATORIAL_CROSSINGS) is an event, handled
                                                exactly as a ThinDisc event (root find, discrete callbacks on the event state,
                                                IntersectedWithGeometry);
                                              - an entry in a step that starts with fewer crossings is passed through (an
                                                ordinary accepted step); exits from the wedge are never events;
                                              - once the count exceeds n the disc is inert: the ray ends at its chart, lambda_max
                                                or callback and is not a hit (its n-th crossing fell outside [r_in, r_out]).
                                            A ray that hits GB200_GEOMETRY_THIN_DISC with count c takes the same steps and the same
                                            event step under order c.  Accepted by gb200_trace*, gb200_render*, gb200_lineprofile*
                                            and gb200_comm_*; gb200_trace_dual*, gb200_trace_target and gb200_trace_path return
                                            GB200_ERR_UNSUPPORTED */

/* ---- user discrete callback: src/tracing/callbacks.jl:31-39 ------------ */
#define GB200_CALLBACK_NONE 0
#define GB200_CALLBACK_UPPER_HEMISPHERE 1 /* r cos(theta) < delta -> OutOfDomain */

/* ---- step-controller pow(): DiffEqBase.fastpow is version dependent ---- */
#define GB200_POW_EXACT 0 /* x^y through double-precision log and exp.  In the throughput kernel the error estimate carries a relative
                            2^-20 from its scale reciprocals and the pair is evaluated to 1e-7 (DESIGN.md, K1); the forward-mode
                            kernel and the oracle evaluate it with libm */
#define GB200_POW_FAST32 1 /* Float32 exp2(y*log2(x)) a la FastPower.jl */

/* ---- integrator failure flags (SciML retcodes are invisible in GeodesicPoint) */
#define GB200_FLAG_MAXITERS 1
#define GB200_FLAG_DT_MIN 2
#define GB200_FLAG_UNSTABLE 4

/*
 * Everything `TracingConfiguration` (src/tracing/configuration.jl:3-88) carries
 * for the in-scope path, flattened.  Integrator: Tsit5 with OrdinaryDiffEq's
 * default PI controller; only the fields below are configurable, anything else
 * the reference would accept as `solver_opts` is rejected by the host shim.
 */
typedef struct gb200_problem {
    int32_t metric_kind;
    int32_t geometry_kind;
    int32_t callback_kind;
    int32_t pow_mode;
    double metric_params[8];
    double observer[4]; /* x = (t, r, theta, phi) shared by all rays unless the IC is explicit */
    double geometry_params[4];
    double gtol;           /* src/geometry/bootstrap.jl:8, default 1e-2 */
    double chart_inner;    /* PolarChart.inner_radius, src/tracing/charts.jl:3-6 */
    double chart_outer;    /* PolarChart.outer_radius */
    double callback_delta; /* domain_upper_hemisphere(delta) */
    double lambda_min;
    double lambda_max;
    double abstol;
    double reltol;
    double dtmax; /* <= 0 -> lambda_max - lambda_min (OrdinaryDiffEq default) */
    double mu;    /* geodesic mass, 0 for photons (constrain_time, auto-diff.jl:161-173); NaN with explicit initial conditions:
                     v^t is kept as given (states taken from an ensemble's prob_func are already constrained) */
    int64_t maxiters; /* <= 0 -> 1000000 */
} gb200_problem;

/* ---- initial conditions ------------------------------------------------ */
#define GB200_IC_RENDER_GRID 0 /* _render_velocity_function, src/rendering/rendering.jl:140-163 */
#define GB200_IC_POLAR_PLANE 1 /* PolarPlane + promote_velfunc, src/image-planes/planes.jl:70-115,180-184 */
#define GB200_IC_EXPLICIT 2    /* prob_func evaluated on the host into SoA (corona ensembles) */
#define GB200_IC_CARTESIAN_PLANE 3 /* CartesianPlane, src/image-planes/planes.jl:130-178 */
#define GB200_IC_IMPACT_PARAMETERS 4 /* map_impact_parameters(m, x, alphas, betas), src/tracing/utility.jl:70-87:
                                        x[0] = alpha[n], x[1] = beta[n] (host arrays); observer = problem.observer;
                                        x[2] = optional height[n]: with GB200_GEOMETRY_DATUM_PLANE each ray meets its own
                                        plane z = height[i] (datumplane(d, r_e) of many emission radii in one launch,
                                        src/geometry/discs/datum-plane.jl:14-19), NULL = geometry_params[0] */

#define GB200_GRID_LINEAR 0    /* src/image-planes/grids.jl:32-36 */
#define GB200_GRID_GEOMETRIC 1 /* grids.jl:11-20 */
#define GB200_GRID_INVERSE 2   /* grids.jl:22-30 */

typedef struct gb200_ic {
    int32_t kind;
    int32_t grid_kind; /* polar plane only */
    /* render grid: ray i (0-based) -> col = i / height, row = i % height;
       alpha = range(alpha_lo, alpha_hi, width)[col] + 1e-6, beta likewise */
    int64_t width;  /* render: image_width ; polar: Nr     ; cartesian: Nx */
    int64_t height; /* render: image_height; polar: Ntheta ; cartesian: Ny */
    double lo0, hi0; /* render: alpha limits; polar: r_min, r_max         ; cartesian: x_min, x_max */
    double lo1, hi1; /* render: beta  limits; polar: theta_min, theta_max ; cartesian: y_min, y_max */
    /* cartesian plane: the grid (grid_kind) is evaluated on Nx/2 and Ny/2 points and mirrored about the first point;
       n = (2(Ny/2) - 1)(2(Nx/2) - 1); ray i -> beta index i % (2(Ny/2) - 1), alpha index i / (2(Ny/2) - 1) */
    /* explicit: host SoA, each pointer addresses n doubles; v[0] (v^t) is
       ignored and re-constrained exactly like wrap_constraint does */
    const double* x[4];
    const double* v[4];
    int64_t n; /* total number of rays described by this IC */
} gb200_ic;

/* Sub-range of rays handled by one call.  Output slot n (0 <= n < count) holds ray
       first + (n / block) * stride * block + n % block,
   i.e. blocks of `block` consecutive rays, every `stride`-th block (block = 1: rays first, first+stride, ...).
   Rays shard trivially across GPUs / ranks; interleaving whole blocks of image columns (block = 4 * image_height)
   keeps neighbouring rays together, which the kernel's warps like (DESIGN.md, "work order"). */
typedef struct gb200_range {
    int64_t first;
    int64_t count;
    int64_t stride; /* >= 1 */
    int64_t block;  /* >= 1; 0 is read as 1 */
} gb200_range;

/* Caller-allocated host SoA, `count` entries each; any pointer may be NULL.
   Field meaning: GeodesicPoint, src/solution-processing.jl:15-32. */
typedef struct gb200_endpoints {
    int32_t* status;
    double* lambda_max;
    double* x[4];
    double* v[4];
    double* x_init[4];
    double* v_init[4];
    int32_t* naccept; /* per-ray integrator statistics */
    int32_t* nreject;
    int32_t* flags;
} gb200_endpoints;

/* ---- point functions: src/const-point-functions.jl --------------------- */
#define GB200_PF_SHADOW 0          /* affine_time o filter_early_term (default pf of render_into_image!, rendering.jl:93-95) */
#define GB200_PF_REDSHIFT 1        /* redshift o filter_intersected (src/redshift.jl:192-220) */
#define GB200_PF_DISC_RADIUS 2     /* r sin(theta) o filter_intersected */
#define GB200_PF_COORDINATE_TIME 3 /* x[1] o filter_intersected */
#define GB200_PF_STATUS 4          /* status as double, no filter */
#define GB200_PF_AFFINE_TIME 5     /* lambda_max, no filter */
#define GB200_PF_RADIUS 6          /* r |sin(theta)| of the end point whatever its status (ConstPointFunctions.radius,
                                      src/const-point-functions.jl; the offset root finder reads it, precision-solvers.jl:124) */
#define GB200_PF_EQUATORIAL_CROSSINGS 7 /* equatorial crossings of the ray, as a double, no filter: the number of accepted steps
                                      whose start and end states differ in the sign of cos(theta) (cos(theta) >= 0 counts as
                                      positive), from 0 at the initial state, up to and including the step that ends the ray at
                                      its chart, lambda_max or a discrete callback.  A step that ends in a disc event does not
                                      count: a hit reports the count at the start of its event step.  Geometry NONE, THIN_DISC
                                      and THIN_DISC_ORDER only; any other geometry is GB200_ERR_UNSUPPORTED (in gb200_render,
                                      gb200_render_batch, gb200_render_device and gb200_comm_render) */

/* ---- emissivity for the binned line profile ---------------------------- */
#define GB200_EMISSIVITY_POWERLAW 0 /* eps(r) = r^(-index) */
#define GB200_EMISSIVITY_TABLE 1    /* linear interpolation in (r, eps), clamped */

typedef struct gb200_emissivity {
    int32_t kind;
    int32_t n;       /* table length */
    double index;    /* power-law index */
    const double* r; /* host, ascending */
    const double* eps;
} gb200_emissivity;

/* Optional plunging-region velocity table for non-Kerr redshift
   (interpolate_redshift, src/redshift.jl:246-276): columns r (ascending), u^t, u^r, u^phi. */
typedef struct gb200_plunging_table {
    int32_t n;
    const double* r;
    const double* ut;
    const double* ur;
    const double* uphi;
} gb200_plunging_table;

typedef struct gb200_lineprofile_opts {
    double min_re;  /* minr_e, default isco(m)  (src/line-profiles.jl:163) */
    double max_re;  /* maxr_e, default 50 */
    int32_t normalise; /* 1: flux ./ sum(flux) (line-profiles.jl:197); 0: raw partial sums (multi-rank) */
    int32_t bin_right_closed; /* 0 (Buckets.Simple): slot i takes bins[i] <= g < bins[i+1], i.e. searchsortedlast, clamped to the
                                 ends -- the convention that reproduces test/unit/emissivity.jl:31-42 to 1e-11;
                                 1: bins[i-1] < g <= bins[i] (searchsortedfirst), kept for callers that label bins by their upper edge */
} gb200_lineprofile_opts;

/* Timing / counters of the last call on a context. */
typedef struct gb200_stats {
    double kernel_ms;      /* CUDA-event time of the trace kernel(s) */
    double total_ms;       /* including H2D/D2H */
    int64_t rays;
    int64_t steps_accepted;
    int64_t steps_rejected;
    int64_t launches;      /* kernels launched by the call */
    int64_t flagged;       /* rays with a non-zero failure flag */
} gb200_stats;

typedef struct gb200_ctx gb200_ctx;

int gb200_version(void);

/* Create a context on CUDA device `device` (ordinal).  One context per GPU;
   multi-GPU callers create one per device (or one per rank). */
int gb200_init(int device, gb200_ctx** out);
void gb200_destroy(gb200_ctx* ctx);
const char* gb200_last_error(gb200_ctx* ctx); /* ctx may be NULL: last global error */
int gb200_get_stats(gb200_ctx* ctx, gb200_stats* out);

/* Cross-section table of GB200_GEOMETRY_THICK_TABLE for this context: n >= 2 points, rho ascending; copied to the device and
   kept until replaced (n = 0 removes it).  A Julia caller tabulates `cross_section(d, rho)` of its ThickDisc once, e.g. on
   Chebyshev nodes of the support so that square-root edges are resolved (tests/test_more_metrics.py uses 4097 nodes for the
   torus of test/smoke-tests/rendergeodesics.jl:8-15). */
int gb200_set_cross_section(gb200_ctx* ctx, const double* rho, const double* height, int32_t n);

/* Validate a configuration without running it (what the Julia shim calls first
   so that unsupported set-ups raise ArgumentError before any work). */
int gb200_validate(const gb200_problem* p, const gb200_ic* ic);

/* Special radii needed to build configurations on the host.
   isco: Kerr analytic (kerr-metric-first-order.jl:336-337); otherwise the root of
   dE/dr (src/special-radii.jl:14-60).  Pure host arithmetic. */
int gb200_isco(int32_t metric_kind, const double* metric_params, double* out);
/* 1 - E_isco, i.e. the default eta of ShakuraSunyaev (shakura-sunyaev.jl:41-50). */
int gb200_radiative_efficiency(int32_t metric_kind, const double* metric_params, double* out);

/* One geodesic with EVERY accepted step recorded (the `save_on = true` single-ray form of tracegeodesics,
   src/tracing/tracing.jl:66-108): u0 = (x[4], v[4]) with v^t re-constrained for mass p->mu; no geometry is used.
   Writes at most `cap` rows: lambda[k], u[8*k .. 8*k+7] (row 0 is the initial state); *nrows receives the number of
   rows the solve produced (may exceed cap), *status the final StatusCodes value.  One GPU thread; a set-up tool. */
int gb200_trace_path(gb200_ctx* ctx, const gb200_problem* p, const double* u0, int32_t cap,
                     double* lambda, double* u, int32_t* nrows, int32_t* status);

/* The objective of optimize_for_target / impact_parameters_for_target (src/tracing/precision-solvers.jl:452-546) for a whole
   set of rays at once: every ray of `ic` / `rg` is traced with the reference's distance callback -- a ContinuousCallback on
   |to_cartesian(u) - to_cartesian(target)| - d_tol with 8 interpolation points that terminates the ray
   (IntersectedWithGeometry) where it first comes within d_tol -- and closest[i] receives the ray's closest approach
   (closest_approach[], :466-481).  The reference records the smallest of the condition's own evaluations (eight samples per
   step), which misses a d_tol sphere lying between two samples; here the distance is also minimised along the dense output
   of each step (golden section around the smallest sample), and coming within d_tol there is an event as well.
   target = (r, theta, phi); p->geometry_kind must be
   GB200_GEOMETRY_NONE (the callback takes the geometry's place), p->callback_kind and the chart apply as usual.  The
   reference minimises this objective one ray at a time (Nelder-Mead); with a device under it the search is a grid of impact
   parameters per call, refined around its minimum (the Python mirror's `optimize_for_target`).  `out` may be NULL. */
int gb200_trace_target(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic, const gb200_range* rg,
                       const double* target, double d_tol, gb200_endpoints* out, double* closest);

/* Plunging-region four-velocity table for the redshift of non-Kerr metrics inside the ISCO
   (interpolate_plunging_velocities, src/orbits/orbit-solving.jl:99-167): a massive geodesic released at
   r_isco - 1e-8 with CircularOrbits.plunging_fourvelocity, traced to 1.000001 r_h on the device, sorted by radius
   with the innermost sample dropped.  Caller provides 4 arrays of `cap` doubles; *n receives the table length. */
int gb200_build_plunging_table(gb200_ctx* ctx, int32_t metric_kind, const double* metric_params, int32_t cap,
                         double* r, double* ut, double* ur, double* uphi, int32_t* n);

/* ensemble_solve_tracing_problem(::EnsembleB200, ...) -> endpoints (tracing.jl:151-196). */
int gb200_trace(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic,
                const gb200_range* range, gb200_endpoints* out);

/* Many short ensembles at once (SURVEY 8f-1: corona / lamp-post emissivity fans over an (a, h) grid,
   src/corona/models/lamp-post.jl:89-100 called once per model).  Equivalent to `nbatch` gb200_trace calls, but every
   ensemble is launched on its own stream of a pool and the host synchronises once, so 1000-ray ensembles overlap
   instead of each paying a launch + copy round trip. */
int gb200_trace_batch(gb200_ctx* ctx, int32_t nbatch, const gb200_problem* problems, const gb200_ic* ics,
                      const gb200_range* ranges, gb200_endpoints* outs);

/* Many fused renders at once: `nbatch` independent (problem, initial conditions, range) triples, the same `npf` point
   functions for all, images[b * npf + k] -> ranges[b].count doubles.  This is the transfer-function table of
   BASELINE config 4 (make_transfer_function_table, src/transfer-functions/cunningham-transfer-functions.jl:507-530: one
   Cunningham transfer-function computation per (a, theta) cell, each a sequence of small probes): every probe round of
   every cell goes out in one call, one launch per cell on a stream pool, one staged H2D and one D2H copy.
   pls: optional array of nbatch plunging-table pointers (NULL, or NULL entries, where none is needed).
   Explicit-SoA initial conditions are not accepted here (gb200_trace_batch batches those). */
int gb200_render_batch(gb200_ctx* ctx, int32_t nbatch, const gb200_problem* problems, const gb200_ic* ics,
                       const gb200_range* ranges, const int32_t* pointfns, int32_t npf,
                       const gb200_plunging_table* const* pls, double* const* images);

/* rendergeodesics fused path (rendering.jl:28-54,89-107): trace + point
   function(s); writes `npf` images of `range->count` doubles each, image k at
   images[k], ray order (for the full range this is the (H,W) column-major image). */
int gb200_render(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic,
                 const gb200_range* range, const int32_t* pointfns, int32_t npf,
                 const gb200_plunging_table* plunging, double* const* images);

/* lineprofile(::BinningMethod) fused path (src/line-profiles.jl:152-198):
   trace + redshift + eps(r) g^3 area + bucket.  flux_out has nbins doubles. */
int gb200_lineprofile(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic,
                      const gb200_range* range, const gb200_emissivity* emis,
                      const gb200_plunging_table* plunging,
                      const double* bins, int32_t nbins,
                      const gb200_lineprofile_opts* opts, double* flux_out);

/* ---- forward-mode (dual-number) traces: the transfer-function solvers ---- */
/* The reference differentiates through the integrator with ForwardDiff: `_make_image_plane_mapper`
   (src/tracing/precision-solvers.jl:73-131) seeds the image-plane offset with one partial for the Newton iteration of
   `_find_offset_for_radius` (:133-241), `jacobian_∂αβ_∂gr` (:401-451) seeds (alpha, beta) with two for
   |d(rho, g) / d(alpha, beta)|.  Ray i starts at problem.observer with impact parameters alpha[i], beta[i]
   (map_impact_parameters, src/tracing/utility.jl:70-87) whose partials are dalpha[k*n + i], dbeta[k*n + i],
   k < npartials; the whole integrator state carries the partials, the step-size control reads them through the error
   norm exactly as DiffEqBase does for dual-valued states (norm_mode), and an event time found on the dense output moves
   with the parameters so that the end point stays on the surface. */
typedef struct gb200_dual_ic {
    int64_t n;
    int32_t npartials;    /* 1 or 2 */
    int32_t reserved;
    const double* alpha;  /* n */
    const double* beta;   /* n */
    const double* dalpha; /* npartials x n */
    const double* dbeta;  /* npartials x n */
    const double* height; /* optional, n: per-ray datum-plane height (GB200_GEOMETRY_DATUM_PLANE), NULL = geometry_params[0] */
} gb200_dual_ic;

/* Caller-allocated host arrays, n entries each (dg, drho: npartials x n); any pointer may be NULL.
   g = redshift (NaN unless the ray intersected the geometry), rho = r sin(theta) of the end point whatever its
   status (`_equatorial_project`, the quantity the offset root finder reads for rays that missed, precision-solvers.jl:124). */
typedef struct gb200_dual_out {
    int32_t* status;
    double* lambda_max;
    double* x[4];
    double* v[4];
    double* g;
    double* dg;
    double* rho;
    double* drho;
    int32_t* naccept;
    int32_t* nreject;
    int32_t* flags;
} gb200_dual_out;

#define GB200_DUAL_NORM_WITH_PARTIALS 0 /* DiffEqBase's ODE_DEFAULT_NORM on duals: partials are error-controlled too */
#define GB200_DUAL_NORM_VALUES_ONLY 1   /* step sequence of the plain trace */

int gb200_trace_dual(gb200_ctx* ctx, const gb200_problem* p, const gb200_dual_ic* ic, int32_t norm_mode,
                     const gb200_plunging_table* plunging, gb200_dual_out* out);

/* `nbatch` independent (problem, rays) pairs in one call (every probe round of a transfer-function table over (a, theta)
   cells, make_transfer_function_table, cunningham-transfer-functions.jl:507-530): one launch per pair on the stream pool,
   one staged copy each way.  pls: optional array of nbatch plunging-table pointers. */
int gb200_trace_dual_batch(gb200_ctx* ctx, int32_t nbatch, const gb200_problem* problems, const gb200_dual_ic* ics,
                           int32_t norm_mode, const gb200_plunging_table* const* pls, gb200_dual_out* outs);

/* Two-dimensional weighted histogram: `bucket(x, y, w, xbins, ybins; reduction = sum)` of bin_transfer_function
   (src/transfer-functions/transfer-functions-2d.jl:100-122), Buckets.Simple in both axes (cell (i, j) takes
   xbins[i] <= x < xbins[i+1], ybins[j] <= y < ybins[j+1], clamped to the ends).  n host samples -> out[i * ny + j] on the
   host.  Weights are accumulated as 64-bit fixed point (2^-62 of sum |w| per sample), so the result does not depend on
   the order of accumulation. */
int gb200_bucket2d(gb200_ctx* ctx, int64_t n, const double* x, const double* y, const double* w,
                   const double* xbins, int32_t nx, const double* ybins, int32_t ny, double* out);

/* ---- binned lag-energy transfer function ------------------------------- */
/* binflux(lagtransfer(m, x, d, model; plane, ...), profile; E0, t0, N_E, N_t, energy_lims, time_lims)
   (src/transfer-functions/transfer-functions-2d.jl:100-122,163-242) from the same traces, binned on the device. */
#define GB200_PROFILE_TIME_NAN_LINEAR 0 /* NaNLinearInterpolator (AnalyticRadialDiscProfile, corona/analytic.jl:1-40) */
#define GB200_PROFILE_TIME_LINEAR 1     /* linear interpolation (RadialDiscProfile, corona/radial.jl:1-37) */

typedef struct gb200_disc_profile { /* eps(rho) and the source-to-disc arrival time t(rho) */
    gb200_emissivity emissivity;    /* POWERLAW or TABLE (r strictly ascending), as for gb200_lineprofile */
    int32_t time_kind;              /* GB200_PROFILE_TIME_*; both clip rho to [r[0], r[n-1]] first */
    int32_t n;                      /* >= 2 */
    const double* r;                /* host, strictly ascending */
    const double* t;
} gb200_disc_profile;

typedef struct gb200_lagtransfer_opts {
    double E0;             /* line energy: E = g E0; positive and finite */
    double t0;             /* subtracted from the returned time edges */
    double energy_lims[2]; /* (lo, hi) with lo < hi, or both NaN: min and max of E over the hits */
    double time_lims[2];   /* likewise for T */
    int32_t N_E, N_t;      /* >= 2 each, N_E * N_t <= 2^26 as gb200_bucket2d */
} gb200_lagtransfer_opts;

/* Traces every ray of a GB200_IC_POLAR_PLANE `ic` (anything else: GB200_ERR_UNSUPPORTED, the r^2 area weight of
   unnormalized_areas, image-planes/planes.jl:108-115, is defined only there) with the point functions of lagtransfer
   (status, redshift, disc radius, coordinate time) and bins its hits -- rays with status IntersectedWithGeometry -- without
   copying per-ray data to the host:
     E = g E0,  T = t(rho) + t,  f = g^3 eps(rho) r^2  (r: the ray's polar-plane radius);
     eb = linspace(E_lo, E_hi, N_E), tb = linspace(T_lo, T_hi, N_t) (edge k = k * step + lo, two roundings, the last = hi);
     tf[i * N_t + j] = (sum of f over the hits in cell (i, j)) / (sum of f over all hits) / ((eb[1] - eb[0]) (tb[1] - tb[0])),
   Buckets.Simple in both axes (cell i takes eb[i] <= E < eb[i+1], clamped at both ends), NaN where no hit with f != 0
   landed.  time_edges = tb - t0 (N_t), energy_edges = eb (N_E), *hits = the number of hits.  f is summed as 64-bit fixed
   point with scale 2^floor(62 - log2(H max|f|)) (H: hits), so the result does not depend on the order of summation or on
   the number of devices.  GB200_ERR_INVALID_ARGUMENT also for automatic limits without hits or with min == max, and for
   a hit whose E, T or f is not finite; these are found after the trace.  Geometry, callback and plunging-table rules are
   those of gb200_render. */
int gb200_lagtransfer(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic, const gb200_disc_profile* profile,
                      const gb200_plunging_table* plunging, const gb200_lagtransfer_opts* opts,
                      double* time_edges, double* energy_edges, double* tf, int64_t* hits);

/* ---- line profiles and lag-energy transfer functions from Cunningham transfer functions ---- */
/* integrate_lineprofile / integrate_lagtransfer (src/transfer-functions/integration.jl:158-207, 233-279, 322-442) for many
   emission models at once.  One table is an InterpolatingTransferBranches (transfer-functions-2d.jl:1-88) as the host holds
   it after interpolate_branches: branch 2k is the lower, 2k+1 the upper branch of radius k, with knots
   [off[b], off[b+1]) of gs / f / t (g* non-decreasing, >= 2 knots).  f and t are NaNLinearInterpolators with default 0:
   NaN knots are allowed, evaluation extrapolates linearly beyond the ends. */
typedef struct gb200_tf_branches {
    int32_t n_radii;                 /* >= 2, r_e strictly ascending */
    int32_t reserved;
    const double *r_e, *gmin, *gmax; /* n_radii each, finite gmin < gmax */
    const int64_t* off;              /* 2 n_radii + 1, off[0] = 0 */
    const double *gs, *f, *t;        /* off[2 n_radii] knots each */
} gb200_tf_branches;

typedef struct gb200_tf_model {
    int32_t table;              /* index into tables[] */
    int32_t n_radii;            /* annuli, >= 2 */
    const double* radii;        /* host, strictly ascending: inverse_grid (line profile) or geometric_grid (lag) of (rmin, rmax) */
    double rmin;                /* r_prev of the first annulus is rmin - (radii[1] - rmin), as on the host */
    double g_scale;             /* bins are g_grid / g_scale; positive and finite */
    gb200_disc_profile profile; /* emissivity for both calls (POWERLAW: r^-index, TABLE: numpy.interp of the clipped radius);
                                   the arrival-time table is read by gb200_tf_lagtransfer only */
} gb200_tf_model;

typedef struct gb200_tf_quad_opts {
    double h;                      /* edge zone in g*, 0 < h < 0.5 */
    double t0;                     /* gb200_tf_lagtransfer: subtracted from the profile's arrival time */
    int32_t upscale;               /* g_grid_upscale >= 1: sub-bins per bin */
    int32_t npoints;               /* Gauss-Legendre points, 1..32 */
    const double *nodes, *weights; /* npoints each: the rule on [-1, 1] (numpy leggauss / FastGaussQuadrature) */
    int32_t normalise;             /* 1: _normalize! (divide bin j by g[j] + g[j+1], then by the total); 0: raw sums */
    int32_t reserved;
} gb200_tf_quad_opts;

/* out[m * ngrid + j]: the line profile of model m, bin j = [g_grid[j], g_grid[j+1]) (the last entry is 0, as on the host).
   Each (model, bin) is one device thread that walks the annuli in the host's order, so every result is independent of the
   other models of the call.  Every argument is checked before the first launch (GB200_ERR_INVALID_ARGUMENT). */
int gb200_tf_lineprofile(gb200_ctx* ctx, int32_t ntables, const gb200_tf_branches* tables, int32_t nmodels,
                         const gb200_tf_model* models, const double* g_grid, int32_t ngrid, const gb200_tf_quad_opts* opts,
                         double* out);
/* out[(m * ngrid + j) * nt + k]: the lag-energy transfer function of model m, energy bin j, time bin k, where a branch's
   contribution lands in the first k with t_grid[k] >= its time (numpy.searchsorted, side left) and is dropped past the
   end.  t_grid: nt >= 1, strictly ascending. */
int gb200_tf_lagtransfer(gb200_ctx* ctx, int32_t ntables, const gb200_tf_branches* tables, int32_t nmodels,
                         const gb200_tf_model* models, const double* g_grid, int32_t ngrid, const double* t_grid, int32_t nt,
                         const gb200_tf_quad_opts* opts, double* out);

/* ---- device-resident variants (inputs/outputs stay in HBM) ------------- */
/* Same as gb200_render but `d_images[k]` are DEVICE pointers on ctx's device and no
   host copy is made; work is enqueued on `cuda_stream` (a cudaStream_t cast to
   void*, NULL = the context's own stream) and the call returns without
   synchronising when `async` != 0.  An asynchronous call leaves kernels running that use the
   context's work queue and scratch buffers: the library orders every later call on the same context (on
   whatever stream) after them with an event, so calls may be issued back to back; the caller only has
   to synchronise `cuda_stream` before it reads the results, and gb200_get_stats reports no step
   counters for asynchronous calls. */
int gb200_render_device(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic,
                        const gb200_range* range, const int32_t* pointfns, int32_t npf,
                        const gb200_plunging_table* plunging, double* const* d_images,
                        void* cuda_stream, int async);

/* Raw (un-normalised) line-profile partial sums into a DEVICE buffer of nbins
   doubles, ready for an NCCL all-reduce issued by the caller on the same stream. */
int gb200_lineprofile_device(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic,
                             const gb200_range* range, const gb200_emissivity* emis,
                             const gb200_plunging_table* plunging,
                             const double* bins, int32_t nbins,
                             const gb200_lineprofile_opts* opts, double* d_flux,
                             void* cuda_stream, int async);

/* ---- several GPUs from ONE process (the Julia extension: EnsembleB200(devices)) ---------------------------- */
/* One context per listed device plus, for more than one device, an NCCL communicator over them (ncclCommInitAll).  NCCL is
   opened at run time (dlopen "libnccl.so.2"): a single-GPU caller does not need it.  Rays are sharded by whole strips of
   four image columns / theta-rows (strip d, d + ndev, ... on device d); the data-path collectives are the
   line-profile histogram, which is summed with one ncclAllReduce(sum, nbins doubles) on the devices' own streams
   (SURVEY 8e), and the lag-energy histogram of gb200_comm_lagtransfer.  torchrun-style callers (one process per GPU) use gb200_lineprofile_device + their own all-reduce instead. */
typedef struct gb200_comm gb200_comm;
int gb200_comm_init(const int32_t* devices, int32_t ndev, gb200_comm** out);
void gb200_comm_destroy(gb200_comm* comm);
int gb200_comm_size(gb200_comm* comm);
gb200_ctx* gb200_comm_context(gb200_comm* comm, int32_t i); /* borrowed: the context of the i-th device */
/* lineprofile(::BinningMethod) over all devices; flux_out: nbins doubles on the host, identical whatever ndev up to the
   order of summation (<= 1e-12 of the peak). */
int gb200_comm_lineprofile(gb200_comm* comm, const gb200_problem* p, const gb200_ic* ic, const gb200_emissivity* emis,
                           const gb200_plunging_table* plunging, const double* bins, int32_t nbins,
                           const gb200_lineprofile_opts* opts, double* flux_out);
/* rendergeodesics over all devices: images[k] -> ic->n doubles on the host in ray order (the (H, W) column-major image). */
int gb200_comm_render(gb200_comm* comm, const gb200_problem* p, const gb200_ic* ic, const int32_t* pointfns, int32_t npf,
                      const gb200_plunging_table* plunging, double* const* images);
/* gb200_lagtransfer over all devices: each bins its strips; the limits, hit count and max |f| are made global with
   ncclAllReduce (min, max, sum) before binning, and the integer cells with one ncclAllReduce(sum), so the result is
   bit-identical to gb200_lagtransfer on one device. */
int gb200_comm_lagtransfer(gb200_comm* comm, const gb200_problem* p, const gb200_ic* ic, const gb200_disc_profile* profile,
                           const gb200_plunging_table* plunging, const gb200_lagtransfer_opts* opts,
                           double* time_edges, double* energy_edges, double* tf, int64_t* hits);

/* Diagnostics: evaluate the device right-hand side (_second_order_ode_f, src/tracing/geodesic-problem.jl:87-92) for
   n states u (row-major n x 8) -> du (n x 8), and the kernel's branch-free elementary functions on n inputs
   (out5 = n x 5: sin x, cos x, 1/x, log|x|, exp(clamp(x, -8, 8))).  Lets tests check the closed forms against the
   oracle's AD-based RHS and libm directly. */
int gb200_debug_rhs(gb200_ctx* ctx, int32_t metric_kind, const double* metric_params, int64_t n, const double* u, double* du);
int gb200_debug_math(gb200_ctx* ctx, int64_t n, const double* x, double* out5);
/* The step controller's own log and exp (evaluated to 1e-7, the accuracy of the error estimate they act on; DESIGN.md K1):
   out2 = n x 2: log|x|, exp(clamp(x, -8, 8)). */
int gb200_debug_math_lo(gb200_ctx* ctx, int64_t n, const double* x, double* out2);

/* Dependent-free DFMA micro-benchmark: measured FP64 FMA throughput of the
   device in TFLOP/s (2 flop per FMA); the roofline denominator. */
int gb200_fp64_peak(gb200_ctx* ctx, double* tflops_out);

/* Diagnostic behind the roofline discussion (DESIGN.md section 4): the DFMA stream of gb200_fp64_peak with `mix` = 1 or 2
   independent integer-pipe instructions per DFMA (do non-FP64 instructions issue in the shadow of the FP64 ones?),
   mix = 3: DFMAs whose three operands are distinct vector registers, mix = 4: DMUL / DADD with register operands,
   mix = 5: three register operands of which one is shared by consecutive DFMAs (operand reuse).
   Returns the FP64 instruction rate x 2 in T/s (= TFLOP/s for the DFMA modes). */
int gb200_fp64_issue_probe(gb200_ctx* ctx, int32_t mix, double* tflops_out);

#ifdef __cplusplus
}
#endif
#endif /* GRADUS_B200_H */
