// gb200_api.cu -- the C ABI of include/gradus_b200.h: context, validation, host-side problem
// set-up (observer LNRF constants, special radii), device buffer management and launches.
// No CPU implementation of the path exists in this library: every compute entry point runs
// the sm_100a kernels of gb200_trace.cu or fails.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h> // types and enums only: the library is opened at run time (see gb200_comm_init)
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <mutex>
#include <string>
#include <functional>
#include <thread>
#include <vector>
#include "gb200_device.cuh"
#include "gb200_internal.h"

// ---------------------------------------------------------------- errors
static thread_local std::string g_last_error;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

struct gb200_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr; // the context's own stream
    cudaStream_t cur = nullptr;    // stream of the call in flight (own stream unless the caller passed one)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr;
    std::string err;
    gb200_stats stats{};
    std::vector<DevBuf> pool;
    unsigned long long* d_queue = nullptr; // [0] queue, [1..3] counters
    std::vector<cudaStream_t> pool_streams; // batch calls, pipelined gb200_render, gb200_comm_render's copies
    std::vector<cudaEvent_t> chunk_events;  // pipelined gb200_render and gb200_comm_render: per chunk
    void* stage = nullptr;                  // pinned host staging for gb200_trace_batch
    size_t stage_cap = 0;
    // An asynchronous call (gb200_render_device / gb200_lineprofile_device with async != 0) returns while its kernels still
    // use the context's work queue and pool buffers: it records `inflight` at its end, and every entry point makes the
    // stream it works on wait for that event before touching the queue or the pool.
    cudaEvent_t inflight = nullptr;
    bool have_inflight = false;
    // cross-section table of GB200_GEOMETRY_THICK_TABLE (gb200_set_cross_section)
    double* d_cs = nullptr; // [rho (n) | height (n)]
    int cs_n = 0;
    double cs_max = 0.0;
};

static int fail(gb200_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    if (ctx) ctx->err = buf;
    return code;
}
#define CU(ctx, call)                                                                                      \
    do {                                                                                                   \
        cudaError_t e__ = (call);                                                                          \
        if (e__ != cudaSuccess) return fail(ctx, GB200_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e__)); \
    } while (0)

// ---------------------------------------------------------------- host-only dual number (d/dr), for the ISCO root find
struct D1 {
    double v, d;
    GB_HD D1(double v_ = 0.0, double d_ = 0.0) : v(v_), d(d_) {}
    GB_HD friend D1 operator+(const D1& a, const D1& b) { return D1(a.v + b.v, a.d + b.d); }
    GB_HD friend D1 operator-(const D1& a, const D1& b) { return D1(a.v - b.v, a.d - b.d); }
    GB_HD friend D1 operator-(const D1& a) { return D1(-a.v, -a.d); }
    GB_HD friend D1 operator*(const D1& a, const D1& b) { return D1(a.v * b.v, a.d * b.v + a.v * b.d); }
    GB_HD friend D1 operator/(const D1& a, const D1& b) { double q = a.v / b.v; return D1(q, (a.d - q * b.d) / b.v); }
};
GB_HD static inline D1 gb_rcp(const D1& a) { return D1(1.0) / a; }
static inline D1 dsqrt(const D1& a) { double s = std::sqrt(a.v); return D1(s, a.d / (2.0 * s)); }
static inline double dsqrt(double a) { return std::sqrt(a); }
static inline double val(const D1& a) { return a.v; }
static inline double val(double a) { return a; }

// E = -u_t of the equatorial circular orbit at radius r (CircularOrbits.energy, src/orbits/circular-orbits.jl:11-52)
template <class S>
static S circular_energy_host(int kind, const double* mp, S r) {
    S g[5], dr[5], dth[5];
    metric_jacobian_kind<S>(kind, mp, r, S(1.0), S(0.0), g, dr, dth);
    const S D = g[0] * g[3] - g[4] * g[4];
    const S gitt = g[3] / D, giphph = g[0] / D, gitph = -g[4] / D;
    const S Om = -(dr[4] - dsqrt(dr[4] * dr[4] - dr[0] * dr[3])) / dr[3];
    const S A = -(Om * gitt - gitph);
    const S B = (Om * gitph - giphph);
    const S denom = B * B * gitt + 2.0 * A * B * gitph + A * A * giphph;
    const double sg = val(denom) > 0 ? 1.0 : (val(denom) < 0 ? -1.0 : 0.0);
    const S ad = val(denom) < 0 ? -denom : denom;
    const S d = -sg * dsqrt(S(1.0) / ad);
    return -(B * d);
}

static double kerr_isco_host(double M, double a) { // Bardeen et al. (1972), kerr-metric-first-order.jl:297-337
    const double x = a / M;
    const double Z1 = 1 + std::cbrt(1 - x * x) * (std::cbrt(1 + x) + std::cbrt(1 - x));
    const double Z2 = std::sqrt(3 * x * x + Z1 * Z1);
    const double s = std::sqrt((3 - Z1) * (3 + Z1 + 2 * Z2));
    return a > 0.0 ? M * (3 + Z2 - s) : M * (3 + Z2 + s);
}

// isco(::AbstractStaticAxisSymmetric): bracket from find_isco_bounds, then the root of dE/dr (special-radii.jl:14-60)
static int generic_isco_host(int kind, const double* mp, double* out) {
    double lower = 0, upper = 0;
    for (long n = 0;; ++n) {
        const double r = 100.0 - 0.005 * (double)n;
        if (r < 1.0) break;
        const double en = circular_energy_host<double>(kind, mp, r);
        if (std::fabs(en) > 1.0) { lower = r; upper = 100.0; break; }
    }
    if (lower == upper) return GB200_ERR_INVALID_ARGUMENT;
    auto dE = [&](double r) { return circular_energy_host<D1>(kind, mp, D1(r, 1.0)).d; };
    double lo = lower, hi = upper, flo = dE(lo);
    for (int it = 0; it < 200; ++it) {
        const double mid = lo + (hi - lo) / 2;
        if (!(mid > lo && mid < hi)) break;
        const double fm = dE(mid);
        if (fm == 0) { lo = hi = mid; break; }
        if ((fm > 0) == (flo > 0)) { lo = mid; flo = fm; } else hi = mid;
    }
    *out = lo + (hi - lo) / 2;
    return GB200_OK;
}

// Start of every entry point that uses the context's queue / pool on `stream`: order it after an earlier asynchronous call.
static int begin_call(gb200_ctx* ctx, cudaStream_t stream) {
    CU(ctx, cudaSetDevice(ctx->device));
    ctx->stats = gb200_stats{};
    ctx->cur = stream;
    if (ctx->have_inflight) CU(ctx, cudaStreamWaitEvent(stream, ctx->inflight, 0));
    return GB200_OK;
}
// End of an asynchronous call: later calls (on any stream) wait for the work enqueued so far.
static int end_async_call(gb200_ctx* ctx, cudaStream_t stream) {
    CU(ctx, cudaEventRecord(ctx->inflight, stream));
    ctx->have_inflight = true;
    return GB200_OK;
}

// ---------------------------------------------------------------- validation
static int validate(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic) {
    if (!p || !ic) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "null problem or ic");
    if (p->metric_kind < 0 || p->metric_kind >= GB200_METRIC_COUNT)
        return fail(ctx, GB200_ERR_UNSUPPORTED, "metric kind %d has no closed-form right-hand side in this library", p->metric_kind);
    const double M = p->metric_params[0], a = p->metric_params[1];
    if (p->metric_kind == GB200_METRIC_MORRIS_THORNE) { // metric_params[0] is the throat size b, there is no mass or spin
        if (!(M == M)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "Morris-Thorne throat size b is NaN");
    } else if (!(M > 0) || !(std::fabs(a) <= M)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "need M > 0 and |a| <= M (M=%g a=%g)", M, a);
    if (p->metric_kind == GB200_METRIC_BUMBLEBEE && (!(p->metric_params[2] > -1.0) || std::fabs(a) > 0.3))
        return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "Bumblebee metric needs l > -1 and |a| <= 0.3 (bumblebee-ad.jl:33-40)");
    if (p->metric_kind == GB200_METRIC_DILATON_AXION && p->metric_params[2] != 0.0 && (a == 0.0 || p->metric_params[3] == 0.0))
        return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "Dilaton-Axion metric with beta != 0 needs a != 0 and b != 0 (beta / a, beta / b; dilaton-axion-ad.jl:24-26)");
    if (p->metric_kind == GB200_METRIC_KERR_NEWMAN && a * a + p->metric_params[2] * p->metric_params[2] > M * M)
        return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "Kerr-Newman metric needs a^2 + Q^2 <= M^2 (kerr-newman-ad.jl:50-52)");
    if ((p->geometry_kind < GB200_GEOMETRY_NONE || p->geometry_kind > GB200_GEOMETRY_THICK_TABLE) && p->geometry_kind != GB200_GEOMETRY_THIN_DISC_ORDER)
        return fail(ctx, GB200_ERR_UNSUPPORTED, "geometry kind %d is outside the hot-path scope", p->geometry_kind);
    if ((p->geometry_kind == GB200_GEOMETRY_THIN_DISC || p->geometry_kind == GB200_GEOMETRY_THIN_DISC_ORDER) && !(p->geometry_params[0] <= p->geometry_params[1]))
        return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "ThinDisc needs inner_radius <= outer_radius");
    if (p->geometry_kind == GB200_GEOMETRY_THIN_DISC_ORDER) {
        const double n = p->geometry_params[2];
        if (!(n >= 0.0 && n <= 2147483647.0 && n == std::floor(n)))
            return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "ImageOrder needs a non-negative integer order below 2^31 (got %g)", n);
    }
    if (p->callback_kind != GB200_CALLBACK_NONE && p->callback_kind != GB200_CALLBACK_UPPER_HEMISPHERE)
        return fail(ctx, GB200_ERR_UNSUPPORTED, "callback kind %d cannot run on the device", p->callback_kind);
    if (p->pow_mode != GB200_POW_EXACT && p->pow_mode != GB200_POW_FAST32) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bad pow_mode");
    if (!(p->mu == p->mu) && ic->kind != GB200_IC_EXPLICIT) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "mu = NaN (keep v^t as given) needs explicit initial conditions");
    if (!(p->lambda_max > p->lambda_min)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "need lambda_max > lambda_min");
    if (!(p->abstol > 0) || !(p->reltol > 0)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "abstol and reltol must be positive");
    if (!(p->chart_outer > p->chart_inner)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "chart outer radius must exceed inner radius");
    if (ic->kind == GB200_IC_RENDER_GRID) {
        if (ic->width < 1 || ic->height < 1) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "image size must be positive");
        if (!(ic->lo0 <= ic->hi0) || !(ic->lo1 <= ic->hi1)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "alpha / beta limits must be sorted");
        if (ic->n != ic->width * ic->height) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "ic.n != width*height");
    } else if (ic->kind == GB200_IC_POLAR_PLANE) {
        if (ic->width < 2 || ic->height < 1) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "PolarPlane needs Nr >= 2, Ntheta >= 1");
        if (ic->grid_kind < GB200_GRID_LINEAR || ic->grid_kind > GB200_GRID_INVERSE) return fail(ctx, GB200_ERR_UNSUPPORTED, "grid kind %d", ic->grid_kind);
        if (!(ic->lo0 > 0) || !(ic->hi0 > ic->lo0)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "PolarPlane needs 0 < r_min < r_max");
        if (ic->n != ic->width * ic->height) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "ic.n != Nr*Ntheta");
    } else if (ic->kind == GB200_IC_CARTESIAN_PLANE) {
        if (ic->width < 4 || ic->height < 4) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "CartesianPlane needs Nx, Ny >= 4");
        if (ic->grid_kind < GB200_GRID_LINEAR || ic->grid_kind > GB200_GRID_INVERSE) return fail(ctx, GB200_ERR_UNSUPPORTED, "grid kind %d", ic->grid_kind);
        if (!(ic->hi0 > ic->lo0) || !(ic->hi1 > ic->lo1)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "CartesianPlane needs x_min < x_max, y_min < y_max");
        if (ic->grid_kind != GB200_GRID_LINEAR && (!(ic->lo0 > 0) || !(ic->lo1 > 0))) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "geometric / inverse grids need positive minima");
        if (ic->n != (2 * (ic->height / 2) - 1) * (2 * (ic->width / 2) - 1)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "ic.n != (2(Ny/2)-1)(2(Nx/2)-1)");
    } else if (ic->kind == GB200_IC_IMPACT_PARAMETERS) {
        if (ic->n < 1 || !ic->x[0] || !ic->x[1]) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "impact-parameter IC needs n >= 1 and alpha / beta arrays");
    } else if (ic->kind == GB200_IC_EXPLICIT) {
        if (ic->n < 1) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "explicit IC needs n >= 1");
        for (int k = 0; k < 4; ++k)
            if (!ic->x[k] || !ic->v[k]) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "explicit IC pointers must be non-null");
    } else return fail(ctx, GB200_ERR_UNSUPPORTED, "ic kind %d", ic->kind);
    return GB200_OK;
}

// The image order is a rule of the throughput kernel's event handling; the generic (forward-mode, target, path) integrator
// does not have it.  Checked before the context, like validate_crossings.
static int reject_image_order(gb200_ctx* ctx, const gb200_problem* p, const char* entry) {
    if (p && p->geometry_kind == GB200_GEOMETRY_THIN_DISC_ORDER)
        return fail(ctx, GB200_ERR_UNSUPPORTED, "%s does not support GB200_GEOMETRY_THIN_DISC_ORDER", entry);
    return GB200_OK;
}

// GB200_PF_EQUATORIAL_CROSSINGS is counted with no geometry and on the thin disc only.  Checked before anything else (a
// device context included), so that callers can probe it without a GPU.
static int validate_crossings(gb200_ctx* ctx, const gb200_problem* p, const int32_t* pfs, int npf) {
    if (!p || !pfs) return GB200_OK;
    for (int k = 0; k < npf && k < GB_MAX_PF; ++k)
        if (pfs[k] == GB200_PF_EQUATORIAL_CROSSINGS && p->geometry_kind != GB200_GEOMETRY_NONE && p->geometry_kind != GB200_GEOMETRY_THIN_DISC &&
            p->geometry_kind != GB200_GEOMETRY_THIN_DISC_ORDER)
            return fail(ctx, GB200_ERR_UNSUPPORTED, "GB200_PF_EQUATORIAL_CROSSINGS needs geometry NONE, THIN_DISC or THIN_DISC_ORDER (got %d)", p->geometry_kind);
    return GB200_OK;
}

// 1..GB_MAX_PF point functions of kinds the kernel evaluates; where `images` is given, a non-null image for each
static int validate_pfs(gb200_ctx* ctx, const int32_t* pfs, int npf, double* const* images) {
    if (npf < 1 || npf > GB_MAX_PF || !pfs) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "need 1..%d point functions", GB_MAX_PF);
    for (int k = 0; k < npf; ++k) {
        if (pfs[k] < GB200_PF_SHADOW || pfs[k] > GB200_PF_EQUATORIAL_CROSSINGS) return fail(ctx, GB200_ERR_UNSUPPORTED, "point function %d", pfs[k]);
        if (images && !images[k]) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "null image pointer");
    }
    return GB200_OK;
}

static int validate_range(gb200_ctx* ctx, const gb200_ic* ic, const gb200_range* rg) {
    if (!rg) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "null range");
    if (rg->count < 0 || rg->first < 0 || rg->stride < 1 || rg->block < 0) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bad range");
    const int64_t blk = rg->block > 0 ? rg->block : 1;
    if (rg->count > 0) {
        const int64_t nlast = rg->count - 1;
        const int64_t last = rg->first + (nlast / blk) * (rg->stride * blk) + nlast % blk;
        if (last >= ic->n) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "range exceeds the %lld rays of the IC", (long long)ic->n);
    }
    return GB200_OK;
}

// ---------------------------------------------------------------- problem -> kernel parameters (host arithmetic)
static void dd_step(double lo, double hi, int64_t n, double* shi, double* slo) { // (hi-lo)/(n-1) as double-double
    if (n <= 1) { *shi = 0; *slo = 0; return; }
    const long double s = ((long double)hi - (long double)lo) / (long double)(n - 1);
    *shi = (double)s;
    *slo = (double)(s - (long double)*shi);
}

// Rays per image column (render grid) or theta-row (polar and Cartesian planes): the fastest-varying extent of the ray
// index, whose multiples of GB_TILE_C make the strips of the tiled work order and of the multi-GPU shards.  0 for ray lists.
static int64_t strip_height(const gb200_ic* ic) {
    if (ic->kind == GB200_IC_RENDER_GRID) return ic->height;
    if (ic->kind == GB200_IC_POLAR_PLANE) return ic->width;
    if (ic->kind == GB200_IC_CARTESIAN_PLANE) return 2 * (ic->height / 2) - 1;
    return 0;
}

static void fill_params(const gb200_problem* p, const gb200_ic* ic, const gb200_range* rg, GbParams& P) {
    memset(&P, 0, sizeof P);
    P.metric_kind = p->metric_kind;
    P.M = p->metric_params[0]; P.a = p->metric_params[1]; P.eps3 = p->metric_params[2];
    P.a2 = P.a * P.a; P.twoM = 2.0 * P.M; P.jp_e = P.eps3 * P.M * P.M * P.M;
    for (int k = 0; k < 8; ++k) P.mp[k] = p->metric_params[k];
    P.lam0 = p->lambda_min; P.lam1 = p->lambda_max; P.abstol = p->abstol; P.reltol = p->reltol;
    P.dtmax = p->dtmax > 0 ? p->dtmax : (p->lambda_max - p->lambda_min);
    P.mu = p->mu;
    P.maxiters = p->maxiters > 0 ? p->maxiters : 1000000;
    P.pow_mode = p->pow_mode;
    P.geometry_kind = p->geometry_kind;
    P.gp0 = p->geometry_params[0]; P.gp1 = p->geometry_params[1]; P.gp2 = p->geometry_params[2];
    P.gtol = p->gtol;
    P.chart_inner = p->chart_inner; P.chart_outer = p->chart_outer;
    P.callback_kind = p->callback_kind; P.callback_delta = p->callback_delta;
    P.ic_kind = ic->kind; P.grid_kind = ic->grid_kind;
    P.width = ic->width; P.height = ic->height;
    for (int k = 0; k < 4; ++k) P.xo[k] = p->observer[k];
    if (ic->kind == GB200_IC_RENDER_GRID) {
        P.lo0 = ic->lo0; dd_step(ic->lo0, ic->hi0, ic->width, &P.step0_hi, &P.step0_lo);
        P.lo1 = ic->lo1; dd_step(ic->lo1, ic->hi1, ic->height, &P.step1_hi, &P.step1_lo);
    } else if (ic->kind == GB200_IC_POLAR_PLANE) {
        P.lo0 = ic->lo0; dd_step(ic->lo0, ic->hi0, ic->width, &P.step0_hi, &P.step0_lo);
        P.geoK = std::pow(ic->hi0 / ic->lo0, 1.0 / (double)(ic->width - 1));
        P.inv_lo_hi = 1.0 / ic->hi0; dd_step(1.0 / ic->hi0, 1.0 / ic->lo0, ic->width, &P.inv_step_hi, &P.inv_step_lo);
        const double dth = (ic->hi1 - ic->lo1) / (double)ic->height; // planes.jl:95-96
        P.lo1 = ic->lo1; dd_step(ic->lo1, ic->hi1 - dth, ic->height, &P.step1_hi, &P.step1_lo);
    }
    if (ic->kind == GB200_IC_CARTESIAN_PLANE) {
        P.n0 = ic->width / 2; P.n1 = ic->height / 2;
        P.lo0 = ic->lo0; dd_step(ic->lo0, ic->hi0, P.n0, &P.step0_hi, &P.step0_lo);
        P.lo1 = ic->lo1; dd_step(ic->lo1, ic->hi1, P.n1, &P.step1_hi, &P.step1_lo);
        if (ic->grid_kind != GB200_GRID_LINEAR) {
            P.geoK = std::pow(ic->hi0 / ic->lo0, 1.0 / (double)(P.n0 - 1));
            P.geoK1 = std::pow(ic->hi1 / ic->lo1, 1.0 / (double)(P.n1 - 1));
            P.inv_lo_hi = 1.0 / ic->hi0; dd_step(1.0 / ic->hi0, 1.0 / ic->lo0, P.n0, &P.inv_step_hi, &P.inv_step_lo);
            P.inv1_lo_hi = 1.0 / ic->hi1; dd_step(1.0 / ic->hi1, 1.0 / ic->lo1, P.n1, &P.inv1_step_hi, &P.inv1_step_lo);
        }
    }
    if (ic->kind != GB200_IC_EXPLICIT) {
        // closed-form LNRF (ZAMO) co-basis at the observer, generic for static axisymmetric g:
        //   e^(t) = N dt, e^(r) = sqrt(g_rr) dr, e^(th) = sqrt(g_thth) dth, e^(ph) = sqrt(g_phph)(dph - w dt)
        double g[5];
        metric_components_rt(P, P.xo[1], P.xo[2], g);
        for (int k = 0; k < 5; ++k) P.go[k] = g[k];
        const double D = g[0] * g[3] - g[4] * g[4];
        const double gitt = g[3] / D, giphph = g[0] / D, gitph = -g[4] / D;
        const double N = std::sqrt(-1.0 / gitt);
        const double om = -g[4] / g[3];
        const double sph = std::sqrt(g[3]);
        P.c_r = 1.0 / std::sqrt(g[1]);
        P.c_th = 1.0 / std::sqrt(g[2]);
        P.c_ph0 = gitph * N;
        P.c_ph1 = (giphph - gitph * om) * sph;
    }
    P.first = rg->first; P.count = rg->count; P.stride = rg->stride;
    P.block = rg->block > 0 ? rg->block : 1;
    // 2-D tiled work order when the range is made of whole strips of GB_TILE_C image columns (or theta-rows of the plane)
    const int64_t h = strip_height(ic), strip = GB_TILE_C * h;
    if (h > 0 && h % GB_TILE_R == 0 && (P.stride == 1 || P.block % strip == 0) && P.first % strip == 0 && P.count % strip == 0) P.tile_h = h;
}

// ---------------------------------------------------------------- device memory
static int pool_get(gb200_ctx* ctx, size_t slot, size_t bytes, void** out) {
    if (ctx->pool.size() <= slot) ctx->pool.resize(slot + 1);
    DevBuf& b = ctx->pool[slot];
    if (b.cap < bytes) {
        if (b.p) cudaFree(b.p);
        b.p = nullptr; b.cap = 0;
        cudaError_t e = cudaMalloc(&b.p, bytes);
        if (e != cudaSuccess) return fail(ctx, GB200_ERR_NOMEM, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
        b.cap = bytes;
    }
    *out = b.p;
    return GB200_OK;
}
// pool slots
enum { SL_STATUS = 0, SL_LAMBDA, SL_X0, SL_V0 = SL_X0 + 4, SL_XI0 = SL_V0 + 4, SL_VI0 = SL_XI0 + 4, SL_NACC = SL_VI0 + 4, SL_NREJ, SL_FLAGS,
       SL_IMG0, SL_G = SL_IMG0 + GB_MAX_PF, SL_F, SL_EX0, SL_EV0 = SL_EX0 + 4, SL_BINS = SL_EV0 + 4, SL_PARTIAL, SL_FLUX, SL_EMR, SL_EME,
       SL_PL0, SL_SCRATCH = SL_PL0 + 4, SL_BATCH, SL_BATCH_QUEUE,
       SL_LAG_SAMPLES, SL_LAG_PARTIAL, SL_LAG_SCAL, SL_LAG_CELLS, SL_LAG_OUT, SL_LAG_PROF, SL_TFQ_IN, SL_TFQ_OUT, SL_COUNT };

// The output arrays of gb200_endpoints: f(host array, GbParams field the kernel writes it through, pool slot of a single
// call) for each, null host arrays included.  Every copy, binding and layout of endpoints goes through this one list.
template <class F> static void endpoint_arrays(const gb200_endpoints& out, GbParams& P, F&& f) {
    f(out.status, P.o_status, SL_STATUS);
    f(out.lambda_max, P.o_lambda, SL_LAMBDA);
    for (int k = 0; k < 4; ++k) {
        f(out.x[k], P.o_x[k], SL_X0 + k);
        f(out.v[k], P.o_v[k], SL_V0 + k);
        f(out.x_init[k], P.o_x0[k], SL_XI0 + k);
        f(out.v_init[k], P.o_v0[k], SL_VI0 + k);
    }
    f(out.naccept, P.o_naccept, SL_NACC);
    f(out.nreject, P.o_nreject, SL_NREJ);
    f(out.flags, P.o_flags, SL_FLAGS);
}

static int upload(gb200_ctx* ctx, size_t slot, const void* host, size_t bytes, const void** dev) {
    void* d = nullptr;
    int rc = pool_get(ctx, slot, bytes, &d);
    if (rc) return rc;
    CU(ctx, cudaMemcpyAsync(d, host, bytes, cudaMemcpyHostToDevice, ctx->cur));
    *dev = d;
    return GB200_OK;
}

static int upload_ic_and_tables(gb200_ctx* ctx, const gb200_ic* ic, const gb200_plunging_table* pl, const gb200_emissivity* em, GbParams& P) {
    if (ic->kind == GB200_IC_IMPACT_PARAMETERS) {
        for (int k = 0; k < 3; ++k) {
            P.ex[k] = nullptr;
            if (k == 2 && !ic->x[2]) continue; // optional per-ray datum-plane heights
            const void* d;
            int rc = upload(ctx, SL_EX0 + k, ic->x[k], sizeof(double) * ic->n, &d); if (rc) return rc;
            P.ex[k] = (const double*)d;
        }
    }
    if (ic->kind == GB200_IC_EXPLICIT) {
        for (int k = 0; k < 4; ++k) {
            const void* d;
            int rc = upload(ctx, SL_EX0 + k, ic->x[k], sizeof(double) * ic->n, &d); if (rc) return rc;
            P.ex[k] = (const double*)d;
            rc = upload(ctx, SL_EV0 + k, ic->v[k], sizeof(double) * ic->n, &d); if (rc) return rc;
            P.ev[k] = (const double*)d;
        }
    }
    if (pl && pl->n >= 2) {
        const double* src[4] = {pl->r, pl->ut, pl->ur, pl->uphi};
        const double* dst[4];
        for (int k = 0; k < 4; ++k) {
            const void* d;
            int rc = upload(ctx, SL_PL0 + k, src[k], sizeof(double) * pl->n, &d); if (rc) return rc;
            dst[k] = (const double*)d;
        }
        P.pl_n = pl->n; P.pl_r = dst[0]; P.pl_ut = dst[1]; P.pl_ur = dst[2]; P.pl_uphi = dst[3];
    }
    if (em) {
        P.emis_kind = em->kind; P.emis_index = em->index; P.emis_n = em->n;
        if (em->kind == GB200_EMISSIVITY_TABLE) {
            if (em->n < 2 || !em->r || !em->eps) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "emissivity table needs n >= 2");
            const void* d;
            int rc = upload(ctx, SL_EMR, em->r, sizeof(double) * em->n, &d); if (rc) return rc;
            P.emis_r = (const double*)d;
            rc = upload(ctx, SL_EME, em->eps, sizeof(double) * em->n, &d); if (rc) return rc;
            P.emis_eps = (const double*)d;
        } else if (em->kind != GB200_EMISSIVITY_POWERLAW) return fail(ctx, GB200_ERR_UNSUPPORTED, "emissivity kind %d", em->kind);
    }
    return GB200_OK;
}

static int check_table(gb200_ctx* ctx, int32_t geometry_kind) {
    if (geometry_kind == GB200_GEOMETRY_THICK_TABLE && ctx->cs_n < 2)
        return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "GB200_GEOMETRY_THICK_TABLE needs a table: call gb200_set_cross_section first");
    return GB200_OK;
}

// GB200_GEOMETRY_THICK_TABLE: point the launch at the context's cross-section table
static int bind_geometry(gb200_ctx* ctx, GbParams& P) {
    { int rc_ = check_table(ctx, P.geometry_kind); if (rc_) return rc_; }
    if (P.geometry_kind != GB200_GEOMETRY_THICK_TABLE) return GB200_OK;
    P.cs_n = ctx->cs_n; P.cs_rho = ctx->d_cs; P.cs_h = ctx->d_cs + ctx->cs_n;
    P.gp0 = ctx->cs_max;
    return GB200_OK;
}

static bool needs_isco(const int32_t* pfs, int npf, bool lineprofile) {
    if (lineprofile) return true;
    for (int k = 0; k < npf; ++k) if (pfs[k] == GB200_PF_REDSHIFT) return true;
    return false;
}

static int set_isco(gb200_ctx* ctx, const gb200_problem* p, GbParams& P) {
    double r = 0;
    int rc = gb200_isco(p->metric_kind, p->metric_params, &r);
    if (rc) return fail(ctx, rc, "no ISCO found for this metric (is it a naked singularity?)");
    P.r_isco = r;
    return GB200_OK;
}

// run the trace kernel on `stream` (queue reset + launch), timing it with events when `timed`
static int run_trace(gb200_ctx* ctx, GbParams& P, cudaStream_t stream, bool timed) {
    P.queue = ctx->d_queue;
    P.counters = ctx->d_queue + 1;
    CU(ctx, cudaMemsetAsync(ctx->d_queue, 0, 4 * sizeof(unsigned long long), stream));
    if (timed) CU(ctx, cudaEventRecord(ctx->ev1, stream));
    int blocks = 0;
    if (P.count > 0) CU(ctx, gb200_launch_trace(P, ctx->sm_count, stream, &blocks));
    if (timed) CU(ctx, cudaEventRecord(ctx->ev2, stream));
    ctx->stats.launches += (P.count > 0) ? 1 : 0;
    return GB200_OK;
}

// add k launches' queue-counter quadruples ([0] ticket queue, [1..3] accepted steps, rejected steps, flagged rays)
static void add_counters(gb200_ctx* ctx, const unsigned long long* c, size_t k) {
    for (size_t i = 0; i < k; ++i) {
        ctx->stats.steps_accepted += (int64_t)c[4 * i + 1]; ctx->stats.steps_rejected += (int64_t)c[4 * i + 2];
        ctx->stats.flagged += (int64_t)c[4 * i + 3];
    }
}

static int finish_stats(gb200_ctx* ctx, int64_t rays) {
    unsigned long long c[4];
    CU(ctx, cudaMemcpyAsync(c, ctx->d_queue, sizeof c, cudaMemcpyDeviceToHost, ctx->cur));
    CU(ctx, cudaEventRecord(ctx->ev3, ctx->cur));
    CU(ctx, cudaStreamSynchronize(ctx->cur));
    float k = 0, tot = 0;
    cudaEventElapsedTime(&k, ctx->ev1, ctx->ev2);
    cudaEventElapsedTime(&tot, ctx->ev0, ctx->ev3);
    ctx->stats.kernel_ms = k; ctx->stats.total_ms = tot; ctx->stats.rays = rays;
    add_counters(ctx, c, 1);
    return GB200_OK;
}

static int ensure_streams(gb200_ctx* ctx, size_t n) {
    while (ctx->pool_streams.size() < n) {
        cudaStream_t st;
        CU(ctx, cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        ctx->pool_streams.push_back(st);
    }
    return GB200_OK;
}

static int ensure_events(gb200_ctx* ctx, size_t n) {
    while (ctx->chunk_events.size() < n) {
        cudaEvent_t ev;
        CU(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        ctx->chunk_events.push_back(ev);
    }
    return GB200_OK;
}

// ---------------------------------------------------------------- pipelined host-output launches
// Large host-output calls are pipelined: the range is cut into chunks of whole tile strips, the chunk kernels alternate
// between two streams (the next chunk's CTAs take over the SMs as the previous chunk drains, so there is no idle tail
// between them) and every chunk's results travel to the host while the following chunks compute.
static int64_t pipeline_unit(const GbParams& P) {
    const int64_t strip = P.tile_h ? (int64_t)GB_TILE_C * P.tile_h : 1;
    return (P.block % strip == 0) ? P.block : ((strip % P.block == 0) ? strip : 0);
}
static bool pipeline_eligible(const GbParams& P, const gb200_range* rg) {
    const int64_t unit = pipeline_unit(P);
    return unit > 0 && rg->count >= (1 << 20) && rg->count / unit >= 8 && !getenv("GB200_NO_PIPELINE");
}
// bind(Pc, slot0): point the chunk's outputs at slot0 of the full-range device buffers;
// copy_back(slot0, cnt, stream): enqueue the device-to-host copies of that chunk.
static int run_pipelined(gb200_ctx* ctx, const gb200_range* rg, const GbParams& P,
                         const std::function<void(GbParams&, int64_t)>& bind,
                         const std::function<cudaError_t(int64_t, int64_t, cudaStream_t)>& copy_back) {
    const int K = 4;
    cudaStream_t stream = ctx->cur;
    const int64_t unit = pipeline_unit(P);
    const int64_t per = ((rg->count / unit + K - 1) / K) * unit;
    int rc = ensure_streams(ctx, 2); if (rc) return rc;
    rc = ensure_events(ctx, (size_t)K + 2); if (rc) return rc;
    cudaStream_t alt = ctx->pool_streams[0], copy = ctx->pool_streams[1];
    void* qv = nullptr;
    rc = pool_get(ctx, SL_BATCH_QUEUE, sizeof(unsigned long long) * 4 * K, &qv); if (rc) return rc;
    unsigned long long* queues = (unsigned long long*)qv;
    CU(ctx, cudaMemsetAsync(queues, 0, sizeof(unsigned long long) * 4 * K, stream));
    CU(ctx, cudaEventRecord(ctx->ev1, stream)); // uploads and queue reset done: the other stream may start
    CU(ctx, cudaStreamWaitEvent(alt, ctx->ev1, 0));
    int nchunks = 0;
    for (int c = 0; c < K; ++c) {
        const int64_t slot0 = (int64_t)c * per;
        if (slot0 >= rg->count) break;
        GbParams Pc = P; // same problem, same tables; only the slot range and the output pointers move
        Pc.first = rg->first + (slot0 / P.block) * (P.stride * P.block);
        Pc.count = (rg->count - slot0 < per) ? rg->count - slot0 : per;
        bind(Pc, slot0);
        Pc.queue = queues + 4 * c;
        Pc.counters = Pc.queue + 1;
        cudaStream_t st = (c % 2 == 0) ? stream : alt;
        int blocks = 0;
        CU(ctx, gb200_launch_trace(Pc, ctx->sm_count, st, &blocks));
        ctx->stats.launches += 1;
        CU(ctx, cudaEventRecord(ctx->chunk_events[(size_t)c], st));
        ++nchunks;
    }
    // join the kernels on the context stream (end of the kernel span) before any copy is enqueued: a device-to-host
    // copy into pageable memory blocks the calling thread, so the copies come after all launches and event records
    for (int c = 1; c < nchunks; c += 2) CU(ctx, cudaStreamWaitEvent(stream, ctx->chunk_events[(size_t)c], 0));
    CU(ctx, cudaEventRecord(ctx->ev2, stream));
    for (int c = 0; c < nchunks; ++c) {
        const int64_t slot0 = (int64_t)c * per;
        const int64_t cnt = (rg->count - slot0 < per) ? rg->count - slot0 : per;
        CU(ctx, cudaStreamWaitEvent(copy, ctx->chunk_events[(size_t)c], 0));
        CU(ctx, copy_back(slot0, cnt, copy));
    }
    CU(ctx, cudaEventRecord(ctx->chunk_events[(size_t)K], copy));
    CU(ctx, cudaStreamWaitEvent(stream, ctx->chunk_events[(size_t)K], 0));
    std::vector<unsigned long long> cq((size_t)4 * K);
    CU(ctx, cudaMemcpyAsync(cq.data(), queues, sizeof(unsigned long long) * cq.size(), cudaMemcpyDeviceToHost, stream));
    CU(ctx, cudaEventRecord(ctx->ev3, stream));
    CU(ctx, cudaStreamSynchronize(stream));
    float kms = 0, tot = 0;
    cudaEventElapsedTime(&kms, ctx->ev1, ctx->ev2);
    cudaEventElapsedTime(&tot, ctx->ev0, ctx->ev3);
    ctx->stats.kernel_ms = kms; ctx->stats.total_ms = tot; ctx->stats.rays = rg->count;
    add_counters(ctx, cq.data(), (size_t)nchunks);
    return GB200_OK;
}

// ---------------------------------------------------------------- batches
// A batch call lays its items out in one device arena, [inputs of every item | outputs of every item], mirrored byte for
// byte by the context's pinned staging buffer, so the whole batch costs one H2D and one D2H copy instead of ~20 small
// ones per item.  An item's layout is written once, as calls of take() on an input and an output Arena, and run in
// passes: with null bases to size the arena, with the staging buffer to stage the inputs, with the device arena to bind
// the kernel's pointers, and with the staging buffer again to find the outputs.  So the passes cannot disagree.
struct Arena {
    char* base;                  // nullptr: the pass only sizes the arena
    bool fill = false;           // base is the staging buffer: copy each input's host array into its place
    size_t used = 0;
    const double* table[4] = {}; // the plunging table placed last (place_plunging)
    template <class T> void take(T*& p, int64_t n, const void* src = nullptr) {
        p = base ? (T*)(base + used) : nullptr;
        const size_t bytes = sizeof(T) * (size_t)n;
        if (fill && src) memcpy((void*)p, src, bytes);
        used += (bytes + 255) & ~(size_t)255;
    }
};

// Plunging table of batch item b, bound into P.  Consecutive items with the same table share one copy in the arena.
static void place_plunging(Arena& in, const gb200_plunging_table* const* pls, int b, GbParams& P) {
    const gb200_plunging_table* pl = pls ? pls[b] : nullptr;
    if (!pl || pl->n < 2) return;
    if (b == 0 || pl != pls[b - 1]) {
        const double* src[4] = {pl->r, pl->ut, pl->ur, pl->uphi};
        for (int k = 0; k < 4; ++k) in.take(in.table[k], pl->n, src[k]);
    }
    P.pl_n = pl->n;
    P.pl_r = in.table[0]; P.pl_ut = in.table[1]; P.pl_ur = in.table[2]; P.pl_uphi = in.table[3];
}

// The output arrays of gb200_dual_out: f(host array, GbDualIO field the kernel writes it through, element count).
template <class F> static void dual_arrays(const gb200_dual_out& out, GbDualIO& io, int64_t n, int64_t npartials, F&& f) {
    f(out.status, io.status, n);
    f(out.lambda_max, io.lambda, n);
    for (int k = 0; k < 4; ++k) {
        f(out.x[k], io.x[k], n);
        f(out.v[k], io.v[k], n);
    }
    f(out.g, io.g, n);
    f(out.dg, io.dg, n * npartials);
    f(out.rho, io.rho, n);
    f(out.drho, io.drho, n * npartials);
    f(out.naccept, io.naccept, n);
    f(out.nreject, io.nreject, n);
    f(out.flags, io.flags, n);
}

static int ensure_stage(gb200_ctx* ctx, size_t total) {
    if (ctx->stage_cap >= total) return GB200_OK;
    if (ctx->stage) cudaFreeHost(ctx->stage);
    ctx->stage = nullptr; ctx->stage_cap = 0;
    CU(ctx, cudaMallocHost(&ctx->stage, total + 256));
    ctx->stage_cap = total;
    return GB200_OK;
}

// the first nstreams pool streams start after the work enqueued on the context stream so far (ev1)
static int fan_out(gb200_ctx* ctx, int nstreams) {
    CU(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    for (int sidx = 0; sidx < nstreams; ++sidx) CU(ctx, cudaStreamWaitEvent(ctx->pool_streams[(size_t)sidx], ctx->ev1, 0));
    return GB200_OK;
}

// join the first nstreams pool streams back into the context stream; ev2 ends recorded on the last of them
static int fan_in(gb200_ctx* ctx, int nstreams) {
    for (int sidx = 0; sidx < nstreams; ++sidx) {
        CU(ctx, cudaEventRecord(ctx->ev2, ctx->pool_streams[(size_t)sidx]));
        CU(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev2, 0));
    }
    return GB200_OK;
}

// The sequence of every batch call, after its validation: lay the items out, stage the inputs, launch the items with rays
// round-robin on up to 32 pool streams, copy the outputs back and scatter them.  The call supplies
//   rays(b)                        item b's ray count (an empty item keeps its place in the layout but does not launch),
//   layout(b, in, out, P, io)      item b's inputs and outputs, as take() calls on the two Arenas,
//   setup(b, P, io) -> rc          the parameters of an item with rays, before its layout binds the device pointers,
//   launch(P, io, stream) -> err   its kernel,
//   scatter(b, P, io)              item b's outputs from the staging buffer to the caller, P and io pointing into it.
// With `queues`, every item gets its own ticket queue and step counters, reset before the launches and added to the stats.
// Set-up stays interleaved with the launches: a non-Kerr ISCO costs milliseconds of host time, during which the items
// already launched run.  stats: launches, rays and counters; kernel_ms = total_ms = the whole call.
template <class Rays, class Layout, class Setup, class Launch, class Scatter>
static int run_batch(gb200_ctx* ctx, int nbatch, bool queues, Rays&& rays, Layout&& layout, Setup&& setup, Launch&& launch, Scatter&& scatter) {
    { int rc_ = begin_call(ctx, ctx->stream); if (rc_) return rc_; }
    const int nstreams = nbatch < 32 ? nbatch : 32;
    int rc = ensure_streams(ctx, (size_t)nstreams); if (rc) return rc;
    GbParams S{}; // pointers of the passes over the staging buffer and of the items that do not launch
    GbDualIO Sio{};
    Arena size_in{nullptr}, size_out{nullptr};
    for (int b = 0; b < nbatch; ++b) layout(b, size_in, size_out, S, Sio);
    const size_t in_bytes = size_in.used, total = in_bytes + size_out.used;
    void* arena_v = nullptr;
    rc = pool_get(ctx, SL_BATCH, total + 256, &arena_v); if (rc) return rc;
    char* arena = (char*)arena_v;
    rc = ensure_stage(ctx, total); if (rc) return rc;
    char* stage = (char*)ctx->stage;
    unsigned long long* qs = nullptr;
    const size_t qbytes = queues ? sizeof(unsigned long long) * 4 * (size_t)nbatch : 0;
    if (queues) { void* qv = nullptr; rc = pool_get(ctx, SL_BATCH_QUEUE, qbytes, &qv); if (rc) return rc; qs = (unsigned long long*)qv; }
    Arena stage_in{stage, true}, stage_out{stage + in_bytes};
    for (int b = 0; b < nbatch; ++b) layout(b, stage_in, stage_out, S, Sio);
    CU(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    if (queues) CU(ctx, cudaMemsetAsync(qs, 0, qbytes, ctx->stream));
    if (in_bytes) CU(ctx, cudaMemcpyAsync(arena, stage, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    rc = fan_out(ctx, nstreams); if (rc) return rc;
    Arena dev_in{arena}, dev_out{arena + in_bytes};
    for (int b = 0; b < nbatch; ++b) {
        if (!rays(b)) { layout(b, dev_in, dev_out, S, Sio); continue; } // the item keeps its place, and its table may be shared
        GbParams P;
        GbDualIO io;
        memset(&io, 0, sizeof io);
        if ((rc = setup(b, P, io))) break;
        layout(b, dev_in, dev_out, P, io);
        if (queues) { P.queue = qs + 4 * (size_t)b; P.counters = P.queue + 1; }
        const cudaError_t e = launch(P, io, ctx->pool_streams[(size_t)(b % nstreams)]);
        if (e != cudaSuccess) { rc = fail(ctx, GB200_ERR_CUDA, "launch of batch item %d: %s", b, cudaGetErrorString(e)); break; }
        ctx->stats.launches += 1;
    }
    const int joined = fan_in(ctx, nstreams);
    if (rc) { // the items launched so far end before the error returns: the next call stages into the same arena
        if (!joined) cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    if (joined) return joined;
    std::vector<unsigned long long> c(qbytes / sizeof(unsigned long long));
    if (total > in_bytes) CU(ctx, cudaMemcpyAsync(stage + in_bytes, arena + in_bytes, total - in_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (queues) CU(ctx, cudaMemcpyAsync(c.data(), qs, qbytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaEventRecord(ctx->ev3, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    Arena host_in{stage}, host_out{stage + in_bytes};
    for (int b = 0; b < nbatch; ++b) {
        layout(b, host_in, host_out, S, Sio);
        if (rays(b)) scatter(b, S, Sio);
        ctx->stats.rays += rays(b);
    }
    float tot = 0;
    cudaEventElapsedTime(&tot, ctx->ev0, ctx->ev3);
    ctx->stats.kernel_ms = tot; ctx->stats.total_ms = tot;
    add_counters(ctx, c.data(), c.size() / 4);
    return GB200_OK;
}

// gb200_fp64_peak and gb200_fp64_issue_probe: launch(d, blocks, iters) runs blocks x 256 threads of 64 FMAs per iteration;
// the rate is the best of repetitions 1..3 (repetition 0 warms up)
template <class Launch> static int fp64_rate(gb200_ctx* ctx, Launch&& launch, double* tflops_out) {
    { int rc_ = begin_call(ctx, ctx->stream); if (rc_) return rc_; }
    void* d;
    int rc = pool_get(ctx, SL_SCRATCH, 64, &d); if (rc) return rc;
    const int blocks = ctx->sm_count * 8, iters = 20000;
    double best = 0;
    for (int rep = 0; rep < 4; ++rep) {
        CU(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        CU(ctx, launch((double*)d, blocks, iters));
        CU(ctx, cudaEventRecord(ctx->ev2, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev1, ctx->ev2);
        const double tf = 2.0 * 64.0 * (double)iters * 256.0 * (double)blocks / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    *tflops_out = best;
    return GB200_OK;
}

// ---------------------------------------------------------------- C ABI
extern "C" {

int gb200_version(void) { return GB200_VERSION; }

const char* gb200_last_error(gb200_ctx* ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }

int gb200_init(int device, gb200_ctx** out) {
    if (!out) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null out pointer");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, GB200_ERR_NO_DEVICE, "no CUDA device available (%s); libgradus_b200 has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "count = 0");
    if (device < 0 || device >= ndev) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "device %d out of range [0, %d)", device, ndev);
    cudaDeviceProp prop;
    CU(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(nullptr, GB200_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    gb200_ctx* ctx = new gb200_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    CU(nullptr, cudaSetDevice(device));
    CU(nullptr, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CU(nullptr, cudaEventCreate(&ctx->ev0)); CU(nullptr, cudaEventCreate(&ctx->ev1));
    CU(nullptr, cudaEventCreate(&ctx->ev2)); CU(nullptr, cudaEventCreate(&ctx->ev3));
    CU(nullptr, cudaEventCreateWithFlags(&ctx->inflight, cudaEventDisableTiming));
    CU(nullptr, cudaMalloc(&ctx->d_queue, 4 * sizeof(unsigned long long)));
    *out = ctx;
    return GB200_OK;
}

int gb200_set_cross_section(gb200_ctx* ctx, const double* rho, const double* height, int32_t n) {
    if (!ctx) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null context");
    if (n != 0 && (n < 2 || !rho || !height)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "cross-section table needs n >= 2 points");
    for (int i = 1; i < n; ++i) if (!(rho[i] > rho[i - 1])) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "cross-section radii must be strictly increasing");
    { int rc_ = begin_call(ctx, ctx->stream); if (rc_) return rc_; }
    CU(ctx, cudaStreamSynchronize(ctx->stream)); // nothing in flight may still read the old table
    if (ctx->d_cs) { cudaFree(ctx->d_cs); ctx->d_cs = nullptr; }
    ctx->cs_n = 0; ctx->cs_max = 0.0;
    if (n == 0) return GB200_OK;
    CU(ctx, cudaMalloc(&ctx->d_cs, sizeof(double) * 2 * (size_t)n));
    CU(ctx, cudaMemcpy(ctx->d_cs, rho, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice));
    CU(ctx, cudaMemcpy(ctx->d_cs + n, height, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice));
    ctx->cs_n = n;
    for (int i = 0; i < n; ++i) ctx->cs_max = std::max(ctx->cs_max, height[i]);
    return GB200_OK;
}

void gb200_destroy(gb200_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->d_cs) cudaFree(ctx->d_cs);
    for (auto& b : ctx->pool) if (b.p) cudaFree(b.p);
    if (ctx->d_queue) cudaFree(ctx->d_queue);
    for (auto st : ctx->pool_streams) cudaStreamDestroy(st);
    for (auto ev : ctx->chunk_events) cudaEventDestroy(ev);
    if (ctx->stage) cudaFreeHost(ctx->stage);
    if (ctx->inflight) cudaEventDestroy(ctx->inflight);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->ev2) cudaEventDestroy(ctx->ev2);
    if (ctx->ev3) cudaEventDestroy(ctx->ev3);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int gb200_get_stats(gb200_ctx* ctx, gb200_stats* out) {
    if (!ctx || !out) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "null argument");
    *out = ctx->stats;
    return GB200_OK;
}

int gb200_validate(const gb200_problem* p, const gb200_ic* ic) { return validate(nullptr, p, ic); }

int gb200_isco(int32_t metric_kind, const double* mp, double* out) {
    if (!mp || !out) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null argument");
    if (metric_kind == GB200_METRIC_KERR) { *out = kerr_isco_host(mp[0], mp[1]); return GB200_OK; }
    if (metric_kind == GB200_METRIC_MORRIS_THORNE)
        return fail(nullptr, GB200_ERR_UNSUPPORTED, "the Morris-Thorne wormhole has no circular-orbit energy minimum: no ISCO");
    if (metric_kind > GB200_METRIC_KERR && metric_kind < GB200_METRIC_COUNT) {
        int rc = generic_isco_host(metric_kind, mp, out);
        if (rc) return fail(nullptr, rc, "No boundaries for minimization could be determined. It is likely this configuration does not have an ISCO solution.");
        return GB200_OK;
    }
    return fail(nullptr, GB200_ERR_UNSUPPORTED, "metric kind %d", metric_kind);
}

int gb200_radiative_efficiency(int32_t metric_kind, const double* mp, double* out) {
    double r = 0;
    int rc = gb200_isco(metric_kind, mp, &r);
    if (rc) return rc;
    *out = 1.0 - circular_energy_host<double>(metric_kind, mp, r);
    return GB200_OK;
}

// gb200_trace and gb200_trace_target: `target` (r, theta, phi) non-null selects the closest-approach objective (the generic
// integrator with the distance condition in place of a geometry); `closest` then receives one distance per ray.
static int trace_common(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic, const gb200_range* rg, gb200_endpoints* out,
                        const double* target, double d_tol, double* closest) {
    if (!ctx) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null context");
    int rc = validate(ctx, p, ic); if (rc) return rc;
    rc = validate_range(ctx, ic, rg); if (rc) return rc;
    static const gb200_endpoints no_endpoints{};
    if (target) {
        if (p->geometry_kind != GB200_GEOMETRY_NONE) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "gb200_trace_target: the distance callback takes the geometry's place (geometry_kind must be NONE)");
        if (!(d_tol > 0) || !closest) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "gb200_trace_target needs d_tol > 0 and a closest[] array");
        if (!out) out = const_cast<gb200_endpoints*>(&no_endpoints);
    } else if (!out) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "null endpoints");
    { int rc_ = begin_call(ctx, ctx->stream); if (rc_) return rc_; }
    CU(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    GbParams P;
    fill_params(p, ic, rg, P);
    { int rcg_ = bind_geometry(ctx, P); if (rcg_) return rcg_; }
    rc = upload_ic_and_tables(ctx, ic, nullptr, nullptr, P); if (rc) return rc;
    const size_t n = (size_t)rg->count;
    void* d;
    if (target) { // to_cartesian(target), src/geometry/geometry.jl:13-16
        P.geometry_kind = GB200_GEOMETRY_TARGET_POINT;
        P.gp0 = target[0] * std::sin(target[1]) * std::cos(target[2]);
        P.gp1 = target[0] * std::sin(target[1]) * std::sin(target[2]);
        P.gp2 = target[0] * std::cos(target[1]);
        P.gtol = d_tol;
        rc = pool_get(ctx, SL_G, n * sizeof(double) + 8, &d); if (rc) return rc;
        P.o_closest = (double*)d;
    }
    endpoint_arrays(*out, P, [&](auto* h, auto*& f, int slot) {
        if (h && !rc && !(rc = pool_get(ctx, (size_t)slot, n * sizeof(*f) + 8, &d))) f = (decltype(h))d;
    });
    if (rc) return rc;
    // the endpoints of slots [s0, s0 + cnt) to the host
    auto copy_back = [&](int64_t s0, int64_t cnt, cudaStream_t copy) -> cudaError_t {
        cudaError_t e = cudaSuccess;
        endpoint_arrays(*out, P, [&](auto* h, auto* f, int) {
            if (e == cudaSuccess && h) e = cudaMemcpyAsync(h + s0, f + s0, (size_t)cnt * sizeof(*f), cudaMemcpyDeviceToHost, copy);
        });
        return e;
    };
    if (!target && pipeline_eligible(P, rg))
        return run_pipelined(ctx, rg, P, [&](GbParams& Pc, int64_t s0) { endpoint_arrays(*out, Pc, [&](auto*, auto*& f, int) { if (f) f += s0; }); },
                             copy_back);
    if (target) { // one ray per thread through the generic integrator; no ticket queue, no step counters
        CU(ctx, cudaMemsetAsync(ctx->d_queue, 0, 4 * sizeof(unsigned long long), ctx->stream));
        CU(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        CU(ctx, gb200_launch_target(P, ctx->stream));
        CU(ctx, cudaEventRecord(ctx->ev2, ctx->stream));
        ctx->stats.launches += n ? 1 : 0;
        if (n) CU(ctx, cudaMemcpyAsync(closest, P.o_closest, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    } else { rc = run_trace(ctx, P, ctx->stream, true); if (rc) return rc; }
    if (n) CU(ctx, copy_back(0, rg->count, ctx->stream));
    return finish_stats(ctx, rg->count);
}

int gb200_trace(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic, const gb200_range* rg, gb200_endpoints* out) {
    return trace_common(ctx, p, ic, rg, out, nullptr, 0.0, nullptr);
}

int gb200_trace_target(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic, const gb200_range* rg, const double* target, double d_tol,
                       gb200_endpoints* out, double* closest) {
    { int rc_ = reject_image_order(ctx, p, "gb200_trace_target"); if (rc_) return rc_; }
    if (!target) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "null target");
    return trace_common(ctx, p, ic, rg, out, target, d_tol, closest);
}

int gb200_trace_batch(gb200_ctx* ctx, int32_t nbatch, const gb200_problem* problems, const gb200_ic* ics,
                      const gb200_range* ranges, gb200_endpoints* outs) {
    if (!ctx) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null context");
    if (nbatch < 1 || !problems || !ics || !ranges || !outs) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bad batch arguments");
    for (int b = 0; b < nbatch; ++b) {
        int rc = validate(ctx, &problems[b], &ics[b]); if (rc) return rc;
        rc = validate_range(ctx, &ics[b], &ranges[b]); if (rc) return rc;
        if (ics[b].kind == GB200_IC_IMPACT_PARAMETERS) return fail(ctx, GB200_ERR_UNSUPPORTED, "impact-parameter lists are not batched; use gb200_trace / gb200_render");
    }
    for (int b = 0; b < nbatch; ++b) { int rc = check_table(ctx, problems[b].geometry_kind); if (rc) return rc; }
    int rc = run_batch(ctx, nbatch, true, [&](int b) { return ranges[b].count; },
        // inputs: the explicit ICs; outputs: the endpoint arrays the caller asked for
        [&](int b, Arena& in, Arena& out, GbParams& P, GbDualIO&) {
            if (ics[b].kind == GB200_IC_EXPLICIT)
                for (int k = 0; k < 4; ++k) { in.take(P.ex[k], ics[b].n, ics[b].x[k]); in.take(P.ev[k], ics[b].n, ics[b].v[k]); }
            endpoint_arrays(outs[b], P, [&](auto* h, auto*& f, int) { if (h) out.take(f, ranges[b].count); });
        },
        [&](int b, GbParams& P, GbDualIO&) {
            fill_params(&problems[b], &ics[b], &ranges[b], P);
            return bind_geometry(ctx, P);
        },
        [&](GbParams& P, GbDualIO&, cudaStream_t st) { int blocks = 0; return gb200_launch_trace(P, ctx->sm_count, st, &blocks); },
        [&](int b, GbParams& S, GbDualIO&) { // the staging buffer into the caller's SoA
            endpoint_arrays(outs[b], S, [&](auto* h, auto* f, int) { if (h) memcpy(h, f, (size_t)ranges[b].count * sizeof(*f)); });
        });
    if (rc) return rc;
    float dev = 0;
    cudaEventElapsedTime(&dev, ctx->ev1, ctx->ev2); // launches only (ev2: the end of the last pool stream), without the two staged copies
    ctx->stats.kernel_ms = dev;
    return GB200_OK;
}

int gb200_trace_path(gb200_ctx* ctx, const gb200_problem* p, const double* u0, int32_t cap, double* lambda, double* u,
                     int32_t* nrows, int32_t* status) {
    { int rc_ = reject_image_order(ctx, p, "gb200_trace_path"); if (rc_) return rc_; }
    if (!ctx) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null context");
    if (!p || !u0 || cap < 1 || !lambda || !u || !nrows || !status) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bad path arguments");
    gb200_ic ic{};
    ic.kind = GB200_IC_EXPLICIT; ic.n = 1;
    for (int k = 0; k < 4; ++k) { ic.x[k] = u0 + k; ic.v[k] = u0 + 4 + k; }
    int rc = validate(ctx, p, &ic); if (rc) return rc;
    { int rc_ = begin_call(ctx, ctx->stream); if (rc_) return rc_; }
    gb200_range rg{0, 1, 1};
    GbParams P;
    fill_params(p, &ic, &rg, P);
    { int rcg_ = bind_geometry(ctx, P); if (rcg_) return rcg_; }
    P.geometry_kind = GB200_GEOMETRY_NONE; // a bare geodesic: chart boundaries and lambda_max only
    P.callback_kind = GB200_CALLBACK_NONE;
    void *d_u0, *d_lam, *d_u, *d_meta;
    rc = pool_get(ctx, SL_EX0, 64, &d_u0); if (rc) return rc;
    rc = pool_get(ctx, SL_LAMBDA, sizeof(double) * (size_t)cap, &d_lam); if (rc) return rc;
    rc = pool_get(ctx, SL_X0, sizeof(double) * 8 * (size_t)cap, &d_u); if (rc) return rc;
    rc = pool_get(ctx, SL_SCRATCH, 64, &d_meta); if (rc) return rc;
    CU(ctx, cudaMemcpyAsync(d_u0, u0, 64, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, gb200_launch_path(P, (const double*)d_u0, cap, (double*)d_lam, (double*)d_u, (int*)d_meta, ctx->stream));
    ctx->stats.launches = 1;
    int meta[2] = {0, 0};
    CU(ctx, cudaMemcpyAsync(meta, d_meta, sizeof meta, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    const int nw = meta[0] < cap ? meta[0] : cap;
    CU(ctx, cudaMemcpy(lambda, d_lam, sizeof(double) * (size_t)nw, cudaMemcpyDeviceToHost));
    CU(ctx, cudaMemcpy(u, d_u, sizeof(double) * 8 * (size_t)nw, cudaMemcpyDeviceToHost));
    *nrows = meta[0];
    *status = meta[1];
    return GB200_OK;
}

int gb200_build_plunging_table(gb200_ctx* ctx, int32_t metric_kind, const double* mp, int32_t cap, double* r, double* ut, double* ur,
                         double* uphi, int32_t* n) {
    if (!ctx) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null context");
    if (!mp || cap < 2 || !r || !ut || !ur || !uphi || !n) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bad plunging-table arguments");
    double risco = 0;
    int rc = gb200_isco(metric_kind, mp, &risco);
    if (rc) return fail(ctx, rc, "no ISCO for this metric");
    // CircularOrbits.plunging_fourvelocity at the ISCO (circular-orbits.jl:129-150)
    double g[5], dr[5], dth[5];
    metric_jacobian_kind<double>(metric_kind, mp, risco, 1.0, 0.0, g, dr, dth);
    const double D = g[0] * g[3] - g[4] * g[4];
    const double gitt = g[3] / D, giphph = g[0] / D, gitph = -g[4] / D;
    const double Om = -(dr[4] - std::sqrt(dr[4] * dr[4] - dr[0] * dr[3])) / dr[3];
    const double A = -(Om * gitt - gitph), B = (Om * gitph - giphph);
    const double denom = B * B * gitt + 2.0 * A * B * gitph + A * A * giphph;
    const double dd = -(denom > 0 ? 1.0 : -1.0) * std::sqrt(1.0 / std::fabs(denom));
    const double ut_ = B * dd, uph_ = A * dd; // covariant u_t, u_phi
    const double E = -ut_, L = uph_;
    const double vt = gitt * ut_ + gitph * uph_, vph = gitph * ut_ + giphph * uph_;
    const double nom = gitt * E * E - 2.0 * gitph * E * L + giphph * L * L + 1.0;
    const double vr = -std::sqrt(std::fabs(nom / (-g[1])));
    gb200_problem p{};
    p.metric_kind = metric_kind;
    for (int k = 0; k < 8; ++k) p.metric_params[k] = mp[k];
    p.mu = 1.0; p.abstol = 1e-9; p.reltol = 1e-9; p.lambda_min = 0.0; p.lambda_max = 50000.0; p.gtol = 1e-2;
    const double q2 = metric_kind == GB200_METRIC_KERR_NEWMAN ? mp[2] * mp[2] : 0.0;
    const double rh = mp[0] + std::sqrt(mp[0] * mp[0] - mp[1] * mp[1] - q2);
    p.chart_inner = rh * 1.000001; p.chart_outer = 12000.0;
    const double u0[8] = {0.0, risco - 1e-8, M_PI / 2, 0.0, vt, vr, 0.0, vph};
    const int pathcap = 1 << 20;
    std::vector<double> lam((size_t)pathcap), u((size_t)pathcap * 8);
    int32_t rows = 0, status = 0;
    rc = gb200_trace_path(ctx, &p, u0, pathcap, lam.data(), u.data(), &rows, &status);
    if (rc) return rc;
    if (rows > pathcap) return fail(ctx, GB200_ERR_NOMEM, "plunging geodesic needs %d rows (> %d)", rows, pathcap);
    // PlungingInterpolation (orbit-solving.jl:99-135): sort by r, drop the innermost sample
    std::vector<int> idx((size_t)rows);
    for (int i = 0; i < rows; ++i) idx[(size_t)i] = i;
    std::stable_sort(idx.begin(), idx.end(), [&](int a_, int b_) { return u[(size_t)a_ * 8 + 1] < u[(size_t)b_ * 8 + 1]; });
    const int nt = rows - 1;
    if (nt > cap) return fail(ctx, GB200_ERR_NOMEM, "plunging table needs %d entries (cap %d)", nt, cap);
    for (int i = 0; i < nt; ++i) {
        const size_t s = (size_t)idx[(size_t)i + 1] * 8;
        r[i] = u[s + 1]; ut[i] = u[s + 4]; ur[i] = u[s + 5]; uphi[i] = u[s + 7];
    }
    *n = nt;
    return GB200_OK;
}

static int render_common(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic, const gb200_range* rg, const int32_t* pfs, int32_t npf,
                         const gb200_plunging_table* pl, double* const* images, bool device_out, cudaStream_t stream, int async) {
    { int rc_ = validate_crossings(ctx, p, pfs, npf); if (rc_) return rc_; }
    if (!ctx) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null context");
    int rc = validate(ctx, p, ic); if (rc) return rc;
    rc = validate_range(ctx, ic, rg); if (rc) return rc;
    if (!images) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "need 1..%d point functions", GB_MAX_PF);
    rc = validate_pfs(ctx, pfs, npf, images); if (rc) return rc;
    { int rc_ = begin_call(ctx, stream); if (rc_) return rc_; }
    CU(ctx, cudaEventRecord(ctx->ev0, stream));
    GbParams P;
    fill_params(p, ic, rg, P);
    { int rcg_ = bind_geometry(ctx, P); if (rcg_) return rcg_; }
    if (needs_isco(pfs, npf, false)) { rc = set_isco(ctx, p, P); if (rc) return rc; }
    rc = upload_ic_and_tables(ctx, ic, pl, nullptr, P); if (rc) return rc;
    const size_t n = (size_t)rg->count;
    P.npf = npf;
    for (int k = 0; k < npf; ++k) {
        P.pf[k] = pfs[k];
        if (device_out) P.o_img[k] = images[k];
        else { void* d; rc = pool_get(ctx, SL_IMG0 + k, n * sizeof(double) + 8, &d); if (rc) return rc; P.o_img[k] = (double*)d; }
    }
    if (!device_out && !async && pipeline_eligible(P, rg)) {
        const GbParams Pfull = P;
        return run_pipelined(ctx, rg, P,
            [&](GbParams& Pc, int64_t slot0) { for (int k = 0; k < npf; ++k) Pc.o_img[k] = Pfull.o_img[k] + slot0; },
            [&](int64_t slot0, int64_t cnt, cudaStream_t copy) -> cudaError_t {
                for (int k = 0; k < npf; ++k) {
                    cudaError_t e = cudaMemcpyAsync(images[k] + slot0, Pfull.o_img[k] + slot0, (size_t)cnt * sizeof(double), cudaMemcpyDeviceToHost, copy);
                    if (e != cudaSuccess) return e;
                }
                return cudaSuccess;
            });
    }
    rc = run_trace(ctx, P, stream, true); if (rc) return rc;
    if (!device_out)
        for (int k = 0; k < npf; ++k)
            if (n) CU(ctx, cudaMemcpyAsync(images[k], P.o_img[k], n * sizeof(double), cudaMemcpyDeviceToHost, stream));
    if (async) { ctx->stats.rays = rg->count; return end_async_call(ctx, stream); }
    return finish_stats(ctx, rg->count);
}

int gb200_render(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic, const gb200_range* rg, const int32_t* pfs, int32_t npf,
                 const gb200_plunging_table* pl, double* const* images) {
    return render_common(ctx, p, ic, rg, pfs, npf, pl, images, false, ctx ? ctx->stream : nullptr, 0);
}

int gb200_render_device(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic, const gb200_range* rg, const int32_t* pfs, int32_t npf,
                        const gb200_plunging_table* pl, double* const* d_images, void* cuda_stream, int async) {
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : (ctx ? ctx->stream : nullptr);
    return render_common(ctx, p, ic, rg, pfs, npf, pl, d_images, true, s, async);
}

int gb200_render_batch(gb200_ctx* ctx, int32_t nbatch, const gb200_problem* problems, const gb200_ic* ics, const gb200_range* ranges,
                       const int32_t* pfs, int32_t npf, const gb200_plunging_table* const* pls, double* const* images) {
    if (problems)
        for (int b = 0; b < nbatch; ++b) { int rc_ = validate_crossings(ctx, &problems[b], pfs, npf); if (rc_) return rc_; }
    if (!ctx) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null context");
    if (nbatch < 1 || !problems || !ics || !ranges || !pfs || !images) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bad batch arguments");
    int rc = validate_pfs(ctx, pfs, npf, nullptr); if (rc) return rc; // the images are checked per item: empty items need none
    for (int b = 0; b < nbatch; ++b) {
        rc = validate(ctx, &problems[b], &ics[b]); if (rc) return rc;
        rc = validate_range(ctx, &ics[b], &ranges[b]); if (rc) return rc;
        if (ics[b].kind == GB200_IC_EXPLICIT) return fail(ctx, GB200_ERR_UNSUPPORTED, "explicit initial conditions are batched by gb200_trace_batch");
        for (int k = 0; k < npf; ++k) if (ranges[b].count && !images[(size_t)b * npf + k]) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "null image pointer");
    }
    for (int b = 0; b < nbatch; ++b) if (ranges[b].count) { rc = check_table(ctx, problems[b].geometry_kind); if (rc) return rc; }
    const bool want_isco = needs_isco(pfs, npf, false);
    return run_batch(ctx, nbatch, true, [&](int b) { return ranges[b].count; },
        // inputs: the impact-parameter lists (+ heights) and the plunging table; outputs: the images
        [&](int b, Arena& in, Arena& out, GbParams& P, GbDualIO&) {
            if (ics[b].kind == GB200_IC_IMPACT_PARAMETERS)
                for (int k = 0; k < 3; ++k) if (ics[b].x[k]) in.take(P.ex[k], ics[b].n, ics[b].x[k]);
            place_plunging(in, pls, b, P);
            for (int k = 0; k < npf; ++k) out.take(P.o_img[k], ranges[b].count);
        },
        [&](int b, GbParams& P, GbDualIO&) {
            fill_params(&problems[b], &ics[b], &ranges[b], P);
            int rc_ = bind_geometry(ctx, P); if (rc_) return rc_;
            if (want_isco) { rc_ = set_isco(ctx, &problems[b], P); if (rc_) return rc_; }
            P.npf = npf;
            for (int k = 0; k < npf; ++k) P.pf[k] = pfs[k];
            return GB200_OK;
        },
        [&](GbParams& P, GbDualIO&, cudaStream_t st) { int blocks = 0; return gb200_launch_trace(P, ctx->sm_count, st, &blocks); },
        [&](int b, GbParams& S, GbDualIO&) {
            for (int k = 0; k < npf; ++k) memcpy(images[(size_t)b * npf + k], S.o_img[k], 8 * (size_t)ranges[b].count);
        });
}

// ---------------------------------------------------------------- forward-mode traces (gb200_dual.cu)
int gb200_trace_dual_batch(gb200_ctx* ctx, int32_t nbatch, const gb200_problem* problems, const gb200_dual_ic* ics, int32_t norm_mode,
                           const gb200_plunging_table* const* pls, gb200_dual_out* outs) {
    if (problems)
        for (int b = 0; b < nbatch; ++b) { int rc_ = reject_image_order(ctx, &problems[b], "gb200_trace_dual"); if (rc_) return rc_; }
    if (!ctx) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null context");
    if (nbatch < 1 || !problems || !ics || !outs) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bad batch arguments");
    if (norm_mode != GB200_DUAL_NORM_WITH_PARTIALS && norm_mode != GB200_DUAL_NORM_VALUES_ONLY) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bad norm_mode");
    std::vector<gb200_ic> fake((size_t)nbatch);
    for (int b = 0; b < nbatch; ++b) {
        const gb200_dual_ic& d = ics[b];
        if (d.n < 0 || (d.npartials != 1 && d.npartials != 2)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "dual IC needs n >= 0 and 1 or 2 partials");
        if (d.n > 0 && (!d.alpha || !d.beta || !d.dalpha || !d.dbeta)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "dual IC needs alpha, beta and their partials");
        gb200_ic& f = fake[(size_t)b];
        memset(&f, 0, sizeof f);
        f.kind = GB200_IC_IMPACT_PARAMETERS; f.n = d.n > 0 ? d.n : 1;
        f.x[0] = d.alpha ? d.alpha : (const double*)&f; f.x[1] = d.beta ? d.beta : (const double*)&f;
        int rc = validate(ctx, &problems[b], &f); if (rc) return rc;
        if (d.height && problems[b].geometry_kind != GB200_GEOMETRY_DATUM_PLANE) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "per-ray heights need GB200_GEOMETRY_DATUM_PLANE");
    }
    for (int b = 0; b < nbatch; ++b) {
        if (!ics[b].n) continue;
        int rc = check_table(ctx, problems[b].geometry_kind); if (rc) return rc;
        if (outs[b].dg && !outs[b].g) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "dg needs g");
    }
    return run_batch(ctx, nbatch, false, [&](int b) { return ics[b].n; },
        // inputs: the seeded impact parameters (+ heights) and the plunging table; outputs: the arrays the caller asked for
        [&](int b, Arena& in, Arena& out, GbParams& P, GbDualIO& io) {
            const gb200_dual_ic& d = ics[b];
            in.take(io.alpha, d.n, d.alpha); in.take(io.beta, d.n, d.beta);
            in.take(io.dalpha, d.n * d.npartials, d.dalpha); in.take(io.dbeta, d.n * d.npartials, d.dbeta);
            if (d.height) in.take(io.height, d.n, d.height);
            place_plunging(in, pls, b, P);
            dual_arrays(outs[b], io, d.n, d.npartials, [&](auto* h, auto*& f, int64_t n) { if (h) out.take(f, n); });
        },
        [&](int b, GbParams& P, GbDualIO& io) {
            const gb200_range rg{0, ics[b].n, 1, 1};
            fill_params(&problems[b], &fake[(size_t)b], &rg, P);
            int rc_ = bind_geometry(ctx, P); if (rc_) return rc_;
            if (outs[b].g) { rc_ = set_isco(ctx, &problems[b], P); if (rc_) return rc_; }
            io.n = ics[b].n; io.npartials = ics[b].npartials; io.norm_partials = (norm_mode == GB200_DUAL_NORM_WITH_PARTIALS) ? 1 : 0;
            return GB200_OK;
        },
        [&](GbParams& P, GbDualIO& io, cudaStream_t st) { return gb200_launch_dual(P, io, st); },
        [&](int b, GbParams&, GbDualIO& Sio) {
            dual_arrays(outs[b], Sio, ics[b].n, ics[b].npartials, [&](auto* h, auto* f, int64_t n) { if (h) memcpy(h, f, (size_t)n * sizeof(*f)); });
        });
}

int gb200_trace_dual(gb200_ctx* ctx, const gb200_problem* p, const gb200_dual_ic* ic, int32_t norm_mode,
                     const gb200_plunging_table* plunging, gb200_dual_out* out) {
    { int rc_ = reject_image_order(ctx, p, "gb200_trace_dual"); if (rc_) return rc_; }
    if (!p || !ic || !out) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "null argument");
    const gb200_plunging_table* pls[1] = {plunging};
    return gb200_trace_dual_batch(ctx, 1, p, ic, norm_mode, pls, out);
}

// the binned line profile to the caller: flux ./ sum(flux) (line-profiles.jl:197), or the raw sums for a multi-rank caller
static void normalise_flux(const std::vector<double>& h, const gb200_lineprofile_opts* opts, double* flux) {
    double tot = 0;
    for (double v : h) tot += v;
    for (size_t b = 0; b < h.size(); ++b) flux[b] = opts->normalise ? h[b] / tot : h[b];
}

static int lineprofile_common(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic, const gb200_range* rg, const gb200_emissivity* em,
                              const gb200_plunging_table* pl, const double* bins, int32_t nbins, const gb200_lineprofile_opts* opts,
                              double* flux, bool device_out, cudaStream_t stream, int async) {
    if (!ctx) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null context");
    int rc = validate(ctx, p, ic); if (rc) return rc;
    rc = validate_range(ctx, ic, rg); if (rc) return rc;
    if (!em || !bins || !opts || !flux || nbins < 1 || nbins > 8192) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bad line-profile arguments (1 <= nbins <= 8192)");
    for (int b = 1; b < nbins; ++b) if (!(bins[b] > bins[b - 1])) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bins must be strictly increasing");
    { int rc_ = begin_call(ctx, stream); if (rc_) return rc_; }
    CU(ctx, cudaEventRecord(ctx->ev0, stream));
    GbParams P;
    fill_params(p, ic, rg, P);
    { int rcg_ = bind_geometry(ctx, P); if (rcg_) return rcg_; }
    rc = set_isco(ctx, p, P); if (rc) return rc;
    rc = upload_ic_and_tables(ctx, ic, pl, em, P); if (rc) return rc;
    P.min_re = opts->min_re; P.max_re = opts->max_re;
    const size_t n = (size_t)rg->count;
    void* d;
    const void* dbins;
    rc = upload(ctx, SL_BINS, bins, sizeof(double) * nbins, &dbins); if (rc) return rc;
    double* dflux = flux;
    if (!device_out) { rc = pool_get(ctx, SL_FLUX, sizeof(double) * nbins, &d); if (rc) return rc; dflux = (double*)d; }
    // Fused path: the histogram is accumulated inside the trace kernel, per CTA in shared memory, as 128-bit fixed point
    // (gb_hist_add).  The scale is a power of two chosen from a generous bound on sum f = sum eps(rho) g^3 area
    // (g <= 1e3), so f * scale is exact and the bins hold the exact sum of the contributions, whatever the order.
    double eps_max = 0.0;
    if (em->kind == GB200_EMISSIVITY_POWERLAW) eps_max = std::max(std::pow(opts->min_re, -em->index), std::pow(opts->max_re, -em->index));
    else for (int k = 0; k < em->n; ++k) eps_max = std::max(eps_max, std::fabs(em->eps[k]));
    const double area_max = (ic->kind == GB200_IC_POLAR_PLANE) ? ic->hi0 * ic->hi0 : 1.0;
    const double bound = (double)(n > 0 ? n : 1) * eps_max * 1e9 * area_max;
    const bool fused = nbins <= 512 && std::isfinite(bound) && bound > 0.0 && !getenv("GB200_HIST_TWO_PASS");
    if (fused) {
        rc = pool_get(ctx, SL_PARTIAL, sizeof(unsigned long long) * 2 * (size_t)nbins, &d); if (rc) return rc;
        P.lp_acc = (unsigned long long*)d;
        P.lp_bins = (const double*)dbins; P.lp_nbins = nbins; P.lp_right_closed = opts->bin_right_closed;
        P.lp_scale = std::exp2(std::floor(120.0 - std::log2(bound)));
        CU(ctx, cudaMemsetAsync(P.lp_acc, 0, sizeof(unsigned long long) * 2 * (size_t)nbins, stream));
        rc = run_trace(ctx, P, stream, true); if (rc) return rc;
        CU(ctx, gb200_launch_hist128_finish(P.lp_acc, nbins, P.lp_scale, dflux, stream));
        ctx->stats.launches += 1;
    } else { // more bins than fit beside the stage data in shared memory: (g, f) per ray through HBM, then the binning kernels
        rc = pool_get(ctx, SL_G, n * sizeof(double) + 8, &d); if (rc) return rc; P.o_g = (double*)d;
        rc = pool_get(ctx, SL_F, n * sizeof(double) + 8, &d); if (rc) return rc; P.o_f = (double*)d;
        const int nblocks = ctx->sm_count * 4;
        rc = pool_get(ctx, SL_PARTIAL, sizeof(double) * (size_t)nblocks * nbins, &d); if (rc) return rc;
        double* dpartial = (double*)d;
        rc = run_trace(ctx, P, stream, true); if (rc) return rc;
        CU(ctx, gb200_launch_hist(P.o_g, P.o_f, rg->count, (const double*)dbins, nbins, opts->bin_right_closed, dpartial, nblocks, dflux, stream));
        ctx->stats.launches += 2;
    }
    if (!device_out) {
        std::vector<double> h((size_t)nbins);
        CU(ctx, cudaMemcpyAsync(h.data(), dflux, sizeof(double) * nbins, cudaMemcpyDeviceToHost, stream));
        CU(ctx, cudaStreamSynchronize(stream));
        normalise_flux(h, opts, flux);
    }
    if (async) { ctx->stats.rays = rg->count; return end_async_call(ctx, stream); }
    return finish_stats(ctx, rg->count);
}

int gb200_lineprofile(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic, const gb200_range* rg, const gb200_emissivity* em,
                      const gb200_plunging_table* pl, const double* bins, int32_t nbins, const gb200_lineprofile_opts* opts, double* flux_out) {
    return lineprofile_common(ctx, p, ic, rg, em, pl, bins, nbins, opts, flux_out, false, ctx ? ctx->stream : nullptr, 0);
}

int gb200_lineprofile_device(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic, const gb200_range* rg, const gb200_emissivity* em,
                             const gb200_plunging_table* pl, const double* bins, int32_t nbins, const gb200_lineprofile_opts* opts,
                             double* d_flux, void* cuda_stream, int async) {
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : (ctx ? ctx->stream : nullptr);
    return lineprofile_common(ctx, p, ic, rg, em, pl, bins, nbins, opts, d_flux, true, s, async);
}

// ---------------------------------------------------------------- single-process multi-GPU (what a Julia caller uses)
// NCCL is opened at run time (dlopen("libnccl.so.2")): a process that already holds an NCCL (PyTorch bundles one) shares it,
// and a single-GPU caller needs none at all.
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool load(std::string* why) {
        if (handle) return true;
        for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
            handle = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (handle) break;
        }
        if (!handle) { *why = dlerror() ? dlerror() : "libnccl.so.2 not found"; return false; }
        CommInitAll = (decltype(CommInitAll))dlsym(handle, "ncclCommInitAll");
        CommDestroy = (decltype(CommDestroy))dlsym(handle, "ncclCommDestroy");
        AllReduce = (decltype(AllReduce))dlsym(handle, "ncclAllReduce");
        GroupStart = (decltype(GroupStart))dlsym(handle, "ncclGroupStart");
        GroupEnd = (decltype(GroupEnd))dlsym(handle, "ncclGroupEnd");
        GetErrorString = (decltype(GetErrorString))dlsym(handle, "ncclGetErrorString");
        if (!CommInitAll || !CommDestroy || !AllReduce || !GroupStart || !GroupEnd || !GetErrorString) { *why = "libnccl lacks a required symbol"; return false; }
        return true;
    }
};
static NcclApi g_nccl;
static std::mutex g_nccl_mutex;

struct gb200_comm {
    std::vector<gb200_ctx*> ctx;
    std::vector<ncclComm_t> nccl; // empty when ndev == 1 and NCCL is unavailable
};
#define NC(call)                                                                                                         \
    do {                                                                                                                 \
        ncclResult_t r__ = (call);                                                                                       \
        if (r__ != ncclSuccess) return fail(nullptr, GB200_ERR_CUDA, "%s: %s", #call, g_nccl.GetErrorString(r__));       \
    } while (0)

// One in-place all-reduce of a device buffer
struct NcclReduce {
    void* buf;
    size_t count;
    ncclDataType_t type;
    ncclRedOp_t op;
};

// ops[d]: the all-reduces of device d, enqueued on its context's stream; all of them run as one NCCL group.  Nothing to do
// on one device.
static int all_reduce(const std::vector<gb200_ctx*>& ctxs, const ncclComm_t* nccl, const std::vector<std::vector<NcclReduce>>& ops) {
    if (ctxs.size() < 2) return GB200_OK;
    NC(g_nccl.GroupStart());
    for (size_t d = 0; d < ctxs.size(); ++d)
        for (const NcclReduce& o : ops[d]) {
            ncclResult_t r = g_nccl.AllReduce(o.buf, o.buf, o.count, o.type, o.op, nccl[d], ctxs[d]->stream);
            if (r != ncclSuccess) { g_nccl.GroupEnd(); return fail(nullptr, GB200_ERR_CUDA, "ncclAllReduce: %s", g_nccl.GetErrorString(r)); }
        }
    NC(g_nccl.GroupEnd());
    return GB200_OK;
}

// rank d's share of the rays: whole strips of four image columns / theta-rows, strip d, d + n, ... (DESIGN.md section 6)
static gb200_range shard_range(const gb200_ic* ic, int d, int n) {
    const int64_t strip = GB_TILE_C * strip_height(ic);
    if (n == 1) return gb200_range{0, ic->n, 1, 1};
    if (strip > 0 && ic->n % strip == 0) {
        const int64_t nstrips = ic->n / strip;
        const int64_t mine = nstrips > d ? (nstrips - d + n - 1) / n : 0;
        return gb200_range{(int64_t)d * strip, mine * strip, n, strip};
    }
    return gb200_range{d, ic->n > d ? (ic->n - d + n - 1) / n : 0, n, 1};
}

int gb200_comm_init(const int32_t* devices, int32_t ndev, gb200_comm** out) {
    if (!devices || ndev < 1 || !out) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "bad communicator arguments");
    *out = nullptr;
    for (int a = 0; a < ndev; ++a)
        for (int b = a + 1; b < ndev; ++b)
            if (devices[a] == devices[b]) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "device %d listed twice", devices[a]);
    gb200_comm* c = new gb200_comm();
    for (int d = 0; d < ndev; ++d) {
        gb200_ctx* ctx = nullptr;
        int rc = gb200_init(devices[d], &ctx);
        if (rc) { gb200_comm_destroy(c); return rc; }
        c->ctx.push_back(ctx);
    }
    std::string why;
    bool have;
    { std::lock_guard<std::mutex> lock(g_nccl_mutex); have = g_nccl.load(&why); }
    if (!have) {
        if (ndev > 1) { gb200_comm_destroy(c); return fail(nullptr, GB200_ERR_UNSUPPORTED, "several devices need NCCL: %s", why.c_str()); }
    } else {
        c->nccl.resize((size_t)ndev);
        std::vector<int> devs(devices, devices + ndev);
        ncclResult_t r = g_nccl.CommInitAll(c->nccl.data(), ndev, devs.data());
        if (r != ncclSuccess) { c->nccl.clear(); gb200_comm_destroy(c); return fail(nullptr, GB200_ERR_CUDA, "ncclCommInitAll: %s", g_nccl.GetErrorString(r)); }
    }
    *out = c;
    return GB200_OK;
}

void gb200_comm_destroy(gb200_comm* c) {
    if (!c) return;
    for (size_t d = 0; d < c->ctx.size(); ++d) {
        if (d < c->nccl.size() && c->nccl[d]) g_nccl.CommDestroy(c->nccl[d]);
        gb200_destroy(c->ctx[d]);
    }
    delete c;
}

int gb200_comm_size(gb200_comm* c) { return c ? (int)c->ctx.size() : 0; }
gb200_ctx* gb200_comm_context(gb200_comm* c, int32_t i) { return (c && i >= 0 && i < (int)c->ctx.size()) ? c->ctx[(size_t)i] : nullptr; }

int gb200_comm_lineprofile(gb200_comm* c, const gb200_problem* p, const gb200_ic* ic, const gb200_emissivity* em, const gb200_plunging_table* pl,
                           const double* bins, int32_t nbins, const gb200_lineprofile_opts* opts, double* flux_out) {
    if (!c || !ic || !opts || !flux_out) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null argument");
    const int n = (int)c->ctx.size();
    // every device traces its strips and bins them into its own raw histogram (asynchronous launches, one host thread) ...
    std::vector<std::vector<NcclReduce>> sums((size_t)n);
    for (int d = 0; d < n; ++d) {
        gb200_ctx* ctx = c->ctx[(size_t)d];
        gb200_range rg = shard_range(ic, d, n);
        void* flux = nullptr;
        CU(ctx, cudaSetDevice(ctx->device));
        int rc = pool_get(ctx, SL_FLUX, sizeof(double) * (size_t)nbins, &flux);
        if (!rc) rc = lineprofile_common(ctx, p, ic, &rg, em, pl, bins, nbins, opts, (double*)flux, true, ctx->stream, 1);
        if (rc) return fail(nullptr, rc, "device %d: %s", ctx->device, ctx->err.c_str());
        sums[(size_t)d] = {{flux, (size_t)nbins, ncclDouble, ncclSum}};
    }
    // ... one all-reduce over NVLink sums them in place on every device's own stream ...
    { int rc_ = all_reduce(c->ctx, c->nccl.data(), sums); if (rc_) return rc_; }
    // ... and device 0 hands the sum to the host, which normalises it (flux ./ sum(flux), line-profiles.jl:197)
    std::vector<double> h((size_t)nbins);
    CU(c->ctx[0], cudaSetDevice(c->ctx[0]->device));
    CU(c->ctx[0], cudaMemcpyAsync(h.data(), sums[0][0].buf, sizeof(double) * (size_t)nbins, cudaMemcpyDeviceToHost, c->ctx[0]->stream));
    for (int d = 0; d < n; ++d) {
        CU(c->ctx[(size_t)d], cudaSetDevice(c->ctx[(size_t)d]->device));
        CU(c->ctx[(size_t)d], cudaStreamSynchronize(c->ctx[(size_t)d]->stream));
    }
    normalise_flux(h, opts, flux_out);
    return GB200_OK;
}

int gb200_comm_render(gb200_comm* c, const gb200_problem* p, const gb200_ic* ic, const int32_t* pfs, int32_t npf,
                      const gb200_plunging_table* pl, double* const* images) {
    if (!c || !ic || !pfs || !images || npf < 1 || npf > GB_MAX_PF) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "bad render arguments");
    const int n = (int)c->ctx.size();
    const int K = 4; // chunks per device: a chunk's images travel to the host while the next chunks compute
    std::vector<gb200_range> rgs((size_t)n);
    std::vector<std::vector<double*>> dimg((size_t)n);
    std::vector<int> nch((size_t)n, 0); // chunks of device d: their kernels end at chunk_events[ch], their copies at [K + ch]
    std::vector<int64_t> per((size_t)n, 0);
    // all launches first (asynchronous, one host thread): the devices compute concurrently
    for (int d = 0; d < n; ++d) {
        gb200_ctx* ctx = c->ctx[(size_t)d];
        gb200_range& rg = rgs[(size_t)d];
        rg = shard_range(ic, d, n);
        if (rg.block < 1) rg.block = 1;
        CU(ctx, cudaSetDevice(ctx->device));
        { int rc = ensure_streams(ctx, 2); if (!rc) rc = ensure_events(ctx, 2 * K); if (rc) return rc; }
        dimg[(size_t)d].resize((size_t)npf);
        for (int k = 0; k < npf; ++k) {
            void* dv = nullptr;
            int rc = pool_get(ctx, SL_IMG0 + k, sizeof(double) * (size_t)rg.count + 8, &dv);
            if (rc) return fail(nullptr, rc, "device %d: %s", ctx->device, ctx->err.c_str());
            dimg[(size_t)d][(size_t)k] = (double*)dv;
        }
        if (rg.count == 0) continue;
        const int64_t nblk = rg.count / rg.block; // strips (or single rays in the fallback decomposition)
        const int chunks = nblk >= 2 * K ? K : 1;
        per[(size_t)d] = ((nblk + chunks - 1) / chunks) * rg.block;
        for (int64_t s0 = 0; s0 < rg.count; s0 += per[(size_t)d]) {
            gb200_range sub{rg.first + (s0 / rg.block) * rg.stride * rg.block, std::min(per[(size_t)d], rg.count - s0), rg.stride, rg.block};
            double* sub_img[GB_MAX_PF];
            for (int k = 0; k < npf; ++k) sub_img[k] = dimg[(size_t)d][(size_t)k] + s0;
            int rc = render_common(ctx, p, ic, &sub, pfs, npf, pl, sub_img, true, ctx->stream, 1);
            if (rc) return fail(nullptr, rc, "device %d: %s", ctx->device, ctx->err.c_str());
            CU(ctx, cudaEventRecord(ctx->chunk_events[(size_t)nch[(size_t)d]++], ctx->stream));
        }
    }
    // Results travel chunk by chunk: a contiguous copy into the device's pinned staging buffer on its copy stream (truly
    // asynchronous, every device on its own PCIe link), then one host thread per device scatters the chunk's strips into
    // the caller's (pageable) images -- strip b of a device sits at ray first + b * stride * block.  A strided copy
    // straight into pageable memory is staged by the driver on the calling thread and serialises the devices (measured:
    // 8 GPUs 15.1 ms for the 2048 x 2048 render whose kernels take 5.3 ms).
    for (int d = 0; d < n; ++d) {
        gb200_ctx* ctx = c->ctx[(size_t)d];
        const gb200_range& rg = rgs[(size_t)d];
        if (rg.count == 0) continue;
        CU(ctx, cudaSetDevice(ctx->device));
        int rc = ensure_stage(ctx, sizeof(double) * (size_t)rg.count * (size_t)npf); if (rc) return rc;
    }
    for (int ch = 0; ch < K; ++ch)
        for (int d = 0; d < n; ++d) {
            if (ch >= nch[(size_t)d]) continue;
            gb200_ctx* ctx = c->ctx[(size_t)d];
            const gb200_range& rg = rgs[(size_t)d];
            const int64_t s0 = (int64_t)ch * per[(size_t)d], cnt = std::min(per[(size_t)d], rg.count - s0);
            CU(ctx, cudaSetDevice(ctx->device));
            cudaStream_t copy = ctx->pool_streams[1];
            CU(ctx, cudaStreamWaitEvent(copy, ctx->chunk_events[(size_t)ch], 0));
            for (int k = 0; k < npf; ++k)
                CU(ctx, cudaMemcpyAsync((double*)ctx->stage + (size_t)k * (size_t)rg.count + s0, dimg[(size_t)d][(size_t)k] + s0,
                                        sizeof(double) * (size_t)cnt, cudaMemcpyDeviceToHost, copy));
            CU(ctx, cudaEventRecord(ctx->chunk_events[(size_t)(K + ch)], copy));
        }
    std::vector<cudaError_t> terr((size_t)n, cudaSuccess);
    std::vector<std::thread> workers;
    for (int d = 0; d < n; ++d) {
        if (!nch[(size_t)d]) continue;
        workers.emplace_back([&, d]() {
            gb200_ctx* ctx = c->ctx[(size_t)d];
            const gb200_range& rg = rgs[(size_t)d];
            const size_t blk = (size_t)rg.block;
            for (int ch = 0; ch < nch[(size_t)d]; ++ch) {
                const cudaError_t e = cudaEventSynchronize(ctx->chunk_events[(size_t)(K + ch)]);
                if (e != cudaSuccess) { terr[(size_t)d] = e; return; }
                const int64_t s0 = (int64_t)ch * per[(size_t)d], cnt = std::min(per[(size_t)d], rg.count - s0);
                for (int k = 0; k < npf; ++k) {
                    const double* src = (const double*)ctx->stage + (size_t)k * (size_t)rg.count + s0;
                    double* dst = images[k] + rg.first + (s0 / rg.block) * rg.stride * rg.block;
                    if (rg.stride == 1) memcpy(dst, src, sizeof(double) * (size_t)cnt);
                    else
                        for (int64_t b_ = 0; b_ < cnt / rg.block; ++b_)
                            memcpy(dst + (size_t)b_ * blk * (size_t)rg.stride, src + (size_t)b_ * blk, sizeof(double) * blk);
                }
            }
        });
    }
    for (auto& w : workers) w.join();
    for (int d = 0; d < n; ++d) {
        gb200_ctx* ctx = c->ctx[(size_t)d];
        if (terr[(size_t)d] != cudaSuccess) return fail(nullptr, GB200_ERR_CUDA, "device %d: %s", ctx->device, cudaGetErrorString(terr[(size_t)d]));
        CU(ctx, cudaSetDevice(ctx->device));
        if (ctx->pool_streams.size() >= 2) CU(ctx, cudaStreamSynchronize(ctx->pool_streams[1]));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return GB200_OK;
}

// ---------------------------------------------------------------- binned lag-energy transfer function
static int validate_lims(gb200_ctx* ctx, const double* lims, const char* axis) {
    if (std::isnan(lims[0]) && std::isnan(lims[1])) return GB200_OK; // automatic: min / max over the hits
    if (!std::isfinite(lims[0]) || !std::isfinite(lims[1]) || !(lims[0] < lims[1]))
        return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "%s limits must be finite with lo < hi, or both NaN (got %g, %g)", axis, lims[0], lims[1]);
    return GB200_OK;
}

static int validate_ascending(gb200_ctx* ctx, const double* r, int32_t n, const char* what) {
    if (n < 2 || !r) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "%s needs n >= 2 radii", what);
    for (int k = 1; k < n; ++k)
        if (!(r[k] > r[k - 1])) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "%s radii must be strictly ascending (index %d)", what, k);
    return GB200_OK;
}

// the emissivity of a gb200_disc_profile and, when `time`, its arrival-time table
static int validate_disc_profile(gb200_ctx* ctx, const gb200_disc_profile* pr, bool time) {
    const gb200_emissivity& em = pr->emissivity;
    int rc;
    if (em.kind == GB200_EMISSIVITY_POWERLAW) {
        if (!std::isfinite(em.index)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "emissivity index must be finite");
    } else if (em.kind == GB200_EMISSIVITY_TABLE) {
        rc = validate_ascending(ctx, em.r, em.n, "emissivity table"); if (rc) return rc;
        if (!em.eps) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "emissivity table without values");
    } else return fail(ctx, GB200_ERR_UNSUPPORTED, "emissivity kind %d", em.kind);
    if (!time) return GB200_OK;
    if (pr->time_kind != GB200_PROFILE_TIME_NAN_LINEAR && pr->time_kind != GB200_PROFILE_TIME_LINEAR)
        return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "profile time kind %d", pr->time_kind);
    rc = validate_ascending(ctx, pr->r, pr->n, "arrival-time profile"); if (rc) return rc;
    if (!pr->t) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "arrival-time profile without times");
    return GB200_OK;
}

// Everything that can be rejected without tracing, for every device, before the first launch.
static int validate_lagtransfer(const std::vector<gb200_ctx*>& ctxs, const gb200_problem* p, const gb200_ic* ic, const gb200_disc_profile* pr,
                                const gb200_lagtransfer_opts* o, const double* time_edges, const double* energy_edges, const double* tf, const int64_t* hits) {
    gb200_ctx* ctx = ctxs[0];
    int rc = validate(ctx, p, ic); if (rc) return rc;
    if (ic->kind != GB200_IC_POLAR_PLANE)
        return fail(ctx, GB200_ERR_UNSUPPORTED, "the lag transfer function needs a PolarPlane: its r^2 area weight is defined only there");
    if (!pr || !o || !time_edges || !energy_edges || !tf || !hits) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "null argument");
    if (o->N_E < 2 || o->N_t < 2 || (int64_t)o->N_E * o->N_t > (1 << 26))
        return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "need N_E, N_t >= 2 and N_E * N_t <= 2^26 (got %d x %d)", o->N_E, o->N_t);
    if (!std::isfinite(o->E0) || !(o->E0 > 0)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "E0 must be positive and finite (got %g)", o->E0);
    if (!std::isfinite(o->t0)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "t0 must be finite");
    rc = validate_lims(ctx, o->energy_lims, "energy"); if (rc) return rc;
    rc = validate_lims(ctx, o->time_lims, "time"); if (rc) return rc;
    rc = validate_disc_profile(ctx, pr, true); if (rc) return rc;
    // what render_common would only find after it has started on the first device
    double r_isco;
    if (gb200_isco(p->metric_kind, p->metric_params, &r_isco)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "no ISCO found for this metric (is it a naked singularity?)");
    for (gb200_ctx* c : ctxs)
        if (p->geometry_kind == GB200_GEOMETRY_THICK_TABLE && c->cs_n < 2)
            return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "GB200_GEOMETRY_THICK_TABLE needs a table on device %d: call gb200_set_cross_section first", c->device);
    return GB200_OK;
}

// gb200_lagtransfer over the devices of `ctxs` (nccl: one communicator per device when there are several).  Every device
// traces its strips and forms its samples; the scalars (limits, hit count, max |f|) are all-reduced; every device bins into
// integer cells with the same edges and scale; the cells are all-reduced and device 0 finishes and copies the result.
static int lagtransfer_run(const std::vector<gb200_ctx*>& ctxs, const ncclComm_t* nccl, const gb200_problem* p, const gb200_ic* ic,
                           const gb200_disc_profile* pr, const gb200_plunging_table* pl, const gb200_lagtransfer_opts* o,
                           double* time_edges, double* energy_edges, double* tf, int64_t* hits) {
    const int n = (int)ctxs.size();
    for (gb200_ctx* c : ctxs) c->stats = gb200_stats{};
    int rc = validate_lagtransfer(ctxs, p, ic, pr, o, time_edges, energy_edges, tf, hits); if (rc) return rc;
    static const int32_t pfs[4] = {GB200_PF_STATUS, GB200_PF_REDSHIFT, GB200_PF_DISC_RADIUS, GB200_PF_COORDINATE_TIME}; // lagtransfer's
    const GbLagLimits L{{o->energy_lims[0], o->energy_lims[1]}, {o->time_lims[0], o->time_lims[1]}, o->N_E, o->N_t};
    const int ncell = o->N_E * o->N_t;
    struct Dev {
        int64_t count;
        double* samples;
        GbLagScalars* scal;
        long long* cells; // ncell + 1: the last is the total
        unsigned* counts;
        double* out;      // tf (ncell) | eb (N_E) | tb (N_t)
    };
    std::vector<Dev> dv((size_t)n);
    for (int d = 0; d < n; ++d) {
        gb200_ctx* ctx = ctxs[(size_t)d];
        Dev& D = dv[(size_t)d];
        const gb200_range rg = shard_range(ic, d, n);
        D.count = rg.count;
        CU(ctx, cudaSetDevice(ctx->device));
        double* img[4];
        void* v;
        for (int k = 0; k < 4; ++k) { rc = pool_get(ctx, SL_IMG0 + k, sizeof(double) * (size_t)rg.count + 8, &v); if (rc) return rc; img[k] = (double*)v; }
        rc = render_common(ctx, p, ic, &rg, pfs, 4, pl, img, true, ctx->stream, 1); if (rc) return rc;
        GbParams P;
        fill_params(p, ic, &rg, P);
        rc = upload_ic_and_tables(ctx, ic, nullptr, &pr->emissivity, P); if (rc) return rc;
        rc = pool_get(ctx, SL_LAG_PROF, sizeof(double) * 2 * (size_t)pr->n, &v); if (rc) return rc;
        const GbLagProfile gp{pr->time_kind, pr->n, (const double*)v, (const double*)v + pr->n};
        CU(ctx, cudaMemcpyAsync((void*)gp.r, pr->r, sizeof(double) * (size_t)pr->n, cudaMemcpyHostToDevice, ctx->stream));
        CU(ctx, cudaMemcpyAsync((void*)gp.t, pr->t, sizeof(double) * (size_t)pr->n, cudaMemcpyHostToDevice, ctx->stream));
        const int nblocks = (int)std::max<int64_t>(1, std::min<int64_t>((rg.count + 255) / 256, (int64_t)ctx->sm_count * 4));
        rc = pool_get(ctx, SL_LAG_SAMPLES, sizeof(double) * 3 * (size_t)rg.count + 8, &v); if (rc) return rc;
        D.samples = (double*)v;
        rc = pool_get(ctx, SL_LAG_PARTIAL, sizeof(GbLagScalars) * (size_t)nblocks, &v); if (rc) return rc;
        GbLagScalars* partial = (GbLagScalars*)v;
        rc = pool_get(ctx, SL_LAG_SCAL, sizeof(GbLagScalars), &v); if (rc) return rc;
        D.scal = (GbLagScalars*)v;
        CU(ctx, gb200_launch_lag_samples(P, img, gp, o->E0, rg.count, D.samples, partial, nblocks, D.scal, ctx->stream));
        ctx->stats.launches += 2;
    }
    std::vector<std::vector<NcclReduce>> ops;
    for (const Dev& D : dv) ops.push_back({{D.scal->mn, 2, ncclDouble, ncclMin}, {D.scal->mx, 4, ncclDouble, ncclMax}, {&D.scal->hits, 1, ncclInt64, ncclSum}});
    rc = all_reduce(ctxs, nccl, ops); if (rc) return rc;
    for (int d = 0; d < n; ++d) {
        gb200_ctx* ctx = ctxs[(size_t)d];
        Dev& D = dv[(size_t)d];
        CU(ctx, cudaSetDevice(ctx->device));
        void* v;
        rc = pool_get(ctx, SL_LAG_CELLS, sizeof(long long) * (size_t)(ncell + 1) + sizeof(unsigned) * (size_t)ncell, &v); if (rc) return rc;
        D.cells = (long long*)v;
        D.counts = (unsigned*)(D.cells + ncell + 1);
        rc = pool_get(ctx, SL_LAG_OUT, sizeof(double) * (size_t)(ncell + o->N_E + o->N_t), &v); if (rc) return rc;
        D.out = (double*)v;
        const int nblocks = (int)std::max<int64_t>(1, std::min<int64_t>((D.count + 255) / 256, (int64_t)ctx->sm_count * 8));
        CU(ctx, gb200_launch_lag_bin(D.scal, L, D.out + ncell, D.out + ncell + o->N_E, D.samples, D.count, D.cells, D.counts, nblocks, ctx->stream));
        ctx->stats.launches += D.count > 0 ? 2 : 1;
    }
    ops.clear();
    for (const Dev& D : dv) ops.push_back({{D.cells, (size_t)ncell + 1, ncclInt64, ncclSum}, {D.counts, (size_t)ncell, ncclUint32, ncclSum}});
    rc = all_reduce(ctxs, nccl, ops); if (rc) return rc;
    gb200_ctx* c0 = ctxs[0];
    const Dev& D0 = dv[0];
    GbLagScalars s;
    CU(c0, cudaSetDevice(c0->device));
    CU(c0, gb200_launch_lag_finish(D0.cells, D0.counts, ncell, D0.scal, D0.out, c0->stream));
    c0->stats.launches += 1;
    CU(c0, cudaMemcpyAsync(tf, D0.out, sizeof(double) * (size_t)ncell, cudaMemcpyDeviceToHost, c0->stream));
    CU(c0, cudaMemcpyAsync(energy_edges, D0.out + ncell, sizeof(double) * (size_t)o->N_E, cudaMemcpyDeviceToHost, c0->stream));
    CU(c0, cudaMemcpyAsync(time_edges, D0.out + ncell + o->N_E, sizeof(double) * (size_t)o->N_t, cudaMemcpyDeviceToHost, c0->stream));
    CU(c0, cudaMemcpyAsync(&s, D0.scal, sizeof s, cudaMemcpyDeviceToHost, c0->stream));
    for (int d = 0; d < n; ++d) {
        CU(ctxs[(size_t)d], cudaSetDevice(ctxs[(size_t)d]->device));
        rc = finish_stats(ctxs[(size_t)d], dv[(size_t)d].count); if (rc) return rc;
    }
    if (s.status == GB_LAG_NONFINITE) return fail(c0, GB200_ERR_INVALID_ARGUMENT, "a hit has a non-finite energy, time or flux (a redshift without a velocity field?)");
    if (s.status == GB_LAG_NO_HITS) return fail(c0, GB200_ERR_INVALID_ARGUMENT, "automatic limits need hits: no ray reached the disc");
    if (s.status == GB_LAG_DEGENERATE) return fail(c0, GB200_ERR_INVALID_ARGUMENT, "automatic limits need min < max over the hits");
    for (int j = 0; j < o->N_t; ++j) time_edges[j] -= o->t0;
    *hits = s.hits;
    return GB200_OK;
}

int gb200_lagtransfer(gb200_ctx* ctx, const gb200_problem* p, const gb200_ic* ic, const gb200_disc_profile* pr, const gb200_plunging_table* pl,
                      const gb200_lagtransfer_opts* opts, double* time_edges, double* energy_edges, double* tf, int64_t* hits) {
    if (!ctx) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null context");
    return lagtransfer_run({ctx}, nullptr, p, ic, pr, pl, opts, time_edges, energy_edges, tf, hits);
}

int gb200_comm_lagtransfer(gb200_comm* c, const gb200_problem* p, const gb200_ic* ic, const gb200_disc_profile* pr, const gb200_plunging_table* pl,
                           const gb200_lagtransfer_opts* opts, double* time_edges, double* energy_edges, double* tf, int64_t* hits) {
    if (!c) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null communicator");
    return lagtransfer_run(c->ctx, c->nccl.data(), p, ic, pr, pl, opts, time_edges, energy_edges, tf, hits);
}

// ---------------------------------------------------------------- quadrature of Cunningham transfer functions
static bool finite_ascending(const double* x, int64_t n, bool strict) {
    for (int64_t k = 0; k < n; ++k) {
        if (!std::isfinite(x[k])) return false;
        if (k > 0 && (strict ? !(x[k] > x[k - 1]) : !(x[k] >= x[k - 1]))) return false;
    }
    return true;
}

static int validate_tf_quad(gb200_ctx* ctx, bool lag, int32_t ntables, const gb200_tf_branches* tables, int32_t nmodels,
                            const gb200_tf_model* models, const double* g_grid, int32_t ngrid, const double* t_grid, int32_t nt,
                            const gb200_tf_quad_opts* o, const double* out) {
    if (!tables || !models || !g_grid || !o || !out || (lag && !t_grid)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "null argument");
    if (ntables < 1 || nmodels < 1) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "need ntables, nmodels >= 1 (got %d, %d)", ntables, nmodels);
    if (ngrid < 2 || ngrid > 65535 * 128) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "need 2 <= ngrid <= %d (got %d)", 65535 * 128, ngrid);
    if (!finite_ascending(g_grid, ngrid, true)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "g_grid must be finite and strictly ascending");
    if (lag && nt < 1) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "need nt >= 1 (got %d)", nt);
    if (lag && !finite_ascending(t_grid, nt, true)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "t_grid must be finite and strictly ascending");
    if (!(o->h > 0.0 && o->h < 0.5)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "need 0 < h < 0.5 (got %g)", o->h);
    if (o->upscale < 1) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "need upscale >= 1 (got %d)", o->upscale);
    if (o->npoints < 1 || o->npoints > 32 || !o->nodes || !o->weights)
        return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "need 1..32 Gauss points with nodes and weights (got %d)", o->npoints);
    for (int k = 0; k < o->npoints; ++k)
        if (!std::isfinite(o->nodes[k]) || !std::isfinite(o->weights[k])) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "Gauss nodes and weights must be finite");
    if (o->normalise != 0 && o->normalise != 1) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "normalise must be 0 or 1");
    if (lag && !std::isfinite(o->t0)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "t0 must be finite");
    for (int i = 0; i < ntables; ++i) {
        const gb200_tf_branches& T = tables[i];
        if (T.n_radii < 2 || !T.r_e || !T.gmin || !T.gmax || !T.off || !T.gs || !T.f || !T.t)
            return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "table %d: need n_radii >= 2 and every array", i);
        if (!finite_ascending(T.r_e, T.n_radii, true)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "table %d: r_e must be finite and strictly ascending", i);
        for (int k = 0; k < T.n_radii; ++k)
            if (!std::isfinite(T.gmin[k]) || !std::isfinite(T.gmax[k]) || !(T.gmin[k] < T.gmax[k]))
                return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "table %d, radius %d: need finite gmin < gmax", i, k);
        if (T.off[0] != 0) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "table %d: off[0] must be 0", i);
        for (int b = 0; b < 2 * T.n_radii; ++b) {
            const int64_t n = T.off[b + 1] - T.off[b];
            if (n < 2 || n > INT32_MAX) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "table %d, branch %d: need at least 2 knots (got %lld)", i, b, (long long)n);
            if (!finite_ascending(T.gs + T.off[b], n, false)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "table %d, branch %d: g* knots must be finite and ascending", i, b);
        }
    }
    for (int m = 0; m < nmodels; ++m) {
        const gb200_tf_model& M = models[m];
        if (M.table < 0 || M.table >= ntables) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "model %d: table index %d out of range [0, %d)", m, M.table, ntables);
        if (M.n_radii < 2 || !M.radii) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "model %d: need n_radii >= 2 (got %d)", m, M.n_radii);
        if (!finite_ascending(M.radii, M.n_radii, true)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "model %d: radii must be finite and strictly ascending", m);
        if (!std::isfinite(M.rmin)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "model %d: rmin must be finite", m);
        if (!std::isfinite(M.g_scale) || !(M.g_scale > 0.0)) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "model %d: g_scale must be positive and finite", m);
        int rc = validate_disc_profile(ctx, &M.profile, lag); if (rc) return rc;
    }
    return GB200_OK;
}

// Both entry points: every array of the call is packed into the pinned staging buffer and crosses in one copy; the result
// comes back in one.
static int tf_quad_run(gb200_ctx* ctx, bool lag, int32_t ntables, const gb200_tf_branches* tables, int32_t nmodels,
                       const gb200_tf_model* models, const double* g_grid, int32_t ngrid, const double* t_grid, int32_t nt,
                       const gb200_tf_quad_opts* o, double* out) {
    if (!ctx) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null context");
    ctx->stats = gb200_stats{};
    int rc = validate_tf_quad(ctx, lag, ntables, tables, nmodels, models, g_grid, ngrid, t_grid, nt, o, out); if (rc) return rc;
    if (!lag) nt = 1;
    std::vector<GbTfTable> tabs((size_t)ntables);
    std::vector<GbTfModel> mods((size_t)nmodels);
    int64_t nrad = 0, noff = 0, nknot = 0, nann = 0, nprof = 0;
    for (int i = 0; i < ntables; ++i) {
        tabs[(size_t)i] = GbTfTable{tables[i].n_radii, nrad, noff};
        nrad += tables[i].n_radii;
        noff += 2 * (int64_t)tables[i].n_radii + 1;
        nknot += tables[i].off[2 * tables[i].n_radii];
    }
    for (int m = 0; m < nmodels; ++m) {
        const gb200_tf_model& M = models[m];
        const gb200_emissivity& em = M.profile.emissivity;
        GbTfModel& G = mods[(size_t)m];
        G = GbTfModel{M.table, M.n_radii, nann, M.rmin, M.g_scale, em.kind, em.kind == GB200_EMISSIVITY_TABLE ? em.n : 0, em.index, nprof,
                      M.profile.time_kind, lag ? M.profile.n : 0, 0};
        nann += M.n_radii;
        nprof += 2 * (int64_t)G.emis_n;
        G.time0 = nprof;
        nprof += 2 * (int64_t)G.time_n;
    }
    // Every array of the call in one arena, laid out as in the batch calls (Arena).  The tables' and the models' arrays are
    // concatenated, so the fill pass copies them piece by piece, the branch offsets becoming knot indices of the whole call.
    GbTfArgs A{};
    auto layout = [&](Arena& a) {
        a.take(A.tables, ntables, tabs.data()); a.take(A.models, nmodels, mods.data());
        a.take(A.r_e, nrad); a.take(A.gmin, nrad); a.take(A.gmax, nrad);
        a.take(A.off, noff); a.take(A.gs, nknot); a.take(A.f, nknot); a.take(A.t, nknot);
        a.take(A.radii, nann); a.take(A.prof, nprof); a.take(A.g_grid, ngrid, g_grid);
        if (lag) a.take(A.t_grid, nt, t_grid);
        a.take(A.nodes, o->npoints, o->nodes); a.take(A.weights, o->npoints, o->weights);
        if (!a.fill) return;
        auto put = [](const auto* dst, int64_t at, const void* src, int64_t n) { memcpy((void*)(dst + at), src, sizeof(*dst) * (size_t)n); };
        int64_t k0 = 0;
        for (int i = 0; i < ntables; ++i) {
            const gb200_tf_branches& T = tables[i];
            const GbTfTable& G = tabs[(size_t)i];
            put(A.r_e, G.radius0, T.r_e, T.n_radii); put(A.gmin, G.radius0, T.gmin, T.n_radii); put(A.gmax, G.radius0, T.gmax, T.n_radii);
            int64_t* off = (int64_t*)A.off + G.off0;
            for (int b = 0; b <= 2 * T.n_radii; ++b) off[b] = k0 + T.off[b];
            const int64_t nk = T.off[2 * T.n_radii];
            put(A.gs, k0, T.gs, nk); put(A.f, k0, T.f, nk); put(A.t, k0, T.t, nk);
            k0 += nk;
        }
        for (int m = 0; m < nmodels; ++m) {
            const gb200_tf_model& M = models[m];
            const GbTfModel& G = mods[(size_t)m];
            put(A.radii, G.radius0, M.radii, M.n_radii);
            if (G.emis_n) { put(A.prof, G.emis0, M.profile.emissivity.r, G.emis_n); put(A.prof, G.emis0 + G.emis_n, M.profile.emissivity.eps, G.emis_n); }
            if (G.time_n) { put(A.prof, G.time0, M.profile.r, G.time_n); put(A.prof, G.time0 + G.time_n, M.profile.t, G.time_n); }
        }
    };
    Arena size{nullptr};
    layout(size);
    const size_t nout = (size_t)nmodels * (size_t)ngrid * (size_t)nt;
    { int rc_ = begin_call(ctx, ctx->stream); if (rc_) return rc_; }
    void *din, *dout;
    rc = pool_get(ctx, SL_TFQ_IN, size.used, &din); if (rc) return rc;
    rc = pool_get(ctx, SL_TFQ_OUT, sizeof(double) * nout, &dout); if (rc) return rc;
    CU(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    rc = ensure_stage(ctx, size.used); if (rc) return rc;
    Arena stage{(char*)ctx->stage, true};
    layout(stage);
    CU(ctx, cudaMemcpyAsync(din, ctx->stage, size.used, cudaMemcpyHostToDevice, ctx->stream));
    Arena dev{(char*)din};
    layout(dev);
    A.nmodels = nmodels; A.ngrid = ngrid; A.nt = nt; A.upscale = o->upscale; A.npoints = o->npoints; A.normalise = o->normalise;
    A.h = o->h; A.t0 = lag ? o->t0 : 0.0;
    A.out = (double*)dout;
    int launches = 0;
    CU(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    CU(ctx, gb200_launch_tf_quad(A, lag, ctx->stream, &launches));
    CU(ctx, cudaEventRecord(ctx->ev2, ctx->stream));
    CU(ctx, cudaMemcpyAsync(out, dout, sizeof(double) * nout, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaEventRecord(ctx->ev3, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    float k = 0, tot = 0;
    cudaEventElapsedTime(&k, ctx->ev1, ctx->ev2);
    cudaEventElapsedTime(&tot, ctx->ev0, ctx->ev3);
    ctx->stats.kernel_ms = k; ctx->stats.total_ms = tot; ctx->stats.launches = launches;
    return GB200_OK;
}

int gb200_tf_lineprofile(gb200_ctx* ctx, int32_t ntables, const gb200_tf_branches* tables, int32_t nmodels, const gb200_tf_model* models,
                         const double* g_grid, int32_t ngrid, const gb200_tf_quad_opts* opts, double* out) {
    return tf_quad_run(ctx, false, ntables, tables, nmodels, models, g_grid, ngrid, nullptr, 0, opts, out);
}

int gb200_tf_lagtransfer(gb200_ctx* ctx, int32_t ntables, const gb200_tf_branches* tables, int32_t nmodels, const gb200_tf_model* models,
                         const double* g_grid, int32_t ngrid, const double* t_grid, int32_t nt, const gb200_tf_quad_opts* opts, double* out) {
    return tf_quad_run(ctx, true, ntables, tables, nmodels, models, g_grid, ngrid, t_grid, nt, opts, out);
}

int gb200_bucket2d(gb200_ctx* ctx, int64_t n, const double* x, const double* y, const double* w, const double* xbins, int32_t nx,
                   const double* ybins, int32_t ny, double* out) {
    if (!ctx) return fail(nullptr, GB200_ERR_INVALID_ARGUMENT, "null context");
    if (n < 0 || (n > 0 && (!x || !y || !w)) || !xbins || !ybins || !out || nx < 1 || ny < 1 || (int64_t)nx * ny > (1 << 26))
        return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bad bucket arguments");
    for (int b = 1; b < nx; ++b) if (!(xbins[b] > xbins[b - 1])) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bins must be strictly increasing");
    for (int b = 1; b < ny; ++b) if (!(ybins[b] > ybins[b - 1])) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bins must be strictly increasing");
    { int rc_ = begin_call(ctx, ctx->stream); if (rc_) return rc_; }
    long double tot = 0.0L;
    for (int64_t i = 0; i < n; ++i) if (w[i] == w[i]) tot += fabsl((long double)w[i]);
    const double scale = tot > 0.0L ? (double)(4611686018427387904.0L / tot) : 1.0; // 2^62 / sum |w|
    void *dx, *dy, *dw, *dxb, *dyb, *dacc, *dout;
    const size_t nb = sizeof(double) * (size_t)(n > 0 ? n : 1), ncell = (size_t)nx * ny;
    int rc = pool_get(ctx, SL_G, nb, &dx); if (rc) return rc;
    rc = pool_get(ctx, SL_F, nb, &dy); if (rc) return rc;
    rc = pool_get(ctx, SL_X0, nb, &dw); if (rc) return rc;
    rc = pool_get(ctx, SL_BINS, sizeof(double) * (size_t)(nx + ny), &dxb); if (rc) return rc;
    dyb = (double*)dxb + nx;
    rc = pool_get(ctx, SL_PARTIAL, sizeof(long long) * ncell, &dacc); if (rc) return rc;
    rc = pool_get(ctx, SL_FLUX, sizeof(double) * ncell, &dout); if (rc) return rc;
    if (n > 0) {
        CU(ctx, cudaMemcpyAsync(dx, x, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
        CU(ctx, cudaMemcpyAsync(dy, y, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
        CU(ctx, cudaMemcpyAsync(dw, w, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    }
    CU(ctx, cudaMemcpyAsync(dxb, xbins, sizeof(double) * (size_t)nx, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemcpyAsync(dyb, ybins, sizeof(double) * (size_t)ny, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, gb200_launch_bucket2d((const double*)dx, (const double*)dy, (const double*)dw, n, (const double*)dxb, nx, (const double*)dyb, ny, scale,
                                  (long long*)dacc, (double*)dout, ctx->sm_count * 8, ctx->stream));
    ctx->stats.launches = 2;
    CU(ctx, cudaMemcpyAsync(out, dout, sizeof(double) * ncell, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return GB200_OK;
}

int gb200_debug_rhs(gb200_ctx* ctx, int32_t metric_kind, const double* mp, int64_t n, const double* u, double* du) {
    if (!ctx || !mp || !u || !du || n < 1) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bad arguments");
    if (metric_kind < 0 || metric_kind >= GB200_METRIC_COUNT) return fail(ctx, GB200_ERR_UNSUPPORTED, "metric kind %d", metric_kind);
    { int rc_ = begin_call(ctx, ctx->stream); if (rc_) return rc_; }
    GbParams P;
    memset(&P, 0, sizeof P);
    P.metric_kind = metric_kind; P.M = mp[0]; P.a = mp[1]; P.eps3 = mp[2];
    P.a2 = P.a * P.a; P.twoM = 2.0 * P.M; P.jp_e = P.eps3 * P.M * P.M * P.M;
    for (int k = 0; k < 8; ++k) P.mp[k] = mp[k];
    void *d_u, *d_du;
    int rc = pool_get(ctx, SL_X0, sizeof(double) * 8 * (size_t)n, &d_u); if (rc) return rc;
    rc = pool_get(ctx, SL_V0, sizeof(double) * 8 * (size_t)n, &d_du); if (rc) return rc;
    CU(ctx, cudaMemcpyAsync(d_u, u, sizeof(double) * 8 * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, gb200_launch_debug_rhs(P, n, (const double*)d_u, (double*)d_du, ctx->stream));
    CU(ctx, cudaMemcpyAsync(du, d_du, sizeof(double) * 8 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return GB200_OK;
}

// gb200_debug_math and gb200_debug_math_lo: `width` outputs per input through `launch`
static int debug_math(gb200_ctx* ctx, int64_t n, const double* x, double* out, int width,
                      cudaError_t (*launch)(long long, const double*, double*, cudaStream_t)) {
    if (!ctx || !x || !out || n < 1) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bad arguments");
    { int rc_ = begin_call(ctx, ctx->stream); if (rc_) return rc_; }
    void *d_x, *d_o;
    int rc = pool_get(ctx, SL_X0, sizeof(double) * (size_t)n, &d_x); if (rc) return rc;
    rc = pool_get(ctx, SL_V0, sizeof(double) * width * (size_t)n, &d_o); if (rc) return rc;
    CU(ctx, cudaMemcpyAsync(d_x, x, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, launch(n, (const double*)d_x, (double*)d_o, ctx->stream));
    CU(ctx, cudaMemcpyAsync(out, d_o, sizeof(double) * width * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return GB200_OK;
}

int gb200_debug_math(gb200_ctx* ctx, int64_t n, const double* x, double* out5) { return debug_math(ctx, n, x, out5, 5, gb200_launch_debug_math); }

int gb200_debug_math_lo(gb200_ctx* ctx, int64_t n, const double* x, double* out2) { return debug_math(ctx, n, x, out2, 2, gb200_launch_debug_math_lo); }

int gb200_fp64_peak(gb200_ctx* ctx, double* tflops_out) {
    if (!ctx || !tflops_out) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "null argument");
    return fp64_rate(ctx, [&](double* d, int blocks, int iters) { return gb200_launch_dfma(d, blocks, iters, ctx->stream); }, tflops_out);
}

int gb200_fp64_issue_probe(gb200_ctx* ctx, int32_t mix, double* tflops_out) {
    if (!ctx || !tflops_out || mix < 0 || mix > 5) return fail(ctx, GB200_ERR_INVALID_ARGUMENT, "bad argument");
    return fp64_rate(ctx, [&](double* d, int blocks, int iters) { return gb200_launch_dfma_mix(d, blocks, iters, mix, ctx->stream); }, tflops_out);
}

} // extern "C"
