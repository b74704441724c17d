// gb200_tfquad.cu -- line profiles and lag-energy transfer functions integrated from Cunningham transfer functions:
// integrate_lineprofile / integrate_lagtransfer (src/transfer-functions/integration.jl:158-207, 233-279, 322-442) for many
// emission models per launch, restating tf_integration.py operation by operation.
//
//   quad        one thread per (model, energy bin) walks the model's annuli in the host's order and accumulates in a
//               register (line profile) or in its own row of the output (lag: the host's np.add.at only ever adds to the
//               row of the bin), so no atomics are needed and no result depends on the other models of the call.  The
//               per-annulus quantities every bin shares (radius interval, blend weight, gmin, gmax, weight, t_sd, the
//               times at the ends of the g* range) are set up once per block, one annulus per thread, in shared memory.
//   normalise   _normalize! (transfer-functions/utils.jl:121-147): the division by g[j] + g[j+1] happens in `quad`, the
//               total over the model's bins is a fixed-order block reduction.
//
// The file is compiled with -fmad=false: the host rounds every product and sum separately, and the time of a branch has to
// be bit-identical to the host's so that it lands in the same time bin.
#include <cuda_runtime.h>
#include "gb200_device.cuh"
#include "gb200_internal.h"

namespace {

constexpr int kThreads = 128;
constexpr double kPi = 3.141592653589793; // math.pi

struct Annulus {
    int64_t k0[4];  // first knot of the lower / upper branch of table radius idx, then of idx + 1
    int32_t n[4];   // their knot counts
    double omth, th; // 1 - theta, theta: the blend between radii idx and idx + 1
    double gmin, gmax, span, weight, t_sd;
    double tend[4]; // lag: blended lower_t(h), upper_t(h), lower_t(1 - h), upper_t(1 - h)
};

// NaNLinearInterpolator of one tabulated branch; a NaN abscissa takes numpy's path (searchsorted puts NaN last)
__device__ __forceinline__ double branch_at(const double* xs, const double* ys, int n, double x) {
    if (x != x) { const double y = ys[n - 1]; return y == y ? y : 0.0; }
    return gb_nan_linear(xs, ys, n, x);
}

// InterpolatingTransferBranches' lazy blend (1 - theta) f1(x) + theta f2(x) of branch b (0 lower, 1 upper) of values v
__device__ __forceinline__ double blend(const GbTfArgs& A, const Annulus& a, const double* v, int b, double x) {
    const double f1 = branch_at(A.gs + a.k0[b], v + a.k0[b], a.n[b], x);
    const double f2 = branch_at(A.gs + a.k0[b + 2], v + a.k0[b + 2], a.n[b + 2], x);
    return a.omth * f1 + a.th * f2;
}

// the integrand g^3 f / sqrt(g*(1 - g*)); which: 0 both branches (line profile), 1 lower, 2 upper (lag)
__device__ __forceinline__ double integrand(const GbTfArgs& A, const Annulus& a, int which, double g) {
    const double gs = (g - a.gmin) / a.span;
    double f;
    if (which == 0) {
        const double fu = blend(A, a, A.f, 1, gs), fl = blend(A, a, A.f, 0, gs);
        f = (fu == fu ? fu : 0.0) + (fl == fl ? fl : 0.0);
    } else {
        f = blend(A, a, A.f, which - 1, gs);
        f = f == f ? f : 0.0;
    }
    return g * g * f * g / sqrt(gs * (1.0 - gs));
}

// integrate_edge: S(gh) |sqrt(gh) - sqrt(lim)| sqrt(h), gh = span lim_gs + gmin
__device__ __forceinline__ double edge(const GbTfArgs& A, const Annulus& a, int which, double lim, double lim_gs, double sqrt_h) {
    const double gh = a.span * lim_gs + a.gmin;
    return integrand(A, a, which, gh) * fabs(sqrt(gh) - sqrt(lim)) * sqrt_h;
}

// _integrate_bins (integration.jl:167-203) for one bin [lo, hi]: the edge rule near g* = 0 and 1, Gauss-Legendre elsewhere.
// The Gauss sum is numpy's pairwise sum of the row (fewer than 8 terms: in order from 0; else eight interleaved partial
// sums combined as ((0+1)+(2+3))+((4+5)+(6+7)), then the remainder in order), kept in eight rotating registers.
__device__ double integrate_bin(const GbTfArgs& A, const Annulus& a, int which, double lo, double hi, double sqrt_h,
                                const double* X, const double* W) {
    const double h = A.h, span = a.gmax - a.gmin;
    double glo = fmin(fmax(lo, a.gmin), a.gmax), ghi = fmin(fmax(hi, a.gmin), a.gmax);
    double lum = 0.0;
    bool live = glo != ghi;
    const double gs_lo = (lo - a.gmin) / span, gs_hi = (hi - a.gmin) / span;
    const bool near_lo = live && gs_lo < h;
    const bool only_lo = near_lo && !(gs_hi > h), part_lo = near_lo && gs_hi > h;
    if (part_lo) {
        lum = lum + edge(A, a, which, glo, h, sqrt_h);
        glo = span * h + a.gmin;
    }
    if (only_lo) lum = edge(A, a, which, glo, gs_hi, sqrt_h);
    live = live && !only_lo;
    const double one_h = 1.0 - h;
    const bool near_hi = live && gs_hi > one_h;
    const bool only_hi = near_hi && !(gs_lo < one_h), part_hi = near_hi && gs_lo < one_h;
    if (part_hi) {
        lum = lum + edge(A, a, which, ghi, one_h, sqrt_h);
        ghi = span * one_h + a.gmin;
    }
    if (only_hi) lum = edge(A, a, which, ghi, gs_lo, sqrt_h);
    live = live && !only_hi;
    if (!live) return lum + 0.0;
    const double q = (ghi - glo) / 2.0;
    const int np = A.npoints, nb = np < 8 ? 0 : np - np % 8;
    double r0 = 0.0, r1 = 0.0, r2 = 0.0, r3 = 0.0, r4 = 0.0, r5 = 0.0, r6 = 0.0, r7 = 0.0, sum = 0.0;
    for (int k = 0; k < np; ++k) {
        const double term = W[k] * integrand(A, a, which, (X[k] + 1.0) * q + glo);
        if (k < nb) { // partial sum k % 8 sits in r0; after a multiple of 8 terms partial j is back in r_j
            const double s = k < 8 ? term : r0 + term;
            r0 = r1; r1 = r2; r2 = r3; r3 = r4; r4 = r5; r5 = r6; r6 = r7; r7 = s;
        } else sum = sum + term;
        if (k + 1 == nb) sum = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7));
    }
    return lum + sum * q;
}

// ε(r): PowerLawEmissivity r^-index (libm pow on the host) or np.interp of the clipped radius
__device__ __forceinline__ double emissivity_at(const GbTfArgs& A, const GbTfModel& M, double r) {
    if (M.emis_kind == GB200_EMISSIVITY_POWERLAW) return pow(r, -M.emis_index);
    return gb_interp_clipped(A.prof + M.emis0, A.prof + M.emis0 + M.emis_n, M.emis_n, r);
}

__device__ __forceinline__ double coordtime_at(const GbTfArgs& A, const GbTfModel& M, double r) {
    const double* rs = A.prof + M.time0;
    const double* ts = rs + M.time_n;
    return M.time_kind == GB200_PROFILE_TIME_NAN_LINEAR ? gb_nan_linear_clipped(rs, ts, M.time_n, r) : gb_interp_clipped(rs, ts, M.time_n, r);
}

// annulus k of model M: InterpolatingTransferBranches(r_e) (transfer-functions-2d.jl:1-88) and the annulus weight
__device__ void set_up_annulus(const GbTfArgs& A, const GbTfModel& M, int k, bool lag, Annulus& a) {
    const GbTfTable T = A.tables[M.table];
    const double* radii = A.radii + M.radius0;
    const double r_e = radii[k];
    const double r_prev = k == 0 ? M.rmin - (radii[1] - M.rmin) : radii[k - 1];
    const double* R = A.r_e + T.radius0;
    int lo = 0, hi = T.n_radii - 1; // searchsorted(radii, r, side="right") - 1, clipped to [0, n - 2]
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (R[mid] <= r_e) lo = mid; else hi = mid; }
    a.th = (r_e - R[lo]) / (R[lo + 1] - R[lo]);
    a.omth = 1.0 - a.th;
    const double* gmin = A.gmin + T.radius0;
    const double* gmax = A.gmax + T.radius0;
    a.gmin = a.omth * gmin[lo] + a.th * gmin[lo + 1];
    a.gmax = a.omth * gmax[lo] + a.th * gmax[lo + 1];
    a.span = a.gmax - a.gmin;
    a.weight = (r_e - r_prev) * r_e * emissivity_at(A, M, r_e) * kPi / a.span;
    const int64_t* off = A.off + T.off0 + 2 * lo;
    for (int b = 0; b < 4; ++b) { a.k0[b] = off[b]; a.n[b] = (int32_t)(off[b + 1] - off[b]); }
    if (lag) {
        a.t_sd = coordtime_at(A, M, r_e) - A.t0;
        const double one_h = 1.0 - A.h;
        a.tend[0] = blend(A, a, A.t, 0, A.h);
        a.tend[1] = blend(A, a, A.t, 1, A.h);
        a.tend[2] = blend(A, a, A.t, 0, one_h);
        a.tend[3] = blend(A, a, A.t, 1, one_h);
    }
}

// _time_gstar / _time_interpolate (integration.jl:73-84): branch b's time at g*, blended with the other branch's within h
// of the ends of the g* range
__device__ __forceinline__ double time_gstar(const GbTfArgs& A, const Annulus& a, int b, double gs) {
    const double h = A.h;
    if (gs < h || gs > 1.0 - h) {
        const bool lo = gs < h;
        const double w = lo ? gs / h : 1.0 - (1.0 - gs) / h;
        const double t1 = a.tend[(lo ? 0 : 2) + b], t2 = a.tend[(lo ? 0 : 2) + (1 - b)];
        return t1 * w + (1.0 - w) * t2;
    }
    return blend(A, a, A.t, b, gs);
}

// numpy.searchsorted(t_grid, T, side="left"); NaN sorts last
__device__ __forceinline__ int time_bin(const double* tg, int nt, double T) {
    if (T != T) return nt;
    int lo = 0, hi = nt;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (tg[mid] < T) lo = mid + 1; else hi = mid; }
    return lo;
}

// The lag kernel asks for three blocks per SM (at most 170 registers) so that it does not spill; 0: no minimum
template <bool LAG>
__global__ void __launch_bounds__(kThreads, LAG ? 3 : 0) gb200_tf_quad_kernel(const GbTfArgs A) {
    __shared__ Annulus sh[kThreads];
    __shared__ double X[32], W[32];
    const int m = blockIdx.x, j = blockIdx.y * kThreads + threadIdx.x;
    const GbTfModel M = A.models[m];
    if (threadIdx.x < A.npoints) { X[threadIdx.x] = A.nodes[threadIdx.x]; W[threadIdx.x] = A.weights[threadIdx.x]; }
    const bool active = j < A.ngrid - 1;
    const double lo = active ? A.g_grid[j] / M.g_scale : 0.0, hi = active ? A.g_grid[j + 1] / M.g_scale : 0.0;
    const double sqrt_h = sqrt(A.h), up = (double)A.upscale;
    double* row = A.out + ((int64_t)m * A.ngrid + j) * (LAG ? A.nt : 1);
    double acc = 0.0;
    for (int base = 0; base < M.n_radii; base += kThreads) {
        __syncthreads(); // the previous chunk is consumed
        if (base + (int)threadIdx.x < M.n_radii) set_up_annulus(A, M, base + threadIdx.x, LAG, sh[threadIdx.x]);
        __syncthreads();
        if (!active) continue;
        const int nk = min(kThreads, M.n_radii - base);
        for (int c = 0; c < nk; ++c) {
            const Annulus& a = sh[c];
            if (!LAG) { // integrate_lineprofile: sub-bins of the unclipped bin
                const double dg = (hi - lo) / up;
                double contrib = 0.0;
                for (int i = 0; i < A.upscale; ++i) {
                    const double flo = lo + (double)i * dg;
                    contrib = contrib + integrate_bin(A, a, 0, flo, flo + dg, sqrt_h, X, W);
                }
                acc = acc + contrib * a.weight;
            } else { // integrate_lagtransfer: sub-bins of the clipped bin, each branch into its own time bin
                const double glo = fmin(fmax(lo, a.gmin), a.gmax), ghi = fmin(fmax(hi, a.gmin), a.gmax);
                if (!(glo != ghi)) continue;
                const double dg = (ghi - glo) / up;
                for (int i = 0; i < A.upscale; ++i) {
                    const double flo = glo + (double)i * dg, fhi = flo + dg;
                    const double k1 = integrate_bin(A, a, 1, flo, fhi, sqrt_h, X, W);
                    const double k2 = integrate_bin(A, a, 2, flo, fhi, sqrt_h, X, W);
                    const double gs_lo = fmin(fmax((flo - a.gmin) / a.span, 0.0), 1.0);
                    const double gs_hi = fmin(fmax((fhi - a.gmin) / a.span, 0.0), 1.0);
                    const double T1 = (time_gstar(A, a, 0, gs_lo) + time_gstar(A, a, 0, gs_hi)) / 2.0 + a.t_sd;
                    const double T2 = (time_gstar(A, a, 1, gs_lo) + time_gstar(A, a, 1, gs_hi)) / 2.0 + a.t_sd;
                    const int i1 = time_bin(A.t_grid, A.nt, T1), i2 = time_bin(A.t_grid, A.nt, T2);
                    if (i1 < A.nt) row[i1] = row[i1] + k1 * a.weight;
                    if (i2 < A.nt) row[i2] = row[i2] + k2 * a.weight;
                }
            }
        }
    }
    if (j >= A.ngrid) return;
    const double gsum = active ? A.g_grid[j + 1] + A.g_grid[j] : 0.0;
    if (!LAG) row[0] = !active ? 0.0 : (A.normalise ? acc / gsum : acc);
    else if (active && A.normalise)
        for (int k = 0; k < A.nt; ++k) row[k] = row[k] / gsum;
}

// divide model blockIdx.x's n values by the sum of its first nsum when that is positive (`if total > 0`)
__global__ void __launch_bounds__(kThreads) gb200_tf_normalise_kernel(double* out, int64_t n, int64_t nsum) {
    __shared__ double part[kThreads];
    double* o = out + (int64_t)blockIdx.x * n;
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < nsum; i += kThreads) s = s + o[i];
    part[threadIdx.x] = s;
    for (int w = kThreads / 2; w > 0; w >>= 1) {
        __syncthreads();
        if ((int)threadIdx.x < w) part[threadIdx.x] = part[threadIdx.x] + part[threadIdx.x + w];
    }
    __syncthreads();
    const double total = part[0];
    if (!(total > 0.0)) return;
    for (int64_t i = threadIdx.x; i < n; i += kThreads) o[i] = o[i] / total;
}

} // namespace

cudaError_t gb200_launch_tf_quad(const GbTfArgs& A, bool lag, cudaStream_t stream, int* launches) {
    const dim3 grid((unsigned)A.nmodels, (unsigned)((A.ngrid + kThreads - 1) / kThreads));
    const int64_t per_model = (int64_t)A.ngrid * (lag ? A.nt : 1);
    if (lag) {
        cudaError_t e = cudaMemsetAsync(A.out, 0, sizeof(double) * (size_t)per_model * (size_t)A.nmodels, stream);
        if (e != cudaSuccess) return e;
        gb200_tf_quad_kernel<true><<<grid, kThreads, 0, stream>>>(A);
    } else gb200_tf_quad_kernel<false><<<grid, kThreads, 0, stream>>>(A);
    *launches = 1;
    if (A.normalise) {
        gb200_tf_normalise_kernel<<<A.nmodels, kThreads, 0, stream>>>(A.out, per_model, (int64_t)(A.ngrid - 1) * (lag ? A.nt : 1));
        *launches = 2;
    }
    return cudaGetLastError();
}
