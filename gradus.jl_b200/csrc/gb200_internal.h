// gb200_internal.h -- launchers shared between gb200_trace.cu (kernels) and gb200_api.cu (C ABI).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
struct GbParams;
cudaError_t gb200_launch_trace(const GbParams& P, int sm_count, cudaStream_t stream, int* blocks_out);
cudaError_t gb200_launch_hist(const double* g, const double* f, int64_t n, const double* bins, int nbins, int right_closed,
                              double* partial, int nblocks, double* out, cudaStream_t stream);
cudaError_t gb200_launch_bucket2d(const double* x, const double* y, const double* w, int64_t n, const double* xb, int nx, const double* yb, int ny,
                                  double scale, long long* acc, double* out, int blocks, cudaStream_t stream);
cudaError_t gb200_launch_hist128_finish(const unsigned long long* acc, int nbins, double scale, double* out, cudaStream_t stream);
cudaError_t gb200_launch_dfma(double* d_out, int blocks, int iters, cudaStream_t stream);
cudaError_t gb200_launch_dfma_mix(double* d_out, int blocks, int iters, int mix, cudaStream_t stream);
cudaError_t gb200_launch_path(const GbParams& P, const double* d_u0, int cap, double* d_lambda, double* d_u, int* d_meta, cudaStream_t stream);
cudaError_t gb200_launch_debug_rhs(const GbParams& P, long long n, const double* d_u, double* d_du, cudaStream_t stream);
cudaError_t gb200_launch_debug_math(long long n, const double* d_x, double* d_out5, cudaStream_t stream);
cudaError_t gb200_launch_debug_math_lo(long long n, const double* d_x, double* d_out2, cudaStream_t stream);

// forward-mode (dual-number) traces and the single-ray path recorder: gb200_dual.cu
struct GbDualIO {
    int64_t n;
    int32_t npartials, norm_partials;
    const double *alpha, *beta, *dalpha, *dbeta, *height; // device
    int32_t* status;
    double* lambda;
    double* x[4];
    double* v[4];
    double *g, *dg, *rho, *drho;
    int32_t *naccept, *nreject, *flags;
};
cudaError_t gb200_launch_dual(const GbParams& P, const GbDualIO& io, cudaStream_t stream);
// closest approach to a target point (optimize_for_target's objective): the generic integrator over the rays of P
cudaError_t gb200_launch_target(const GbParams& P, cudaStream_t stream);

// binned lag-energy transfer function (gb200_lag.cu; host side gb200_lagtransfer in gb200_api.cu)
struct GbLagProfile { // t(rho) of gb200_disc_profile on the device
    int32_t time_kind, n;
    const double* r;
    const double* t;
};
struct GbLagLimits { // (lo, hi) of each axis, NaN = min / max over the hits; N_E, N_t >= 2
    double energy[2], time[2];
    int32_t N_E, N_t;
};
enum { GB_LAG_NONFINITE = 1, GB_LAG_NO_HITS = 2, GB_LAG_DEGENERATE = 3 };
struct GbLagScalars {
    // reduced over the hits of every device (the NCCL all-reduce works on these three groups)
    double mn[2];   // min E, min T (finite samples)
    double mx[4];   // max E, max T, max |f| (finite samples), 1 if any hit has a non-finite E, T or f
    long long hits;
    // derived from them by the edges kernel, the same on every device
    double scale, dedt; // fixed-point scale, (eb[1] - eb[0]) (tb[1] - tb[0])
    int32_t status;     // 0 or GB_LAG_*
};
cudaError_t gb200_launch_lag_samples(const GbParams& P, const double* const* img, const GbLagProfile& pr, double E0, int64_t n, double* samples,
                                     GbLagScalars* partial, int nblocks, GbLagScalars* scal, cudaStream_t stream);
cudaError_t gb200_launch_lag_bin(GbLagScalars* scal, const GbLagLimits& L, double* eb, double* tb, const double* samples, int64_t n,
                                 long long* cells, unsigned* counts, int nblocks, cudaStream_t stream);
cudaError_t gb200_launch_lag_finish(const long long* cells, const unsigned* counts, int ncell, const GbLagScalars* scal, double* tf, cudaStream_t stream);

// line profiles and lag-energy transfer functions from Cunningham transfer functions (gb200_tfquad.cu; host side
// gb200_tf_lineprofile / gb200_tf_lagtransfer in gb200_api.cu).  All arrays live in one device arena.
struct GbTfTable { // one gb200_tf_branches
    int32_t n_radii;
    int64_t radius0; // its radius 0 in r_e / gmin / gmax
    int64_t off0;    // its off[0] in off; off holds knot indices into gs / f / t of the whole call
};
struct GbTfModel { // one gb200_tf_model
    int32_t table, n_radii;
    int64_t radius0; // its first annulus in radii
    double rmin, g_scale;
    int32_t emis_kind, emis_n; // emissivity table: r at prof[emis0], eps at prof[emis0 + emis_n]
    double emis_index;
    int64_t emis0;
    int32_t time_kind, time_n; // arrival-time table: r at prof[time0], t at prof[time0 + time_n]
    int64_t time0;
};
struct GbTfArgs {
    const GbTfTable* tables;
    const GbTfModel* models;
    const double *r_e, *gmin, *gmax;
    const int64_t* off;
    const double *gs, *f, *t;
    const double* radii;
    const double* prof;
    const double* g_grid;
    const double* t_grid; // lag only
    const double *nodes, *weights;
    int32_t nmodels, ngrid, nt, upscale, npoints, normalise;
    double h, t0;
    double* out; // nmodels x ngrid (x nt)
};
cudaError_t gb200_launch_tf_quad(const GbTfArgs& A, bool lag, cudaStream_t stream, int* launches);
