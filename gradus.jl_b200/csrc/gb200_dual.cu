// gb200_dual.cu -- kernels over the generic-scalar integrator of gb200_generic.cuh:
//   gb200_dual_kernel<N>   forward-mode traces (N = 1: Newton derivative of the offset search, N = 2: Jacobian over
//                          (alpha, beta)) for the transfer-function solvers, src/tracing/precision-solvers.jl:73-131,401-451
//   gb200_path_kernel      one geodesic with every accepted step recorded (save_on = true, src/tracing/tracing.jl:66-108)
// One ray per thread.  These launches carry 10^2..10^5 rays between host-side root-finding rounds: they are latency
// bound, not throughput bound: their integrator is not the throughput kernel's of gb200_trace.cu, but the metric closed
// forms, the disc conditions, the endpoint redshift and the v^t constraint are the same templates of gb200_device.cuh --
// tests/test_gpu_dual.py holds the two integrators to the same end points.
#include <cuda_runtime.h>
#include "gb200_generic.cuh"
#include "gb200_internal.h"

struct GbNoRecord {
    template <class U> GB_HD void operator()(double, const U*) const {}
};

template <int N, int MK>
__global__ void __launch_bounds__(64) gb200_dual_kernel(const __grid_constant__ GbParams P, const __grid_constant__ GbDualIO io) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= io.n) return;
    typedef GD<N> S;
    S al(io.alpha[i]), be(io.beta[i]);
    for (int k = 0; k < N; ++k) { al.d[k] = io.dalpha[(size_t)k * io.n + i]; be.d[k] = io.dbeta[(size_t)k * io.n + i]; }
    S u0[8], E_obs;
    gen_initial_state<N>(P, al, be, u0, E_obs);
    const double hgt = io.height ? io.height[i] : P.gp0;
    GenResult<N> res;
    gen_trace_ray<N, MK>(P, u0, hgt, io.norm_partials != 0, res, GbNoRecord());
    if (io.status) io.status[i] = res.status;
    if (io.lambda) io.lambda[i] = res.lambda;
    for (int k = 0; k < 4; ++k) {
        if (io.x[k]) io.x[k][i] = res.u[k].v;
        if (io.v[k]) io.v[k][i] = res.u[4 + k].v;
    }
    if (io.naccept) io.naccept[i] = res.naccept;
    if (io.nreject) io.nreject[i] = res.nreject;
    if (io.flags) io.flags[i] = res.flags;
    S sth, cth;
    gd_sincos(res.u[2], sth, cth);
    const S rho = res.u[1] * sth; // _equatorial_project(gp.x), whatever the status
    if (io.rho) io.rho[i] = rho.v;
    if (io.drho) for (int k = 0; k < N; ++k) io.drho[(size_t)k * io.n + i] = rho.d[k];
    if (io.g) {
        const bool hit = res.status == GB200_STATUS_INTERSECTED_WITH_GEOMETRY && res.flags == 0;
        S g_(nan(""));
        if (hit) g_ = redshift_endpoint<-1>(P, res.u, res.u + 4, E_obs);
        io.g[i] = g_.v;
        if (io.dg) for (int k = 0; k < N; ++k) io.dg[(size_t)k * io.n + i] = hit ? g_.d[k] : nan("");
    }
}

cudaError_t gb200_launch_dual(const GbParams& P, const GbDualIO& io, cudaStream_t stream) {
    if (io.n <= 0) return cudaSuccess;
    const unsigned grid = (unsigned)((io.n + 63) / 64);
    const bool kerr = P.metric_kind == GB200_METRIC_KERR; // its own instantiation: a third of the code of the run-time-metric one
    if (io.npartials == 1) { if (kerr) gb200_dual_kernel<1, GB200_METRIC_KERR><<<grid, 64, 0, stream>>>(P, io); else gb200_dual_kernel<1, -1><<<grid, 64, 0, stream>>>(P, io); }
    else if (io.npartials == 2) { if (kerr) gb200_dual_kernel<2, GB200_METRIC_KERR><<<grid, 64, 0, stream>>>(P, io); else gb200_dual_kernel<2, -1><<<grid, 64, 0, stream>>>(P, io); }
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}

// ---------------------------------------------------------------- closest approach to a target point
// The objective of optimize_for_target (src/tracing/precision-solvers.jl:452-546) over a set of rays: one ray per thread
// through the generic integrator with the distance condition (disc_condition, GB200_GEOMETRY_TARGET_POINT).
template <int MK>
__global__ void __launch_bounds__(64) gb200_target_kernel(const __grid_constant__ GbParams P) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= P.count) return;
    GbRayInit ri;
    ray_initial_state(P, ray_index_of_slot(P, s), ri);
    GD<0> u[8];
    for (int k = 0; k < 4; ++k) { u[k] = GD<0>(ri.x[k]); u[4 + k] = GD<0>(ri.v[k]); }
    GenResult<0> res;
    gen_trace_ray<0, MK>(P, u, 0.0, false, res, GbNoRecord());
    if (P.o_status) P.o_status[s] = res.status;
    if (P.o_lambda) P.o_lambda[s] = res.lambda;
    for (int k = 0; k < 4; ++k) {
        if (P.o_x[k]) P.o_x[k][s] = res.u[k].v;
        if (P.o_v[k]) P.o_v[k][s] = res.u[4 + k].v;
        if (P.o_x0[k]) P.o_x0[k][s] = ri.x[k];
        if (P.o_v0[k]) P.o_v0[k][s] = ri.v[k];
    }
    if (P.o_naccept) P.o_naccept[s] = res.naccept;
    if (P.o_nreject) P.o_nreject[s] = res.nreject;
    if (P.o_flags) P.o_flags[s] = res.flags;
    if (P.o_closest) P.o_closest[s] = res.closest;
}

cudaError_t gb200_launch_target(const GbParams& P, cudaStream_t stream) {
    if (P.count <= 0) return cudaSuccess;
    const unsigned grid = (unsigned)((P.count + 63) / 64);
    if (P.metric_kind == GB200_METRIC_KERR) gb200_target_kernel<GB200_METRIC_KERR><<<grid, 64, 0, stream>>>(P);
    else gb200_target_kernel<-1><<<grid, 64, 0, stream>>>(P);
    return cudaGetLastError();
}

// ---------------------------------------------------------------- single-ray path recorder
struct GbPathRecord {
    int cap;
    double* lam;
    double* u;
    int* rows;
    GB_HD void operator()(double t, const GD<0>* x) const {
        const int r = *rows;
        if (r < cap) { lam[r] = t; for (int i = 0; i < 8; ++i) u[8 * r + i] = x[i].v; }
        *rows = r + 1;
    }
};

__global__ void gb200_path_kernel(const __grid_constant__ GbParams P, const double* __restrict__ u0in, int cap, double* __restrict__ lam_out,
                                  double* __restrict__ u_out, int* __restrict__ meta) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    GD<0> u[8];
    for (int i = 0; i < 8; ++i) u[i] = GD<0>(u0in[i]);
    if (P.mu == P.mu) { // constrain_all for mass P.mu at the starting point (mu = NaN: v^t is kept as given)
        GD<0> s, c, g[5], dr[5], dth[5];
        gd_sincos(u[2], s, c);
        metric_jacobian_kind<GD<0>>(P.metric_kind, P.mp, u[1], s, c, g, dr, dth);
        u[4] = constrain_vt(g, u[5], u[6], u[7], P.mu);
    }
    int rows = 0;
    GbPathRecord rec{cap, lam_out, u_out, &rows};
    GenResult<0> res;
    gen_trace_ray<0, -1>(P, u, P.gp0, false, res, rec);
    meta[0] = rows;
    meta[1] = res.status;
}

cudaError_t gb200_launch_path(const GbParams& P, const double* d_u0, int cap, double* d_lambda, double* d_u, int* d_meta, cudaStream_t stream) {
    gb200_path_kernel<<<1, 32, 0, stream>>>(P, d_u0, cap, d_lambda, d_u, d_meta);
    return cudaGetLastError();
}
