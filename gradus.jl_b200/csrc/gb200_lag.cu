// gb200_lag.cu -- the binned lag-energy transfer function on the device: binflux(lagtransfer(...)) of
// src/transfer-functions/transfer-functions-2d.jl:100-122,163-242 after the fused render of gb200_trace.cu.
//
//   samples   per ray slot (E, T, f) = (g E0, t_src(rho) + t, g^3 eps(rho) r^2), NaN for a miss; per-block min / max / count
//   reduce    the block partials -> one GbLagScalars (min, max and count do not depend on the order of reduction)
//   edges     linspace edges of both axes and the fixed-point scale, from the (all-reduced) scalars
//   bin       Buckets.Simple into 64-bit fixed-point cells, plus a count of contributing samples per cell
//   finish    tf = cell / total / (de dt), NaN where no sample contributed
//
// The cells are integers, so their sum over samples, blocks and devices is exact in any order: one device and eight give
// the same bits.
#include <cuda_runtime.h>
#include "gb200_device.cuh"
#include "gb200_internal.h"

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kThreads = 256;

// numpy.linspace(lo, hi, N)[k]: k * step + lo with step = (hi - lo) / (N - 1), two roundings, the last edge exactly hi
__device__ double lag_edge(double lo, double hi, int N, int k) {
    if (k == N - 1) return hi;
    return __dadd_rn(__dmul_rn((double)k, (hi - lo) / (double)(N - 1)), lo);
}

__device__ void lag_identity(GbLagScalars& s) {
    s.mn[0] = s.mn[1] = INFINITY;
    s.mx[0] = s.mx[1] = -INFINITY;
    s.mx[2] = s.mx[3] = 0.0;
    s.hits = 0;
    s.scale = s.dedt = 0.0;
    s.status = 0;
}

__device__ void lag_combine(GbLagScalars& a, const GbLagScalars& b) {
    for (int k = 0; k < 2; ++k) a.mn[k] = fmin(a.mn[k], b.mn[k]);
    for (int k = 0; k < 4; ++k) a.mx[k] = fmax(a.mx[k], b.mx[k]);
    a.hits += b.hits;
}

// block-wide combination of every thread's `s` into thread 0's
__device__ void lag_block_reduce(GbLagScalars& s) {
    __shared__ GbLagScalars sh[kThreads / 32];
    for (int off = 16; off > 0; off >>= 1) {
        GbLagScalars o;
        for (int k = 0; k < 2; ++k) o.mn[k] = __shfl_down_sync(kFull, s.mn[k], off);
        for (int k = 0; k < 4; ++k) o.mx[k] = __shfl_down_sync(kFull, s.mx[k], off);
        o.hits = __shfl_down_sync(kFull, s.hits, off);
        lag_combine(s, o);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) sh[warp] = s;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int w = 1; w < kThreads / 32; ++w) lag_combine(s, sh[w]);
}

__global__ void __launch_bounds__(kThreads) gb200_lag_samples_kernel(const GbParams P, const double* __restrict__ status, const double* __restrict__ g,
                                                                    const double* __restrict__ rho, const double* __restrict__ t, GbLagProfile pr,
                                                                    double E0, int64_t n, double* __restrict__ samples, GbLagScalars* __restrict__ partial) {
    GbLagScalars s;
    lag_identity(s);
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads) {
        double E = nan(""), T = nan(""), f = nan("");
        if (status[i] == (double)GB200_STATUS_INTERSECTED_WITH_GEOMETRY) {
            GbRayInit ri; // the polar plane's r^2 (unnormalized_areas, image-planes/planes.jl:108-115)
            ray_initial_state(P, ray_index_of_slot(P, i), ri);
            const double gi = g[i], r = rho[i];
            E = gi * E0;
            T = (pr.time_kind == GB200_PROFILE_TIME_NAN_LINEAR ? gb_nan_linear_clipped(pr.r, pr.t, pr.n, r) : gb_interp_clipped(pr.r, pr.t, pr.n, r)) + t[i];
            f = pow(gi, 3.0) * emissivity_eval(P, r) * ri.area; // g .^ 3 is libm pow on the host, not g * g * g
            if (isfinite(E) && isfinite(T) && isfinite(f)) {
                s.mn[0] = fmin(s.mn[0], E); s.mx[0] = fmax(s.mx[0], E);
                s.mn[1] = fmin(s.mn[1], T); s.mx[1] = fmax(s.mx[1], T);
                s.mx[2] = fmax(s.mx[2], fabs(f));
            } else s.mx[3] = 1.0;
            s.hits += 1;
        }
        samples[i] = E; samples[n + i] = T; samples[2 * n + i] = f;
    }
    lag_block_reduce(s);
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

__global__ void __launch_bounds__(kThreads) gb200_lag_reduce_kernel(const GbLagScalars* __restrict__ partial, int nblocks, GbLagScalars* __restrict__ out) {
    GbLagScalars s;
    lag_identity(s);
    for (int b = threadIdx.x; b < nblocks; b += kThreads) lag_combine(s, partial[b]);
    lag_block_reduce(s);
    if (threadIdx.x == 0) *out = s;
}

// Edges of both axes from the global scalars, and the fixed-point scale: the largest power of two with
// scale * H * max|f| <= 2^62, i.e. 2^floor(62 - log2(H max|f|)).  It depends only on the global hit count and maximum,
// so every device uses the same one, and it bounds sum |q| by 2^62 + H/2: the int64 cells cannot overflow.
__global__ void gb200_lag_edges_kernel(GbLagScalars* __restrict__ s, GbLagLimits L, double* __restrict__ eb, double* __restrict__ tb) {
    const bool autoE = L.energy[0] != L.energy[0], autoT = L.time[0] != L.time[0];
    const double Elo = autoE ? s->mn[0] : L.energy[0], Ehi = autoE ? s->mx[0] : L.energy[1];
    const double Tlo = autoT ? s->mn[1] : L.time[0], Thi = autoT ? s->mx[1] : L.time[1];
    int status = 0;
    if (s->mx[3] != 0.0) status = GB_LAG_NONFINITE;
    else if ((autoE || autoT) && s->hits == 0) status = GB_LAG_NO_HITS;
    else if ((autoE && !(Elo < Ehi)) || (autoT && !(Tlo < Thi))) status = GB_LAG_DEGENERATE;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (status == 0 && i < L.N_E) eb[i] = lag_edge(Elo, Ehi, L.N_E, i);
    if (status == 0 && i < L.N_t) tb[i] = lag_edge(Tlo, Thi, L.N_t, i);
    if (i == 0) { // the only writer; the fields it writes are not read by this kernel
        const double x = (double)s->hits * s->mx[2];
        double scale = 1.0;
        if (x > 0.0) {
            int e;
            const double m = frexp(x, &e); // x = m 2^e, m in [0.5, 1)
            scale = ldexp(1.0, (m == 0.5 ? 63 : 62) - e);
        }
        s->scale = scale;
        s->dedt = (lag_edge(Elo, Ehi, L.N_E, 1) - Elo) * (lag_edge(Tlo, Thi, L.N_t, 1) - Tlo);
        s->status = status;
    }
}

__global__ void __launch_bounds__(kThreads) gb200_lag_bin_kernel(const double* __restrict__ samples, int64_t n, const double* __restrict__ eb, int NE,
                                                                const double* __restrict__ tb, int Nt, const GbLagScalars* __restrict__ s,
                                                                long long* __restrict__ cells, unsigned* __restrict__ counts) {
    if (s->status != 0) return;
    const double scale = s->scale;
    const unsigned lane = threadIdx.x & 31u;
    const int64_t ncell = (int64_t)NE * Nt;
    long long tot = 0;
    for (int64_t base = (int64_t)blockIdx.x * kThreads; base < n; base += (int64_t)gridDim.x * kThreads) {
        const int64_t i = base + threadIdx.x;
        int cell = -1;
        long long q = 0;
        bool nz = false;
        if (i < n) {
            const double E = samples[i];
            if (E == E) {
                const double T = samples[n + i], f = samples[2 * n + i];
                cell = gb_simple_bucket(eb, NE, E) * Nt + gb_simple_bucket(tb, Nt, T);
                q = __double2ll_rn(f * scale);
                nz = f != 0.0;
            }
        }
        tot += q;
        const unsigned active = __ballot_sync(kFull, cell >= 0);
        const unsigned nzmask = __ballot_sync(kFull, nz);
        if (cell >= 0) { // lanes of the warp that share a cell are combined first, as in gb200_bucket2d_kernel
            const unsigned peers = __match_any_sync(active, cell);
            long long sum = 0;
            unsigned rem = peers;
            while (rem) { const int src = __ffs(rem) - 1; sum += __shfl_sync(peers, q, src); rem &= rem - 1; }
            if ((int)lane == __ffs(peers) - 1) {
                atomicAdd((unsigned long long*)&cells[cell], (unsigned long long)sum);
                const unsigned c = (unsigned)__popc(peers & nzmask);
                if (c) atomicAdd(&counts[cell], c);
            }
        }
    }
    for (int off = 16; off > 0; off >>= 1) tot += __shfl_down_sync(kFull, tot, off);
    if (lane == 0 && tot != 0) atomicAdd((unsigned long long*)&cells[ncell], (unsigned long long)tot); // cells[ncell]: the total, sum of all cells
}

__global__ void gb200_lag_finish_kernel(const long long* __restrict__ cells, const unsigned* __restrict__ counts, int ncell,
                                        const GbLagScalars* __restrict__ s, double* __restrict__ tf) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncell) return;
    tf[c] = (s->status != 0 || counts[c] == 0) ? nan("") : ((double)cells[c] / (double)cells[ncell]) / s->dedt;
}

} // namespace

cudaError_t gb200_launch_lag_samples(const GbParams& P, const double* const* img, const GbLagProfile& pr, double E0, int64_t n, double* samples,
                                     GbLagScalars* partial, int nblocks, GbLagScalars* scal, cudaStream_t stream) {
    gb200_lag_samples_kernel<<<nblocks, kThreads, 0, stream>>>(P, img[0], img[1], img[2], img[3], pr, E0, n, samples, partial);
    gb200_lag_reduce_kernel<<<1, kThreads, 0, stream>>>(partial, nblocks, scal);
    return cudaGetLastError();
}

cudaError_t gb200_launch_lag_bin(GbLagScalars* scal, const GbLagLimits& L, double* eb, double* tb, const double* samples, int64_t n,
                                 long long* cells, unsigned* counts, int nblocks, cudaStream_t stream) {
    const int ncell = L.N_E * L.N_t, nedge = L.N_E > L.N_t ? L.N_E : L.N_t;
    cudaError_t e = cudaMemsetAsync(cells, 0, sizeof(long long) * (size_t)(ncell + 1), stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(counts, 0, sizeof(unsigned) * (size_t)ncell, stream);
    if (e != cudaSuccess) return e;
    gb200_lag_edges_kernel<<<(nedge + kThreads - 1) / kThreads, kThreads, 0, stream>>>(scal, L, eb, tb);
    if (n > 0) gb200_lag_bin_kernel<<<nblocks, kThreads, 0, stream>>>(samples, n, eb, L.N_E, tb, L.N_t, scal, cells, counts);
    return cudaGetLastError();
}

cudaError_t gb200_launch_lag_finish(const long long* cells, const unsigned* counts, int ncell, const GbLagScalars* scal, double* tf, cudaStream_t stream) {
    gb200_lag_finish_kernel<<<(ncell + kThreads - 1) / kThreads, kThreads, 0, stream>>>(cells, counts, ncell, scal, tf);
    return cudaGetLastError();
}
