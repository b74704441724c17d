// gb200_trace.cu -- the hot path: persistent-thread FP64 adaptive Tsit5 ray tracer for sm_100a.
//
// One ray per thread, one warp per CTA.  Registers hold the previous and the proposed state, the FSAL slope and k7,
// running sums and the controller; the stage values k2..k6 live in shared memory (GbK).  A step attempt is
// straight-line code committed with selects (no taken branch, the loop-carried state stays in the same registers on
// every path): reciprocals, sincos and the controller's log / exp are branch-free with their coefficients in the
// constant bank, and the 6 interior event samples are skipped when a bound on the dense output proves that the disc
// condition cannot change sign.  Warps stay full through a work queue: a global ticket counter hands out ray slots,
// and a warp refills its lanes (one warp-aggregated atomicAdd) once GB_REFILL_THRESH of them have terminated.
// Terminated lanes keep their last step and are finalised together (event root find on the dense output, discrete
// callbacks, point function, endpoint store), so the divergent epilogue is paid once per batch, not once per ray.
// The measurements behind each of these choices are in profiles/r0{1,2}_tuning_log.md.
//
// What it replaces in the reference (all per ray, on CPU threads):
//   prob_func -> velfunc(i) -> constrain_all         src/tracing/geodesic-problem.jl:121-154
//   _solve_reinit! / auto_dt_reset! / solve!          src/tracing/tracing.jl:234-252
//   OrdinaryDiffEq Tsit5 perform_step! + PI controller, DiffEqBase ContinuousCallback
//   (interp_points = 8, left root find) and DiscreteCallbacks of create_callback_set
//                                                     src/tracing/callbacks.jl:25-28
//   unpack_solution / point functions                 src/solution-processing.jl:86-112,
//                                                     src/rendering/rendering.jl:103-107
#include <cstdio>
#include <cuda_runtime.h>
#include "gb200_device.cuh"
#include "gb200_internal.h"

constexpr int GB_BLOCK = 32;         // one warp per CTA: the service decision needs no cross-warp barrier (v21 sweep, profiles/r01_tuning_log.md)
constexpr int GB_MIN_BLOCKS = 12;    // 12 warps per SM at 168 registers per thread
constexpr int GB_REFILL_THRESH = 16; // idle lanes per warp that trigger a service pass (per CTA: x warps per CTA)
constexpr int GB_SYNC_EVERY = 16;    // service decision (a single-warp barrier count) every n-th attempt

#define LANE_EMPTY 0
#define LANE_RUN 1
#define LANE_PENDING 2
#define FULLMASK 0xffffffffu

// Storage of the stage values of one component: get(0) = k1 (FSAL), get(1..5) = k2..k6, get(6) = k7.  k2..k6 sit in
// shared memory ([stage][thread], conflict-free) instead of 60 registers, k1 and k7 in registers; the indices are
// compile-time constants after unrolling, so the selection folds away.
struct GbK {
    double k1, k7;
    double* p; // &sh_k[first row of this component][threadIdx.x]
    GB_D double get(int j) const { return j == 0 ? k1 : (j == 6 ? k7 : p[(j - 1) * GB_BLOCK]); }
    GB_D void set(int j, double v) { if (j == 0) k1 = v; else if (j == 6) k7 = v; else p[(j - 1) * GB_BLOCK] = v; }
};
// stage input  u + dt * sum_{l<S} a_{S+1,l+1} k_l   (S = 1..6 -> stages 2..7), summed left to right like the reference.
// k0 is the FSAL slope (k1 of the tableau); k[1..5] are k2..k6.
template <int S>
GB_D double comb(double u, double dt, double k0, const GbK& k) {
    if (S == 1) return fma(dt * GB_C(A21), k0, u);
    if (S == 2) return fma(dt, fma(GB_C(A32), k.get(1), GB_C(A31) * k0), u);
    if (S == 3) return fma(dt, fma(GB_C(A43), k.get(2), fma(GB_C(A42), k.get(1), GB_C(A41) * k0)), u);
    if (S == 4) return fma(dt, fma(GB_C(A54), k.get(3), fma(GB_C(A53), k.get(2), fma(GB_C(A52), k.get(1), GB_C(A51) * k0))), u);
    if (S == 5) return fma(dt, fma(GB_C(A65), k.get(4), fma(GB_C(A64), k.get(3), fma(GB_C(A63), k.get(2), fma(GB_C(A62), k.get(1), GB_C(A61) * k0)))), u);
    return fma(dt, fma(GB_C(A76), k.get(5), fma(GB_C(A75), k.get(4), fma(GB_C(A74), k.get(3), fma(GB_C(A73), k.get(2), fma(GB_C(A72), k.get(1), GB_C(A71) * k0))))), u);
}
template <int S> GB_D constexpr double a7coef() {
    return S == 0 ? GB_C(A71) : S == 1 ? GB_C(A72) : S == 2 ? GB_C(A73) : S == 3 ? GB_C(A74) : S == 4 ? GB_C(A75) : GB_C(A76);
}
template <int S> GB_D constexpr double btcoef() {
    return S == 0 ? GB_C(BT1) : S == 1 ? GB_C(BT2) : S == 2 ? GB_C(BT3) : S == 3 ? GB_C(BT4) : S == 4 ? GB_C(BT5) : S == 5 ? GB_C(BT6) : GB_C(BT7);
}
// dense-output polynomial coefficients  u(Th) = u0 + dt*Th*(k0 + Th*(C2 + Th*(C3 + Th*C4)))
GB_D void dense_coeffs(double k0, const GbK& k, double k6, double& C2, double& C3, double& C4) {
    const double k2 = k.get(1), k3 = k.get(2), k4 = k.get(3), k5 = k.get(4), k6_ = k.get(5);
    C2 = fma(GB_C(R72), k6, fma(GB_C(R62), k6_, fma(GB_C(R52), k5, fma(GB_C(R42), k4, fma(GB_C(R32), k3, fma(GB_C(R22), k2, GB_C(R12) * k0))))));
    C3 = fma(GB_C(R73), k6, fma(GB_C(R63), k6_, fma(GB_C(R53), k5, fma(GB_C(R43), k4, fma(GB_C(R33), k3, fma(GB_C(R23), k2, GB_C(R13) * k0))))));
    C4 = fma(GB_C(R74), k6, fma(GB_C(R64), k6_, fma(GB_C(R54), k5, fma(GB_C(R44), k4, fma(GB_C(R34), k3, fma(GB_C(R24), k2, GB_C(R14) * k0))))));
}
GB_D double dense_eval(double u0, double dt, double Th, double C1, double C2, double C3, double C4) {
    return fma(dt * Th, fma(Th, fma(Th, fma(Th, C4, C3), C2), C1), u0);
}
GB_D double sgn(double x) { return (x > 0.0) ? 1.0 : ((x < 0.0) ? -1.0 : 0.0); }

// controller power x^y (PI controller, OrdinaryDiffEq): exp(y log x) is within 2 ulp of pow(x, y) here
GB_D double ctrl_pow_log(double logx, double x, double y, int mode) {
    if (mode == GB200_POW_FAST32) return (double)exp2f((float)y * log2f((float)x));
    return exp(y * logx);
}

// The step acceptance test EEst^2 <= 1.  Written as a call it yields the same instructions as the comparison written
// in place, but a different schedule of the step counters that follow it.
GB_D bool gb_le_one(double a) { return a <= 1.0; }

// 1 / (abstol + reltol max(|a|, |b|)): the reciprocal error scale of one component (calculate_residuals,
// DiffEqBase).  The estimate it feeds enters the controller through EEst^(7/50) and the test EEst <= 1, and the reference
// itself evaluates that power at Float32 accuracy (FastPower), so the scale does not need 53 bits: the hardware seed alone
// (rcp.approx.f64: 2^-20 and better) is used, two DFMAs fewer per component than one Newton step on it.  Measured on C2
// (profiles/r02_tuning_log.md): 39.93 ms; seed + one Newton step (2^-40) 40.48 ms; the scale in Float32 on the FP32 /
// integer / special-function pipes 39.79 ms, but its truncated |u| biases every scale by up to 1e-6 and moves 36 of 1.94 M
// disc hits across the grazing band, where the seed moves one.
GB_D double gb_inv_scale(double a, double b, double reltol, double abstol) {
    // fabs is applied to the argument of larger magnitude as an operand modifier: selecting |a| or |b| directly makes the
    // compiler materialise both absolute values with two extra FP64 instructions
    const double m = fabs(a) > fabs(b) ? a : b;
    double y;
    const double x = fma(fabs(m), reltol, abstol);
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    return y;
}

// Can the disc condition become negative anywhere on this step?  Conservative bound from the dense-output
// polynomial: |u(Th) - u0| <= |dt| (|C1| + |C2| + |C3| + |C4|) for Th in [0, 1], and |cos| is 1-Lipschitz.
// Returning false lets the caller skip the 6 interior samples (they would all be positive).
template <int GEOM>
GB_D bool scan_needed(const GbParams& P, double r0, double acos0, double cprev, double Bth, double Br) {
    const double slack = 1.0 + 1e-9;
    if (GEOM == GB200_GEOMETRY_THIN_DISC) return !(acos0 - Bth > P.gtol * slack + 1e-12);
    if (GEOM == GB200_GEOMETRY_SHAKURA_SUNYAEV) {
        const double hmax = 3.0 * P.gp1 * P.gp0;
        return !((acos0 - Bth) > 0.0 && (acos0 - Bth) * (r0 - Br) > hmax * slack + 1e-12);
    }
    if (GEOM == GB200_GEOMETRY_DATUM_PLANE) return !(fabs(cprev) > (Br + (fabs(r0) + Br) * Bth) * slack + 1e-12);
    if (GEOM == GB200_GEOMETRY_THICK_TABLE) return !((acos0 - Bth) > 0.0 && (acos0 - Bth) * (r0 - Br) > P.gp0 * slack + 1e-12); // gp0 = max of the table
    return false;
}


// ---------------------------------------------------------------- fused line-profile histogram
// bucket(Simple(), g, f, bins) (src/line-profiles.jl:196) accumulated where the ray is finalised: the (g, f) pair never
// goes through HBM.  Each CTA owns a histogram in shared memory; contributions are added as 128-bit fixed-point integers
// (two 64-bit words with carry), because integer addition is associative: which CTA finalises which ray, in what order,
// on how many GPUs -- the tickets are handed out dynamically -- cannot change a single bit of the result.
__device__ __forceinline__ void gb_acc128(unsigned long long* lo, unsigned long long* hi, unsigned long long vlo, unsigned long long vhi) {
    const unsigned long long old = atomicAdd(lo, vlo);
    if (old + vlo < old) ++vhi; // carry out of the low word
    if (vhi) atomicAdd(hi, vhi);
}
__device__ __noinline__ void gb_hist_add(const GbParams& P, unsigned long long* sh_hist, double g, double f) {
    int lo = 0, hi = P.lp_nbins; // right_closed: first idx with bins[idx] >= g; else first idx with bins[idx] > g, minus 1
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const bool go_right = P.lp_right_closed ? (P.lp_bins[mid] < g) : (P.lp_bins[mid] <= g);
        if (go_right) lo = mid + 1; else hi = mid;
    }
    int bin = P.lp_right_closed ? lo : lo - 1;
    bin = bin < 0 ? 0 : (bin > P.lp_nbins - 1 ? P.lp_nbins - 1 : bin);
    const double v = fmin(f * P.lp_scale, 8.5e37); // < 2^126: the host chooses lp_scale from a bound on sum f
    if (!(v > 0.0)) return;
    const double vh = floor(v * 5.421010862427522e-20); // v / 2^64: exact, v has 53 significant bits
    const unsigned long long whi = __double2ull_rz(vh);
    const unsigned long long wlo = __double2ull_rz(fma(-vh, 18446744073709551616.0, v));
    gb_acc128(&sh_hist[bin], &sh_hist[P.lp_nbins + bin], wlo, whi);
}

// Equatorial crossings (GB200_PF_EQUATORIAL_CROSSINGS) are counted only by instantiations that need them: GEOM is then a
// public geometry kind plus GB_GEOM_COUNTING (NONE and THIN_DISC), or GB200_GEOMETRY_THIN_DISC_ORDER, which always counts.
// Every other instantiation compiles exactly the code it had before the counter existed.
constexpr int GB_GEOM_COUNTING = 16;
template <int GEOM> GB_HD constexpr bool gb_counts() { return GEOM >= GB_GEOM_COUNTING || GEOM == GB200_GEOMETRY_THIN_DISC_ORDER; }
// the disc whose condition the kernel evaluates: the order-n image is the thin disc's wedge
template <int GEOM> GB_HD constexpr int gb_disc_kind() {
    return GEOM == GB200_GEOMETRY_THIN_DISC_ORDER ? GB200_GEOMETRY_THIN_DISC : (GEOM >= GB_GEOM_COUNTING ? GEOM - GB_GEOM_COUNTING : GEOM);
}

template <int METRIC, int GEOM>
__global__ void __launch_bounds__(GB_BLOCK, GB_MIN_BLOCKS) gb200_trace_kernel(const __grid_constant__ GbParams P) {
    constexpr bool COUNT = gb_counts<GEOM>();
    constexpr bool ORDER = GEOM == GB200_GEOMETRY_THIN_DISC_ORDER;
    constexpr int DISC = gb_disc_kind<GEOM>();
    const unsigned lane = threadIdx.x & 31u;
    const double abstol = P.abstol, reltol = P.reltol;
    const double tstop = P.lam1;
    const double dtmax = P.dtmax;
    const double dtmin = 2.220446049250313e-16;
    const double beta1 = 7.0 / 50.0, beta2 = 2.0 / 25.0, gamma = 9.0 / 10.0, qmin = 1.0 / 5.0, qmax = 10.0;
    const double log_qoldinit = -9.210340371976182; // log(1e-4)

    // ---- per-lane integrator state (registers)
    double lam = 0;                                                         // affine parameter at u_prev (integrator.t)
    double ct = 0, r = 0, th = 0, ph = 0, vt = 0, vr = 0, vth = 0, vph = 0; // u_prev (ct = coordinate time x^t)
    double nct = 0, nr = 0, nth = 0, nph = 0, nvt = 0, nvr = 0, nvth = 0, nvph = 0; // u (proposed / final)
    GbK kA0, kA1, kA2, kA3; // accelerations: get(0) = FSAL k1, get(1..5) = k2..k6, get(6) = k7
    GbK kR, kT;             // stage velocities v^r, v^theta of k2..k6 (k1, k7 unused: those are vr, vth and nvr, nvth)
    double dt = 0, cprev = 1, acos_prev = 1, ev_lo = 0, ev_hi = 0;
    double qoldpow = 1; // controller memory: beta2 * log(qold) (POW_EXACT) or qold^beta2 (POW_FAST32)
    double tfinal = 0;
    double E_obs = 0, area = 1; // per-ray constants fixed at refill (redshift numerator, image-plane area weight)
    double hgt = P.gp0;         // datum-plane height of this ray (only read when GEOM is the datum plane)
    int state = LANE_EMPTY, pend_status = GB200_STATUS_NO_STATUS;
    bool pend_event = false;
    int naccept = 0, nreject = 0, flags = 0;
    int64_t slot = -1;
    const int maxit = (int)(P.maxiters < 0x7fffffff ? P.maxiters : 0x7fffffff); // step attempts are counted in 32 bits
    bool exhausted = false;
    unsigned long long tot_acc = 0, tot_rej = 0, tot_flag = 0;
    // COUNT: equatorial crossings of the accepted steps so far and the sign of cos(theta) at u_prev; ORDER: the image order
    int crossings = 0;
    bool cpos_prev = true;
    const int order = ORDER ? (int)P.gp2 : 0;
    // k2..k6 of the four accelerations and of the r, theta stage velocities: 30 rows; rows 30..33 park the k7
    // accelerations of a lane whose step ended in a disc event until it is finalised.
    __shared__ double sh_k[34][GB_BLOCK];
    kA0.p = &sh_k[0][threadIdx.x]; kA1.p = &sh_k[5][threadIdx.x]; kA2.p = &sh_k[10][threadIdx.x]; kA3.p = &sh_k[15][threadIdx.x];
    kR.p = &sh_k[20][threadIdx.x]; kT.p = &sh_k[25][threadIdx.x];
    kR.k1 = kR.k7 = kT.k1 = kT.k7 = 0.0;
#pragma unroll
    for (int j = 0; j < 34; ++j) sh_k[j][threadIdx.x] = 0.0;
#pragma unroll
    for (int j = 0; j < 7; ++j) { kA0.set(j, 0.0); kA1.set(j, 0.0); kA2.set(j, 0.0); kA3.set(j, 0.0); }
#pragma unroll
    for (int j = 1; j < 6; ++j) { kR.set(j, 0.0); kT.set(j, 0.0); }

    extern __shared__ unsigned long long sh_hist[]; // 2 * lp_nbins words when the line-profile histogram is fused, else empty
    if (P.lp_bins)
        for (int b = threadIdx.x; b < 2 * P.lp_nbins; b += GB_BLOCK) sh_hist[b] = 0ull;
    unsigned loop_count = 0;
    __shared__ int sh_exhausted;
    if (threadIdx.x == 0) sh_exhausted = 0;
    __syncthreads();
    for (;;) {
        // A barrier every GB_SYNC_EVERY-th step attempt: the warps of a CTA walk the (long, straight-line) step code
        // together and share its instruction-cache lines, and the decision to run the cold service code is CTA-uniform,
        // so that code is fetched once per CTA instead of once per warp.
        bool service = false;
        if ((loop_count++ % GB_SYNC_EVERY) == 0) {
            const int idle_cta = __syncthreads_count(state != LANE_RUN);
            service = idle_cta >= GB_REFILL_THRESH * (GB_BLOCK / 32) || idle_cta == GB_BLOCK;
        }
        if (service) {
            // ================= finalise terminated lanes =================
            if (state == LANE_PENDING) {
                int status = pend_status;
                if (DISC != GB200_GEOMETRY_NONE && pend_event) {
                    kA0.k7 = sh_k[30][threadIdx.x]; kA1.k7 = sh_k[31][threadIdx.x]; kA2.k7 = sh_k[32][threadIdx.x]; kA3.k7 = sh_k[33][threadIdx.x];
                    // ContinuousCallback root find on the dense output (DiffEqBase find_callback_time, LeftRootFind)
                    double C2r, C3r, C4r, C2t, C3t, C4t;
                    dense_coeffs(vr, kR, nvr, C2r, C3r, C4r);
                    dense_coeffs(vth, kT, nvth, C2t, C3t, C4t);
                    const double sprev = sgn(cprev);
                    double lo = ev_lo, hi = ev_hi;
                    double flo, fhi;
                    {
                        double s_, c_;
                        if (lo > 0.0) {
                            gb_sincos(dense_eval(th, dt, lo, vth, C2t, C3t, C4t), &s_, &c_);
                            flo = disc_condition<DISC>(P, dense_eval(r, dt, lo, vr, C2r, C3r, C4r), s_, c_, hgt);
                        } else flo = cprev;
                        gb_sincos(dense_eval(th, dt, hi, vth, C2t, C3t, C4t), &s_, &c_);
                        fhi = disc_condition<DISC>(P, dense_eval(r, dt, hi, vr, C2r, C3r, C4r), s_, c_, hgt);
                    }
                    if (fhi == 0.0) lo = hi;
                    else {
                        int side = 0;
#pragma unroll 1
                        for (int it = 0; it < 100; ++it) {
                            const double w = hi - lo;
                            if (w <= 1e-15) break;
                            // Illinois-modified regula falsi, falling back to bisection for the discontinuous case
                            double mid = (it < 40 && flo * fhi < 0.0) ? (lo * fhi - hi * flo) / (fhi - flo) : 0.5 * (lo + hi);
                            if (!(mid > lo && mid < hi)) mid = 0.5 * (lo + hi);
                            if (!(mid > lo && mid < hi)) break;
                            double s_, c_;
                            gb_sincos(dense_eval(th, dt, mid, vth, C2t, C3t, C4t), &s_, &c_);
                            const double fm = disc_condition<DISC>(P, dense_eval(r, dt, mid, vr, C2r, C3r, C4r), s_, c_, hgt);
                            if (fm != 0.0 && (fm > 0.0) == (sprev > 0.0)) {
                                lo = mid; flo = fm;
                                if (side == -1) fhi *= 0.5;
                                side = -1;
                            } else {
                                hi = mid; fhi = fm;
                                if (fm == 0.0) { fhi = -sprev * 1e-300; }
                                if (side == 1) flo *= 0.5;
                                side = 1;
                            }
                        }
                    }
                    // change_t_via_interpolation!: full state from the Tsit5 interpolant at Theta = lo
                    const double Th = lo, Th2 = Th * Th;
                    double b[7];
                    b[0] = Th * fma(Th, fma(Th, fma(Th, GB_C(R14), GB_C(R13)), GB_C(R12)), 1.0);
                    b[1] = Th2 * fma(Th, fma(Th, GB_C(R24), GB_C(R23)), GB_C(R22));
                    b[2] = Th2 * fma(Th, fma(Th, GB_C(R34), GB_C(R33)), GB_C(R32));
                    b[3] = Th2 * fma(Th, fma(Th, GB_C(R44), GB_C(R43)), GB_C(R42));
                    b[4] = Th2 * fma(Th, fma(Th, GB_C(R54), GB_C(R53)), GB_C(R52));
                    b[5] = Th2 * fma(Th, fma(Th, GB_C(R64), GB_C(R63)), GB_C(R62));
                    b[6] = Th2 * fma(Th, fma(Th, GB_C(R74), GB_C(R73)), GB_C(R72));
                    // stage v^t, v^phi are recomputed from the stored accelerations (bitwise the same values)
                    double W0[7], W3[7], WR[7], WT[7];
                    double st = 0, sr = 0, sth = 0, sph = 0, s0 = 0, s1 = 0, s2 = 0, s3 = 0;
                    W0[0] = vt; W3[0] = vph; WR[0] = vr; WT[0] = vth;
                    W0[1] = comb<1>(vt, dt, kA0.get(0), kA0); W3[1] = comb<1>(vph, dt, kA3.get(0), kA3);
                    W0[2] = comb<2>(vt, dt, kA0.get(0), kA0); W3[2] = comb<2>(vph, dt, kA3.get(0), kA3);
                    W0[3] = comb<3>(vt, dt, kA0.get(0), kA0); W3[3] = comb<3>(vph, dt, kA3.get(0), kA3);
                    W0[4] = comb<4>(vt, dt, kA0.get(0), kA0); W3[4] = comb<4>(vph, dt, kA3.get(0), kA3);
                    W0[5] = comb<5>(vt, dt, kA0.get(0), kA0); W3[5] = comb<5>(vph, dt, kA3.get(0), kA3);
                    W0[6] = nvt; W3[6] = nvph; WR[6] = nvr; WT[6] = nvth;
#pragma unroll
                    for (int j = 1; j < 6; ++j) { WR[j] = kR.get(j); WT[j] = kT.get(j); }
#pragma unroll
                    for (int j = 0; j < 7; ++j) {
                        st = fma(b[j], W0[j], st); sr = fma(b[j], WR[j], sr); sth = fma(b[j], WT[j], sth); sph = fma(b[j], W3[j], sph);
                        s0 = fma(b[j], kA0.get(j), s0); s1 = fma(b[j], kA1.get(j), s1); s2 = fma(b[j], kA2.get(j), s2); s3 = fma(b[j], kA3.get(j), s3);
                    }
                    nct = fma(dt, st, ct); nr = fma(dt, sr, r); nth = fma(dt, sth, th); nph = fma(dt, sph, ph);
                    nvt = fma(dt, s0, vt); nvr = fma(dt, s1, vr); nvth = fma(dt, s2, vth); nvph = fma(dt, s3, vph);
                    tfinal = fma(Th, dt, tfinal); // tfinal held lambda_prev for event lanes
                    status = GB200_STATUS_INTERSECTED_WITH_GEOMETRY;
                    // DiscreteCallbacks still run on the event state (handle_callbacks!): user, then chart
                    if (P.callback_kind == GB200_CALLBACK_UPPER_HEMISPHERE && nr * cos(nth) < P.callback_delta) status = GB200_STATUS_OUT_OF_DOMAIN;
                    if (nr <= P.chart_inner) status = GB200_STATUS_WITHIN_INNER_BOUNDARY;
                    else if (nr > P.chart_outer) status = GB200_STATUS_OUT_OF_DOMAIN;
                }
                // ---- store: GeodesicPoint fields, point functions, line-profile samples
                const int64_t n = slot;
                const bool failed = flags != 0; // integrator failure: last accepted state
                const double xe[4] = {failed ? ct : nct, failed ? r : nr, failed ? th : nth, failed ? ph : nph};
                const double ve[4] = {failed ? vt : nvt, failed ? vr : nvr, failed ? vth : nvth, failed ? vph : nvph};
                if (P.o_status) P.o_status[n] = status;
                if (P.o_lambda) P.o_lambda[n] = tfinal;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (P.o_x[k]) P.o_x[k][n] = xe[k];
                    if (P.o_v[k]) P.o_v[k][n] = ve[k];
                }
                if (P.o_naccept) P.o_naccept[n] = naccept;
                if (P.o_nreject) P.o_nreject[n] = nreject;
                if (P.o_flags) P.o_flags[n] = flags;
                tot_acc += (unsigned)naccept; tot_rej += (unsigned)nreject; tot_flag += (flags != 0);
                if (P.npf > 0 || P.o_g != nullptr || P.lp_bins != nullptr) {
                    const bool hit = (status == GB200_STATUS_INTERSECTED_WITH_GEOMETRY);
                    double g_red = nan("");
                    bool have_g = false;
                    for (int k = 0; k < P.npf; ++k) {
                        double val = nan("");
                        const int pf = P.pf[k];
                        if (pf == GB200_PF_SHADOW) { if (tfinal < P.lam1) val = tfinal; }
                        else if (pf == GB200_PF_REDSHIFT) {
                            if (hit) { if (!have_g) { g_red = redshift_endpoint<METRIC>(P, xe, ve, E_obs); have_g = true; } val = g_red; }
                        } else if (pf == GB200_PF_DISC_RADIUS) { if (hit) val = xe[1] * fabs(sin(xe[2])); }
                        else if (pf == GB200_PF_COORDINATE_TIME) { if (hit) val = xe[0]; }
                        else if (pf == GB200_PF_STATUS) val = (double)status;
                        else if (pf == GB200_PF_AFFINE_TIME) val = tfinal;
                        else if (pf == GB200_PF_RADIUS) val = xe[1] * fabs(sin(xe[2]));
                        else if (COUNT && pf == GB200_PF_EQUATORIAL_CROSSINGS) val = (double)crossings;
                        P.o_img[k][n] = val;
                    }
                    if (P.o_g || P.lp_bins) { // lineprofile BinningMethod, src/line-profiles.jl:186-194
                        double gg = nan(""), ff = 0.0;
                        if (hit) {
                            const double rho = xe[1] * fabs(sin(xe[2]));
                            if (P.min_re <= rho && rho <= P.max_re) {
                                gg = have_g ? g_red : redshift_endpoint<METRIC>(P, xe, ve, E_obs);
                                ff = emissivity_eval(P, rho) * gg * gg * gg * area;
                            }
                        }
                        if (P.o_g) { P.o_g[n] = gg; P.o_f[n] = ff; }
                        if (P.lp_bins && gg == gg) gb_hist_add(P, sh_hist, gg, ff);
                    }
                }
                state = LANE_EMPTY;
            }
            // ================= refill empty lanes from the work queue =================
            if (!exhausted) {
                const unsigned emask = __ballot_sync(FULLMASK, state == LANE_EMPTY);
                const int nfree = __popc(emask);
                unsigned long long base = 0;
                if (lane == 0) base = atomicAdd(P.queue, (unsigned long long)nfree);
                base = __shfl_sync(FULLMASK, base, 0);
                if (state == LANE_EMPTY) {
                    const int64_t ticket = (int64_t)base + __popc(emask & ((1u << lane) - 1u));
                    if (ticket < P.count) {
                        const int64_t s = slot_of_ticket(P, ticket);
                        slot = s;
                        GbRayInit ri;
                        ray_initial_state(P, ray_index_of_slot(P, s), ri);
                        lam = P.lam0; ct = ri.x[0]; r = ri.x[1]; th = ri.x[2]; ph = ri.x[3];
                        vt = ri.v[0]; vr = ri.v[1]; vth = ri.v[2]; vph = ri.v[3];
                        area = ri.area;
                        if (DISC == GB200_GEOMETRY_DATUM_PLANE && P.ic_kind == GB200_IC_IMPACT_PARAMETERS && P.ex[2])
                            hgt = P.ex[2][ray_index_of_slot(P, s)];
#pragma unroll
                        for (int k = 0; k < 4; ++k) { // GeodesicPoint.x_init / v_init are known now
                            if (P.o_x0[k]) P.o_x0[k][s] = ri.x[k];
                            if (P.o_v0[k]) P.o_v0[k][s] = ri.v[k];
                        }
                        if (P.ic_kind == GB200_IC_EXPLICIT) {
                            double go[5], sx, cx;
                            sincos(th, &sx, &cx);
                            metric_components_t<METRIC>(P, r, sx, cx, go);
                            E_obs = go[0] * vt + go[4] * vph;
                        } else E_obs = P.go[0] * vt + P.go[4] * vph;
                        naccept = 0; nreject = 0; flags = 0;
                        pend_event = false;
                        // f0 and the Hairer-Wanner initial step (ode_determine_initdt)
                        double acc[4], s_, c_;
                        rhs_accel<METRIC>(P, r, th, vt, vr, vth, vph, acc, s_, c_);
                        if (DISC != GB200_GEOMETRY_NONE) cprev = disc_condition<DISC>(P, r, s_, c_, hgt);
                        acos_prev = fabs(c_);
                        if (COUNT) { crossings = 0; cpos_prev = c_ >= 0.0; }
                        const double u0[8] = {ct, r, th, ph, vt, vr, vth, vph};
                        const double f0[8] = {vt, vr, vth, vph, acc[0], acc[1], acc[2], acc[3]};
                        double sk[8], d0 = 0, d1 = 0;
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
                            sk[k] = gb_rcp(fma(fabs(u0[k]), reltol, abstol)); // 1/sk
                            const double a0 = u0[k] * sk[k], a1 = f0[k] * sk[k];
                            d0 = fma(a0, a0, d0); d1 = fma(a1, a1, d1);
                        }
                        d0 = sqrt(d0 / 8.0); d1 = sqrt(d1 / 8.0);
                        double dt0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : (d0 / d1) / 100.0;
                        dt0 = fmin(dt0, dtmax);
                        double acc1[4];
                        rhs_accel<METRIC>(P, fma(dt0, vr, r), fma(dt0, vth, th), fma(dt0, acc[0], vt), fma(dt0, acc[1], vr),
                                          fma(dt0, acc[2], vth), fma(dt0, acc[3], vph), acc1, s_, c_);
                        const double f1[8] = {fma(dt0, acc[0], vt), fma(dt0, acc[1], vr), fma(dt0, acc[2], vth), fma(dt0, acc[3], vph),
                                              acc1[0], acc1[1], acc1[2], acc1[3]};
                        double d2 = 0;
#pragma unroll
                        for (int k = 0; k < 8; ++k) { const double a2 = (f1[k] - f0[k]) * sk[k]; d2 = fma(a2, a2, d2); }
                        d2 = sqrt(d2 / 8.0) / dt0;
                        const double md = fmax(d1, d2);
                        // 10^(-(2 + log10 md)/5) = (100 md)^(-1/5)
                        const double dt1 = (md <= 1e-15) ? fmax(1e-6, dt0 * 1e-3) : exp(-0.2 * log(100.0 * md));
                        dt = fmax(dtmin, fmin(fmin(100.0 * dt0, dt1), dtmax));
                        kA0.set(0, acc[0]); kA1.set(0, acc[1]); kA2.set(0, acc[2]); kA3.set(0, acc[3]);
                        qoldpow = (P.pow_mode == GB200_POW_FAST32) ? ctrl_pow_log(log_qoldinit, 1e-4, beta2, P.pow_mode) : beta2 * log_qoldinit;
                        state = LANE_RUN;
                    }
                }
                if ((int64_t)base + nfree >= P.count) {
                    exhausted = true;
                    if (lane == 0) *(volatile int*)&sh_exhausted = 1;
                }
            }
            const int running_cta = __syncthreads_count(state == LANE_RUN);
            exhausted = (*(volatile int*)&sh_exhausted) != 0; // written only inside a service pass, read only after its closing barrier
            if (running_cta == 0) break;                       // CTA-uniform: queue drained and every lane finalised
        }

        // ================= one Tsit5 step attempt for every running lane (straight-line: no taken branches) ==========
        if (state == LANE_RUN) {
            // dt arrives clamped to [dtmin, dtmax] (refill and commit do it); modify_dt_for_tstops! clips it to the end
            const double rem = tstop - lam;
            int fail = 0;
            if (naccept + nreject >= maxit) fail = GB200_FLAG_MAXITERS;
            else if (!(dt == dt) || !(r == r)) fail = GB200_FLAG_UNSTABLE;
            else if (!(gb_min(dt, rem) > dtmin) && rem > dtmin) fail = GB200_FLAG_DT_MIN;
            dt = gb_min(dt, rem);
            if (fail) { // integrator failure: the ray keeps NoStatus at its last accepted state (finalise reads u_prev for flagged rays)
                flags |= fail;
                tfinal = lam; pend_status = GB200_STATUS_NO_STATUS; pend_event = false; state = LANE_PENDING;
            }
        }
        if (state == LANE_RUN) {
            double acc[4], s_ = 0, c_ = 1;
            double tsum = GB_C(A71) * vt, psum = GB_C(A71) * vph; // sum_j a7j k_j[1], k_j[4]
            double terr = GB_C(BT1) * vt, perr = GB_C(BT1) * vph; // sum_j btilde_j k_j[1], k_j[4]
            // the other six error sums are accumulated stage by stage too (btilde_1 .. btilde_7 in order): their FMAs fill
            // the latency gaps of the next stage instead of forming a serial tail after the seventh
            double rerr = GB_C(BT1) * vr, therr = GB_C(BT1) * vth;
            double a0err = GB_C(BT1) * kA0.get(0), a1err = GB_C(BT1) * kA1.get(0), a2err = GB_C(BT1) * kA2.get(0), a3err = GB_C(BT1) * kA3.get(0);
            // running maxima of the high words of |k_j[r]|, |k_j[theta]| for the event-scan pre-test (no re-read from shared memory)
            int mxr = __double2hiint(vr) & 0x7fffffff, mxt = __double2hiint(vth) & 0x7fffffff;
#define GB_STAGE(S)                                                                                                     \
    {                                                                                                                   \
        const double xr = comb<S>(r, dt, vr, kR), xt = comb<S>(th, dt, vth, kT);                                        \
        const double w0 = comb<S>(vt, dt, kA0.get(0), kA0), w1 = comb<S>(vr, dt, kA1.get(0), kA1),                      \
                     w2 = comb<S>(vth, dt, kA2.get(0), kA2), w3 = comb<S>(vph, dt, kA3.get(0), kA3);                    \
        kR.set(S, w1); kT.set(S, w2);                                                                                   \
        mxr = max(mxr, __double2hiint(w1) & 0x7fffffff); mxt = max(mxt, __double2hiint(w2) & 0x7fffffff);              \
        tsum = fma(a7coef<S>(), w0, tsum); psum = fma(a7coef<S>(), w3, psum);                                           \
        terr = fma(btcoef<S>(), w0, terr); perr = fma(btcoef<S>(), w3, perr);                                           \
        rerr = fma(btcoef<S>(), w1, rerr); therr = fma(btcoef<S>(), w2, therr);                                         \
        rhs_accel<METRIC>(P, xr, xt, w0, w1, w2, w3, acc, s_, c_);                                                      \
        kA0.set(S, acc[0]); kA1.set(S, acc[1]); kA2.set(S, acc[2]); kA3.set(S, acc[3]);                                 \
        a0err = fma(btcoef<S>(), acc[0], a0err); a1err = fma(btcoef<S>(), acc[1], a1err);                               \
        a2err = fma(btcoef<S>(), acc[2], a2err); a3err = fma(btcoef<S>(), acc[3], a3err);                               \
    }
            GB_STAGE(1) GB_STAGE(2) GB_STAGE(3) GB_STAGE(4) GB_STAGE(5)
#undef GB_STAGE
            const double th6 = comb<5>(th, dt, vth, kT); // the sixth stage's polar angle (the compiler merges it with the stage's own)
            // 7th stage = the proposed state (FSAL)
            nr = comb<6>(r, dt, vr, kR); nth = comb<6>(th, dt, vth, kT);
            nvt = comb<6>(vt, dt, kA0.get(0), kA0); nvr = comb<6>(vr, dt, kA1.get(0), kA1);
            nvth = comb<6>(vth, dt, kA2.get(0), kA2); nvph = comb<6>(vph, dt, kA3.get(0), kA3);
            nct = fma(dt, tsum, ct); nph = fma(dt, psum, ph);
            terr = fma(GB_C(BT7), nvt, terr); perr = fma(GB_C(BT7), nvph, perr);
            rerr = fma(GB_C(BT7), nvr, rerr); therr = fma(GB_C(BT7), nvth, therr);
            // the eight error scales only need u_prev and u: they are formed while the seventh RHS is in flight
            const double is0 = gb_inv_scale(ct, nct, reltol, abstol), is1 = gb_inv_scale(r, nr, reltol, abstol);
            const double is2 = gb_inv_scale(th, nth, reltol, abstol), is3 = gb_inv_scale(ph, nph, reltol, abstol);
            const double is4 = gb_inv_scale(vt, nvt, reltol, abstol), is5 = gb_inv_scale(vr, nvr, reltol, abstol);
            const double is6 = gb_inv_scale(vth, nvth, reltol, abstol), is7 = gb_inv_scale(vph, nvph, reltol, abstol);
            double ee = 0;
            {
                double q_;
                q_ = terr * is0; ee = fma(q_, q_, ee);
                q_ = rerr * is1; ee = fma(q_, q_, ee);
                q_ = therr * is2; ee = fma(q_, q_, ee);
                q_ = perr * is3; ee = fma(q_, q_, ee);
            }
            rhs_accel_near<METRIC>(P, nr, nth, nvt, nvr, nvth, nvph, th6, s_, c_, acc, s_, c_);
            kA0.set(6, acc[0]); kA1.set(6, acc[1]); kA2.set(6, acc[2]); kA3.set(6, acc[3]);
            // ---- error estimate: rms( dt*sum btilde_j k_j / (abstol + max(|u_prev|,|u|) reltol) )
            {
                double q_;
                q_ = fma(GB_C(BT7), acc[0], a0err) * is4; ee = fma(q_, q_, ee);
                q_ = fma(GB_C(BT7), acc[1], a1err) * is5; ee = fma(q_, q_, ee);
                q_ = fma(GB_C(BT7), acc[2], a2err) * is6; ee = fma(q_, q_, ee);
                q_ = fma(GB_C(BT7), acc[3], a3err) * is7; ee = fma(q_, q_, ee);
            }
            // EEst^2 = dt^2 sum_i (.)^2 / 8; the controller only needs log EEst = log(EEst^2) / 2 and the test EEst <= 1, so no
            // square root is taken (the Float32 controller mode takes it where it needs EEst itself).  An exactly zero
            // estimate is raised to 1e-150: the controller clamps q to 1/qmax and qold to 1e-4 either way.
            const double EEst2 = gb_max((dt * dt) * (ee * 0.125), 1e-300);
            // PI controller (stepsize_controller!, OrdinaryDiffEq): q = EEst^beta1 / qold^beta2 / gamma, clamped; a rejected
            // attempt uses EEst^beta1 / gamma (step_reject_controller!).  One log and one exp serve both:
            // exp(beta1 log EEst - [accepted] beta2 log qold).
            const bool accept = gb_le_one(EEst2);
            const bool fast32 = (P.pow_mode == GB200_POW_FAST32);
            const double logE = 0.5 * gb_log_pos_lo(EEst2);
            double EEst = 1.0; // only the Float32 mode reads it
            if (fast32) EEst = gb_sqrt_pos(EEst2);
            double Epow;
            if (fast32) {
                Epow = ctrl_pow_log(logE, EEst, beta1, P.pow_mode);
                if (accept) Epow *= gb_rcp(qoldpow);
            } else {
                const double arg = accept ? fma(beta1, logE, -qoldpow) : beta1 * logE; // qoldpow = beta2 * log(qold) in this mode
                const double carg = gb_max(-8.0, gb_min(8.0, arg));
                Epow = gb_exp_small_lo(carg); // q is clamped to [1/qmax, 1/qmin] = exp(-2.2 .. 1.7) afterwards
            }
            const double q = gb_max(1.0 / qmax, gb_min(1.0 / qmin, Epow * (1.0 / gamma)));
            // ---- accept / reject, callbacks and the commit of the step.  Everything up to the commit is computed
            // unconditionally and committed with selects: the loop-carried state then lives in the same registers on
            // every path (the branchy form cost ~200 register moves per attempt where the paths merged).
            // Measured alternatives (profiles/r02_tuning_log.md): forming 1/q directly, with no reciprocal here and no
            // division in dtrej, was within the spread; one Newton step instead of gb_rcp's third-order correction gained nothing.
            const double dtnew = dt * gb_rcp(q);
            const double ttmp = lam + dt;
            const double tnew = (fabs(ttmp - tstop) < 100.0 * (fabs(tstop) * 2.220446049250313e-16)) ? tstop : ttmp;
            const double dtprop = gb_max(gb_min(dtmax, dtnew), dtmin);
            double dtrej = dt;
            if (!accept) dtrej = gb_max(dt / gb_min(1.0 / qmin, Epow / gamma), dtmin);
            // ---- callbacks: continuous (disc) first, then discrete (user, chart)
            bool event = false;
            double cnext = 1.0;
            if (DISC != GB200_GEOMETRY_NONE) {
                cnext = disc_condition<DISC>(P, nr, s_, c_, hgt);
                const double sprev = sgn(cprev);
                // the order-n image: only an entry into the wedge (sprev > 0) in a step that starts with n crossings is an
                // event; inside the wedge, before the n-th crossing and after it, the event test and the scan are skipped
                if (accept && (ORDER ? (sprev > 0.0 && crossings == order) : sprev != 0.0)) {
                    if (sprev * sgn(cnext) <= 0.0) { event = true; ev_lo = 0.0; ev_hi = 1.0; }
                    else {
                        // cheap bound first: |u(Th) - u0| <= |dt| * L * max_j |k_j| with L = max_Th sum_j |b_j(Th)| = 7.5822
                        // for the Tsit5 dense output; only when it is inconclusive are the polynomial coefficients formed
                        const double adt = fabs(dt);
                        // max_j |k_j| bounded from the high words alone (integer pipe): doubles order like their bit
                        // patterns, and (hi + 1, 0) exceeds every double whose high word is hi.  inf/nan give a nan bound,
                        // which the comparisons in scan_needed treat as "cannot skip".
                        const double mth = __hiloint2double(max(mxt, __double2hiint(nvth) & 0x7fffffff) + 1, 0);
                        const double mr = __hiloint2double(max(mxr, __double2hiint(nvr) & 0x7fffffff) + 1, 0);
                        bool need = (!ORDER && sprev < 0.0) || scan_needed<DISC>(P, r, acos_prev, cprev, adt * 7.5823 * mth, adt * 7.5823 * mr);
                        double C2r = 0, C3r = 0, C4r = 0, C2t = 0, C3t = 0, C4t = 0;
                        if (need) {
                            dense_coeffs(vth, kT, nvth, C2t, C3t, C4t);
                            dense_coeffs(vr, kR, nvr, C2r, C3r, C4r);
                            const double Bth = adt * (fabs(vth) + fabs(C2t) + fabs(C3t) + fabs(C4t));
                            const double Br = adt * (fabs(vr) + fabs(C2r) + fabs(C3r) + fabs(C4r));
                            need = (!ORDER && sprev < 0.0) || scan_needed<DISC>(P, r, acos_prev, cprev, Bth, Br);
                        }
                        if (need) {
#pragma unroll 1
                            for (int i = 1; i <= 6; ++i) { // interp_points = 8: Theta = 1/7 .. 6/7 (7/7 is u itself)
                                const double Th = (double)i / 7.0;
                                double si, ci;
                                gb_sincos(dense_eval(th, dt, Th, vth, C2t, C3t, C4t), &si, &ci);
                                const double cn = disc_condition<DISC>(P, dense_eval(r, dt, Th, vr, C2r, C3r, C4r), si, ci, hgt);
                                if (sprev * cn < 0.0) { event = true; ev_lo = (double)(i - 1) / 7.0; ev_hi = Th; break; }
                            }
                        }
                    }
                }
            }
            if (DISC != GB200_GEOMETRY_NONE && event) { // k2..k6 are in shared memory already; k7 joins them
                sh_k[30][threadIdx.x] = kA0.k7; sh_k[31][threadIdx.x] = kA1.k7; sh_k[32][threadIdx.x] = kA2.k7; sh_k[33][threadIdx.x] = kA3.k7;
            }
            int status = GB200_STATUS_NO_STATUS;
            bool term = false;
            if (P.callback_kind == GB200_CALLBACK_UPPER_HEMISPHERE && nr * c_ < P.callback_delta) { status = GB200_STATUS_OUT_OF_DOMAIN; term = true; }
            if (nr <= P.chart_inner) { status = GB200_STATUS_WITHIN_INNER_BOUNDARY; term = true; }
            else if (nr > P.chart_outer) { status = GB200_STATUS_OUT_OF_DOMAIN; term = true; }
            if (!(tnew < tstop)) term = true; // reached lambda_max: NoStatus unless a callback fired
            const bool finish = accept && (event || term);
            const bool advance = accept && !finish; // apply_step!: u_prev <- u, FSAL
            naccept += accept ? 1 : 0;
            nreject += accept ? 0 : 1;
            if (accept) { // controller memory
                if (fast32) qoldpow = ctrl_pow_log(fmax(logE, log_qoldinit), fmax(EEst, 1e-4), beta2, P.pow_mode);
                else qoldpow = beta2 * gb_max(logE, log_qoldinit);
            }
            // an event keeps u_prev, the stage data and dt (= the step's dt) in registers: the root find happens at
            // finalise; tfinal holds lambda_prev for event lanes, the end of the step otherwise
            tfinal = event ? lam : tnew;
            pend_event = event;
            pend_status = event ? GB200_STATUS_INTERSECTED_WITH_GEOMETRY : status;
            state = finish ? LANE_PENDING : LANE_RUN;
            lam = advance ? tnew : lam;
            ct = advance ? nct : ct; r = advance ? nr : r; th = advance ? nth : th; ph = advance ? nph : ph;
            vt = advance ? nvt : vt; vr = advance ? nvr : vr; vth = advance ? nvth : vth; vph = advance ? nvph : vph;
            kA0.set(0, advance ? kA0.get(6) : kA0.get(0)); kA1.set(0, advance ? kA1.get(6) : kA1.get(0));
            kA2.set(0, advance ? kA2.get(6) : kA2.get(0)); kA3.set(0, advance ? kA3.get(6) : kA3.get(0));
            cprev = advance ? cnext : cprev; acos_prev = advance ? fabs(c_) : acos_prev;
            if (COUNT) { // every accepted step counts except one that ends in a disc event (the ray stops at u_prev + a root)
                const bool cpos = c_ >= 0.0;
                crossings += (accept && !event && cpos != cpos_prev) ? 1 : 0;
                cpos_prev = advance ? cpos : cpos_prev;
            }
            dt = advance ? dtprop : (accept ? dt : dtrej);
        }
    }
    if (P.lp_bins) { // this CTA's histogram joins the launch's (carry-correct 128-bit adds: order independent)
        __syncthreads();
        for (int b = threadIdx.x; b < P.lp_nbins; b += GB_BLOCK) {
            const unsigned long long wlo = sh_hist[b], whi = sh_hist[P.lp_nbins + b];
            if (wlo | whi) gb_acc128(&P.lp_acc[b], &P.lp_acc[P.lp_nbins + b], wlo, whi);
        }
    }
    // ---- flush per-thread counters (warp-reduced)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        tot_acc += __shfl_down_sync(FULLMASK, tot_acc, o);
        tot_rej += __shfl_down_sync(FULLMASK, tot_rej, o);
        tot_flag += __shfl_down_sync(FULLMASK, tot_flag, o);
    }
    if (lane == 0 && P.counters) {
        atomicAdd(&P.counters[0], tot_acc);
        atomicAdd(&P.counters[1], tot_rej);
        if (tot_flag) atomicAdd(&P.counters[2], tot_flag);
    }
}

// ---------------------------------------------------------------- launch
template <int METRIC, int GEOM>
static cudaError_t launch_one(const GbParams& P, int sm_count, cudaStream_t stream, int* blocks_out) {
    int per_sm = 0;
    const size_t dyn = P.lp_bins ? sizeof(unsigned long long) * 2 * (size_t)P.lp_nbins : 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gb200_trace_kernel<METRIC, GEOM>, GB_BLOCK, dyn);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    long long want = ((long long)P.count + GB_BLOCK - 1) / GB_BLOCK;
    long long grid = (long long)sm_count * per_sm; // persistent: one wave, sized in multiples of the SM count
    if (want < grid) grid = want > 0 ? want : 1;
    if (blocks_out) *blocks_out = (int)grid;
    gb200_trace_kernel<METRIC, GEOM><<<(unsigned)grid, GB_BLOCK, dyn, stream>>>(P);
    return cudaGetLastError();
}

template <int METRIC>
static cudaError_t launch_geom(const GbParams& P, int sm_count, cudaStream_t stream, int* blocks_out) {
    bool count = false; // the counting instantiations run only for calls that ask for the crossings
    for (int k = 0; k < P.npf; ++k) count = count || P.pf[k] == GB200_PF_EQUATORIAL_CROSSINGS;
    if (count && P.geometry_kind == GB200_GEOMETRY_NONE)
        return launch_one<METRIC, GB200_GEOMETRY_NONE + GB_GEOM_COUNTING>(P, sm_count, stream, blocks_out);
    if (count && P.geometry_kind == GB200_GEOMETRY_THIN_DISC)
        return launch_one<METRIC, GB200_GEOMETRY_THIN_DISC + GB_GEOM_COUNTING>(P, sm_count, stream, blocks_out);
    if (count && P.geometry_kind != GB200_GEOMETRY_THIN_DISC_ORDER) return cudaErrorInvalidValue; // the host rejects this first
    switch (P.geometry_kind) {
    case GB200_GEOMETRY_NONE: return launch_one<METRIC, GB200_GEOMETRY_NONE>(P, sm_count, stream, blocks_out);
    case GB200_GEOMETRY_THIN_DISC: return launch_one<METRIC, GB200_GEOMETRY_THIN_DISC>(P, sm_count, stream, blocks_out);
    case GB200_GEOMETRY_THIN_DISC_ORDER: return launch_one<METRIC, GB200_GEOMETRY_THIN_DISC_ORDER>(P, sm_count, stream, blocks_out);
    case GB200_GEOMETRY_SHAKURA_SUNYAEV: return launch_one<METRIC, GB200_GEOMETRY_SHAKURA_SUNYAEV>(P, sm_count, stream, blocks_out);
    case GB200_GEOMETRY_DATUM_PLANE: return launch_one<METRIC, GB200_GEOMETRY_DATUM_PLANE>(P, sm_count, stream, blocks_out);
    case GB200_GEOMETRY_THICK_TABLE: return launch_one<METRIC, GB200_GEOMETRY_THICK_TABLE>(P, sm_count, stream, blocks_out);
    }
    return cudaErrorInvalidValue;
}

cudaError_t gb200_launch_trace(const GbParams& P, int sm_count, cudaStream_t stream, int* blocks_out) {
    switch (P.metric_kind) {
    case GB200_METRIC_KERR: return launch_geom<GB200_METRIC_KERR>(P, sm_count, stream, blocks_out);
    case GB200_METRIC_JOHANNSEN_PSALTIS: return launch_geom<GB200_METRIC_JOHANNSEN_PSALTIS>(P, sm_count, stream, blocks_out);
    case GB200_METRIC_JOHANNSEN: return launch_geom<GB200_METRIC_JOHANNSEN>(P, sm_count, stream, blocks_out);
    case GB200_METRIC_BUMBLEBEE: return launch_geom<GB200_METRIC_BUMBLEBEE>(P, sm_count, stream, blocks_out);
    case GB200_METRIC_KERR_NEWMAN: return launch_geom<GB200_METRIC_KERR_NEWMAN>(P, sm_count, stream, blocks_out);
    case GB200_METRIC_MORRIS_THORNE: return launch_geom<GB200_METRIC_MORRIS_THORNE>(P, sm_count, stream, blocks_out);
    case GB200_METRIC_DILATON_AXION: return launch_geom<GB200_METRIC_DILATON_AXION>(P, sm_count, stream, blocks_out);
    }
    return cudaErrorInvalidValue;
}

// ---------------------------------------------------------------- line-profile histogram (Buckets.bucket(Simple(), g, f, bins))
// Shared-memory FP64 bins; lanes of a warp that hit the same bin are combined first
// (__match_any_sync) so one shared atomic per distinct bin per warp is issued; each block
// then writes its partial histogram to its own row and a second kernel sums the rows in a
// fixed order, so the result does not depend on atomic arrival order across blocks.
__global__ void __launch_bounds__(256) gb200_hist_kernel(const double* __restrict__ g, const double* __restrict__ f, int64_t n,
                                                         const double* __restrict__ bins, int nbins, int right_closed,
                                                         double* __restrict__ partial, int hist_rows) {
    extern __shared__ double sh[];
    double* sbins = sh;
    // one histogram row per warp when they fit (rows = warps per block), else one row for the block: with a row of
    // its own a warp's additions happen in program order, so the block's result does not depend on which warp's
    // atomic arrives first and the whole histogram is bitwise reproducible
    const int rows = hist_rows;
    double* shist = sh + nbins + (rows > 1 ? (int)(threadIdx.x >> 5) * nbins : 0);
    for (int b = threadIdx.x; b < nbins; b += blockDim.x) sbins[b] = bins[b];
    for (int b = threadIdx.x; b < nbins * rows; b += blockDim.x) sh[nbins + b] = 0.0;
    __syncthreads();
    const unsigned lane = threadIdx.x & 31u;
    const int64_t per_block = (n + gridDim.x - 1) / gridDim.x;
    const int64_t begin = (int64_t)blockIdx.x * per_block;
    const int64_t end = (begin + per_block < n) ? begin + per_block : n;
    for (int64_t base = begin; base < end; base += blockDim.x) {
        const int64_t i = base + threadIdx.x;
        int bin = -1;
        double val = 0.0;
        if (i < end) {
            const double gi = g[i];
            if (gi == gi) {
                int lo = 0, hi = nbins; // right_closed: first idx with bins[idx] >= g ; else first idx with bins[idx] > g, minus 1
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    const bool go_right = right_closed ? (sbins[mid] < gi) : (sbins[mid] <= gi);
                    if (go_right) lo = mid + 1; else hi = mid;
                }
                bin = right_closed ? lo : lo - 1;
                bin = bin < 0 ? 0 : (bin > nbins - 1 ? nbins - 1 : bin);
                val = f[i];
            }
        }
        // warp aggregation: leader (lowest lane of each equal-bin group) adds the group's sum in lane order
        const unsigned active = __ballot_sync(FULLMASK, bin >= 0);
        if (bin >= 0) {
            const unsigned peers = __match_any_sync(active, bin);
            const int leader = __ffs(peers) - 1;
            double sum = 0.0;
            unsigned rem = peers;
            while (rem) { // fixed lane order -> deterministic group sum
                const int src = __ffs(rem) - 1;
                sum += __shfl_sync(peers, val, src);
                rem &= rem - 1;
            }
            if ((int)lane == leader) atomicAdd(&shist[bin], sum);
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b < nbins; b += blockDim.x) {
        double s = 0.0;
        for (int w = 0; w < rows; ++w) s += sh[nbins + w * nbins + b]; // fixed warp order
        partial[(size_t)blockIdx.x * nbins + b] = s;
    }
}

__global__ void gb200_hist_reduce_kernel(const double* __restrict__ partial, int nblocks, int nbins, double* __restrict__ out, int accumulate) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nbins) return;
    double s = 0.0;
    for (int k = 0; k < nblocks; ++k) s += partial[(size_t)k * nbins + b];
    out[b] = accumulate ? out[b] + s : s;
}

// (high, low) 128-bit fixed-point bins -> doubles: out[b] = (hi 2^64 + lo) / scale
__global__ void gb200_hist128_finish_kernel(const unsigned long long* __restrict__ acc, int nbins, double inv_scale, double* __restrict__ out) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < nbins) out[b] = fma((double)acc[nbins + b], 18446744073709551616.0, (double)acc[b]) * inv_scale;
}
cudaError_t gb200_launch_hist128_finish(const unsigned long long* acc, int nbins, double scale, double* out, cudaStream_t stream) {
    gb200_hist128_finish_kernel<<<(nbins + 127) / 128, 128, 0, stream>>>(acc, nbins, 1.0 / scale, out);
    return cudaGetLastError();
}

cudaError_t gb200_launch_hist(const double* g, const double* f, int64_t n, const double* bins, int nbins, int right_closed,
                              double* partial, int nblocks, double* out, cudaStream_t stream) {
    const int rows = ((size_t)nbins * 9 * sizeof(double) <= 96 * 1024) ? 8 : 1; // 256 threads = 8 warps
    const size_t smem = (size_t)nbins * (1 + rows) * sizeof(double);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(gb200_hist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    gb200_hist_kernel<<<nblocks, 256, smem, stream>>>(g, f, n, bins, nbins, right_closed, partial, rows);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    gb200_hist_reduce_kernel<<<(nbins + 127) / 128, 128, 0, stream>>>(partial, nblocks, nbins, out, 0);
    return cudaGetLastError();
}

// ---------------------------------------------------------------- two-dimensional bucket (lag-energy transfer functions)
// `bucket(energy, time, flux, energy_bins, time_bins; reduction = sum)` of bin_transfer_function
// (src/transfer-functions/transfer-functions-2d.jl:100-122, Buckets.Simple in both axes).  300 x 300 bins do not fit shared
// memory, so the bins live in HBM; to keep the result independent of the order in which atomics arrive (and of how the
// samples are split over GPUs) the weights are accumulated as 64-bit fixed-point integers -- integer addition is
// associative -- with the scale chosen from sum |w|, so that the quantisation (2^-62 of the total per sample) is far below
// the rounding of a floating-point sum.  Lanes of a warp that hit the same cell are combined first (__match_any_sync).
__global__ void __launch_bounds__(256) gb200_bucket2d_kernel(const double* __restrict__ x, const double* __restrict__ y, const double* __restrict__ w,
                                                             int64_t n, const double* __restrict__ xb, int nx, const double* __restrict__ yb, int ny,
                                                             double scale, long long* __restrict__ acc) {
    const unsigned lane = threadIdx.x & 31u;
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < n; base += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = base + threadIdx.x;
        int cell = -1;
        long long q = 0;
        if (i < n) {
            const double xi = x[i], yi = y[i], wi = w[i];
            if (xi == xi && yi == yi && wi == wi) {
                cell = gb_simple_bucket(xb, nx, xi) * ny + gb_simple_bucket(yb, ny, yi);
                q = __double2ll_rn(wi * scale);
            }
        }
        const unsigned active = __ballot_sync(FULLMASK, cell >= 0);
        if (cell >= 0) {
            const unsigned peers = __match_any_sync(active, cell);
            long long sum = 0;
            unsigned rem = peers;
            while (rem) { const int src = __ffs(rem) - 1; sum += __shfl_sync(peers, q, src); rem &= rem - 1; }
            if ((int)lane == __ffs(peers) - 1) atomicAdd((unsigned long long*)&acc[cell], (unsigned long long)sum);
        }
    }
}
__global__ void gb200_bucket2d_finish_kernel(const long long* __restrict__ acc, int ncell, double inv_scale, double* __restrict__ out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < ncell) out[c] = (double)acc[c] * inv_scale;
}
cudaError_t gb200_launch_bucket2d(const double* x, const double* y, const double* w, int64_t n, const double* xb, int nx, const double* yb, int ny,
                                  double scale, long long* acc, double* out, int blocks, cudaStream_t stream) {
    const int ncell = nx * ny;
    cudaError_t e = cudaMemsetAsync(acc, 0, sizeof(long long) * (size_t)ncell, stream);
    if (e != cudaSuccess) return e;
    if (n > 0) gb200_bucket2d_kernel<<<blocks, 256, 0, stream>>>(x, y, w, n, xb, nx, yb, ny, scale, acc);
    gb200_bucket2d_finish_kernel<<<(ncell + 255) / 256, 256, 0, stream>>>(acc, ncell, 1.0 / scale, out);
    return cudaGetLastError();
}

// ---------------------------------------------------------------- diagnostics
template <int METRIC>
__global__ void gb200_debug_rhs_kernel(const GbParams P, long long n, const double* __restrict__ u, double* __restrict__ du) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double acc[4], s_, c_;
    rhs_accel<METRIC>(P, u[8 * i + 1], u[8 * i + 2], u[8 * i + 4], u[8 * i + 5], u[8 * i + 6], u[8 * i + 7], acc, s_, c_);
    for (int k = 0; k < 4; ++k) { du[8 * i + k] = u[8 * i + 4 + k]; du[8 * i + 4 + k] = acc[k]; }
}
__global__ void gb200_debug_math_kernel(long long n, const double* __restrict__ x, double* __restrict__ out5) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double s_, c_;
    gb_sincos(x[i], &s_, &c_);
    out5[5 * i] = s_; out5[5 * i + 1] = c_; out5[5 * i + 2] = gb_rcp(x[i]);
    out5[5 * i + 3] = gb_log_pos(fabs(x[i]));
    out5[5 * i + 4] = gb_exp_small(fmax(-8.0, fmin(8.0, x[i])));
}
__global__ void gb200_debug_math_lo_kernel(long long n, const double* __restrict__ x, double* __restrict__ out2) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out2[2 * i] = gb_log_pos_lo(fabs(x[i]));
    out2[2 * i + 1] = gb_exp_small_lo(fmax(-8.0, fmin(8.0, x[i])));
}
cudaError_t gb200_launch_debug_math_lo(long long n, const double* d_x, double* d_out2, cudaStream_t stream) {
    gb200_debug_math_lo_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(n, d_x, d_out2);
    return cudaGetLastError();
}
cudaError_t gb200_launch_debug_rhs(const GbParams& P, long long n, const double* d_u, double* d_du, cudaStream_t stream) {
    const unsigned grid = (unsigned)((n + 127) / 128);
    switch (P.metric_kind) {
    case GB200_METRIC_KERR: gb200_debug_rhs_kernel<GB200_METRIC_KERR><<<grid, 128, 0, stream>>>(P, n, d_u, d_du); break;
    case GB200_METRIC_JOHANNSEN_PSALTIS: gb200_debug_rhs_kernel<GB200_METRIC_JOHANNSEN_PSALTIS><<<grid, 128, 0, stream>>>(P, n, d_u, d_du); break;
    case GB200_METRIC_JOHANNSEN: gb200_debug_rhs_kernel<GB200_METRIC_JOHANNSEN><<<grid, 128, 0, stream>>>(P, n, d_u, d_du); break;
    case GB200_METRIC_BUMBLEBEE: gb200_debug_rhs_kernel<GB200_METRIC_BUMBLEBEE><<<grid, 128, 0, stream>>>(P, n, d_u, d_du); break;
    case GB200_METRIC_MORRIS_THORNE: gb200_debug_rhs_kernel<GB200_METRIC_MORRIS_THORNE><<<grid, 128, 0, stream>>>(P, n, d_u, d_du); break;
    case GB200_METRIC_DILATON_AXION: gb200_debug_rhs_kernel<GB200_METRIC_DILATON_AXION><<<grid, 128, 0, stream>>>(P, n, d_u, d_du); break;
    default: gb200_debug_rhs_kernel<GB200_METRIC_KERR_NEWMAN><<<grid, 128, 0, stream>>>(P, n, d_u, d_du); break;
    }
    return cudaGetLastError();
}
cudaError_t gb200_launch_debug_math(long long n, const double* d_x, double* d_out5, cudaStream_t stream) {
    gb200_debug_math_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(n, d_x, d_out5);
    return cudaGetLastError();
}

// ---------------------------------------------------------------- FP64 peak micro-benchmark (roofline denominator)
__global__ void __launch_bounds__(256) gb200_dfma_kernel(double* out, int iters, double seed) {
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
            a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
        }
    }
    const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 12345.678) out[0] = s; // never true: keeps the chain alive
}

// The same DFMA stream with MIX independent integer-pipe instructions (LOP3) per DFMA: probes whether non-FP64
// instructions issue in the shadow of the two-cycle FP64 instructions or add to them.
template <int MIX>
__global__ void __launch_bounds__(256) gb200_dfma_mix_kernel(double* out, int iters, double seed) {
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    unsigned b0 = threadIdx.x, b1 = b0 + 1, b2 = b0 + 2, b3 = b0 + 3, b4 = b0 + 4, b5 = b0 + 5, b6 = b0 + 6, b7 = b0 + 7;
    const unsigned x = blockIdx.x | 1u, y = gridDim.x;
    const double m = 1.0000001, c = 1e-9;
#define GB_LOP(b) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(b) : "r"(x), "r"(y));
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
            a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
#pragma unroll
            for (int v = 0; v < MIX; ++v) { GB_LOP(b0) GB_LOP(b1) GB_LOP(b2) GB_LOP(b3) GB_LOP(b4) GB_LOP(b5) GB_LOP(b6) GB_LOP(b7) }
        }
    }
#undef GB_LOP
    const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    const unsigned t = b0 ^ b1 ^ b2 ^ b3 ^ b4 ^ b5 ^ b6 ^ b7;
    if (s == 12345.678 || t == 0xdeadbeefu) out[0] = s + t; // practically never true: keeps both chains alive
}
// DFMA / DMUL streams whose operands are all distinct vector registers (the probes above multiply by a uniform constant):
// mode 3 = DFMA a <- a * m_k + c_k with per-thread m_k, c_k; mode 4 = the same with DMUL + DADD pairs.
template <int MODE>
__global__ void __launch_bounds__(256) gb200_dfma_reg_kernel(double* out, int iters, double seed) {
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m0 = 1.0 + 1e-9 * threadIdx.x, m1 = m0 + 1e-9, m2 = m0 + 2e-9, m3 = m0 + 3e-9;
    const double c0 = 1e-9 * (threadIdx.x + 1), c1 = c0 * 2, c2 = c0 * 3, c3 = c0 * 4;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            if (MODE == 5) { // one register operand shared by consecutive DFMAs (operand reuse cache)
                a0 = fma(a0, m0, c0); a1 = fma(a1, m0, c1); a2 = fma(a2, m0, c2); a3 = fma(a3, m0, c3);
                a4 = fma(a4, m0, c1); a5 = fma(a5, m0, c2); a6 = fma(a6, m0, c3); a7 = fma(a7, m0, c0);
            } else if (MODE == 3) {
                a0 = fma(a0, m0, c0); a1 = fma(a1, m1, c1); a2 = fma(a2, m2, c2); a3 = fma(a3, m3, c3);
                a4 = fma(a4, m0, c1); a5 = fma(a5, m1, c2); a6 = fma(a6, m2, c3); a7 = fma(a7, m3, c0);
            } else {
                a0 = __dmul_rn(a0, m0); a1 = __dadd_rn(a1, c1); a2 = __dmul_rn(a2, m2); a3 = __dadd_rn(a3, c3);
                a4 = __dmul_rn(a4, m0); a5 = __dadd_rn(a5, c2); a6 = __dmul_rn(a6, m2); a7 = __dadd_rn(a7, c0);
            }
        }
    }
    const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 12345.678) out[0] = s;
}

cudaError_t gb200_launch_dfma_mix(double* d_out, int blocks, int iters, int mix, cudaStream_t stream) {
    if (mix == 3) { gb200_dfma_reg_kernel<3><<<blocks, 256, 0, stream>>>(d_out, iters, 0.5); return cudaGetLastError(); }
    if (mix == 4) { gb200_dfma_reg_kernel<4><<<blocks, 256, 0, stream>>>(d_out, iters, 0.5); return cudaGetLastError(); }
    if (mix == 5) { gb200_dfma_reg_kernel<5><<<blocks, 256, 0, stream>>>(d_out, iters, 0.5); return cudaGetLastError(); }
    if (mix == 0) gb200_dfma_mix_kernel<0><<<blocks, 256, 0, stream>>>(d_out, iters, 0.5);
    else if (mix == 1) gb200_dfma_mix_kernel<1><<<blocks, 256, 0, stream>>>(d_out, iters, 0.5);
    else if (mix == 2) gb200_dfma_mix_kernel<2><<<blocks, 256, 0, stream>>>(d_out, iters, 0.5);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}

cudaError_t gb200_launch_dfma(double* d_out, int blocks, int iters, cudaStream_t stream) {
    gb200_dfma_kernel<<<blocks, 256, 0, stream>>>(d_out, iters, 0.5);
    return cudaGetLastError();
}
