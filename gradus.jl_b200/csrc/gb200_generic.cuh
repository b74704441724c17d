// gb200_generic.cuh -- a second integrator beside the warp-cooperative one of gb200_trace.cu, written over a generic
// scalar: one ray per thread, plain loops, every quantity of the state a dual number GD<N> carrying N partial derivatives
// (N = 0: plain doubles).  The step loop and the right-hand sides are its own; the disc conditions, the endpoint
// redshift, the v^t constraint and the Tsit5 tableau are gb200_device.cuh's, instantiated on GD<N> (the overloads of
// gd_sqrt, gd_abs, gd_sin, gd_cos, gd_fmin and gd_fmax below keep each scalar type's own arithmetic).
//
// Two users:
//   * N = 1, 2: the forward-mode traces of the transfer-function solvers.  The reference pushes ForwardDiff duals through
//     the ODE solve: `_make_image_plane_mapper` (src/tracing/precision-solvers.jl:73-131) for the Newton derivative of
//     `_find_offset_for_radius` (:133-241) and `jacobian_∂αβ_∂gr` (:401-451) for |d(rho, g) / d(alpha, beta)|.
//   * N = 0 with a record hook: the single-geodesic path recorder (`save_on = true`, src/tracing/tracing.jl:66-108) behind
//     gb200_trace_path and the plunging-velocity table (src/orbits/orbit-solving.jl:137-167).
//
// Semantics are those of gb200_trace_kernel (Hairer-Wanner initial dt, Tsit5 with FSAL, PI controller, tstop snapping,
// ContinuousCallback with 8 interpolation points and a left-biased root find on the dense output, DiscreteCallbacks in
// the reference's order); tests/test_gpu_dual.py requires the N = 0 instantiation to reproduce the ensemble kernel's end
// points.  What a dual-valued state changes (DiffEqBase's ForwardDiff extension, un-vendored, restated):
//   * the error norm: ODE_DEFAULT_NORM(u) = sqrt(sum(value^2 + partials^2) / (length (1 + N))) for arrays and
//     sqrt(value^2 + sum partials^2) for one dual -- partials are error-controlled like values (norm_partials);
//   * control flow reads values only;
//   * the event time found on the dense output carries partials (the root find runs on dual-valued samples of the
//     condition): to first order Theta_p = -(dc/dp) / (dc/dTheta), so the end point slides along the ray and stays on
//     the surface as the parameters move.
#pragma once
#include "gb200_device.cuh"

template <int N>
struct GD {
    double v;
    double d[N > 0 ? N : 1];
    GB_HD GD() : v(0.0) { for (int i = 0; i < N; ++i) d[i] = 0.0; }
    GB_HD GD(double x) : v(x) { for (int i = 0; i < N; ++i) d[i] = 0.0; }
};
#define GD_T template <int N> GB_HD inline
GD_T GD<N> operator+(const GD<N>& a, const GD<N>& b) { GD<N> r; r.v = a.v + b.v; for (int i = 0; i < N; ++i) r.d[i] = a.d[i] + b.d[i]; return r; }
GD_T GD<N> operator-(const GD<N>& a, const GD<N>& b) { GD<N> r; r.v = a.v - b.v; for (int i = 0; i < N; ++i) r.d[i] = a.d[i] - b.d[i]; return r; }
GD_T GD<N> operator-(const GD<N>& a) { GD<N> r; r.v = -a.v; for (int i = 0; i < N; ++i) r.d[i] = -a.d[i]; return r; }
GD_T GD<N> operator*(const GD<N>& a, const GD<N>& b) { GD<N> r; r.v = a.v * b.v; for (int i = 0; i < N; ++i) r.d[i] = a.d[i] * b.v + a.v * b.d[i]; return r; }
// 1 / x: branch-free reciprocal (<= 1 ulp) on the device, where an IEEE division costs ~10x as many instructions
GB_HD inline double gd_inv(double x) {
#ifdef __CUDA_ARCH__
    return gb_rcp(x);
#else
    return 1.0 / x;
#endif
}
GD_T GD<N> operator/(const GD<N>& a, const GD<N>& b) {
    GD<N> r; const double ib = gd_inv(b.v); r.v = a.v * ib;
    for (int i = 0; i < N; ++i) r.d[i] = (a.d[i] - r.v * b.d[i]) * ib;
    return r;
}
GD_T GD<N> operator+(const GD<N>& a, double c) { GD<N> r = a; r.v += c; return r; }
GD_T GD<N> operator+(double c, const GD<N>& a) { GD<N> r = a; r.v += c; return r; }
GD_T GD<N> operator-(const GD<N>& a, double c) { GD<N> r = a; r.v -= c; return r; }
GD_T GD<N> operator-(double c, const GD<N>& a) { GD<N> r; r.v = c - a.v; for (int i = 0; i < N; ++i) r.d[i] = -a.d[i]; return r; }
GD_T GD<N> operator*(const GD<N>& a, double c) { GD<N> r; r.v = a.v * c; for (int i = 0; i < N; ++i) r.d[i] = a.d[i] * c; return r; }
GD_T GD<N> operator*(double c, const GD<N>& a) { return a * c; }
GD_T GD<N> operator/(const GD<N>& a, double c) { GD<N> r; const double ic = gd_inv(c); r.v = a.v * ic; for (int i = 0; i < N; ++i) r.d[i] = a.d[i] * ic; return r; }
GD_T GD<N> operator/(double c, const GD<N>& a) {
    GD<N> r; const double ib = gd_inv(a.v); r.v = c * ib;
    for (int i = 0; i < N; ++i) r.d[i] = -r.v * a.d[i] * ib;
    return r;
}
GD_T bool operator<(const GD<N>& a, const GD<N>& b) { return a.v < b.v; }
GD_T bool operator>(const GD<N>& a, const GD<N>& b) { return a.v > b.v; }
GD_T bool operator<=(const GD<N>& a, const GD<N>& b) { return a.v <= b.v; }
GD_T bool operator>=(const GD<N>& a, const GD<N>& b) { return a.v >= b.v; }
GD_T bool operator<(const GD<N>& a, double b) { return a.v < b; }
GD_T bool operator>(const GD<N>& a, double b) { return a.v > b; }
GD_T bool operator<=(const GD<N>& a, double b) { return a.v <= b; }
GD_T bool operator>=(const GD<N>& a, double b) { return a.v >= b; }
GD_T bool operator<=(double a, const GD<N>& b) { return a <= b.v; }
GD_T GD<N> gb_rcp(const GD<N>& a) { return 1.0 / a; } // the generated metric code calls gb_rcp on its scalar type
GD_T GD<N> gd_sqrt(const GD<N>& a) { GD<N> r; r.v = sqrt(a.v); const double h = 0.5 / r.v; for (int i = 0; i < N; ++i) r.d[i] = h * a.d[i]; return r; }
GD_T GD<N> gd_abs(const GD<N>& a) { return a.v < 0.0 ? -a : a; }
GD_T void gd_sincos(const GD<N>& a, GD<N>& s, GD<N>& c) {
    double sv, cv;
#ifdef __CUDA_ARCH__
    gb_sincos(a.v, &sv, &cv); // the polar angle stays far below 2^20 rad: no Payne-Hanek path needed
#else
    sincos(a.v, &sv, &cv);
#endif
    s.v = sv; c.v = cv;
    for (int i = 0; i < N; ++i) { s.d[i] = cv * a.d[i]; c.d[i] = -sv * a.d[i]; }
}
GD_T GD<N> gd_sin(const GD<N>& a) { GD<N> s, c; gd_sincos(a, s, c); return s; }
GD_T GD<N> gd_cos(const GD<N>& a) { GD<N> s, c; gd_sincos(a, s, c); return c; }
// clamps by compares and selects: a clamped value carries no derivative
GD_T GD<N> gd_fmin(const GD<N>& a, double b) { return a > b ? GD<N>(b) : a; }
GD_T GD<N> gd_fmax(const GD<N>& a, double b) { return a < b ? GD<N>(b) : a; }
// |u| as DiffEqBase's internalnorm sees one dual: sqrt(value^2 + sum partials^2); values only: |value|
GD_T double gd_norm1(const GD<N>& a, bool partials) {
    if (!partials || N == 0) return fabs(a.v);
    double s = a.v * a.v;
    for (int i = 0; i < N; ++i) s += a.d[i] * a.d[i];
    return sqrt(s);
}
GD_T double gd_norm8(const GD<N> a[8], bool partials) {
    double s = 0.0;
    for (int i = 0; i < 8; ++i) {
        s += a[i].v * a[i].v;
        if (partials) for (int k = 0; k < N; ++k) s += a[i].d[k] * a[i].d[k];
    }
    return sqrt(s / ((partials && N > 0) ? 8.0 * (1 + N) : 8.0));
}

// ---------------------------------------------------------------- right-hand side over S
// geodesic_equation with d_t = d_phi = 0 written out (auto-diff.jl:59-76,115-141), same algebra as geodesic_accel
template <class S>
GB_HD inline void geodesic_accel_g(const S g[5], const S dr[5], const S dth[5], const S& vt, const S& vr, const S& vth, const S& vph,
                                   S acc[4], S gi[5]) {
    const S D = g[0] * g[3] - g[4] * g[4];
    const S iD = 1.0 / D;
    gi[0] = g[3] * iD; gi[3] = g[0] * iD; gi[4] = -(g[4] * iD);
    gi[1] = 1.0 / g[1]; gi[2] = 1.0 / g[2];
    const S d0 = vr * dr[0] + vth * dth[0];
    const S d3 = vr * dr[3] + vth * dth[3];
    const S d4 = vr * dr[4] + vth * dth[4];
    const S Pt = d0 * vt + d4 * vph;
    const S Pp = d4 * vt + d3 * vph;
    const S vtt = vt * vt, vrr = vr * vr, vthth = vth * vth, vpp = vph * vph, vtp2 = 2.0 * (vt * vph);
    const S X = vr * vth;
    const S Br = dr[0] * vtt - dr[1] * vrr + dr[2] * vthth + dr[3] * vpp + dr[4] * vtp2;
    const S Bt = dth[0] * vtt + dth[1] * vrr - dth[2] * vthth + dth[3] * vpp + dth[4] * vtp2;
    acc[0] = -(gi[0] * Pt) - gi[4] * Pp;
    acc[1] = gi[1] * (0.5 * Br - dth[1] * X);
    acc[2] = gi[2] * (0.5 * Bt - dr[2] * X);
    acc[3] = -(gi[4] * Pt) - gi[3] * Pp;
}
// Lorentz force of the Kerr-Newman field on a charged test particle (kerr_newman_lorentz over S)
template <class S>
GB_HD inline void kerr_newman_lorentz_g(const double* mp, const S& r, const S& s, const S& c, const S gi[5],
                                        const S& vt, const S& vr, const S& vth, const S& vph, S acc[4]) {
    const double a = mp[1], Q = mp[2], q = mp[3];
    const double a2 = a * a;
    const S s2 = s * s, sc2 = 2.0 * (s * c);
    const S Sig = r * r + a2 * (c * c);
    const S iS = 1.0 / Sig;
    const S At = Q * r * iS;
    const S At_r = Q * (Sig - 2.0 * (r * r)) * iS * iS;
    const S At_t = At * a2 * sc2 * iS;
    const S Ap_r = -a * s2 * At_r;
    const S Ap_t = -a * (sc2 * At + s2 * At_t);
    const S wt = At_r * vr + At_t * vth, wp = Ap_r * vr + Ap_t * vth;
    const S wr = -(At_r * vt + Ap_r * vph), wth = -(At_t * vt + Ap_t * vph);
    acc[0] = acc[0] + q * (gi[0] * wt + gi[4] * wp);
    acc[1] = acc[1] + q * gi[1] * wr;
    acc[2] = acc[2] + q * gi[2] * wth;
    acc[3] = acc[3] + q * (gi[4] * wt + gi[3] * wp);
}
// Kerr accelerations in closed form over S: the Euler-Lagrange form of kerr_rhs_accel_sq (gb200_device.cuh) -- two thirds
// of the operations of the generic metric Jacobian + contraction, which matters threefold on GD<2>
template <class S>
GB_HD inline void kerr_accel_g(double M, double a, const S& r, const S& s, const S& c, const S& vt, const S& vr, const S& vth, const S& vph, S acc[4]) {
    const double a2 = a * a;
    const S s2 = s * s, sin2 = 2.0 * (s * c), r2 = r * r;
    const S rho2 = r2 + a2;
    const S Sig = r2 + a2 * (c * c), Del = r * (r - 2.0 * M) + a2;
    const S iSig = 1.0 / Sig, iDel = 1.0 / Del;
    const S w = (2.0 * M) * r * iSig;
    const S hw_r = (M - w * r) * iSig; // w_r / 2
    const S a2sin2 = a2 * sin2;
    const S as2 = a * s2;
    const S A = vt - as2 * vph, U = w * A;
    const S h = a2sin2 * vth;
    const S wdot = 2.0 * (hw_r * vr) + (w * iSig) * h;
    const S rr = r * vr;
    const S Udot = ((rho2 * wdot) * A - (w * h) * U + 2.0 * (((w * as2) * rr) * vph)) * iDel;
    const S pp = vph * vph, tt = vth * vth, rr2 = vr * vr, X = vr * vth;
    acc[0] = Udot;
    acc[1] = (Del * iSig) * (r * (s2 * pp + tt) + hw_r * (A * A)) - (r * iSig - (r - M) * iDel) * rr2 + (a2sin2 * iSig) * X;
    acc[2] = iSig * ((0.5 * sin2) * (rho2 * pp - (2.0 * a) * (U * vph) + a2 * (tt - rr2 * iDel + (U * A) * iSig)) - 2.0 * (r * X));
    const S m = (sin2 / s2) * vth;
    acc[3] = (a * (m * U + Udot) - 2.0 * (rr * vph)) / rho2 - m * vph;
}

// _second_order_ode_f (src/tracing/geodesic-problem.jl:87-92): du = (v, a); also returns sin, cos of theta
// MK >= 0 fixes the metric kind at compile time (the Kerr instantiation of the forward-mode kernel then carries no other
// metric's code: a lone warp walks the step code once per attempt, and what does not fit the instruction cache is fetched
// again every attempt); MK = -1 reads it from P.
template <int N, int MK = -1>
GB_HD inline void rhs_g(const GbParams& P, const GD<N> u[8], GD<N> du[8], GD<N>& s, GD<N>& c) {
    typedef GD<N> S;
    const int mk = (MK >= 0) ? MK : P.metric_kind;
    gd_sincos(u[2], s, c);
    S acc[4];
    if (mk == GB200_METRIC_KERR) kerr_accel_g<S>(P.M, P.a, u[1], s, c, u[4], u[5], u[6], u[7], acc);
    else {
        S g[5], dr[5], dth[5], gi[5];
        metric_jacobian_kind<S>(mk, P.mp, u[1], s, c, g, dr, dth);
        geodesic_accel_g<S>(g, dr, dth, u[4], u[5], u[6], u[7], acc, gi);
        if (mk == GB200_METRIC_KERR_NEWMAN && P.mp[3] != 0.0) kerr_newman_lorentz_g<S>(P.mp, u[1], s, c, gi, u[4], u[5], u[6], u[7], acc);
    }
    for (int i = 0; i < 4; ++i) { du[i] = u[4 + i]; du[4 + i] = acc[i]; }
}

// ---------------------------------------------------------------- the integrator
template <int N>
struct GenResult {
    int status, naccept, nreject, flags;
    double lambda;
    GD<N> u[8];     // end state
    GD<N> E_obs;    // g_{mu nu}(x_init) v_init^mu (1,0,0,0)^nu
    double closest; // GB200_GEOMETRY_TARGET_POINT: the smallest distance to the target over every evaluation of the condition
};

GB_HD inline void gen_dense_weights(double Th, double b[7], double db[7]) { // b_j(Theta) and d b_j / d Theta of the Tsit5 interpolant
    // R_jk by name: indexing the list as gb_const(GB_I_R12 + 3 j) inside the loop costs the forward-mode kernels registers
    // and stack (-Xptxas -v: 2 more registers in gb200_target_kernel<Kerr>, 352 bytes more stack in gb200_dual_kernel<1, Kerr>)
    const double R2[7] = {gb_const(GB_I_R12), gb_const(GB_I_R22), gb_const(GB_I_R32), gb_const(GB_I_R42), gb_const(GB_I_R52), gb_const(GB_I_R62), gb_const(GB_I_R72)};
    const double R3[7] = {gb_const(GB_I_R13), gb_const(GB_I_R23), gb_const(GB_I_R33), gb_const(GB_I_R43), gb_const(GB_I_R53), gb_const(GB_I_R63), gb_const(GB_I_R73)};
    const double R4[7] = {gb_const(GB_I_R14), gb_const(GB_I_R24), gb_const(GB_I_R34), gb_const(GB_I_R44), gb_const(GB_I_R54), gb_const(GB_I_R64), gb_const(GB_I_R74)};
    for (int j = 0; j < 7; ++j) {
        const double lead = (j == 0) ? 1.0 : 0.0;
        b[j] = Th * (lead + Th * (R2[j] + Th * (R3[j] + Th * R4[j])));
        db[j] = lead + Th * (2.0 * R2[j] + Th * (3.0 * R3[j] + Th * (4.0 * R4[j])));
    }
}

// Can the disc condition change sign inside this step?  |u(Theta) - u0| <= |dt| L max_j |k_j| with L = max sum_j |b_j(Theta)| =
// 7.5822 for the Tsit5 interpolant, and |cos| is 1-Lipschitz: when the bound keeps the ray outside the surface the six
// interior samples (all of the previous sign) are skipped.  Same test as scan_needed<GEOM> of the ensemble kernel.
template <int N>
GB_HD inline bool gen_scan_needed(const GbParams& P, double r0, double cprev, double sprev, double hgt, double dt, const GD<N> k[7][8]) {
    if (sprev < 0.0) return true;
    double mr = 0.0, mth = 0.0;
    for (int j = 0; j < 7; ++j) { mr = fmax(mr, fabs(k[j][1].v)); mth = fmax(mth, fabs(k[j][2].v)); }
    const double Br = fabs(dt) * 7.5823 * mr, Bth = fabs(dt) * 7.5823 * mth, slack = 1.0 + 1e-9;
    if (P.geometry_kind == GB200_GEOMETRY_DATUM_PLANE) return !(fabs(cprev) > (Br + (fabs(r0) + Br) * Bth) * slack + 1e-12);
    if (P.geometry_kind == GB200_GEOMETRY_THIN_DISC) {
        // inside the radial range the condition is r |cos| - gtol |r| = cprev; outside it is 1: bound |cos| from below
        return true;
    }
    return true;
}

// Stage input u + dt sum_l a_{S+1,l+1} k_l with the stage number as a template parameter: the coefficients are immediates
// and the k rows are read at constant offsets (the run-time loop over l cost a fifth of the forward-mode kernel's
// instructions in index arithmetic, compares and branches).  Same order of operations as the run-time loop.
template <int N, int S>
GB_HD inline void gen_stage_input(const GD<N> u[8], double dt, const GD<N> k[7][8], GD<N> tmp[8]) {
    constexpr int a = GB_I_A21 + S * (S - 1) / 2; // a_{S+1,1}: the list holds the a_ij row by row
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        if (S == 1) tmp[i] = u[i] + (dt * gb_const(a)) * k[0][i];
        else {
            GD<N> acc = gb_const(a) * k[0][i];
#pragma unroll
            for (int l = 1; l < S; ++l) acc = acc + gb_const(a + l) * k[l][i];
            tmp[i] = u[i] + dt * acc;
        }
    }
}

// REC: callable (double lambda, const GD<N> u[8]) invoked with the initial state and after every accepted step
template <int N, int MK = -1, class REC>
GB_HD inline void gen_trace_ray(const GbParams& P, const GD<N> u_init[8], double hgt, bool norm_partials, GenResult<N>& res, REC&& rec) {
    typedef GD<N> S;
    const double abstol = P.abstol, reltol = P.reltol, dtmax = P.dtmax, dtmin = 2.220446049250313e-16, tstop = P.lam1;
    const double beta1 = 7.0 / 50.0, beta2 = 2.0 / 25.0, gamma = 9.0 / 10.0, qmin = 1.0 / 5.0, qmax = 10.0, qoldinit = 1e-4;
    const bool fast32 = P.pow_mode == GB200_POW_FAST32;
    const bool has_geom = P.geometry_kind != GB200_GEOMETRY_NONE;
    S u[8], un[8], k[7][8], tmp[8];
    for (int i = 0; i < 8; ++i) u[i] = u_init[i];
    double t = P.lam0;
    res.status = GB200_STATUS_NO_STATUS; res.naccept = 0; res.nreject = 0; res.flags = 0;
    rec(t, u);
    S s_, c_;
    rhs_g<N, MK>(P, u, k[0], s_, c_);
    const bool target = P.geometry_kind == GB200_GEOMETRY_TARGET_POINT;
    double cprev = has_geom ? disc_condition<-1>(P, u[1], s_, c_, hgt, u[3].v).v : 1.0;
    res.closest = target ? cprev + P.gtol : nan("");
    double dt;
    { // ode_determine_initdt
        double sk[8];
        S w[8];
        for (int i = 0; i < 8; ++i) { sk[i] = abstol + gd_norm1(u[i], norm_partials) * reltol; w[i] = u[i] / sk[i]; }
        const double d0 = gd_norm8(w, norm_partials);
        for (int i = 0; i < 8; ++i) w[i] = k[0][i] / sk[i];
        const double d1 = gd_norm8(w, norm_partials);
        double dt0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : (d0 / d1) / 100.0;
        dt0 = fmin(dt0, dtmax);
        for (int i = 0; i < 8; ++i) tmp[i] = u[i] + dt0 * k[0][i];
        rhs_g<N, MK>(P, tmp, k[1], s_, c_);
        for (int i = 0; i < 8; ++i) w[i] = (k[1][i] - k[0][i]) / sk[i];
        const double d2 = gd_norm8(w, norm_partials) / dt0;
        const double md = fmax(d1, d2);
        const double dt1 = (md <= 1e-15) ? fmax(1e-6, dt0 * 1e-3) : exp(-0.2 * log(100.0 * md));
        dt = fmax(dtmin, fmin(fmin(100.0 * dt0, dt1), dtmax));
    }
    double qold = qoldinit;
    const int64_t maxit = P.maxiters;
    for (int64_t iter = 0;; ++iter) {
        const double rem = tstop - t;
        if (iter >= maxit) { res.flags |= GB200_FLAG_MAXITERS; break; }
        if (!(dt == dt) || !(u[1].v == u[1].v)) { res.flags |= GB200_FLAG_UNSTABLE; break; }
        if (!(fmin(dt, rem) > dtmin) && rem > dtmin) { res.flags |= GB200_FLAG_DT_MIN; break; }
        dt = fmin(dt, rem);
#ifdef __CUDA_ARCH__
#pragma unroll 1 /* one copy of the right-hand side in the step loop: the loop body then stays inside the instruction cache */
#endif
        for (int s = 1; s < 7; ++s) {
            switch (s) {
            case 1: gen_stage_input<N, 1>(u, dt, k, tmp); break;
            case 2: gen_stage_input<N, 2>(u, dt, k, tmp); break;
            case 3: gen_stage_input<N, 3>(u, dt, k, tmp); break;
            case 4: gen_stage_input<N, 4>(u, dt, k, tmp); break;
            case 5: gen_stage_input<N, 5>(u, dt, k, tmp); break;
            default: gen_stage_input<N, 6>(u, dt, k, tmp); break;
            }
            if (s == 6) for (int i = 0; i < 8; ++i) un[i] = tmp[i];
            rhs_g<N, MK>(P, tmp, k[s], s_, c_);
        }
        double EEst;
        {
            S at[8];
            for (int i = 0; i < 8; ++i) {
                S e = gb_const(GB_I_BT1) * k[0][i];
                for (int l = 1; l < 7; ++l) e = e + gb_const(GB_I_BT1 + l) * k[l][i];
                at[i] = (dt * e) / (abstol + fmax(gd_norm1(u[i], norm_partials), gd_norm1(un[i], norm_partials)) * reltol);
            }
            EEst = gd_norm8(at, norm_partials);
        }
        // PI controller (stepsize_controller!, step_accept_controller!, step_reject_controller!)
        double q11 = 0.0, q;
        if (EEst == 0.0) q = 1.0 / qmax;
        else {
            q11 = fast32 ? (double)exp2f((float)beta1 * log2f((float)EEst)) : exp(beta1 * log(EEst));
            const double qo = fast32 ? (double)exp2f((float)beta2 * log2f((float)qold)) : exp(beta2 * log(qold));
            q = fmax(1.0 / qmax, fmin(1.0 / qmin, q11 / qo / gamma));
        }
        if (!(EEst <= 1.0)) {
            ++res.nreject;
            dt = fmax(dt / fmin(1.0 / qmin, q11 / gamma), dtmin);
            continue;
        }
        ++res.naccept;
        qold = fmax(EEst, qoldinit);
        const double ttmp = t + dt;
        double tnew = (fabs(ttmp - tstop) < 100.0 * (fabs(tstop) * 2.220446049250313e-16)) ? tstop : ttmp;
        const double dtprop = fmax(fmin(dtmax, dt / q), dtmin);
        // ---- ContinuousCallback (decisions on values), interp_points = 8
        bool event = false;
        double cnext = 1.0;
        if (has_geom) {
            cnext = disc_condition<-1>(P, un[1], s_, c_, hgt, un[3].v).v;
            if (target) res.closest = fmin(res.closest, cnext + P.gtol);
            const double sprev = (cprev > 0.0) ? 1.0 : ((cprev < 0.0) ? -1.0 : 0.0);
            const double snext = (cnext > 0.0) ? 1.0 : ((cnext < 0.0) ? -1.0 : 0.0);
            double ev_lo = 0.0, ev_hi = 1.0;
            // value of the condition on the dense output at Theta
            auto cond_at = [&](double Th) -> double {
                double b[7], db[7];
                gen_dense_weights(Th, b, db);
                double rr = 0.0, tt = 0.0, pp = 0.0;
                for (int j = 0; j < 7; ++j) { rr += b[j] * k[j][1].v; tt += b[j] * k[j][2].v; }
                if (target) for (int j = 0; j < 7; ++j) pp += b[j] * k[j][3].v;
                rr = u[1].v + dt * rr; tt = u[2].v + dt * tt; pp = u[3].v + dt * pp;
                double sv, cv;
                sincos(tt, &sv, &cv);
                const double cv_ = disc_condition<-1>(P, rr, sv, cv, hgt, pp);
                if (target) res.closest = fmin(res.closest, cv_ + P.gtol); // closest_approach[] is updated by every evaluation
                return cv_;
            };
            if (sprev != 0.0) {
                if (target) {
                    // The reference's objective is the smallest of the condition's own evaluations -- eight samples per step,
                    // which miss a d_tol sphere lying between two of them (steps are ~ 1 long near the hole, d_tol = 1e-2), plus
                    // whatever the root finder happens to touch.  Here the distance is minimised along the dense output of
                    // the step: all samples, then a golden-section search around the smallest one; the ray ends (event) at
                    // its first entry into the d_tol sphere, and closest is the minimum over the whole step either way, so it
                    // does not depend on which points a root finder visits.
                    double best = cprev, bestTh = 0.0;
                    int first_neg = 0;
                    for (int i = 1; i <= 7; ++i) {
                        const double Th = (double)i / 7.0, cv = (i == 7) ? cnext : cond_at(Th);
                        if (cv < 0.0 && !first_neg) first_neg = i;
                        if (cv < best) { best = cv; bestTh = Th; }
                    }
                    double a = fmax(bestTh - 1.0 / 7.0, 0.0), b = fmin(bestTh + 1.0 / 7.0, 1.0);
                    const double gr = 0.6180339887498949;
                    double x1 = b - gr * (b - a), x2 = a + gr * (b - a), f1 = cond_at(x1), f2 = cond_at(x2);
                    for (int it = 0; it < 30; ++it) {
                        if (f1 < f2) { b = x2; x2 = x1; f2 = f1; x1 = b - gr * (b - a); f1 = cond_at(x1); }
                        else { a = x1; x1 = x2; f1 = f2; x2 = a + gr * (b - a); f2 = cond_at(x2); }
                    }
                    const double xm = (f1 < f2) ? x1 : x2, fm = fmin(f1, f2);
                    if (first_neg) { event = true; ev_lo = (double)(first_neg - 1) / 7.0; ev_hi = (double)first_neg / 7.0; }
                    else if (fm < 0.0) { event = true; ev_lo = fmax(bestTh - 1.0 / 7.0, 0.0); ev_hi = xm; }
                } else if (sprev * snext <= 0.0) event = true;
                else if (gen_scan_needed(P, u[1].v, cprev, sprev, hgt, dt, k))
                    for (int i = 1; i <= 6; ++i) {
                        const double Th = (double)i / 7.0;
                        if (sprev * cond_at(Th) < 0.0) { event = true; ev_lo = (double)(i - 1) / 7.0; ev_hi = Th; break; }
                    }
            }
            if (event) {
                // left-biased root find (find_callback_time, LeftRootFind): Illinois regula falsi with a bisection fallback
                double lo = ev_lo, hi = ev_hi;
                double flo = (lo > 0.0) ? cond_at(lo) : cprev;
                double fhi = (hi < 1.0) ? cond_at(hi) : cnext;
                if (fhi == 0.0) lo = hi;
                else {
                    int side = 0;
                    for (int it = 0; it < 100; ++it) {
                        const double w = hi - lo;
                        if (w <= 1e-15) break;
                        double mid = (it < 40 && flo * fhi < 0.0) ? (lo * fhi - hi * flo) / (fhi - flo) : 0.5 * (lo + hi);
                        if (!(mid > lo && mid < hi)) mid = 0.5 * (lo + hi);
                        if (!(mid > lo && mid < hi)) break;
                        const double fm = cond_at(mid);
                        if (fm != 0.0 && (fm > 0.0) == (sprev > 0.0)) { lo = mid; flo = fm; if (side == -1) fhi *= 0.5; side = -1; }
                        else { hi = mid; fhi = fm; if (fm == 0.0) fhi = -sprev * 1e-300; if (side == 1) flo *= 0.5; side = 1; }
                    }
                }
                // change_t_via_interpolation!: the state from the interpolant at Theta = lo, partials included
                const double Th = lo;
                double b[7], db[7];
                gen_dense_weights(Th, b, db);
                S ue[8];
                double dudTh[8];
                for (int i = 0; i < 8; ++i) {
                    S acc = b[0] * k[0][i];
                    double ds = db[0] * k[0][i].v;
                    for (int j = 1; j < 7; ++j) { acc = acc + b[j] * k[j][i]; ds += db[j] * k[j][i].v; }
                    ue[i] = u[i] + dt * acc;
                    dudTh[i] = dt * ds;
                }
                if (N > 0) { // the event time moves with the parameters: Theta_p = -(dc/dp) / (dc/dTheta)
                    S se, ce;
                    gd_sincos(ue[2], se, ce);
                    const S cD = disc_condition<-1>(P, ue[1], se, ce, hgt);
                    GD<2> r2(ue[1].v), t2(ue[2].v), s2, c2;
                    r2.d[0] = 1.0; t2.d[1] = 1.0;
                    gd_sincos(t2, s2, c2);
                    const GD<2> cg = disc_condition<-1>(P, r2, s2, c2, hgt);
                    const double dcdTh = cg.d[0] * dudTh[1] + cg.d[1] * dudTh[2];
                    if (dcdTh != 0.0 && dcdTh == dcdTh && fabs(dcdTh) < 1e300)
                        for (int kk = 0; kk < N; ++kk) {
                            const double Thp = -cD.d[kk] / dcdTh;
                            for (int i = 0; i < 8; ++i) ue[i].d[kk] += dudTh[i] * Thp;
                        }
                }
                for (int i = 0; i < 8; ++i) un[i] = ue[i];
                tnew = t + Th * dt;
                gd_sincos(un[2], s_, c_);
            }
        }
        // ---- DiscreteCallbacks in CallbackSet order: user, then chart (the later one overwrites the status)
        int status = event ? GB200_STATUS_INTERSECTED_WITH_GEOMETRY : GB200_STATUS_NO_STATUS;
        bool term = event;
        if (P.callback_kind == GB200_CALLBACK_UPPER_HEMISPHERE && un[1].v * c_.v < P.callback_delta) { status = GB200_STATUS_OUT_OF_DOMAIN; term = true; }
        if (un[1].v <= P.chart_inner) { status = GB200_STATUS_WITHIN_INNER_BOUNDARY; term = true; }
        else if (un[1].v > P.chart_outer) { status = GB200_STATUS_OUT_OF_DOMAIN; term = true; }
        if (!(tnew < tstop)) term = true;
        t = tnew;
        for (int i = 0; i < 8; ++i) { u[i] = un[i]; k[0][i] = k[6][i]; }
        cprev = cnext;
        dt = dtprop;
        rec(t, u);
        if (term) { res.status = status; break; }
    }
    res.lambda = t;
    for (int i = 0; i < 8; ++i) res.u[i] = u[i];
}

// map_impact_parameters + constrain_all over S: the closed-form LNRF constants of the launch are plain doubles (the
// observer carries no partials in the reference either: x_dual has zero partials, precision-solvers.jl:82-87)
template <int N>
GB_HD inline void gen_initial_state(const GbParams& P, const GD<N>& alpha, const GD<N>& beta, GD<N> u0[8], GD<N>& E_obs) {
    typedef GD<N> S;
    for (int k = 0; k < 4; ++k) u0[k] = S(P.xo[k]);
    const S b = beta / P.xo[1], a = alpha / P.xo[1];
    const S pr = -1.0 / gd_sqrt(1.0 + a * a + b * b);
    const S pth = b * pr, pph = a * pr;
    u0[5] = P.c_r * pr;
    u0[6] = P.c_th * pth;
    u0[7] = P.c_ph0 + P.c_ph1 * pph;
    S go[5];
    for (int k = 0; k < 5; ++k) go[k] = S(P.go[k]);
    u0[4] = constrain_vt(go, u0[5], u0[6], u0[7], P.mu);
    E_obs = P.go[0] * u0[4] + P.go[4] * u0[7];
}
