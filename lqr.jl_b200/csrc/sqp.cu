// sqp.cu — batched Dubins SQP driver, everything on device.
//
// Outer loop      solve!/step!            src/cholesky_solver.jl:109-153  (<= iters steps, converge at
//                                         feas_p, feas_d < eps, :131-137)
// Linearisation   update!                 src/cholesky_solver.jl:155-164  (third-party numerics in the
//                                         reference; re-derived here for the Dubins car, RK3 as
//                                         test/cartpole.jl:38, cost expansion scaled by dt on non-terminal
//                                         knots as test/sparse_solver.jl:67-72 pins)
// QP step         _solve!                 src/cholesky_solver.jl:166-182  (the batched KKT kernel)
// Globalisation   line_search (spec)      src/sqp.jl:72-94: L1 merit phi = f + mu*||c||_1,
//                                         phi' = grad f'dx - mu*||c||_1, eta = 1e-4, rho = 0.5, <= 10
//                                         trials, second-order correction tried only at alpha = 1:
//                                         dx^ = -A'(AA')^-1 c(x+dx)  (= second_order_correction!,
//                                         src/cholesky_solver.jl:254-273, the Ginv=false chain)
// The merit penalty rule (TO.update_penalty!, third-party, unpinned) is mu <- max(mu, 1.1*||lambda||_inf).
//
// One thread per instance; every per-instance array is tiled batch-minor [tile][row][32].
#include <algorithm>
#include <cmath>

#include "common.cuh"
#include "kkt_kernels.cuh"

namespace {

constexpr int n = 3, m = 2, w = n + m;
// packed KKT rows for p = [3, 0, ..., 0, 3], HESS_DIAG (see lqrb200.h)
constexpr int ROWS_FIRST = w + w + n * w + n + n * w + n;  // H g D1 d C c = 46
constexpr int ROWS_MID = w + w + n * w + n;                // 28
constexpr int ROWS_LAST = n + n + n * n + n;               // 18

struct Opts {
    int N;
    double dt, qd, rd, qfd;
};

__device__ __forceinline__ int64_t knot_row(int k, int N) {
    return k == 0 ? 0 : (int64_t)ROWS_FIRST + (int64_t)(k - 1) * ROWS_MID;
}
__device__ __forceinline__ int64_t data_rows(int N) { return ROWS_FIRST + (int64_t)(N - 2) * ROWS_MID + ROWS_LAST; }
__device__ __forceinline__ int64_t mult_row(int k) { return k == 0 ? 0 : (int64_t)n + n + (int64_t)(k - 1) * n; }

// RK3 step of the Dubins car (x, y, theta; v, omega) and the averaged heading terms.
__device__ __forceinline__ void dubins_avg(double th, double om, double dt, double &cb, double &sb, double &dcb,
                                           double &dsb) {
    const double t2 = th + 0.5 * dt * om, t3 = th + dt * om;
    double s1, c1, s2, c2, s3, c3;
    sincos(th, &s1, &c1);
    sincos(t2, &s2, &c2);
    sincos(t3, &s3, &c3);
    cb = (c1 + 4.0 * c2 + c3) / 6.0;
    sb = (s1 + 4.0 * s2 + s3) / 6.0;
    dcb = (-4.0 * s2 * 0.5 * dt - s3 * dt) / 6.0;  // d cb / d omega
    dsb = (4.0 * c2 * 0.5 * dt + c3 * dt) / 6.0;
}

struct Stats {  // per-instance scalars, stored as rows of a [S_COUNT][32]-tiled array
    enum { F0 = 0, C1, CINF, FEASD, MU, PHI0, DPHI0, ALPHA, DONE, CONV, ITERS, S_COUNT };
};

// ---------------------------------------------------------------------------------------------
// linearise at Z: writes the packed KKT data and per-instance f, ||c||_1, ||c||_inf, feas_d.
// feas_d = || (||g_k + D1_k'lam_k + C_k'mu_k + D2_k'lam_{k-1}||)_k ||  with the previous multipliers
// (residual(solver, recalculate=false), src/cholesky_solver.jl:130,238-252).
template <bool WRITE>
__global__ void __launch_bounds__(64) dubins_linearize_kernel(const double *__restrict__ Z, const double *__restrict__ x0,
                                                              const double *__restrict__ xf, const double *__restrict__ mult,
                                                              double *__restrict__ data, double *__restrict__ stats,
                                                              Opts o, int64_t batch, int check_conv, double eps_p,
                                                              double eps_d) {
    const int64_t inst = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= batch) return;
    const int64_t tile = inst >> 5;
    const int lane = (int)(inst & 31);
    const int N = o.N;
    const int64_t NN = (int64_t)N * n + (int64_t)(N - 1) * m, P = (int64_t)(N - 1) * n + 2 * n;
    const double *zb = Z + tile * NN * 32 + lane;
    const double *mb = mult + tile * P * 32 + lane;
    double *db = WRITE ? data + tile * data_rows(N) * 32 + lane : nullptr;  // WRITE = false: statistics only
    double *sb = stats + tile * Stats::S_COUNT * 32 + lane;
    const double *x0b = x0 + tile * n * 32 + lane, *xfb = xf + tile * n * 32 + lane;
    double xg[n];
    for (int i = 0; i < n; ++i) xg[i] = xfb[i * 32];

    double f = 0.0, c1 = 0.0, cinf = 0.0, fd2 = 0.0;
    double x[n], xn[n], lam_prev[n] = {0.0, 0.0, 0.0};
    for (int i = 0; i < n; ++i) x[i] = zb[i * 32];
    for (int k = 0; k < N; ++k) {
        double *kp = db + knot_row(k, N) * 32;
        const bool last = k == N - 1;
        const double qs = last ? o.qfd : o.qd * o.dt, rs = o.rd * o.dt;
        double g[w], res[w];
        // cost expansion (diagonal): H = diag(Q dt, R dt), g = [Q (x - xf) dt; R u dt]
        for (int i = 0; i < n; ++i) {
            const double e = x[i] - xg[i];
            if (WRITE) kp[i * 32] = qs;
            g[i] = qs * e;
            f += 0.5 * qs * e * e;
        }
        if (last) {
            double *Cp = kp + 2 * n * 32;  // C = I, c = x_N - xf
            if (WRITE) {
                for (int i = 0; i < n; ++i) kp[(n + i) * 32] = g[i];
                for (int j = 0; j < n; ++j)
                    for (int i = 0; i < n; ++i) Cp[(i + j * n) * 32] = (i == j) ? 1.0 : 0.0;
            }
            const double *mu = mb + mult_row(k) * 32;
            for (int i = 0; i < n; ++i) {
                const double c = x[i] - xg[i];
                if (WRITE) Cp[(n * n + i) * 32] = c;
                c1 += fabs(c);
                cinf = fmax(cinf, fabs(c));
                res[i] = g[i] + mu[i * 32] - lam_prev[i];
                fd2 += res[i] * res[i];
            }
            break;
        }
        double u[m];
        for (int i = 0; i < m; ++i) {
            u[i] = zb[((int64_t)k * w + n + i) * 32];
            if (WRITE) kp[(n + i) * 32] = rs;
            g[n + i] = rs * u[i];
            f += 0.5 * rs * u[i] * u[i];
        }
        if (WRITE)
            for (int i = 0; i < w; ++i) kp[(w + i) * 32] = g[i];
        // dynamics: RK3 map, Jacobians A (3x3), B (3x2); D1 = [A B] column-major 3 x 5
        double cb, sbar, dcb, dsb;
        dubins_avg(x[2], u[1], o.dt, cb, sbar, dcb, dsb);
        const double v = u[0];
        double D1[n * w];
        for (int e = 0; e < n * w; ++e) D1[e] = 0.0;
        D1[0 + 0 * n] = 1.0; D1[1 + 1 * n] = 1.0; D1[2 + 2 * n] = 1.0;
        D1[0 + 2 * n] = -o.dt * v * sbar;
        D1[1 + 2 * n] = o.dt * v * cb;
        D1[0 + 3 * n] = o.dt * cb;
        D1[1 + 3 * n] = o.dt * sbar;
        D1[0 + 4 * n] = o.dt * v * dcb;
        D1[1 + 4 * n] = o.dt * v * dsb;
        D1[2 + 4 * n] = o.dt;
        double *D1p = kp + 2 * w * 32;
        if (WRITE)
            for (int e = 0; e < n * w; ++e) D1p[e * 32] = D1[e];
        for (int i = 0; i < n; ++i) xn[i] = zb[((int64_t)(k + 1) * w + i) * 32];
        const double fx[n] = {x[0] + o.dt * v * cb, x[1] + o.dt * v * sbar, x[2] + o.dt * u[1]};
        const double *lam = mb + (mult_row(k) + (k == 0 ? n : 0)) * 32;
        double lk[n];
        for (int i = 0; i < n; ++i) {
            const double d = fx[i] - xn[i];  // d_k = f(z_k) - x_{k+1}   (test/cartpole.jl:34-42)
            if (WRITE) D1p[(n * w + i) * 32] = d;
            c1 += fabs(d);
            cinf = fmax(cinf, fabs(d));
            lk[i] = lam[i * 32];
        }
        for (int j = 0; j < w; ++j) {
            double s = g[j];
            for (int i = 0; i < n; ++i) s = fma(D1[i + j * n], lk[i], s);
            if (j < n && k > 0) s -= lam_prev[j];
            res[j] = s;
        }
        if (k == 0) {  // C = [I 0], c = x_1 - x0
            double *Cp = D1p + (n * w + n) * 32;
            const double *mu = mb;
            if (WRITE)
                for (int j = 0; j < w; ++j)
                    for (int i = 0; i < n; ++i) Cp[(i + j * n) * 32] = (i == j) ? 1.0 : 0.0;
            for (int i = 0; i < n; ++i) {
                const double c = x[i] - x0b[i * 32];
                if (WRITE) Cp[(n * w + i) * 32] = c;
                c1 += fabs(c);
                cinf = fmax(cinf, fabs(c));
                res[i] += mu[i * 32];
            }
        }
        for (int j = 0; j < w; ++j) fd2 += res[j] * res[j];
        for (int i = 0; i < n; ++i) {
            lam_prev[i] = lk[i];
            x[i] = xn[i];
        }
    }
    const double feasd = sqrt(fd2);
    sb[Stats::F0 * 32] = f;
    sb[Stats::C1 * 32] = c1;
    sb[Stats::CINF * 32] = cinf;
    sb[Stats::FEASD * 32] = feasd;
    if (check_conv && sb[Stats::CONV * 32] == 0.0 && cinf < eps_p && feasd < eps_d) sb[Stats::CONV * 32] = 1.0;
}

// cost and constraint 1-norm / values at a trial point Zt = Z + alpha*dz (+ dzh)
// WRITE_C: 0 nothing; 1 into the c/d rows of the packed KKT data; 2 into a compact array with the row order of
// the multipliers [c_1; d_1; ...; d_{N-1}; c_N] (fused path: the SOC solve rebuilds everything else from Z)
template <int WRITE_C>
__device__ __forceinline__ void dubins_eval(const double *zb, const double *dzb, const double *dhb, double alpha,
                                            const double *x0b, const double *xg, const Opts &o, double *db,
                                            double &f, double &c1) {
    const int N = o.N;
    f = 0.0;
    c1 = 0.0;
    auto at = [&](int64_t row) {
        double v = fma(alpha, dzb[row * 32], zb[row * 32]);
        if (dhb) v += dhb[row * 32];
        return v;
    };
    double x[n], xn[n];
    for (int i = 0; i < n; ++i) x[i] = at(i);
    for (int i = 0; i < n; ++i) {
        const double c = x[i] - x0b[i * 32];
        c1 += fabs(c);
        if (WRITE_C == 1) db[(2 * w + n * w + n + n * w + i) * 32] = c;
        if (WRITE_C == 2) db[i * 32] = c;
    }
    for (int k = 0; k < N - 1; ++k) {
        double u[m];
        for (int i = 0; i < m; ++i) u[i] = at((int64_t)k * w + n + i);
        for (int i = 0; i < n; ++i) {
            const double e = x[i] - xg[i];
            f += 0.5 * o.qd * o.dt * e * e;
        }
        for (int i = 0; i < m; ++i) f += 0.5 * o.rd * o.dt * u[i] * u[i];
        double cb, sbar, dcb, dsb;
        dubins_avg(x[2], u[1], o.dt, cb, sbar, dcb, dsb);
        const double fx[n] = {x[0] + o.dt * u[0] * cb, x[1] + o.dt * u[0] * sbar, x[2] + o.dt * u[1]};
        for (int i = 0; i < n; ++i) xn[i] = at((int64_t)(k + 1) * w + i);
        for (int i = 0; i < n; ++i) {
            const double d = fx[i] - xn[i];
            c1 += fabs(d);
            if (WRITE_C == 1) db[(knot_row(k, N) + 2 * w + n * w + i) * 32] = d;
            if (WRITE_C == 2) db[(mult_row(k) + (k == 0 ? n : 0) + i) * 32] = d;
            x[i] = xn[i];
        }
    }
    for (int i = 0; i < n; ++i) {
        const double e = x[i] - xg[i];
        f += 0.5 * o.qfd * e * e;
        c1 += fabs(e);
        if (WRITE_C == 1) db[(knot_row(N - 1, N) + 2 * n + n * n + i) * 32] = e;
        if (WRITE_C == 2) db[(mult_row(N - 1) + i) * 32] = e;
    }
}

// ---------------------------------------------------------------------------------------------
// Fused linearisation + KKT solve: the thread-per-instance KKT sweeps of kkt_kernels.cuh, fed from a
// thread-local knot that is linearised on the fly from the iterate (update!, src/cholesky_solver.jl:155-164)
// instead of being written to HBM by one kernel and streamed back twice by the next.  SOC: H = I, g = 0 and
// the constraint values are c(x + dx) from `cvals` (second_order_correction!, :254-273).
template <int KIND, bool SOC>  // KIND 0 first, 1 middle, 2 last knot
__device__ __forceinline__ void dubins_build_knot(double *kn, const double *x, const double *u, const double *xn,
                                                  const double *x0v, const double *xg, const Opts &o,
                                                  const double *cd, const double *cc) {
    if (KIND == 2) {  // H (3) | g (3) | C = I (9) | c (3)
        SM_UNROLL
        for (int i = 0; i < n; ++i) {
            kn[i] = o.qfd;
            kn[n + i] = o.qfd * (x[i] - xg[i]);
            SM_UNROLL
            for (int j = 0; j < n; ++j) kn[2 * n + i + j * n] = (i == j) ? 1.0 : 0.0;
            kn[2 * n + n * n + i] = SOC ? cc[i * 32] : x[i] - xg[i];
        }
        return;
    }
    const double qs = o.qd * o.dt, rs = o.rd * o.dt;
    SM_UNROLL
    for (int i = 0; i < n; ++i) {
        kn[i] = qs;
        kn[w + i] = qs * (x[i] - xg[i]);
    }
    SM_UNROLL
    for (int i = 0; i < m; ++i) {
        kn[n + i] = rs;
        kn[w + n + i] = rs * u[i];
    }
    double cb, sbar, dcb, dsb;
    dubins_avg(x[2], u[1], o.dt, cb, sbar, dcb, dsb);
    const double v = u[0];
    double *D1 = kn + 2 * w;
    SM_UNROLL
    for (int e = 0; e < n * w; ++e) D1[e] = 0.0;
    D1[0 + 0 * n] = 1.0; D1[1 + 1 * n] = 1.0; D1[2 + 2 * n] = 1.0;
    D1[0 + 2 * n] = -o.dt * v * sbar;
    D1[1 + 2 * n] = o.dt * v * cb;
    D1[0 + 3 * n] = o.dt * cb;
    D1[1 + 3 * n] = o.dt * sbar;
    D1[0 + 4 * n] = o.dt * v * dcb;
    D1[1 + 4 * n] = o.dt * v * dsb;
    D1[2 + 4 * n] = o.dt;
    const double fx[n] = {x[0] + o.dt * v * cb, x[1] + o.dt * v * sbar, x[2] + o.dt * u[1]};
    SM_UNROLL
    for (int i = 0; i < n; ++i) D1[n * w + i] = SOC ? cd[i * 32] : fx[i] - xn[i];
    if (KIND == 0) {  // C = [I 0], c = x_1 - x0
        double *Cp = D1 + n * w + n;
        SM_UNROLL
        for (int j = 0; j < w; ++j)
            SM_UNROLL
            for (int i = 0; i < n; ++i) Cp[i + j * n] = (i == j) ? 1.0 : 0.0;
        SM_UNROLL
        for (int i = 0; i < n; ++i) Cp[n * w + i] = SOC ? cc[i * 32] : x[i] - x0v[i];
    }
}

template <bool SOC>
__global__ void __launch_bounds__(64, 8)
    dubins_kkt_fused_kernel(const double *__restrict__ Z, const double *__restrict__ x0, const double *__restrict__ xf,
                            const double *__restrict__ cvals, double *__restrict__ scratch, double *__restrict__ dz,
                            double *__restrict__ mult, int32_t *__restrict__ info, Opts o, int64_t batch) {
    using L = KktLayout<n, m, n, 0, n, LQRB_HESS_DIAG>;
    constexpr int HD = LQRB_HESS_DIAG;
    const int64_t inst = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= batch) return;
    const int64_t tile = inst >> 5;
    const int lane = (int)(inst & 31);
    const int N = o.N;
    const int64_t NN = (int64_t)N * n + (int64_t)(N - 1) * m, P = (int64_t)(N - 1) * n + 2 * n;
    const double *zb = Z + tile * NN * 32 + lane;
    const double *cvb = SOC ? cvals + tile * P * 32 + lane : nullptr;
    double *sb = scratch + tile * L::rec_rows(N) * 32 + lane;
    double *dzb = dz + tile * NN * 32 + lane;
    double *mb = mult + tile * P * 32 + lane;
    double xg[n], x0v[n];
    SM_UNROLL
    for (int i = 0; i < n; ++i) {
        xg[i] = xf[tile * n * 32 + lane + i * 32];
        x0v[i] = x0[tile * n * 32 + lane + i * 32];
    }
    auto ldz = [&](int64_t row) { return zb[row * 32]; };
    double kn[ROWS_FIRST], x[n], u[m], xn[n];

    // ---------------- forward sweep
    FwdCarry<n> cy;
    SM_UNROLL
    for (int i = 0; i < n; ++i) { x[i] = ldz(i); xn[i] = ldz(w + i); }
    SM_UNROLL
    for (int i = 0; i < m; ++i) u[i] = ldz(n + i);
    dubins_build_knot<0, SOC>(kn, x, u, xn, x0v, xg, o, SOC ? cvb + n * 32 : nullptr, cvb);
    int st = kkt_fwd_knot<n, m, 0, n, n, HD, SOC, 1>(kn, sb, cy, 0);
    for (int k = 1; k < N - 1; ++k) {
        SM_UNROLL
        for (int i = 0; i < n; ++i) { x[i] = xn[i]; xn[i] = ldz((int64_t)(k + 1) * w + i); }
        SM_UNROLL
        for (int i = 0; i < m; ++i) u[i] = ldz((int64_t)k * w + n + i);
        dubins_build_knot<1, SOC>(kn, x, u, xn, x0v, xg, o, SOC ? cvb + mult_row(k) * 32 : nullptr, nullptr);
        const int s2 = kkt_fwd_knot<n, m, n, 0, n, HD, SOC, 1>(
            kn, sb + ((int64_t)L::RF::ROWS + (int64_t)(k - 1) * L::RM::ROWS) * 32, cy, k);
        if (!st) st = s2;
    }
    const int64_t rlast = (int64_t)L::RF::ROWS + (int64_t)(N - 2) * L::RM::ROWS;
    {
        SM_UNROLL
        for (int i = 0; i < n; ++i) x[i] = xn[i];
        dubins_build_knot<2, SOC>(kn, x, u, xn, x0v, xg, o, nullptr, SOC ? cvb + mult_row(N - 1) * 32 : nullptr);
        const int s2 = kkt_fwd_knot<n, 0, n, n, 0, HD, SOC, 1>(kn, sb + rlast * 32, cy, N - 1);
        if (!st) st = s2;
    }
    if (info) info[inst] = st;

    // ---------------- backward sweep (the knot is linearised again: cheaper than a round trip through HBM)
    double lam[n];
    const int64_t mlast = (int64_t)n + n + (int64_t)(N - 2) * n;
    const int64_t zlast = (int64_t)(N - 1) * w;
    kkt_bwd_knot<n, 0, n, n, 0, HD, SOC, 1>(kn, sb + rlast * 32, lam, dzb + zlast * 32, mb + mlast * 32,
                                            mb + (mlast - n) * 32, nullptr);
    for (int k = N - 2; k >= 1; --k) {
        SM_UNROLL
        for (int i = 0; i < n; ++i) { xn[i] = x[i]; x[i] = ldz((int64_t)k * w + i); }
        SM_UNROLL
        for (int i = 0; i < m; ++i) u[i] = ldz((int64_t)k * w + n + i);
        dubins_build_knot<1, SOC>(kn, x, u, xn, x0v, xg, o, SOC ? cvb + mult_row(k) * 32 : nullptr, nullptr);
        const int64_t mo = (int64_t)n + n + (int64_t)(k - 1) * n;
        kkt_bwd_knot<n, m, n, 0, n, HD, SOC, 1>(kn, sb + ((int64_t)L::RF::ROWS + (int64_t)(k - 1) * L::RM::ROWS) * 32, lam,
                                                dzb + (int64_t)k * w * 32, mb + mo * 32, mb + (mo - n) * 32, nullptr);
    }
    SM_UNROLL
    for (int i = 0; i < n; ++i) { xn[i] = x[i]; x[i] = ldz(i); }
    SM_UNROLL
    for (int i = 0; i < m; ++i) u[i] = ldz(n + i);
    dubins_build_knot<0, SOC>(kn, x, u, xn, x0v, xg, o, SOC ? cvb + n * 32 : nullptr, cvb);
    kkt_bwd_knot<n, m, 0, n, n, HD, SOC, 1>(kn, sb, lam, dzb, mb, mb, nullptr);
}

// ---------------------------------------------------------------------------------------------
// One whole SQP iteration per launch (full fusion): forward sweep = linearise + statistics (f, ||c||_1,
// feas_p, feas_d with the kept multipliers, convergence freeze, :126-137) + KKT forward elimination;
// backward sweep = back-substitution + primal step + the alpha = 1 trial of the line search accumulated on
// the fly (grad f'dx, ||Lambda||_inf, f(x+dx), ||c(x+dx)||_1, c(x+dx) stored for a possible SOC solve);
// epilogue = stage 0 of dubins_linesearch_kernel (penalty, phi0, phi'0, Armijo test, accept or flag for SOC).
// L2 prefetch of one 256-byte row of a packed tile (one request per 32-byte sector): the kernel runs ~3.5 warps
// per scheduler, so the loads at the top of every knot are latency the other warps cannot cover; prefetching the
// next knot's rows costs no registers.
__device__ __forceinline__ void prefetch_row_l2(const double *p, int lane) {
    if ((lane & 3) == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

// Per-thread asynchronous prefetch ring in shared memory (cp.async, 8 bytes per row and thread): a thread copies the
// rows IT will read two knots later, so only cp.async.wait_group orders the data — no barrier.  The kernel runs one
// instance per thread with ~14 warps per SM (the batch is one wave), and ncu showed 4.5 long-scoreboard stall cycles
// per issued instruction: the loads at the top of every knot were latency nothing else could cover.
__device__ __forceinline__ void cp_async8(double *smem_dst, const double *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int PENDING>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(PENDING) : "memory"); }

// PF = true: cp.async ring (3 slots, 2 knots ahead) and 7 CTAs per SM (144 registers; 1,024 CTAs still fit in the one
// wave of 148 x 7 = 1,036); PF = false: the round-1 kernel (L2 prefetch only, 8 CTAs per SM at 128 registers).
template <bool PF>
__device__ __forceinline__ void
    dubins_sqp_step_body(double *__restrict__ Z, const double *__restrict__ x0, const double *__restrict__ xf,
                           double *__restrict__ mult_kept, double *__restrict__ cvals, double *__restrict__ scratch,
                           double *__restrict__ dz, int32_t *__restrict__ info, double *__restrict__ stats, Opts o,
                           int64_t batch, double eps_p, double eps_d, int full_step, int *__restrict__ counters) {
    using L = KktLayout<n, m, n, 0, n, LQRB_HESS_DIAG>;
    constexpr int HD = LQRB_HESS_DIAG;
    const int64_t inst = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= batch) return;
    const int64_t tile = inst >> 5;
    const int lane = (int)(inst & 31);
    const int N = o.N;
    const int64_t NN = (int64_t)N * n + (int64_t)(N - 1) * m, P = (int64_t)(N - 1) * n + 2 * n;
    double *st = stats + tile * Stats::S_COUNT * 32 + lane;
    if (st[Stats::CONV * 32] != 0.0) return;  // converged instances are frozen (:135-137)
    double *zb = Z + tile * NN * 32 + lane;
    double *cvb = cvals + tile * P * 32 + lane;
    double *sb = scratch + tile * L::rec_rows(N) * 32 + lane;
    double *dzb = dz + tile * NN * 32 + lane;
    double *mb = mult_kept + tile * P * 32 + lane;
    double xg[n], x0v[n];
    SM_UNROLL
    for (int i = 0; i < n; ++i) {
        xg[i] = xf[tile * n * 32 + lane + i * 32];
        x0v[i] = x0[tile * n * 32 + lane + i * 32];
    }
    auto ldz = [&](int64_t row) { return zb[row * 32]; };
    const double qs = o.qd * o.dt, rs = o.rd * o.dt;
    double kn[ROWS_FIRST], x[n], u[m], xn[n];

    // ---------------- forward sweep: statistics at Z + elimination
    double f = 0.0, c1 = 0.0, cinf = 0.0, fd2 = 0.0, lam_prev[n] = {0.0, 0.0, 0.0};
    // knot with controls: g at kn[w..], D1 at kn[2w..], d after D1 (and C | c of the first knot after that)
    // ---- prefetch ring: [slot][row][thread]; forward rows: x_{k+1} (n) | u_k (m) | kept lam_k (n); backward rows:
    // x_k (n) | u_k (m) | record of knot k (RM::ROWS)
    constexpr int PF_ROWS = n + m + (L::RM::ROWS > n ? L::RM::ROWS : n);
    __shared__ double pfbuf[PF ? 3 * PF_ROWS * 64 : 1];
    double *pft = pfbuf + threadIdx.x;
    auto pf_issue_fwd = [&](int k) {  // rows of knot k (1 <= k <= N-2)
        double *dst = pft + (k % 3) * PF_ROWS * 64;
        SM_UNROLL
        for (int i = 0; i < n; ++i) cp_async8(dst + i * 64, zb + ((int64_t)(k + 1) * w + i) * 32);
        SM_UNROLL
        for (int i = 0; i < m; ++i) cp_async8(dst + (n + i) * 64, zb + ((int64_t)k * w + n + i) * 32);
        SM_UNROLL
        for (int i = 0; i < n; ++i) cp_async8(dst + (w + i) * 64, mb + (mult_row(k) + i) * 32);
    };
    auto pf_issue_bwd = [&](int k) {  // rows of knot k (1 <= k <= N-2)
        double *dst = pft + (k % 3) * PF_ROWS * 64;
        SM_UNROLL
        for (int i = 0; i < w; ++i) cp_async8(dst + i * 64, zb + ((int64_t)k * w + i) * 32);
        const double *rp = sb + ((int64_t)L::RF::ROWS + (int64_t)(k - 1) * L::RM::ROWS) * 32;
        SM_UNROLL
        for (int i = 0; i < L::RM::ROWS; ++i) cp_async8(dst + (w + i) * 64, rp + i * 32);
    };
    double lk[n];
    auto knot_stats = [&](int k) {
        const double *D1 = kn + 2 * w;
        SM_UNROLL
        for (int i = 0; i < n; ++i) {
            const double e = x[i] - xg[i];
            f += 0.5 * qs * e * e;
            const double d = D1[n * w + i];
            c1 += fabs(d);
            cinf = fmax(cinf, fabs(d));
        }
        SM_UNROLL
        for (int i = 0; i < m; ++i) f += 0.5 * rs * u[i] * u[i];
        SM_UNROLL
        for (int j = 0; j < w; ++j) {
            double s = kn[w + j];
            SM_UNROLL
            for (int i = 0; i < n; ++i) s = fma(D1[i + j * n], lk[i], s);
            if (j < n) {
                if (k > 0) s -= lam_prev[j];
                else {
                    const double c = D1[n * w + n + n * w + j];  // c = x_1 - x0
                    c1 += fabs(c);
                    cinf = fmax(cinf, fabs(c));
                    s += mb[j * 32];
                }
            }
            fd2 += s * s;
        }
        SM_UNROLL
        for (int i = 0; i < n; ++i) lam_prev[i] = lk[i];
    };
    FwdCarry<n> cy;
    if constexpr (PF) {  // two knots ahead; empty groups keep the group count uniform
        if (1 < N - 1) pf_issue_fwd(1);
        cp_async_commit();
        if (2 < N - 1) pf_issue_fwd(2);
        cp_async_commit();
    }
    SM_UNROLL
    for (int i = 0; i < n; ++i) { x[i] = ldz(i); xn[i] = ldz(w + i); lk[i] = mb[(n + i) * 32]; }
    SM_UNROLL
    for (int i = 0; i < m; ++i) u[i] = ldz(n + i);
    dubins_build_knot<0, false>(kn, x, u, xn, x0v, xg, o, nullptr, nullptr);
    knot_stats(0);
    int s1 = kkt_fwd_knot<n, m, 0, n, n, HD, false, 1>(kn, sb, cy, 0);
    for (int k = 1; k < N - 1; ++k) {
        if constexpr (PF) {
            cp_async_wait<1>();  // the group of knot k has landed (at most the one of knot k+1 is pending)
            const double *src = pft + (k % 3) * PF_ROWS * 64;
            SM_UNROLL
            for (int i = 0; i < n; ++i) { x[i] = xn[i]; xn[i] = src[i * 64]; lk[i] = src[(w + i) * 64]; }
            SM_UNROLL
            for (int i = 0; i < m; ++i) u[i] = src[(n + i) * 64];
            if (k + 2 < N - 1) pf_issue_fwd(k + 2);  // slot (k+2) % 3: not the one just read, not the pending one
            cp_async_commit();
        } else {
            if (k + 2 < N) {  // next knot: u_{k+1}, x_{k+2}, kept lam_{k+1}
                SM_UNROLL
                for (int i = 0; i < w; ++i) prefetch_row_l2(zb + ((int64_t)(k + 1) * w + n + i) * 32, lane);
                SM_UNROLL
                for (int i = 0; i < n; ++i) prefetch_row_l2(mb + (mult_row(k + 1) + i) * 32, lane);
            }
            SM_UNROLL
            for (int i = 0; i < n; ++i) { x[i] = xn[i]; xn[i] = ldz((int64_t)(k + 1) * w + i); lk[i] = mb[(mult_row(k) + i) * 32]; }
            SM_UNROLL
            for (int i = 0; i < m; ++i) u[i] = ldz((int64_t)k * w + n + i);
        }
        dubins_build_knot<1, false>(kn, x, u, xn, x0v, xg, o, nullptr, nullptr);
        knot_stats(k);
        const int s2 = kkt_fwd_knot<n, m, n, 0, n, HD, false, 1>(
            kn, sb + ((int64_t)L::RF::ROWS + (int64_t)(k - 1) * L::RM::ROWS) * 32, cy, k);
        if (!s1) s1 = s2;
    }
    const int64_t rlast = (int64_t)L::RF::ROWS + (int64_t)(N - 2) * L::RM::ROWS;
    {
        SM_UNROLL
        for (int i = 0; i < n; ++i) x[i] = xn[i];
        dubins_build_knot<2, false>(kn, x, u, xn, x0v, xg, o, nullptr, nullptr);
        SM_UNROLL
        for (int i = 0; i < n; ++i) {  // terminal knot: g = Qf (x - xf), c = x_N - xf
            const double e = x[i] - xg[i];
            f += 0.5 * o.qfd * e * e;
            c1 += fabs(e);
            cinf = fmax(cinf, fabs(e));
            const double r = kn[n + i] + mb[(mult_row(N - 1) + i) * 32] - lam_prev[i];
            fd2 += r * r;
        }
        const int s2 = kkt_fwd_knot<n, 0, n, n, 0, HD, false, 1>(kn, sb + rlast * 32, cy, N - 1);
        if (!s1) s1 = s2;
    }
    if (info) info[inst] = s1;
    const double feasd = sqrt(fd2);
    st[Stats::F0 * 32] = f;
    st[Stats::C1 * 32] = c1;
    st[Stats::CINF * 32] = cinf;
    st[Stats::FEASD * 32] = feasd;
    if (cinf < eps_p && feasd < eps_d) {
        st[Stats::CONV * 32] = 1.0;
        return;
    }

    // ---------------- backward sweep: step, multipliers (kept for the next feas_d) and the alpha = 1 trial
    if constexpr (PF) {
        cp_async_wait<0>();
        if (N - 2 >= 1) pf_issue_bwd(N - 2);
        cp_async_commit();
        if (N - 3 >= 1) pf_issue_bwd(N - 3);
        cp_async_commit();
    }
    double lam[n], dzr[w], xtn[n];
    double gdx = 0.0, linf = 0.0, ft = 0.0, c1t = 0.0;
    const int64_t mlast = (int64_t)n + n + (int64_t)(N - 2) * n;
    const int64_t zlast = (int64_t)(N - 1) * w;
    kkt_bwd_knot<n, 0, n, n, 0, HD, false, 1>(kn, sb + rlast * 32, lam, dzb + zlast * 32, mb + mlast * 32,
                                              mb + (mlast - n) * 32, nullptr, dzr, &linf);
    SM_UNROLL
    for (int i = 0; i < n; ++i) {
        gdx = fma(kn[n + i], dzr[i], gdx);
        xtn[i] = x[i] + dzr[i];
        const double e = xtn[i] - xg[i];
        ft += 0.5 * o.qfd * e * e;
        c1t += fabs(e);
        cvb[(mult_row(N - 1) + i) * 32] = e;
    }
    auto knot_trial = [&](int k) {
        double xt[n], ut[m];
        SM_UNROLL
        for (int j = 0; j < w; ++j) gdx = fma(kn[w + j], dzr[j], gdx);
        SM_UNROLL
        for (int i = 0; i < n; ++i) {
            xt[i] = x[i] + dzr[i];
            const double e = xt[i] - xg[i];
            ft += 0.5 * qs * e * e;
        }
        SM_UNROLL
        for (int i = 0; i < m; ++i) {
            ut[i] = u[i] + dzr[n + i];
            ft += 0.5 * rs * ut[i] * ut[i];
        }
        double cb, sbar, dcb, dsb;
        dubins_avg(xt[2], ut[1], o.dt, cb, sbar, dcb, dsb);
        const double fx[n] = {xt[0] + o.dt * ut[0] * cb, xt[1] + o.dt * ut[0] * sbar, xt[2] + o.dt * ut[1]};
        SM_UNROLL
        for (int i = 0; i < n; ++i) {
            const double d = fx[i] - xtn[i];
            c1t += fabs(d);
            cvb[(mult_row(k) + (k == 0 ? n : 0) + i) * 32] = d;
            xtn[i] = xt[i];
        }
    };
    for (int k = N - 2; k >= 1; --k) {
        const int64_t mo = (int64_t)n + n + (int64_t)(k - 1) * n;
        if constexpr (PF) {
            cp_async_wait<1>();
            const double *src = pft + (k % 3) * PF_ROWS * 64;
            double rl[L::RM::ROWS];
            SM_UNROLL
            for (int i = 0; i < n; ++i) { xn[i] = x[i]; x[i] = src[i * 64]; }
            SM_UNROLL
            for (int i = 0; i < m; ++i) u[i] = src[(n + i) * 64];
            SM_UNROLL
            for (int i = 0; i < L::RM::ROWS; ++i) rl[i] = src[(w + i) * 64];
            if (k - 2 >= 1) pf_issue_bwd(k - 2);
            cp_async_commit();
            dubins_build_knot<1, false>(kn, x, u, xn, x0v, xg, o, nullptr, nullptr);
            kkt_bwd_knot<n, m, n, 0, n, HD, false, 1, 1>(kn, rl, lam, dzb + (int64_t)k * w * 32, mb + mo * 32,
                                                         mb + (mo - n) * 32, nullptr, dzr, &linf);
        } else {
            if (k >= 2) {  // previous knot: z_{k-1} and its record
                SM_UNROLL
                for (int i = 0; i < w; ++i) prefetch_row_l2(zb + ((int64_t)(k - 1) * w + i) * 32, lane);
                const double *rp = sb + ((int64_t)L::RF::ROWS + (int64_t)(k - 2) * L::RM::ROWS) * 32;
                SM_UNROLL
                for (int i = 0; i < L::RM::ROWS; ++i) prefetch_row_l2(rp + i * 32, lane);
            }
            SM_UNROLL
            for (int i = 0; i < n; ++i) { xn[i] = x[i]; x[i] = ldz((int64_t)k * w + i); }
            SM_UNROLL
            for (int i = 0; i < m; ++i) u[i] = ldz((int64_t)k * w + n + i);
            dubins_build_knot<1, false>(kn, x, u, xn, x0v, xg, o, nullptr, nullptr);
            kkt_bwd_knot<n, m, n, 0, n, HD, false, 1>(kn, sb + ((int64_t)L::RF::ROWS + (int64_t)(k - 1) * L::RM::ROWS) * 32, lam,
                                                      dzb + (int64_t)k * w * 32, mb + mo * 32, mb + (mo - n) * 32, nullptr,
                                                      dzr, &linf);
        }
        knot_trial(k);
    }
    if constexpr (PF) cp_async_wait<0>();
    SM_UNROLL
    for (int i = 0; i < n; ++i) { xn[i] = x[i]; x[i] = ldz(i); }
    SM_UNROLL
    for (int i = 0; i < m; ++i) u[i] = ldz(n + i);
    dubins_build_knot<0, false>(kn, x, u, xn, x0v, xg, o, nullptr, nullptr);
    kkt_bwd_knot<n, m, 0, n, n, HD, false, 1>(kn, sb, lam, dzb, mb, mb, nullptr, dzr, &linf);
    knot_trial(0);
    SM_UNROLL
    for (int i = 0; i < n; ++i) {  // c_1(x + dx) = x_1 + dx_1 - x0
        const double c = xtn[i] - x0v[i];
        c1t += fabs(c);
        cvb[i * 32] = c;
    }

    // ---------------- stage 0 of the line search (src/sqp.jl:72-94)
    st[Stats::ITERS * 32] += 1.0;
    bool take = full_step != 0;
    if (!take) {
        const double eta = 1e-4;
        const double mu = fmax(st[Stats::MU * 32], 1.1 * linf);  // mu <- max(mu, 1.1 ||lambda||_inf)
        st[Stats::MU * 32] = mu;
        const double phi0 = f + mu * c1, dphi0 = gdx - mu * c1;
        st[Stats::PHI0 * 32] = phi0;
        st[Stats::DPHI0 * 32] = dphi0;
        take = ft + mu * c1t <= phi0 + eta * dphi0;
    }
    st[Stats::ALPHA * 32] = 1.0;
    if (take) {
        for (int64_t r = 0; r < NN; ++r) zb[r * 32] += dzb[r * 32];
        st[Stats::DONE * 32] = 1.0;
    } else {
        st[Stats::DONE * 32] = 0.0;
        atomicAdd(&counters[0], 1);  // needs the second-order correction solve
    }
}

// 65,536 instances = 1,024 CTAs of 64 threads must fit in ONE wave: 148 x 8 at 128 registers (round-1 kernel), or
// 148 x 7 = 1,036 at 144 registers for the prefetching variant (its ring takes 21.5 KB of shared memory per CTA).
__global__ void __launch_bounds__(64, 8)
    dubins_sqp_step_kernel(double *__restrict__ Z, const double *__restrict__ x0, const double *__restrict__ xf,
                           double *__restrict__ mult_kept, double *__restrict__ cvals, double *__restrict__ scratch,
                           double *__restrict__ dz, int32_t *__restrict__ info, double *__restrict__ stats, Opts o,
                           int64_t batch, double eps_p, double eps_d, int full_step, int *__restrict__ counters) {
    dubins_sqp_step_body<false>(Z, x0, xf, mult_kept, cvals, scratch, dz, info, stats, o, batch, eps_p, eps_d, full_step, counters);
}
__global__ void __maxnreg__(144)
    dubins_sqp_step_pf_kernel(double *__restrict__ Z, const double *__restrict__ x0, const double *__restrict__ xf,
                              double *__restrict__ mult_kept, double *__restrict__ cvals, double *__restrict__ scratch,
                              double *__restrict__ dz, int32_t *__restrict__ info, double *__restrict__ stats, Opts o,
                              int64_t batch, double eps_p, double eps_d, int full_step, int *__restrict__ counters) {
    dubins_sqp_step_body<true>(Z, x0, xf, mult_kept, cvals, scratch, dz, info, stats, o, batch, eps_p, eps_d, full_step, counters);
}

// Line search stages (src/sqp.jl:72-94).
//   stage 0: penalty update, phi0, phi'0; trial alpha = 1; on failure write c(x+dx) into the data rows
//            for the second-order correction solve and set need_soc.
//   stage 1: second-order-correction trial x + dx + dx^; on failure alpha = rho.
//   stage 2: trial at the current alpha; on failure alpha *= rho.
// full_step != 0 skips the tests and takes alpha = 1 (line_search = 0).
template <bool FUSED>
__global__ void __launch_bounds__(64) dubins_linesearch_kernel(double *__restrict__ Z, const double *__restrict__ dz,
                                                               const double *__restrict__ dzh, const double *__restrict__ mult,
                                                               double *__restrict__ mult_kept,
                                                               const double *__restrict__ x0, const double *__restrict__ xf,
                                                               double *__restrict__ data, double *__restrict__ stats, Opts o,
                                                               int64_t batch, int stage, int full_step,
                                                               int *__restrict__ counters) {
    const int64_t inst = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= batch) return;
    const int64_t tile = inst >> 5;
    const int lane = (int)(inst & 31);
    const int N = o.N;
    const int64_t NN = (int64_t)N * n + (int64_t)(N - 1) * m, P = (int64_t)(N - 1) * n + 2 * n;
    double *zb = Z + tile * NN * 32 + lane;
    const double *dzb = dz + tile * NN * 32 + lane;
    const double *dhb = dzh ? dzh + tile * NN * 32 + lane : nullptr;
    double *db = data + tile * (FUSED ? P : data_rows(N)) * 32 + lane;  // FUSED: compact constraint values
    double *sb = stats + tile * Stats::S_COUNT * 32 + lane;
    const double *x0b = x0 + tile * n * 32 + lane, *xfb = xf + tile * n * 32 + lane;
    if (sb[Stats::CONV * 32] != 0.0) return;  // converged instances are frozen (:135-137)
    if (stage > 0 && sb[Stats::DONE * 32] != 0.0) return;
    double xg[n];
    for (int i = 0; i < n; ++i) xg[i] = xfb[i * 32];
    const double eta = 1e-4, rho = 0.5;

    auto accept = [&](double alpha, bool with_soc) {
        for (int64_t r = 0; r < NN; ++r) {
            double v = fma(alpha, dzb[r * 32], zb[r * 32]);
            if (with_soc) v += dhb[r * 32];
            zb[r * 32] = v;
        }
        sb[Stats::DONE * 32] = 1.0;
        sb[Stats::ALPHA * 32] = alpha;
    };

    if (stage == 0) {
        sb[Stats::ITERS * 32] += 1.0;
        sb[Stats::DONE * 32] = 0.0;
        {   // the multipliers of this QP step become the solver's current ones (converged instances keep theirs)
            const double *mb = mult + tile * P * 32 + lane;
            double *mk = mult_kept + tile * P * 32 + lane;
            for (int64_t r = 0; r < P; ++r) mk[r * 32] = mb[r * 32];
        }
        if (full_step) {
            accept(1.0, false);
            return;
        }
        // penalty: mu <- max(mu, 1.1 ||lambda||_inf)
        const double *mb = mult + tile * P * 32 + lane;
        double linf = 0.0;
        for (int64_t r = 0; r < P; ++r) linf = fmax(linf, fabs(mb[r * 32]));
        const double mu = fmax(sb[Stats::MU * 32], 1.1 * linf);
        sb[Stats::MU * 32] = mu;
        // phi'(x, dx) = grad f'dx - mu ||c(x)||_1  with grad f = the g rows of the packed data
        double gdx = 0.0;
        for (int k = 0; k < N; ++k) {
            const int wk = k < N - 1 ? w : n;
            if (FUSED) {  // g = [Q (x - xf) dt; R u dt] (terminal: Qf), the same numbers the linearisation forms
                const double qs = k < N - 1 ? o.qd * o.dt : o.qfd, rs = o.rd * o.dt;
                for (int j = 0; j < wk; ++j) {
                    const double zj = zb[((int64_t)k * w + j) * 32];
                    const double gj = j < n ? qs * (zj - xg[j]) : rs * zj;
                    gdx = fma(gj, dzb[((int64_t)k * w + j) * 32], gdx);
                }
            } else {
                const double *gp = db + (knot_row(k, N) + wk) * 32;
                for (int j = 0; j < wk; ++j) gdx = fma(gp[j * 32], dzb[((int64_t)k * w + j) * 32], gdx);
            }
        }
        const double phi0 = sb[Stats::F0 * 32] + mu * sb[Stats::C1 * 32];
        const double dphi0 = gdx - mu * sb[Stats::C1 * 32];
        sb[Stats::PHI0 * 32] = phi0;
        sb[Stats::DPHI0 * 32] = dphi0;
        double f, c1;
        dubins_eval<FUSED ? 2 : 1>(zb, dzb, nullptr, 1.0, x0b, xg, o, db, f, c1);
        if (f + mu * c1 <= phi0 + eta * dphi0) {
            accept(1.0, false);
        } else {
            sb[Stats::ALPHA * 32] = 1.0;
            atomicAdd(&counters[0], 1);  // needs the second-order correction solve
        }
        return;
    }
    const double mu = sb[Stats::MU * 32], phi0 = sb[Stats::PHI0 * 32], dphi0 = sb[Stats::DPHI0 * 32];
    double f, c1;
    if (stage == 1) {
        dubins_eval<0>(zb, dzb, dhb, 1.0, x0b, xg, o, db, f, c1);
        if (f + mu * c1 < phi0 + eta * dphi0) {
            accept(1.0, true);
        } else {
            sb[Stats::ALPHA * 32] = rho;
            atomicAdd(&counters[1], 1);
        }
        return;
    }
    const double alpha = sb[Stats::ALPHA * 32];
    dubins_eval<0>(zb, dzb, nullptr, alpha, x0b, xg, o, db, f, c1);
    if (f + mu * c1 <= phi0 + eta * alpha * dphi0) {
        accept(alpha, false);
    } else {
        sb[Stats::ALPHA * 32] = alpha * rho;
        atomicAdd(&counters[1], 1);
    }
}

__global__ void stats_init_kernel(double *stats, int64_t batch) {
    const int64_t inst = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= batch) return;
    double *sb = stats + (inst >> 5) * Stats::S_COUNT * 32 + (inst & 31);
    for (int r = 0; r < Stats::S_COUNT; ++r) sb[r * 32] = 0.0;
    sb[Stats::MU * 32] = 1.0;  // reset!: merit.mu = 1 (src/cholesky_solver.jl:88-94)
}

__global__ void stats_export_kernel(const double *stats, double *feas_p, double *feas_d, int32_t *iters, int64_t batch) {
    const int64_t inst = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= batch) return;
    const double *sb = stats + (inst >> 5) * Stats::S_COUNT * 32 + (inst & 31);
    if (feas_p) feas_p[inst] = sb[Stats::CINF * 32];
    if (feas_d) feas_d[inst] = sb[Stats::FEASD * 32];
    if (iters) iters[inst] = (int32_t)sb[Stats::ITERS * 32];
}

}  // namespace

extern "C" int32_t lqrb_sqp_dubins_f64(lqrb_handle_t h, int64_t batch, const lqrb_sqp_options_t *opts,
                                       const double *x0, const double *xf, double *Z, double *feas_p,
                                       double *feas_d, int32_t *iters_done, int64_t *kkt_solves) {
    if (!h) return -1;
    if (batch < 0) return lqrb_fail(h, -2, "batch < 0");
    if (!opts || opts->N < 3 || opts->iters < 0 || !(opts->dt > 0.0)) return lqrb_fail(h, -3, "bad options");
    if (!x0) return lqrb_fail(h, -4, "x0 is NULL");
    if (!xf) return lqrb_fail(h, -5, "xf is NULL");
    if (!Z) return lqrb_fail(h, -6, "Z is NULL");
    if (kkt_solves) *kkt_solves = 0;
    if (batch == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const int N = opts->N;
    const int64_t NN = lqrb_num_vars(n, m, N), P = (int64_t)(N - 1) * n + 2 * n;
    const int64_t ldb = lqrb_padded_batch(batch);
    std::vector<int32_t> p((size_t)N, 0);
    p[0] = n;
    p[N - 1] = n;
    const int64_t drows = lqrb_kkt_data_rows(n, m, N, p.data(), LQRB_HESS_DIAG, 0);

    // fused (default): the KKT kernel linearises each knot on the fly; sqp_fused = 0 keeps the three-kernel
    // path (linearise -> packed data -> generic KKT solve) that it is tested against
    const bool fused = h->opt("sqp_fused", 1) != 0;
    // device buffers: [Zp | dz | dzh | mult | multh | x0p | xfp | stats] in SQP0, data (or c values) in SQP1
    const size_t nd = (size_t)ldb * (3 * NN + 3 * P + 2 * n + Stats::S_COUNT);
    double *buf = (double *)lqrb_scratch(h, SCR_SQP0, nd * 8);
    double *data = (double *)lqrb_scratch(h, SCR_SQP1, (size_t)ldb * (fused ? P : drows) * 8);
    using FL = KktLayout<n, m, n, 0, n, LQRB_HESS_DIAG>;
    double *frec = fused ? (double *)lqrb_scratch(h, SCR_FACT, (size_t)ldb * FL::rec_rows(N) * 8) : nullptr;
    if (fused && !frec) return 1000 + (int)cudaErrorMemoryAllocation;
    int *counters = (int *)lqrb_scratch(h, SCR_SQP2, 64);
    int32_t *dinfo = (int32_t *)lqrb_scratch(h, SCR_SQP3, (size_t)ldb * 4);
    if (!buf || !data || !counters || !dinfo) return 1000 + (int)cudaErrorMemoryAllocation;
    double *Zp = buf, *dz = Zp + ldb * NN, *dzh = dz + ldb * NN, *mult = dzh + ldb * NN, *multh = mult + ldb * P,
           *multk = multh + ldb * P, *x0p = multk + ldb * P, *xfp = x0p + ldb * n, *stats = xfp + ldb * n;

    // Z is updated in place; the scratch above belongs to lane 0, where a call in one chunk runs
    int64_t solves = 0;
    const int32_t rc = lqrb_for_chunks(
        h, batch, batch, {{Z, NN * 8}, {x0, n * 8}, {xf, n * 8}}, {{Z, NN * 8}, {feas_p, 8}, {feas_d, 8}, {iters_done, 4}},
        [&](Lane lane, int64_t, const void *const *in, void *const *out) -> int32_t {
            const cudaStream_t s = lane.stream;
            ArrayTable t = {};
            t.ptr[0] = (const double *)in[0]; t.stride[0] = NN;
            int32_t rc = lqrb_gather_pack(h, lqrb_identity_map(h, NN), t, batch, LQRB_TILE, Zp, s);
            if (rc) return rc;
            t.ptr[0] = (const double *)in[1]; t.stride[0] = n;
            rc = lqrb_gather_pack(h, lqrb_identity_map(h, n), t, batch, LQRB_TILE, x0p, s);
            if (rc) return rc;
            t.ptr[0] = (const double *)in[2];
            rc = lqrb_gather_pack(h, lqrb_identity_map(h, n), t, batch, LQRB_TILE, xfp, s);
            if (rc) return rc;
            LQRB_CUDA(h, cudaMemsetAsync(multk, 0, (size_t)ldb * P * 8, s));

            const Opts o{N, opts->dt, opts->q_diag, opts->r_diag, opts->qf_diag};
            const unsigned grid = (unsigned)((batch + 63) / 64);
            stats_init_kernel<<<grid, 64, 0, s>>>(stats, batch);
            LQRB_LAUNCH_CHECK(h, "stats_init_kernel");
            int hc[2];
            for (int it = 0; it < opts->iters; ++it) {
                // update! + convergence check (:126-137)
                if (fused) {
                    // update! + convergence check + _solve! + line-search stage 0 in one kernel
                    LQRB_CUDA(h, cudaMemsetAsync(counters, 0, 8, s));
                    // the cp.async ring measured SLOWER than the L2 prefetch (config 4: 23.9 vs 18.7 ms, same box): option only
                    if (h->opt("sqp_prefetch", 0))
                        dubins_sqp_step_pf_kernel<<<grid, 64, 0, s>>>(Zp, x0p, xfp, multk, data, frec, dz, dinfo, stats, o, batch,
                                                                         opts->eps_p, opts->eps_d, opts->line_search ? 0 : 1, counters);
                    else
                        dubins_sqp_step_kernel<<<grid, 64, 0, s>>>(Zp, x0p, xfp, multk, data, frec, dz, dinfo, stats, o, batch,
                                                                          opts->eps_p, opts->eps_d, opts->line_search ? 0 : 1, counters);
                    h->kernel_name = "dubins_sqp_step<3,2,p=3/0/3,hess=2>";
                    LQRB_LAUNCH_CHECK(h, "dubins_sqp_step_kernel");
                } else {
                    dubins_linearize_kernel<true><<<grid, 64, 0, s>>>(Zp, x0p, xfp, multk, data, stats, o, batch, 1, opts->eps_p, opts->eps_d);
                    LQRB_LAUNCH_CHECK(h, "dubins_linearize_kernel");
                    // _solve! (:143)
                    rc = lqrb_kkt_solve_packed_on(h, n, m, N, batch, p.data(), LQRB_HESS_DIAG, 0, 0, data, dz, mult, nullptr, dinfo, lane);
                    if (rc) return rc;
                }
                solves += batch;
                // line search (:146; spec src/sqp.jl:72-94)
                if (!fused) {
                    LQRB_CUDA(h, cudaMemsetAsync(counters, 0, 8, s));
                    dubins_linesearch_kernel<false><<<grid, 64, 0, s>>>(Zp, dz, nullptr, mult, multk, x0p, xfp, data, stats, o, batch, 0,
                                                                        opts->line_search ? 0 : 1, counters);
                    LQRB_LAUNCH_CHECK(h, "dubins_linesearch_kernel");
                }
                if (!opts->line_search) continue;
                LQRB_CUDA(h, cudaMemcpyAsync(hc, counters, 8, cudaMemcpyDeviceToHost, s));
                LQRB_CUDA(h, cudaStreamSynchronize(s));
                if (hc[0] == 0) continue;
                // second-order correction: same chain with Ginv=false on c(x+dx) (:254-273)
                if (fused) {
                    dubins_kkt_fused_kernel<true><<<grid, 64, 0, s>>>(Zp, x0p, xfp, data, frec, dzh, multh, dinfo, o, batch);
                    LQRB_LAUNCH_CHECK(h, "dubins_kkt_fused_kernel");
                } else {
                    rc = lqrb_kkt_solve_packed_on(h, n, m, N, batch, p.data(), LQRB_HESS_DIAG, 0, LQRB_FLAG_SOC, data, dzh, multh,
                                                  nullptr, dinfo, lane);
                    if (rc) return rc;
                }
                solves += batch;
                int pending = hc[0];
                // trial 1 = the SOC step; trials 2..10 = the reference's back-tracking iterations i = 2..10 (alpha = rho^1..rho^9,
                // src/sqp.jl:76-92)
                for (int trial = 1; trial < 11 && pending > 0; ++trial) {
                    LQRB_CUDA(h, cudaMemsetAsync(counters, 0, 8, s));
                    if (fused)
                        dubins_linesearch_kernel<true><<<grid, 64, 0, s>>>(Zp, dz, dzh, mult, multk, x0p, xfp, data, stats, o, batch,
                                                                           trial == 1 ? 1 : 2, 0, counters);
                    else
                        dubins_linesearch_kernel<false><<<grid, 64, 0, s>>>(Zp, dz, dzh, mult, multk, x0p, xfp, data, stats, o, batch,
                                                                            trial == 1 ? 1 : 2, 0, counters);
                    LQRB_LAUNCH_CHECK(h, "dubins_linesearch_kernel");
                    LQRB_CUDA(h, cudaMemcpyAsync(hc, counters, 8, cudaMemcpyDeviceToHost, s));
                    LQRB_CUDA(h, cudaStreamSynchronize(s));
                    pending = hc[1];
                }
            }
            // final feasibility numbers at the returned iterate
            dubins_linearize_kernel<false><<<grid, 64, 0, s>>>(Zp, x0p, xfp, multk, nullptr, stats, o, batch, 0, opts->eps_p, opts->eps_d);
            LQRB_LAUNCH_CHECK(h, "dubins_linearize_kernel");

            // export
            ArrayTableOut to = {};
            to.ptr[0] = (double *)out[0]; to.stride[0] = NN;
            rc = lqrb_scatter_unpack(h, lqrb_identity_map(h, NN), to, batch, LQRB_TILE, Zp, s);
            if (rc) return rc;
            stats_export_kernel<<<grid, 64, 0, s>>>(stats, (double *)out[1], (double *)out[2], (int32_t *)out[3], batch);
            LQRB_LAUNCH_CHECK(h, "stats_export_kernel");
            return 0;
        });
    if (rc) return rc;
    if (kkt_solves) *kkt_solves = solves;
    return 0;
}
