/*
 * lqrb200.h — C ABI of liblqrb200.so, the B200 (sm_100a) batched LQR / KKT solver.
 *
 * This is the drop-in boundary for the hot path of bjack205/LQR.jl.  The reference is pure Julia
 * with no FFI of its own (SURVEY §8b), so each entry point below names the Julia function(s) it
 * replaces; the Julia `ccall` shim that re-exposes the reference's names on top of this header is
 * lqr.jl_b200/julia/LQRB200.jl, and INTEGRATION.md shows the binding a maintainer would add.
 *
 * Conventions
 *   - plain C types only; every array is caller-owned; the library owns only its handle and internal scratch.
 *   - instance-major arrays may be host or device memory.  A call is device-resident when every non-NULL
 *     array it is given, inputs and outputs alike, is device or managed memory (cudaPointerGetAttributes):
 *     it then runs on the handle's stream and returns without synchronising.  Any other call is staged:
 *     its arrays are copied through device buffers in chunks over two internal streams (each copy
 *     cudaMemcpyDefault, so device arrays in a staged call are fine), and it returns when done.
 *   - every function returns int32: 0 ok; -i = argument i (1-based) invalid (LAPACK style);
 *     >0 = 1000 + cudaError_t.  Nothing throws across the ABI.  lqrb_last_error_string() explains.
 *   - numerical failure never aborts a batch: per-instance `info[batch]` mirrors the potrf `info`
 *     the reference surfaces at src/cholesky_solve.jl:1-3:
 *         0 ok;  otherwise (knot+1)*1000 + stage*100 + (1-based pivot index),
 *         stage 0 = cost-Hessian / Riccati E block, 1 = Schur B block, 2 = Schur C block;
 *     pivots count in the caller's numbering (a padded shape's codes are mapped back).  KKT: as in the
 *     reference, which factors every H_k first, a Hessian failure at any knot takes precedence over a
 *     Schur-block failure; otherwise the first failure in knot order is reported.
 *   - one handle per host thread / GPU, stream ordered, no global state (SURVEY §8b threading).
 *
 * Two data layouts
 *   INSTANCE-MAJOR ("Julia order"): what LQR.jl holds — one instance contiguous, every small matrix
 *     column-major, knot index next, batch index outermost.  E.g. A is Float64[n, n, N-1, batch].
 *   PACKED tiled batch-minor SoA (device resident, the layout the kernels stream): [tile][rows][T]
 *     doubles, a tile = T consecutive instances, element (row, inst) at
 *         ((inst / T) * rows + row) * T + inst % T,        ldb = lqrb_padded_batch(batch) instances.
 *     T depends on the size class: T = 32 where one THREAD owns an instance (a warp reads one row of
 *     its tile as one 256-byte line), T = 1 (plain per-instance records in the same row order) where a
 *     half-warp, warp or CTA owns an instance and bulk-copies whole knot records.  Query it with
 *     lqrb_riccati_tile_width / lqrb_kkt_tile_width; the *_pack_f64 / *_unpack_f64 entry points apply
 *     it themselves.  "[rows][ldb]" in the comments below is shorthand for this tiled layout.  Row
 *     maps are given by the *_layout functions below.
 */
#ifndef LQRB200_H
#define LQRB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LQRB_VERSION 100 /* 0.1.0 */

/* Hessian storage modes = the three BlockCholesky modes, src/block_cholesky.jl:55-91 */
#define LQRB_HESS_DENSE 0     /* H_k = [Q Hux'; Hux R], whole-matrix potrf (:55-66)            */
#define LQRB_HESS_BLOCKDIAG 1 /* Hux = 0, separate potrf of Q and R (:69-77)                   */
#define LQRB_HESS_DIAG 2      /* Diagonal storage: stores the inverse, solve = multiply (:82-91) */

/* flags */
#define LQRB_FLAG_SOC 1     /* Ginv=false: H=I, g=0 (second_order_correction!, src/cholesky_solver.jl:254-273) */
#define LQRB_FLAG_LTI 2     /* Riccati: A,B,Q,R,q,r carry no knot axis (LQRProblem, src/lqr_problem.jl:1-11) */
#define LQRB_FLAG_NO_AFFINE 4 /* Riccati: q, r, qf are absent/zero (the reference's DPSolver form) */

typedef struct lqrb_context *lqrb_handle_t;

/* ---------------------------------------------------------------- library / handle ---------- */
int32_t lqrb_version(void);
int32_t lqrb_device_count(int32_t *count);
int32_t lqrb_create(lqrb_handle_t *handle, int32_t device);
int32_t lqrb_destroy(lqrb_handle_t handle);
const char *lqrb_last_error_string(lqrb_handle_t handle);
/* cudaStream_t to order all work of this handle on (NULL = the handle's own stream). */
int32_t lqrb_set_stream(lqrb_handle_t handle, void *cuda_stream);
int32_t lqrb_synchronize(lqrb_handle_t handle);
/* number of kernels this handle has launched so far (bench.py's gpu_launches). */
int64_t lqrb_launch_count(lqrb_handle_t handle);
/* kernel variant used by the last solve on this handle ("riccati_tpi<4,1>", ...). */
const char *lqrb_last_kernel_name(lqrb_handle_t handle);
/* tuning knob: 0 = default choice, otherwise force a variant (see DESIGN.md). */
int32_t lqrb_set_option(lqrb_handle_t handle, const char *name, int64_t value);

/* Diagnostic: best FP64 throughput (TFLOP/s) of this device over `seconds` of back-to-back launches of a
 * register-only kernel; kind 0 = DFMA (vector pipe), 1 = DMMA (mma.sync.m8n8k4.f64, tensor pipe).  These are the
 * peaks the FP64-bound rooflines in DESIGN.md / bench.py are quoted against (SURVEY §8d: "to be measured"). */
int32_t lqrb_fp64_peak_f64(lqrb_handle_t handle, int32_t kind, double seconds, double *tflops);

/* ---------------------------------------------------------------- layouts -------------------- */
int64_t lqrb_padded_batch(int64_t batch); /* ldb: batch rounded up to a multiple of 32 */

/* LQRProblem / Primals sizes: src/lqr_problem.jl:21-25 (num_vars = N*n + (N-1)*m). */
int64_t lqrb_num_vars(int32_t n, int32_t m, int32_t N);
/* number of constraint rows P = sum(p) + (N-1)*n   (src/conblocks.jl:74-96 with dynamics coupling). */
int64_t lqrb_num_cons(int32_t n, int32_t N, const int32_t *p);

/* Riccati packed rows.
 *   knots : [(LTI ? 1 : N-1)][F][ldb]  per knot: A (n*n col-major) | B (n*m) | Q (upper packed,
 *           idx(i,j)=j(j+1)/2+i) | R (upper packed) | q (n) | r (m);  F = rows_per_knot (for n = 8, 12 with
 *           m = 2, 3 one padding row follows r so that F is even: take F from lqrb_riccati_layout)
 *   term  : [n(n+1)/2 + 2n][ldb]       Qf (upper packed) | qf (n) | x0 (n)
 *   Z     : [N*n+(N-1)*m][ldb]         Primals order [x1;u1;x2;u2;...;xN] (src/lqr_problem.jl:46-73)
 *   K     : [(N-1)*(m*n+m)][ldb]       per knot: K (m*n col-major) | kff (m)                      */
typedef struct {
    int64_t rows_per_knot, knot_count, term_rows, z_rows, gain_rows;
} lqrb_riccati_layout_t;
int32_t lqrb_riccati_layout(int32_t n, int32_t m, int32_t N, int32_t flags,
                            lqrb_riccati_layout_t *out);

/* KKT packed rows (one "data" array, knot after knot; offsets in the layout struct).
 *   knot k: H_k (DIAG: w | BLOCKDIAG: tri(n)+tri(m_k) | DENSE: tri(w), upper packed) | g_k (w)
 *           | [k<N-1] D1_k=[A_k B_k] (n*w col-major) | d_k (n)
 *           | [k>0 and explicit D2] D2_k (n*w col-major)
 *           | C_k (p_k*w col-major) | c_k (p_k)                 with w = n + (k<N-1 ? m : 0)
 *   outputs: dz [NN][ldb] Primals order; mult [P][ldb] order [mu_1;lam_1;...;mu_N]
 *            (src/jacobian_blocks.jl:181-195); res [NN][ldb] = D1'lam+C'mu+D2'lam_prev+g
 *            (src/cholesky_solver.jl:201-236).                                                   */
int64_t lqrb_kkt_data_rows(int32_t n, int32_t m, int32_t N, const int32_t *p, int32_t hess_mode,
                           int32_t explicit_d2);
/* row offset of knot k in the packed data array (k = N gives the total). */
int64_t lqrb_kkt_knot_offset(int32_t n, int32_t m, int32_t N, const int32_t *p, int32_t hess_mode,
                             int32_t explicit_d2, int32_t k);

/* ---------------------------------------------------------------- Riccati ------------------- */
/* Replaces DPSolver solve! : src/dynamic_programming.jl:54-72 (compute_gain! :37-43,
 * compute_ctg! :48-52, chol_solve! :28-31) and the rollout of src/least_squares.jl:195-202,
 * generalised to per-knot (LTV) data and affine cost terms (SURVEY Appendix A).
 *
 * Instance-major arrays (host or device):
 *   A[n,n,Kn,batch] B[n,m,Kn,batch] Q[n,n,Kn,batch] R[m,m,Kn,batch] q[n,Kn,batch] r[m,Kn,batch]
 *   Qf[n,n,batch] qf[n,batch] x0[n,batch]       Kn = (flags & LTI) ? 1 : N-1; q, r, qf may be NULL
 * Outputs: Z[NN,batch] (Primals order), optional K[m,n,N-1,batch], kff[m,N-1,batch], info[batch].
 * With host pointers the call does H2D -> pack -> solve -> unpack -> D2H, chunked over two
 * streams so copies overlap compute.                                                             */
int32_t lqrb_riccati_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                         int32_t flags, const double *A, const double *B, const double *Q,
                         const double *R, const double *q, const double *r, const double *Qf,
                         const double *qf, const double *x0, double *Z, double *K, double *kff,
                         int32_t *info);

/* Gradient of a scalar loss l(Z) through lqrb_riccati_f64: given the inputs, that call's output Z and dZ = dl/dZ
 * (same shape as Z), writes dl/d of every input.  The adjoint LQR (same A, B, Q, R, Qf, linear terms dZ, initial
 * state 0) is solved by the same kernels as the forward solve, then one backward sweep forms the costates and the
 * gradients (DESIGN §4.8).
 *   inputs as in lqrb_riccati_f64 (x0 is not needed); Z[NN,batch], dZ[NN,batch]
 *   outputs gA, gB, gQ, gR, gq, gr, gQf, gqf, gx0: the shape of their input (Kn = 1 under LQRB_FLAG_LTI: the sum over
 *   the knots); any may be NULL, not all.  gq, gr, gqf are available with LQRB_FLAG_NO_AFFINE or NULL q, r, qf.
 *   The kernels read only the upper triangle of Q, R, Qf: their gradients are returned as the symmetric matrices
 *   (1/2)(x^ x' + x x^'); a finite-difference check perturbs (i,j) and (j,i) together.
 *   info[batch] | NULL: the potrf info of the adjoint solve (the same matrices as the forward solve).  The gradients
 *   of an instance with info != 0 carry no meaning.
 * Host or device pointers, with the staged / device-resident rule of every entry point.                      */
int32_t lqrb_riccati_grad_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                              int32_t flags, const double *A, const double *B, const double *Q,
                              const double *R, const double *q, const double *r, const double *Qf,
                              const double *qf, const double *Z, const double *dZ, double *gA, double *gB,
                              double *gQ, double *gR, double *gq, double *gr, double *gQf, double *gqf,
                              double *gx0, int32_t *info);

/* Gradient of a scalar loss l(Z, K, kff) through lqrb_riccati_f64, the policy outputs included: given the inputs,
 * that call's Z and the cotangents dZ = dl/dZ, dK = dl/dK, dkff = dl/dkff, writes the total dl/d of every input.  The
 * Z part is lqrb_riccati_grad_f64's; the gains part recomputes the recursion into a per-knot tape and runs its adjoint
 * forward over the knots (DESIGN §4.10).
 *   inputs and outputs as in lqrb_riccati_grad_f64; dK[m,n,N-1,batch], dkff[m,N-1,batch] in the layout of the forward
 *   call's K, kff.  dZ, dK, dkff may each be NULL, not all three; Z is read only when dZ is given.  With dZ = NULL, gx0
 *   is written as zeros (the gains do not depend on x0).  With dK = dkff = NULL the result is bitwise that of
 *   lqrb_riccati_grad_f64.
 *   info[batch] | NULL: 0, or the forward solve's code for the first failed factorisation.
 *   Error codes: -6 flags other than LTI / NO_AFFINE; -7..-10, -13 A, B, Q, R or Qf NULL; -15 Z NULL while dZ is
 *   given; -16 every cotangent NULL; -19 every output NULL; shapes the solve rejects with the solve's code.
 * Host or device pointers, with the staged / device-resident rule of every entry point.                      */
int32_t lqrb_riccati_grad_gains_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                                    int32_t flags, const double *A, const double *B, const double *Q,
                                    const double *R, const double *q, const double *r, const double *Qf,
                                    const double *qf, const double *Z, const double *dZ, const double *dK,
                                    const double *dkff, double *gA, double *gB, double *gQ, double *gR, double *gq,
                                    double *gr, double *gQf, double *gqf, double *gx0, int32_t *info);

/* Device-resident split of the same call (all pointers are DEVICE pointers). */
int32_t lqrb_riccati_pack_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                              int32_t flags, const double *A, const double *B, const double *Q,
                              const double *R, const double *q, const double *r, const double *Qf,
                              const double *qf, const double *x0, double *knots, double *term);
/* gains may be NULL (internal scratch is used); info may be NULL. */
int32_t lqrb_riccati_solve_packed_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N,
                                      int64_t batch, int32_t flags, const double *knots,
                                      const double *term, double *Z, double *gains, int32_t *info);
/* tile width T (1 or 32) of the packed arrays of this size class on this handle (> 0; < 0 = bad argument). */
int32_t lqrb_riccati_tile_width(lqrb_handle_t handle, int32_t n, int32_t m);
/* packed outputs of lqrb_riccati_solve_packed_f64 -> instance-major Z[NN,batch], optional
 * K[m,n,N-1,batch], kff[m,N-1,batch] (gains may be NULL when neither is wanted); device pointers. */
int32_t lqrb_riccati_unpack_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                                const double *Z_packed, const double *gains_packed, double *Z,
                                double *K, double *kff);
/* generic: packed [tile][rows][T] -> instance-major [rows, batch] (and back); device pointers;
 * `tile` = the T of the size class that produced / will consume the array (1 or 32). */
int32_t lqrb_unpack_rows_f64(lqrb_handle_t handle, int64_t rows, int64_t batch, int32_t tile,
                             const double *packed, double *instance_major);
int32_t lqrb_pack_rows_f64(lqrb_handle_t handle, int64_t rows, int64_t batch, int32_t tile,
                           const double *instance_major, double *packed);

/* forward simulate with given controls: rollout!, src/least_squares.jl:195-202.
 * Instance-major, host or device: A,B as above, x0[n,batch], U[m,N-1,batch] -> X[n,N,batch]. */
int32_t lqrb_rollout_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                         int32_t flags, const double *A, const double *B, const double *x0,
                         const double *U, double *X);

/* Replaces solve!(sol, ::LeastSquaresSolver, prob) : src/least_squares.jl:158-190 — the condensed form of the
 * unconstrained LTI problem: T (block Toeplitz, build_toeplitz :136-156), (T' Qbar T + Rbar) U = -T' Qbar L x0 by
 * Cholesky (:176-178), then rollout! (:195-202).  O((N m)^3) work and (N m)^2 doubles per instance: for short
 * horizons, and the reference's independent cross-check of the Riccati path (test/least_squares.jl:38).
 *   A[n,n,batch] B[n,m,batch] Q[n,n,batch] R[m,m,batch] Qf[n,n,batch] x0[n,batch] (host or device)
 *   -> Z[NN,batch] (Primals order), info[batch] | NULL (potrf info of the condensed Hessian).               */
int32_t lqrb_lsq_solve_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                           const double *A, const double *B, const double *Q, const double *R,
                           const double *Qf, const double *x0, double *Z, int32_t *info);

/* ---------------------------------------------------------------- DARE ---------------------- */
/* The discrete algebraic Riccati equation of the infinite-horizon LQR,  P = Q + A'PA - A'PB (R + B'PB)^-1 B'PA,  its
 * stabilising solution P and stationary gain K = (R + B'PB)^-1 B'PA (u = -K x, the sign of lqrb_riccati_f64), by the
 * structured doubling algorithm: quadratic convergence, 7-10 doubling steps on the benchmark draws (DESIGN §4.11).
 * P is the terminal cost Qf that makes a finite-horizon lqrb_riccati_f64 consistent with its stage cost.
 *   A[n,n,batch] B[n,m,batch] Q[n,n,batch] R[m,m,batch] (instance-major, column-major; only the upper triangles of Q
 *   and R are read), 1 <= n <= 64, 1 <= m <= n.
 *   -> P[n,n,batch] (both triangles) | NULL, K[m,n,batch] | NULL (not both NULL), iters[batch] | NULL (doubling steps
 *   taken), info[batch] | NULL.
 *   Stopping rule: ||dH||_F <= 2^-52 ||H||_F for the increment dH of the last step, at most 64 steps.
 *   info: 0 ok; 1 not converged within 64 steps (no stabilising solution, or a NaN / Inf input); 1000 + j R not positive
 *   definite at pivot j; 2000 + j a zero pivot at column j of W = I + G_k H_k; 3000 + j R + B'PB not positive definite
 *   at pivot j (formed when K is requested).  A failed instance's P and K are NaN; the other instances are not affected.
 *   Error codes: -2 n, -3 m, -4 batch, -5..-8 A, B, Q, R NULL, -9 P and K both NULL.
 * Host or device pointers, with the staged / device-resident rule of every entry point.                         */
int32_t lqrb_dare_f64(lqrb_handle_t handle, int32_t n, int32_t m, int64_t batch, const double *A, const double *B,
                      const double *Q, const double *R, double *P, double *K, int32_t *iters, int32_t *info);

/* Gradient of a scalar loss l(P, K) through lqrb_dare_f64: given A, B, R, that call's P and the cotangents dP = dl/dP
 * [n,n,batch], dK = dl/dK [m,n,batch] (either may be NULL, not both), writes dl/dA, dl/dB, dl/dQ, dl/dR in the shapes
 * of the inputs (any may be NULL, not all).  K and R + B'PB are rebuilt from P (its upper triangle is read).  One
 * Stein equation Y = Acl Y Acl' + S (Acl = A - BK) is solved by Smith doubling with the stopping rule of
 * lqrb_dare_f64, the gradients are products of Y, P, K (DESIGN §4.11).  gQ and gR are returned as the symmetric
 * matrices (Q and R enter through their upper triangles); a finite-difference check perturbs (i,j) and (j,i) together.
 *   info: 0 ok; 1 the Stein doubling did not converge (rho(Acl) >= 1: P is not stabilising); 3000 + j R + B'PB not
 *   positive definite at pivot j.  A failed instance's gradients are NaN.
 *   Error codes: -2 n, -3 m, -4 batch, -5..-8 A, B, R, P NULL, -9 dP and dK both NULL, -11 every output NULL.
 * Host or device pointers, with the staged / device-resident rule of every entry point.                         */
int32_t lqrb_dare_grad_f64(lqrb_handle_t handle, int32_t n, int32_t m, int64_t batch, const double *A,
                           const double *B, const double *R, const double *P, const double *dP, const double *dK,
                           double *gA, double *gB, double *gQ, double *gR, int32_t *info);

/* ---------------------------------------------------------------- box-constrained MPC (ADMM) - */
/* Box-constrained LTI MPC by ADMM on a cached infinite-horizon Riccati factor (the algorithm of TinyMPC, Nguyen et al.,
 * ICRA 2024; DESIGN §4.12).  Per instance, with x_1 = x0:
 *     min  sum_{k=1}^{N-1} 1/2 (x_k - xref_k)'Q(x_k - xref_k) + 1/2 (u_k - uref_k)'R(u_k - uref_k)
 *          + 1/2 (x_N - xref_N)'Qf(x_N - xref_N)
 *     s.t. x_{k+1} = A x_k + B u_k,  umin_k <= u_k <= umax_k (k = 1..N-1),  xmin_k <= x_k <= xmax_k (k = 2..N)
 * THE TERMINAL COST DEPENDS ON rho: Qf = Pt - rho I with Pt = DARE(A, B, Q + rho I, R + rho I) (Pt >= Q + rho I, so
 * Qf >= Q).  With that Qf the finite-horizon gains of the rho-augmented problem equal the stationary K at every knot,
 * so one cached factor serves every iteration and every horizon.
 * Iteration (scaled duals; z, y, v, g start at 0 on a cold start):
 *   1. qt_k = -Q xref_k - rho (v_k - g_k), rt_k = -R uref_k - rho (z_k - y_k), p_N = -Qf xref_N - rho (v_N - g_N);
 *   2. for k = N-1..1: d_k = C1 (B'p_{k+1} + rt_k), p_k = qt_k + C2 p_{k+1} - K'rt_k   (C1 = (R + rho I + B'Pt B)^-1,
 *      C2 = (A - BK)');
 *   3. u_k = -K x_k - d_k, x_{k+1} = A x_k + B u_k;
 *   4. z = clamp(u + y, umin, umax), v = clamp(x + g, xmin, xmax);   5. y += u - z, g += x - v;
 *   6. r_pri = max(|u - z|_inf, |x - v|_inf), r_dual = rho max(|z - z_prev|_inf, |v - v_prev|_inf);
 *   7. stop when r_pri <= eps_pri and r_dual <= eps_dual, or after max_iter iterations.
 * The returned trajectory is the last primal iterate (x, u): dynamically exact, within r_pri of the bounds.
 *
 * lqrb_admm_cache_f64: the cache of (A, B, Q, R, rho).
 *   A[n,n,batch] B[n,m,batch] Q[n,n,batch] R[m,m,batch] (only the upper triangles of Q and R are read), rho > 0 finite
 *   (one value for the batch), 1 <= n <= 32, 1 <= m <= n.
 *   -> cache[L,batch], L = 4n^2 + 2nm + 2m^2 + 1 doubles per instance, column-major blocks in this order:
 *      A (n x n) | B (n x m) | Q (n x n) | R (m x m) | Qf (n x n) | K (m x n) | C1 (m x m) | C2 (n x n) | rho,
 *      Q and R symmetric (from their upper triangles), K the DARE gain of the rho-augmented costs (u = -K x);
 *      info[batch] | NULL: the codes of lqrb_dare_f64 for (A, B, Q + rho I, R + rho I): 0, 1, 1000 + j, 2000 + j,
 *      3000 + j.  A failed instance's record is NaN (a solve on it reports info 2); the others are not affected.
 *   Error codes: -2 n, -3 m, -4 batch, -5 rho, -6..-9 A, B, Q, R NULL, -10 cache NULL.
 *
 * lqrb_admm_solve_f64: the ADMM iterations, each instance to its own stopping point.
 *   flags: 0 or LQRB_FLAG_WARM_START (start from `state` instead of zeros).
 *   opts: max_iter >= 1, eps_pri >= 0, eps_dual >= 0 (eps = 0: exactly max_iter iterations).
 *   cache[L,batch] from lqrb_admm_cache_f64 with the same n, m; x0[n,batch];
 *   xref[n,N,batch] | NULL (0), uref[m,N-1,batch] | NULL (0), umin, umax[m,N-1,batch] | NULL (-inf, +inf),
 *   xmin, xmax[n,N-1,batch] | NULL (-inf, +inf; knots 2..N).  Infinite bound entries are legal; a NaN anywhere is not.
 *   state[2(N-1)(m+n),batch] | NULL, in/out, per instance [z (m,N-1); y (m,N-1); v (n,N-1); g (n,N-1)] (v, g at knots
 *   2..N): read only under LQRB_FLAG_WARM_START, written whenever given (the receding-horizon loop passes it back).
 *   -> Z[N*n+(N-1)*m,batch] (Primals order, as lqrb_riccati_f64), iters[batch] | NULL (iterations run),
 *      res[2,batch] | NULL (r_pri, r_dual of the last iteration), info[batch] | NULL:
 *      0 converged; 1 max_iter reached (the last iterate is written); 2 a NaN in the instance's inputs (cache record,
 *      x0, references, bounds, warm-start state) or in an iterate; 3 an empty box (min > max) somewhere.  Under 2 and
 *      3 the instance's Z, state and res are NaN.  The other instances of the batch are not affected.
 *   Each instance's working set (2n^2 + 2nm + m^2 + (N-1)(6n + 6m) doubles) stays in shared memory for all
 *   iterations; a shape where it exceeds 227 KB is rejected with -4 (N too long for this n, m).
 *   Error codes: -2 n, -3 m, -4 N < 2 or the working set above, -5 batch, -6 flags (or WARM_START without state),
 *   -7 opts NULL or out of range, -8 cache NULL, -9 x0 NULL, -17 Z NULL.
 * Both: host or device pointers, with the staged / device-resident rule of every entry point.  Not differentiable. */
#define LQRB_FLAG_WARM_START 8
typedef struct {
    int32_t max_iter;
    double eps_pri, eps_dual;
} lqrb_admm_options_t;
int32_t lqrb_admm_cache_f64(lqrb_handle_t handle, int32_t n, int32_t m, int64_t batch, double rho, const double *A,
                            const double *B, const double *Q, const double *R, double *cache, int32_t *info);
int32_t lqrb_admm_solve_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch, int32_t flags,
                            const lqrb_admm_options_t *opts, const double *cache, const double *x0, const double *xref,
                            const double *uref, const double *umin, const double *umax, const double *xmin,
                            const double *xmax, double *state, double *Z, int32_t *iters, double *res, int32_t *info);

/* ---------------------------------------------------------------- BlockCholesky ------------- */
/* Replaces cholesky!(chol, A, B[, C]) : src/block_cholesky.jl:55-91.  Instance-major:
 *   A[n,n,batch] B[m,m,batch] C[m,n,batch] (C NULL unless DENSE) -> M[(n+m),(n+m),batch]
 * M holds the upper factor (strict lower untouched = zero here), or for DIAG the reciprocals on
 * its diagonal, exactly as the reference's `chol.M`.                                            */
int32_t lqrb_block_cholesky_f64(lqrb_handle_t handle, int32_t n, int32_t m, int64_t batch,
                                int32_t hess_mode, const double *A, const double *B,
                                const double *C, double *M, int32_t *info);
/* Replaces ldiv!(chol, b) and chol \ b : src/block_cholesky.jl:93-101.
 *   M as produced above, b[(n+m), nrhs, batch] overwritten with the solution.                    */
int32_t lqrb_block_ldiv_f64(lqrb_handle_t handle, int32_t n, int32_t m, int64_t batch,
                            int32_t hess_mode, const double *M, int32_t nrhs, double *b);

/* ---------------------------------------------------------------- constrained KKT solve ------ */
/* Replaces _solve!(::CholeskySolver) : src/cholesky_solver.jl:166-182, i.e.
 *   calculate_shur_factors! (src/jacobian_blocks.jl:220-286), cholesky!(chol, shur)
 *   (src/cholesky_solve.jl:28-67), forward/backward_substitution! (:93-143) and
 *   calculate_primals! (src/cholesky_solver.jl:185-236); with LQRB_FLAG_SOC it is
 *   second_order_correction!'s chain (:254-273).
 *
 * Instance-major arrays (host or device):
 *   Q[n,n,N,batch] R[m,m,N-1,batch] Hux[m,n,N-1,batch]|NULL q[n,N,batch] r[m,N-1,batch]
 *   A[n,n,N-1,batch] B[n,m,N-1,batch] d[n,N-1,batch]           (D1_k = [A_k B_k], y_k = [c_k; d_k])
 *   D2: NULL => D2_k = [-I 0] (test/cartpole.jl:34-42); else concat over k=2..N of [n,w_k] blocks
 *   p[N] (host int32): stage-constraint rows per knot; C: concat over k of C_k[p_k,w_k]; c likewise
 * Outputs (instance-major): dz[NN,batch], mult[P,batch], res[NN,batch]|NULL, info[batch]|NULL.  */
int32_t lqrb_kkt_solve_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                           const int32_t *p, int32_t hess_mode, int32_t flags, const double *Q,
                           const double *R, const double *Hux, const double *q, const double *r,
                           const double *A, const double *B, const double *d, const double *D2,
                           const double *C, const double *c, double *dz, double *mult, double *res,
                           int32_t *info);

/* Gradient of a scalar loss l(dz, mult) through lqrb_kkt_solve_f64: given the inputs, that call's outputs dz, mult and
 * the cotangents dz_bar = dl/d dz, mult_bar = dl/d mult (same shapes), writes dl/d of every input.  The same KKT
 * matrices are solved once more with g := dz_bar and [c; d] := mult_bar, by the same kernels as the forward solve; one
 * kernel then forms every gradient as outer products of the two solutions (DESIGN §4.9).
 *   inputs as in lqrb_kkt_solve_f64 (q, r, d, c are not needed); flags must be 0 (-8: LQRB_FLAG_SOC has no gradient);
 *   dz_bar[NN,batch] | NULL, mult_bar[P,batch] | NULL (zero), not both NULL.
 *   outputs gQ, gR, gHux, gq, gr, gA, gB, gd, gD2, gC, gc: the shape of their input (gD2, gC, gc: the same ragged
 *   concatenations); any may be NULL, not all.  gHux needs LQRB_HESS_DENSE, gD2 an explicit D2, gC / gc sum(p) > 0.
 *   The kernels read only the upper triangle of Q, R (LQRB_HESS_DIAG: the diagonal): their gradients are returned as
 *   the symmetric matrices (1/2)(x^ x' + x x^'), under LQRB_HESS_DIAG only their diagonal (the rest is 0); a
 *   finite-difference check perturbs (i,j) and (j,i) together.  gHux = u^ x' + u x^' (the solve reads Hux once).
 *   info[batch] | NULL: the potrf info of the adjoint solve (the same matrices as the forward solve).  The gradients of
 *   an instance with info != 0 carry no meaning.  The call leaves the kept factorisation (lqrb_kkt_factor_f64) and the
 *   record of lqrb_kkt_last_condition as they were.
 * Host or device pointers, with the staged / device-resident rule of every entry point.                          */
int32_t lqrb_kkt_grad_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                          const int32_t *p, int32_t hess_mode, int32_t flags,
                          const double *Q, const double *R, const double *Hux, const double *A, const double *B,
                          const double *D2, const double *C,
                          const double *dz, const double *mult, const double *dz_bar, const double *mult_bar,
                          double *gQ, double *gR, double *gHux, double *gq, double *gr, double *gA, double *gB,
                          double *gd, double *gD2, double *gC, double *gc, int32_t *info);

/* Device-resident split (DEVICE pointers; `data` has lqrb_kkt_data_rows() x ldb doubles). */
int32_t lqrb_kkt_pack_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                          const int32_t *p, int32_t hess_mode, const double *Q, const double *R,
                          const double *Hux, const double *q, const double *r, const double *A,
                          const double *B, const double *d, const double *D2, const double *C,
                          const double *c, double *data);
int32_t lqrb_kkt_solve_packed_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N,
                                  int64_t batch, const int32_t *p, int32_t hess_mode,
                                  int32_t explicit_d2, int32_t flags, const double *data,
                                  double *dz, double *mult, double *res, int32_t *info);

/* tile width T (1 or 32) of `data`, dz, mult, res for this shape on this handle (> 0; < 0 = bad argument). */
int32_t lqrb_kkt_tile_width(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, const int32_t *p,
                            int32_t hess_mode, int32_t explicit_d2);
/* packed outputs of lqrb_kkt_solve_packed_f64 -> instance-major dz[NN,batch], mult[P,batch],
 * res[NN,batch] | NULL; device pointers. */
int32_t lqrb_kkt_unpack_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                            const int32_t *p, int32_t hess_mode, int32_t explicit_d2,
                            const double *dz_packed, const double *mult_packed,
                            const double *res_packed, double *dz, double *mult, double *res);

/* ---- the five steps of _solve! one by one, with the factor kept for further right-hand sides (SURVEY §8f-3) ----
 * The reference keeps `shur_blocks` / `chol_blocks` (Vector{BlockUpperTriangular3}, src/jacobian_blocks.jl:95-169) in
 * the solver and re-uses them (test/cholesky_solve.jl:14-35).  Here the HANDLE keeps one factorisation on the device:
 *
 * lqrb_kkt_factor_f64  = calculate_shur_factors! (matrix part, src/jacobian_blocks.jl:220-286) + cholesky!(U, F)
 *   (src/cholesky_solve.jl:28-67): S = D H^-1 D' factored block row by block row as U'U; LQRB_FLAG_SOC: S = D D'.
 *   Arrays as in lqrb_kkt_solve_f64 (instance-major, host or device).  info[batch] | NULL.
 * lqrb_kkt_solve_factored_f64 = the right-hand-side part of calculate_shur_factors! (h = D H^-1 g - d) +
 *   forward_substitution! (:93-117) + backward_substitution! (:119-143) + calculate_primals!
 *   (src/cholesky_solver.jl:185-236) with the kept U — no O(n^3) work.  q, r, d, c: the new right-hand side
 *   (the second-order correction's constraint values, a refinement residual, ...); shape, batch and flags must
 *   be those of the kept factorisation (else -1).  Runs on the general (any size / stage pattern) kernel.     */
int32_t lqrb_kkt_factor_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                            const int32_t *p, int32_t hess_mode, int32_t flags, const double *Q,
                            const double *R, const double *Hux, const double *A, const double *B,
                            const double *D2, const double *C, int32_t *info);
int32_t lqrb_kkt_solve_factored_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                                    const int32_t *p, int32_t hess_mode, int32_t explicit_d2, int32_t flags,
                                    const double *q, const double *r, const double *d, const double *c,
                                    double *dz, double *mult, double *res, int32_t *info);
/* Replaces get_shur_factors (src/cholesky_solver.jl:333-341) and get_cholesky (:352-359), i.e. copy_shur_factors!
 * (src/jacobian_blocks.jl:173-211) on the device's block rows: dense column-major S[P,P,batch] (symmetric, both
 * triangles filled), h[P,batch] = D H^-1 g - d, U[P,P,batch] (upper triangular, U'U = S), in the multiplier order
 * [mu_1; lam_1; ...; mu_N].  Any of S, h, U may be NULL.  Debug / parity path: P^2 doubles per instance.      */
int32_t lqrb_kkt_get_shur_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                              const int32_t *p, int32_t hess_mode, int32_t flags, const double *Q,
                              const double *R, const double *Hux, const double *q, const double *r,
                              const double *A, const double *B, const double *d, const double *D2,
                              const double *C, const double *c, double *S, double *h, double *U,
                              int32_t *info);

/* Diagnostic of the last lqrb_kkt_solve_f64 / lqrb_kkt_solve_packed_f64 call on this handle that used one of the
 * tuned large-size kernels (which carry explicit block inverses): log2 of the worst pivot ratio met in any Schur block
 * of each instance of the call, in instance order however the call was chunked (-1 = not tracked), and how many of
 * its instances were found ill-conditioned (>= 2^kkt_cond_bits, option, default 6) and solved again by the
 * Cholesky-based general kernel, the reference's own operation order (src/cholesky_solve.jl:47-67).  Either output
 * may be NULL.                                                                                                   */
int32_t lqrb_kkt_last_condition(lqrb_handle_t handle, int64_t count, int32_t *log2_pivot_ratio,
                                int64_t *resolved);

/* Replaces residual(solver; recalculate=true) : src/cholesky_solver.jl:238-252 — calc_residual! (:201-236)
 * with the KEPT multipliers of an earlier solve and freshly evaluated Jacobians / gradients (what step!
 * reports as feas_d, :126-134):
 *   res_k = D1_k' lam_k + C_k' mu_k + D2_k' lam_{k-1} + g_k,   norms[i] = || (||res_k||)_k || = ||res||_2.
 * Arrays as in lqrb_kkt_solve_f64 (instance-major, host or device); mult[P,batch] in the reference's
 * multiplier order.  LQRB_FLAG_SOC drops g (Ginv = false, :229-231; q, r may then be NULL).
 * res[NN,batch] | NULL, norms[batch] | NULL (not both NULL).                                            */
int32_t lqrb_kkt_residual_f64(lqrb_handle_t handle, int32_t n, int32_t m, int32_t N, int64_t batch,
                              const int32_t *p, int32_t flags, const double *q, const double *r,
                              const double *A, const double *B, const double *D2, const double *C,
                              const double *mult, double *res, double *norms);

/* ---------------------------------------------------------------- Dubins SQP ---------------- */
/* Fixed-count SQP outer loop (solve!/step!, src/cholesky_solver.jl:109-153, globalised as the
 * in-repo spec src/sqp.jl:72-94: L1 merit, eta=1e-4, rho=0.5, <=10 trials, SOC tried at alpha=1)
 * on the Dubins car turn problem, everything on device: RK3 linearisation, cost expansion
 * (dt-scaled, test/sparse_solver.jl:67-72), one constrained KKT solve per iteration.
 *   x0[3,batch] xf[3,batch] (host or device), Z[NN,batch] in/out (initial guess -> solution),
 *   feas_p[batch], feas_d[batch] out, iters_done[batch] out, kkt_solves (host) total KKT solves. */
typedef struct {
    int32_t N, iters;
    double dt, q_diag, r_diag, qf_diag;
    double eps_p, eps_d; /* convergence: 1e-5 each, src/cholesky_solver.jl:131-132 */
    int32_t line_search; /* 0 = full steps, 1 = L1 merit back-tracking + SOC */
} lqrb_sqp_options_t;
int32_t lqrb_sqp_dubins_f64(lqrb_handle_t handle, int64_t batch, const lqrb_sqp_options_t *opts,
                            const double *x0, const double *xf, double *Z, double *feas_p,
                            double *feas_d, int32_t *iters_done, int64_t *kkt_solves);

#ifdef __cplusplus
}
#endif
#endif /* LQRB200_H */
