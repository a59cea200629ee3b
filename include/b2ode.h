/*
 * b2ode.h -- C ABI of libb2ode.so: the sm_100a kernels behind tfdiffeq's odeint() Runge-Kutta hot path.
 *
 * The reference (titu1994/tfdiffeq) is pure Python on TensorFlow-Eager and has no FFI layer; its seam
 * is the solver protocol `SOLVERS[method](func, y0, rtol=, atol=, **options).integrate(t)`
 * (tfdiffeq/odeint.py:77-78).  This library sits directly below that seam: every entry point replaces
 * the per-step tensor arithmetic of one group of reference functions (cited per function, paths
 * relative to the reference root).  The user's func(t, y) stays a host-side callable (a PyTorch
 * nn.Module); its outputs land in device tensors whose pointers are handed to these calls.
 *
 * Conventions
 *  - plain C: pointers, sizes, ints.  No torch / C++ types cross this boundary.
 *  - every function returns 0 on success, a negative B2ODE_E* code for an invalid argument, or a
 *    positive cudaError_t; b2ode_last_error() returns a thread-local description.  Nothing throws.
 *  - all device pointers are CALLER-OWNED (allocated by the host framework's allocator) and must stay
 *    valid until the stream reaches the call.  The library never allocates device memory and never
 *    synchronises the host, with the single exception of b2ode_poll_sync().
 *  - "segments": a state that is a tuple of tensors (tfdiffeq/misc.py:292-305) is a list of up to
 *    B2ODE_MAXSEG flat arrays; the error norm is computed per segment (tfdiffeq/misc.py:250-264).
 *  - dtype: 0 = float32, 1 = float64.  Time (t0, t1, dt, output times) is always float64
 *    (tfdiffeq/solvers.py:30); stage arithmetic is in the state dtype (tfdiffeq/rk_common.py:45-46).
 *  - vector (16-byte) loads are used for a segment when every pointer of that segment is 16-byte
 *    aligned; otherwise that segment takes the scalar path.  No alignment is *required*.
 */
#ifndef B2ODE_H_
#define B2ODE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2ODE_ABI_VERSION 1
#define B2ODE_MAXSEG 12     /* tuple components per state (odeint_adjoint of an n-tuple needs 2n + 2) */
#define B2ODE_MAXK 14       /* k-buffers per step (dopri8: 14)                 */
#define B2ODE_MAXPEERS 8    /* ranks in a shared-step group (one NVSwitch box) */

#define B2ODE_F32 0
#define B2ODE_F64 1

/* error codes (negative) */
#define B2ODE_EINVAL (-1)   /* bad argument                               */
#define B2ODE_ESTATE (-2)   /* call sequence violated (e.g. not bound)    */
#define B2ODE_ENOMEM (-3)   /* caller-provided workspace too small        */

/* status bits of b2ode_state.status; the host driver re-raises them with the reference's messages */
#define B2ODE_ST_UNDERFLOW 1u   /* `assert t0 + dt > t0`          tfdiffeq/dopri5.py:98  */
#define B2ODE_ST_NONFINITE 2u   /* `assert _is_finite(abs(y0))`   tfdiffeq/dopri5.py:100 */
#define B2ODE_ST_MAXSTEPS 4u    /* `assert n_steps < max_num_steps` tfdiffeq/dopri5.py:85 */

/* controller flavours */
#define B2ODE_CTRL_REFERENCE 0  /* tfdiffeq/misc.py:267-287 (sqrt, float32-rounded exponent, per-segment msr, max) */
#define B2ODE_CTRL_TSIT5 1      /* tfdiffeq/tsit5.py:53-62,134-138 (pooled msr, no sqrt, exact exponent)           */

/* Mirror of the device-resident solver state (tfdiffeq/rk_common.py:8-19 `_RungeKuttaState`, minus the
 * tensors).  b2ode_poll_async() copies it to pinned host memory. 256 bytes. */
typedef struct b2ode_state {
    double t0;              /* start of the last accepted step                           */
    double t1;              /* current time = end of the last accepted step              */
    double dt;              /* size of the NEXT attempt                                  */
    double dt_last;         /* size of the attempt just finalized                        */
    double msr_max;         /* max over segments of the last mean-square error ratio     */
    double h0;              /* initial-step probe size (misc.py:232-236)                 */
    double reserved_d[2];
    uint64_t n_acc;         /* accepted steps                                            */
    uint64_t n_rej;         /* rejected attempts                                         */
    uint64_t attempt;       /* attempts finalized so far (sequence number)               */
    int64_t n_steps_adv;    /* attempts since the last emitted output (max_num_steps)    */
    int32_t accept;         /* 1 iff the attempt just finalized was accepted             */
    int32_t done;           /* all output points emitted, or status != 0                 */
    uint32_t status;        /* B2ODE_ST_* bits                                           */
    int32_t cursor;         /* next output index to emit                                 */
    int32_t emit_j0;        /* outputs [emit_j0, emit_j1) fall in the step just accepted */
    int32_t emit_j1;
    uint32_t ticket;        /* last-block-done counter of the reduction kernels          */
    uint32_t reserved_u;
    uint64_t xseq;          /* cross-GPU exchange sequence number                        */
    uint64_t klast[B2ODE_MAXSEG]; /* device address of k_{s-1} of the attempt just finalized, per segment:
                                     read by the next attempt's stage 0 when it commits an accepted step  */
    double reserved_t[3];
} b2ode_state;

/* Description of an adaptive Runge-Kutta solve.  Restates `_ButcherTableau` (tfdiffeq/rk_common.py:5) plus
 * the solver options of tfdiffeq/dopri5.py:50-68 (same in dopri8.py, bosh3.py, tsit5.py, adaptive_huen.py). */
typedef struct b2ode_adaptive_desc {
    int32_t dtype;                      /* B2ODE_F32 / B2ODE_F64                                   */
    int32_t nseg;                       /* tuple components                                        */
    int64_t seg_len[B2ODE_MAXSEG];      /* elements per component                                  */
    int32_t n_k;                        /* number of k buffers s (dopri5: 7); func evals/attempt = s-1 */
    int32_t fsal;                       /* rk_common.py:54 shortcut holds (y1 = last stage input)  */
    double alpha[B2ODE_MAXK];           /* s-1 entries                                             */
    double beta[B2ODE_MAXK][B2ODE_MAXK];/* row i (0-based, i < s-1) has i+1 entries                */
    double c_sol[B2ODE_MAXK];           /* s entries (used only when !fsal)                        */
    double c_error[B2ODE_MAXK];         /* s entries                                               */
    double c_mid[B2ODE_MAXK];           /* s entries; ignored when dense_kind != 0                 */
    int32_t dense_kind;                 /* 0: quartic fit through y_mid (interp.py:6-67); 1: tsit5.py:33-50 */
    int32_t controller;                 /* B2ODE_CTRL_*                                            */
    double rtol[B2ODE_MAXSEG];
    double atol[B2ODE_MAXSEG];
    double safety, ifactor, dfactor;    /* already rounded through float32 as the reference does   */
    double exponent;                    /* 1/order as the reference rounds it (misc.py:281-282)    */
    int64_t max_num_steps;              /* per advance(), tfdiffeq/dopri5.py:83-88                 */
    int32_t init_order;                 /* order passed to _select_initial_step (dopri5.py:74)     */
    int32_t sm_count;                   /* SMs of the device (grid sizing); 0 -> 148               */
} b2ode_adaptive_desc;

/* Caller-owned device buffers of one solve. */
typedef struct b2ode_adaptive_buffers {
    void *state;                        /* sizeof(b2ode_state) bytes, zeroed by b2ode_adaptive_init  */
    void *workspace;                    /* b2ode_workspace_bytes() bytes (reduction partials)        */
    size_t workspace_bytes;
    void *y0[B2ODE_MAXSEG];             /* current accepted state per segment (y0 of the step)       */
    void *f0[B2ODE_MAXSEG];             /* derivative at y0 (k_1)                                    */
    void *ystage[B2ODE_MAXSEG];         /* stage input handed to func; holds y1 after the last stage */
    void *tstage;                       /* n_k state-dtype scalars: time argument of each func call  */
    const double *t_out;                /* n_out output times (float64, increasing)                  */
    int32_t n_out;
    void *out[B2ODE_MAXSEG];            /* per segment: (n_out, seg_len) row-major solution slab     */
} b2ode_adaptive_buffers;

typedef struct b2ode_solver b2ode_solver;   /* opaque host-side handle */

int b2ode_version(void);
const char *b2ode_last_error(void);
size_t b2ode_state_bytes(void);
size_t b2ode_workspace_bytes(const b2ode_adaptive_desc *desc);

/* ---- adaptive Runge-Kutta (tfdiffeq/solvers.py:27-35, dopri5.py:70-121 and siblings) ---------------- */

int b2ode_adaptive_create(b2ode_solver **out, const b2ode_adaptive_desc *desc);
void b2ode_adaptive_destroy(b2ode_solver *s);
int b2ode_adaptive_bind(b2ode_solver *s, const b2ode_adaptive_buffers *buf, void *cuda_stream);
/* Redirect subsequent launches to another stream (e.g. the stream a CUDA graph of one attempt is captured on:
 * no kernel argument changes between attempts, so an attempt -- func included -- can be captured once and replayed). */
int b2ode_set_stream(b2ode_solver *s, void *cuda_stream);

/* Replaces Dopri5Solver.before_integrate's state construction (dopri5.py:78): zero the state, set
 * t0 = t1 = t_start (= t_out[0]), copy y0 into out[.][0], write the stage-time scalars.  If first_step is not NaN it
 * becomes dt (dopri5.py:76); otherwise call the two initial-step functions below.  y0/f0 must be filled. */
int b2ode_adaptive_init(b2ode_solver *s, double t_start, double first_step);

/* `_select_initial_step` (tfdiffeq/misc.py:183-247), first half: d0, d1, h0 and the Euler probe
 * ystage = y0 + h0*f0, tstage[0] = t0 + h0 (:216-237).  The host then evaluates f1 = func(tstage[0], ystage). */
int b2ode_initial_step_probe(b2ode_solver *s);
/* second half (:238-247): d2, h1, dt = min(100*h0, h1); then rewrites the stage times for the first attempt. */
int b2ode_initial_step_finish(b2ode_solver *s, const void *const *f1);

/* `_runge_kutta_step` stage combine (tfdiffeq/rk_common.py:49-51 via misc.py:118-121):
 *   ystage = y0 + sum_{j<=i} (dt*beta[i][j]) * k_j     for stage i = 0 .. n_k-2,
 * with dt read from the device state.  `k_new` = per-segment pointers of k_i, the output of the func call
 * that followed stage i-1 (ignored for i == 0, where k_0 = f0).  Stage 0 also commits the previous attempt
 * if it was accepted (y0 <- y1, f0 <- k_last: dopri5.py:113-114) -- the accept decision lives on the device.
 * i == n_k-1 is the extra solution combine with c_sol for non-FSAL tableaus (rk_common.py:54-56). */
int b2ode_rk_stage(b2ode_solver *s, int i, const void *const *k_new);

/* Everything after the last func call of an attempt (k_last = k_{s-1} = f1), fused:
 *   error combine (rk_common.py:60), `_compute_error_ratio` (misc.py:250-264), finite check
 *   (misc.py:147-150 / dopri5.py:100), accept decision (dopri5.py:108), `_optimal_step_size`
 *   (misc.py:267-287 or tsit5.py:53-62), state update (dopri5.py:113-120), max_num_steps / dt-underflow
 *   asserts (dopri5.py:85,98) as status bits, stage times of the next attempt;
 * then, iff accepted and output times fall inside the step, the dense output for ALL of them:
 *   `_interp_fit` + `_interp_evaluate` (interp.py:6-67, y_mid from dopri5.py:42) written straight into
 *   out[.][j] -- the interpolation coefficients never touch HBM. */
int b2ode_rk_finalize(b2ode_solver *s, const void *const *k_last);

/* Asynchronous copy of the device state to (pinned) host memory on the solver's stream. */
int b2ode_poll_async(b2ode_solver *s, b2ode_state *host_dst);
/* Blocking variant (the only call that synchronises): copy + cudaStreamSynchronize. */
int b2ode_poll_sync(b2ode_solver *s, b2ode_state *host_dst);

/* ---- shared-step groups across GPUs (new; the reference has no distributed code, SURVEY 8e) --------- */

/* Per-rank mailbox for the per-attempt exchange of {sum err^2, max|y0|, max|y1|, non-finite} per segment.
 * `mailboxes[r]` is the address, in THIS process, of rank r's mailbox (peer-mapped via CUDA IPC for r != rank;
 * every mailbox comes from b2ode_mailbox_create, which initialises it: sequence numbers zero, the persistent kernel's
 * receive area filled with a pattern no exchange validates).  After this call b2ode_rk_finalize and the
 * initial-step functions push their partials to every peer with st.global stores over NVLink and spin on the
 * arrival flags inside the same kernel (last block), so every rank takes the same accept / dt decision. */
size_t b2ode_mailbox_bytes(void);
int b2ode_comm_attach(b2ode_solver *s, int rank, int nranks, void *const *mailboxes);

/* Mailbox memory is the one thing the library allocates itself (cudaMalloc, so that a CUDA IPC handle can be
 * taken): create on each rank, exchange the 64-byte handles out of band, open the peers', attach. */
int b2ode_mailbox_create(void **dev_ptr, unsigned char handle_out[64]);
int b2ode_mailbox_open(const unsigned char handle[64], void **peer_ptr);
int b2ode_mailbox_close(void *peer_ptr);
int b2ode_mailbox_destroy(void *dev_ptr);
/* element count of every segment over the WHOLE group (the mean in misc.py:262 is over all ranks' elements) */
int b2ode_comm_set_global_len(b2ode_solver *s, const int64_t *global_len);
/* bit i set: tuple component i is REPLICATED -- every rank holds the whole component with bit-identical values (the
 * parameter / time adjoints of odeint_adjoint after their all-reduce, tfdiffeq/adjoint.py:97-107): its error-norm
 * partials are taken from the local rank alone and its global_len is the local length. */
int b2ode_comm_set_replicated(b2ode_solver *s, unsigned segment_mask);

/* ---- built-in right-hand sides: the whole adaptive solve in one persistent kernel (SURVEY 8f-2) ---------- */

#define B2ODE_RHS_LORENZ 0          /* (B,3): s(y-x), x(r-z)-y, xy-bz ; params {sigma, beta, rho}   examples/lorenz_attractor.py:20-37 */
#define B2ODE_RHS_LOTKA_VOLTERRA 1  /* (B,2): ax-bxz, -cz+dxz        ; params {a, b, c, d}          README.md:67-81                   */
#define B2ODE_RHS_CUBIC_MLP 2       /* (B,2): W2 tanh(W1 y^3 + b1) + b2; params {H <= 128, cube}; rhs_data = packed
                                       [W1 (2 x H) | b1 (H) | W2 (H x 2) | b2 (2)] in the state dtype   examples/ode_demo.py:115-129 */

#define B2ODE_RHS_KEPLER 3         /* (B, 4 m): m two-body orbits [x, y, vx, vy] per row; no params   tests/DETEST/detest.py:263-283 */
#define B2ODE_RHS_LINEAR 4         /* (B, D): y @ A (+ b), k[r, c] = sum_d y[r, d] A[d, c]; params {D, has_bias}, 1 <= D <= 128;
                                      data = A row-major D x D in the state dtype, then b (D values) iff has_bias.  Stage
                                      kernels only (b2ode_rhs_eval / b2ode_rk_stage_rhs, fp64 GEMM on DMMA): b2ode_fused_capacity
                                      returns 0 and the persistent / fixed-grid solves reject it   tests/problems.py:43-68 */

/* A built-in right-hand side as the kernels see it. */
typedef struct b2ode_rhs_desc {
    int32_t kind;                       /* B2ODE_RHS_*                                                   */
    int32_t n_params;
    double params[8];
    const void *data;                   /* staged weights (B2ODE_RHS_CUBIC_MLP, B2ODE_RHS_LINEAR), else NULL */
    double time_sign;                   /* -1: the reversed system of tfdiffeq/misc.py:318-321           */
} b2ode_rhs_desc;

/* k_out = f(t, y) for a built-in right-hand side: one elementwise pass over n state elements (rows of the
 * right-hand side's dimension); `t_scalar` is a device scalar of the state dtype.  Used for the first derivative
 * (dopri5.py:71), the initial-step probe (misc.py:237) and stage 0. */
int b2ode_rhs_eval(int dtype, const b2ode_rhs_desc *rhs, const void *t_scalar, const void *y, void *k_out, int64_t n,
                   int sm_count, void *cuda_stream);

/* b2ode_rk_stage for stage i in [1, n_k - 2] WITH the evaluation of a built-in right-hand side in the same launch
 * (tfdiffeq/rk_common.py:49-52: y_i = y0 + sum (dt beta_ij) k_j ; k_{i+1} = func(t_i, y_i)): registers k_i = k_new,
 * writes k_{i+1} to k_out (caller-owned, n elements) and, for the last stage, the stage input to ystage.  For batches
 * the persistent kernel below cannot keep co-resident.  Single-tensor states. */
int b2ode_rk_stage_rhs(b2ode_solver *s, int i, const void *const *k_new, const b2ode_rhs_desc *rhs, void *k_out);

/* Replaces the WHOLE of AdaptiveStepsizeODESolver.integrate (tfdiffeq/solvers.py:27-35) for a func the library
 * knows: every trajectory stays in one thread's registers (state + all k's) for the entire solve, one grid-wide
 * reduction per attempt keeps the reference's single shared step / global scalar tolerance; HBM traffic is the
 * (n_out, B, D) solution slab only.  Same arithmetic and operation order as the generic kernels.  `desc` must
 * describe ONE segment of B*D elements and a quartic dense output; `state` receives the final b2ode_state.
 * Returns B2ODE_ENOMEM when the batch exceeds what the device can keep co-resident (caller falls back to the
 * generic path).  time_sign = -1 integrates the reversed system of tfdiffeq/misc.py:318-321. */
size_t b2ode_fused_workspace_bytes(int64_t n_trajectories);
/* Largest per-device batch b2ode_fused_solve keeps co-resident for this tableau / dtype / right-hand side on the
 * current device (< 0: error).  Asked before launching so that all shards of a shared-step group take the same path. */
int64_t b2ode_fused_capacity(const b2ode_adaptive_desc *desc, int rhs_kind);
/* Everything b2ode_fused_solve needs besides the tableau / tolerances of `b2ode_adaptive_desc`. */
typedef struct b2ode_fused_desc {
    int32_t rhs_kind;                   /* B2ODE_RHS_*                                                            */
    int32_t n_rhs_params;
    double rhs_params[8];
    const void *rhs_data;               /* staged weights (B2ODE_RHS_CUBIC_MLP), else NULL                        */
    double time_sign;                   /* -1 integrates the reversed system of tfdiffeq/misc.py:318-321          */
    const void *y0;                     /* (B, D) initial state                                                   */
    void *out;                          /* (n_out, B, D) solution slab                                            */
    const double *t_out;                /* n_out output times (device memory, float64, increasing)                */
    int32_t n_out;
    double t_start, first_step;         /* first_step NaN -> _select_initial_step (misc.py:183-247)               */
    void *state;                        /* receives the final b2ode_state                                         */
    void *workspace;                    /* b2ode_fused_workspace_bytes(B) bytes, 16-byte aligned                  */
    size_t workspace_bytes;
    int32_t rank, nranks;               /* shared-step group (nranks <= 1: none)                                  */
    void *const *mailboxes;             /* nranks mailbox addresses in this process (b2ode_mailbox_create/open)   */
    int64_t n_traj_rank[B2ODE_MAXPEERS];/* trajectories of every rank: each rank derives every rank's kernel grid */
    void *cuda_stream;
    int32_t *host_mark;                 /* optional: page-locked, device-mapped int.  While the solve runs the kernel keeps
                                           it at the number of leading rows of `out` that are complete on the device, so
                                           the caller can stream the solution to the host behind the solve (the value only
                                           grows; rows [0, *host_mark) may be copied without further synchronisation)      */
} b2ode_fused_desc;
int b2ode_fused_solve(const b2ode_adaptive_desc *desc, const b2ode_fused_desc *fused);

/* Fixed-grid methods (0 euler, 1 midpoint, 2 heun, 3 rk4 3/8 rule) with a built-in right-hand side: replaces the
 * whole of FixedGridODESolver.integrate (tfdiffeq/solvers.py:82-104); no reductions, one launch.  The host
 * supplies, in the state dtype, the stage times of every grid cell ([n_steps][4]), dt per cell, and for the
 * outputs: j0[i]..j0[i+1] = outputs inside cell i, ends[i] = the cell ends exactly on its last output (then y1 is
 * stored, otherwise the linear interpolation of solvers.py:106-115 with s1[i] = t1 - t0 and s2[j] = t_j - t0). */
int b2ode_fused_fixed_solve(int dtype, int method, int rhs_kind, const double *rhs_params, int n_rhs_params,
                            const void *rhs_data, double time_sign, const void *y0, void *out, int64_t n_traj,
                            int n_steps, int n_out, const void *times, const void *dts, const int32_t *j0,
                            const unsigned char *ends, const void *s1, const void *s2, int sm_count, void *cuda_stream);

/* ---- multistep solvers (SURVEY 8f-4: tfdiffeq/fixed_adams.py, tfdiffeq/adams.py) ----------------------- */

/* out = base + scale * sum_{j < nterms} coef[j] * x[j]   over all segments; products and sums in the state dtype,
 * left to right (the order of `dt * _scaled_dot_product(scale, coeffs, f)`, misc.py:118-121, fixed_adams.py:196-204,
 * adams.py:144-157).  `base` may be NULL (no addend); scale == 1 skips the multiplication.  xs[j * nseg + s] is term
 * j of segment s; 1 <= nterms <= 16.  Covers the Adams-Bashforth predictor, the Adams-Moulton corrector update,
 * phi scaling and phi differences (adams.py:46, :73-75), and copies. */
int b2ode_lincomb(int dtype, int nseg, const int64_t *seg_len, void *const *out, const void *const *base, double scale,
                  int nterms, const void *const *xs, const double *coef, int sm_count, void *cuda_stream);

/* Per-segment reductions; out[2*s], out[2*s+1] (device doubles), deterministic (fixed combine order).
 *   B2ODE_RED_ABSMAX2       { max|a|, max|b| }, NaN-propagating                      misc.py:257 / adams.py:160-163
 *   B2ODE_RED_RATIO_SUMSQ   { sum ((p0[s] * a) / p1[s])^2, 0 }  (the caller divides by the element count)
 *                                                                                      misc.py:259-264 / adams.py:164-166
 *   B2ODE_RED_NOT_CONVERGED { number of elements with NOT |a-b| < p1[s] + p0[s]*max(|a|,|b|), 0 }   misc.py:129-134
 * `workspace`: b2ode_reduce_workspace_bytes(sm_count) bytes of device memory, zero-filled once by the caller and
 * reusable by later calls on the same stream. */
#define B2ODE_RED_ABSMAX2 0
#define B2ODE_RED_RATIO_SUMSQ 1
#define B2ODE_RED_NOT_CONVERGED 2
size_t b2ode_reduce_workspace_bytes(int sm_count);
int b2ode_reduce(int dtype, int mode, int nseg, const int64_t *seg_len, const void *const *a, const void *const *b,
                 const double *p0, const double *p1, double *out, void *workspace, size_t workspace_bytes, int sm_count,
                 void *cuda_stream);

/* ---- GEMM-backed func on tensor cores (SURVEY 8f-3) ---------------------------------------------------- */

/* One dense layer of an ODENet-style func (tfdiffeq/models/dense_odenet.py:85-92) on tcgen05 / TMEM:
 *     out[M, N] = act( A[M, K] . W[N, K]^T + bias[N] ),   fp32 storage, TF32 tensor-core math,
 * act: 0 none, 1 relu, 2 tanh, 3 softplus.  With nk == 0, A = x.  With nk > 0 the Runge-Kutta stage combine
 * (tfdiffeq/rk_common.py:51) is the A-operand producer: A = x + sum_j (dt * coef[j]) * k[j] with dt read from
 * `state` (x = y0 of the step); if `ystage` is non-null the stage input is also stored there (the last stage
 * needs it: it is y1).  W is torch's nn.Linear.weight layout.  N must be a multiple of 16. */
/* Registers k_i with the solver without launching the stage kernel (the combine then happens inside
 * b2ode_dense_layer as the A-operand producer). */
int b2ode_set_k(b2ode_solver *s, int i, const void *const *k_new);
int b2ode_dense_layer(const void *x, const void *const *k, const double *coef, int nk, const void *state, void *ystage,
                      const void *W, const void *bias, void *out, int64_t M, int K, int N, int act, void *cuda_stream);

/* Same layer with fp32-accurate products ("3xTF32"): W_hi = tf32(W), W_lo = tf32(W - W_hi), both [N, K]; the kernel
 * splits A = A_hi + A_lo the same way while staging it and accumulates A_lo.W_hi + A_hi.W_lo + A_hi.W_hi in the fp32
 * TMEM accumulator (the dropped A_lo.W_lo term is 2^-22 relative).  This is the default numeric mode of the
 * tensor-core func: it keeps the solution within north_star's 1e-3 fp32 bar of the reference's fp32 matmuls
 * (tfdiffeq/models/dense_odenet.py:85-92, conv_odenet.py:80-86 1x1 convolutions on NHWC = this GEMM with M = B*H*W). */
int b2ode_dense_layer_x3(const void *x, const void *const *k, const double *coef, int nk, const void *state, void *ystage,
                         const void *W_hi, const void *W_lo, const void *bias, void *out, int64_t M, int K, int N, int act,
                         void *cuda_stream);

/* The whole three-layer func (dense_odenet.py:85-92: fc1 -> act -> fc2 -> act -> fc3) in ONE launch: per 128-row
 * tile the hidden activations stay in shared memory / TMEM, so an evaluation moves only the input tile(s) and the
 * output tile through HBM.  out[M, D] = W3 . act(W2 . act(W1 . A + b1) + b2) + b3 with A as in b2ode_dense_layer
 * (x, or the stage combine of x and k[0..nk)).  W1 [H, D], W2 [H, H], W3 [D, H] in nn.Linear layout; D and H
 * multiples of 16 in [16, 256].
 *   b2ode_mlp3_packed_bytes : size of the packed weight image (-1 for unsupported widths)
 *   b2ode_mlp3_pack         : rounds the weights to TF32 and lays them out as the kernel's shared-memory image
 *                             (once per weight version; `packed` is caller-owned device memory, 16-byte aligned)
 *   b2ode_mlp3              : one evaluation */
int64_t b2ode_mlp3_packed_bytes(int D, int H);
int b2ode_mlp3_pack(const void *W1, const void *W2, const void *W3, int D, int H, void *packed, void *cuda_stream);
int b2ode_mlp3(const void *x, const void *const *k, const double *coef, int nk, const void *state, void *ystage,
               const void *packed, const void *b1, const void *b2, const void *b3, void *out, int64_t M, int D, int H,
               int act, void *cuda_stream);

/* ---- measurement hooks (bench.py) --------------------------------------------------------------------- */
unsigned long long b2ode_launch_count(void);            /* kernels launched by this library so far          */
/* families: 0 stage 0, 1 stage, 2 finalize, 3 dense output, 4 initial step, 5 fixed grid, 6 persistent solve,
 * 7 linear stage GEMM (B2ODE_RHS_LINEAR's stage / evaluation kernel) */
int b2ode_timing_enable(unsigned family_mask);          /* CUDA-event timing per kernel family; 0 = off     */
int b2ode_timing_read(int family, double *total_ms, int *count);

/* ---- fixed-grid steppers (tfdiffeq/solvers.py:82-115, fixed_grid.py, rk_common.py:73-81) ------------ */

#define B2ODE_OP_EULER 0        /* out = y + dt*a                                  fixed_grid.py:6-7 + solvers.py:95 */
#define B2ODE_OP_HALF_STEP 1    /* out = y + (a*dt)/2                              fixed_grid.py:17                  */
#define B2ODE_OP_HEUN_FINAL 2   /* out = y + (dt/2)*(a + b)                        fixed_grid.py:32                  */
#define B2ODE_OP_RK4_S2 3       /* out = y + (dt*a)/3                              rk_common.py:77                   */
#define B2ODE_OP_RK4_S3 4       /* out = y + dt*(a/(-3) + b)                       rk_common.py:78                   */
#define B2ODE_OP_RK4_S4 5       /* out = y + dt*((a - b) + c)                      rk_common.py:79-80                */
#define B2ODE_OP_RK4_FINAL 6    /* out = y + (((a + 3b) + 3c) + d)*(dt/8)          rk_common.py:81                   */
#define B2ODE_OP_LERP 7         /* out = y + ((a - y)/s1)*s2   (s1 = t1-t0, s2 = t-t0)  solvers.py:106-115            */

/* One elementwise op over all segments.  dt, s1, s2 are host scalars already rounded to the state dtype
 * (the fixed-grid loop has no device-side decisions).  Unused operands may be NULL. */
int b2ode_fixed_op(int dtype, int op, int nseg, const int64_t *seg_len, void *const *out, const void *const *y,
                   const void *const *a, const void *const *b, const void *const *c, const void *const *d,
                   double dt, double s1, double s2, int sm_count, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* B2ODE_H_ */
