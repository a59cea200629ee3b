#include <cstddef>
#include <vector>
// b2ode.cu -- sm_100a kernels + C ABI for the Runge-Kutta hot path of tfdiffeq's odeint().
//
// Reference citations are relative to the reference repository root (titu1994/tfdiffeq).
//
// Design (B200-first, see DESIGN.md):
//  * every kernel is a streaming, HBM-bound elementwise pass with 16-byte vector loads/stores and a
//    grid sized from the SM count; there is no GEMM-shaped work here, so no tensor cores.
//  * the step size, the accept/reject decision, the output cursor and all counters live in a 256-byte
//    device-resident state (b2ode_state); no kernel argument depends on them, so the host enqueues whole
//    attempts without reading anything back.
//  * stage arithmetic uses explicit round-to-nearest mul/add intrinsics (no FMA contraction) in the
//    reference's operation order, so single-kernel results are bit-identical to the oracle.
//  * the error-norm reduction is warp-shuffle tree -> per-block partial -> last block (ticket) in a fixed
//    order: deterministic.  The last block also runs the controller, so "finalize" is one launch; with a
//    shared-step group attached it additionally exchanges the partials with the peer GPUs over NVLink
//    (st/ld on peer-mapped mailboxes) inside the same kernel.
//  * the dense output is evaluated for every output time inside the accepted step from registers; the
//    quartic's coefficients are never written to HBM.

#include "b2ode_dev.cuh"
#include "b2ode_rhs.cuh"
#include <stdlib.h>

static thread_local char g_err[512] = "";

int b2_fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

// ------------------------------------------------------------------------------------------------
// K1: stage combine   ystage = y0 + sum_j (dt*beta_j) * k_j        (rk_common.py:51, misc.py:118-121)
// ------------------------------------------------------------------------------------------------
template <int NK>
struct StageParams {
    SegGeom g;
    const b2ode_state *st;
    const void *y0[B2ODE_MAXSEG];
    void *out[B2ODE_MAXSEG];
    const void *k[NK][B2ODE_MAXSEG];
    double coef[NK];
};

template <typename T, int NK>
__global__ void __launch_bounds__(kThreads, B2_MINB_STAGE) k_rk_stage(const __grid_constant__ StageParams<NK> p) {
    const int s = find_seg(p.g, blockIdx.x);
    const int bl = blockIdx.x - p.g.blk_begin[s], nb = p.g.blk_begin[s + 1] - p.g.blk_begin[s];
    const T dt = (T)p.st->dt;
    T c[NK];
#pragma unroll
    for (int j = 0; j < NK; ++j) c[j] = Ar<T>::mul(dt, (T)p.coef[j]);   // (scale * x), misc.py:121
    const T *y0 = (const T *)p.y0[s];
    T *out = (T *)p.out[s];
    const T *k[NK];
#pragma unroll
    for (int j = 0; j < NK; ++j) k[j] = (const T *)p.k[j][s];
    seg_for_each<T>(p.g.n[s], (p.g.vec_mask >> s) & 1u, bl, nb, [&](auto vt, long long i) {
        constexpr int V = decltype(vt)::value;
        Pack<T, V> yv = ld_pack<T, V>(y0, i);
        Pack<T, V> kv[NK];
#pragma unroll
        for (int j = 0; j < NK; ++j) kv[j] = ld_pack<T, V>(k[j], i);
        Pack<T, V> o;
#pragma unroll
        for (int e = 0; e < V; ++e) {
            T acc = Ar<T>::mul(c[0], kv[0].v[e]);
#pragma unroll
            for (int j = 1; j < NK; ++j) acc = Ar<T>::add(acc, Ar<T>::mul(c[j], kv[j].v[e]));   // add_n, left to right
            o.v[e] = Ar<T>::add(yv.v[e], acc);
        }
        st_pack<T, V>(out, i, o);
    });
}

// ------------------------------------------------------------------------------------------------
// K1 + func: stage combine with a BUILT-IN right-hand side evaluated in the same pass (SURVEY 8f-2 for batches / tableaus
// the one-launch persistent kernel cannot hold: BASELINE config 5's 131 072 Kepler orbits under dopri8, Lorenz batches
// beyond 71 040 trajectories).  One thread per ROW of RHS::D state elements:
//     y_i = y0 + sum_j (dt * beta_ij) k_j        (rk_common.py:51, same operation order as k_rk_stage)
//     k_{i+1} = f(t_i, y_i)                      (rk_common.py:52; f = the library's right-hand side, same arithmetic as rhs.py)
// so a stage is ONE launch that reads (NK + 1) N and writes N, instead of the stage kernel, a 2 N round trip of the stage
// input and the ~6 elementwise torch kernels of the module's forward.  NK = 0: plain evaluation k = f(t, y) of an
// existing buffer (first derivative, initial-step probe, stage 0 after the commit kernel).
// ------------------------------------------------------------------------------------------------
template <int NK>
struct StageRhsParams {
    const b2ode_state *st;
    const void *y0;
    const void *k[NK > 0 ? NK : 1];
    double coef[NK > 0 ? NK : 1];
    void *ystage;              // optional: also materialise the stage input (the last stage's input is y1)
    void *k_out;
    const void *t_scalar;      // device scalar of the state dtype: the stage time
    long long rows;
    double time_sign;
    double rhs[8];
    const void *rhs_data;
};

template <typename T, typename RHS, int NK>
__global__ void __launch_bounds__(kThreads) k_rk_stage_rhs(const __grid_constant__ StageRhsParams<NK> p) {
    constexpr int D = RHS::D;
    __shared__ T sw[RHS::kSmem];
    if (RHS::kSmem > 1) {
        const int nw = (int)p.rhs[0] * 5 + 2;
        for (int q = threadIdx.x; q < nw && q < RHS::kSmem; q += kThreads) sw[q] = ((const T *)p.rhs_data)[q];
        __syncthreads();
    }
    T c[NK > 0 ? NK : 1];
    if (NK > 0) {
        const T dt = (T)p.st->dt;
#pragma unroll
        for (int j = 0; j < NK; ++j) c[j] = Ar<T>::mul(dt, (T)p.coef[j]);
    }
    const T ti = *reinterpret_cast<const T *>(p.t_scalar);
    const T sgn = (T)p.time_sign;
    const T *y0 = (const T *)p.y0;
    T *ys = (T *)p.ystage, *ko = (T *)p.k_out;
    for (long long r = (long long)blockIdx.x * kThreads + threadIdx.x; r < p.rows; r += (long long)gridDim.x * kThreads) {
        T y[D], kv[NK > 0 ? NK : 1][D];
#pragma unroll
        for (int d = 0; d < D; ++d) y[d] = y0[r * D + d];
#pragma unroll
        for (int j = 0; j < NK; ++j)
#pragma unroll
            for (int d = 0; d < D; ++d) kv[j][d] = ((const T *)p.k[j])[r * D + d];
        if (NK > 0) {
#pragma unroll
            for (int d = 0; d < D; ++d) {
                T acc = Ar<T>::mul(c[0], kv[0][d]);
#pragma unroll
                for (int j = 1; j < NK; ++j) acc = Ar<T>::add(acc, Ar<T>::mul(c[j], kv[j][d]));   // add_n, left to right
                y[d] = Ar<T>::add(y[d], acc);
            }
            if (ys) {
#pragma unroll
                for (int d = 0; d < D; ++d) ys[r * D + d] = y[d];
            }
        }
        T dy[D];
        if (sgn < T(0)) {                                              // reverse-time wrapper of misc.py:318-321
            RHS::eval(p.rhs, sw, -ti, y, dy);
#pragma unroll
            for (int d = 0; d < D; ++d) dy[d] = -dy[d];
        } else {
            RHS::eval(p.rhs, sw, ti, y, dy);
        }
#pragma unroll
        for (int d = 0; d < D; ++d) ko[r * D + d] = dy[d];
    }
}

// Stage 0 with the deferred commit of the previous attempt (dopri5.py:113-114: y_next = y1 if accept ...).
// If the previous attempt was accepted: y0 <- ystage (= y1), f0 <- k_last, all in this pass; ystage is then
// overwritten in place with the first stage input.  One extra N write per array, only after an accept.
struct Stage0Params {
    SegGeom g;
    const b2ode_state *st;
    void *y0[B2ODE_MAXSEG];
    void *f0[B2ODE_MAXSEG];
    void *ystage[B2ODE_MAXSEG];
    double coef;
};

template <typename T>
__global__ void __launch_bounds__(kThreads) k_rk_stage0(const __grid_constant__ Stage0Params p) {
    const int s = find_seg(p.g, blockIdx.x);
    const int bl = blockIdx.x - p.g.blk_begin[s], nb = p.g.blk_begin[s + 1] - p.g.blk_begin[s];
    const T c = Ar<T>::mul((T)p.st->dt, (T)p.coef);
    // k_{s-1} of the previous attempt: its address was left in the state by that attempt's finalize kernel
    const T *kl = reinterpret_cast<const T *>(p.st->klast[s]);
    const bool commit = p.st->accept != 0 && kl != nullptr;
    T *y0 = (T *)p.y0[s], *f0 = (T *)p.f0[s], *ys = (T *)p.ystage[s];
    // kl is a func output whose address the host never sees here: check its 16-byte alignment on the device
    const bool vec_ok = ((p.g.vec_mask >> s) & 1u) && ((reinterpret_cast<unsigned long long>(kl) & 15ull) == 0);
    if (commit) {
        seg_for_each<T>(p.g.n[s], vec_ok, bl, nb, [&](auto vt, long long i) {
            constexpr int V = decltype(vt)::value;
            Pack<T, V> yv = ld_pack<T, V>(ys, i);
            Pack<T, V> fv = ld_pack<T, V>(kl, i);
            Pack<T, V> o;
#pragma unroll
            for (int e = 0; e < V; ++e) o.v[e] = Ar<T>::add(yv.v[e], Ar<T>::mul(c, fv.v[e]));
            st_pack<T, V>(y0, i, yv);
            st_pack<T, V>(f0, i, fv);
            st_pack<T, V>(ys, i, o);
        });
    } else {
        seg_for_each<T>(p.g.n[s], (p.g.vec_mask >> s) & 1u, bl, nb, [&](auto vt, long long i) {
            constexpr int V = decltype(vt)::value;
            Pack<T, V> yv = ld_pack<T, V>(y0, i);
            Pack<T, V> fv = ld_pack<T, V>(f0, i);
            Pack<T, V> o;
#pragma unroll
            for (int e = 0; e < V; ++e) o.v[e] = Ar<T>::add(yv.v[e], Ar<T>::mul(c, fv.v[e]));
            st_pack<T, V>(ys, i, o);
        });
    }
}

// ------------------------------------------------------------------------------------------------
// K2+K3: error combine + error-ratio reduction + finite check + controller + state update
// ------------------------------------------------------------------------------------------------
template <int NK>
struct FinalizeParams {
    SegGeom g;
    b2ode_state *st;
    Partial *part;
    const void *y0[B2ODE_MAXSEG];
    const void *y1[B2ODE_MAXSEG];
    const void *k[NK][B2ODE_MAXSEG];
    double coef[NK];
    const void *klast[B2ODE_MAXSEG];   // k_{s-1} (= f1) of this attempt, recorded in the state for the next stage 0
    CtrlParams c;
    CommParams comm;
};

// misc.py:250-264 + dopri5.py:106-120 + misc.py:267-287 (or tsit5.py:53-62,134-138).
// Called by ONE WARP (the first warp of the last block): every lane evaluates the (cheap) scalar controller
// redundantly, the output-cursor search and the stage-time writes are spread over the lanes, lane 0 stores.
// The state is read once, up front, so the serial tail of the finalize kernel is two dependent memory
// round trips (state, then t_out) instead of a dozen.
template <typename T>
__device__ void control_step(b2ode_state *st, const CtrlParams &c, const Partial *tot, int nseg,
                             const void *const *klast) {
    const int lane = threadIdx.x & 31;
    const double dt = st->dt;
    const double t_cur = st->t1;
    unsigned status = st->status;
    int cur = st->cursor;
    const long long nadv0 = st->n_steps_adv;
    const unsigned long long n_acc = st->n_acc, n_rej = st->n_rej, attempt = st->attempt;
    const CtrlDecision dec = ctrl_decide<T>(c, tot, nseg, dt);
    const bool accept = dec.accept, bad0 = dec.bad0;
    const double m = dec.m, dt_next = dec.dt_next;
    if (bad0) status |= B2ODE_ST_NONFINITE;   // the reference asserts this before taking the step
    const double t1_new = accept ? t_cur + dt : t_cur;
    // outputs inside the accepted step: every t_out[j] with t_out[j] <= t1 (advance(): `while next_t > t1`);
    // t_out is increasing, so each 32-wide ballot is a run of ones followed by zeros
    const int j0 = cur;
    if (accept && !bad0) {
        for (;;) {
            const int j = cur + lane;
            const bool in = (j < c.n_out) && (c.t_out[j] <= t1_new);
            const unsigned b = __ballot_sync(0xffffffffu, in);
            const int cnt = (b == 0xffffffffu) ? 32 : (__ffs((int)~b) - 1);
            cur += cnt;
            if (cnt < 32) break;
        }
    }
    const long long nadv = (cur > j0) ? 0 : nadv0 + 1;
    int done = (cur >= c.n_out) ? 1 : 0;
    if (!done) {
        if (nadv >= c.max_num_steps) status |= B2ODE_ST_MAXSTEPS;        // dopri5.py:85
        if (!(t1_new + dt_next > t1_new)) status |= B2ODE_ST_UNDERFLOW;  // dopri5.py:98 (NaN dt lands here too)
    }
    if (status) done = 1;
    if (lane == 0) {
        st->dt_last = dt;
        st->msr_max = m;
        if (accept) {
            st->t0 = t_cur;
            st->t1 = t1_new;
            st->n_acc = n_acc + 1;
        } else {
            st->n_rej = n_rej + 1;
        }
        st->accept = accept ? 1 : 0;
        st->attempt = attempt + 1;
        st->dt = dt_next;
        st->cursor = cur;
        st->emit_j0 = j0;
        st->emit_j1 = cur;
        st->n_steps_adv = nadv;
        st->status = status;
        st->done = done;
    }
    if (lane < nseg) st->klast[lane] = reinterpret_cast<unsigned long long>(klast[lane]);
    // stage times of the next attempt (rk_common.py:45-50), one lane each
    if (lane + 1 < c.n_k) {
        T *ts = reinterpret_cast<T *>(c.tstage);
        ts[lane] = Ar<T>::add((T)t1_new, Ar<T>::mul((T)c.alpha[lane], (T)dt_next));
    }
}

template <typename T, int NK>
__global__ void __launch_bounds__(kThreads, B2_MINB_FINALIZE) k_rk_finalize(const __grid_constant__ FinalizeParams<NK> p) {
    const int s = find_seg(p.g, blockIdx.x);
    const int bl = blockIdx.x - p.g.blk_begin[s], nb = p.g.blk_begin[s + 1] - p.g.blk_begin[s];
    const T dt = (T)p.st->dt;
    T c[NK];
#pragma unroll
    for (int j = 0; j < NK; ++j) c[j] = Ar<T>::mul(dt, (T)p.coef[j]);
    const T *y0 = (const T *)p.y0[s], *y1 = (const T *)p.y1[s];
    const T *k[NK];
#pragma unroll
    for (int j = 0; j < NK; ++j) k[j] = (const T *)p.k[j][s];
    double sum = 0.0;
    AbsMax<T> m0, m1;
    bool bad = false;
    seg_for_each<T>(p.g.n[s], (p.g.vec_mask >> s) & 1u, bl, nb, [&](auto vt, long long i) {
        constexpr int V = decltype(vt)::value;
        Pack<T, V> a = ld_pack<T, V>(y0, i);
        Pack<T, V> b = ld_pack<T, V>(y1, i);
        Pack<T, V> kv[NK];
#pragma unroll
        for (int j = 0; j < NK; ++j) kv[j] = ld_pack<T, V>(k[j], i);
#pragma unroll
        for (int e = 0; e < V; ++e) {
            T err = Ar<T>::mul(c[0], kv[0].v[e]);
#pragma unroll
            for (int j = 1; j < NK; ++j) err = Ar<T>::add(err, Ar<T>::mul(c[j], kv[j].v[e]));
            const double ed = (double)err;
            sum += ed * ed;
            m0.see(a.v[e]);
            m1.see(b.v[e]);
            bad |= !isfinite((double)a.v[e]);
        }
    });
    // columns: 0 = sum err^2, 1 = max|y0|, 2 = max|y1| (NaN poisons the tolerance like reduce_max), 3 = non-finite y0
    constexpr unsigned MM = 0xEu;
    Partial mine;
    mine.v[0] = sum;
    mine.v[1] = m0.value();
    mine.v[2] = m1.value();
    mine.v[3] = bad ? 1.0 : 0.0;
    Partial r = block_reduce<MM>(mine);
    if (threadIdx.x == 0) p.part[blockIdx.x] = r;
    if (!last_block_arrives(&p.st->ticket)) return;
    __shared__ Partial tot[B2ODE_MAXSEG];
    reduce_partials<MM>(p.g, p.part, tot);
    group_combine<MM>(p.comm, p.st, tot, p.g.nseg);
    if (threadIdx.x < 32) {
        control_step<T>(p.st, p.c, tot, p.g.nseg, p.klast);
        if (threadIdx.x == 0) p.st->ticket = 0;
    }
}

// ------------------------------------------------------------------------------------------------
// K2+K3, bulk-copy variant (A/B, B2ODE_FINALIZE_BULK=1): the same pass with its (NK + 2) read streams staged through
// shared memory by the TMA engine in linear mode -- one thread issues cp.async.bulk copies of kBulkTile elements per
// stream into a kBulkStages-deep ring, an mbarrier transaction count tells the block when a stage has landed.  north_star
// asks for "TMA-staged shared-memory tiles for the k-stage buffer"; there is no reuse and no tile structure in this pass,
// so the question is only whether the copy engine feeds HBM better than 16-byte LDGs with eight streams in flight per
// thread.  Measured at 65 536 x 128 fp64: profiles/r02_finalize_bulk_ab.md.  One segment, 16-byte aligned pointers.
// ------------------------------------------------------------------------------------------------
constexpr int kBulkTile = 512;       // elements per stream per stage (4 KB fp64, 2 KB fp32)
constexpr int kBulkStages = 3;

__device__ __forceinline__ unsigned smem_addr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait_parity(unsigned long long *bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t}" ::"r"(smem_addr(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst)),
                 "l"(src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}

template <typename T, int NK>
__global__ void __launch_bounds__(kThreads) k_rk_finalize_bulk(const __grid_constant__ FinalizeParams<NK> p) {
    extern __shared__ __align__(128) unsigned char bulk_smem[];
    __shared__ __align__(8) unsigned long long full[kBulkStages];
    constexpr int NS = NK + 2;                                   // streams: y0, y1, k...
    T *ring = reinterpret_cast<T *>(bulk_smem);                  // [stage][stream][kBulkTile]
    const long long n = p.g.n[0];
    const long long ntiles = n / kBulkTile;                      // full tiles; the remainder is read directly
    const T dt = (T)p.st->dt;
    T c[NK];
#pragma unroll
    for (int j = 0; j < NK; ++j) c[j] = Ar<T>::mul(dt, (T)p.coef[j]);
    const T *src[NS];
    src[0] = (const T *)p.y0[0];
    src[1] = (const T *)p.y1[0];
#pragma unroll
    for (int j = 0; j < NK; ++j) src[2 + j] = (const T *)p.k[j][0];
    if (threadIdx.x == 0) {
        for (int s = 0; s < kBulkStages; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    auto issue = [&](long long tile, int stage) {
        mbar_expect_tx(&full[stage], (unsigned)(NS * kBulkTile * sizeof(T)));
#pragma unroll
        for (int q = 0; q < NS; ++q)
            bulk_g2s(ring + ((size_t)stage * NS + q) * kBulkTile, src[q] + tile * kBulkTile, (unsigned)(kBulkTile * sizeof(T)), &full[stage]);
    };
    if (threadIdx.x == 0) {
        for (int s = 0; s < kBulkStages; ++s) {
            const long long tile = (long long)blockIdx.x + (long long)s * gridDim.x;
            if (tile < ntiles) issue(tile, s);
        }
    }
    double sum = 0.0;
    AbsMax<T> m0, m1;
    bool bad = false;
    auto one = [&](T a, T b, const T(&kk)[NK]) {
        T err = Ar<T>::mul(c[0], kk[0]);
#pragma unroll
        for (int j = 1; j < NK; ++j) err = Ar<T>::add(err, Ar<T>::mul(c[j], kk[j]));
        const double ed = (double)err;
        sum += ed * ed;
        m0.see(a);
        m1.see(b);
        bad |= !isfinite((double)a);
    };
    int it = 0;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
        const int stage = it % kBulkStages;
        mbar_wait_parity(&full[stage], (unsigned)((it / kBulkStages) & 1));
        const T *base = ring + (size_t)stage * NS * kBulkTile;
#pragma unroll
        for (int e = threadIdx.x; e < kBulkTile; e += kThreads) {
            T kk[NK];
#pragma unroll
            for (int j = 0; j < NK; ++j) kk[j] = base[(2 + j) * kBulkTile + e];
            one(base[e], base[kBulkTile + e], kk);
        }
        __syncthreads();                                         // everyone has read the stage: it may be refilled
        const long long next = tile + (long long)kBulkStages * gridDim.x;
        if (threadIdx.x == 0 && next < ntiles) issue(next, stage);
    }
    // remainder (n not a multiple of the tile): plain loads, one block
    if (blockIdx.x == 0) {
        for (long long i = ntiles * kBulkTile + threadIdx.x; i < n; i += kThreads) {
            T kk[NK];
#pragma unroll
            for (int j = 0; j < NK; ++j) kk[j] = src[2 + j][i];
            one(src[0][i], src[1][i], kk);
        }
    }
    constexpr unsigned MM = 0xEu;
    Partial mine;
    mine.v[0] = sum;
    mine.v[1] = m0.value();
    mine.v[2] = m1.value();
    mine.v[3] = bad ? 1.0 : 0.0;
    Partial r = block_reduce<MM>(mine);
    if (threadIdx.x == 0) p.part[blockIdx.x] = r;
    if (!last_block_arrives(&p.st->ticket)) return;
    __shared__ Partial tot[B2ODE_MAXSEG];
    reduce_partials<MM>(p.g, p.part, tot);
    group_combine<MM>(p.comm, p.st, tot, p.g.nseg);
    if (threadIdx.x < 32) {
        control_step<T>(p.st, p.c, tot, p.g.nseg, p.klast);
        if (threadIdx.x == 0) p.st->ticket = 0;
    }
}

// ------------------------------------------------------------------------------------------------
// K5: dense output for all output times inside the accepted step
//   y_mid (dopri5.py:42) + _interp_fit (interp.py:22-36) + _interp_evaluate (interp.py:55-67), fused.
// ------------------------------------------------------------------------------------------------
template <int NK>
struct EmitParams {
    SegGeom g;
    const b2ode_state *st;
    const void *y0[B2ODE_MAXSEG];
    const void *y1[B2ODE_MAXSEG];
    const void *k[NK][B2ODE_MAXSEG];   // union of {k_j : c_mid_j != 0} and {f0 = k_0, f1 = k_{s-1}}
    double coef[NK];                   // c_mid of each listed k (0 for f0/f1 if they carry no weight)
    unsigned mid_mask;                 // which listed k's enter y_mid
    void *out[B2ODE_MAXSEG];           // (n_out, n_s) row-major
    const double *t_out;
};

template <typename T, int NK>
__global__ void __launch_bounds__(kThreads) k_emit_quartic(const __grid_constant__ EmitParams<NK> p) {
    const b2ode_state *st = p.st;
    const int j0 = st->emit_j0, j1 = st->emit_j1;
    if (!st->accept || j1 <= j0) return;
    const int s = find_seg(p.g, blockIdx.x);
    const int bl = blockIdx.x - p.g.blk_begin[s], nb = p.g.blk_begin[s + 1] - p.g.blk_begin[s];
    const long long n = p.g.n[s];
    const T dt = (T)st->dt_last;                       // dopri5.py:41 `dt = tf.cast(dt, y0[0].dtype)`
    const T t0 = (T)st->t0, t1 = (T)st->t1;            // interp.py:55-57
    const T den = Ar<T>::sub(t1, t0);
    T c[NK];
#pragma unroll
    for (int j = 0; j < NK; ++j) c[j] = Ar<T>::mul(dt, (T)p.coef[j]);
    const T m2dt = Ar<T>::mul(T(-2), dt), p2dt = Ar<T>::mul(T(2), dt), p5dt = Ar<T>::mul(T(5), dt);
    const T m3dt = Ar<T>::mul(T(-3), dt), m4dt = Ar<T>::mul(T(-4), dt);
    const T *y0 = (const T *)p.y0[s], *y1 = (const T *)p.y1[s];
    T *out = (T *)p.out[s];
    const T *k[NK];
#pragma unroll
    for (int j = 0; j < NK; ++j) k[j] = (const T *)p.k[j][s];
    // rows of `out` keep the 16-byte alignment of the base only if the row length is a multiple of the pack
    constexpr int VW = 16 / sizeof(T);
    const bool vec_ok = ((p.g.vec_mask >> s) & 1u) && (n % VW == 0);
    seg_for_each<T>(n, vec_ok, bl, nb, [&](auto vt, long long i) {
        constexpr int V = decltype(vt)::value;
        Pack<T, V> a0 = ld_pack<T, V>(y0, i);
        Pack<T, V> a1 = ld_pack<T, V>(y1, i);
        Pack<T, V> kv[NK];
#pragma unroll
        for (int j = 0; j < NK; ++j) kv[j] = ld_pack<T, V>(k[j], i);
        T ca[V], cb[V], cc[V], cd[V];
#pragma unroll
        for (int e = 0; e < V; ++e) {
            // y_mid = y0 + sum (dt*c_mid_j) k_j
            T acc = T(0);
            bool first = true;
#pragma unroll
            for (int j = 0; j < NK; ++j) {
                if ((p.mid_mask >> j) & 1u) {
                    const T term = Ar<T>::mul(c[j], kv[j].v[e]);
                    acc = first ? term : Ar<T>::add(acc, term);
                    first = false;
                }
            }
            const T ymid = Ar<T>::add(a0.v[e], acc);
            const T f0 = kv[0].v[e], f1 = kv[NK - 1].v[e], y0e = a0.v[e], y1e = a1.v[e];   // list is k-ordered: f0 first, f1 last
            // interp.py:22-36, python sum() left to right
            T a = Ar<T>::mul(m2dt, f0);
            a = Ar<T>::add(a, Ar<T>::mul(p2dt, f1));
            a = Ar<T>::add(a, Ar<T>::mul(T(-8), y0e));
            a = Ar<T>::add(a, Ar<T>::mul(T(-8), y1e));
            a = Ar<T>::add(a, Ar<T>::mul(T(16), ymid));
            T b = Ar<T>::mul(p5dt, f0);
            b = Ar<T>::add(b, Ar<T>::mul(m3dt, f1));
            b = Ar<T>::add(b, Ar<T>::mul(T(18), y0e));
            b = Ar<T>::add(b, Ar<T>::mul(T(14), y1e));
            b = Ar<T>::add(b, Ar<T>::mul(T(-32), ymid));
            T cq = Ar<T>::mul(m4dt, f0);
            cq = Ar<T>::add(cq, Ar<T>::mul(dt, f1));
            cq = Ar<T>::add(cq, Ar<T>::mul(T(-11), y0e));
            cq = Ar<T>::add(cq, Ar<T>::mul(T(-5), y1e));
            cq = Ar<T>::add(cq, Ar<T>::mul(T(16), ymid));
            ca[e] = a;
            cb[e] = b;
            cc[e] = cq;
            cd[e] = Ar<T>::mul(dt, f0);
        }
        for (int j = j0; j < j1; ++j) {
            const T x = Ar<T>::div(Ar<T>::sub((T)p.t_out[j], t0), den);   // interp.py:60
            const T x2 = Ar<T>::mul(x, x), x3 = Ar<T>::mul(x2, x), x4 = Ar<T>::mul(x3, x);
            Pack<T, V> o;
#pragma unroll
            for (int e = 0; e < V; ++e) {
                T r = Ar<T>::mul(ca[e], x4);
                r = Ar<T>::add(r, Ar<T>::mul(cb[e], x3));
                r = Ar<T>::add(r, Ar<T>::mul(cc[e], x2));
                r = Ar<T>::add(r, Ar<T>::mul(cd[e], x));
                r = Ar<T>::add(r, a0.v[e]);      // e * 1
                o.v[e] = r;
            }
            st_pack<T, V>(out + (long long)j * n, i, o);
        }
    });
}

// tsit5.py:33-50 as written (the "y0" it adds is k[0] = f0, :47): out = f0 + sum_j (dt*b_j(x)) k_j, all 7 k's.
struct EmitTsitParams {
    SegGeom g;
    const b2ode_state *st;
    const void *k[7][B2ODE_MAXSEG];
    void *out[B2ODE_MAXSEG];
    const double *t_out;
};

template <typename T>
__global__ void __launch_bounds__(kThreads) k_emit_tsit5(const __grid_constant__ EmitTsitParams p) {
    const b2ode_state *st = p.st;
    const int j0 = st->emit_j0, j1 = st->emit_j1;
    if (!st->accept || j1 <= j0) return;
    const int s = find_seg(p.g, blockIdx.x);
    const int bl = blockIdx.x - p.g.blk_begin[s], nb = p.g.blk_begin[s + 1] - p.g.blk_begin[s];
    const long long n = p.g.n[s];
    const double dt = st->t1 - st->t0;
    const T *k[7];
#pragma unroll
    for (int j = 0; j < 7; ++j) k[j] = (const T *)p.k[j][s];
    T *out = (T *)p.out[s];
    constexpr int VW = 16 / sizeof(T);
    const bool vec_ok = ((p.g.vec_mask >> s) & 1u) && (n % VW == 0);
    seg_for_each<T>(n, vec_ok, bl, nb, [&](auto vt, long long i) {
        constexpr int V = decltype(vt)::value;
        Pack<T, V> kv[7];
#pragma unroll
        for (int j = 0; j < 7; ++j) kv[j] = ld_pack<T, V>(k[j], i);
        for (int jj = j0; jj < j1; ++jj) {
            const double t = __ddiv_rn(__dsub_rn(p.t_out[jj], st->t0), dt);
            const double t2 = __dmul_rn(t, t);
            double b[7];
            // tsit5.py:35-41, python operator order
            b[0] = __dmul_rn(__dmul_rn(__dmul_rn(-1.0530884977290216, t), __dsub_rn(t, 1.3299890189751412)),
                             __dadd_rn(__dsub_rn(t2, __dmul_rn(1.4364028541716351, t)), 0.7139816917074209));
            b[1] = __dmul_rn(__dmul_rn(0.1017, t2), __dadd_rn(__dsub_rn(t2, __dmul_rn(2.1966568338249754, t)), 1.2949852507374631));
            b[2] = __dmul_rn(__dmul_rn(2.490627285651252793, t2),
                             __dadd_rn(__dsub_rn(t2, __dmul_rn(2.38535645472061657, t)), 1.57803468208092486));
            b[3] = __dmul_rn(__dmul_rn(__dmul_rn(-16.54810288924490272, __dsub_rn(t, 1.21712927295533244)),
                                       __dsub_rn(t, 0.61620406037800089)), t2);
            b[4] = __dmul_rn(__dmul_rn(__dmul_rn(47.37952196281928122, __dsub_rn(t, 1.203071208372362603)),
                                       __dsub_rn(t, 0.658047292653547382)), t2);
            b[5] = __dmul_rn(__dmul_rn(__dmul_rn(-34.87065786149660974, __dsub_rn(t, 1.2)),
                                       __dsub_rn(t, 0.666666666666666667)), t2);
            b[6] = __dmul_rn(__dmul_rn(__dmul_rn(2.5, __dsub_rn(t, 1.0)), __dsub_rn(t, 0.6)), t2);
            T c[7];
#pragma unroll
            for (int j = 0; j < 7; ++j) c[j] = (T)__dmul_rn(dt, b[j]);
            Pack<T, V> o;
#pragma unroll
            for (int e = 0; e < V; ++e) {
                T acc = Ar<T>::mul(c[0], kv[0].v[e]);
#pragma unroll
                for (int j = 1; j < 7; ++j) acc = Ar<T>::add(acc, Ar<T>::mul(c[j], kv[j].v[e]));
                o.v[e] = Ar<T>::add(kv[0].v[e], acc);
            }
            st_pack<T, V>(out + (long long)jj * n, i, o);
        }
    });
}

// ------------------------------------------------------------------------------------------------
// K6: _select_initial_step (misc.py:183-247)
// ------------------------------------------------------------------------------------------------
struct InitParams {
    SegGeom g;
    b2ode_state *st;
    Partial *part;
    const void *y0[B2ODE_MAXSEG];
    const void *f0[B2ODE_MAXSEG];
    const void *f1[B2ODE_MAXSEG];
    void *ystage[B2ODE_MAXSEG];
    double rtol0, atol0;       // the reference passes rtol[0], atol[0] for every component (dopri5.py:74)
    CtrlParams c;
    CommParams comm;
};

// pass 1: d0 = rms(y0/scale), d1 = rms(f0/scale) per segment; last block derives h0 (misc.py:226-234)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_init_norms(const __grid_constant__ InitParams p) {
    const int s = find_seg(p.g, blockIdx.x);
    const int bl = blockIdx.x - p.g.blk_begin[s], nb = p.g.blk_begin[s + 1] - p.g.blk_begin[s];
    const T *y0 = (const T *)p.y0[s], *f0 = (const T *)p.f0[s];
    const T rtol = (T)p.rtol0, atol = (T)p.atol0;
    double s0 = 0.0, s1 = 0.0;
    seg_for_each<T>(p.g.n[s], (p.g.vec_mask >> s) & 1u, bl, nb, [&](auto vt, long long i) {
        constexpr int V = decltype(vt)::value;
        Pack<T, V> a = ld_pack<T, V>(y0, i);
        Pack<T, V> f = ld_pack<T, V>(f0, i);
#pragma unroll
        for (int e = 0; e < V; ++e) {
            const T scale = Ar<T>::add(atol, Ar<T>::mul(Ar<T>::abs(a.v[e]), rtol));
            const double q0 = (double)Ar<T>::div(a.v[e], scale), q1 = (double)Ar<T>::div(f.v[e], scale);
            s0 += q0 * q0;
            s1 += q1 * q1;
        }
    });
    Partial mine;
    mine.v[0] = s0;
    mine.v[1] = s1;
    mine.v[2] = mine.v[3] = 0.0;
    Partial r = block_reduce<0u>(mine);
    if (threadIdx.x == 0) p.part[blockIdx.x] = r;
    if (!last_block_arrives(&p.st->ticket)) return;
    __shared__ Partial tot[B2ODE_MAXSEG];
    reduce_partials<0u>(p.g, p.part, tot);
    group_combine<0u>(p.comm, p.st, tot, p.g.nseg);
    if (threadIdx.x == 0) {
        b2ode_state *st = p.st;
        T d1max;
        const T h0 = init_h0<T>(p.c, tot, p.g.nseg, &d1max);
        st->h0 = (double)h0;
        st->reserved_d[0] = (double)d1max;
        T *ts = reinterpret_cast<T *>(p.c.tstage);
        ts[0] = Ar<T>::add((T)st->t1, h0);                                        // fun(t0 + h0, y1), misc.py:237
        st->ticket = 0;
    }
}

// pass 2: the explicit Euler probe y1 = y0 + h0 * f0 (misc.py:236)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_init_probe(const __grid_constant__ InitParams p) {
    const int s = find_seg(p.g, blockIdx.x);
    const int bl = blockIdx.x - p.g.blk_begin[s], nb = p.g.blk_begin[s + 1] - p.g.blk_begin[s];
    const T h0 = (T)p.st->h0;
    const T *y0 = (const T *)p.y0[s], *f0 = (const T *)p.f0[s];
    T *ys = (T *)p.ystage[s];
    seg_for_each<T>(p.g.n[s], (p.g.vec_mask >> s) & 1u, bl, nb, [&](auto vt, long long i) {
        constexpr int V = decltype(vt)::value;
        Pack<T, V> a = ld_pack<T, V>(y0, i);
        Pack<T, V> f = ld_pack<T, V>(f0, i);
        Pack<T, V> o;
#pragma unroll
        for (int e = 0; e < V; ++e) o.v[e] = Ar<T>::add(a.v[e], Ar<T>::mul(h0, f.v[e]));
        st_pack<T, V>(ys, i, o);
    });
}

// pass 3: d2 = rms((f1 - f0)/scale) / h0; h1; dt = min(100 h0, h1) (misc.py:238-247)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_init_finish(const __grid_constant__ InitParams p) {
    const int s = find_seg(p.g, blockIdx.x);
    const int bl = blockIdx.x - p.g.blk_begin[s], nb = p.g.blk_begin[s + 1] - p.g.blk_begin[s];
    const T *y0 = (const T *)p.y0[s], *f0 = (const T *)p.f0[s], *f1 = (const T *)p.f1[s];
    const T rtol = (T)p.rtol0, atol = (T)p.atol0;
    double s2 = 0.0;
    seg_for_each<T>(p.g.n[s], (p.g.vec_mask >> s) & 1u, bl, nb, [&](auto vt, long long i) {
        constexpr int V = decltype(vt)::value;
        Pack<T, V> a = ld_pack<T, V>(y0, i);
        Pack<T, V> f = ld_pack<T, V>(f0, i);
        Pack<T, V> g = ld_pack<T, V>(f1, i);
#pragma unroll
        for (int e = 0; e < V; ++e) {
            const T scale = Ar<T>::add(atol, Ar<T>::mul(Ar<T>::abs(a.v[e]), rtol));
            const double q = (double)Ar<T>::div(Ar<T>::sub(g.v[e], f.v[e]), scale);
            s2 += q * q;
        }
    });
    Partial mine;
    mine.v[0] = s2;
    mine.v[1] = mine.v[2] = mine.v[3] = 0.0;
    Partial r = block_reduce<0u>(mine);
    if (threadIdx.x == 0) p.part[blockIdx.x] = r;
    if (!last_block_arrives(&p.st->ticket)) return;
    __shared__ Partial tot[B2ODE_MAXSEG];
    reduce_partials<0u>(p.g, p.part, tot);
    group_combine<0u>(p.comm, p.st, tot, p.g.nseg);
    if (threadIdx.x == 0) {
        b2ode_state *st = p.st;
        const T h0 = (T)st->h0;
        const T d1max = (T)st->reserved_d[0];
        const T dt0 = init_dt<T>(p.c, tot, p.g.nseg, h0, d1max);
        st->dt = (double)dt0;                                                     // cast to float64, dopri5.py:75
        if (!(st->t1 + st->dt > st->t1) && st->cursor < p.c.n_out) {
            st->status |= B2ODE_ST_UNDERFLOW;
            st->done = 1;
        }
        write_stage_times<T>(p.c, st->t1, st->dt);
        st->ticket = 0;
    }
}

// state construction (dopri5.py:78); one thread
struct StateInitParams {
    b2ode_state *st;
    double t_start, first_step;
    int have_first_step;
    CtrlParams c;
};
template <typename T>
__global__ void k_state_init(const __grid_constant__ StateInitParams p) {
    b2ode_state z;
    memset(&z, 0, sizeof(z));
    z.t0 = p.t_start;
    z.t1 = p.t_start;
    z.cursor = 1;                         // out[.][0] = y0 (solvers.py:29)
    z.emit_j0 = z.emit_j1 = 1;
    z.done = (p.c.n_out <= 1) ? 1 : 0;
    if (p.have_first_step) {
        z.dt = p.first_step;
        if (!z.done && !(z.t1 + z.dt > z.t1)) {
            z.status |= B2ODE_ST_UNDERFLOW;
            z.done = 1;
        }
    }
    *p.st = z;
    if (p.have_first_step) write_stage_times<T>(p.c, p.t_start, p.first_step);
}

// ------------------------------------------------------------------------------------------------
// K7: fixed-grid ops (fixed_grid.py, rk_common.py:73-81, solvers.py:95,106-115)
// ------------------------------------------------------------------------------------------------
struct FixedParams {
    SegGeom g;
    int op;
    void *out[B2ODE_MAXSEG];
    const void *y[B2ODE_MAXSEG];
    const void *a[B2ODE_MAXSEG];
    const void *b[B2ODE_MAXSEG];
    const void *c[B2ODE_MAXSEG];
    const void *d[B2ODE_MAXSEG];
    double dt, s1, s2;
};

template <typename T, int OP>
__device__ __forceinline__ T fixed_eval(T y, T a, T b, T c, T d, T dt, T s1, T s2) {
    using A = Ar<T>;
    if constexpr (OP == B2ODE_OP_EULER) return A::add(y, A::mul(dt, a));
    if constexpr (OP == B2ODE_OP_HALF_STEP) return A::add(y, A::div(A::mul(a, dt), T(2)));
    if constexpr (OP == B2ODE_OP_HEUN_FINAL) return A::add(y, A::mul(A::div(dt, T(2)), A::add(a, b)));
    if constexpr (OP == B2ODE_OP_RK4_S2) return A::add(y, A::div(A::mul(dt, a), T(3)));
    if constexpr (OP == B2ODE_OP_RK4_S3) return A::add(y, A::mul(dt, A::add(A::div(a, T(-3)), b)));
    if constexpr (OP == B2ODE_OP_RK4_S4) return A::add(y, A::mul(dt, A::add(A::sub(a, b), c)));
    if constexpr (OP == B2ODE_OP_RK4_FINAL)
        return A::add(y, A::mul(A::add(A::add(A::add(a, A::mul(T(3), b)), A::mul(T(3), c)), d), A::div(dt, T(8))));
    if constexpr (OP == B2ODE_OP_LERP) return A::add(y, A::mul(A::div(A::sub(a, y), s1), s2));
    return y;
}

template <int OP>
struct FixedArity {
    static constexpr int n = (OP == B2ODE_OP_HEUN_FINAL || OP == B2ODE_OP_RK4_S3)  ? 2
                             : (OP == B2ODE_OP_RK4_S4)                             ? 3
                             : (OP == B2ODE_OP_RK4_FINAL)                          ? 4
                                                                                   : 1;
};

template <typename T, int OP>
__global__ void __launch_bounds__(kThreads) k_fixed(const __grid_constant__ FixedParams p) {
    const int s = find_seg(p.g, blockIdx.x);
    const int bl = blockIdx.x - p.g.blk_begin[s], nb = p.g.blk_begin[s + 1] - p.g.blk_begin[s];
    constexpr int NA = FixedArity<OP>::n;
    const T dt = (T)p.dt, s1 = (T)p.s1, s2 = (T)p.s2;
    const T *y = (const T *)p.y[s];
    const T *in[4] = {(const T *)p.a[s], (const T *)p.b[s], (const T *)p.c[s], (const T *)p.d[s]};
    T *out = (T *)p.out[s];
    seg_for_each<T>(p.g.n[s], (p.g.vec_mask >> s) & 1u, bl, nb, [&](auto vt, long long i) {
        constexpr int V = decltype(vt)::value;
        Pack<T, V> yv = ld_pack<T, V>(y, i);
        Pack<T, V> iv[4];
#pragma unroll
        for (int j = 0; j < NA; ++j) iv[j] = ld_pack<T, V>(in[j], i);
        Pack<T, V> o;
#pragma unroll
        for (int e = 0; e < V; ++e)
            o.v[e] = fixed_eval<T, OP>(yv.v[e], iv[0].v[e], NA > 1 ? iv[1].v[e] : T(0), NA > 2 ? iv[2].v[e] : T(0),
                                       NA > 3 ? iv[3].v[e] : T(0), dt, s1, s2);
        st_pack<T, V>(out, i, o);
    });
}

// ================================================================================================
// host side
// ================================================================================================
struct b2ode_solver {
    b2ode_adaptive_desc d;
    b2ode_adaptive_buffers b;
    bool bound;
    cudaStream_t stream;
    SegGeom geom;          // blocks per segment; vec_mask filled per launch
    int grid;
    CtrlParams ctrl;
    CommParams comm;
    const void *k[B2ODE_MAXK][B2ODE_MAXSEG];   // k pointers of the current attempt (k[0] = f0)
    // compacted (zero-skipping) coefficient lists
    int st_nk[B2ODE_MAXK];
    int st_idx[B2ODE_MAXK][B2ODE_MAXK];
    double st_coef[B2ODE_MAXK][B2ODE_MAXK];
    int err_nk;
    int err_idx[B2ODE_MAXK];
    double err_coef[B2ODE_MAXK];
    int mid_nk;
    int mid_idx[B2ODE_MAXK];
    double mid_coef[B2ODE_MAXK];
    unsigned mid_mask;
    int mid_if0, mid_if1;
};

static bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static void build_geom(SegGeom *g, int dtype, int nseg, const int64_t *seg_len, int sm_count) {
    const int vw = dtype == B2ODE_F64 ? 2 : 4;
    const int sms = sm_count > 0 ? sm_count : 148;
    const long long cap = (long long)sms * 8;     // 8 x 256 threads = 2048 resident threads per SM
    long long need[B2ODE_MAXSEG], tot = 0;
    for (int s = 0; s < nseg; ++s) {
        long long nv = (seg_len[s] + vw - 1) / vw;
        need[s] = (nv + kThreads - 1) / kThreads;
        if (need[s] < 1) need[s] = 1;
        tot += need[s];
    }
    g->nseg = nseg;
    g->blk_begin[0] = 0;
    for (int s = 0; s < nseg; ++s) {
        long long nb = need[s];
        if (tot > cap) {
            nb = (long long)((double)cap * (double)need[s] / (double)tot);
            if (nb < 1) nb = 1;
        }
        g->blk_begin[s + 1] = g->blk_begin[s] + (int)nb;
        g->n[s] = seg_len[s];
    }
    g->vec_mask = 0;
}

extern "C" int b2ode_version(void) { return B2ODE_ABI_VERSION; }
extern "C" const char *b2ode_last_error(void) { return g_err; }
extern "C" size_t b2ode_state_bytes(void) { return sizeof(b2ode_state); }
extern "C" size_t b2ode_mailbox_bytes(void) { return sizeof(Mailbox); }

extern "C" size_t b2ode_workspace_bytes(const b2ode_adaptive_desc *desc) {
    if (!desc || desc->nseg < 1 || desc->nseg > B2ODE_MAXSEG) return 0;
    SegGeom g;
    build_geom(&g, desc->dtype, desc->nseg, desc->seg_len, desc->sm_count);
    return (size_t)g.blk_begin[g.nseg] * sizeof(Partial);
}

extern "C" int b2ode_adaptive_create(b2ode_solver **out, const b2ode_adaptive_desc *desc) {
    if (!out || !desc) return b2_fail(B2ODE_EINVAL, "null argument");
    if (desc->dtype != B2ODE_F32 && desc->dtype != B2ODE_F64) return b2_fail(B2ODE_EINVAL, "dtype must be 0 or 1");
    if (desc->nseg < 1 || desc->nseg > B2ODE_MAXSEG) return b2_fail(B2ODE_EINVAL, "nseg must be in [1, %d]", B2ODE_MAXSEG);
    if (desc->n_k < 2 || desc->n_k > B2ODE_MAXK) return b2_fail(B2ODE_EINVAL, "n_k must be in [2, %d]", B2ODE_MAXK);
    for (int s = 0; s < desc->nseg; ++s)
        if (desc->seg_len[s] < 0) return b2_fail(B2ODE_EINVAL, "negative segment length");
    if (desc->dense_kind == 1 && desc->n_k != 7) return b2_fail(B2ODE_EINVAL, "tsit5 dense output needs n_k == 7");
    b2ode_solver *s = new (std::nothrow) b2ode_solver();
    if (!s) return b2_fail(B2ODE_ENOMEM, "host allocation failed");
    memset(s, 0, sizeof(*s));
    s->d = *desc;
    build_geom(&s->geom, desc->dtype, desc->nseg, desc->seg_len, desc->sm_count);
    s->grid = s->geom.blk_begin[s->geom.nseg];
    const int nk = desc->n_k;
    // stage rows 0..nk-2 from beta; row nk-1 = c_sol (only launched when !fsal)
    for (int i = 0; i < nk; ++i) {
        int cnt = 0;
        const int len = (i < nk - 1) ? i + 1 : nk;
        for (int j = 0; j < len; ++j) {
            const double v = (i < nk - 1) ? desc->beta[i][j] : desc->c_sol[j];
            if (v != 0.0) {
                s->st_idx[i][cnt] = j;
                s->st_coef[i][cnt] = v;
                ++cnt;
            }
        }
        if (cnt == 0) {   // keep at least one (zero-weight) term so the kernel has something to read
            s->st_idx[i][0] = 0;
            s->st_coef[i][0] = 0.0;
            cnt = 1;
        }
        s->st_nk[i] = cnt;
    }
    s->err_nk = 0;
    for (int j = 0; j < nk; ++j)
        if (desc->c_error[j] != 0.0) {
            s->err_idx[s->err_nk] = j;
            s->err_coef[s->err_nk] = desc->c_error[j];
            ++s->err_nk;
        }
    if (s->err_nk == 0) {
        s->err_idx[0] = 0;
        s->err_coef[0] = 0.0;
        s->err_nk = 1;
    }
    // dense output list: nonzero c_mid, plus f0 and f1
    s->mid_nk = 0;
    s->mid_mask = 0;
    s->mid_if0 = s->mid_if1 = -1;
    if (desc->dense_kind == 0) {
        for (int j = 0; j < nk; ++j) {
            const bool w = desc->c_mid[j] != 0.0;
            if (w || j == 0 || j == nk - 1) {
                if (w) s->mid_mask |= 1u << s->mid_nk;
                if (j == 0) s->mid_if0 = s->mid_nk;
                if (j == nk - 1) s->mid_if1 = s->mid_nk;
                s->mid_idx[s->mid_nk] = j;
                s->mid_coef[s->mid_nk] = desc->c_mid[j];
                ++s->mid_nk;
            }
        }
    }
    CtrlParams &c = s->ctrl;
    c.n_k = nk;
    c.controller = desc->controller;
    for (int i = 0; i < B2ODE_MAXK; ++i) c.alpha[i] = desc->alpha[i];
    for (int i = 0; i < B2ODE_MAXSEG; ++i) {
        c.rtol[i] = desc->rtol[i];
        c.atol[i] = desc->atol[i];
        c.n_global[i] = desc->seg_len[i];
    }
    c.safety = desc->safety;
    c.ifactor = desc->ifactor;
    c.dfactor = desc->dfactor;
    c.exponent = desc->exponent;
    c.inv_safety = 1.0 / desc->safety;
    c.inv_ifactor = 1.0 / desc->ifactor;
    c.inv_dfactor = 1.0 / desc->dfactor;
    c.max_num_steps = desc->max_num_steps;
    c.init_order = desc->init_order;
    s->comm.nranks = 0;
    *out = s;
    return 0;
}

extern "C" void b2ode_adaptive_destroy(b2ode_solver *s) { delete s; }

extern "C" int b2ode_adaptive_bind(b2ode_solver *s, const b2ode_adaptive_buffers *buf, void *cuda_stream) {
    if (!s || !buf) return b2_fail(B2ODE_EINVAL, "null argument");
    if (!buf->state || !buf->workspace || !buf->tstage) return b2_fail(B2ODE_EINVAL, "state/workspace/tstage is null");
    if (buf->workspace_bytes < (size_t)s->grid * sizeof(Partial))
        return b2_fail(B2ODE_ENOMEM, "workspace too small: %zu < %zu", buf->workspace_bytes, (size_t)s->grid * sizeof(Partial));
    if (buf->n_out < 1 || (!buf->t_out && buf->n_out > 0)) return b2_fail(B2ODE_EINVAL, "t_out / n_out invalid");
    for (int i = 0; i < s->d.nseg; ++i) {
        if (s->d.seg_len[i] > 0 && (!buf->y0[i] || !buf->f0[i] || !buf->ystage[i] || !buf->out[i]))
            return b2_fail(B2ODE_EINVAL, "segment %d has a null buffer", i);
    }
    if (!aligned16(buf->state)) return b2_fail(B2ODE_EINVAL, "state must be 16-byte aligned");
    s->b = *buf;
    s->stream = (cudaStream_t)cuda_stream;
    s->ctrl.n_out = buf->n_out;
    s->ctrl.t_out = buf->t_out;
    s->ctrl.tstage = buf->tstage;
    for (int i = 0; i < s->d.nseg; ++i) s->k[0][i] = buf->f0[i];
    s->bound = true;
    return 0;
}

extern "C" int b2ode_set_stream(b2ode_solver *s, void *cuda_stream) {
    if (!s) return b2_fail(B2ODE_EINVAL, "null solver");
    s->stream = (cudaStream_t)cuda_stream;
    return 0;
}

extern "C" int b2ode_comm_attach(b2ode_solver *s, int rank, int nranks, void *const *mailboxes) {
    if (!s) return b2_fail(B2ODE_EINVAL, "null solver");
    if (nranks < 1 || nranks > B2ODE_MAXPEERS || rank < 0 || rank >= nranks) return b2_fail(B2ODE_EINVAL, "bad rank/nranks");
    if (nranks > 1 && !mailboxes) return b2_fail(B2ODE_EINVAL, "mailboxes is null");
    s->comm.rank = rank;
    s->comm.nranks = nranks;
    for (int r = 0; r < nranks; ++r) {
        if (nranks > 1 && !mailboxes[r]) return b2_fail(B2ODE_EINVAL, "mailbox %d is null", r);
        s->comm.box[r] = nranks > 1 ? (Mailbox *)mailboxes[r] : nullptr;
    }
    return 0;
}

// the group-wide element counts (used for the mean in the error ratio) -- set by the host driver after attach
extern "C" int b2ode_comm_set_global_len(b2ode_solver *s, const int64_t *global_len) {
    if (!s || !global_len) return b2_fail(B2ODE_EINVAL, "null argument");
    for (int i = 0; i < s->d.nseg; ++i) {
        if (global_len[i] < s->d.seg_len[i]) return b2_fail(B2ODE_EINVAL, "global length smaller than the local one");
        s->ctrl.n_global[i] = global_len[i];
    }
    return 0;
}

// Segments every rank holds in full with bit-identical values (e.g. the parameter adjoint of odeint_adjoint after its
// all-reduce): their partials are taken from the local rank alone; global_len of such a segment is its local length.
extern "C" int b2ode_comm_set_replicated(b2ode_solver *s, unsigned segment_mask) {
    if (!s) return b2_fail(B2ODE_EINVAL, "null solver");
    s->comm.repl_mask = segment_mask;
    return 0;
}

#define B2_REQUIRE_BOUND(s)                                              \
    do {                                                                 \
        if (!(s)) return b2_fail(B2ODE_EINVAL, "null solver");              \
        if (!(s)->bound) return b2_fail(B2ODE_ESTATE, "solver is not bound"); \
    } while (0)

// ---- launch accounting (bench.py's gpu_launches) and optional per-kernel-family event timing -------------
static unsigned long long g_launches = 0;
void b2_count_launch(void) { ++g_launches; }

enum { B2_FAM_STAGE0 = 0, B2_FAM_STAGE = 1, B2_FAM_FINALIZE = 2, B2_FAM_EMIT = 3, B2_FAM_INIT = 4, B2_FAM_FIXED = 5, B2_FAM_FUSED = 6,
       B2_FAM_STAGE_GEMM = 7, B2_NFAM = 8 };
static_assert(B2_FAM_STAGE_GEMM == kFamStageGemm, "linear stage kernel timing family");
constexpr int kMaxTimed = 2048;   // event pairs per family

struct Timing {
    unsigned mask;
    int n[B2_NFAM];
    cudaEvent_t ev[B2_NFAM][kMaxTimed][2];
    bool created[B2_NFAM];
};
static Timing *g_timing = nullptr;

template <typename K, typename P>
static int launch(K kernel, int grid, cudaStream_t st, const P &p, int fam = -1, size_t dyn_smem = 0) {
    if (grid <= 0) return 0;
    Timing *tm = g_timing;
    bool timed = tm && fam >= 0 && ((tm->mask >> fam) & 1u) && tm->n[fam] < kMaxTimed;
    if (timed) {   // event pairs cannot be read back from a captured graph: only time eager launches
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) timed = false;
    }
    if (timed) B2_CUDA(cudaEventRecord(tm->ev[fam][tm->n[fam]][0], st));
    kernel<<<grid, kThreads, dyn_smem, st>>>(p);
    B2_CUDA(cudaGetLastError());
    if (timed) {
        B2_CUDA(cudaEventRecord(tm->ev[fam][tm->n[fam]][1], st));
        tm->n[fam] += 1;
    }
    ++g_launches;
    return 0;
}

extern "C" unsigned long long b2ode_launch_count(void) { return g_launches; }

// event pair around a launch made elsewhere (b2ode_fused.cu); returns the slot or -1
int b2_timing_begin(int fam, cudaStream_t st) {
    Timing *tm = g_timing;
    if (!(tm && fam >= 0 && fam < B2_NFAM && ((tm->mask >> fam) & 1u) && tm->n[fam] < kMaxTimed)) return -1;
    if (cudaEventRecord(tm->ev[fam][tm->n[fam]][0], st) != cudaSuccess) return -1;
    return tm->n[fam];
}
void b2_timing_end(int fam, int slot, cudaStream_t st) {
    if (slot < 0) return;
    Timing *tm = g_timing;
    if (cudaEventRecord(tm->ev[fam][slot][1], st) == cudaSuccess) tm->n[fam] = slot + 1;
}

// Enable CUDA-event timing of the kernel families in `family_mask` (bit f = family f: 0 stage0, 1 stage,
// 2 finalize, 3 dense output, 4 initial step, 5 fixed grid, 6 fused persistent solve, 7 linear stage GEMM); 0 disables.
// Resets the counters.
extern "C" int b2ode_timing_enable(unsigned family_mask) {
    if (!g_timing) {
        g_timing = new (std::nothrow) Timing();
        if (!g_timing) return b2_fail(B2ODE_ENOMEM, "host allocation failed");
        memset(g_timing, 0, sizeof(Timing));
    }
    for (int f = 0; f < B2_NFAM; ++f) {
        if (((family_mask >> f) & 1u) && !g_timing->created[f]) {
            for (int i = 0; i < kMaxTimed; ++i) {
                B2_CUDA(cudaEventCreate(&g_timing->ev[f][i][0]));
                B2_CUDA(cudaEventCreate(&g_timing->ev[f][i][1]));
            }
            g_timing->created[f] = true;
        }
        g_timing->n[f] = 0;
    }
    g_timing->mask = family_mask;
    return 0;
}

// Sum of the recorded launch durations of one family (synchronises on the last recorded event).
extern "C" int b2ode_timing_read(int family, double *total_ms, int *count) {
    if (!g_timing || family < 0 || family >= B2_NFAM || !total_ms || !count) return b2_fail(B2ODE_EINVAL, "bad timing query");
    double tot = 0.0;
    const int n = g_timing->n[family];
    for (int i = 0; i < n; ++i) {
        float ms = 0.f;
        B2_CUDA(cudaEventSynchronize(g_timing->ev[family][i][1]));
        B2_CUDA(cudaEventElapsedTime(&ms, g_timing->ev[family][i][0], g_timing->ev[family][i][1]));
        tot += (double)ms;
    }
    *total_ms = tot;
    *count = n;
    return 0;
}

// ---- mailboxes of a shared-step group: the one place the library owns device memory ---------------------
// (cudaMalloc'ed so that a CUDA IPC handle can be taken; 87 KB per rank: 7 KB of sequence-numbered slots for the generic kernels,
// 80 KB of 16-byte partial slots for the persistent kernel)
extern "C" int b2ode_mailbox_create(void **dev_ptr, unsigned char handle_out[64]) {
    if (!dev_ptr || !handle_out) return b2_fail(B2ODE_EINVAL, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle is 64 bytes");
    void *p = nullptr;
    B2_CUDA(cudaMalloc(&p, sizeof(Mailbox)));
    B2_CUDA(cudaMemset(p, 0, sizeof(Mailbox)));
    {   // the fused kernel's receive area starts out poisoned (see Mailbox::fused_part)
        constexpr size_t n = sizeof(((Mailbox *)nullptr)->fused_part) / 16;
        std::vector<unsigned long long> poison(2 * n);
        for (size_t i = 0; i < n; ++i) {
            poison[2 * i] = kPoisonW0;
            poison[2 * i + 1] = kPoisonW1;
        }
        B2_CUDA(cudaMemcpy((char *)p + offsetof(Mailbox, fused_part), poison.data(), 16 * n, cudaMemcpyHostToDevice));
    }
    B2_CUDA(cudaDeviceSynchronize());
    cudaIpcMemHandle_t h;
    B2_CUDA(cudaIpcGetMemHandle(&h, p));
    memcpy(handle_out, &h, 64);
    *dev_ptr = p;
    return 0;
}
extern "C" int b2ode_mailbox_open(const unsigned char handle[64], void **peer_ptr) {
    if (!handle || !peer_ptr) return b2_fail(B2ODE_EINVAL, "null argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    B2_CUDA(cudaIpcOpenMemHandle(peer_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}
extern "C" int b2ode_mailbox_close(void *peer_ptr) {
    if (peer_ptr) B2_CUDA(cudaIpcCloseMemHandle(peer_ptr));
    return 0;
}
extern "C" int b2ode_mailbox_destroy(void *dev_ptr) {
    if (dev_ptr) B2_CUDA(cudaFree(dev_ptr));
    return 0;
}

extern "C" int b2ode_adaptive_init(b2ode_solver *s, double t_start, double first_step) {
    B2_REQUIRE_BOUND(s);
    StateInitParams p;
    p.st = (b2ode_state *)s->b.state;
    p.t_start = t_start;
    p.first_step = first_step;
    p.have_first_step = (first_step == first_step) ? 1 : 0;
    p.c = s->ctrl;
    if (s->d.dtype == B2ODE_F64)
        k_state_init<double><<<1, 1, 0, s->stream>>>(p);
    else
        k_state_init<float><<<1, 1, 0, s->stream>>>(p);
    B2_CUDA(cudaGetLastError());
    ++g_launches;
    const size_t esz = s->d.dtype == B2ODE_F64 ? 8 : 4;
    for (int i = 0; i < s->d.nseg; ++i)
        if (s->d.seg_len[i] > 0)
            B2_CUDA(cudaMemcpyAsync(s->b.out[i], s->b.y0[i], (size_t)s->d.seg_len[i] * esz, cudaMemcpyDeviceToDevice, s->stream));
    for (int i = 0; i < s->d.nseg; ++i) s->k[0][i] = s->b.f0[i];
    return 0;
}

static unsigned vec_mask_of(const b2ode_solver *s, const void *const *const *lists, int nlists) {
    unsigned m = 0;
    for (int sg = 0; sg < s->d.nseg; ++sg) {
        bool ok = true;
        for (int l = 0; l < nlists && ok; ++l)
            if (lists[l] && lists[l][sg] && !aligned16(lists[l][sg])) ok = false;
        if (ok) m |= 1u << sg;
    }
    return m;
}

static void fill_init_params(b2ode_solver *s, InitParams *p, const void *const *f1) {
    p->g = s->geom;
    p->st = (b2ode_state *)s->b.state;
    p->part = (Partial *)s->b.workspace;
    for (int i = 0; i < B2ODE_MAXSEG; ++i) {
        p->y0[i] = s->b.y0[i];
        p->f0[i] = s->b.f0[i];
        p->f1[i] = f1 ? f1[i] : nullptr;
        p->ystage[i] = s->b.ystage[i];
    }
    p->rtol0 = s->d.rtol[0];
    p->atol0 = s->d.atol[0];
    p->c = s->ctrl;
    p->comm = s->comm;
    const void *const *lists[4] = {(const void *const *)s->b.y0, (const void *const *)s->b.f0,
                                   (const void *const *)s->b.ystage, f1};
    p->g.vec_mask = vec_mask_of(s, lists, 4);
}

extern "C" int b2ode_initial_step_probe(b2ode_solver *s) {
    B2_REQUIRE_BOUND(s);
    InitParams p;
    fill_init_params(s, &p, nullptr);
    int rc;
    if (s->d.dtype == B2ODE_F64) {
        if ((rc = launch(k_init_norms<double>, s->grid, s->stream, p, B2_FAM_INIT))) return rc;
        return launch(k_init_probe<double>, s->grid, s->stream, p, B2_FAM_INIT);
    }
    if ((rc = launch(k_init_norms<float>, s->grid, s->stream, p, B2_FAM_INIT))) return rc;
    return launch(k_init_probe<float>, s->grid, s->stream, p, B2_FAM_INIT);
}

extern "C" int b2ode_initial_step_finish(b2ode_solver *s, const void *const *f1) {
    B2_REQUIRE_BOUND(s);
    if (!f1) return b2_fail(B2ODE_EINVAL, "f1 is null");
    InitParams p;
    fill_init_params(s, &p, f1);
    if (s->d.dtype == B2ODE_F64) return launch(k_init_finish<double>, s->grid, s->stream, p, B2_FAM_INIT);
    return launch(k_init_finish<float>, s->grid, s->stream, p, B2_FAM_INIT);
}

template <typename T, int NK>
static int launch_stage(b2ode_solver *s, int row) {
    StageParams<NK> p;
    p.g = s->geom;
    p.st = (const b2ode_state *)s->b.state;
    const void *const *lists[NK + 2];
    for (int sg = 0; sg < B2ODE_MAXSEG; ++sg) {
        p.y0[sg] = s->b.y0[sg];
        p.out[sg] = s->b.ystage[sg];
    }
    lists[0] = (const void *const *)s->b.y0;
    lists[1] = (const void *const *)s->b.ystage;
    for (int j = 0; j < NK; ++j) {
        const int kj = s->st_idx[row][j];
        p.coef[j] = s->st_coef[row][j];
        for (int sg = 0; sg < B2ODE_MAXSEG; ++sg) p.k[j][sg] = s->k[kj][sg];
        lists[j + 2] = s->k[kj];
    }
    p.g.vec_mask = vec_mask_of(s, lists, NK + 2);
    return launch(k_rk_stage<T, NK>, s->grid, s->stream, p, B2_FAM_STAGE);
}

template <typename T>
static int dispatch_stage(b2ode_solver *s, int row) {
    switch (s->st_nk[row]) {
#define B2_CASE(N) \
    case N:        \
        return launch_stage<T, N>(s, row);
        B2_CASE(1) B2_CASE(2) B2_CASE(3) B2_CASE(4) B2_CASE(5) B2_CASE(6) B2_CASE(7) B2_CASE(8) B2_CASE(9) B2_CASE(10)
        B2_CASE(11) B2_CASE(12) B2_CASE(13) B2_CASE(14)
#undef B2_CASE
    }
    return b2_fail(B2ODE_EINVAL, "unsupported number of stage terms %d", s->st_nk[row]);
}

// Register k_i (the output of the func call that followed stage i-1) WITHOUT launching the stage kernel: used when
// the stage combine runs as the A-operand producer of a tensor-core dense layer (b2ode_dense_layer) instead.
extern "C" int b2ode_set_k(b2ode_solver *s, int i, const void *const *k_new) {
    B2_REQUIRE_BOUND(s);
    if (i < 1 || i > s->d.n_k - 1 || !k_new) return b2_fail(B2ODE_EINVAL, "bad b2ode_set_k arguments");
    for (int sg = 0; sg < s->d.nseg; ++sg) {
        if (!k_new[sg] && s->d.seg_len[sg] > 0) return b2_fail(B2ODE_EINVAL, "k_new[%d] is null", sg);
        s->k[i][sg] = k_new[sg];
    }
    return 0;
}

extern "C" int b2ode_rk_stage(b2ode_solver *s, int i, const void *const *k_new) {
    B2_REQUIRE_BOUND(s);
    const int nk = s->d.n_k;
    if (i < 0 || i > nk - 1) return b2_fail(B2ODE_EINVAL, "stage index %d out of range", i);
    if (i == nk - 1 && s->d.fsal) return b2_fail(B2ODE_EINVAL, "solution combine requested for an FSAL tableau");
    if (i > 0) {
        if (!k_new) return b2_fail(B2ODE_EINVAL, "k_new is null for stage %d", i);
        for (int sg = 0; sg < s->d.nseg; ++sg) {
            if (!k_new[sg] && s->d.seg_len[sg] > 0) return b2_fail(B2ODE_EINVAL, "k_new[%d] is null", sg);
            s->k[i][sg] = k_new[sg];
        }
    }
    if (i == 0) {
        Stage0Params p;
        p.g = s->geom;
        p.st = (const b2ode_state *)s->b.state;
        for (int sg = 0; sg < B2ODE_MAXSEG; ++sg) {
            p.y0[sg] = s->b.y0[sg];
            p.f0[sg] = s->b.f0[sg];
            p.ystage[sg] = s->b.ystage[sg];
        }
        p.coef = s->d.beta[0][0];
        const void *const *lists[3] = {(const void *const *)s->b.y0, (const void *const *)s->b.f0,
                                       (const void *const *)s->b.ystage};
        p.g.vec_mask = vec_mask_of(s, lists, 3);
        if (s->d.dtype == B2ODE_F64) return launch(k_rk_stage0<double>, s->grid, s->stream, p, B2_FAM_STAGE0);
        return launch(k_rk_stage0<float>, s->grid, s->stream, p, B2_FAM_STAGE0);
    }
    if (s->d.dtype == B2ODE_F64) return dispatch_stage<double>(s, i);
    return dispatch_stage<float>(s, i);
}

// ---- stage kernels with a built-in right-hand side ------------------------------------------------------------------
static int rhs_row_dim(const b2ode_rhs_desc *r) {
    switch (r->kind) {
        case B2ODE_RHS_LORENZ: return 3;
        case B2ODE_RHS_LOTKA_VOLTERRA:
        case B2ODE_RHS_CUBIC_MLP: return 2;
        case B2ODE_RHS_KEPLER: return 4;
        case B2ODE_RHS_LINEAR: return r->n_params >= 1 ? (int)r->params[0] : -1;
    }
    return -1;
}

struct RhsCall {
    int kind;
    double prm[8];
    const void *data;
    double time_sign;
};

template <typename T, typename RHS, int NK>
static int launch_stage_rhs_t(const StageRhsParams<NK> &p, int sm_count, cudaStream_t st) {
    const long long need = (p.rows + kThreads - 1) / kThreads;
    const long long cap = (long long)(sm_count > 0 ? sm_count : 148) * 8;
    const int grid = (int)(need < cap ? (need < 1 ? 1 : need) : cap);
    return launch(k_rk_stage_rhs<T, RHS, NK>, grid, st, p, B2_FAM_STAGE);
}

// B2ODE_RHS_LINEAR: the stage combine feeds a DMMA GEMM in b2ode_linear.cu (its own kernel, timing family 7)
template <typename T, int NK>
static int launch_stage_linear(const StageRhsParams<NK> &p, int sm_count, cudaStream_t st) {
    LinearStageArgs a;
    memset(&a, 0, sizeof(a));
    a.st = p.st;
    a.y0 = p.y0;
    for (int j = 0; j < NK; ++j) {
        a.k[j] = p.k[j];
        a.coef[j] = p.coef[j];
    }
    a.nk = NK;
    a.ystage = p.ystage;
    a.k_out = p.k_out;
    a.rows = p.rows;
    a.D = (int)p.rhs[0];
    a.has_bias = p.rhs[1] != 0.0;
    a.data = p.rhs_data;
    a.time_sign = p.time_sign;
    return b2_launch_stage_linear(std::is_same<T, double>::value ? B2ODE_F64 : B2ODE_F32, a, sm_count, st);
}

template <typename T, int NK>
static int launch_stage_rhs_k(int kind, const StageRhsParams<NK> &p, int sm_count, cudaStream_t st) {
    switch (kind) {
        case B2ODE_RHS_LINEAR: return launch_stage_linear<T, NK>(p, sm_count, st);
        case B2ODE_RHS_LORENZ: return launch_stage_rhs_t<T, RhsLorenz<T>, NK>(p, sm_count, st);
        case B2ODE_RHS_LOTKA_VOLTERRA: return launch_stage_rhs_t<T, RhsLotkaVolterra<T>, NK>(p, sm_count, st);
        case B2ODE_RHS_CUBIC_MLP: return launch_stage_rhs_t<T, RhsCubicMLP<T>, NK>(p, sm_count, st);
        case B2ODE_RHS_KEPLER: return launch_stage_rhs_t<T, RhsKepler<T>, NK>(p, sm_count, st);
    }
    return b2_fail(B2ODE_EINVAL, "unknown built-in right-hand side %d", kind);
}

template <int NK>
static void fill_rhs(StageRhsParams<NK> *p, const b2ode_rhs_desc *r) {
    for (int i = 0; i < 8; ++i) p->rhs[i] = i < r->n_params ? r->params[i] : 0.0;
    p->rhs_data = r->data;
    p->time_sign = r->time_sign;
}

static int check_rhs(const b2ode_rhs_desc *r, long long seg_len, long long *rows) {
    if (!r) return b2_fail(B2ODE_EINVAL, "null right-hand side");
    if (r->n_params < 0 || r->n_params > 8) return b2_fail(B2ODE_EINVAL, "bad rhs params");
    if (r->kind == B2ODE_RHS_LINEAR) {
        const double d = r->n_params >= 1 ? r->params[0] : 0.0;
        if (!(d >= 1.0 && d <= (double)kLinearMaxD) || d != (double)(int)d)
            return b2_fail(B2ODE_EINVAL, "linear right-hand side needs params {D, has_bias} with 1 <= D <= %d", kLinearMaxD);
        if (!r->data) return b2_fail(B2ODE_EINVAL, "linear right-hand side needs its matrix (rhs data)");
    }
    const int D = rhs_row_dim(r);
    if (D < 0) return b2_fail(B2ODE_EINVAL, "unknown built-in right-hand side %d", r->kind);
    if (seg_len % D != 0) return b2_fail(B2ODE_EINVAL, "state length %lld is not a multiple of the row size %d", seg_len, D);
    if (r->kind == B2ODE_RHS_CUBIC_MLP && (!r->data || r->n_params < 2 || r->params[0] < 1 || r->params[0] > 128))
        return b2_fail(B2ODE_EINVAL, "cubic-MLP right-hand side needs {H <= 128, cube} and its weights");
    *rows = seg_len / D;
    return 0;
}

extern "C" int b2ode_rhs_eval(int dtype, const b2ode_rhs_desc *rhs, const void *t_scalar, const void *y, void *k_out, int64_t n,
                              int sm_count, void *cuda_stream) {
    if (!t_scalar || !y || !k_out || n < 1) return b2_fail(B2ODE_EINVAL, "bad arguments");
    long long rows = 0;
    const int rc = check_rhs(rhs, n, &rows);
    if (rc) return rc;
    StageRhsParams<0> p;
    memset(&p, 0, sizeof(p));
    p.y0 = y;
    p.k_out = k_out;
    p.t_scalar = t_scalar;
    p.rows = rows;
    fill_rhs(&p, rhs);
    if (dtype == B2ODE_F64) return launch_stage_rhs_k<double, 0>(rhs->kind, p, sm_count, (cudaStream_t)cuda_stream);
    if (dtype == B2ODE_F32) return launch_stage_rhs_k<float, 0>(rhs->kind, p, sm_count, (cudaStream_t)cuda_stream);
    return b2_fail(B2ODE_EINVAL, "dtype must be 0 or 1");
}

template <typename T, int NK>
static int launch_stage_rhs(b2ode_solver *s, int row, const b2ode_rhs_desc *rhs, void *k_out, long long rows) {
    StageRhsParams<NK> p;
    memset(&p, 0, sizeof(p));
    p.st = (const b2ode_state *)s->b.state;
    p.y0 = s->b.y0[0];
    for (int j = 0; j < NK; ++j) {
        p.k[j] = s->k[s->st_idx[row][j]][0];
        p.coef[j] = s->st_coef[row][j];
    }
    p.ystage = (row == s->d.n_k - 2) ? s->b.ystage[0] : nullptr;     // the last stage's input is y1 (FSAL) / feeds the commit
    p.k_out = k_out;
    p.t_scalar = (const char *)s->b.tstage + (size_t)row * (s->d.dtype == B2ODE_F64 ? 8 : 4);
    p.rows = rows;
    fill_rhs(&p, rhs);
    return launch_stage_rhs_k<T, NK>(rhs->kind, p, s->d.sm_count, s->stream);
}

template <typename T>
static int dispatch_stage_rhs(b2ode_solver *s, int row, const b2ode_rhs_desc *rhs, void *k_out, long long rows) {
    switch (s->st_nk[row]) {
#define B2_CASE(N) \
    case N:        \
        return launch_stage_rhs<T, N>(s, row, rhs, k_out, rows);
        B2_CASE(1) B2_CASE(2) B2_CASE(3) B2_CASE(4) B2_CASE(5) B2_CASE(6) B2_CASE(7) B2_CASE(8) B2_CASE(9) B2_CASE(10)
        B2_CASE(11) B2_CASE(12) B2_CASE(13)
#undef B2_CASE
    }
    return b2_fail(B2ODE_EINVAL, "unsupported number of stage terms %d", s->st_nk[row]);
}

extern "C" int b2ode_rk_stage_rhs(b2ode_solver *s, int i, const void *const *k_new, const b2ode_rhs_desc *rhs, void *k_out) {
    B2_REQUIRE_BOUND(s);
    const int nk = s->d.n_k;
    if (s->d.nseg != 1) return b2_fail(B2ODE_EINVAL, "built-in right-hand sides take a single-tensor state");
    if (i < 1 || i > nk - 2) return b2_fail(B2ODE_EINVAL, "stage index %d out of range for a fused right-hand side", i);
    if (!k_new || !k_new[0] || !k_out) return b2_fail(B2ODE_EINVAL, "null k buffer");
    long long rows = 0;
    const int rc = check_rhs(rhs, s->d.seg_len[0], &rows);
    if (rc) return rc;
    s->k[i][0] = k_new[0];
    if (s->d.dtype == B2ODE_F64) return dispatch_stage_rhs<double>(s, i, rhs, k_out, rows);
    return dispatch_stage_rhs<float>(s, i, rhs, k_out, rows);
}

template <typename T, int NK>
static int launch_finalize(b2ode_solver *s) {
    FinalizeParams<NK> p;
    p.g = s->geom;
    p.st = (b2ode_state *)s->b.state;
    p.part = (Partial *)s->b.workspace;
    const void *const *lists[NK + 2];
    for (int sg = 0; sg < B2ODE_MAXSEG; ++sg) {
        p.y0[sg] = s->b.y0[sg];
        p.y1[sg] = s->b.ystage[sg];
    }
    lists[0] = (const void *const *)s->b.y0;
    lists[1] = (const void *const *)s->b.ystage;
    for (int j = 0; j < NK; ++j) {
        const int kj = s->err_idx[j];
        p.coef[j] = s->err_coef[j];
        for (int sg = 0; sg < B2ODE_MAXSEG; ++sg) p.k[j][sg] = s->k[kj][sg];
        lists[j + 2] = s->k[kj];
    }
    for (int sg = 0; sg < B2ODE_MAXSEG; ++sg) p.klast[sg] = s->k[s->d.n_k - 1][sg];
    p.c = s->ctrl;
    p.comm = s->comm;
    p.g.vec_mask = vec_mask_of(s, lists, NK + 2);
    static int bulk = -1;            // A/B switch (profiles/r02_finalize_bulk_ab.md); default = the LDG kernel
    if (bulk < 0) {
        const char *e = getenv("B2ODE_FINALIZE_BULK");
        bulk = (e && e[0] == '1') ? 1 : 0;
    }
    if (bulk && s->d.nseg == 1 && (p.g.vec_mask & 1u) && s->d.seg_len[0] >= (long long)kBulkTile * 4) {
        const size_t smem = (size_t)kBulkStages * (NK + 2) * kBulkTile * sizeof(T);
        if (smem <= 200 * 1024) {
            static bool configured[64][15] = {};
            int dev = 0;
            B2_CUDA(cudaGetDevice(&dev));
            if (dev >= 0 && dev < 64 && !configured[dev][NK]) {
                B2_CUDA(cudaFuncSetAttribute(k_rk_finalize_bulk<T, NK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                configured[dev][NK] = true;
            }
            const long long ntiles = s->d.seg_len[0] / kBulkTile;
            const int sms = s->d.sm_count > 0 ? s->d.sm_count : 148;
            const int per_sm = (int)((220 * 1024) / (smem + 1024)) < 1 ? 1 : (int)((220 * 1024) / (smem + 1024));
            long long grid = (long long)sms * per_sm;
            if (grid > ntiles) grid = ntiles;
            if (grid > s->grid) grid = s->grid;          // the partial array was sized for s->grid blocks
            p.g.blk_begin[1] = (int)grid;                 // reduce_partials walks [blk_begin[0], blk_begin[1])
            return launch(k_rk_finalize_bulk<T, NK>, (int)grid, s->stream, p, B2_FAM_FINALIZE, smem);
        }
    }
    return launch(k_rk_finalize<T, NK>, s->grid, s->stream, p, B2_FAM_FINALIZE);
}

template <typename T, int NK>
static int launch_emit(b2ode_solver *s) {
    EmitParams<NK> p;
    p.g = s->geom;
    p.st = (const b2ode_state *)s->b.state;
    const void *const *lists[NK + 3];
    for (int sg = 0; sg < B2ODE_MAXSEG; ++sg) {
        p.y0[sg] = s->b.y0[sg];
        p.y1[sg] = s->b.ystage[sg];
        p.out[sg] = s->b.out[sg];
    }
    lists[0] = (const void *const *)s->b.y0;
    lists[1] = (const void *const *)s->b.ystage;
    lists[2] = (const void *const *)s->b.out;
    for (int j = 0; j < NK; ++j) {
        const int kj = s->mid_idx[j];
        p.coef[j] = s->mid_coef[j];
        for (int sg = 0; sg < B2ODE_MAXSEG; ++sg) p.k[j][sg] = s->k[kj][sg];
        lists[j + 3] = s->k[kj];
    }
    p.mid_mask = s->mid_mask;
    p.t_out = s->b.t_out;
    p.g.vec_mask = vec_mask_of(s, lists, NK + 3);
    return launch(k_emit_quartic<T, NK>, s->grid, s->stream, p, B2_FAM_EMIT);
}

template <typename T>
static int launch_emit_tsit5(b2ode_solver *s) {
    EmitTsitParams p;
    p.g = s->geom;
    p.st = (const b2ode_state *)s->b.state;
    const void *const *lists[8];
    for (int sg = 0; sg < B2ODE_MAXSEG; ++sg) p.out[sg] = s->b.out[sg];
    lists[0] = (const void *const *)s->b.out;
    for (int j = 0; j < 7; ++j) {
        for (int sg = 0; sg < B2ODE_MAXSEG; ++sg) p.k[j][sg] = s->k[j][sg];
        lists[j + 1] = s->k[j];
    }
    p.t_out = s->b.t_out;
    p.g.vec_mask = vec_mask_of(s, lists, 8);
    return launch(k_emit_tsit5<T>, s->grid, s->stream, p, B2_FAM_EMIT);
}

template <typename T>
static int dispatch_finalize(b2ode_solver *s) {
    int rc = B2ODE_EINVAL;
    switch (s->err_nk) {
#define B2_CASE(N)                      \
    case N:                             \
        rc = launch_finalize<T, N>(s);  \
        break;
        B2_CASE(1) B2_CASE(2) B2_CASE(3) B2_CASE(4) B2_CASE(5) B2_CASE(6) B2_CASE(7) B2_CASE(8) B2_CASE(9) B2_CASE(10)
        B2_CASE(11) B2_CASE(12) B2_CASE(13) B2_CASE(14)
#undef B2_CASE
    }
    if (rc) return rc;
    if (s->d.dense_kind == 1) return launch_emit_tsit5<T>(s);
    switch (s->mid_nk) {
#define B2_CASE(N) \
    case N:        \
        return launch_emit<T, N>(s);
        B2_CASE(1) B2_CASE(2) B2_CASE(3) B2_CASE(4) B2_CASE(5) B2_CASE(6) B2_CASE(7) B2_CASE(8) B2_CASE(9) B2_CASE(10)
        B2_CASE(11) B2_CASE(12) B2_CASE(13) B2_CASE(14)
#undef B2_CASE
    }
    return b2_fail(B2ODE_EINVAL, "unsupported dense-output list length %d", s->mid_nk);
}

extern "C" int b2ode_rk_finalize(b2ode_solver *s, const void *const *k_last) {
    B2_REQUIRE_BOUND(s);
    if (!k_last) return b2_fail(B2ODE_EINVAL, "k_last is null");
    const int nk = s->d.n_k;
    for (int sg = 0; sg < s->d.nseg; ++sg) {
        if (!k_last[sg] && s->d.seg_len[sg] > 0) return b2_fail(B2ODE_EINVAL, "k_last[%d] is null", sg);
        s->k[nk - 1][sg] = k_last[sg];
    }
    int rc = (s->d.dtype == B2ODE_F64) ? dispatch_finalize<double>(s) : dispatch_finalize<float>(s);
    return rc;
}

extern "C" int b2ode_poll_async(b2ode_solver *s, b2ode_state *host_dst) {
    B2_REQUIRE_BOUND(s);
    if (!host_dst) return b2_fail(B2ODE_EINVAL, "host_dst is null");
    B2_CUDA(cudaMemcpyAsync(host_dst, s->b.state, sizeof(b2ode_state), cudaMemcpyDeviceToHost, s->stream));
    return 0;
}

extern "C" int b2ode_poll_sync(b2ode_solver *s, b2ode_state *host_dst) {
    int rc = b2ode_poll_async(s, host_dst);
    if (rc) return rc;
    B2_CUDA(cudaStreamSynchronize(s->stream));
    return 0;
}

// ---- fixed grid --------------------------------------------------------------------------------
template <typename T>
static int dispatch_fixed(int op, int grid, cudaStream_t st, const FixedParams &p) {
    switch (op) {
#define B2_CASE(OP) \
    case OP:        \
        return launch(k_fixed<T, OP>, grid, st, p, B2_FAM_FIXED);
        B2_CASE(B2ODE_OP_EULER) B2_CASE(B2ODE_OP_HALF_STEP) B2_CASE(B2ODE_OP_HEUN_FINAL) B2_CASE(B2ODE_OP_RK4_S2)
        B2_CASE(B2ODE_OP_RK4_S3) B2_CASE(B2ODE_OP_RK4_S4) B2_CASE(B2ODE_OP_RK4_FINAL) B2_CASE(B2ODE_OP_LERP)
#undef B2_CASE
    }
    return b2_fail(B2ODE_EINVAL, "unknown fixed-grid op %d", op);
}

extern "C" int b2ode_fixed_op(int dtype, int op, int nseg, const int64_t *seg_len, void *const *out, const void *const *y,
                              const void *const *a, const void *const *b, const void *const *c, const void *const *d,
                              double dt, double s1, double s2, int sm_count, void *cuda_stream) {
    if (dtype != B2ODE_F32 && dtype != B2ODE_F64) return b2_fail(B2ODE_EINVAL, "dtype must be 0 or 1");
    if (nseg < 1 || nseg > B2ODE_MAXSEG || !seg_len || !out || !y || !a) return b2_fail(B2ODE_EINVAL, "bad segment arguments");
    int arity = 1;
    switch (op) {
        case B2ODE_OP_HEUN_FINAL:
        case B2ODE_OP_RK4_S3: arity = 2; break;
        case B2ODE_OP_RK4_S4: arity = 3; break;
        case B2ODE_OP_RK4_FINAL: arity = 4; break;
        default: break;
    }
    if ((arity > 1 && !b) || (arity > 2 && !c) || (arity > 3 && !d)) return b2_fail(B2ODE_EINVAL, "op %d needs %d operands", op, arity);
    FixedParams p;
    memset(&p, 0, sizeof(p));
    build_geom(&p.g, dtype, nseg, seg_len, sm_count);
    p.op = op;
    unsigned mask = 0;
    for (int s = 0; s < nseg; ++s) {
        if (seg_len[s] < 0) return b2_fail(B2ODE_EINVAL, "negative segment length");
        p.out[s] = out[s];
        p.y[s] = y[s];
        p.a[s] = a[s];
        p.b[s] = arity > 1 ? b[s] : nullptr;
        p.c[s] = arity > 2 ? c[s] : nullptr;
        p.d[s] = arity > 3 ? d[s] : nullptr;
        if (seg_len[s] > 0 && (!p.out[s] || !p.y[s] || !p.a[s] || (arity > 1 && !p.b[s]) || (arity > 2 && !p.c[s]) ||
                               (arity > 3 && !p.d[s])))
            return b2_fail(B2ODE_EINVAL, "segment %d has a null operand", s);
        if (aligned16(p.out[s]) && aligned16(p.y[s]) && aligned16(p.a[s]) && aligned16(p.b[s]) && aligned16(p.c[s]) &&
            aligned16(p.d[s]))
            mask |= 1u << s;
    }
    p.g.vec_mask = mask;
    p.dt = dt;
    p.s1 = s1;
    p.s2 = s2;
    const int grid = p.g.blk_begin[nseg];
    if (dtype == B2ODE_F64) return dispatch_fixed<double>(op, grid, (cudaStream_t)cuda_stream, p);
    return dispatch_fixed<float>(op, grid, (cudaStream_t)cuda_stream, p);
}

// ================================================================================================
// multistep solvers (SURVEY 8f-4: tfdiffeq/fixed_adams.py, tfdiffeq/adams.py)
//
// Their arithmetic is linear combinations of stored derivative tensors plus three reductions; the step logic
// (history, order selection, functional iteration) is host code like the reference's.  Two kernels:
//   k_lincomb : out = base + scale * sum_j coef[j] * x[j]      (products and sums in the state dtype, left to right,
//               no contraction: the order of `dt * _scaled_dot_product(...)`, misc.py:118-121)
//   k_reduce  : per segment, two numbers, deterministic (block partials combined in block order by the last block)
// ================================================================================================
constexpr int kMaxTerms = 16;

struct LincombParams {
    SegGeom g;
    void *out[B2ODE_MAXSEG];
    const void *base[B2ODE_MAXSEG];
    const void *x[kMaxTerms][B2ODE_MAXSEG];
    double coef[kMaxTerms];
    double scale;
    int nterms, has_base, has_scale;
};

template <typename T>
__global__ void __launch_bounds__(kThreads) k_lincomb(const __grid_constant__ LincombParams p) {
    const int s = find_seg(p.g, blockIdx.x);
    const int bl = blockIdx.x - p.g.blk_begin[s], nb = p.g.blk_begin[s + 1] - p.g.blk_begin[s];
    T *out = (T *)p.out[s];
    const T *base = (const T *)p.base[s];
    const T scale = (T)p.scale;
    seg_for_each<T>(p.g.n[s], (p.g.vec_mask >> s) & 1u, bl, nb, [&](auto vt, long long i) {
        constexpr int V = decltype(vt)::value;
        Pack<T, V> acc;
#pragma unroll
        for (int e = 0; e < V; ++e) acc.v[e] = T(0);
        for (int j = 0; j < p.nterms; ++j) {
            const Pack<T, V> xv = ld_pack<T, V>((const T *)p.x[j][s], i);
            const T c = (T)p.coef[j];
#pragma unroll
            for (int e = 0; e < V; ++e) {
                const T term = Ar<T>::mul(c, xv.v[e]);
                acc.v[e] = j ? Ar<T>::add(acc.v[e], term) : term;
            }
        }
        if (p.has_scale) {
#pragma unroll
            for (int e = 0; e < V; ++e) acc.v[e] = Ar<T>::mul(scale, acc.v[e]);
        }
        if (p.has_base) {
            const Pack<T, V> bv = ld_pack<T, V>(base, i);
#pragma unroll
            for (int e = 0; e < V; ++e) acc.v[e] = Ar<T>::add(bv.v[e], acc.v[e]);
        }
        st_pack<T, V>(out, i, acc);
    });
}

extern "C" int b2ode_lincomb(int dtype, int nseg, const int64_t *seg_len, void *const *out, const void *const *base, double scale,
                             int nterms, const void *const *xs, const double *coef, int sm_count, void *cuda_stream) {
    if (dtype != B2ODE_F32 && dtype != B2ODE_F64) return b2_fail(B2ODE_EINVAL, "dtype must be 0 or 1");
    if (nseg < 1 || nseg > B2ODE_MAXSEG || !seg_len || !out) return b2_fail(B2ODE_EINVAL, "bad segment arguments");
    if (nterms < 1 || nterms > kMaxTerms || !xs || !coef) return b2_fail(B2ODE_EINVAL, "lincomb takes 1..%d terms", kMaxTerms);
    LincombParams p;
    memset(&p, 0, sizeof(p));
    build_geom(&p.g, dtype, nseg, seg_len, sm_count);
    unsigned mask = 0;
    for (int s = 0; s < nseg; ++s) {
        if (seg_len[s] < 0) return b2_fail(B2ODE_EINVAL, "negative segment length");
        p.out[s] = out[s];
        p.base[s] = base ? base[s] : nullptr;
        bool al = aligned16(p.out[s]) && aligned16(p.base[s]);
        if (seg_len[s] > 0 && (!p.out[s] || (base && !p.base[s]))) return b2_fail(B2ODE_EINVAL, "segment %d has a null operand", s);
        for (int j = 0; j < nterms; ++j) {
            p.x[j][s] = xs[(size_t)j * nseg + s];
            if (seg_len[s] > 0 && !p.x[j][s]) return b2_fail(B2ODE_EINVAL, "term %d of segment %d is null", j, s);
            al = al && aligned16(p.x[j][s]);
        }
        if (al) mask |= 1u << s;
    }
    p.g.vec_mask = mask;
    for (int j = 0; j < nterms; ++j) p.coef[j] = coef[j];
    p.scale = scale;
    p.nterms = nterms;
    p.has_base = base ? 1 : 0;
    p.has_scale = scale != 1.0 ? 1 : 0;      // 1 * x is exact: skipping it changes nothing
    const int grid = p.g.blk_begin[nseg];
    if (dtype == B2ODE_F64) return launch(k_lincomb<double>, grid, (cudaStream_t)cuda_stream, p, B2_FAM_FIXED);
    return launch(k_lincomb<float>, grid, (cudaStream_t)cuda_stream, p, B2_FAM_FIXED);
}

struct ReduceParams {
    SegGeom g;
    const void *a[B2ODE_MAXSEG];
    const void *b[B2ODE_MAXSEG];
    double p0[B2ODE_MAXSEG], p1[B2ODE_MAXSEG];
    Partial *partials;
    unsigned *ticket;
    double *out;
};

// MODE B2ODE_RED_ABSMAX2   : out = { max|a|, max|b| }                (NaN-propagating; misc.py:257, adams.py:160-163)
//      B2ODE_RED_RATIO_SUMSQ: out = { sum ((p0 * a) / p1)^2, 0 }     (misc.py:259-264 with error_tol given: adams.py:164-166)
//      B2ODE_RED_NOT_CONVERGED: out = { #elements with NOT |a-b| < p1 + p0 * max(|a|,|b|), 0 }   (misc.py:129-134)
template <typename T, int MODE>
__global__ void __launch_bounds__(kThreads) k_reduce(const __grid_constant__ ReduceParams p) {
    constexpr unsigned MM = MODE == B2ODE_RED_ABSMAX2 ? 0x3u : 0x0u;
    const int s = find_seg(p.g, blockIdx.x);
    const int bl = blockIdx.x - p.g.blk_begin[s], nb = p.g.blk_begin[s + 1] - p.g.blk_begin[s];
    const T *a = (const T *)p.a[s];
    const T *b = (const T *)p.b[s];
    const T p0 = (T)p.p0[s], p1 = (T)p.p1[s];
    AbsMax<T> ma, mb;
    double sum = 0.0;
    seg_for_each<T>(p.g.n[s], (p.g.vec_mask >> s) & 1u, bl, nb, [&](auto vt, long long i) {
        constexpr int V = decltype(vt)::value;
        const Pack<T, V> av = ld_pack<T, V>(a, i);
        if constexpr (MODE == B2ODE_RED_RATIO_SUMSQ) {
#pragma unroll
            for (int e = 0; e < V; ++e) {
                const T r = Ar<T>::div(Ar<T>::mul(p0, av.v[e]), p1);
                sum += (double)Ar<T>::mul(r, r);
            }
        } else {
            const Pack<T, V> bv = ld_pack<T, V>(b, i);
#pragma unroll
            for (int e = 0; e < V; ++e) {
                if constexpr (MODE == B2ODE_RED_ABSMAX2) {
                    ma.see(av.v[e]);
                    mb.see(bv.v[e]);
                } else {
                    const T aa = Ar<T>::abs(av.v[e]), ab = Ar<T>::abs(bv.v[e]);
                    const T mx = (aa != aa || ab != ab) ? (T)NAN : (aa > ab ? aa : ab);
                    const T tol = Ar<T>::add(p1, Ar<T>::mul(p0, mx));
                    const T err = Ar<T>::abs(Ar<T>::sub(av.v[e], bv.v[e]));
                    sum += (err < tol) ? 0.0 : 1.0;
                }
            }
        }
    });
    Partial mine = identity<MM>();
    if (MODE == B2ODE_RED_ABSMAX2) {
        mine.v[0] = ma.value();
        mine.v[1] = mb.value();
    } else {
        mine.v[0] = sum;
    }
    mine = block_reduce<MM>(mine);
    if (threadIdx.x == 0) p.partials[blockIdx.x] = mine;
    if (last_block_arrives(p.ticket)) {
        if ((int)threadIdx.x < p.g.nseg) {
            const int sg = threadIdx.x;
            Partial tot = p.partials[p.g.blk_begin[sg]];
            for (int q = p.g.blk_begin[sg] + 1; q < p.g.blk_begin[sg + 1]; ++q) tot = combine<MM>(tot, p.partials[q]);
            p.out[2 * sg + 0] = tot.v[0];
            p.out[2 * sg + 1] = tot.v[1];
        }
        if (threadIdx.x == 0) *p.ticket = 0u;                   // ready for the next launch on the same workspace
    }
}

extern "C" size_t b2ode_reduce_workspace_bytes(int sm_count) {
    const int sms = sm_count > 0 ? sm_count : 148;
    return 64 + sizeof(Partial) * ((size_t)sms * 8 + 2 * B2ODE_MAXSEG);
}

extern "C" int b2ode_reduce(int dtype, int mode, int nseg, const int64_t *seg_len, const void *const *a, const void *const *b,
                            const double *p0, const double *p1, double *out, void *workspace, size_t workspace_bytes, int sm_count,
                            void *cuda_stream) {
    if (dtype != B2ODE_F32 && dtype != B2ODE_F64) return b2_fail(B2ODE_EINVAL, "dtype must be 0 or 1");
    if (nseg < 1 || nseg > B2ODE_MAXSEG || !seg_len || !a || !out || !workspace) return b2_fail(B2ODE_EINVAL, "bad segment arguments");
    if (mode < B2ODE_RED_ABSMAX2 || mode > B2ODE_RED_NOT_CONVERGED) return b2_fail(B2ODE_EINVAL, "unknown reduction %d", mode);
    if (mode != B2ODE_RED_RATIO_SUMSQ && !b) return b2_fail(B2ODE_EINVAL, "reduction %d needs two operands", mode);
    if (mode != B2ODE_RED_ABSMAX2 && (!p0 || !p1)) return b2_fail(B2ODE_EINVAL, "reduction %d needs its scalars", mode);
    if (workspace_bytes < b2ode_reduce_workspace_bytes(sm_count) || ((uintptr_t)workspace & 15u))
        return b2_fail(B2ODE_EINVAL, "reduce workspace too small or misaligned");
    ReduceParams p;
    memset(&p, 0, sizeof(p));
    build_geom(&p.g, dtype, nseg, seg_len, sm_count);
    unsigned mask = 0;
    for (int s = 0; s < nseg; ++s) {
        if (seg_len[s] < 0) return b2_fail(B2ODE_EINVAL, "negative segment length");
        p.a[s] = a[s];
        p.b[s] = b ? b[s] : nullptr;
        if (seg_len[s] > 0 && (!p.a[s] || (mode != B2ODE_RED_RATIO_SUMSQ && !p.b[s])))
            return b2_fail(B2ODE_EINVAL, "segment %d has a null operand", s);
        if (aligned16(p.a[s]) && aligned16(p.b[s])) mask |= 1u << s;
        p.p0[s] = p0 ? p0[s] : 0.0;
        p.p1[s] = p1 ? p1[s] : 0.0;
    }
    p.g.vec_mask = mask;
    p.ticket = (unsigned *)workspace;
    p.partials = (Partial *)((char *)workspace + 64);
    p.out = out;
    const int grid = p.g.blk_begin[nseg];
    cudaStream_t st = (cudaStream_t)cuda_stream;
#define B2_RED(T)                                                                                                        \
    (mode == B2ODE_RED_ABSMAX2       ? launch(k_reduce<T, B2ODE_RED_ABSMAX2>, grid, st, p, B2_FAM_FIXED)                 \
     : mode == B2ODE_RED_RATIO_SUMSQ ? launch(k_reduce<T, B2ODE_RED_RATIO_SUMSQ>, grid, st, p, B2_FAM_FIXED)             \
                                     : launch(k_reduce<T, B2ODE_RED_NOT_CONVERGED>, grid, st, p, B2_FAM_FIXED))
    return dtype == B2ODE_F64 ? B2_RED(double) : B2_RED(float);
#undef B2_RED
}
