// b2ode_fused.cu -- whole adaptive solve in ONE persistent kernel for built-in right-hand sides.
//
// SURVEY.md 8(f)-2.  When `func` is one of the library's own right-hand sides (tfdiffeq_b200/rhs.py), the user
// callable does not have to be called from the host at all: every trajectory of the batch lives in the
// registers of one thread -- state, all s stage derivatives -- for the entire solve; the only HBM traffic is
// the (T, B, D) solution slab, written once.  The reference semantics are kept exactly: ONE step size for
// the whole batch and a tolerance that is a global scalar over the whole tensor (tfdiffeq/misc.py:257), so
// every attempt needs one grid-wide reduction; it is done with a sense-reversing grid barrier (cooperative
// launch guarantees co-residency) and evaluated redundantly -- and bit-identically -- by every thread.
// The arithmetic is the same as the generic path's kernels (same helpers from b2ode_dev.cuh, same operation
// order: rk_common.py:49-60, misc.py:250-287, interp.py:6-67), only the reduction order differs.

#include "b2ode_dev.cuh"
#include "b2ode_rhs.cuh"
#include "b2ode_pay16.cuh"
#include <stdlib.h>

// ------------------------------------------------------------------------------------------------
// optional timeline stamps (-DB2ODE_FUSED_TRACE, scripts/fused_trace.py): thread 0 of two blocks records clock64() at the
// phase boundaries of attempts [8, 8 + kTraceAttempts); compiled out of the shipped library
// ------------------------------------------------------------------------------------------------
#ifdef B2ODE_FUSED_TRACE
constexpr int kTraceAttempts = 64, kTracePhases = 16;
__device__ unsigned long long g_fused_trace[2 * kTraceAttempts * kTracePhases];
// `dep` is a value that only exists after the event being stamped (a word read after a barrier / received from a poll):
// the clock read is predicated on it, so ptxas cannot hoist the read above the event (an unanchored clock64() was observed
// to float above BAR.SYNC)
#define FTRACE_DEP(att, ph, dep)                                                                                 \
    do {                                                                                                         \
        if ((unsigned)(dep) != 0x7ffffff3u && (threadIdx.x == 0 || threadIdx.x == blockDim.x - 32) /* single-GPU traces: the control warp is the last warp */ &&            \
            (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1) && (att) >= 8 && (att) < 8 + kTraceAttempts)        \
            g_fused_trace[((blockIdx.x == 0 ? 0 : 1) * kTraceAttempts + ((att)-8)) * kTracePhases + (ph)] = clock64(); \
    } while (0)
#define FTRACE(att, ph) FTRACE_DEP(att, ph, 0)
extern "C" int b2ode_debug_fused_trace(unsigned long long *out) {
    B2_CUDA(cudaMemcpyFromSymbol(out, g_fused_trace, sizeof(g_fused_trace)));
    return 0;
}
#else
#define FTRACE(att, ph) do { } while (0)
#define FTRACE_DEP(att, ph, dep) do { } while (0)
#endif

// Block size is a template parameter: 512 threads (one block per SM, the fewest barrier arrivals and partials)
// when the kernel fits in 128 registers per thread, 128 threads otherwise.

// ------------------------------------------------------------------------------------------------
// Grid-wide (and group-wide) all-reduce of two 64-bit values per attempt, built for LATENCY: measured on the round-1
// kernel (scripts/fused_trace.py) an attempt cost 15.7k cycles of which only 3.1k were the Runge-Kutta arithmetic; the
// rest was two block reductions with __syncthreads (1.2k + 2.9k), an atomic grid barrier (2.5k), the serial controller
// (3.1k) and the dense output (2.4k), all on every thread's critical path.  Now:
//   * one CONTROL WARP per block owns the whole protocol; the compute warps hand it their warp partials through shared
//     memory and a named barrier (bar.arrive, they do not wait), write the dense output of the step SPECULATIVELY while
//     the control warp talks to the rest of the GPU, and pick the decision up at a second named barrier;
//   * no atomics, no fences: a value travels as 8-byte words {32 data bits | 32-bit sequence number} (the idea of NCCL's
//     LL protocol) -- a word is valid the moment its sequence number matches;
//   * block 0's control warp gathers the 4-word partials of all blocks (one 16-byte-pair poll per block, 5 per lane),
//     reduces them in a fixed order and publishes the GPU total; with a shared-step group it pushes the total to every
//     peer's mailbox over NVLink instead, and EVERY block polls its own rank's mailbox (one hop after the push);
//   * every control warp then evaluates the (cheap, now low-latency) controller redundantly and bit-identically.
// ------------------------------------------------------------------------------------------------
struct FusedParams {
    b2ode_state *st;
    unsigned long long *part2;   // [2][gridDim.x][2] u64: 16-byte tagged block partials, double buffered by exchange parity
    unsigned *ctr;               // monotonically increasing arrival counter (zeroed by the host before the launch)
    const void *y0;
    void *out;
    // optional streaming of the solution to the host: `progress` counts output rows completed over all blocks, `host_mark`
    // (page-locked host memory, mapped) receives the number of leading rows that are complete on EVERY block, so that the
    // host can issue device-to-host copies behind the solve (b2ode_fused_desc.host_mark)
    unsigned *progress;
    int *host_mark;
    long long n_traj;       // trajectories on this rank
    int have_first_step;
    double t_start, first_step;
    double time_sign;       // -1 when integrating the reversed system (misc.py:318-321)
    double rhs[8];
    const void *rhs_data;   // device buffer of staged weights (RhsCubicMLP), else null
    // tableau (runtime values).  Structural zeros are multiplied like any other coefficient, as the reference does
    // (misc.py:114-121: its zero test never fires): x + 0 * k == x for finite k, so results equal the generic path's
    double beta[B2ODE_MAXK][B2ODE_MAXK];
    double c_sol[B2ODE_MAXK], c_error[B2ODE_MAXK], c_mid[B2ODE_MAXK];
    int fsal;
    double rtol0, atol0;
    CtrlParams c;
    CommParams comm;
};

__device__ __forceinline__ unsigned long long umax64(unsigned long long a, unsigned long long b) { return a > b ? a : b; }

// two 64-bit lanes of payload + one flag bit.  MODE 0: (a: sum >= 0, b: bit pattern of a non-negative double, combined
// with an unsigned max -- NaN patterns sort above +inf, so it is a NaN-propagating max for free); MODE 1: (a, b: sums)
template <int MODE>
__device__ __forceinline__ Pay pay_identity() {
    Pay r;
    r.a = 0.0;
    r.b = 0ull;       // +0.0 as a double, 0 as a max identity
    r.flag = 0u;
    return r;
}

template <int MODE>
__device__ __forceinline__ Pay pay_combine(const Pay &x, const Pay &y) {
    Pay r;
    r.a = x.a + y.a;
    if (MODE == 0) r.b = x.b > y.b ? x.b : y.b;
    else r.b = (unsigned long long)__double_as_longlong(__longlong_as_double((long long)x.b) + __longlong_as_double((long long)y.b));
    r.flag = x.flag | y.flag;
    return r;
}

template <int MODE>
__device__ __forceinline__ Pay pay_warp_reduce(Pay x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        Pay y;
        y.a = __shfl_xor_sync(0xffffffffu, x.a, o);
        y.b = __shfl_xor_sync(0xffffffffu, x.b, o);
        y.flag = __shfl_xor_sync(0xffffffffu, x.flag, o);
        x = pay_combine<MODE>(x, y);
    }
    return x;       // every lane holds the warp total (a + b == b + a bitwise, so all lanes agree)
}

// transport form: 4 words, the flag rides in the sign bit of `a` (a is a sum of squares: never negative; a NaN is made
// canonical first so that its sign bit is free too)
__device__ __forceinline__ void pay_pack(const Pay &x, unsigned seq, unsigned long long (&w)[4]) {
    unsigned long long ab = (unsigned long long)__double_as_longlong(x.a);
    if (x.a != x.a) ab = 0x7ff8000000000000ull;
    ab = (ab & 0x7fffffffffffffffull) | ((unsigned long long)(x.flag & 1u) << 63);
    const unsigned long long s = (unsigned long long)seq << 32;
    w[0] = s | (ab & 0xffffffffull);
    w[1] = s | (ab >> 32);
    w[2] = s | (x.b & 0xffffffffull);
    w[3] = s | (x.b >> 32);
}

__device__ __forceinline__ Pay pay_unpack(const unsigned long long (&w)[4]) {
    const unsigned long long ab = (w[0] & 0xffffffffull) | (w[1] << 32);
    Pay r;
    r.flag = (unsigned)(ab >> 63);
    r.a = __longlong_as_double((long long)(ab & 0x7fffffffffffffffull));
    r.b = (w[2] & 0xffffffffull) | (w[3] << 32);
    return r;
}

template <bool SYS>
__device__ __forceinline__ void ll_store4(unsigned long long *dst, const unsigned long long (&w)[4]) {
    if (SYS) {
        asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(dst), "l"(w[0]), "l"(w[1]) : "memory");
        asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(dst + 2), "l"(w[2]), "l"(w[3]) : "memory");
    } else {
        asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(dst), "l"(w[0]), "l"(w[1]) : "memory");
        asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(dst + 2), "l"(w[2]), "l"(w[3]) : "memory");
    }
}

// spin until all four words carry `seq`; every 8-byte word is written atomically, so each is checked on its own
template <bool SYS>
__device__ __forceinline__ Pay ll_wait4(const unsigned long long *src, unsigned seq) {
    unsigned long long w[4];
    for (;;) {
        if (SYS) {
            asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(w[0]), "=l"(w[1]) : "l"(src) : "memory");
            asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(w[2]), "=l"(w[3]) : "l"(src + 2) : "memory");
        } else {
            asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(w[0]), "=l"(w[1]) : "l"(src) : "memory");
            asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(w[2]), "=l"(w[3]) : "l"(src + 2) : "memory");
        }
        if ((unsigned)(w[0] >> 32) == seq && (unsigned)(w[1] >> 32) == seq && (unsigned)(w[2] >> 32) == seq &&
            (unsigned)(w[3] >> 32) == seq)
            break;
    }
    return pay_unpack(w);
}

__device__ __forceinline__ void named_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void named_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }

// The polls below use WEAK loads (ld.global.cg: they overlap; strong loads of one warp do not), and to the PTX memory
// model a weak load of an unchanged address may be assumed to return the same value again: ptxas is entitled to hoist such
// a load out of a polling loop, or to drop the loop ("it must terminate, so its condition holds") -- and does, once the loop
// is simple enough.  Every polling round therefore offsets its addresses by this value, which is always 0 but which ptxas
// cannot know: the loads are loop-variant and have to be issued again.
__device__ __forceinline__ unsigned long long opaque_zero() {
    unsigned long long c;
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(c));
    return c >> 63;
}

constexpr int kGatherPerLane = 5;        // 160 blocks gathered with every poll in flight (148 SMs x 1 block)

// shared scratch of one block
struct FusedShared {
    Pay part[16];                  // compute-warp partials
    unsigned long long rlane[B2ODE_MAXPEERS][32][2];   // per-lane sums of the OTHER ranks' partials (comm warp -> control warp)
    Pay tot;                       // totals of the initial-step reductions (read by every thread)
    struct {
        double dt_next;
        int accept, done;
        unsigned status;
    } ctl;                         // what the control warp hands to the compute warps
};

constexpr int kBarPartials = 1, kBarDecision = 2, kBarRows = 3, kBarRowsReady = 4, kBarRemote = 5;

// Called by the COMM warp (blocks of a shared-step group have one: a second service warp without trajectories): fetch the
// partials every peer wrote into this rank's mailbox over NVLink and leave, per source rank, each LANE's share (blocks
// lane, lane + 32, ... summed in that order) in shared memory; the control warp folds the ranks in rank order and does the
// one butterfly.  The comm warp starts polling the moment an exchange begins, so the peers' data is fetched while the
// control warp is still in the intra-GPU phase: the NVLink hop (~2070 cycles) hides behind it.  B2ODE_COMM_RG source ranks
// (three: 15 weak loads per lane) are polled together, round by round, until every partial carries the tag of `seq`.
template <int MODE>
__device__ __forceinline__ void remote_gather(const FusedParams &p, FusedShared &sh, unsigned seq) {
    const int nranks = p.comm.nranks, lane = threadIdx.x & 31, rank = p.comm.rank;
#ifndef B2ODE_COMM_RG
#define B2ODE_COMM_RG 3
#endif
    constexpr int RG = B2ODE_COMM_RG;                       // source ranks per batch
    constexpr int NL = RG * kGatherPerLane;                 // loads in flight per lane
    const unsigned long long *base = &p.comm.box[rank]->fused_part[seq & 1u][0][0][0] + (size_t)lane * 2;
    const unsigned tag = pay_tag(seq);
    for (int i0 = 0; i0 < nranks - 1; i0 += RG) {
        // The poll loop is INSTRUCTION bound (one warp, every load followed by its validation), so it is kept minimal: one
        // pointer per source rank, loads at immediate offsets and without predicates -- a slot past the source's grid, or
        // of a rank past the group, is just memory of the mailbox (fused_part has kMaxFusedBlocks >= 32 * kGatherPerLane
        // slots per rank) whose content is ignored -- and a two-instruction tag test per load.  Slots that were valid a
        // round ago stay valid (a buffer is rewritten two exchanges later), so every round simply reloads everything.
        unsigned long long g0[NL], g1[NL];
        const unsigned long long *ptr[RG];
        unsigned mine = 0u;
#pragma unroll
        for (int r = 0; r < RG; ++r) {
            const int i = i0 + r;
            const bool ok = i < nranks - 1;
            const int src = ok ? (i < rank ? i : i + 1) : rank;
            const int G = ok ? p.comm.grid_of[src] : 0;
            ptr[r] = base + (size_t)src * (kMaxFusedBlocks * 2);
            asm volatile("" : "+l"(ptr[r]));                 // (keep it in a register: do not recompute it per load)
#pragma unroll
            for (int q = 0; q < kGatherPerLane; ++q)
                if (lane + 32 * q < G) mine |= 1u << (r * kGatherPerLane + q);
        }
        unsigned got;
        do {
            const unsigned long long z = opaque_zero();
#pragma unroll
            for (int r = 0; r < RG; ++r)
#pragma unroll
                for (int q = 0; q < kGatherPerLane; ++q)
                    asm volatile("ld.global.cg.v2.u64 {%0, %1}, [%2];"
                                 : "=l"(g0[r * kGatherPerLane + q]), "=l"(g1[r * kGatherPerLane + q])
                                 : "l"(ptr[r] + z + 64 * q)
                                 : "memory");
            got = 0u;
#pragma unroll
            for (int k = 0; k < NL; ++k) {
                got |= (pay_mismatch(g0[k], g1[k], tag) == 0u) ? (1u << k) : 0u;
            }
        } while ((got & mine) != mine);
#pragma unroll
        for (int r = 0; r < RG; ++r) {
            const int i = i0 + r;
            if (i >= nranks - 1) continue;
            const int src = i < rank ? i : i + 1;
            Pay acc = pay_identity<MODE>();
#pragma unroll
            for (int q = 0; q < kGatherPerLane; ++q)
                if ((mine >> (r * kGatherPerLane + q)) & 1u)
                    acc = pay_combine<MODE>(acc, pay_unpack16(g0[r * kGatherPerLane + q], g1[r * kGatherPerLane + q]));   // fixed order
            const int G = p.comm.grid_of[src];
            for (int b = lane + 32 * kGatherPerLane; b < G; b += 32) {       // grids beyond 32 * kGatherPerLane blocks
                const unsigned long long *sl = base + (size_t)src * (kMaxFusedBlocks * 2) + (size_t)(b - lane) * 2;
                unsigned long long a0, a1;
                do {
                    asm volatile("ld.global.cg.v2.u64 {%0, %1}, [%2];" : "=l"(a0), "=l"(a1) : "l"(sl + opaque_zero()) : "memory");
                } while (!pay_valid16(a0, a1, seq));
                acc = pay_combine<MODE>(acc, pay_unpack16(a0, a1));
            }
#ifdef B2ODE_COMM_RTOT
            acc = pay_warp_reduce<MODE>(acc);                // A/B variant: the comm warp does one butterfly per source rank
#endif
            unsigned long long ab = (unsigned long long)__double_as_longlong(acc.a);
            if (acc.a != acc.a) ab = 0x7ff8000000000000ull;
            sh.rlane[src][lane][0] = (ab & 0x7fffffffffffffffull) | ((unsigned long long)(acc.flag & 1u) << 63);
            sh.rlane[src][lane][1] = acc.b;
        }
    }
    asm volatile("bar.arrive %0, %1;" ::"r"(kBarRemote), "r"(64) : "memory");
}

// Called by the CONTROL warp (all 32 lanes, convergent) once the compute warps' partials are in sh.part[0 .. ncw).
// `epoch` counts the exchanges of this launch (1, 2, ...).  Returns the group-wide totals in every lane of every block of
// every rank, bit-identical everywhere.
//
// What the microbenchmarks showed on B200 (scripts/micro/grid_barrier.cu, nvlink_pingpong.cu; profiles/r02_fused_exchange_ab.md):
//   * a gpu- or sys-scope STRONG load (ld.relaxed / acquire / volatile, atomic read) costs 500-700 cycles and the strong loads
//     of one warp do not overlap: a flag protocol that polls k words pays k round trips per poll; a leader gathering 147
//     messages with 5 polls per lane pays ~10 serialised round trips (7.3k cycles per all-reduce; two-level 13.4k);
//   * one atomic arrival counter + one polled word: 1.9k; weak ld.global.cg loads always read the L2 and pipeline;
//   * a fence (red.release) in front of the arrival costs a MEMBAR.GPU = the store's round trip;
//   * one NVLink hop (remote write -> visible to a poll of local memory) is ~2070 cycles whatever the instructions, +520 per
//     extra polled word; REMOTE atomics on one address serialise badly (147 blocks x 7 peers bumping per-source counters:
//     11.5 us per attempt at 8 GPUs against 4.2 us on one); an intra-GPU all-reduce followed by one message per peer puts
//     the hop behind the whole local phase (+3.1 us per attempt at 2 GPUs).
// Hence: every block stores its 16-byte tagged partial LOCALLY and, over NVLink, into EVERY peer's mailbox (plain stores: the
// tag validates the data, no flag, no remote atomic).  Inside the GPU one RELAXED arrival atomic orders nothing (no fence: a
// reader that finds a stale tag re-reads), lane 0 spins on the counter with one strong load per poll, then all partials
// are fetched with weak loads that overlap.  The peers' partials, which travel during the local phase, are gathered by a
// dedicated COMM warp (remote_gather) and handed to the control warp through shared memory; ranks combine in rank order.
template <int MODE>
__device__ __forceinline__ Pay control_allreduce(const FusedParams &p, FusedShared &sh, int ncw, unsigned epoch, unsigned seq0,
                                                 unsigned long long hw2 = 0ull /* Mailbox::fused_hw[0..1] at kernel start */,
                                                 int att = -1) {
    const int lane = threadIdx.x & 31;
    Pay x = (lane < ncw) ? sh.part[lane] : pay_identity<MODE>();
    x = pay_warp_reduce<MODE>(x);                                         // block total, all lanes
    FTRACE_DEP(att, 2, __double_as_longlong(x.a));
    const int nranks = p.comm.nranks > 1 ? p.comm.nranks : 1, rank = p.comm.rank;
    const int G = (int)gridDim.x;
    // buffer parity follows the PERSISTENT sequence number, so the alternation continues across launches: a rank that has
    // already started the next solve cannot overwrite a partial a slower rank has not read yet
    const unsigned seq = seq0 + epoch, par = seq & 1u;
    unsigned long long w0, w1;
    pay_pack16(x, seq, w0, w1);
    if (nranks > 1 && epoch <= 2u && lane < nranks && lane != rank) {
        // first use of this buffer in this solve: slots the previous writer of the buffer filled and this (smaller) grid does
        // not are poisoned in every peer's mailbox, so that no later solve can take them for fresh partials
        const int hw = (int)(par ? (unsigned)(hw2 >> 32) : (unsigned)hw2);
        for (int b = G + (int)blockIdx.x; b < hw && b < kMaxFusedBlocks; b += G) {
            unsigned long long *dst = &p.comm.box[lane]->fused_part[par][rank][b][0];
            asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(dst), "l"(kPoisonW0), "l"(kPoisonW1) : "memory");
        }
    }
    if (nranks > 1 && lane < nranks && lane != rank) {                    // lane q: this block's partial -> rank q, over NVLink
        unsigned long long *dst = &p.comm.box[lane]->fused_part[par][rank][blockIdx.x][0];
        asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(dst), "l"(w0), "l"(w1) : "memory");
    }
    if (G > 1) {
        unsigned long long *slots = p.part2 + (size_t)par * G * 2;
        if (lane == 0) {
            asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(slots + (size_t)blockIdx.x * 2), "l"(w0), "l"(w1) : "memory");
            asm volatile("red.relaxed.gpu.global.add.u32 [%0], 1;" ::"l"(p.ctr) : "memory");
            const unsigned target = epoch * (unsigned)G;
            unsigned v;
            do {
                asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p.ctr) : "memory");
            } while ((int)(v - target) < 0);
        }
        __syncwarp();
        FTRACE(att, 3);
        // this LANE's share of this GPU's partials (blocks lane, lane + 32, ...: fixed order).  All arrivals have been seen, so
        // the partials are almost always there: five unconditional weak loads in flight (a lane without a block at
        // lane + 32 q reads slot 0 and ignores it), then the tag test; a stale tag -- the relaxed arrival overtook its
        // data -- is re-read with strong loads, which the compiler may not hoist or elide.
        unsigned long long g0[kGatherPerLane], g1[kGatherPerLane];
#pragma unroll
        for (int q = 0; q < kGatherPerLane; ++q) {
            const int b = lane + 32 * q;
            asm volatile("ld.global.cg.v2.u64 {%0, %1}, [%2];" : "=l"(g0[q]), "=l"(g1[q]) : "l"(slots + (size_t)(b < G ? b : 0) * 2) : "memory");
        }
        x = pay_identity<MODE>();
#pragma unroll
        for (int q = 0; q < kGatherPerLane; ++q) {
            const int b = lane + 32 * q;
            if (b < G) {
                while (!pay_valid16(g0[q], g1[q], seq))
                    asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(g0[q]), "=l"(g1[q]) : "l"(slots + (size_t)b * 2) : "memory");
                x = pay_combine<MODE>(x, pay_unpack16(g0[q], g1[q]));
            }
        }
        for (int b = lane + 32 * kGatherPerLane; b < G; b += 32) {         // grids beyond 32 * kGatherPerLane blocks
            unsigned long long a0, a1;
            do {
                asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(a0), "=l"(a1) : "l"(slots + (size_t)b * 2) : "memory");
            } while (!pay_valid16(a0, a1, seq));
            x = pay_combine<MODE>(x, pay_unpack16(a0, a1));
        }
    } else {
        x = (lane == 0) ? pay_unpack16(w0, w1) : pay_identity<MODE>();   // (the transported form, like everybody else's)
    }
    if (nranks == 1) return pay_warp_reduce<MODE>(x);
#ifdef B2ODE_COMM_RTOT
    x = pay_warp_reduce<MODE>(x);
#endif
    asm volatile("bar.sync %0, %1;" ::"r"(kBarRemote), "r"(64) : "memory");                    // the comm warp has the peers' lane sums
    Pay tot = pay_identity<MODE>();
    for (int q = 0; q < nranks; ++q) {                                     // rank order, per lane: identical on every GPU
        Pay v = x;
        if (q != rank) {
            const unsigned long long a = sh.rlane[q][lane][0];
            v.flag = (unsigned)(a >> 63);
            v.a = __longlong_as_double((long long)(a & 0x7fffffffffffffffull));
            v.b = sh.rlane[q][lane][1];
        }
        tot = (q == 0) ? v : pay_combine<MODE>(tot, v);
    }
#ifdef B2ODE_COMM_RTOT
    return tot;
#else
    return pay_warp_reduce<MODE>(tot);                                     // one butterfly for the whole group
#endif
}

// The controller of the persistent kernel (one segment, the reference's controller: misc.py:250-287), written for the
// shortest dependent chain -- it sits on the critical path of every attempt with the whole GPU waiting:
//   accept  <=>  mean((err/tol)^2) <= 1  <=>  sum err^2 <= tol^2 * n         (no division; fp32 states compare in fp32,
//                                                                             i.e. against the largest double that rounds to 1.0f)
//   dt_next = dt / clamp(sqrt(m)^e / safety, 1/ifactor, 1/dfactor) = dt * clamp(safety * 2^(-e/2 * log2 m), dfactor', ifactor)
//   with log2 m = log2(sum err^2) - log2(tol^2 n): two independent logarithms, one exp2, no division, no sqrt.
// dt_next differs from the oracle's expression in the last ulps (an fp32 state: ~1e-7 relative, the oracle rounds sqrt(m)
// to fp32) -- dt is a free parameter of the method; the parity bars are on the solution (1e-6 / 1e-3).
// Called by all 32 lanes of the control warp, convergent (it shuffles).
template <typename T>
__device__ __forceinline__ CtrlDecision ctrl_fast(const CtrlParams &c, double ssq, double mm, bool bad0, double dt) {
    const T tol = Ar<T>::add((T)c.atol[0], Ar<T>::mul((T)c.rtol[0], (T)mm));
    const double tol2n = (double)tol * (double)tol * (double)c.n_global[0];
    const double bound = std::is_same<T, float>::value ? tol2n * (1.0 + 5.9604644775390625e-08) : tol2n;
    CtrlDecision d;
    d.bad0 = bad0;
    d.accept = ssq <= bound;
    {
        // the two logarithms are independent: lane 0 takes log2(ssq), the other lanes log2(tol2n) (one log2 on the chain)
        const double lg = log2(((threadIdx.x & 31) == 0) ? ssq : tol2n);
        const double L = __shfl_sync(0xffffffffu, lg, 0) - __shfl_sync(0xffffffffu, lg, 1);
        const double df = (ssq < tol2n) ? 1.0 : c.dfactor;
        const double rf = c.safety * exp2(-0.5 * c.exponent * L);
        d.dt_next = (ssq == 0.0) ? dt * c.ifactor : dt * nan_min(c.ifactor, nan_max(df, rf));
    }
    d.m = 0.0;       // filled in off the critical path
    return d;
}

// ------------------------------------------------------------------------------------------------
// the persistent solve.  Block = NCW compute warps (one trajectory per thread) + 1 control warp (the last one).
// ------------------------------------------------------------------------------------------------
template <typename T, typename RHS, int S, int MAXT>
__global__ void __launch_bounds__(MAXT) k_fused_adaptive(const __grid_constant__ FusedParams p) {
    using A = Ar<T>;
    constexpr int D = RHS::D;
    __shared__ FusedShared sh;
    __shared__ T sw[RHS::kSmem];
    constexpr int kDenseRows = (3 * (MAXT - 32) * D * (int)sizeof(T) + (int)sizeof(FusedShared) + RHS::kSmem * (int)sizeof(T) + 256 <= 48 * 1024) ? 3 : 2;
    __shared__ __align__(16) T s_rows[kDenseRows][(MAXT - 32) * D];     // dense-output rows of the step, waiting for the decision
    const int nthreads = blockDim.x;
    const bool grouped = p.comm.nranks > 1;
    const int nsvc = grouped ? 2 : 1;                    // service warps: control (+ comm with a shared-step group)
    const int ncw = (nthreads >> 5) - nsvc;              // compute warps
    const int nloc = 32 * (ncw + 1);                     // compute warps + control warp (barriers the comm warp is not part of)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool is_control = warp == ncw;
    // persistent exchange number of the cross-GPU receive area (it survives across solves in the mailbox)
    const unsigned ll_base = grouped ? (unsigned)p.comm.box[p.comm.rank]->ll_seq : 0u;
    const unsigned long long hw2 = (grouped && is_control) ? *(const volatile unsigned long long *)p.comm.box[p.comm.rank]->fused_hw : 0ull;
    if (RHS::kSmem > 1) {
        const int nw = (int)p.rhs[0] * 5 + 2;
        for (int q = threadIdx.x; q < nw && q < RHS::kSmem; q += nthreads) sw[q] = ((const T *)p.rhs_data)[q];
        __syncthreads();
    }
    const int n_out = p.c.n_out;
    const double *__restrict__ t_out = p.c.t_out;

    if (is_control) {
        // ================================ control warp =================================================
        unsigned epoch = 0;
        double t_cur = p.t_start, dt;
        unsigned status = 0;
        if (p.have_first_step) {
            dt = p.first_step;
        } else {
            // misc.py:226-247 with the two reductions of _select_initial_step
            named_sync(kBarPartials, nloc);
            Pay r = control_allreduce<1>(p, sh, ncw, ++epoch, ll_base, hw2);
            if (lane == 0) sh.tot = r;
            named_arrive(kBarDecision, nthreads);
            Partial tot;
            tot.v[0] = r.a;
            tot.v[1] = __longlong_as_double((long long)r.b);
            tot.v[2] = tot.v[3] = 0.0;
            T d1max;
            const T h0 = init_h0<T>(p.c, &tot, 1, &d1max);
            named_sync(kBarPartials, nloc);
            r = control_allreduce<1>(p, sh, ncw, ++epoch, ll_base, hw2);
            if (lane == 0) sh.tot = r;
            named_arrive(kBarDecision, nthreads);
            tot.v[0] = r.a;
            dt = (double)init_dt<T>(p.c, &tot, 1, h0, d1max);
        }
        int cur = 1;
        int done = (n_out <= 1) ? 1 : 0;
        if (!done && !(t_cur + dt > t_cur)) {
            status |= B2ODE_ST_UNDERFLOW;
            done = 1;
        }
        // bookkeeping for the final state
        int late_rows = 0;     // host streaming: rows of a long step whose completion is accounted one barrier later
        double m_last = 0.0, t_prev = t_cur, dt_last = 0.0;
        unsigned long long n_acc = 0, n_rej = 0;
        long long nadv = 0;
        int att = 0;
        while (!done) {
            FTRACE(att, 0);
            // everything that does not depend on the reduction, computed while the compute warps work
            const double t1_acc = t_cur + dt;
            int c2 = cur;
            while (c2 < n_out && __ldg(t_out + c2) <= t1_acc) ++c2;             // advance(): `while next_t > t1`
            if (c2 > cur) named_arrive(kBarRows, nloc);                    // the previous step's rows have been copied out
            named_sync(kBarPartials, nloc);                                // the compute warps' partials are in
            if (late_rows) {
                // a long step's extra rows were stored by the compute warps themselves, before this barrier
                __threadfence();
                if (lane == 0) {
                    const unsigned old = atomicAdd(p.progress, (unsigned)late_rows);
                    if (old + (unsigned)late_rows == (unsigned)(cur - 1) * gridDim.x) {
                        __threadfence_system();
                        *(volatile int *)p.host_mark = cur;
                    }
                }
                late_rows = 0;
            }
            FTRACE_DEP(att, 1, sh.part[0].flag);
            const Pay r = control_allreduce<0>(p, sh, ncw, ++epoch, ll_base, hw2, att);
            FTRACE_DEP(att, 4, __double_as_longlong(r.a));
            Partial tot;
            tot.v[0] = r.a;
            tot.v[1] = tot.v[2] = __longlong_as_double((long long)r.b);        // max(max|y0|, max|y1|)
            tot.v[3] = r.flag ? 1.0 : 0.0;                                      // inf or NaN somewhere in y0
            CtrlDecision dec = ctrl_fast<T>(p.c, tot.v[0], tot.v[1], r.flag != 0u, dt);
            unsigned st_bits = status;
            if (dec.bad0) st_bits |= B2ODE_ST_NONFINITE;
            const bool adv = dec.accept && !dec.bad0;
            const double t1n = dec.accept ? t1_acc : t_cur;
            const int c_new = adv ? c2 : cur;
            const long long nadv2 = (c_new > cur) ? 0 : nadv + 1;
            int dn = (c_new >= n_out) ? 1 : 0;
            if (!dn) {
                if (nadv2 >= p.c.max_num_steps) st_bits |= B2ODE_ST_MAXSTEPS;
                if (!(t1n + dec.dt_next > t1n)) st_bits |= B2ODE_ST_UNDERFLOW;
            }
            if (st_bits) dn = 1;
            if (lane == 0) {
                sh.ctl.dt_next = dec.dt_next;
                sh.ctl.accept = dec.accept ? 1 : 0;
                sh.ctl.done = dn;
                sh.ctl.status = st_bits;
            }
            named_arrive(kBarDecision, nthreads);
            FTRACE_DEP(att, 5, __double_as_longlong(dec.dt_next));
            if (c2 > cur) named_sync(kBarRowsReady, nloc);                  // the compute warps' rows are in shared memory
            if (adv && c2 > cur) {
                // The accepted step's dense-output rows wait in shared memory (written by the compute warps before the
                // decision barrier): this otherwise idle warp streams them to the solution slab with 16-byte stores while
                // the compute warps are already in the next attempt's stages.  The block's part of an output row is one
                // contiguous run of nblk * D elements.
                const long long first = (long long)blockIdx.x * (ncw * 32);
                long long nblk = p.n_traj - first;
                if (nblk > ncw * 32) nblk = ncw * 32;
                const int nel = (int)(nblk > 0 ? nblk * D : 0);
                const long long Nrow = p.n_traj * D;
                const int nrows = (c2 - cur) < kDenseRows ? (c2 - cur) : kDenseRows;
                for (int q = 0; q < nrows; ++q) {
                    T *row = (T *)p.out + (long long)(cur + q) * Nrow + first * D;
                    const T *src = s_rows[q];
                    constexpr int V = 16 / sizeof(T);
                    if ((reinterpret_cast<uintptr_t>(row) & 15u) == 0) {
                        const int nv = nel / V;
                        for (int e = lane; e < nv; e += 32)
                            reinterpret_cast<int4 *>(row)[e] = reinterpret_cast<const int4 *>(src)[e];
                        for (int e = nv * V + lane; e < nel; e += 32) row[e] = src[e];
                    } else {
                        for (int e = lane; e < nel; e += 32) row[e] = src[e];
                    }
                }
                if (p.host_mark) {
                    if (c2 - cur > kDenseRows) {
                        late_rows = c2 - cur;                       // compute warps are still writing rows: account later
                    } else {
                        __threadfence();                            // my rows are visible device-wide before the count moves
                        if (lane == 0) {
                            const unsigned old = atomicAdd(p.progress, (unsigned)(c2 - cur));
                            // rows 1 .. c2-1 complete on every block  <=>  the count reached (c2 - 1) * blocks
                            if (old + (unsigned)(c2 - cur) == (unsigned)(c2 - 1) * gridDim.x) {
                                __threadfence_system();
                                *(volatile int *)p.host_mark = c2;
                            }
                        }
                    }
                }
            }
            {   // the reported error ratio (b2ode_state.msr_max), off the critical path
                const T tol = Ar<T>::add((T)p.c.atol[0], Ar<T>::mul((T)p.c.rtol[0], (T)tot.v[1]));
                dec.m = (double)(T)(tot.v[0] / ((double)tol * (double)tol * (double)p.c.n_global[0]));
            }
            m_last = dec.m;
            dt_last = dt;
            if (dec.accept) {
                n_acc += 1;
                t_prev = t_cur;
                t_cur = t1n;
            } else {
                n_rej += 1;
            }
            cur = c_new;
            nadv = nadv2;
            dt = dec.dt_next;
            status = st_bits;
            done = dn;
            ++att;
        }
        if (blockIdx.x == 0 && lane == 0) {
            b2ode_state z;
            memset(&z, 0, sizeof(z));
            z.t0 = t_prev;
            z.t1 = t_cur;
            z.dt = dt;
            z.dt_last = dt_last;
            z.msr_max = m_last;
            z.n_acc = n_acc;
            z.n_rej = n_rej;
            z.attempt = n_acc + n_rej;
            z.n_steps_adv = nadv;
            z.done = 1;
            z.status = status;
            z.cursor = cur;
            z.xseq = p.st->xseq;
            *p.st = z;
        }
        if (blockIdx.x == 0 && grouped) {
            if (lane == 0) {
                Mailbox *mb = p.comm.box[p.comm.rank];
                mb->ll_seq = (unsigned long long)(ll_base + epoch);
                if (epoch >= 1u) mb->fused_hw[(ll_base + 1u) & 1u] = gridDim.x;     // what this solve left in each buffer
                if (epoch >= 2u) mb->fused_hw[(ll_base + 2u) & 1u] = gridDim.x;
            }
        }
        return;
    }

    if (warp == ncw + 1) {
        // ================================ comm warp (shared-step groups only) ===========================
        // mirrors the sequence of exchanges: per exchange, gather every peer's partials, then wait for the decision
        unsigned epoch = 0;
        double t_cur = p.t_start, dt;
        if (p.have_first_step) {
            dt = p.first_step;
        } else {
            remote_gather<1>(p, sh, ll_base + (++epoch));
            named_sync(kBarDecision, nthreads);
            Partial tot;
            tot.v[0] = sh.tot.a;
            tot.v[1] = __longlong_as_double((long long)sh.tot.b);
            tot.v[2] = tot.v[3] = 0.0;
            T d1max;
            const T h0 = init_h0<T>(p.c, &tot, 1, &d1max);
            remote_gather<1>(p, sh, ll_base + (++epoch));
            named_sync(kBarDecision, nthreads);
            tot.v[0] = sh.tot.a;
            dt = (double)init_dt<T>(p.c, &tot, 1, h0, d1max);
        }
        int done = (n_out <= 1) ? 1 : 0;
        if (!done && !(t_cur + dt > t_cur)) done = 1;
        while (!done) {
            remote_gather<0>(p, sh, ll_base + (++epoch));
            named_sync(kBarDecision, nthreads);
            done = sh.ctl.done;
        }
        return;
    }

    // ================================ compute warps ====================================================
    const long long i = (long long)blockIdx.x * (ncw * 32) + threadIdx.x;
    const bool live = i < p.n_traj;
    const long long N = p.n_traj * D;
    const T *y0g = (const T *)p.y0;
    T *out = (T *)p.out;
    const T tsign = (T)p.time_sign;
    T y[D], f0[D];
#pragma unroll
    for (int d = 0; d < D; ++d) y[d] = live ? y0g[i * D + d] : T(0);
    if (live) {
#pragma unroll
        for (int d = 0; d < D; ++d) out[i * D + d] = y[d];                 // solution[0] = y0 (solvers.py:29)
    }
    auto rhs = [&](T t, const T(&yy)[D], T(&dy)[D]) {
        // reverse-time wrapper of misc.py:318-321: f'(t, y) = -f(-t, y)
        if (tsign < T(0)) {
            RHS::eval(p.rhs, sw, -t, yy, dy);
#pragma unroll
            for (int d = 0; d < D; ++d) dy[d] = -dy[d];
        } else {
            RHS::eval(p.rhs, sw, t, yy, dy);
        }
    };
    // hand this warp's share to the control warp; do not wait
    unsigned xepoch = 0;              // exchanges so far (the control warp counts the same)
    auto contribute = [&](const Pay &mine, auto mode) {
        constexpr int MODE = decltype(mode)::value;
        const Pay w = pay_warp_reduce<MODE>(mine);
        if (lane == 0) sh.part[warp] = w;
        named_arrive(kBarPartials, nloc);
        ++xepoch;
    };
    double t_cur = p.t_start;
    rhs((T)t_cur, y, f0);                                                    // dopri5.py:71

    // ---- first step: given (dopri5.py:76) or _select_initial_step (misc.py:183-247) ----------------------
    double dt;
    if (p.have_first_step) {
        dt = p.first_step;
    } else {
        const T rtol = (T)p.rtol0, atol = (T)p.atol0;
        T scale[D];
        Pay mine = pay_identity<1>();
        double s0 = 0.0, s1 = 0.0;
#pragma unroll
        for (int d = 0; d < D; ++d) {
            scale[d] = A::add(atol, A::mul(A::abs(y[d]), rtol));
            if (live) {
                const double q0 = (double)A::div(y[d], scale[d]), q1 = (double)A::div(f0[d], scale[d]);
                s0 += q0 * q0;
                s1 += q1 * q1;
            }
        }
        mine.a = s0;
        mine.b = (unsigned long long)__double_as_longlong(s1);
        contribute(mine, IC<1>{});
        named_sync(kBarDecision, nthreads);
        Partial tot;
        tot.v[0] = sh.tot.a;
        tot.v[1] = __longlong_as_double((long long)sh.tot.b);
        tot.v[2] = tot.v[3] = 0.0;
        T d1max;
        const T h0 = init_h0<T>(p.c, &tot, 1, &d1max);
        T y1[D], f1[D];
#pragma unroll
        for (int d = 0; d < D; ++d) y1[d] = A::add(y[d], A::mul(h0, f0[d]));
        rhs(A::add((T)t_cur, h0), y1, f1);
        double s2 = 0.0;
        if (live) {
#pragma unroll
            for (int d = 0; d < D; ++d) {
                const double q = (double)A::div(A::sub(f1[d], f0[d]), scale[d]);
                s2 += q * q;
            }
        }
        mine.a = s2;
        mine.b = 0ull;
        contribute(mine, IC<1>{});
        named_sync(kBarDecision, nthreads);
        tot.v[0] = sh.tot.a;
        dt = (double)init_dt<T>(p.c, &tot, 1, h0, d1max);
    }
    int cur = 1;
    int done = (n_out <= 1) ? 1 : 0;
    if (!done && !(t_cur + dt > t_cur)) done = 1;

    // ---- attempts -------------------------------------------------------------------------------------
    int att = 0;
    while (!done) {
        const T t0c = (T)t_cur, dtc = (T)dt;                               // rk_common.py:45-46
        T k[S][D];
#pragma unroll
        for (int d = 0; d < D; ++d) k[0][d] = f0[d];
        T yi[D];
#pragma unroll
        for (int s = 0; s < S - 1; ++s) {
            const T ti = A::add(t0c, A::mul((T)p.c.alpha[s], dtc));
            T acc[D];
#pragma unroll
            for (int j = 0; j <= s; ++j) {
                const T c = A::mul(dtc, (T)p.beta[s][j]);                  // (scale * x), misc.py:121
#pragma unroll
                for (int d = 0; d < D; ++d) {
                    const T term = A::mul(c, k[j][d]);
                    acc[d] = (j == 0) ? term : A::add(acc[d], term);
                }
            }
#pragma unroll
            for (int d = 0; d < D; ++d) yi[d] = A::add(y[d], acc[d]);
            rhs(ti, yi, k[s + 1]);
        }
        if (!p.fsal) {                                                     // rk_common.py:54-56
            T acc[D];
#pragma unroll
            for (int j = 0; j < S; ++j) {
                const T c = A::mul(dtc, (T)p.c_sol[j]);
#pragma unroll
                for (int d = 0; d < D; ++d) {
                    const T term = A::mul(c, k[j][d]);
                    acc[d] = (j == 0) ? term : A::add(acc[d], term);
                }
            }
#pragma unroll
            for (int d = 0; d < D; ++d) yi[d] = A::add(y[d], acc[d]);
        }
        // error estimate + this thread's share of the reduction (rk_common.py:60, misc.py:256-263)
        {
            Pay mine = pay_identity<0>();
            T err[D];
#pragma unroll
            for (int j = 0; j < S; ++j) {
                const T c = A::mul(dtc, (T)p.c_error[j]);
#pragma unroll
                for (int d = 0; d < D; ++d) {
                    const T term = A::mul(c, k[j][d]);
                    err[d] = (j == 0) ? term : A::add(err[d], term);
                }
            }
            if (live) {
                double sum = 0.0;
                unsigned long long m0 = 0ull, m1 = 0ull;
#pragma unroll
                for (int d = 0; d < D; ++d) {
                    const double ed = (double)err[d];
                    sum += ed * ed;
                    m0 = umax64(m0, (unsigned long long)__double_as_longlong(fabs((double)y[d])));
                    m1 = umax64(m1, (unsigned long long)__double_as_longlong(fabs((double)yi[d])));
                }
                mine.a = sum;
                mine.b = umax64(m0, m1);
                mine.flag = (m0 >= 0x7ff0000000000000ull) ? 1u : 0u;     // inf or NaN in y0 (dopri5.py:100)
            }
            contribute(mine, IC<0>{});
        }
        FTRACE(att, 8);
        // ---- dense output (dopri5.py:39-45, interp.py:22-67): the VALUES of the first kDenseRows output rows of the step are
        // computed now, while the control warp runs the reduction (the arithmetic overlaps the exchange latency); they are
        // STORED only once the step is known to be accepted -- the stores then drain under the next attempt's stages instead
        // of queueing in front of the control warp's loads (measured: speculative stores tripled the exchange time)
        const double t1_acc = t_cur + dt;
        int c2 = cur;
        while (c2 < n_out && __ldg(t_out + c2) <= t1_acc) ++c2;                 // advance(): `while next_t > t1`
        const T t0s = t0c, t1s = (T)t1_acc;
        const T den = A::sub(t1s, t0s);
        auto fit = [&](T(&ca)[D], T(&cb)[D], T(&cc)[D], T(&cd)[D]) {
            const T m2dt = A::mul(T(-2), dtc), p2dt = A::mul(T(2), dtc), p5dt = A::mul(T(5), dtc);
            const T m3dt = A::mul(T(-3), dtc), m4dt = A::mul(T(-4), dtc);
            T ymid[D];
            {
                T acc[D];
#pragma unroll
                for (int j = 0; j < S; ++j) {
                    const T c = A::mul(dtc, (T)p.c_mid[j]);
#pragma unroll
                    for (int d = 0; d < D; ++d) {
                        const T term = A::mul(c, k[j][d]);
                        acc[d] = (j == 0) ? term : A::add(acc[d], term);
                    }
                }
#pragma unroll
                for (int d = 0; d < D; ++d) ymid[d] = A::add(y[d], acc[d]);
            }
#pragma unroll
            for (int d = 0; d < D; ++d) {
                const T f0e = k[0][d], f1e = k[S - 1][d], y0e = y[d], y1e = yi[d];
                T a = A::mul(m2dt, f0e);
                a = A::add(a, A::mul(p2dt, f1e));
                a = A::add(a, A::mul(T(-8), y0e));
                a = A::add(a, A::mul(T(-8), y1e));
                a = A::add(a, A::mul(T(16), ymid[d]));
                T b = A::mul(p5dt, f0e);
                b = A::add(b, A::mul(m3dt, f1e));
                b = A::add(b, A::mul(T(18), y0e));
                b = A::add(b, A::mul(T(14), y1e));
                b = A::add(b, A::mul(T(-32), ymid[d]));
                T cq = A::mul(m4dt, f0e);
                cq = A::add(cq, A::mul(dtc, f1e));
                cq = A::add(cq, A::mul(T(-11), y0e));
                cq = A::add(cq, A::mul(T(-5), y1e));
                cq = A::add(cq, A::mul(T(16), ymid[d]));
                ca[d] = a;
                cb[d] = b;
                cc[d] = cq;
                cd[d] = A::mul(dtc, f0e);
            }
        };
        auto eval_row = [&](int j, const T(&ca)[D], const T(&cb)[D], const T(&cc)[D], const T(&cd)[D], T(&r)[D]) {
            const T x = A::div(A::sub((T)__ldg(t_out + j), t0s), den);
            const T x2 = A::mul(x, x), x3 = A::mul(x2, x), x4 = A::mul(x3, x);
#pragma unroll
            for (int d = 0; d < D; ++d) {
                T v = A::mul(ca[d], x4);
                v = A::add(v, A::mul(cb[d], x3));
                v = A::add(v, A::mul(cc[d], x2));
                v = A::add(v, A::mul(cd[d], x));
                r[d] = A::add(v, y[d]);
            }
        };
        // the rows wait in shared memory, laid out exactly like the block's contiguous chunk of an output row
        const bool blk_out = c2 > cur;                                        // uniform over the grid
        if (blk_out) {
            named_sync(kBarRows, nloc);                                   // the control warp has copied the previous step's rows out
            if (live) {
                T ca[D], cb[D], cc[D], cd[D];
                fit(ca, cb, cc, cd);
#pragma unroll
                for (int q = 0; q < kDenseRows; ++q) {
                    if (cur + q < c2) {
                        T r[D];
                        eval_row(cur + q, ca, cb, cc, cd, r);
#pragma unroll
                        for (int d = 0; d < D; ++d) s_rows[q][threadIdx.x * D + d] = r[d];
                    }
                }
            }
        }
        if (blk_out) named_arrive(kBarRowsReady, nloc);                   // rows handed to the control warp
        FTRACE(att, 9);
        named_sync(kBarDecision, nthreads);                                 // the control warp's decision
        const bool accept = sh.ctl.accept != 0;
        FTRACE_DEP(att, 10, sh.ctl.accept);
        // state update (dopri5.py:113-120)
        if (accept) {
            if (blk_out) {
                if (cur + kDenseRows < c2 && live) {                         // long steps: the remaining rows, after the fact
                    T ca[D], cb[D], cc[D], cd[D];
                    fit(ca, cb, cc, cd);                                     // (recomputed: not kept live over the barrier)
                    for (int j = cur + kDenseRows; j < c2; ++j) {
                        T r[D];
                        eval_row(j, ca, cb, cc, cd, r);
                        T *row = out + (long long)j * N + i * D;
#pragma unroll
                        for (int d = 0; d < D; ++d) row[d] = r[d];
                    }
                }
            }
            t_cur = t1_acc;
            cur = c2;                     // (a non-finite y0 also sets `done`, so the cursor is moot in that case)
#pragma unroll
            for (int d = 0; d < D; ++d) {
                y[d] = yi[d];
                f0[d] = k[S - 1][d];
            }
        }
        dt = sh.ctl.dt_next;
        done = sh.ctl.done;
        ++att;
    }
}

// ================================================================================================
// host side
// ================================================================================================
// Block geometry: NCW compute warps + 1 control warp.  One block per SM when the batch allows it (fewest partials to
// gather, all 148 SMs busy): NCW = ceil(ceil(n / SMs) / 32), capped by the register budget of the instantiation; if
// that does not keep the batch co-resident, the largest block that does (smaller blocks can pack more warps per SM when
// the register file, not the block size, is the limit).  A pure function of (n, device, instantiation): every rank of a
// shared-step group computes the same geometry for every other rank's shard.
template <typename T, typename RHS, int S, int MAXT>
static int fused_geometry(long long n_traj, int nsm, int nsvc, int *ncw_out, int *grid_out) {
    const int kMaxNcw = MAXT / 32 - nsvc;
    long long per_block = (n_traj + nsm - 1) / nsm;
    int ncw = (int)((per_block + 31) / 32);
    if (ncw < 1) ncw = 1;
    if (ncw > kMaxNcw) ncw = kMaxNcw;
    for (; ncw >= 1; --ncw) {
        int per_sm = 0;
        const int grid = (int)((n_traj + (long long)ncw * 32 - 1) / ((long long)ncw * 32));
        B2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_fused_adaptive<T, RHS, S, MAXT>, 32 * (ncw + nsvc), 0));
        if (grid <= per_sm * nsm) {
            *ncw_out = ncw;
            *grid_out = grid;
            return 0;
        }
    }
    return b2_fail(B2ODE_ENOMEM, "batch of %lld trajectories cannot stay co-resident on %d SMs", n_traj, nsm);
}

// `capacity` != null: only report how many trajectories this instantiation can keep co-resident on the current device.
// n_traj_rank: trajectories of every rank of the group (null / ignored without a group).
template <typename T, typename RHS, int S, int MAXT>
static int fused_launch(const FusedParams &p_in, long long n_traj, cudaStream_t st, long long *capacity, const int64_t *n_traj_rank) {
    int dev = 0, coop = 0, nsm = 0, per_sm = 0;
    B2_CUDA(cudaGetDevice(&dev));
    B2_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
    B2_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
    if (capacity) {
        // (reported for the geometry with both service warps, so that a batch that fits alone also fits in a group)
        long long best = 0;
        for (int ncw = MAXT / 32 - 2; ncw >= 1 && coop; --ncw) {
            B2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_fused_adaptive<T, RHS, S, MAXT>, 32 * (ncw + 2), 0));
            const long long cap = (long long)per_sm * nsm * ncw * 32;
            if (cap > best) best = cap;
        }
        *capacity = best;
        return 0;
    }
    if (!coop) return b2_fail(B2ODE_ESTATE, "device does not support cooperative launch");
    FusedParams p = p_in;
    const int nsvc = p.comm.nranks > 1 ? 2 : 1;        // control warp (+ comm warp with a shared-step group)
    int ncw = 0, grid = 0;
    {
        const int rc = fused_geometry<T, RHS, S, MAXT>(n_traj, nsm, nsvc, &ncw, &grid);
        if (rc) return rc;
    }
    if (p.comm.nranks > 1) {
        for (int r = 0; r < p.comm.nranks; ++r) {
            int ncw_r = 0, grid_r = 0;
            const int rc = fused_geometry<T, RHS, S, MAXT>(n_traj_rank[r], nsm, nsvc, &ncw_r, &grid_r);
            if (rc) return rc;
            if (grid_r > kMaxFusedBlocks)
                return b2_fail(B2ODE_ENOMEM, "rank %d needs %d blocks, the group mailbox holds %d", r, grid_r, kMaxFusedBlocks);
            p.comm.grid_of[r] = grid_r;
        }
        if (p.comm.grid_of[p.comm.rank] != grid) return b2_fail(B2ODE_ESTATE, "inconsistent shard size for this rank");
    }
    void *args[] = {(void *)&p};
    const int slot = b2_timing_begin(6 /* B2_FAM_FUSED */, st);
    B2_CUDA(cudaLaunchCooperativeKernel((const void *)k_fused_adaptive<T, RHS, S, MAXT>, dim3(grid), dim3(32 * (ncw + nsvc)), args, 0, st));
    b2_timing_end(6, slot, st);
    b2_count_launch();
    return 0;
}

template <typename T, typename RHS>
static int fused_dispatch_s(const FusedParams &p, int n_k, long long n_traj, cudaStream_t st, long long *capacity,
                            const int64_t *ntr) {
    // up to 512 threads per block (<= 128 registers per thread) for the tableaus whose k-set fits; 256 otherwise
    switch (n_k) {
        case 2: return fused_launch<T, RHS, 2, 512>(p, n_traj, st, capacity, ntr);
        case 4: return fused_launch<T, RHS, 4, 512>(p, n_traj, st, capacity, ntr);
        case 7: return fused_launch<T, RHS, 7, 512>(p, n_traj, st, capacity, ntr);
        case 14: return fused_launch<T, RHS, 14, 256>(p, n_traj, st, capacity, ntr);
    }
    return b2_fail(B2ODE_EINVAL, "fused solve supports tableaus with 2, 4, 7 or 14 k's (got %d)", n_k);
}

template <typename T>
static int fused_dispatch_rhs(const FusedParams &p, int rhs_kind, int n_k, long long n_traj, cudaStream_t st,
                              long long *capacity = nullptr, const int64_t *ntr = nullptr) {
    switch (rhs_kind) {
        case B2ODE_RHS_LORENZ: return fused_dispatch_s<T, RhsLorenz<T>>(p, n_k, n_traj, st, capacity, ntr);
        case B2ODE_RHS_LOTKA_VOLTERRA: return fused_dispatch_s<T, RhsLotkaVolterra<T>>(p, n_k, n_traj, st, capacity, ntr);
        case B2ODE_RHS_CUBIC_MLP: return fused_dispatch_s<T, RhsCubicMLP<T>>(p, n_k, n_traj, st, capacity, ntr);
        case B2ODE_RHS_KEPLER: return fused_dispatch_s<T, RhsKepler<T>>(p, n_k, n_traj, st, capacity, ntr);
    }
    return b2_fail(B2ODE_EINVAL, "unknown built-in right-hand side %d", rhs_kind);
}

// Largest batch (trajectories on this device) b2ode_fused_solve can keep co-resident for this tableau / dtype / right-hand
// side: the host asks BEFORE launching, so that the shards of a shared-step group can agree on one path.  < 0: error.
extern "C" int64_t b2ode_fused_capacity(const b2ode_adaptive_desc *desc, int rhs_kind) {
    if (!desc) return b2_fail(B2ODE_EINVAL, "null argument");
    if (rhs_kind == B2ODE_RHS_LINEAR) return 0;     // a row of up to 128 values does not fit one thread's registers
    FusedParams p;
    memset(&p, 0, sizeof(p));
    long long cap = 0;
    int rc;
    if (desc->dtype == B2ODE_F64) rc = fused_dispatch_rhs<double>(p, rhs_kind, desc->n_k, 0, nullptr, &cap);
    else if (desc->dtype == B2ODE_F32) rc = fused_dispatch_rhs<float>(p, rhs_kind, desc->n_k, 0, nullptr, &cap);
    else return b2_fail(B2ODE_EINVAL, "dtype must be 0 or 1");
    if (rc) return rc < 0 ? rc : -rc;
    return (int64_t)cap;
}

static int rhs_dim(int kind) {
    return kind == B2ODE_RHS_LORENZ ? 3 : (kind == B2ODE_RHS_LOTKA_VOLTERRA || kind == B2ODE_RHS_CUBIC_MLP) ? 2 : kind == B2ODE_RHS_KEPLER ? 4 : -1;
}

static int rhs_check(int kind, const double *prm, int n_prm, const void *rhs_data) {
    if (kind == B2ODE_RHS_CUBIC_MLP) {
        if (n_prm < 2 || !rhs_data) return b2_fail(B2ODE_EINVAL, "cubic-MLP right-hand side needs {H, cube} and its weights");
        if (prm[0] < 1 || prm[0] > 128) return b2_fail(B2ODE_EINVAL, "cubic-MLP hidden width must be in [1, 128]");
    }
    return 0;
}

extern "C" size_t b2ode_fused_workspace_bytes(int64_t n_traj) {
    const long long grid_max = (n_traj + 31) / 32;       // the smallest block has one compute warp
    // [arrival counter, 128 B][row progress counter, 128 B][partials 2 x grid x 16 B (no shared-step group)]
    return (size_t)256 + (size_t)grid_max * 32;
}

extern "C" int b2ode_fused_solve(const b2ode_adaptive_desc *desc, const b2ode_fused_desc *f) {
    if (!desc || !f) return b2_fail(B2ODE_EINVAL, "null argument");
    if (!f->y0 || !f->out || !f->t_out || !f->state || !f->workspace) return b2_fail(B2ODE_EINVAL, "null buffer");
    const int rhs_kind = f->rhs_kind;
    if (rhs_kind == B2ODE_RHS_LINEAR) return b2_fail(B2ODE_EINVAL, "the linear right-hand side has no persistent kernel");
    const int D = rhs_dim(rhs_kind);
    if (D < 0) return b2_fail(B2ODE_EINVAL, "unknown built-in right-hand side %d", rhs_kind);
    if (desc->nseg != 1 || desc->seg_len[0] % D != 0) return b2_fail(B2ODE_EINVAL, "state must be one (B, %d) tensor", D);
    if (desc->dense_kind != 0) return b2_fail(B2ODE_EINVAL, "fused solve supports the quartic dense output only");
    if (f->n_rhs_params < 0 || f->n_rhs_params > 8) return b2_fail(B2ODE_EINVAL, "bad rhs params");
    const long long n_traj = desc->seg_len[0] / D;
    if (n_traj < 1) return b2_fail(B2ODE_EINVAL, "empty batch");
    if (f->workspace_bytes < b2ode_fused_workspace_bytes(n_traj)) return b2_fail(B2ODE_ENOMEM, "workspace too small");
    cudaStream_t st = (cudaStream_t)f->cuda_stream;
    unsigned char *w = (unsigned char *)f->workspace;
    if ((uintptr_t)w & 15u) return b2_fail(B2ODE_EINVAL, "workspace must be 16-byte aligned");
    const int nranks = f->nranks > 1 ? f->nranks : 1;
    FusedParams p;
    memset(&p, 0, sizeof(p));
    B2_CUDA(cudaMemsetAsync(w, 0, 256, st));
    p.progress = (unsigned *)(w + 128);
    p.host_mark = (int *)f->host_mark;
    p.st = (b2ode_state *)f->state;
    p.y0 = f->y0;
    p.out = f->out;
    p.n_traj = n_traj;
    p.have_first_step = (f->first_step == f->first_step) ? 1 : 0;
    p.t_start = f->t_start;
    p.first_step = f->first_step;
    p.time_sign = f->time_sign;
    for (int i = 0; i < f->n_rhs_params; ++i) p.rhs[i] = f->rhs_params[i];
    p.rhs_data = f->rhs_data;
    {
        const int rc_ = rhs_check(rhs_kind, f->rhs_params, f->n_rhs_params, f->rhs_data);
        if (rc_) return rc_;
    }
    const int nk = desc->n_k;
    for (int i = 0; i < B2ODE_MAXK; ++i) {
        for (int j = 0; j < B2ODE_MAXK; ++j) p.beta[i][j] = desc->beta[i][j];
        p.c_sol[i] = desc->c_sol[i];
        p.c_error[i] = desc->c_error[i];
        p.c_mid[i] = desc->c_mid[i];
        p.c.alpha[i] = desc->alpha[i];
    }
    p.fsal = desc->fsal;
    p.rtol0 = desc->rtol[0];
    p.atol0 = desc->atol[0];
    p.c.n_k = nk;
    p.c.controller = desc->controller;
    p.c.rtol[0] = desc->rtol[0];
    p.c.atol[0] = desc->atol[0];
    p.c.safety = desc->safety;
    p.c.ifactor = desc->ifactor;
    p.c.dfactor = desc->dfactor;
    p.c.exponent = desc->exponent;
    p.c.inv_safety = 1.0 / desc->safety;
    p.c.inv_ifactor = 1.0 / desc->ifactor;
    p.c.inv_dfactor = 1.0 / desc->dfactor;
    p.c.max_num_steps = desc->max_num_steps;
    p.c.init_order = desc->init_order;
    p.c.n_out = f->n_out;
    p.c.t_out = f->t_out;
    p.c.tstage = nullptr;
    long long n_glob = n_traj;
    p.comm.rank = 0;
    p.comm.nranks = 0;
    if (nranks > 1) {
        if (!f->mailboxes || nranks > B2ODE_MAXPEERS || f->rank < 0 || f->rank >= nranks) return b2_fail(B2ODE_EINVAL, "bad group arguments");
        n_glob = 0;
        for (int r = 0; r < nranks; ++r) {
            if (!f->mailboxes[r] || f->n_traj_rank[r] < 1) return b2_fail(B2ODE_EINVAL, "bad mailbox / shard size of rank %d", r);
            n_glob += f->n_traj_rank[r];
            p.comm.box[r] = (Mailbox *)f->mailboxes[r];
        }
        if (f->n_traj_rank[f->rank] != n_traj) return b2_fail(B2ODE_EINVAL, "n_traj_rank[rank] does not match the state");
        p.comm.rank = f->rank;
        p.comm.nranks = nranks;
    }
    // intra-GPU receive area = the caller's workspace: [arrival counter][row progress][partials 2 x grid x 16 B], zeroed per launch
    B2_CUDA(cudaMemsetAsync(w + 256, 0, b2ode_fused_workspace_bytes(n_traj) - 256, st));
    p.ctr = (unsigned *)w;
    p.part2 = (unsigned long long *)(w + 256);
    p.c.n_global[0] = n_glob * D;
    if (desc->dtype == B2ODE_F64) return fused_dispatch_rhs<double>(p, rhs_kind, nk, n_traj, st, nullptr, f->n_traj_rank);
    if (desc->dtype == B2ODE_F32) return fused_dispatch_rhs<float>(p, rhs_kind, nk, n_traj, st, nullptr, f->n_traj_rank);
    return b2_fail(B2ODE_EINVAL, "dtype must be 0 or 1");
}

// ================================================================================================
// fixed-grid methods with a built-in right-hand side: no step-size control, hence no reductions at all --
// every thread integrates its trajectory through the whole grid and writes its outputs
// (tfdiffeq/solvers.py:82-115, fixed_grid.py, rk_common.py:73-81; same operation order as k_fixed<T, OP>)
// ================================================================================================
struct FusedFixedParams {
    const void *y0;
    void *out;
    long long n_traj;
    int n_steps, n_out, method;     // method: 0 euler, 1 midpoint, 2 heun, 3 rk4 (3/8 rule)
    const void *times;              // [n_steps][4] stage times, state dtype
    const void *dts;                // [n_steps]
    const int *j0;                  // [n_steps + 1]: outputs inside cell i are [j0[i], j0[i+1])
    const unsigned char *ends;      // [n_steps]: the cell ends exactly on its last output
    const void *s1;                 // [n_steps]  t1 - t0
    const void *s2;                 // [n_out]    t_out[j] - t0 of its cell
    double time_sign;
    double rhs[8];
    const void *rhs_data;
};

template <typename T, typename RHS>
__global__ void __launch_bounds__(256) k_fused_fixed(const __grid_constant__ FusedFixedParams p) {
    using A = Ar<T>;
    constexpr int D = RHS::D;
    __shared__ T sw[RHS::kSmem];
    if (RHS::kSmem > 1) {
        const int nw = (int)p.rhs[0] * 5 + 2;
        for (int q = threadIdx.x; q < nw && q < RHS::kSmem; q += 256) sw[q] = ((const T *)p.rhs_data)[q];
        __syncthreads();
    }
    const T tsign = (T)p.time_sign;
    auto rhs = [&](T t, const T(&yy)[D], T(&dy)[D]) {
        if (tsign < T(0)) {
            RHS::eval(p.rhs, sw, -t, yy, dy);
#pragma unroll
            for (int d = 0; d < D; ++d) dy[d] = -dy[d];
        } else {
            RHS::eval(p.rhs, sw, t, yy, dy);
        }
    };
    const long long N = p.n_traj * D;
    const T *times = (const T *)p.times, *dts = (const T *)p.dts, *s1 = (const T *)p.s1, *s2 = (const T *)p.s2;
    T *out = (T *)p.out;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < p.n_traj; i += (long long)gridDim.x * 256) {
        T y[D];
#pragma unroll
        for (int d = 0; d < D; ++d) {
            y[d] = ((const T *)p.y0)[i * D + d];
            out[i * D + d] = y[d];
        }
        for (int s = 0; s < p.n_steps; ++s) {
            const T dt = dts[s];
            const T *tm = times + 4 * s;
            T y1[D], k1[D], k2[D], k3[D], k4[D], ys[D];
            rhs(tm[0], y, k1);
            if (p.method == 0) {
#pragma unroll
                for (int d = 0; d < D; ++d) y1[d] = A::add(y[d], A::mul(dt, k1[d]));                       // B2ODE_OP_EULER
            } else if (p.method == 1) {
#pragma unroll
                for (int d = 0; d < D; ++d) ys[d] = A::add(y[d], A::div(A::mul(k1[d], dt), T(2)));         // HALF_STEP
                rhs(tm[1], ys, k2);
#pragma unroll
                for (int d = 0; d < D; ++d) y1[d] = A::add(y[d], A::mul(dt, k2[d]));
            } else if (p.method == 2) {
#pragma unroll
                for (int d = 0; d < D; ++d) ys[d] = A::add(y[d], A::mul(dt, k1[d]));
                rhs(tm[1], ys, k2);
#pragma unroll
                for (int d = 0; d < D; ++d) y1[d] = A::add(y[d], A::mul(A::div(dt, T(2)), A::add(k1[d], k2[d])));   // HEUN_FINAL
            } else {
#pragma unroll
                for (int d = 0; d < D; ++d) ys[d] = A::add(y[d], A::div(A::mul(dt, k1[d]), T(3)));         // RK4_S2
                rhs(tm[1], ys, k2);
#pragma unroll
                for (int d = 0; d < D; ++d) ys[d] = A::add(y[d], A::mul(dt, A::add(A::div(k1[d], T(-3)), k2[d])));   // RK4_S3
                rhs(tm[2], ys, k3);
#pragma unroll
                for (int d = 0; d < D; ++d) ys[d] = A::add(y[d], A::mul(dt, A::add(A::sub(k1[d], k2[d]), k3[d])));   // RK4_S4
                rhs(tm[3], ys, k4);
#pragma unroll
                for (int d = 0; d < D; ++d)
                    y1[d] = A::add(y[d], A::mul(A::add(A::add(A::add(k1[d], A::mul(T(3), k2[d])), A::mul(T(3), k3[d])), k4[d]),
                                                A::div(dt, T(8))));                                          // RK4_FINAL
            }
            const int ja = p.j0[s], jb = p.j0[s + 1];
            for (int j = ja; j < jb; ++j) {
                T *row = out + (long long)j * N + i * D;
                if (j == jb - 1 && p.ends[s]) {
#pragma unroll
                    for (int d = 0; d < D; ++d) row[d] = y1[d];
                } else {
#pragma unroll
                    for (int d = 0; d < D; ++d) row[d] = A::add(y[d], A::mul(A::div(A::sub(y1[d], y[d]), s1[s]), s2[j]));   // LERP
                }
            }
#pragma unroll
            for (int d = 0; d < D; ++d) y[d] = y1[d];
        }
    }
}

template <typename T>
static int fused_fixed_dispatch(const FusedFixedParams &p, int rhs_kind, int sm_count, cudaStream_t st) {
    const long long blocks_needed = (p.n_traj + 255) / 256;
    const long long cap = (long long)(sm_count > 0 ? sm_count : 148) * 8;
    const int grid = (int)(blocks_needed < cap ? blocks_needed : cap);
    switch (rhs_kind) {
        case B2ODE_RHS_LORENZ: k_fused_fixed<T, RhsLorenz<T>><<<grid, 256, 0, st>>>(p); break;
        case B2ODE_RHS_LOTKA_VOLTERRA: k_fused_fixed<T, RhsLotkaVolterra<T>><<<grid, 256, 0, st>>>(p); break;
        case B2ODE_RHS_CUBIC_MLP: k_fused_fixed<T, RhsCubicMLP<T>><<<grid, 256, 0, st>>>(p); break;
        case B2ODE_RHS_KEPLER: k_fused_fixed<T, RhsKepler<T>><<<grid, 256, 0, st>>>(p); break;
        default: return b2_fail(B2ODE_EINVAL, "unknown built-in right-hand side %d", rhs_kind);
    }
    B2_CUDA(cudaGetLastError());
    b2_count_launch();
    return 0;
}

extern "C" int b2ode_fused_fixed_solve(int dtype, int method, int rhs_kind, const double *rhs_params, int n_rhs_params,
                                       const void *rhs_data, double time_sign, const void *y0, void *out, int64_t n_traj,
                                       int n_steps, int n_out, const void *times, const void *dts, const int32_t *j0,
                                       const unsigned char *ends, const void *s1, const void *s2, int sm_count,
                                       void *cuda_stream) {
    if (!y0 || !out || n_traj < 1 || n_out < 1 || n_steps < 0) return b2_fail(B2ODE_EINVAL, "bad arguments");
    if (n_steps > 0 && (!times || !dts || !j0 || !ends || !s1 || !s2)) return b2_fail(B2ODE_EINVAL, "null grid array");
    if (method < 0 || method > 3) return b2_fail(B2ODE_EINVAL, "method must be 0..3");
    if (rhs_kind == B2ODE_RHS_LINEAR) return b2_fail(B2ODE_EINVAL, "the linear right-hand side has no one-launch fixed-grid kernel");
    if (rhs_dim(rhs_kind) < 0) return b2_fail(B2ODE_EINVAL, "unknown built-in right-hand side %d", rhs_kind);
    if (n_rhs_params < 0 || n_rhs_params > 8 || (n_rhs_params && !rhs_params)) return b2_fail(B2ODE_EINVAL, "bad rhs params");
    const int rc = rhs_check(rhs_kind, rhs_params, n_rhs_params, rhs_data);
    if (rc) return rc;
    FusedFixedParams p;
    memset(&p, 0, sizeof(p));
    p.y0 = y0;
    p.out = out;
    p.n_traj = n_traj;
    p.n_steps = n_steps;
    p.n_out = n_out;
    p.method = method;
    p.times = times;
    p.dts = dts;
    p.j0 = j0;
    p.ends = ends;
    p.s1 = s1;
    p.s2 = s2;
    p.time_sign = time_sign;
    for (int i = 0; i < n_rhs_params; ++i) p.rhs[i] = rhs_params[i];
    p.rhs_data = rhs_data;
    if (dtype == B2ODE_F64) return fused_fixed_dispatch<double>(p, rhs_kind, sm_count, (cudaStream_t)cuda_stream);
    if (dtype == B2ODE_F32) return fused_fixed_dispatch<float>(p, rhs_kind, sm_count, (cudaStream_t)cuda_stream);
    return b2_fail(B2ODE_EINVAL, "dtype must be 0 or 1");
}
