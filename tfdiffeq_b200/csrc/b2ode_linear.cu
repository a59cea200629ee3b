// b2ode_linear.cu -- the linear built-in right-hand side k = s * (y @ A + b) (B2ODE_RHS_LINEAR, rhs.py's LinearSystem),
// evaluated inside the Runge-Kutta stage kernel on the fp64 tensor cores (DMMA, mma.sync m8n8k4 f64).
//
// One launch per stage i of an attempt on a (rows, D) state, 1 <= D <= 128:
//     y_i     = y0 + sum_j (dt * beta_ij) k_j      (rk_common.py:51; k_rk_stage's operations and order, bit for bit)
//     k_{i+1} = s * (y_i @ A + b)                  (s = time_sign: -1 is the reversed system of misc.py:318-321)
// The stage input is formed tile by tile in shared memory and is the GEMM's A-operand; it reaches HBM only for the last
// stage (it is y1 there: finalize, the dense output and the next commit read it).  NK = 0 is plain evaluation of an
// existing buffer (first derivative, initial-step probe, stage 0 after k_rk_stage0's commit).
//
// Layout (DESIGN.md 4.2 (c)): one persistent block per SM, 512 threads.  A (zero-padded to Dp = D rounded up to 8) stays
// in shared memory for the whole launch.  Warps 0-7 produce 32-row stage-input tiles into two shared buffers; warps 8-15
// multiply the other buffer by A and store k.  Named barriers hand the buffers back and forth, so the stream of the next
// tile overlaps the DMMA work of the current one.  The K dimension is accumulated in ascending order: deterministic.
// fp32 states take the same pipeline with fp32 FMAs on the CUDA cores (single-pass TF32 would miss fp32 accuracy).
#include "b2ode_rhs.cuh"

namespace {

constexpr int kLinThreads = 512;               // 8 producer + 8 consumer warps
constexpr int kLinTM = 32;                     // rows per stage-input tile
constexpr int kBarFull = 1, kBarEmpty = 3;     // named barriers 1,2 (buffer full) and 3,4 (buffer free); 0 is __syncthreads

struct LinGeom {
    int D, Dp, lda, ldy;
};

__host__ __device__ inline LinGeom lin_geom(int D) {
    LinGeom g;
    g.D = D;
    g.Dp = (D + 7) & ~7;
    g.lda = (g.Dp % 16 == 0) ? g.Dp + 8 : g.Dp;   // lda = 8 mod 16 doubles: a B fragment (4 k-rows x 8 cols) is 2 wavefronts
    g.ldy = g.Dp + 4;                              // ldy = 4 mod 8 doubles: an A fragment (8 rows x 4 k) is 2 wavefronts
    return g;
}

template <typename T>
size_t lin_smem_bytes(int D) {
    const LinGeom g = lin_geom(D);
    return sizeof(T) * ((size_t)g.Dp * g.lda + 2 * (size_t)kLinTM * g.ldy + g.Dp);
}

}  // namespace

template <int NK>
struct LinParams {
    const b2ode_state *st;
    const void *y0;
    const void *k[NK > 0 ? NK : 1];
    double coef[NK > 0 ? NK : 1];
    void *ystage;
    void *k_out;
    const void *A;               // D x D row-major, then b (D) if has_bias
    long long rows;
    int D, has_bias, vec_in, vec_out;
    double time_sign;
};

namespace {

__device__ __forceinline__ void bar_sync(int id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(kLinThreads) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(kLinThreads) : "memory"); }

__device__ __forceinline__ void dmma884(double (&c)[2], double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
        : "+d"(c[0]), "+d"(c[1])
        : "d"(a), "d"(b));
}

// Producer: the stage input of rows [r0, r0 + nr) into ys (row stride ldy), optionally also to ystage.  Flat over the
// tile's nr * D contiguous elements with 16-byte packs where every pointer allows it.
template <typename T, int NK>
__device__ __forceinline__ void produce_tile(const LinParams<NK> &p, const LinGeom &g, const T (&c)[NK > 0 ? NK : 1],
                                             T *ys, long long r0, int nr, int tid) {
    constexpr int V = 16 / sizeof(T);
    constexpr int U = NK <= 6 ? 2 : 1;        // packs in flight per thread (register budget of the 512-thread block)
    const long long base = r0 * g.D;
    const int n_el = nr * g.D;
    const T *y0 = (const T *)p.y0 + base;
    T *yst = p.ystage ? (T *)p.ystage + base : nullptr;
    auto put = [&](int e, T v) { ys[(e / g.D) * g.ldy + (e % g.D)] = v; };
    auto combine = [&](T y, const T (&kv)[NK > 0 ? NK : 1]) {
        if (NK == 0) return y;
        T acc = Ar<T>::mul(c[0], kv[0]);
#pragma unroll
        for (int j = 1; j < NK; ++j) acc = Ar<T>::add(acc, Ar<T>::mul(c[j], kv[j]));   // add_n, left to right
        return Ar<T>::add(y, acc);
    };
    int e0 = 0;
    if (p.vec_in) {
        const int np = n_el / V;
        for (int q0 = tid; q0 < np; q0 += 256 * U) {
            Pack<T, V> yv[U], kv[U][NK > 0 ? NK : 1];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int q = q0 + 256 * u;
                if (q < np) {
                    yv[u] = ld_pack<T, V>(y0, q);
#pragma unroll
                    for (int j = 0; j < NK; ++j) kv[u][j] = ld_pack<T, V>((const T *)p.k[j] + base, q);
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int q = q0 + 256 * u;
                if (q < np) {
                    Pack<T, V> o;
#pragma unroll
                    for (int v = 0; v < V; ++v) {
                        T kk[NK > 0 ? NK : 1];
#pragma unroll
                        for (int j = 0; j < NK; ++j) kk[j] = kv[u][j].v[v];
                        o.v[v] = combine(yv[u].v[v], kk);
                        put(q * V + v, o.v[v]);
                    }
                    if (NK > 0 && yst) st_pack<T, V>(yst, q, o);
                }
            }
        }
        e0 = np * V;
    }
    for (int e = e0 + tid; e < n_el; e += 256) {
        T kk[NK > 0 ? NK : 1];
#pragma unroll
        for (int j = 0; j < NK; ++j) kk[j] = ((const T *)p.k[j])[base + e];
        const T o = combine(y0[e], kk);
        put(e, o);
        if (NK > 0 && yst) yst[e] = o;
    }
}

// Consumer, fp64: k rows [r0, r0 + nr) = ys @ A on DMMA.  Warp w (0..7) owns m-tiles 2(w>>2), 2(w>>2)+1 (16 rows) and a
// quarter of the n-tiles (at most 4 of 16); per k-step: 2 A fragments + up to 4 B fragments for up to 8 DMMAs.
__device__ __forceinline__ void consume_tile(const LinGeom &g, const double *As, const double *ys, const double *bs,
                                             bool has_bias, double sgn, double *ko, long long r0, int nr, bool vec_out,
                                             int w, int lane) {
    const int NT = g.Dp / 8, NQ = (NT + 3) / 4;
    const int j0 = (w & 3) * NQ;
    const int nj = min(NQ, NT - j0);
    if (nj <= 0) return;
    const int mrow = 16 * (w >> 2);
    const int gr = lane >> 2, gc = lane & 3;
    double acc[2][4][2];
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[m][j][0] = acc[m][j][1] = 0.0;
    const double *ya = ys + (mrow + gr) * g.ldy + gc;
    const double *bb = As + gc * g.lda + j0 * 8 + gr;
#pragma unroll 2
    for (int k0 = 0; k0 < g.Dp; k0 += 4) {
        const double a0 = ya[k0], a1 = ya[8 * g.ldy + k0];
        const double *bk = bb + k0 * g.lda;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j < nj) {
                const double b = bk[8 * j];
                dmma884(acc[0][j], a0, b);
                dmma884(acc[1][j], a1, b);
            }
        }
    }
#pragma unroll
    for (int m = 0; m < 2; ++m) {
        const int rl = mrow + 8 * m + gr;
        if (rl >= nr) continue;
        double *orow = ko + (r0 + rl) * g.D;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j >= nj) continue;
            const int col = (j0 + j) * 8 + 2 * gc;
            double v[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                double x = acc[m][j][h];
                if (has_bias) x = Ar<double>::add(x, bs[col + h]);
                v[h] = sgn < 0.0 ? -x : x;
            }
            if (vec_out) {
                if (col < g.D) *reinterpret_cast<double2 *>(orow + col) = make_double2(v[0], v[1]);
            } else {
                if (col < g.D) orow[col] = v[0];
                if (col + 1 < g.D) orow[col + 1] = v[1];
            }
        }
    }
}

// Consumer, fp32: fp32 FMAs on the CUDA cores, ascending over K.  Warp w owns rows 4w..4w+3, lane the columns lane + 32 j.
__device__ __forceinline__ void consume_tile(const LinGeom &g, const float *As, const float *ys, const float *bs,
                                             bool has_bias, float sgn, float *ko, long long r0, int nr, bool /*vec_out*/,
                                             int w, int lane) {
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const float *yr = ys + 4 * w * g.ldy;
    for (int d = 0; d < g.D; ++d) {
        float yv[4], av[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) yv[i] = yr[i * g.ldy + d];
#pragma unroll
        for (int j = 0; j < 4; ++j) av[j] = (lane + 32 * j < g.D) ? As[d * g.lda + lane + 32 * j] : 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(yv[i], av[j], acc[i][j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int rl = 4 * w + i;
        if (rl >= nr) continue;
        float *orow = ko + (r0 + rl) * g.D;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int col = lane + 32 * j;
            if (col >= g.D) continue;
            float x = acc[i][j];
            if (has_bias) x = Ar<float>::add(x, bs[col]);
            orow[col] = sgn < 0.f ? -x : x;
        }
    }
}

}  // namespace

template <typename T, int NK>
__global__ void __launch_bounds__(kLinThreads, 1) k_rk_stage_linear(const __grid_constant__ LinParams<NK> p) {
    extern __shared__ __align__(16) unsigned char lin_smem[];
    const LinGeom g = lin_geom(p.D);
    T *As = reinterpret_cast<T *>(lin_smem);
    T *const ysb = As + g.Dp * g.lda;                 // two stage-input buffers of kLinTM x ldy
    T *const bs = ysb + 2 * kLinTM * g.ldy;
    const T *Ag = (const T *)p.A;
    // A zero-padded to Dp x lda, both stage-input buffers zeroed (their padding columns are never written again)
    for (int q = threadIdx.x; q < g.Dp * g.lda; q += kLinThreads) {
        const int d = q / g.lda, cc = q % g.lda;
        As[q] = (d < g.D && cc < g.D) ? Ag[d * g.D + cc] : T(0);
    }
    for (int q = threadIdx.x; q < 2 * kLinTM * g.ldy; q += kLinThreads) ysb[q] = T(0);
    for (int q = threadIdx.x; q < g.Dp; q += kLinThreads) bs[q] = (p.has_bias && q < g.D) ? Ag[g.D * g.D + q] : T(0);
    __syncthreads();

    const long long ntiles = (p.rows + kLinTM - 1) / kLinTM;
    const int mine = ntiles > blockIdx.x ? (int)((ntiles - 1 - blockIdx.x) / gridDim.x + 1) : 0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp < 8) {
        T c[NK > 0 ? NK : 1];
        if (NK > 0) {
            const T dt = (T)p.st->dt;
#pragma unroll
            for (int j = 0; j < NK; ++j) c[j] = Ar<T>::mul(dt, (T)p.coef[j]);   // (scale * x), misc.py:121
        }
        for (int it = 0; it < mine; ++it) {
            const int b = it & 1;
            const long long r0 = (blockIdx.x + (long long)it * gridDim.x) * kLinTM;
            const int nr = (int)min((long long)kLinTM, p.rows - r0);
            if (it >= 2) bar_sync(kBarEmpty + b);
            produce_tile<T, NK>(p, g, c, ysb + b * kLinTM * g.ldy, r0, nr, threadIdx.x);
            bar_arrive(kBarFull + b);
        }
    } else {
        const T sgn = (T)p.time_sign;
        for (int it = 0; it < mine; ++it) {
            const int b = it & 1;
            const long long r0 = (blockIdx.x + (long long)it * gridDim.x) * kLinTM;
            const int nr = (int)min((long long)kLinTM, p.rows - r0);
            bar_sync(kBarFull + b);
            consume_tile(g, As, ysb + b * kLinTM * g.ldy, bs, p.has_bias != 0, sgn, (T *)p.k_out, r0, nr, p.vec_out != 0, warp - 8, lane);
            if (it + 2 < mine) bar_arrive(kBarEmpty + b);
        }
    }
}

namespace {

bool aligned16p(const void *q) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & 15u) == 0; }

template <typename T, int NK>
int launch_linear(const LinearStageArgs &a, int sm_count, cudaStream_t st) {
    LinParams<NK> p;
    memset(&p, 0, sizeof(p));
    p.st = a.st;
    p.y0 = a.y0;
    bool vin = aligned16p(a.y0) && aligned16p(a.ystage);
    for (int j = 0; j < NK; ++j) {
        p.k[j] = a.k[j];
        p.coef[j] = a.coef[j];
        vin = vin && aligned16p(a.k[j]);
    }
    p.ystage = NK > 0 ? a.ystage : nullptr;
    p.k_out = a.k_out;
    p.A = a.data;
    p.rows = a.rows;
    p.D = a.D;
    p.has_bias = a.has_bias;
    p.vec_in = vin ? 1 : 0;
    p.vec_out = (aligned16p(a.k_out) && a.D % 2 == 0) ? 1 : 0;
    p.time_sign = a.time_sign;
    const size_t smem = lin_smem_bytes<T>(a.D);
    static unsigned attr_done = 0;    // per device: opt in to > 48 KB of dynamic shared memory once
    int dev = 0;
    B2_CUDA(cudaGetDevice(&dev));
    if (dev >= 32 || !((attr_done >> dev) & 1u)) {
        B2_CUDA(cudaFuncSetAttribute(k_rk_stage_linear<T, NK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)lin_smem_bytes<T>(kLinearMaxD)));
        if (dev < 32) attr_done |= 1u << dev;
    }
    const long long ntiles = (a.rows + kLinTM - 1) / kLinTM;
    const long long nsm = sm_count > 0 ? sm_count : 148;
    const int grid = (int)(ntiles < nsm ? ntiles : nsm);
    if (grid <= 0) return 0;
    // event timing (family B2_FAM_STAGE_GEMM) of eager launches only: events cannot be read back from a captured graph
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    B2_CUDA(cudaStreamIsCapturing(st, &cs));
    const int slot = cs == cudaStreamCaptureStatusNone ? b2_timing_begin(kFamStageGemm, st) : -1;
    k_rk_stage_linear<T, NK><<<grid, kLinThreads, smem, st>>>(p);
    B2_CUDA(cudaGetLastError());
    b2_timing_end(kFamStageGemm, slot, st);
    b2_count_launch();
    return 0;
}

template <typename T>
int dispatch_linear(const LinearStageArgs &a, int sm_count, cudaStream_t st) {
    switch (a.nk) {
#define B2_CASE(N) \
    case N:        \
        return launch_linear<T, N>(a, sm_count, st);
        B2_CASE(0) B2_CASE(1) B2_CASE(2) B2_CASE(3) B2_CASE(4) B2_CASE(5) B2_CASE(6) B2_CASE(7) B2_CASE(8) B2_CASE(9)
        B2_CASE(10) B2_CASE(11) B2_CASE(12) B2_CASE(13)
#undef B2_CASE
    }
    return b2_fail(B2ODE_EINVAL, "unsupported number of stage terms %d", a.nk);
}

}  // namespace

int b2_launch_stage_linear(int dtype, const LinearStageArgs &a, int sm_count, cudaStream_t st) {
    if (a.D < 1 || a.D > kLinearMaxD || !a.data || !a.y0 || !a.k_out) return b2_fail(B2ODE_EINVAL, "bad linear stage arguments");
    if (dtype == B2ODE_F64) return dispatch_linear<double>(a, sm_count, st);
    if (dtype == B2ODE_F32) return dispatch_linear<float>(a, sm_count, st);
    return b2_fail(B2ODE_EINVAL, "dtype must be 0 or 1");
}
