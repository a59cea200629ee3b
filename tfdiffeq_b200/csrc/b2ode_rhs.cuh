// b2ode_rhs.cuh -- the library's built-in right-hand sides (tfdiffeq_b200/rhs.py), shared by the persistent fused kernels
// (b2ode_fused.cu) and the stage kernels with a fused right-hand side of the generic path (b2ode.cu).
#pragma once
#include "b2ode_dev.cuh"

// ------------------------------------------------------------------------------------------------
// built-in right-hand sides: explicit mul/add in the order of the torch expressions in rhs.py
// ------------------------------------------------------------------------------------------------
template <typename T>
struct RhsLorenz {   // examples/lorenz_attractor.py:20-37 ; params {sigma, beta, rho}
    static constexpr int D = 3;
    static constexpr int kSmem = 1;      // no staged weights
    static __device__ __forceinline__ void eval(const double *prm, const T * /*sw*/, T /*t*/, const T (&y)[3], T (&dy)[3]) {
        using A = Ar<T>;
        const T sigma = (T)prm[0], beta = (T)prm[1], rho = (T)prm[2];
        dy[0] = A::mul(sigma, A::sub(y[1], y[0]));                          // sigma * (y - x)
        dy[1] = A::sub(A::mul(y[0], A::sub(rho, y[2])), y[1]);              // x * (rho - z) - y
        dy[2] = A::sub(A::mul(y[0], y[1]), A::mul(beta, y[2]));             // x * y - beta * z
    }
};

template <typename T>
struct RhsLotkaVolterra {   // README.md:67-81 ; params {a, b, c, d}
    static constexpr int D = 2;
    static constexpr int kSmem = 1;
    static __device__ __forceinline__ void eval(const double *prm, const T * /*sw*/, T /*t*/, const T (&y)[2], T (&dy)[2]) {
        using A = Ar<T>;
        const T a = (T)prm[0], b = (T)prm[1], c = (T)prm[2], d = (T)prm[3];
        dy[0] = A::sub(A::mul(a, y[0]), A::mul(A::mul(b, y[0]), y[1]));     // a*x - b*x*z
        dy[1] = A::add(A::mul(-c, y[1]), A::mul(A::mul(d, y[0]), y[1]));    // -c*z + d*x*z
    }
};

// examples/ode_demo.py:115-129 (BASELINE config 3): W2 . tanh(W1 . y**3 + b1) + b2, 2 -> H -> 2, H <= 128.
// params {H, cube}; weights staged in shared memory, packed [W1 (2 x H) | b1 (H) | W2 (H x 2) | b2 (2)].
// torch evaluates the two products with cuBLAS (its own FMA order), so this right-hand side agrees with the
// module's forward to rounding, not bit for bit.
template <typename T>
struct RhsCubicMLP {
    static constexpr int D = 2;
    static constexpr int kMaxH = 128;
    static constexpr int kSmem = 2 * kMaxH + kMaxH + 2 * kMaxH + 2;
    static __device__ __forceinline__ void eval(const double *prm, const T *sw, T /*t*/, const T (&y)[2], T (&dy)[2]) {
        using A = Ar<T>;
        const int H = (int)prm[0];
        const bool cube = prm[1] != 0.0;
        const T u0 = cube ? A::mul(A::mul(y[0], y[0]), y[0]) : y[0];
        const T u1 = cube ? A::mul(A::mul(y[1], y[1]), y[1]) : y[1];
        const T *W1 = sw, *b1 = sw + 2 * H, *W2 = sw + 3 * H, *b2 = sw + 5 * H;
        T o0 = T(0), o1 = T(0);
        for (int h = 0; h < H; ++h) {
            const T a = A::add(A::add(A::mul(u0, W1[h]), A::mul(u1, W1[H + h])), b1[h]);
            const T z = act_dispatch(a);
            o0 = A::add(o0, A::mul(z, W2[2 * h]));
            o1 = A::add(o1, A::mul(z, W2[2 * h + 1]));
        }
        dy[0] = A::add(o0, b2[0]);
        dy[1] = A::add(o1, b2[1]);
    }
    static __device__ __forceinline__ float act_dispatch(float a) { return tanhf(a); }
    static __device__ __forceinline__ double act_dispatch(double a) { return tanh(a); }
};


// B2ODE_RHS_LINEAR (rhs.py's LinearSystem): k = s * (y @ A + b) on rows of D <= 128, with the stage combine fused in front of
// the GEMM (b2ode_linear.cu).  Rows do not fit one thread's registers, so this kind has its own kernel rather than an eval().
constexpr int kLinearMaxD = 128;
constexpr int kFamStageGemm = 7;   // B2_FAM_STAGE_GEMM: timing family of the linear stage kernel (b2ode.cu)
struct LinearStageArgs {
    const b2ode_state *st;
    const void *y0;
    const void *k[B2ODE_MAXK];
    double coef[B2ODE_MAXK];
    int nk;                      // stage terms, 0 = plain evaluation of y0
    void *ystage;                // optional: also store the stage input (the last stage's input is y1)
    void *k_out;
    long long rows;
    int D, has_bias;
    const void *data;            // A (D x D row-major), then b (D) if has_bias; state dtype
    double time_sign;
};
int b2_launch_stage_linear(int dtype, const LinearStageArgs &a, int sm_count, cudaStream_t st);

// DETEST class D (tests/DETEST/detest.py:263-283): a two-body orbit, state [x, y, vx, vy] per row; BASELINE config 5 stacks 32
// of them per batch row (dim 128), i.e. the (B, 128) state is (32 B) rows of 4.  r^3 = (x^2 + y^2)^1.5 like the torch module.
template <typename T>
struct RhsKepler {
    static constexpr int D = 4;
    static constexpr int kSmem = 1;
    static __device__ __forceinline__ void eval(const double * /*prm*/, const T * /*sw*/, T /*t*/, const T (&y)[4], T (&dy)[4]) {
        using A = Ar<T>;
        const T r2 = A::add(A::mul(y[0], y[0]), A::mul(y[1], y[1]));
        const T r3 = A::pow(r2, T(1.5));
        dy[0] = y[2];
        dy[1] = y[3];
        dy[2] = A::div(-y[0], r3);
        dy[3] = A::div(-y[1], r3);
    }
};
