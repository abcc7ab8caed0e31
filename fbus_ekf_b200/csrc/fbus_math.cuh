// fbus_math.cuh -- per-filter math of the batched FBUS-EKF hot path (device inlines).
//
// One CUDA thread owns one filter.  The 18x18 covariance is kept PACKED-SYMMETRIC (171 doubles) in
// shared memory, laid out [element][thread] so that a warp touches 32 consecutive doubles per access;
// the nominal state (29 doubles) lives in registers.  All loops are compile-time unrolled: every
// shared-memory address is an immediate offset from one base register.
//
// The arithmetic exploits the structure the reference multiplies out densely:
//   F = I + N has six small non-zero blocks (filter.cpp:598-604); Gamma*Q*Gamma^T is diagonal
//   (filter.hpp:108-125); H has two non-zero block columns (filter.cpp:690-694).
// Results agree with the dense reference evaluation to rounding (~1e-16 relative), far inside the
// 1e-9 parity tolerance; see DESIGN.md for the derivations and tests/ for the parity checks.
//
// The header also compiles for the host (FBUS_HD expands to nothing without nvcc) -- used only by
// tests/host_math_harness.cpp to debug the math against the oracle on machines without a GPU.  The
// product never runs this code on the CPU.
#pragma once

#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define FBUS_HD __host__ __device__ __forceinline__
#define FBUS_UNROLL _Pragma("unroll")
#ifdef __CUDA_ARCH__
#define FBUS_FENCE asm volatile("" ::: "memory")
#else
#define FBUS_FENCE ((void)0)
#endif
#else
#define FBUS_FENCE ((void)0)
#define FBUS_HD inline
#define FBUS_UNROLL
#endif

// scheduling fences inside propagate_cov: level 2 = between every stage, 1 = between phases only, 0 = none
#ifndef FBUS_COV_FENCES
#define FBUS_COV_FENCES 2
#endif
#if FBUS_COV_FENCES >= 2
#define FBUS_FENCE_A FBUS_FENCE
#else
#define FBUS_FENCE_A ((void)0)
#endif
#if FBUS_COV_FENCES >= 1
#define FBUS_FENCE_B FBUS_FENCE
#else
#define FBUS_FENCE_B ((void)0)
#endif

namespace fbus {

constexpr int NX = 18;
constexpr int NPK = 171;
constexpr int MAXM = 16;  // marker-map capacity (FBUS_MAX_MARKERS)

// packed upper-triangular index of P(i,j)
FBUS_HD constexpr int pidx_u(int i, int j) { return i * NX - (i * (i - 1)) / 2 + (j - i); }
FBUS_HD constexpr int pidx(int i, int j) { return i <= j ? pidx_u(i, j) : pidx_u(j, i); }

// per-run constants (derived on the host from fbus_config; passed by value as a kernel parameter)
struct MarkerConst {
    double p[3];    // positionAtG
    double q[4];    // quaternionM2G = Quaterniond(rotation), main.cpp:201
    double CM[16];  // R(Q_M) * L(Q_IL) * L2   (constant factor of H[3:7,6:9], filter.cpp:693-694)
    int32_t id;
    int32_t pad;
};
struct DevConsts {
    double R_IL[9], Q_IL[4], P_IL[3];  // filter view: T_C_I * T_SC_left (filter.hpp:67-69)
    double Qd[4];                      // accel_n, gyro_n, accel_b, gyro_b covariances
    double Rp, Rq;                     // pos / quat measurement covariances
    double max_dist, switch_thres, reset_gap;
    double R_RL[9], P_LR[3];           // vision view: raw T_SC (vision.cpp:476-481)
    double a0, a1;                     // n_air/n_glass, n_glass/n_water
    double d_air, d_glass, normal[3], dect_thres;
    double rod_s, rod_c;               // sin/cos of -3.1415926/4 (common.hpp:14, vision.cpp:740)
    double cam_k[2][4], cam_d[2][4];   // fisheye intrinsics (fx fy cx cy) and Kannala-Brandt coefficients, left / right
    double T_LR_air[12];               // in-air stereo: [R_IR R_IL^T | P_LI - R P_RI], row-major 3x4 (vision.cpp:402-408)
    int32_t air_lt_glass, glass_gt_water;
    int32_t n_markers, flags;
    double imu_g;                      // IMUInfo.g: scale of float32 sensor accelerations (main.cpp:252-254)
};
// marker map: lives in device global memory (dynamic indexing of kernel parameters would force a
// local-memory copy of the whole table)
struct MarkerTable {
    MarkerConst mk[MAXM];
};

// nominal state held in registers (NominalState, common.hpp:205-225)
struct Nominal {
    double t, q[4], R[9], p[3], v[3], ba[3], bg[3], g[3];
};

// ------------------------------------------------------------------------------------------------
// quaternion / rotation device inlines (matrix_math.hpp + the Eigen rules of SURVEY A.1)
// ------------------------------------------------------------------------------------------------
FBUS_HD void qmul(const double* a, const double* b, double* o) {
    const double w = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3];
    const double x = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2];
    const double y = a[0] * b[2] + a[2] * b[0] + a[3] * b[1] - a[1] * b[3];
    const double z = a[0] * b[3] + a[3] * b[0] + a[1] * b[2] - a[2] * b[1];
    o[0] = w; o[1] = x; o[2] = y; o[3] = z;
}
FBUS_HD void qmul_conjb(const double* a, const double* b, double* o) {  // a * conj(b)
    const double bb[4] = {b[0], -b[1], -b[2], -b[3]};
    qmul(a, bb, o);
}
// reciprocal square root: one MUFU.RSQ64H + Newton steps on the device (1-2 ulp) instead of a correctly rounded
// sqrt followed by a correctly rounded division (~4x the instructions); the host build keeps 1/sqrt
// Device versions are call-free on purpose (hardware seed + Newton steps, no out-of-line slow path: fewer instructions and
// nothing for the register allocator to save around a call).  Arguments on these paths are far inside the normal range;
// 0 gives NaN (the callers treat 0 separately or want it).
FBUS_HD double rsqrt_d(double x) {
#ifdef __CUDA_ARCH__
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double hx = 0.5 * x;
    y = fma(y, fma(-hx * y, y, 0.5), y);  // y += y (1/2 - x y^2 / 2)
    y = fma(y, fma(-hx * y, y, 0.5), y);
    return y;
#else
    return 1.0 / sqrt(x);
#endif
}
// one Newton step only: relative error ~1e-13, for iterations that correct themselves (the inner Newton of the GN projection)
FBUS_HD double rsqrt_d1(double x) {
#ifdef __CUDA_ARCH__
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    return fma(y, fma(-0.5 * x * y, y, 0.5), y);
#else
    return 1.0 / sqrt(x);
#endif
}
// sqrt to ~1 ulp: x * rsqrt(x), exactly 0 at 0
FBUS_HD double sqrt_d(double x) {
#ifdef __CUDA_ARCH__
    return x > 0.0 ? x * rsqrt_d(x) : (x == 0.0 ? 0.0 : x * rsqrt_d(x));
#else
    return sqrt(x);
#endif
}
// sin and cos together, call-free: two-term Cody-Waite reduction by pi/2 with FMA (exact enough for |x| < ~1e5; the angles
// here are half rotation increments, << 1) and the fdlibm kernel polynomials on [-pi/4, pi/4] (< 1 ulp)
FBUS_HD void sincos_d(double x, double* sn, double* cs) {
#ifdef __CUDA_ARCH__
    const double kf = rint(x * 0.63661977236758138);  // 2/pi
    double r = fma(-kf, 1.5707963267948966, x);
    r = fma(-kf, 6.123233995736766e-17, r);
    const double z = r * r;
    double ps = 1.58969099521155010221e-10;
    ps = fma(ps, z, -2.50507602534068634195e-08);
    ps = fma(ps, z, 2.75573137070700676789e-06);
    ps = fma(ps, z, -1.98412698298579493134e-04);
    ps = fma(ps, z, 8.33333333332248946124e-03);
    ps = fma(ps, z, -1.66666666666666324348e-01);
    const double s0 = fma(r * z, ps, r);
    double pc = -1.13596475577881948265e-11;
    pc = fma(pc, z, 2.08757232129817482790e-09);
    pc = fma(pc, z, -2.75573143513906633035e-07);
    pc = fma(pc, z, 2.48015872894767294178e-05);
    pc = fma(pc, z, -1.38888888888741095749e-03);
    pc = fma(pc, z, 4.16666666666666019037e-02);
    const double c0 = fma(z * z, pc, fma(-0.5, z, 1.0));
    const int q = (int)kf & 3;
    const double sv = (q & 1) ? c0 : s0, cv = (q & 1) ? s0 : c0;
    *sn = (q & 2) ? -sv : sv;
    *cs = ((q + 1) & 2) ? -cv : cv;
#else
    *sn = sin(x);
    *cs = cos(x);
#endif
}
// reciprocal: hardware seed (~20 bits) + two Newton steps (~1 ulp), without the slow-path call of a correctly rounded
// division; arguments here are well inside the normal range
FBUS_HD double rcp_d(double x) {
#ifdef __CUDA_ARCH__
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(fma(-x, r, 1.0), r, r);
    r = fma(fma(-x, r, 1.0), r, r);
    return r;
#else
    return 1.0 / x;
#endif
}
FBUS_HD void qnormalize(double* q) {
    const double inv = rsqrt_d(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    q[0] *= inv; q[1] *= inv; q[2] *= inv; q[3] *= inv;
}
// An expression like  t1*x - t2*w  has two products, and the compiler may contract either into the FMA: which one it picks can differ
// between two instantiations of the same kernel (it did: the float32-sensor and the double instantiation of the lane kernel rounded
// R(q) differently in the last bit, and the bitwise tests between the two element formats caught it).  Where a sum has more than one
// product the pairing is therefore written out: FBUS_PROD is a product rounded on its own, the other one goes into an explicit fma.
#ifdef __CUDA_ARCH__
#define FBUS_PROD(a, b) __dmul_rn((a), (b))
#else
#define FBUS_PROD(a, b) ((a) * (b))
#endif
FBUS_HD void q2R(const double* q, double* R) {  // Eigen toRotationMatrix, literal also for non-unit q
    const double w = q[0], x = q[1], y = q[2], z = q[3];
    const double tx = 2 * x, ty = 2 * y, tz = 2 * z;
    const double twx = FBUS_PROD(tx, w), twy = FBUS_PROD(ty, w), twz = FBUS_PROD(tz, w);
    const double tyy = FBUS_PROD(ty, y), tzz = FBUS_PROD(tz, z);
    R[0] = 1 - fma(ty, y, tzz);  R[1] = fma(ty, x, -twz);     R[2] = fma(tz, x, twy);
    R[3] = fma(ty, x, twz);      R[4] = 1 - fma(tx, x, tzz);  R[5] = fma(tz, y, -twx);
    R[6] = fma(tz, x, -twy);     R[7] = fma(tz, y, twx);      R[8] = 1 - fma(tx, x, tyy);
}
FBUS_HD void R2q(const double* m, double* q) {  // Eigen Quaterniond(Matrix3d), not normalised
    double t = m[0] + m[4] + m[8];
    if (t > 0) {
        t = sqrt(t + 1.0);
        q[0] = 0.5 * t;
        t = 0.5 / t;
        q[1] = (m[7] - m[5]) * t;
        q[2] = (m[2] - m[6]) * t;
        q[3] = (m[3] - m[1]) * t;
    } else {
        // branch-per-case keeps every index static (no local-memory arrays on the device)
        if (m[0] >= m[4] && m[0] >= m[8]) {  // i=0,j=1,k=2   (ties -> lowest index, as Eigen)
            t = sqrt(m[0] - m[4] - m[8] + 1.0);
            q[1] = 0.5 * t; t = 0.5 / t;
            q[0] = (m[7] - m[5]) * t; q[2] = (m[3] + m[1]) * t; q[3] = (m[6] + m[2]) * t;
        } else if (m[4] > m[0] && m[4] >= m[8]) {  // i=1,j=2,k=0
            t = sqrt(m[4] - m[8] - m[0] + 1.0);
            q[2] = 0.5 * t; t = 0.5 / t;
            q[0] = (m[2] - m[6]) * t; q[3] = (m[7] + m[5]) * t; q[1] = (m[1] + m[3]) * t;
        } else {  // i=2,j=0,k=1
            t = sqrt(m[8] - m[0] - m[4] + 1.0);
            q[3] = 0.5 * t; t = 0.5 / t;
            q[0] = (m[3] - m[1]) * t; q[1] = (m[2] + m[6]) * t; q[2] = (m[5] + m[7]) * t;
        }
    }
}
FBUS_HD void mat3_vec(const double* M, const double* v, double* o) {
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i) o[i] = M[i * 3] * v[0] + M[i * 3 + 1] * v[1] + M[i * 3 + 2] * v[2];
}
FBUS_HD void mat3t_vec(const double* M, const double* v, double* o) {  // M^T v
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i) o[i] = M[i] * v[0] + M[3 + i] * v[1] + M[6 + i] * v[2];
}
FBUS_HD double norm3(const double* v) { return sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); }

// ------------------------------------------------------------------------------------------------
// covariance accessor: packed symmetric storage with element stride S (S = block size in shared
// memory on the device, 1 on the host harness)
// ------------------------------------------------------------------------------------------------
// TLR = true: the top-left 9x9 block (rows/cols 0..8: p, v, theta) lives in the caller's registers TL[45] (packed by
// tlidx) instead of in the strided array; every index is a compile-time constant after unrolling, so the choice is static.
FBUS_HD constexpr int tlidx(int i, int j) {
    return (i <= j) ? (i * 9 - (i * (i - 1)) / 2 + (j - i)) : (j * 9 - (j * (j - 1)) / 2 + (i - j));
}
template <int S, bool TLR = false>
struct CovX {
    static constexpr bool kTLR = TLR;
    static constexpr bool kBlocked = false;  // element access is as cheap as block access
    double* s;
    double* TL = nullptr;
    FBUS_HD void fence_st() const {}  // accessors with asynchronous stores (tensor memory) order them here
    // asynchronous-load API of the tensor-memory accessor (fbus_tmem.cuh); plain loads here
    FBUS_HD void ldblk_nw(int bi, int bj, double* X) const { ldany(bi, bj, X); }
    // cross blocks of rows 1, 2 (bi in {1,2}, k in 3..5)
    FBUS_HD void ldtr_nw(int bi, int k, double* X, bool) const { ldany(bi, k, X); }
    FBUS_HD void sttr(int bi, int k, const double* X) const { stblk(bi, k, X); }
    FBUS_HD void wait_ld() const {}
    FBUS_HD void fix(int, int, double*) const {}
    FBUS_HD double ld(int i, int j) const {
        if (TLR && i < 9 && j < 9) return TL[tlidx(i, j)];
        return s[pidx(i, j) * S];
    }
    FBUS_HD void st(int i, int j, double v) const {
        if (TLR && i < 9 && j < 9) TL[tlidx(i, j)] = v;
        else s[pidx(i, j) * S] = v;
    }
    // X[r*3+c] = P[3bi+r][3bj+c]  (off-diagonal block, any order of bi,bj)
    FBUS_HD void ldblk(int bi, int bj, double* X) const {
        FBUS_UNROLL
        for (int r = 0; r < 3; ++r)
            FBUS_UNROLL
            for (int c = 0; c < 3; ++c) X[r * 3 + c] = ld(3 * bi + r, 3 * bj + c);
    }
    // diagonal block expanded to a full symmetric 3x3 (6 loads)
    FBUS_HD void lddiag(int b, double* X) const {
        FBUS_UNROLL
        for (int r = 0; r < 3; ++r)
            FBUS_UNROLL
            for (int c = r; c < 3; ++c) {
                const double v = ld(3 * b + r, 3 * b + c);
                X[r * 3 + c] = v;
                X[c * 3 + r] = v;
            }
    }
    FBUS_HD void ldany(int bi, int bj, double* X) const {
        if (bi == bj) lddiag(bi, X);
        else ldblk(bi, bj, X);
    }
    FBUS_HD void stblk(int bi, int bj, const double* X) const {  // bi < bj
        FBUS_UNROLL
        for (int r = 0; r < 3; ++r)
            FBUS_UNROLL
            for (int c = 0; c < 3; ++c) st(3 * bi + r, 3 * bj + c, X[r * 3 + c]);
    }
    FBUS_HD void stdiag(int b, const double* X) const {  // upper 6 of X
        FBUS_UNROLL
        for (int r = 0; r < 3; ++r)
            FBUS_UNROLL
            for (int c = r; c < 3; ++c) st(3 * b + r, 3 * b + c, X[r * 3 + c]);
    }
};
template <int S>
using Cov = CovX<S, false>;

// ------------------------------------------------------------------------------------------------
// F1: covariance propagation  P <- F P F^T + diag(Qbar)   (FILTER::UpdateCovariance, filter.cpp:588-616)
//
// F = E2*E1*E0 with block-row operations
//   row0 += dt*row1 ;  row1 += A*row2 + B*row3 + dt*row5 ;  row2 <- (I+Wm)*row2 - dt*row4
//   A = -R*[a]x*dt,  B = -R*dt,  Wm = -[w]x*dt     (R = CARRIED rotmatI2G, a/w bias-corrected)
// Only the 126 entries of block rows 0..2 change; rows 3..5 (b_a, b_g, g) only receive Qbar.
// Evaluation: (1) top-left 3x3 blocks from OLD values, (2) block columns 4,3,5 of rows 0..2, folding
// their contribution into the top-left accumulators.  ~650 FMA instead of the 2*18^3 dense product.
// ------------------------------------------------------------------------------------------------
constexpr int NTL = 45;  // packed size of the top-left 9x9 (tlidx)
template <int S, class CV = Cov<S>>
FBUS_HD void tl_load(const CV P, double* TL) {
    FBUS_UNROLL
    for (int i = 0; i < 9; ++i)
        FBUS_UNROLL
        for (int j = i; j < 9; ++j) TL[tlidx(i, j)] = P.ld(i, j);
}
template <int S, class CV = Cov<S>>
FBUS_HD void tl_store(const CV P, const double* TL) {
    FBUS_UNROLL
    for (int i = 0; i < 9; ++i)
        FBUS_UNROLL
        for (int j = i; j < 9; ++j) P.st(i, j, TL[tlidx(i, j)]);
}
// coefficients of F for one IMU sample: A = -R*[a]x*dt, B = -R*dt (row-major 3x3), u = w*dt
FBUS_HD void cov_coeffs(const double* R, const double* acc, const double* w, double dt, double* A, double* B, double* u) {
    const double ndt = -dt;
    const double s0 = acc[0] * ndt, s1 = acc[1] * ndt, s2 = acc[2] * ndt;  // -dt * a
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i) {
        // (R * [v]x)[i][:] = (R[i][1]v2 - R[i][2]v1, R[i][2]v0 - R[i][0]v2, R[i][0]v1 - R[i][1]v0)
        A[i * 3 + 0] = fma(R[i * 3 + 1], s2, -FBUS_PROD(R[i * 3 + 2], s1));
        A[i * 3 + 1] = fma(R[i * 3 + 2], s0, -FBUS_PROD(R[i * 3 + 0], s2));
        A[i * 3 + 2] = fma(R[i * 3 + 0], s1, -FBUS_PROD(R[i * 3 + 1], s0));
        FBUS_UNROLL
        for (int j = 0; j < 3; ++j) B[i * 3 + j] = R[i * 3 + j] * ndt;
    }
    // Wm = -[w]x dt :  Wm01 = w2 dt, Wm02 = -w1 dt, Wm10 = -w2 dt, Wm12 = w0 dt, Wm20 = w1 dt, Wm21 = -w0 dt
    u[0] = w[0] * dt; u[1] = w[1] * dt; u[2] = w[2] * dt;
}

// TLR = true: the top-left 9x9 (p, v, theta covariance: read AND written by every step) is held in the caller's
// registers TL[45] across the IMU samples of a window instead of making a round trip through shared memory per step.
template <int S, bool TLR = false, class CV = Cov<S>>
FBUS_HD void propagate_cov_core(const CV P, const double* A, const double* B, double u0, double u1, double u2, double dt,
                                const double* Qd, double* TL = nullptr) {
// element (r, c) of block (bi, bj) loaded with ldblk_nw: a blocked accessor delivers the stored block (min, max), i.e. the
// transpose when bi > bj
#define FBUS_BLK(X, bi, bj, r, c) ((CV::kBlocked && (bi) > (bj)) ? X[(c) * 3 + (r)] : X[(r) * 3 + (c)])
#define FBUS_TLLD(i, j) (TLR ? TL[tlidx((i), (j))] : P.ld((i), (j)))
#define FBUS_TLST(i, j, v)                        \
    do {                                          \
        if (TLR) TL[tlidx((i), (j))] = (v);       \
        else P.st((i), (j), (v));                 \
    } while (0)
// block loads/stores of the top-left part through the same switch
#define FBUS_TL_LDBLK(bi, bj, X)                                                        \
    do {                                                                                \
        FBUS_UNROLL                                                                     \
        for (int r_ = 0; r_ < 3; ++r_)                                                  \
            FBUS_UNROLL                                                                 \
            for (int c_ = 0; c_ < 3; ++c_) X[r_ * 3 + c_] = FBUS_TLLD(3 * (bi) + r_, 3 * (bj) + c_); \
    } while (0)
#define FBUS_TL_STBLK(bi, bj, X)                                                        \
    do {                                                                                \
        FBUS_UNROLL                                                                     \
        for (int r_ = 0; r_ < 3; ++r_)                                                  \
            FBUS_UNROLL                                                                 \
            for (int c_ = ((bi) == (bj) ? r_ : 0); c_ < 3; ++c_) FBUS_TLST(3 * (bi) + r_, 3 * (bj) + c_, X[r_ * 3 + c_]); \
    } while (0)
    // Every sum below is written as a chain  s += x*y  so that it compiles to one DFMA per term.
    const double a = dt;
// s += (Wm X)[i][j]  and  s += (X Wm^T)[i][j] = sum_k X[i][k] Wm[j][k]   (two DFMA each)
#define FBUS_WX_ACC(s, X, i, j)                                                \
    do {                                                                       \
        if ((i) == 0) { s += u2 * X[3 + (j)]; s -= u1 * X[6 + (j)]; }          \
        else if ((i) == 1) { s += u0 * X[6 + (j)]; s -= u2 * X[(j)]; }         \
        else { s += u1 * X[(j)]; s -= u0 * X[3 + (j)]; }                       \
    } while (0)
#define FBUS_XWT_ACC(s, X, i, j)                                               \
    do {                                                                       \
        if ((j) == 0) { s += u2 * X[(i)*3 + 1]; s -= u1 * X[(i)*3 + 2]; }      \
        else if ((j) == 1) { s += u0 * X[(i)*3 + 2]; s -= u2 * X[(i)*3]; }     \
        else { s += u1 * X[(i)*3]; s -= u0 * X[(i)*3 + 1]; }                   \
    } while (0)

    // ---------------- phase 1: top-left blocks from old values -------------------------------
    // Staged so that few blocks are live at a time (FBUS_FENCE stops the scheduler hoisting every
    // shared-memory load to the top, which would blow the 255-register budget).
    {
        double P11[9], P12[9];
        FBUS_TL_LDBLK(1, 2, P12);
        double M12[9];
        {   // 1c: P'22 (without the -a*M24 term) ; M12 = P12 + A*P22 (+ more below)
            double P22[9], P24[9], U22[9], acc22[9];
            FBUS_TL_LDBLK(2, 2, P22);
            P.ldtr_nw(2, 4, P24, false);
            P.wait_ld();
            FBUS_UNROLL
            for (int i = 0; i < 3; ++i)
                FBUS_UNROLL
                for (int j = 0; j < 3; ++j) {
                    double s = P12[i * 3 + j];
                    FBUS_UNROLL
                    for (int k = 0; k < 3; ++k) s += A[i * 3 + k] * P22[k * 3 + j];
                    M12[i * 3 + j] = s;
                    double t = P22[i * 3 + j];
                    t -= a * P24[j * 3 + i];
                    FBUS_WX_ACC(t, P22, i, j);
                    U22[i * 3 + j] = t;
                }
            FBUS_UNROLL
            for (int i = 0; i < 3; ++i)
                FBUS_UNROLL
                for (int j = i; j < 3; ++j) {
                    double t = U22[i * 3 + j];
                    if (i == j) t += Qd[1];  // + gyro noise on theta
                    FBUS_XWT_ACC(t, U22, i, j);
                    acc22[i * 3 + j] = t;
                }
            FBUS_TL_STBLK(2, 2, acc22);
        }
        FBUS_FENCE_A;
        {   // M12 += B*P23^T + a*P25^T
            double P23[9], P25[9];
            P.ldtr_nw(2, 3, P23, false);
            P.ldtr_nw(2, 5, P25, false);
            P.wait_ld();
            FBUS_UNROLL
            for (int i = 0; i < 3; ++i)
                FBUS_UNROLL
                for (int j = 0; j < 3; ++j) {
                    double s = M12[i * 3 + j];
                    s += a * P25[j * 3 + i];
                    FBUS_UNROLL
                    for (int k = 0; k < 3; ++k) s += B[i * 3 + k] * P23[j * 3 + k];
                    M12[i * 3 + j] = s;
                }
        }
        FBUS_FENCE_A;
        {   // 1b: P'11 (without the M13*B^T + a*M15 term), P'12 (without -a*M14)
            double P13[9], P15[9], acc11[9], acc12[9];
            FBUS_TL_LDBLK(1, 1, P11);
            P.ldtr_nw(1, 3, P13, false);
            P.ldtr_nw(1, 5, P15, false);
            P.wait_ld();
            FBUS_UNROLL
            for (int i = 0; i < 3; ++i)
                FBUS_UNROLL
                for (int j = 0; j < 3; ++j) {
                    double t = M12[i * 3 + j];
                    FBUS_XWT_ACC(t, M12, i, j);
                    acc12[i * 3 + j] = t;
                    if (j >= i) {
                        double s = P11[i * 3 + j];
                        if (i == j) s += Qd[0];  // + accel noise on v
                        s += a * P15[j * 3 + i];
                        FBUS_UNROLL
                        for (int k = 0; k < 3; ++k) {
                            s += A[i * 3 + k] * P12[j * 3 + k];
                            s += B[i * 3 + k] * P13[j * 3 + k];
                            s += M12[i * 3 + k] * A[j * 3 + k];
                        }
                        acc11[i * 3 + j] = s;
                    }
                }
            FBUS_TL_STBLK(1, 1, acc11);
            FBUS_TL_STBLK(1, 2, acc12);
        }
        FBUS_FENCE_A;
        {   // 1a: P'00, P'01 (without M03*B^T + a*M05), P'02 (without -a*M04); uses OLD P11, P12 kept in registers
            double P00[9], P01[9], P02[9], acc00[9], acc01[9], acc02[9];
            FBUS_TL_LDBLK(0, 0, P00);
            FBUS_TL_LDBLK(0, 1, P01);
            FBUS_TL_LDBLK(0, 2, P02);
            FBUS_UNROLL
            for (int i = 0; i < 3; ++i)
                FBUS_UNROLL
                for (int j = i; j < 3; ++j) {
                    double m01 = P01[i * 3 + j];
                    m01 += a * P11[i * 3 + j];  // M01[i][j]
                    double t = P00[i * 3 + j];
                    t += a * P01[j * 3 + i];    // M00[i][j]
                    t += a * m01;
                    acc00[i * 3 + j] = t;
                }
            FBUS_UNROLL
            for (int e = 0; e < 9; ++e) {
                P01[e] += a * P11[e];  // M01
                P02[e] += a * P12[e];  // M02
            }
            FBUS_UNROLL
            for (int i = 0; i < 3; ++i)
                FBUS_UNROLL
                for (int j = 0; j < 3; ++j) {
                    double s = P01[i * 3 + j];
                    FBUS_UNROLL
                    for (int k = 0; k < 3; ++k) s += P02[i * 3 + k] * A[j * 3 + k];
                    acc01[i * 3 + j] = s;
                    double t = P02[i * 3 + j];
                    FBUS_XWT_ACC(t, P02, i, j);
                    acc02[i * 3 + j] = t;
                }
            FBUS_TL_STBLK(0, 0, acc00);
            FBUS_TL_STBLK(0, 1, acc01);
            FBUS_TL_STBLK(0, 2, acc02);
        }
    }
    FBUS_FENCE_B;
    // ---------------- phase 2: block columns 4, 3, 5 of rows 0..2 -----------------------------
    // the new cross blocks are computed and folded into the top-left block
    double d01[9], d11[9];
    FBUS_UNROLL
    for (int kk = 0; kk < 3; ++kk) {
        const int k = (kk == 0) ? 4 : (kk == 1) ? 3 : 5;
        double X1[9], X2[9], M0[9], M2[9];
        {
            P.ldtr_nw(1, k, X1, false);
            P.ldblk_nw(0, k, M0);
            P.ldtr_nw(2, k, X2, false);
            P.wait_ld();
            // row 0: M0 = P0k + a*P1k
            FBUS_UNROLL
            for (int e = 0; e < 9; ++e) M0[e] += a * X1[e];
            P.stblk(0, k, M0);
        }
        {
            if (k == 4) {  // P'02 -= a*M04
                FBUS_UNROLL
                for (int i = 0; i < 3; ++i)
                    FBUS_UNROLL
                    for (int j = 0; j < 3; ++j) {
                        double t = FBUS_TLLD(i, 6 + j);
                        t -= a * M0[i * 3 + j];
                        FBUS_TLST(i, 6 + j, t);
                    }
            } else if (k == 3) {  // d01 = M03*B^T
                FBUS_UNROLL
                for (int i = 0; i < 3; ++i)
                    FBUS_UNROLL
                    for (int j = 0; j < 3; ++j) {
                        double s = M0[i * 3] * B[j * 3];
                        s += M0[i * 3 + 1] * B[j * 3 + 1];
                        s += M0[i * 3 + 2] * B[j * 3 + 2];
                        d01[i * 3 + j] = s;
                    }
            } else {  // P'01 += d01 + a*M05
                FBUS_UNROLL
                for (int i = 0; i < 3; ++i)
                    FBUS_UNROLL
                    for (int j = 0; j < 3; ++j) {
                        double t = FBUS_TLLD(i, 3 + j) + d01[i * 3 + j];
                        t += a * M0[i * 3 + j];
                        FBUS_TLST(i, 3 + j, t);
                    }
            }
        }
        FBUS_FENCE_A;
        double X4[9];
        {   // row 1: M1 = P1k + A*P2k + B*P3k + a*P5k
            double X3[9], X5[9];
            P.ldblk_nw(3, k, X3);
            P.ldblk_nw(5, k, X5);
            P.ldblk_nw(4, k, X4);
            P.wait_ld();  // blocks below the diagonal arrive transposed from a blocked accessor: FBUS_BLK indexes them
            FBUS_UNROLL
            for (int i = 0; i < 3; ++i)
                FBUS_UNROLL
                for (int j = 0; j < 3; ++j) {
                    double s = X1[i * 3 + j];
                    s += a * FBUS_BLK(X5, 5, k, i, j);
                    FBUS_UNROLL
                    for (int c = 0; c < 3; ++c) {
                        s += A[i * 3 + c] * X2[c * 3 + j];
                        s += B[i * 3 + c] * FBUS_BLK(X3, 3, k, c, j);
                    }
                    X1[i * 3 + j] = s;  // M1 in place (X1[i][j] is not read again)
                }
            P.sttr(1, k, X1);
            if (k == 3) {  // accel-bias process noise on P33's diagonal
                FBUS_UNROLL
                for (int i = 0; i < 3; ++i) P.st(9 + i, 9 + i, X3[i * 3 + i] + Qd[2]);
            }
        }
        {
            if (k == 4) {  // P'12 -= a*M14
                FBUS_UNROLL
                for (int i = 0; i < 3; ++i)
                    FBUS_UNROLL
                    for (int j = 0; j < 3; ++j) {
                        double t = FBUS_TLLD(3 + i, 6 + j);
                        t -= a * X1[i * 3 + j];
                        FBUS_TLST(3 + i, 6 + j, t);
                    }
            } else if (k == 3) {  // d11 = M13*B^T (upper)
                FBUS_UNROLL
                for (int i = 0; i < 3; ++i)
                    FBUS_UNROLL
                    for (int j = i; j < 3; ++j) {
                        double s = X1[i * 3] * B[j * 3];
                        s += X1[i * 3 + 1] * B[j * 3 + 1];
                        s += X1[i * 3 + 2] * B[j * 3 + 2];
                        d11[i * 3 + j] = s;
                    }
            } else {  // P'11 += d11 + a*M15 (upper)
                FBUS_UNROLL
                for (int i = 0; i < 3; ++i)
                    FBUS_UNROLL
                    for (int j = i; j < 3; ++j) {
                        double t = FBUS_TLLD(3 + i, 3 + j) + d11[i * 3 + j];
                        t += a * X1[i * 3 + j];
                        FBUS_TLST(3 + i, 3 + j, t);
                    }
            }
        }
        FBUS_FENCE_A;
        {   // row 2: M2 = (I+Wm)*P2k - a*P4k
            FBUS_UNROLL
            for (int i = 0; i < 3; ++i)
                FBUS_UNROLL
                for (int j = 0; j < 3; ++j) {
                    double t = X2[i * 3 + j];
                    t -= a * FBUS_BLK(X4, 4, k, i, j);
                    FBUS_WX_ACC(t, X2, i, j);
                    M2[i * 3 + j] = t;
                }
            P.sttr(2, k, M2);
            if (k == 4) {  // gyro-bias process noise on P44's diagonal
                FBUS_UNROLL
                for (int i = 0; i < 3; ++i) P.st(12 + i, 12 + i, X4[i * 3 + i] + Qd[3]);
            }
        }
        if (k == 4) {  // P'22 -= a*M24 (upper)
            FBUS_UNROLL
            for (int i = 0; i < 3; ++i)
                FBUS_UNROLL
                for (int j = i; j < 3; ++j) {
                    double t = FBUS_TLLD(6 + i, 6 + j);
                    t -= a * M2[i * 3 + j];
                    FBUS_TLST(6 + i, 6 + j, t);
                }
        }
        FBUS_FENCE_B;
    }
#undef FBUS_WX_ACC
#undef FBUS_XWT_ACC
#undef FBUS_BLK
#undef FBUS_TLLD
#undef FBUS_TLST
#undef FBUS_TL_LDBLK
#undef FBUS_TL_STBLK
}

template <int S>
FBUS_HD void propagate_cov(const Cov<S> P, const double* R, const double* acc, const double* w, double dt, const double* Qd) {
    double A[9], B[9], u[3];
    cov_coeffs(R, acc, w, dt, A, B, u);
    propagate_cov_core<S, false>(P, A, B, u[0], u[1], u[2], dt, Qd, nullptr);
}

// ------------------------------------------------------------------------------------------------
// F2: nominal state propagation (FILTER::UpdateNominalState, filter.cpp:533-582)
// ------------------------------------------------------------------------------------------------
// The step in two halves.  nominal_increment: everything that depends on the sample, the biases and dt only (bias-corrected rate,
// the half- and full-interval increment quaternions): independent from sample to sample, so the lanes-per-filter kernel evaluates
// it for all samples of a window in parallel lanes.  nominal_apply: the part that is a chain through q, v, p.
FBUS_HD void nominal_increment(const double* w, double dt, double* dqh, double* dq) {
    const double wn2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
    const double inv = rsqrt_d(wn2);  // 1/|w| (inf for w = 0: only used in the branch below)
    const double wn = wn2 * inv;      // |w|
    // Both forms of the increment are evaluated and the one the reference's branch takes (filter.cpp:544-561) is selected:
    // straight-line code instead of a divergent region, so that the scheduler can overlap the sincos chain with the rest
    // of the step.  The values selected are exactly those the branch would have produced (a zero rate gives inf / NaN in
    // the unused axis-angle form, which the select discards).
    const bool big = wn > 10e-5;
    const double ax[3] = {w[0] * inv, w[1] * inv, w[2] * inv};
    // one sincos: the half-interval quaternion needs angle/2 = wn*dt/4, the full one twice that
    // (double-angle identities; ~1 ulp from evaluating sin/cos of wn*dt/2 directly)
    double sh, ch;
    sincos_d(big ? wn * dt * 0.25 : 0.0, &sh, &ch);
    const double sf = 2.0 * sh * ch, cf = 1.0 - 2.0 * sh * sh;
    dqh[0] = big ? ch : 1.0;
    dq[0] = big ? cf : 1.0;
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i) {
        dqh[1 + i] = big ? sh * ax[i] : 0.25 * dt * w[i];
        dq[1 + i] = big ? sf * ax[i] : 0.5 * dt * w[i];
    }
}
// the velocity / position half of nominal_apply: q0, R0 = quaternion and rotation matrix before the step, Rn = after it.  Not part of
// the chain through q, so the lanes-per-filter kernel runs it one sample behind (dt = 0 and a = 0 leave v and p as they are).
FBUS_HD void nominal_apply_vp(Nominal& n, double dt, const double* q0, const double* dqh, const double* a, const double* R0, const double* Rn) {
    double qh[4], Rh[9];
    qmul(q0, dqh, qh);
    qnormalize(qh);
    q2R(qh, Rh);
    double k1[3], k2[3], k4[3];
    mat3_vec(R0, a, k1);
    mat3_vec(Rh, a, k2);
    mat3_vec(Rn, a, k4);
    const double dt6 = dt * (1.0 / 6.0), dt2 = dt * 0.5;
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i) {
        const double kv1 = k1[i] + n.g[i], kv2 = k2[i] + n.g[i], kv4 = k4[i] + n.g[i];
        const double v0 = n.v[i];
        n.v[i] = v0 + dt6 * (kv1 + 2 * kv2 + 2 * kv2 + kv4);
        const double kp2 = v0 + kv1 * dt2, kp3 = v0 + kv2 * dt2;
        n.p[i] = n.p[i] + dt6 * (v0 + 2 * kp2 + 2 * kp3 + kp3);
    }
}
// the quaternion half: q <- normalised q * dq, rotmatI2G <- R(q)
FBUS_HD void nominal_apply_q(Nominal& n, const double* dq) {
    double qn[4];
    qmul(n.q, dq, qn);
    qnormalize(qn);
    FBUS_UNROLL
    for (int i = 0; i < 4; ++i) n.q[i] = qn[i];
    q2R(n.q, n.R);
}
// ---- the same arithmetic written for a LONE warp ------------------------------------------------------------------------------
// A warp that has its scheduler to itself (the nominal lane of the lanes-per-filter kernel) pays the full 8-clock latency of every
// dependent FP64 instruction, and ptxas keeps independent chains that are far apart in the source far apart in the code: F2 written
// as above ran at ~8 clk per instruction.  These versions evaluate TWO independent chains statement by statement next to each other
// (value for value the expressions of qmul / qnormalize / q2R, so the results are bit-identical).
FBUS_HD void qmul2(const double* a, const double* b, double* o, const double* c, const double* d, double* p) {
    const double w1 = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3];
    const double w2 = c[0] * d[0] - c[1] * d[1] - c[2] * d[2] - c[3] * d[3];
    const double x1 = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2];
    const double x2 = c[0] * d[1] + c[1] * d[0] + c[2] * d[3] - c[3] * d[2];
    const double y1 = a[0] * b[2] + a[2] * b[0] + a[3] * b[1] - a[1] * b[3];
    const double y2 = c[0] * d[2] + c[2] * d[0] + c[3] * d[1] - c[1] * d[3];
    const double z1 = a[0] * b[3] + a[3] * b[0] + a[1] * b[2] - a[2] * b[1];
    const double z2 = c[0] * d[3] + c[3] * d[0] + c[1] * d[2] - c[2] * d[1];
    o[0] = w1; o[1] = x1; o[2] = y1; o[3] = z1;
    p[0] = w2; p[1] = x2; p[2] = y2; p[3] = z2;
}
FBUS_HD void qnormalize2(double* q, double* r) {
    const double s1 = q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
    const double s2 = r[0] * r[0] + r[1] * r[1] + r[2] * r[2] + r[3] * r[3];
#ifdef __CUDA_ARCH__
    double y1, y2;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y1) : "d"(s1));
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y2) : "d"(s2));
    const double h1 = 0.5 * s1, h2 = 0.5 * s2;
    double e1 = fma(-h1 * y1, y1, 0.5), e2 = fma(-h2 * y2, y2, 0.5);
    y1 = fma(y1, e1, y1);
    y2 = fma(y2, e2, y2);
    e1 = fma(-h1 * y1, y1, 0.5);
    e2 = fma(-h2 * y2, y2, 0.5);
    y1 = fma(y1, e1, y1);
    y2 = fma(y2, e2, y2);
#else
    const double y1 = 1.0 / sqrt(s1), y2 = 1.0 / sqrt(s2);
#endif
    q[0] *= y1; r[0] *= y2; q[1] *= y1; r[1] *= y2; q[2] *= y1; r[2] *= y2; q[3] *= y1; r[3] *= y2;
}
FBUS_HD void q2R2(const double* q, double* R, const double* p, double* S) {
    const double w = q[0], x = q[1], y = q[2], z = q[3];
    const double a = p[0], b = p[1], c = p[2], d = p[3];
    const double tx = 2 * x, ty = 2 * y, tz = 2 * z;
    const double tb = 2 * b, tc = 2 * c, td = 2 * d;
    const double twx = FBUS_PROD(tx, w), twy = FBUS_PROD(ty, w), twz = FBUS_PROD(tz, w);
    const double tab = FBUS_PROD(tb, a), tac = FBUS_PROD(tc, a), tad = FBUS_PROD(td, a);
    const double tyy = FBUS_PROD(ty, y), tzz = FBUS_PROD(tz, z);
    const double tcc = FBUS_PROD(tc, c), tdd = FBUS_PROD(td, d);
    R[0] = 1 - fma(ty, y, tzz);  S[0] = 1 - fma(tc, c, tdd);
    R[1] = fma(ty, x, -twz);     S[1] = fma(tc, b, -tad);
    R[2] = fma(tz, x, twy);      S[2] = fma(td, b, tac);
    R[3] = fma(ty, x, twz);      S[3] = fma(tc, b, tad);
    R[4] = 1 - fma(tx, x, tzz);  S[4] = 1 - fma(tb, b, tdd);
    R[5] = fma(tz, y, -twx);     S[5] = fma(td, c, -tab);
    R[6] = fma(tz, x, -twy);     S[6] = fma(td, b, -tac);
    R[7] = fma(tz, y, twx);      S[7] = fma(td, c, tab);
    R[8] = 1 - fma(tx, x, tyy);  S[8] = 1 - fma(tb, b, tcc);
}
// One sample of the pipelined F2: the quaternion half of THIS sample (q <- normalised q * dq, rotmatI2G <- R(q)) side by side with
// the velocity / position half of the PREVIOUS one (nominal_apply_vp with its operands pq, pdqh, pa, pR0, pdt; its R-after-the-step is
// the current R(q), Rq).  On return Rq = R of the new quaternion.
FBUS_HD void nominal_apply_dual(Nominal& n, double* Rq, double pdt, const double* pq, const double* pdqh, const double* pa, const double* pR0,
                                const double* dq) {
    double qn[4], qh[4], Rh[9], k1[3], k2[3], k4[3];
    qmul2(n.q, dq, qn, pq, pdqh, qh);
    mat3_vec(pR0, pa, k1);
    mat3_vec(Rq, pa, k4);
    qnormalize2(qn, qh);
    FBUS_UNROLL
    for (int i = 0; i < 4; ++i) n.q[i] = qn[i];
    q2R2(n.q, n.R, qh, Rh);
    mat3_vec(Rh, pa, k2);
    const double dt6 = pdt * (1.0 / 6.0), dt2 = pdt * 0.5;
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i) {
        const double kv1 = k1[i] + n.g[i], kv2 = k2[i] + n.g[i], kv4 = k4[i] + n.g[i];
        const double v0 = n.v[i];
        n.v[i] = v0 + dt6 * (kv1 + 2 * kv2 + 2 * kv2 + kv4);
        const double kp2 = v0 + kv1 * dt2, kp3 = v0 + kv2 * dt2;
        n.p[i] = n.p[i] + dt6 * (v0 + 2 * kp2 + 2 * kp3 + kp3);
    }
    FBUS_UNROLL
    for (int i = 0; i < 9; ++i) Rq[i] = n.R[i];
}
FBUS_HD void nominal_apply(Nominal& n, double dt, const double* dqh, const double* dq, const double* a) {
    double R0[9], q0[4];
    q2R(n.q, R0);
    FBUS_UNROLL
    for (int i = 0; i < 4; ++i) q0[i] = n.q[i];
    nominal_apply_q(n, dq);
    nominal_apply_vp(n, dt, q0, dqh, a, R0, n.R);
}
FBUS_HD void propagate_nominal(Nominal& n, double dt, const double* accel, const double* gyro) {
    double w[3], a[3], dqh[4], dq[4];
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i) {
        w[i] = gyro[i] - n.bg[i];
        a[i] = accel[i] - n.ba[i];
    }
    nominal_increment(w, dt, dqh, dq);
    nominal_apply(n, dt, dqh, dq, a);
}

// ------------------------------------------------------------------------------------------------
// MATLAB-semantics mode (FBUS_FLAG_MATLAB): the numerics of matlab/*.m where they differ from filter.cpp (SURVEY A.4)
// ------------------------------------------------------------------------------------------------
// quaternion_to_rotmat.m:24-32: the w^2+x^2-y^2-z^2 form (equal to Eigen's toRotationMatrix only for a unit quaternion; the
// MATLAB filter applies it to un-normalised products)
FBUS_HD void q2R_matlab(const double* q, double* R) {
    const double w = q[0], x = q[1], y = q[2], z = q[3];
    const double ww = FBUS_PROD(w, w), wx = FBUS_PROD(w, x), wy = FBUS_PROD(w, y), wz = FBUS_PROD(w, z);  // (pairing written out: see q2R)
    R[0] = fma(-z, z, fma(-y, y, fma(x, x, ww)));  R[1] = 2 * fma(x, y, -wz);                     R[2] = 2 * fma(x, z, wy);
    R[3] = 2 * fma(x, y, wz);                      R[4] = fma(-z, z, fma(y, y, fma(-x, x, ww)));  R[5] = 2 * fma(y, z, -wx);
    R[6] = 2 * fma(x, z, -wy);                     R[7] = 2 * fma(y, z, wx);                      R[8] = fma(z, z, fma(-y, y, fma(-x, x, ww)));
}
// ImuUpdate.m:37-60,76-79: always the axis-angle increment (axis = w/|w|: NaN for w = 0, as MATLAB), rotation matrices of
// the UN-normalised products, R0 = the carried State.rotateMat, State.rotateMat <- R(qT), State.quaternion <- qT/|qT|
FBUS_HD void propagate_nominal_matlab(Nominal& n, double dt, const double* accel, const double* gyro) {
    double w[3];
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i) w[i] = gyro[i] - n.bg[i];
    const double wn2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
    const double inv = rsqrt_d(wn2);
    const double wn = wn2 * inv;
    const double ax[3] = {w[0] * inv, w[1] * inv, w[2] * inv};
    const double dth = wn * (dt < 0 ? -dt : dt);  // norm(w*dt)
    double sh, ch;
    sincos_d(dth * 0.25, &sh, &ch);               // qHalfT: axisangle(w, dtheta/2) -> half angle dtheta/4
    const double sf = 2.0 * sh * ch, cf = 1.0 - 2.0 * sh * sh;
    const double dqh[4] = {ch, sh * ax[0], sh * ax[1], sh * ax[2]};
    const double dq[4] = {cf, sf * ax[0], sf * ax[1], sf * ax[2]};
    double qh[4], qn[4], R0[9], Rh[9];
    qmul(n.q, dqh, qh);
    qmul(n.q, dq, qn);
    FBUS_UNROLL
    for (int i = 0; i < 9; ++i) R0[i] = n.R[i];
    q2R_matlab(qh, Rh);
    q2R_matlab(qn, n.R);
    qnormalize(qn);
    FBUS_UNROLL
    for (int i = 0; i < 4; ++i) n.q[i] = qn[i];
    double a[3], k1[3], k2[3], k4[3];
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i) a[i] = accel[i] - n.ba[i];
    mat3_vec(R0, a, k1);
    mat3_vec(Rh, a, k2);
    mat3_vec(n.R, a, k4);
    const double dt6 = dt * (1.0 / 6.0), dt2 = dt * 0.5;
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i) {
        const double kv1 = k1[i] + n.g[i], kv2 = k2[i] + n.g[i], kv4 = k4[i] + n.g[i];
        const double v0 = n.v[i];
        n.v[i] = v0 + dt6 * (kv1 + 2 * kv2 + 2 * kv2 + kv4);
        const double kp2 = v0 + kv1 * dt2, kp3 = v0 + kv2 * dt2;
        n.p[i] = n.p[i] + dt6 * (v0 + 2 * kp2 + 2 * kp3 + kp3);
    }
}
// ImuUpdate.m:68: Fx(7:9,7:9) = expm(-[w]x dt), returned as W = expm(-[w]x dt) - I (the kernels add the identity themselves).
// Rodrigues: expm(-K) = I - (sin t / t) K + ((1 - cos t) / t^2) K^2 with K = [w dt]x, t = |w dt|.
FBUS_HD void expm_rot_minus_I(const double* w, double dt, double* W) {
    const double v[3] = {w[0] * dt, w[1] * dt, w[2] * dt};
    const double t2 = v[0] * v[0] + v[1] * v[1] + v[2] * v[2];
    double s1 = 1.0, c1 = 0.5;  // limits for t -> 0
    if (t2 > 1e-16) {
        const double it = rsqrt_d(t2), t = t2 * it;
        double sh, ch;
        sincos_d(0.5 * t, &sh, &ch);
        s1 = 2.0 * sh * ch * it;         // sin t / t
        c1 = 2.0 * sh * sh * (it * it);  // (1 - cos t) / t^2
    }
    // K = [v]x ; K^2 = v v^T - t^2 I
    const double K[9] = {0.0, -v[2], v[1], v[2], 0.0, -v[0], -v[1], v[0], 0.0};
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i)
        FBUS_UNROLL
        for (int j = 0; j < 3; ++j) {
            const double k2 = v[i] * v[j] - ((i == j) ? t2 : 0.0);
            W[i * 3 + j] = c1 * k2 - s1 * K[i * 3 + j];
        }
}

// ------------------------------------------------------------------------------------------------
// marker-map lookup (std::map::find on markerPoseServer_, filter.cpp:353,442,671)
// ------------------------------------------------------------------------------------------------
FBUS_HD int find_marker(const DevConsts& k, const MarkerTable* tab, int id) {
    int m = -1;
    for (int i = 0; i < k.n_markers; ++i)
        if (tab->mk[i].id == id) m = (m < 0) ? i : m;
    return m;
}

// vision-only pose (shared by InitializePose filter.cpp:379-384 and ResetSystemState :454-459):
//   q = Q_M * conj(Q_ML) * Q_IL ;  Rq = R(q) ;  p = P_M - Rq*P_IL - Rq*R_IL^T*P_ML
template <bool MATLAB = false>
FBUS_HD void vision_pose(const DevConsts& k, const MarkerConst& mk, const double* pml, const double* qml, double* q,
                         double* Rq, double* p) {
    double t1[4];
    qmul_conjb(mk.q, qml, t1);
    qmul(t1, k.Q_IL, q);
    if (MATLAB) q2R_matlab(q, Rq);  // InitPositionAndQuaternion.m / ResetState.m: quaternion_to_rotmat of the un-normalised Q_IG
    else q2R(q, Rq);
    double u[3], r1[3], r2[3];
    mat3t_vec(k.R_IL, pml, u);  // R_IL^T * P_ML
    mat3_vec(Rq, k.P_IL, r1);
    mat3_vec(Rq, u, r2);
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i) p[i] = (mk.p[i] - r1[i]) - r2[i];
}

// ------------------------------------------------------------------------------------------------
// F4: measurement update (FILTER::ObservationUpdate, filter.cpp:677-739) for the chosen detection.
//
// H = [Hp0 0 Hp2 0 0 0 ; 0 0 Hq 0 0 0] only touches block rows/cols 0 (p) and 2 (theta):
//   with G = P[{0,1,2,6,7,8}, :] (6x18), Hs = [Hp0 Hp2; 0 Hq] (7x6), P6 = G[:, {0,1,2,6,7,8}]
//   S = Hs P6 Hs^T + R ;  K = G^T Hs^T S^-1 ;  dx = G^T u, u = Hs^T S^-1 r ;
//   (I-KH)P = P - G^T C G,  C = Hs^T S^-1 Hs = Lc Lc^T  ->  P' = P - Z^T Z,  Z = Lc^T G.
// Z is applied in two half-rank sweeps (rows 0..2 then 3..5) so that only 54 doubles are live;
// G's theta rows are rebuilt between the sweeps (see DESIGN.md "update without scratch").
// S is SPD, so Cholesky replaces the reference's LDLT (filter.cpp:711).  Measured against a 50-digit evaluation of one update
// (tests/test_precision_host.py, host build of this header), the error of the updated (p, theta) block whitened by its exact
// value stays within 1.2 to 3.4x of the dense double oracle's own error for R from 1e-3 down to 1e-12: 3e-16 at the default
// R = 1e-3, 3e-12 at the noise sweep's corner (pos 1e-8, quat 1e-7), 8e-10 at 1e-10 and 7e-8 at 1e-12.  Both forms lose about
// eps * |P6 before| / |P6 after| to the cancellation in P - K H P; tests/test_gpu_precision.py holds every kernel form to 8x the
// oracle's error and to 1e-9 on the sweep's range (R >= 1e-8).
// ------------------------------------------------------------------------------------------------
// In-place Cholesky of a packed lower-triangular matrix (row-major packed: L[i*(i+1)/2 + j]); also returns the
// reciprocal diagonal.  Template recursion instead of a loop over columns: nvcc does not fully unroll the
// column loop (it contains sqrt/division slow paths), and a rolled loop would index L dynamically and push
// it to local memory.
template <int N, int J>
struct CholStep {
    static FBUS_HD void run(double* L, double* Li) {
        double s = L[J * (J + 1) / 2 + J];
        FBUS_UNROLL
        for (int c = 0; c < J; ++c) s -= L[J * (J + 1) / 2 + c] * L[J * (J + 1) / 2 + c];
        const double di = rsqrt_d(s);  // 1/sqrt(s) by MUFU.RSQ64H + Newton (1-2 ulp); d = s * di
        const double d = s * di;
        L[J * (J + 1) / 2 + J] = d;
        Li[J] = di;
        FBUS_UNROLL
        for (int i = J + 1; i < N; ++i) {
            double s2 = L[i * (i + 1) / 2 + J];
            FBUS_UNROLL
            for (int c = 0; c < J; ++c) s2 -= L[i * (i + 1) / 2 + c] * L[J * (J + 1) / 2 + c];
            L[i * (i + 1) / 2 + J] = s2 * di;
        }
        CholStep<N, J + 1>::run(L, Li);
    }
};
template <int N>
struct CholStep<N, N> {
    static FBUS_HD void run(double*, double*) {}
};

// First half: predicted measurement, Hs, S = Hs P6 Hs^T + R = L L^T, X = L^-1 Hs (7x6, left in scr with element stride XS) and
// z = L^-1 r.  With these alone (I-KH)P = P - (X G)^T (X G) and dx = (X G)^T z (the lanes-per-filter kernel stops here: a
// 7-row factor costs its parallel sweep little and saves the serial second factorisation); the second half below reduces
// the factor to 6 rows.
// the state-only part: Hs = [Hp0 Hp2; 0 Hq] and the residual r (filter.cpp:677-721); needs nothing of P
struct UpdHs {
    double Hp0[9], Hp2[9], Hq[12], r[7];
};
// Measurement noise of one filter (rows 4, 5 of the per-filter noise buffer of fbus_set_noise).  The update functions read
// R from `kr.Rp` / `kr.Rq` of a template type KR: DevConsts itself on the default path (the same constant loads as before),
// this struct where every filter has its own values.
struct MeasNoise {
    double Rp, Rq;
};
template <bool MATLAB = false>
FBUS_HD void update_hs(const Nominal& n, const DevConsts& k, const MarkerConst& mk, const double* yP, const double* yQ, UpdHs& hh) {
    double* const Hp0 = hh.Hp0;
    double* const Hp2 = hh.Hp2;
    double* const Hq = hh.Hq;
    double* const r = hh.r;
    {
        double dp[3], rtdp[3], RP[3], d2[3], rt2[3], hP[3];
        FBUS_UNROLL
        for (int i = 0; i < 3; ++i) dp[i] = mk.p[i] - n.p[i];
        mat3t_vec(n.R, dp, rtdp);  // R^T (P_M - p)
        mat3_vec(n.R, k.P_IL, RP);
        FBUS_UNROLL
        for (int i = 0; i < 3; ++i) d2[i] = dp[i] - RP[i];
        mat3t_vec(n.R, d2, rt2);
        mat3_vec(k.R_IL, rt2, hP);  // hP = R_IL R^T (P_M - p - R P_IL)
        FBUS_UNROLL
        for (int i = 0; i < 3; ++i) r[i] = yP[i] - hP[i];
        // Hp0 = -R_IL R^T ; Hp2 = R_IL [R^T(P_M - p)]x
        FBUS_UNROLL
        for (int i = 0; i < 3; ++i)
            FBUS_UNROLL
            for (int j = 0; j < 3; ++j) {
                double s = k.R_IL[i * 3] * n.R[j * 3];
                s += k.R_IL[i * 3 + 1] * n.R[j * 3 + 1];
                s += k.R_IL[i * 3 + 2] * n.R[j * 3 + 2];
                Hp0[i * 3 + j] = -s;
            }
        FBUS_UNROLL
        for (int i = 0; i < 3; ++i) {
            const double a0 = k.R_IL[i * 3], a1 = k.R_IL[i * 3 + 1], a2 = k.R_IL[i * 3 + 2];
            Hp2[i * 3 + 0] = a1 * rtdp[2] - a2 * rtdp[1];
            Hp2[i * 3 + 1] = a2 * rtdp[0] - a0 * rtdp[2];
            Hp2[i * 3 + 2] = a0 * rtdp[1] - a1 * rtdp[0];
        }
        // hQ = Q_IL * conj(q) * Q_M ; Hq = CM * (L(q) L1),  L(q) L1 = 0.5*[[-x,-y,-z],[w,-z,y],[z,w,-x],[-y,x,w]]
        double t1[4], hQ[4];
        qmul_conjb(k.Q_IL, n.q, t1);
        qmul(t1, mk.q, hQ);
        double k1 = 0.0, k2 = 0.0;
        FBUS_UNROLL
        for (int i = 0; i < 4; ++i) {
            k1 += (yQ[i] - hQ[i]) * (yQ[i] - hQ[i]);
            k2 += (yQ[i] + hQ[i]) * (yQ[i] + hQ[i]);
        }
        const double sg = (k1 > k2) ? -1.0 : 1.0;  // filter.cpp:702-706 (strict >): flips hQ and H[3:7,6:9]
        const double hs = 0.5 * sg;
        const double w = hs * n.q[0], x = hs * n.q[1], y = hs * n.q[2], z = hs * n.q[3];
        const double LL[12] = {-x, -y, -z, w, -z, y, z, w, -x, -y, x, w};
        FBUS_UNROLL
        for (int i = 0; i < 4; ++i)
            FBUS_UNROLL
            for (int j = 0; j < 3; ++j) {
                double s = mk.CM[i * 4] * LL[j];
                FBUS_UNROLL
                for (int c = 1; c < 4; ++c) s += mk.CM[i * 4 + c] * LL[c * 3 + j];
                Hq[i * 3 + j] = s;
            }
        FBUS_UNROLL
        for (int i = 0; i < 4; ++i) r[3 + i] = MATLAB ? 0.0 : (yQ[i] - sg * hQ[i]);  // MeasureUpdate.m:88 zeroes the quaternion rows
    }
}
template <int S, int XS, class CV = Cov<S>, class KR = DevConsts>
FBUS_HD void update_prologue_sx(const CV P, const KR& k, const UpdHs& hh, double* L, double* Li, double* z, double* scr) {
    // scr: 42 doubles of scratch with element stride XS (shared memory in the warp-specialised kernel) for X = L^-1 Hs
    const double* const Hp0 = hh.Hp0;
    const double* const Hp2 = hh.Hp2;
    const double* const Hq = hh.Hq;
    const double* const r = hh.r;
    // ---- S = Hs P6 Hs^T + R (lower triangle, packed in L) --------------------------------------
    // L[28]: row-major packed lower triangle: L[i*(i+1)/2 + j]
#define FBUS_L(i, j) L[(i) * ((i) + 1) / 2 + (j)]
    {
        double P00[9], P02[9], P22[9];
        P.lddiag(0, P00);
        P.ldblk(0, 2, P02);
        P.lddiag(2, P22);
        double Ep[18], Eq[24];  // Ep = [Hp0 Hp2] P6 (3x6) ; Eq = Hq [P20 P22] (4x6)
        FBUS_UNROLL
        for (int i = 0; i < 3; ++i)
            FBUS_UNROLL
            for (int j = 0; j < 3; ++j) {
                double s0 = Hp0[i * 3] * P00[j], s1 = Hp0[i * 3] * P02[j];
                FBUS_UNROLL
                for (int c = 1; c < 3; ++c) {
                    s0 += Hp0[i * 3 + c] * P00[c * 3 + j];
                    s1 += Hp0[i * 3 + c] * P02[c * 3 + j];
                }
                FBUS_UNROLL
                for (int c = 0; c < 3; ++c) {
                    s0 += Hp2[i * 3 + c] * P02[j * 3 + c];
                    s1 += Hp2[i * 3 + c] * P22[c * 3 + j];
                }
                Ep[i * 6 + j] = s0;
                Ep[i * 6 + 3 + j] = s1;
            }
        FBUS_UNROLL
        for (int i = 0; i < 4; ++i)
            FBUS_UNROLL
            for (int j = 0; j < 3; ++j) {
                double s0 = Hq[i * 3] * P02[j * 3], s1 = Hq[i * 3] * P22[j];
                FBUS_UNROLL
                for (int c = 1; c < 3; ++c) {
                    s0 += Hq[i * 3 + c] * P02[j * 3 + c];
                    s1 += Hq[i * 3 + c] * P22[c * 3 + j];
                }
                Eq[i * 6 + j] = s0;
                Eq[i * 6 + 3 + j] = s1;
            }
        FBUS_UNROLL
        for (int i = 0; i < 3; ++i)
            FBUS_UNROLL
            for (int j = 0; j <= i; ++j) {
                double s = (i == j) ? k.Rp : 0.0;
                FBUS_UNROLL
                for (int c = 0; c < 3; ++c) {
                    s += Ep[i * 6 + c] * Hp0[j * 3 + c];
                    s += Ep[i * 6 + 3 + c] * Hp2[j * 3 + c];
                }
                FBUS_L(i, j) = s;
            }
        FBUS_UNROLL
        for (int i = 0; i < 4; ++i) {
            FBUS_UNROLL
            for (int j = 0; j < 3; ++j) {  // S[3+i][j] = Eq[i][0:3] Hp0[j]^T + Eq[i][3:6] Hp2[j]^T
                double s = Eq[i * 6] * Hp0[j * 3];
                FBUS_UNROLL
                for (int c = 1; c < 3; ++c) s += Eq[i * 6 + c] * Hp0[j * 3 + c];
                FBUS_UNROLL
                for (int c = 0; c < 3; ++c) s += Eq[i * 6 + 3 + c] * Hp2[j * 3 + c];
                FBUS_L(3 + i, j) = s;
            }
            FBUS_UNROLL
            for (int j = 0; j <= i; ++j) {
                double s = (i == j) ? k.Rq : 0.0;
                FBUS_UNROLL
                for (int c = 0; c < 3; ++c) s += Eq[i * 6 + 3 + c] * Hq[j * 3 + c];
                FBUS_L(3 + i, 3 + j) = s;
            }
        }
    }
    // ---- Cholesky S = L L^T (in place), reciprocal diagonal in Li -------------------------------
    CholStep<7, 0>::run(L, Li);
    // ---- X = L^-1 Hs (7x6), z = L^-1 r -----------------------------------------------------------
#define FBUS_X(i) scr[(i) * XS]
    {
        FBUS_UNROLL
        for (int i = 0; i < 7; ++i) {
            FBUS_UNROLL
            for (int c = 0; c < 6; ++c) {
                double s = (i < 3) ? ((c < 3) ? Hp0[i * 3 + c] : Hp2[i * 3 + (c - 3)]) : ((c < 3) ? 0.0 : Hq[(i - 3) * 3 + (c - 3)]);
                FBUS_UNROLL
                for (int j = 0; j < i; ++j) s -= FBUS_L(i, j) * FBUS_X(j * 6 + c);
                FBUS_X(i * 6 + c) = s * Li[i];
            }
            double s = r[i];
            FBUS_UNROLL
            for (int j = 0; j < i; ++j) s -= FBUS_L(i, j) * z[j];
            z[i] = s * Li[i];
        }
    }
#undef FBUS_L
#undef FBUS_X
}

// Prologue of the update: everything up to the gain factors.  Reads only the 21 entries of P6 = P[{p,theta},{p,theta}].
// Outputs Cm = lower-packed Cholesky factor Lc of C = Hs^T S^-1 Hs and y = Lc^-1 u (u = Hs^T S^-1 r), so that
//   (I-KH)P = P - Z^T Z with Z = Lc^T G, and dx = K r = Z^T y.
// kr: where R comes from (DevConsts or MeasNoise, see MeasNoise)
// zo (optional): receives z = L^-1 r (7 doubles), whose squared norm is the update's NIS r^T S^-1 r (the innovation gate)
template <int S, int XS, bool JOSEPH = false, class CV = Cov<S>, class KR = DevConsts>
FBUS_HD void update_prologue(const CV P, const Nominal& n, const DevConsts& k, const KR& kr, const MarkerConst& mk, const double* yP,
                             const double* yQ, double* Cm, double* y, double* scr, double* zo = nullptr) {
    double L[28], Li[7], z[7];
    {
        UpdHs hh;
        update_hs(n, k, mk, yP, yQ, hh);
        update_prologue_sx<S, XS, CV>(P, kr, hh, L, Li, z, scr);
    }
    if (zo) {
        FBUS_UNROLL
        for (int i = 0; i < 7; ++i) zo[i] = z[i];
    }
#define FBUS_L(i, j) L[(i) * ((i) + 1) / 2 + (j)]
#define FBUS_X(i) scr[(i) * XS]
    // ---- C = X^T X ; u = X^T z -------------------------------------------------------------------
    double u[6];  // (Cm: C lower packed, Cm[i*(i+1)/2+j])
#define FBUS_C(i, j) Cm[(i) * ((i) + 1) / 2 + (j)]
    {
        FBUS_UNROLL
        for (int i = 0; i < 6; ++i) {
            FBUS_UNROLL
            for (int j = 0; j <= i; ++j) {
                double s = FBUS_X(i) * FBUS_X(j);
                FBUS_UNROLL
                for (int c = 1; c < 7; ++c) s += FBUS_X(c * 6 + i) * FBUS_X(c * 6 + j);
                FBUS_C(i, j) = s;
            }
            double s = FBUS_X(i) * z[0];
            FBUS_UNROLL
            for (int c = 1; c < 7; ++c) s += FBUS_X(c * 6 + i) * z[c];
            u[i] = s;
        }
    }
    if (JOSEPH) {
        // FBUS_FLAG_JOSEPH (compile-time variant so that the default path carries none of this code): Joseph-form covariance update  P' = (I-KH) P (I-KH)^T + K R K^T  evaluated in the same reduced
        // space.  With K = G^T Hs^T S^-1 it equals  P - G^T C_J G,  C_J = 2C - C P6 C - D,  D = Y^T R Y,  Y = S^-1 Hs
        // (C P6 C + D = C in exact arithmetic, so C_J = C up to rounding; the default is the reference's (I-KH)P).
        // P - G^T C_J G subtracts from P like the standard form, so this has the standard form's accuracy, not the dense Joseph
        // form's: at the sweep's corner (R = 1e-8 / 1e-7) the whitened P6 error is 6e-12 against 2e-15 for the oracle's dense
        // (I-KH) P (I-KH)^T + K R K^T, and 7e-8 against 7e-16 at R = 1e-12 (host build, tests/test_precision_host.py).
        double Y[42];  // S^-1 Hs = L^-T X  (back substitution)
        FBUS_UNROLL
        for (int i = 6; i >= 0; --i)
            FBUS_UNROLL
            for (int c = 0; c < 6; ++c) {
                double s = FBUS_X(i * 6 + c);
                FBUS_UNROLL
                for (int j = i + 1; j < 7; ++j) s -= FBUS_L(j, i) * Y[j * 6 + c];
                Y[i * 6 + c] = s * Li[i];
            }
        double P6[36];  // [[P00 P02],[P02^T P22]]
        FBUS_UNROLL
        for (int i = 0; i < 6; ++i)
            FBUS_UNROLL
            for (int j = 0; j < 6; ++j) P6[i * 6 + j] = P.ld(i < 3 ? i : i + 3, j < 3 ? j : j + 3);
        double CP[36];  // C P6 (C symmetric, lower packed)
        FBUS_UNROLL
        for (int i = 0; i < 6; ++i)
            FBUS_UNROLL
            for (int j = 0; j < 6; ++j) {
                double s = 0.0;
                FBUS_UNROLL
                for (int c = 0; c < 6; ++c) s += ((i >= c) ? FBUS_C(i, c) : FBUS_C(c, i)) * P6[c * 6 + j];
                CP[i * 6 + j] = s;
            }
        double CJ[21];
        FBUS_UNROLL
        for (int i = 0; i < 6; ++i)
            FBUS_UNROLL
            for (int j = 0; j <= i; ++j) {
                double s = 2.0 * FBUS_C(i, j);
                FBUS_UNROLL
                for (int c = 0; c < 6; ++c) s -= CP[i * 6 + c] * ((c >= j) ? FBUS_C(c, j) : FBUS_C(j, c));
                FBUS_UNROLL
                for (int c = 0; c < 7; ++c) s -= ((c < 3) ? kr.Rp : kr.Rq) * Y[c * 6 + i] * Y[c * 6 + j];
                CJ[i * (i + 1) / 2 + j] = s;
            }
        FBUS_UNROLL
        for (int i = 0; i < 21; ++i) Cm[i] = CJ[i];
    }
#undef FBUS_L
#undef FBUS_X
    // ---- Cholesky C = Lc Lc^T (in place in Cm) ; y = Lc^-1 u -------------------------------------
    // dx = K r = G^T u = Z^T y = Za^T y[0:3] + Zb^T y[3:6]
    {
        double Lci[6];
        CholStep<6, 0>::run(Cm, Lci);
        FBUS_UNROLL
        for (int i = 0; i < 6; ++i) {
            double s = u[i];
            FBUS_UNROLL
            for (int j = 0; j < i; ++j) s -= FBUS_C(i, j) * y[j];
            y[i] = s * Lci[i];
        }
    }
#undef FBUS_C
}
// R from the constants
template <int S, int XS, bool JOSEPH = false, class CV = Cov<S>>
FBUS_HD void update_prologue(const CV P, const Nominal& n, const DevConsts& k, const MarkerConst& mk, const double* yP,
                             const double* yQ, double* Cm, double* y, double* scr) {
    update_prologue<S, XS, JOSEPH, CV>(P, n, k, k, mk, yP, yQ, Cm, y, scr);
}

// rows 0..2 of Z = Lc^T G from the current P (G = rows {0,1,2,6,7,8} of P)
#define FBUS_C(i, j) Cm[(i) * ((i) + 1) / 2 + (j)]
template <int S>
FBUS_HD void update_Za(const Cov<S> P, const double* Cm, double* Z) {
    FBUS_UNROLL
    for (int m = 0; m < 6; ++m) {
        const int row = (m < 3) ? m : (3 + m);  // 0,1,2,6,7,8
        FBUS_UNROLL
        for (int c = 0; c < 18; ++c) {
            const double g = P.ld(row, c);
            FBUS_UNROLL
            for (int kz = 0; kz < 3; ++kz) {
                if (m == kz) Z[kz * 18 + c] = FBUS_C(m, kz) * g;
                else if (m > kz) Z[kz * 18 + c] += FBUS_C(m, kz) * g;
            }
        }
    }
}
// rows 3..5 of Z = Lc^T G from the current (not yet swept) P: only the theta rows 6..8 are needed
template <int S>
FBUS_HD void update_Zb(const Cov<S> P, const double* Cm, double* Z) {
    FBUS_UNROLL
    for (int c = 0; c < 18; ++c) {
        const double g3 = P.ld(6, c), g4 = P.ld(7, c), g5 = P.ld(8, c);
        double t3 = FBUS_C(3, 3) * g3;
        t3 += FBUS_C(4, 3) * g4;
        t3 += FBUS_C(5, 3) * g5;
        double t4 = FBUS_C(4, 4) * g4;
        t4 += FBUS_C(5, 4) * g5;
        Z[c] = t3;
        Z[18 + c] = t4;
        Z[36 + c] = FBUS_C(5, 5) * g5;
    }
}
#undef FBUS_C
// same from the six entries of Lc's rows 3..5 alone (what the nominal warp of the split kernel receives)
template <int S>
FBUS_HD void update_Zb6(const Cov<S> P, double c33, double c43, double c44, double c53, double c54, double c55, double* Z) {
    FBUS_UNROLL
    for (int c = 0; c < 18; ++c) {
        const double g3 = P.ld(6, c), g4 = P.ld(7, c), g5 = P.ld(8, c);
        double t3 = c33 * g3;
        t3 += c43 * g4;
        t3 += c53 * g5;
        double t4 = c44 * g4;
        t4 += c54 * g5;
        Z[c] = t3;
        Z[18 + c] = t4;
        Z[36 + c] = c55 * g5;
    }
}
// P[i][j] -= sum_k Z[k][i] Z[k][j] for rows R0 <= i < R1 (j >= i)
// `on` = false turns the stores off (predicated stores: the split kernel keeps the code between two barriers free of
// divergent regions, because ptxas parks values that live across such regions in local memory)
template <int S, int R0, int R1>
FBUS_HD void update_sweep(const Cov<S> P, const double* Z, bool on = true) {
    FBUS_UNROLL
    for (int i = R0; i < R1; ++i)
        FBUS_UNROLL
        for (int j = i; j < 18; ++j) {
            double v = P.ld(i, j);
            v -= Z[i] * Z[j];
            v -= Z[18 + i] * Z[18 + j];
            v -= Z[36 + i] * Z[36 + j];
            if (on) P.st(i, j, v);
        }
}
// dx[c] (+)= y0 Z[0][c] + y1 Z[1][c] + y2 Z[2][c]
template <bool ACC>
FBUS_HD void update_dx(const double* Z, double y0, double y1, double y2, double* dx) {
    FBUS_UNROLL
    for (int c = 0; c < 18; ++c) {
        double s = ACC ? dx[c] : 0.0;
        s += y0 * Z[c];
        s += y1 * Z[18 + c];
        s += y2 * Z[36 + c];
        dx[c] = s;
    }
}
// error-state injection (filter.cpp:726-733); rotmatI2G deliberately NOT refreshed (SURVEY A.3-2)
FBUS_HD void inject_error_state(Nominal& n, const double* dx) {
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i) {
        n.p[i] += dx[i];
        n.v[i] += dx[3 + i];
        n.ba[i] += dx[9 + i];
        n.bg[i] += dx[12 + i];
        n.g[i] += dx[15 + i];
    }
    // VectorToQuaterniond (matrix_math.hpp:90-99): v/|v| * sin(|v|/2); NaN at exactly zero, as the reference
    const double v2 = dx[6] * dx[6] + dx[7] * dx[7] + dx[8] * dx[8];
    const double iv = rsqrt_d(v2);  // inf at exactly zero -> NaN below, as the reference's 0/0
    const double vn = v2 * iv;
    double sh, ch;
    sincos_d(vn * 0.5, &sh, &ch);
    const double sc = iv * sh;
    const double dq[4] = {ch, dx[6] * sc, dx[7] * sc, dx[8] * sc};
    double qn[4];
    qmul(n.q, dq, qn);
    qnormalize(qn);
    FBUS_UNROLL
    for (int i = 0; i < 4; ++i) n.q[i] = qn[i];
}

// Cooperative form used by the warp-specialised kernel (here executed by one thread, for the host harness): both
// half-rank factors are taken from the OLD covariance, then applied; algebraically identical to measurement_update.
template <int S>
FBUS_HD void measurement_update_coop(const Cov<S> P, Nominal& n, const DevConsts& k, const MarkerConst& mk, const double* yP,
                                     const double* yQ) {
    double Cm[21], y[6], Za[54], Zb[54], dx[18], xloc[42];
    update_prologue<S, 1>(P, n, k, mk, yP, yQ, Cm, y, xloc);
    update_Za<S>(P, Cm, Za);
    update_Zb<S>(P, Cm, Zb);
    update_sweep<S, 0, 18>(P, Za);
    update_sweep<S, 0, 18>(P, Zb);
    update_dx<false>(Za, y[0], y[1], y[2], dx);
    update_dx<true>(Zb, y[3], y[4], y[5], dx);
    inject_error_state(n, dx);
}

// ------------------------------------------------------------------------------------------------------------------
// One-pass form of the covariance update (default, FBUS_UPDATE_ONEPASS=1): every entry of P is read once and written
// once.  Z = Lc^T G (6 x 18) is never held whole: the columns of the p/v/theta block (0..8) stay in registers (54
// doubles), the columns of the bias/gravity block (9..17) are produced one at a time from the OLD rows of G, used for the
// 9 cross entries of that column, and parked in `stash` (54 doubles, stride XS: the exchange area of the split kernel)
// for the bottom-right block.  Shared-memory accesses per update: 495 instead of the two-sweep form's 846, and no
// rebuild of the old theta rows.  Per entry the six FMAs run in the same order as in the two-sweep form.
// ------------------------------------------------------------------------------------------------------------------
#ifndef FBUS_UPDATE_ONEPASS
#define FBUS_UPDATE_ONEPASS 1
#endif
template <int S, int XS, class CV = Cov<S>>
FBUS_HD void update_onepass(const CV P, Nominal& n, const double* Cm, const double* y, double* stash) {
#define FBUS_C(i, j) Cm[(i) * ((i) + 1) / 2 + (j)]
#define FBUS_GROW(m) (((m) < 3) ? (m) : (3 + (m)))  // rows of G: 0,1,2,6,7,8
    double dth[3] = {0.0, 0.0, 0.0};
    double Z1[54];  // Z[k][c], c = 0..8, at Z1[k * 9 + c]
    // ---- phase 1: Z columns 0..8 from the top-left block ----------------------------------------------
    FBUS_UNROLL
    for (int c = 0; c < 9; ++c) {
        double g[6];
        FBUS_UNROLL
        for (int m = 0; m < 6; ++m) g[m] = P.ld(FBUS_GROW(m), c);
        FBUS_UNROLL
        for (int kz = 0; kz < 6; ++kz) {
            double z = FBUS_C(kz, kz) * g[kz];
            FBUS_UNROLL
            for (int m = kz + 1; m < 6; ++m) z += FBUS_C(m, kz) * g[m];
            Z1[kz * 9 + c] = z;
        }
    }
    // error-state injection (filter.cpp:726-733), columns 0..8: dx[c] = sum_k y[k] Z[k][c]
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i) {
        FBUS_UNROLL
        for (int kz = 0; kz < 6; ++kz) {
            n.p[i] += y[kz] * Z1[kz * 9 + i];
            n.v[i] += y[kz] * Z1[kz * 9 + 3 + i];
            dth[i] += y[kz] * Z1[kz * 9 + 6 + i];
        }
    }
    FBUS_FENCE;
    // top-left block
    FBUS_UNROLL
    for (int i = 0; i < 9; ++i)
        FBUS_UNROLL
        for (int j = i; j < 9; ++j) {
            double v = P.ld(i, j);
            FBUS_UNROLL
            for (int kz = 0; kz < 6; ++kz) v -= Z1[kz * 9 + i] * Z1[kz * 9 + j];
            P.st(i, j, v);
        }
    FBUS_FENCE;
    P.fence_st();
    // ---- phase 2: columns 9..17: Z column from the OLD G entries of that column, cross entries, stash ------
    FBUS_UNROLL
    for (int c = 9; c < 18; ++c) {
        double col[9];
        FBUS_UNROLL
        for (int i = 0; i < 9; ++i) col[i] = P.ld(i, c);
        double z[6];
        FBUS_UNROLL
        for (int kz = 0; kz < 6; ++kz) {
            double t = FBUS_C(kz, kz) * col[FBUS_GROW(kz)];
            FBUS_UNROLL
            for (int m = kz + 1; m < 6; ++m) t += FBUS_C(m, kz) * col[FBUS_GROW(m)];
            z[kz] = t;
            stash[(size_t)((c - 9) * 6 + kz) * XS] = t;
        }
        {
            double* dst = (c < 12) ? &n.ba[c - 9] : (c < 15) ? &n.bg[c - 12] : &n.g[c - 15];
            double d = *dst;
            FBUS_UNROLL
            for (int kz = 0; kz < 6; ++kz) d += y[kz] * z[kz];
            *dst = d;
        }
        FBUS_UNROLL
        for (int i = 0; i < 9; ++i) {
            double v = col[i];
            FBUS_UNROLL
            for (int kz = 0; kz < 6; ++kz) v -= Z1[kz * 9 + i] * z[kz];
            P.st(i, c, v);
        }
    }
    FBUS_FENCE;
    P.fence_st();
    // ---- phase 3: bottom-right block from the stashed columns -------------------------------------------
    {
        double Z2[54];  // Z[k][c], c = 9..17, at Z2[(c - 9) * 6 + k]
        FBUS_UNROLL
        for (int e = 0; e < 54; ++e) Z2[e] = stash[(size_t)e * XS];
        FBUS_UNROLL
        for (int i = 9; i < 18; ++i)
            FBUS_UNROLL
            for (int j = i; j < 18; ++j) {
                double v = P.ld(i, j);
                FBUS_UNROLL
                for (int kz = 0; kz < 6; ++kz) v -= Z2[(i - 9) * 6 + kz] * Z2[(j - 9) * 6 + kz];
                P.st(i, j, v);
            }
    }
#undef FBUS_GROW
#undef FBUS_C
    {   // VectorToQuaterniond (matrix_math.hpp:90-99): v/|v| * sin(|v|/2); NaN at exactly zero, as the reference
        const double v2 = dth[0] * dth[0] + dth[1] * dth[1] + dth[2] * dth[2];
        const double iv = rsqrt_d(v2);  // inf at exactly zero -> NaN below, as the reference's 0/0
        const double vn = v2 * iv;
        double sh, ch;
        sincos_d(vn * 0.5, &sh, &ch);
        const double sc = iv * sh;
        const double dq[4] = {ch, dth[0] * sc, dth[1] * sc, dth[2] * sc};
        double qn[4];
        qmul(n.q, dq, qn);
        qnormalize(qn);
        FBUS_UNROLL
        for (int i = 0; i < 4; ++i) n.q[i] = qn[i];
    }
}

// JMODE: 0 = reference form (I-KH)P, 1 = Joseph form, -1 = decided at run time from k.flags (host harness, un-split kernel)
// Block form of the one-pass update for accessors whose natural unit is a 3x3 block (tensor memory): same arithmetic per
// entry (six FMAs in the same order), the entries are visited block by block.
//   1. Z columns 0..8 from the blocks (0,0) (0,1) (0,2) (1,2) (2,2); sweep of the six top-left blocks;
//   2a. Z columns 9..17 from the blocks (0,k), (2,k), k = 3..5 -> stash (Lc is dead afterwards);
//   2b. sweep of the nine cross blocks (Z columns of block column k re-read from the stash);
//   3.  sweep of the six bottom-right blocks from the stashed columns.
template <int S, int XS, class CV>
FBUS_HD void update_onepass_blk(const CV P, Nominal& n, const double* Cm, const double* y, double* stash) {
#define FBUS_C(i, j) Cm[(i) * ((i) + 1) / 2 + (j)]
    double dth[3] = {0.0, 0.0, 0.0};
    double Z1[54];  // Z[k][c], c = 0..8, at Z1[k * 9 + c]
    {
        double B00[9], B01[9], B02[9], B12[9], B22[9];
        P.ldblk_nw(0, 0, B00); P.ldblk_nw(0, 1, B01); P.ldblk_nw(0, 2, B02); P.ldblk_nw(1, 2, B12); P.ldblk_nw(2, 2, B22);
        P.wait_ld();
        FBUS_UNROLL
        for (int c = 0; c < 9; ++c) {
            double g[6];
            FBUS_UNROLL
            for (int m = 0; m < 3; ++m) {
                g[m] = (c < 3) ? B00[m * 3 + c] : (c < 6) ? B01[m * 3 + (c - 3)] : B02[m * 3 + (c - 6)];
                g[3 + m] = (c < 3) ? B02[c * 3 + m] : (c < 6) ? B12[(c - 3) * 3 + m] : B22[m * 3 + (c - 6)];
            }
            FBUS_UNROLL
            for (int kz = 0; kz < 6; ++kz) {
                double z = FBUS_C(kz, kz) * g[kz];
                FBUS_UNROLL
                for (int m = kz + 1; m < 6; ++m) z += FBUS_C(m, kz) * g[m];
                Z1[kz * 9 + c] = z;
            }
        }
    }
    FBUS_UNROLL
    for (int i = 0; i < 3; ++i) {
        FBUS_UNROLL
        for (int kz = 0; kz < 6; ++kz) {
            n.p[i] += y[kz] * Z1[kz * 9 + i];
            n.v[i] += y[kz] * Z1[kz * 9 + 3 + i];
            dth[i] += y[kz] * Z1[kz * 9 + 6 + i];
        }
    }
    FBUS_FENCE;
    FBUS_UNROLL
    for (int bj = 0; bj < 3; ++bj)
        FBUS_UNROLL
        for (int bi = 0; bi <= bj; ++bi) {
            double T[9];
            P.ldblk_nw(bi, bj, T);
            P.wait_ld();
            FBUS_UNROLL
            for (int r = 0; r < 3; ++r)
                FBUS_UNROLL
                for (int c = (bi == bj ? r : 0); c < 3; ++c) {
                    double v = T[r * 3 + c];
                    FBUS_UNROLL
                    for (int kz = 0; kz < 6; ++kz) v -= Z1[kz * 9 + 3 * bi + r] * Z1[kz * 9 + 3 * bj + c];
                    T[r * 3 + c] = v;
                }
            if (bi == bj) P.stdiag(bi, T);
            else P.stblk(bi, bj, T);
        }
    FBUS_FENCE;
    // ---- 2a: Z columns 9..17 -> stash ------------------------------------------------------------------
    FBUS_UNROLL
    for (int k = 3; k < 6; ++k) {
        double B0[9], B2[9];
        P.ldblk_nw(0, k, B0); P.ldblk_nw(2, k, B2);
        P.wait_ld();
        FBUS_UNROLL
        for (int c = 0; c < 3; ++c) {
            double z[6];
            FBUS_UNROLL
            for (int kz = 0; kz < 6; ++kz) {
                double t = FBUS_C(kz, kz) * ((kz < 3) ? B0[kz * 3 + c] : B2[(kz - 3) * 3 + c]);
                FBUS_UNROLL
                for (int m = kz + 1; m < 6; ++m) t += FBUS_C(m, kz) * ((m < 3) ? B0[m * 3 + c] : B2[(m - 3) * 3 + c]);
                z[kz] = t;
                stash[(size_t)(((k - 3) * 3 + c) * 6 + kz) * XS] = t;
            }
            double* dst = (k == 3) ? &n.ba[c] : (k == 4) ? &n.bg[c] : &n.g[c];
            double d = *dst;
            FBUS_UNROLL
            for (int kz = 0; kz < 6; ++kz) d += y[kz] * z[kz];
            *dst = d;
        }
    }
#undef FBUS_C
    FBUS_FENCE;
    // ---- 2b: cross blocks -----------------------------------------------------------------------------
    FBUS_UNROLL
    for (int k = 3; k < 6; ++k) {
        double zc[18];  // z of columns 3k..3k+2: zc[c * 6 + kz]
        FBUS_UNROLL
        for (int e = 0; e < 18; ++e) zc[e] = stash[(size_t)((k - 3) * 18 + e) * XS];
        FBUS_UNROLL
        for (int bi = 0; bi < 3; ++bi) {
            double T[9];
            P.ldblk_nw(bi, k, T);
            P.wait_ld();
            FBUS_UNROLL
            for (int r = 0; r < 3; ++r)
                FBUS_UNROLL
                for (int c = 0; c < 3; ++c) {
                    double v = T[r * 3 + c];
                    FBUS_UNROLL
                    for (int kz = 0; kz < 6; ++kz) v -= Z1[kz * 9 + 3 * bi + r] * zc[c * 6 + kz];
                    T[r * 3 + c] = v;
                }
            P.stblk(bi, k, T);
        }
    }
    FBUS_FENCE;
    // ---- 3: bottom-right blocks -----------------------------------------------------------------------
    {
        double Z2[54];  // Z[k][c], c = 9..17, at Z2[(c - 9) * 6 + k]
        FBUS_UNROLL
        for (int e = 0; e < 54; ++e) Z2[e] = stash[(size_t)e * XS];
        FBUS_UNROLL
        for (int bj = 3; bj < 6; ++bj)
            FBUS_UNROLL
            for (int bi = 3; bi <= bj; ++bi) {
                double T[9];
                P.ldblk_nw(bi, bj, T);
                P.wait_ld();
                FBUS_UNROLL
                for (int r = 0; r < 3; ++r)
                    FBUS_UNROLL
                    for (int c = (bi == bj ? r : 0); c < 3; ++c) {
                        double v = T[r * 3 + c];
                        FBUS_UNROLL
                        for (int kz = 0; kz < 6; ++kz) v -= Z2[(3 * (bi - 3) + r) * 6 + kz] * Z2[(3 * (bj - 3) + c) * 6 + kz];
                        T[r * 3 + c] = v;
                    }
                if (bi == bj) P.stdiag(bi, T);
                else P.stblk(bi, bj, T);
            }
    }
    {   // VectorToQuaterniond (matrix_math.hpp:90-99): v/|v| * sin(|v|/2); NaN at exactly zero, as the reference
        const double v2 = dth[0] * dth[0] + dth[1] * dth[1] + dth[2] * dth[2];
        const double iv = rsqrt_d(v2);  // inf at exactly zero -> NaN below, as the reference's 0/0
        const double vn = v2 * iv;
        double sh, ch;
        sincos_d(vn * 0.5, &sh, &ch);
        const double sc = iv * sh;
        const double dq[4] = {ch, dth[0] * sc, dth[1] * sc, dth[2] * sc};
        double qn[4];
        qmul(n.q, dq, qn);
        qnormalize(qn);
        FBUS_UNROLL
        for (int i = 0; i < 4; ++i) n.q[i] = qn[i];
    }
}

// stash: 54 doubles of scratch with stride XS (nullptr: a private array); kr: where R comes from (DevConsts or MeasNoise)
template <int S, int JMODE = -1, int XS = 1, class CV = Cov<S>, class KR = DevConsts>
FBUS_HD void measurement_update(const CV P, Nominal& n, const DevConsts& k, const KR& kr, const MarkerConst& mk, const double* yP,
                                const double* yQ, double* stash, bool on) {
    double Cm[21], y[6];
    {
        double xloc[42];  // X = L^-1 Hs stays private
        if (JMODE == 1 || (JMODE < 0 && (k.flags & 1))) update_prologue<S, 1, true>(P, n, k, kr, mk, yP, yQ, Cm, y, xloc);
        else update_prologue<S, 1, false>(P, n, k, kr, mk, yP, yQ, Cm, y, xloc);
    }
    if (!on) {  // lane without an update inside a warp that must stay convergent: zero gain, P and the state keep their values
        FBUS_UNROLL
        for (int i = 0; i < 21; ++i) Cm[i] = 0.0;
        FBUS_UNROLL
        for (int i = 0; i < 6; ++i) y[i] = 0.0;
    }
#if FBUS_UPDATE_ONEPASS
    if (CV::kBlocked) {
        update_onepass_blk<S, XS>(P, n, Cm, y, stash);
    } else if (stash != nullptr) {
        update_onepass<S, XS>(P, n, Cm, y, stash);
    } else {
        double loc[54];
        update_onepass<S, 1>(P, n, Cm, y, loc);
    }
    return;
#endif
#define FBUS_C(i, j) Cm[(i) * ((i) + 1) / 2 + (j)]
    double dth[3];  // attitude part of dx (needed whole before the quaternion injection)
    double Z[54];   // 3 x 18
    // ---- stream G (rows 0..2 and 6..8 of P): Za = rows 0..2 of Lc^T G -----------------------------
    FBUS_UNROLL
    for (int m = 0; m < 6; ++m) {
        const int row = (m < 3) ? m : (3 + m);  // 0,1,2,6,7,8
        FBUS_UNROLL
        for (int c = 0; c < 18; ++c) {
            const double g = P.ld(row, c);
            FBUS_UNROLL
            for (int kz = 0; kz < 3; ++kz) {
                if (m == kz) Z[kz * 18 + c] = FBUS_C(m, kz) * g;
                else if (m > kz) Z[kz * 18 + c] += FBUS_C(m, kz) * g;
            }
        }
    }
    // error-state injection, first half (filter.cpp:726-733); rotmatI2G deliberately NOT refreshed
#define FBUS_DX_ACC(dst, c)       \
    do {                          \
        dst += y0 * Z[c];         \
        dst += y1 * Z[18 + (c)];  \
        dst += y2 * Z[36 + (c)];  \
    } while (0)
    {
        const double y0 = y[0], y1 = y[1], y2 = y[2];
        FBUS_UNROLL
        for (int i = 0; i < 3; ++i) {
            FBUS_DX_ACC(n.p[i], i);
            FBUS_DX_ACC(n.v[i], 3 + i);
            dth[i] = 0.0;
            FBUS_DX_ACC(dth[i], 6 + i);
            FBUS_DX_ACC(n.ba[i], 9 + i);
            FBUS_DX_ACC(n.bg[i], 12 + i);
            FBUS_DX_ACC(n.g[i], 15 + i);
        }
    }
    FBUS_FENCE;
    // ---- sweep 1: P -= Za^T Za -----------------------------------------------------------------
    FBUS_UNROLL
    for (int i = 0; i < 18; ++i)
        FBUS_UNROLL
        for (int j = i; j < 18; ++j) {
            double v = P.ld(i, j);
            v -= Z[i] * Z[j];
            v -= Z[18 + i] * Z[18 + j];
            v -= Z[36 + i] * Z[36 + j];
            P.st(i, j, v);
        }
    FBUS_FENCE;
    // ---- rebuild G_b = P_old[6..8,:] = P1[6..8,:] + Za[:,6..8]^T Za, then Zb = Lbb^T G_b in place ----
    {
        const double z06 = Z[6], z07 = Z[7], z08 = Z[8], z16 = Z[18 + 6], z17 = Z[18 + 7], z18 = Z[18 + 8], z26 = Z[36 + 6],
                     z27 = Z[36 + 7], z28 = Z[36 + 8];
        FBUS_UNROLL
        for (int c = 0; c < 18; ++c) {
            const double za0 = Z[c], za1 = Z[18 + c], za2 = Z[36 + c];
            double g3 = P.ld(6, c), g4 = P.ld(7, c), g5 = P.ld(8, c);
            g3 += z06 * za0; g3 += z16 * za1; g3 += z26 * za2;
            g4 += z07 * za0; g4 += z17 * za1; g4 += z27 * za2;
            g5 += z08 * za0; g5 += z18 * za1; g5 += z28 * za2;
            double t3 = FBUS_C(3, 3) * g3;
            t3 += FBUS_C(4, 3) * g4;
            t3 += FBUS_C(5, 3) * g5;
            double t4 = FBUS_C(4, 4) * g4;
            t4 += FBUS_C(5, 4) * g5;
            Z[c] = t3;
            Z[18 + c] = t4;
            Z[36 + c] = FBUS_C(5, 5) * g5;
        }
    }
#undef FBUS_C
    {   // injection, second half
        const double y0 = y[3], y1 = y[4], y2 = y[5];
        FBUS_UNROLL
        for (int i = 0; i < 3; ++i) {
            FBUS_DX_ACC(n.p[i], i);
            FBUS_DX_ACC(n.v[i], 3 + i);
            FBUS_DX_ACC(dth[i], 6 + i);
            FBUS_DX_ACC(n.ba[i], 9 + i);
            FBUS_DX_ACC(n.bg[i], 12 + i);
            FBUS_DX_ACC(n.g[i], 15 + i);
        }
    }
#undef FBUS_DX_ACC
    FBUS_FENCE;
    // ---- sweep 2: P -= Zb^T Zb -----------------------------------------------------------------
    FBUS_UNROLL
    for (int i = 0; i < 18; ++i)
        FBUS_UNROLL
        for (int j = i; j < 18; ++j) {
            double v = P.ld(i, j);
            v -= Z[i] * Z[j];
            v -= Z[18 + i] * Z[18 + j];
            v -= Z[36 + i] * Z[36 + j];
            P.st(i, j, v);
        }
    {   // VectorToQuaterniond (matrix_math.hpp:90-99): v/|v| * sin(|v|/2); NaN at exactly zero, as the reference
        const double v2 = dth[0] * dth[0] + dth[1] * dth[1] + dth[2] * dth[2];
        const double iv = rsqrt_d(v2);  // inf at exactly zero -> NaN below, as the reference's 0/0
        const double vn = v2 * iv;
        double sh, ch;
        sincos_d(vn * 0.5, &sh, &ch);
        const double sc = iv * sh;
        const double dq[4] = {ch, dth[0] * sc, dth[1] * sc, dth[2] * sc};
        double qn[4];
        qmul(n.q, dq, qn);
        qnormalize(qn);
        FBUS_UNROLL
        for (int i = 0; i < 4; ++i) n.q[i] = qn[i];
    }
}
// R from the constants
template <int S, int JMODE = -1, int XS = 1, class CV = Cov<S>>
FBUS_HD void measurement_update(const CV P, Nominal& n, const DevConsts& k, const MarkerConst& mk, const double* yP,
                                const double* yQ, double* stash = nullptr, bool on = true) {
    measurement_update<S, JMODE, XS, CV>(P, n, k, k, mk, yP, yQ, stash, on);
}

}  // namespace fbus
