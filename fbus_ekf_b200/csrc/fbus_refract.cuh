// fbus_refract.cuh -- refractive flat-port marker-pose solve, per-marker device inlines.
//   R1  VISION::RefractionTriangulation  (C++/src/vision.cpp:488-608)
//   R2  VISION::ComputeMarkerPose        (C++/src/vision.cpp:635-759)
// One thread per marker; everything lives in registers.  Also host-compilable (tests only).
#pragma once

#include "fbus_math.cuh"

// cap of the Newton steps on the characteristic polynomial / Rayleigh-quotient polish of the plane normal (smallest_eigvec_sym3)
#ifndef FBUS_EIG_NEWTON
#define FBUS_EIG_NEWTON 60
#endif
#ifndef FBUS_EIG_POLISH
#define FBUS_EIG_POLISH 0
#endif

namespace fbus {

// common.hpp:14 -- the reference overrides M_PI; R2's -pi/4 rotation must use this value (A.3-1)
constexpr double REF_M_PI = 3.1415926;

// Snell refraction of unit ray r at a plane with normal nv (vision.cpp:505-543):
//   r' = alpha*r + beta*nv, beta = sqrt(1-alpha^2(1-v^2)) - alpha*v  (or its negation, see `rule`)
FBUS_HD void refract_ray(const double* r, const double* nv, double alpha, int rule, double* out, double* v_out) {
    const double v = r[0] * nv[0] + r[1] * nv[1] + r[2] * nv[2];
    const double arg = 1 - alpha * alpha * (1 - v * v);
    const double root = arg * rsqrt_d(arg);  // sqrt to ~1 ulp without the correctly-rounded sequence (NaN for arg <= 0: total reflection)
    const double beta = rule ? (root - alpha * v) : (alpha * v - root);
    FBUS_UNROLL
    for (int j = 0; j < 3; ++j) out[j] = alpha * r[j] + beta * nv[j];
    *v_out = v;
}

FBUS_HD double det3_cols(const double* a, const double* b, const double* c) {  // det of [a b c] (columns)
    // cofactor expansion along the first row of the matrix whose columns are a,b,c
    return a[0] * (b[1] * c[2] - c[1] * b[2]) - b[0] * (a[1] * c[2] - c[1] * a[2]) + c[0] * (a[1] * b[2] - b[1] * a[2]);
}

// R1 for one stereo corner pair: (xl,yl),(xr,yr) float32-valued normalised coordinates -> P (3), flipped
// by R_I_C = diag(-1,-1,1); returns |P| (the unflipped norm, vision.cpp:601)
FBUS_HD double triangulate_corner(const DevConsts& k, double xl, double yl, double xr, double yr, double* Pout) {
    double r0L[3] = {xl, yl, 1.0}, r0R[3] = {xr, yr, 1.0};
    {
        const double il = rsqrt_d(r0L[0] * r0L[0] + r0L[1] * r0L[1] + 1.0), ir = rsqrt_d(r0R[0] * r0R[0] + r0R[1] * r0R[1] + 1.0);
        FBUS_UNROLL
        for (int j = 0; j < 3; ++j) { r0L[j] *= il; r0R[j] *= ir; }
    }
    double r1L[3], r1R[3], r2L[3], r2R[3], v0L, v0R, v1L, v1R;
    refract_ray(r0L, k.normal, k.a0, k.air_lt_glass, r1L, &v0L);
    refract_ray(r0R, k.normal, k.a0, k.air_lt_glass, r1R, &v0R);
    refract_ray(r1L, k.normal, k.a1, k.glass_gt_water, r2L, &v1L);
    refract_ray(r1R, k.normal, k.a1, k.glass_gt_water, r2R, &v1R);
    double P1L[3], P1R[3];
    {
        // d_air / v0 and d_glass / v1 from ONE reciprocal per ray: 1 / (v0 v1)
        const double iL = rcp_d(v0L * v1L), iR = rcp_d(v0R * v1R);
        const double s0L = k.d_air * (v1L * iL), s0R = k.d_air * (v1R * iR), s1L = k.d_glass * (v0L * iL), s1R = k.d_glass * (v0R * iR);
        FBUS_UNROLL
        for (int j = 0; j < 3; ++j) {
            P1L[j] = s0L * r0L[j] + s1L * r1L[j];
            P1R[j] = s0R * r0R[j] + s1R * r1R[j];
        }
    }
    double rR[3], pR[3];
    mat3_vec(k.R_RL, r2R, rR);
    mat3_vec(k.R_RL, P1R, pR);
    FBUS_UNROLL
    for (int j = 0; j < 3; ++j) pR[j] += k.P_LR[j];
    const double c[3] = {r2L[1] * rR[2] - r2L[2] * rR[1], r2L[2] * rR[0] - r2L[0] * rR[2], r2L[0] * rR[1] - r2L[1] * rR[0]};
    const double d[3] = {pR[0] - P1L[0], pR[1] - P1L[1], pR[2] - P1L[2]};
    const double inv3 = rcp_d(c[0] * c[0] + c[1] * c[1] + c[2] * c[2]);  // det[c, rL, rR] = c . (rL x rR) = |c|^2
    const double t1 = det3_cols(c, d, rR) * inv3;
    const double t2 = -det3_cols(c, r2L, d) * inv3;
    double P[3];
    FBUS_UNROLL
    for (int j = 0; j < 3; ++j) P[j] = 0.5 * (P1L[j] + t1 * r2L[j] + pR[j] + t2 * rR[j]);
    Pout[0] = -P[0]; Pout[1] = -P[1]; Pout[2] = P[2];
    const double n2 = P[0] * P[0] + P[1] * P[1] + P[2] * P[2];
    return n2 * rsqrt_d(n2);  // |P|, only compared with the detection-distance threshold
}

// unit eigenvector of the smallest eigenvalue of a symmetric 3x3 (stands in for EigenSolver<Matrix3d>,
// vision.cpp:679-696; only this eigenvector is used and its sign is re-fixed by the caller).
// Closed-form eigenvalue (trigonometric) -> null vector of (M - lambda I) by the largest row cross product
// -> one Rayleigh-quotient polish.  The smallest eigenvalue of the corner scatter matrix is well separated
// (the two large ones are nearly equal for a square marker), so this is well conditioned.
FBUS_HD void null_vec(const double* M, double lam, double* v) {
    const double r0[3] = {M[0] - lam, M[1], M[2]}, r1[3] = {M[3], M[4] - lam, M[5]}, r2[3] = {M[6], M[7], M[8] - lam};
    const double c0[3] = {r0[1] * r1[2] - r0[2] * r1[1], r0[2] * r1[0] - r0[0] * r1[2], r0[0] * r1[1] - r0[1] * r1[0]};
    const double c1[3] = {r0[1] * r2[2] - r0[2] * r2[1], r0[2] * r2[0] - r0[0] * r2[2], r0[0] * r2[1] - r0[1] * r2[0]};
    const double c2[3] = {r1[1] * r2[2] - r1[2] * r2[1], r1[2] * r2[0] - r1[0] * r2[2], r1[0] * r2[1] - r1[1] * r2[0]};
    const double n0 = c0[0] * c0[0] + c0[1] * c0[1] + c0[2] * c0[2];
    const double n1 = c1[0] * c1[0] + c1[1] * c1[1] + c1[2] * c1[2];
    const double n2 = c2[0] * c2[0] + c2[1] * c2[1] + c2[2] * c2[2];
    double b0 = c0[0], b1 = c0[1], b2 = c0[2], nb = n0;
    if (n1 > nb) { b0 = c1[0]; b1 = c1[1]; b2 = c1[2]; nb = n1; }
    if (n2 > nb) { b0 = c2[0]; b1 = c2[1]; b2 = c2[2]; nb = n2; }
    const double inv = rsqrt_d(nb);
    v[0] = b0 * inv; v[1] = b1 * inv; v[2] = b2 * inv;
}
FBUS_HD void smallest_eigvec_sym3(const double* M, double* z) {
    // Smallest root of the characteristic polynomial f(l) = l^3 - c2 l^2 + c1 l - c0 by Newton from l = 0: M is positive
    // semi-definite, so f(0) = -det M <= 0 and f is increasing and concave left of its smallest root -- the iterates rise
    // monotonically to it and never overshoot.  For the corner scatter matrix (smallest eigenvalue ~ noise^2, the other two
    // ~ side^2) the first step already has a relative error of ~l_min/l_2; the Rayleigh polish below removes what is left.
    const double c2 = M[0] + M[4] + M[8];
    const double c1 = (M[0] * M[4] - M[1] * M[1]) + (M[0] * M[8] - M[2] * M[2]) + (M[4] * M[8] - M[5] * M[5]);
    const double c0 = M[0] * (M[4] * M[8] - M[5] * M[5]) - M[1] * (M[1] * M[8] - M[5] * M[2]) + M[2] * (M[1] * M[5] - M[4] * M[2]);
    // Iterated to convergence: two or three steps for a clean marker; up to FBUS_EIG_NEWTON when the corner noise is so large
    // that the smallest eigenvalue is no longer well separated (the monotone iteration is then slower, but still safe).
    double lam = 0.0;
    for (int it = 0; it < FBUS_EIG_NEWTON; ++it) {
        const double f = ((lam - c2) * lam + c1) * lam - c0;
        const double df = (3.0 * lam - 2.0 * c2) * lam + c1;
        const double step = f * rcp_d(df);
        lam -= step;
        if (!((step < 0 ? -step : step) > 2.3e-16 * c2)) break;  // also leaves on NaN
    }
#if FBUS_EIG_POLISH
    double v[3];
    null_vec(M, lam, v);
    // Rayleigh-quotient polish
    double Mv[3];
    mat3_vec(M, v, Mv);
    lam = v[0] * Mv[0] + v[1] * Mv[1] + v[2] * Mv[2];
#endif
    null_vec(M, lam, z);
}

FBUS_HD double signum_ref(double x) { return x < 0 ? -1.0 : 1.0; }  // matrix_math.hpp:9-15

// R2 for one marker: C[12] = 4 corners x 3 -> p (corner 0 projected), q = Quaterniond([X Y Z])
// rod_s, rod_c = sin/cos of -REF_M_PI/4 (computed once on the host)
FBUS_HD void marker_pose(const double* C, double rod_s, double rod_c, double* p, double* q) {
    const double* c0 = C; const double* c1 = C + 3; const double* c2 = C + 6; const double* c3 = C + 9;
    double M[9];
    {
        double v[6][3];
        FBUS_UNROLL
        for (int j = 0; j < 3; ++j) {
            v[0][j] = c1[j] - c0[j]; v[1][j] = c2[j] - c0[j]; v[2][j] = c3[j] - c0[j];
            v[3][j] = c2[j] - c1[j]; v[4][j] = c3[j] - c1[j]; v[5][j] = c3[j] - c2[j];
        }
        FBUS_UNROLL
        for (int i = 0; i < 3; ++i)
            FBUS_UNROLL
            for (int j = i; j < 3; ++j) {
                double s = 0.0;
                FBUS_UNROLL
                for (int e = 0; e < 6; ++e) s += v[e][i] * v[e][j];
                M[i * 3 + j] = s;
                M[j * 3 + i] = s;
            }
    }
    double Z[3];
    smallest_eigvec_sym3(M, Z);
    {   // vision.cpp:697-709
        double s = 1.0;
        if (Z[2] > 0.1) s = -1.0;
        else if (Z[2] < -0.1) s = 1.0;
        else s = -signum_ref(c0[0]) * signum_ref(Z[0]);
        Z[0] *= s; Z[1] *= s; Z[2] *= s;
    }
    const double D = 0.25 * (Z[0] * (c0[0] + c1[0] + c2[0] + c3[0]) + Z[1] * (c0[1] + c1[1] + c2[1] + c3[1]) +
                             Z[2] * (c0[2] + c1[2] + c2[2] + c3[2]));
    double P1[3], P2[3], P4[3];
    {
        const double t1 = (Z[0] * c0[0] + Z[1] * c0[1] + Z[2] * c0[2]) - D;
        const double t2 = (Z[0] * c1[0] + Z[1] * c1[1] + Z[2] * c1[2]) - D;
        const double t4 = (Z[0] * c3[0] + Z[1] * c3[1] + Z[2] * c3[2]) - D;
        FBUS_UNROLL
        for (int j = 0; j < 3; ++j) {
            P1[j] = c0[j] - t1 * Z[j];
            P2[j] = c1[j] - t2 * Z[j];
            P4[j] = c3[j] - t4 * Z[j];
        }
    }
    double m[3];
    {
        double V12[3], V14[3];
        FBUS_UNROLL
        for (int j = 0; j < 3; ++j) { V12[j] = P2[j] - P1[j]; V14[j] = P4[j] - P1[j]; }
        const double i12 = rsqrt_d(V12[0] * V12[0] + V12[1] * V12[1] + V12[2] * V12[2]);
        const double i14 = rsqrt_d(V14[0] * V14[0] + V14[1] * V14[1] + V14[2] * V14[2]);
        FBUS_UNROLL
        for (int j = 0; j < 3; ++j) m[j] = V12[j] * i12 + V14[j] * i14;
    }
    // Rm = AngleAxisd(-REF_M_PI/4, Z).matrix() (Rodrigues, SURVEY A.1-3) ; X = Rm*m/|m|
    double X[3];
    {
        const double sa[3] = {rod_s * Z[0], rod_s * Z[1], rod_s * Z[2]};
        const double ca[3] = {(1 - rod_c) * Z[0], (1 - rod_c) * Z[1], (1 - rod_c) * Z[2]};
        double Rm[9];
        double tmp;
        tmp = ca[0] * Z[1]; Rm[1] = tmp - sa[2]; Rm[3] = tmp + sa[2];
        tmp = ca[0] * Z[2]; Rm[2] = tmp + sa[1]; Rm[6] = tmp - sa[1];
        tmp = ca[1] * Z[2]; Rm[5] = tmp - sa[0]; Rm[7] = tmp + sa[0];
        Rm[0] = ca[0] * Z[0] + rod_c; Rm[4] = ca[1] * Z[1] + rod_c; Rm[8] = ca[2] * Z[2] + rod_c;
        double Rmm[3];
        mat3_vec(Rm, m, Rmm);
        const double im = rsqrt_d(m[0] * m[0] + m[1] * m[1] + m[2] * m[2]);
        FBUS_UNROLL
        for (int j = 0; j < 3; ++j) X[j] = Rmm[j] * im;
    }
    const double Y[3] = {Z[1] * X[2] - Z[2] * X[1], Z[2] * X[0] - Z[0] * X[2], Z[0] * X[1] - Z[1] * X[0]};
    const double R[9] = {X[0], Y[0], Z[0], X[1], Y[1], Z[1], X[2], Y[2], Z[2]};
    R2q(R, q);
    p[0] = P1[0]; p[1] = P1[1]; p[2] = P1[2];
}

}  // namespace fbus

// -------------------------------------------------------------------------------------------------
// N4: cv::fisheye::undistortPoints with R = P = identity (OpenCV 3.4.3 semantics, the version the reference links):
//   pw = ((u-cx)/fx, (v-cy)/fy); theta_d = |pw| clamped to [-pi/2, pi/2]; Newton on
//   theta (1 + k1 th^2 + k2 th^4 + k3 th^6 + k4 th^8) = theta_d (at most 10 iterations, |step| < 1e-8 stops);
//   out = pw * tan(theta)/theta_d, rounded to float32 (cv::Point2f).
// -------------------------------------------------------------------------------------------------
namespace fbus {
FBUS_HD void undistort_fisheye_point(const double* K4, const double* D4, double u, double v, float* xo, float* yo) {
    const double px = (u - K4[2]) / K4[0], py = (v - K4[3]) / K4[1];
    double scale = 1.0;
    double theta_d = sqrt(px * px + py * py);
    const double half_pi = 1.5707963267948966;  // CV_PI / 2 (OpenCV's own constant, not the reference's truncated M_PI)
    theta_d = theta_d < -half_pi ? -half_pi : (theta_d > half_pi ? half_pi : theta_d);
    if (theta_d > 1e-8) {
        double theta = theta_d;
        for (int j = 0; j < 10; ++j) {
            const double t2 = theta * theta, t4 = t2 * t2, t6 = t4 * t2, t8 = t6 * t2;
            const double k0 = D4[0] * t2, k1 = D4[1] * t4, k2 = D4[2] * t6, k3 = D4[3] * t8;
            const double fix = (theta * (1 + k0 + k1 + k2 + k3) - theta_d) / (1 + 3 * k0 + 5 * k1 + 7 * k2 + 9 * k3);
            theta = theta - fix;
            if ((fix < 0 ? -fix : fix) < 1e-8) break;
        }
        scale = tan(theta) / theta_d;
    }
    *xo = (float)(px * scale);
    *yo = (float)(py * scale);
}
}  // namespace fbus

// -------------------------------------------------------------------------------------------------
// N3: in-air stereo triangulation, VISION::NormalTriangulation (vision.cpp:395-466): homogeneous DLT
//   A = [ [xL]x [I|0] ; [xR]x T_L_R ]  (6x4),  P = right singular vector of the smallest singular value.
// That vector is the eigenvector of the smallest eigenvalue of the symmetric 4x4 A^T A, found here by cyclic Jacobi
// rotations (the reference uses Eigen's JacobiSVD; the result is a direction, its sign cancels in P[0:3]/P[3]).
// -------------------------------------------------------------------------------------------------
namespace fbus {

FBUS_HD void smallest_eigvec_sym4(double* A /*[16], destroyed*/, double* v) {
    double V[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    for (int sweep = 0; sweep < 10; ++sweep) {
        FBUS_UNROLL
        for (int p = 0; p < 3; ++p)
            FBUS_UNROLL
            for (int q = p + 1; q < 4; ++q) {
                const double apq = A[p * 4 + q];
                const double app = A[p * 4 + p], aqq = A[q * 4 + q];
                // rotation angle: tan(2 phi) = 2 apq / (aqq - app); stable t = sgn(th) / (|th| + sqrt(th^2 + 1))
                double c = 1.0, sn = 0.0;
                if (apq != 0.0) {
                    const double th = (aqq - app) / (2.0 * apq);
                    const double t = (th >= 0 ? 1.0 : -1.0) / ((th >= 0 ? th : -th) + sqrt(th * th + 1.0));
                    c = rsqrt_d(t * t + 1.0);
                    sn = t * c;
                }
                FBUS_UNROLL
                for (int k = 0; k < 4; ++k) {  // A <- A J
                    const double akp = A[k * 4 + p], akq = A[k * 4 + q];
                    A[k * 4 + p] = c * akp - sn * akq;
                    A[k * 4 + q] = sn * akp + c * akq;
                }
                FBUS_UNROLL
                for (int k = 0; k < 4; ++k) {  // A <- J^T A
                    const double apk = A[p * 4 + k], aqk = A[q * 4 + k];
                    A[p * 4 + k] = c * apk - sn * aqk;
                    A[q * 4 + k] = sn * apk + c * aqk;
                }
                FBUS_UNROLL
                for (int k = 0; k < 4; ++k) {
                    const double vkp = V[k * 4 + p], vkq = V[k * 4 + q];
                    V[k * 4 + p] = c * vkp - sn * vkq;
                    V[k * 4 + q] = sn * vkp + c * vkq;
                }
            }
    }
    // column of the smallest diagonal entry (static selects: no dynamic register indexing)
    const double d0 = A[0], d1 = A[5], d2 = A[10], d3 = A[15];
    const bool s1 = d1 < d0;
    const double m01 = s1 ? d1 : d0;
    const bool s3 = d3 < d2;
    const double m23 = s3 ? d3 : d2;
    const bool hi = m23 < m01;
    FBUS_UNROLL
    for (int k = 0; k < 4; ++k) {
        const double a = s1 ? V[k * 4 + 1] : V[k * 4 + 0];
        const double b = s3 ? V[k * 4 + 3] : V[k * 4 + 2];
        v[k] = hi ? b : a;
    }
}

// one stereo corner pair (undistorted normalised coordinates) -> corner in the flipped left frame with z > 0;
// returns |P| for the range gate, or -1 when the homogeneous coordinate vanishes (the reference `continue`s)
FBUS_HD double triangulate_corner_inair(const DevConsts& k, double xl, double yl, double xr, double yr, double* Pout) {
    // rows of [x]x M for x = (x, y, 1):  ( -M1 + y M2,  M0 - x M2,  -y M0 + x M1 )  with M's rows M0, M1, M2
    double A[24];
    {   // left: M = [I | 0]
        const double M0[4] = {1, 0, 0, 0}, M1[4] = {0, 1, 0, 0}, M2[4] = {0, 0, 1, 0};
        FBUS_UNROLL
        for (int c = 0; c < 4; ++c) {
            A[0 * 4 + c] = -M1[c] + yl * M2[c];
            A[1 * 4 + c] = M0[c] - xl * M2[c];
            A[2 * 4 + c] = -yl * M0[c] + xl * M1[c];
        }
    }
    FBUS_UNROLL
    for (int c = 0; c < 4; ++c) {
        const double m0 = k.T_LR_air[c], m1 = k.T_LR_air[4 + c], m2 = k.T_LR_air[8 + c];
        A[3 * 4 + c] = -m1 + yr * m2;
        A[4 * 4 + c] = m0 - xr * m2;
        A[5 * 4 + c] = -yr * m0 + xr * m1;
    }
    double G[16];
    FBUS_UNROLL
    for (int i = 0; i < 4; ++i)
        FBUS_UNROLL
        for (int j = i; j < 4; ++j) {
            double s = 0.0;
            FBUS_UNROLL
            for (int r = 0; r < 6; ++r) s += A[r * 4 + i] * A[r * 4 + j];
            G[i * 4 + j] = s;
            G[j * 4 + i] = s;
        }
    double P[4];
    smallest_eigvec_sym4(G, P);
    if (P[3] == 0.0) { Pout[0] = 0; Pout[1] = 0; Pout[2] = 0; return -1.0; }
    const double iw = 1.0 / P[3];
    const double Pn[3] = {-P[0] * iw, -P[1] * iw, P[2] * iw};  // R_I_C = diag(-1,-1,1)
    const double sg = signum_ref(Pn[2]);
    Pout[0] = sg * Pn[0]; Pout[1] = sg * Pn[1]; Pout[2] = sg * Pn[2];
    return norm3(Pn);
}

}  // namespace fbus

// =================================================================================================
// R3 (north_star; NOT in the reference -> "parity unpinned"): Gauss-Newton refinement of the marker pose.
// Minimises sum over 4 corners x 2 cameras of | pi_refr(x_c) - u |^2 over (R_M, p) in the flipped left-camera frame,
// seeded by the closed-form solve above.  pi_refr = flat-port forward projection (air -> glass -> water): solve the
// monotone equation  d0 t(s0) + d1 t(k1 s0) + (Z-d0-d1) t(k2 s0) = rho,  t(s) = s/sqrt(1-s^2),  for s0 = sin(theta_air)
// (SURVEY A.1-4); Jacobian by the implicit-function theorem (SURVEY A.6).  Right perturbation R_M <- R_M Exp(dphi).
// =================================================================================================
#ifndef FBUS_GN_UNROLL_ON
#define FBUS_GN_UNROLL_ON 0  // 1: inline all 8 projections of a Gauss-Newton iteration (warm starts in registers)
#endif
#ifndef FBUS_GN_NEWTON_TOL
#define FBUS_GN_NEWTON_TOL 1e-7
#endif
#if FBUS_GN_UNROLL_ON
#define FBUS_GN_UNROLL FBUS_UNROLL
#else
#define FBUS_GN_UNROLL _Pragma("unroll 1")
#endif
namespace fbus {

struct GnConsts {
    double d0, d1, k1, k2;       // air / glass thickness, n_air/n_glass, n_air/n_water
    double R_RL_inv[9], P_LR[3];  // TRUE inverse of R_RL (the calibration is ~2.5e-6 non-orthonormal, SURVEY A.3-5)
    double size;                  // marker side (0.28 m, vision.hpp:114)
    double tol;                   // > 0: stop iterating once an applied step is below this in every component (fbus_config.gn_tol)
};

// projects X (camera frame) -> uv (2) and, when JAC, the 2x3 Jacobian d(uv)/dX (row-major J[0..2] = du/dX,
// J[3..5] = dv/dX).  s_io: warm start for s0 = sin(theta_air) (<= 0: straight-line guess) and, on return, the root --
// the Gauss-Newton loop carries it from one iteration to the next, where the pose moves by ~the pixel noise and Newton
// needs two steps instead of six.
// FAST: stop Newton one evaluation early (see the loop); exact root for uv, 1e-9-relative Jacobian -- for the GN loop.
template <bool JAC = true, bool FAST = false>
FBUS_HD void project_refr(const GnConsts& g, const double* X, double* uv, double* J, double& s_io) {
    const double rho2 = X[0] * X[0] + X[1] * X[1];
    const double Zw = X[2] - g.d0 - g.d1;
    const double rho = sqrt(rho2);
    if (rho < 1e-12) {  // paraxial limit
        const double den = 1.0 / (g.d0 + g.k1 * g.d1 + g.k2 * Zw);
        uv[0] = X[0] * den; uv[1] = X[1] * den;
        if (JAC) {
            J[0] = den; J[1] = 0.0; J[2] = -X[0] * den * den * g.k2;
            J[3] = 0.0; J[4] = den; J[5] = -X[1] * den * den * g.k2;
        }
        s_io = 0.0;
        return;
    }
    // Newton on f(s) = d0 t(s) + d1 t(k1 s) + Zw t(k2 s) - rho.  f is increasing and convex on [0,1): from any start
    // the first step lands right of the root and the iteration then decreases monotonically to it; the only safeguard
    // needed is to stay inside the domain.  The loop leaves with r0,r1,r2 evaluated AT the accepted s.
    double s = (s_io > 0.0 && s_io < 1.0) ? s_io : rho * rsqrt_d(rho2 + X[2] * X[2]);
    const double k1s = g.k1 * g.k1, k2s = g.k2 * g.k2, a1 = g.d1 * g.k1, a2 = Zw * g.k2;
    double r0, r1, r2, gs, ds = 0.0;
    for (int it = 0; it < 50; ++it) {
        const double s2 = s * s;
        if (FAST) {  // 1e-13-accurate reciprocal roots are enough inside the GN loop (tau inherits that error, parity needs 1e-8)
            r0 = rsqrt_d1(1.0 - s2); r1 = rsqrt_d1(1.0 - k1s * s2); r2 = rsqrt_d1(1.0 - k2s * s2);
        } else {
            r0 = rsqrt_d(1.0 - s2); r1 = rsqrt_d(1.0 - k1s * s2); r2 = rsqrt_d(1.0 - k2s * s2);
        }
        gs = g.d0 * (r0 * r0) * r0 + a1 * (r1 * r1) * r1 + a2 * (r2 * r2) * r2;
        const double f = s * (g.d0 * r0 + a1 * r1 + a2 * r2) - rho;
        double sn = s - f * rcp_d(gs);
        if (!(sn < 1.0)) sn = 0.5 * (s + 1.0);
        if (!(sn > 0.0)) sn = 0.5 * s;
        ds = sn - s;
        // |ds| <= 1e-7 s: the Newton step that follows would move s by ~ds^2 (1e-14 s): sn is the root to rounding.
        // r0..gs were evaluated at s = sn - ds; tau below is corrected to first order (error ~ t'' ds^2 / 2 < 1e-12),
        // the Jacobian keeps a 1e-9 relative error, which only perturbs the GN step by 1e-9 of its length.
        if ((ds < 0 ? -ds : ds) <= (FAST ? FBUS_GN_NEWTON_TOL : 4.5e-16) * s) break;
        s = sn;
        ds = 0.0;
    }
    s_io = s + ds;
    const double t0 = s * r0 + (r0 * r0) * r0 * ds;
    const double ir = rcp_d(rho);
    const double xh = X[0] * ir, yh = X[1] * ir;
    uv[0] = t0 * xh; uv[1] = t0 * yh;
    if (JAC) {
        const double t2 = g.k2 * s * r2, dt0 = (r0 * r0) * r0;
        const double a = t0 * ir;      // tau / rho
        const double igs = rcp_d(gs);
        const double b = dt0 * igs;    // t'(s0) / g_s
        J[0] = a * (1.0 - xh * xh) + b * xh * xh; J[1] = (b - a) * xh * yh;
        J[3] = J[1];                               J[4] = a * (1.0 - yh * yh) + b * yh * yh;
        const double cz = -dt0 * t2 * igs;
        J[2] = cz * xh; J[5] = cz * yh;
    }
}
FBUS_HD void project_refr(const GnConsts& g, const double* X, double* uv, double* J) {
    double s = 0.0;
    project_refr<true, false>(g, X, uv, J, s);
}

// residuals and normal equations for pose (Rm row-major 3x3, p) against the 16 observed coordinates c[16]
// (Lx0,Ly0..Lx3,Ly3,Rx0..Ry3).  H: 6x6 lower-packed J^T J, gvec: J^T r, returns the cost sum r^2.  sw[8]: Newton warm
// starts per (corner, camera), carried across Gauss-Newton iterations.  JAC = false: cost only (H, gvec untouched).
template <bool JAC = true>
FBUS_HD double gn_normal_eq(const GnConsts& g, const double* c, const double* Rm, const double* p, double* H, double* gvec, double* sw) {
    if (JAC) {
        FBUS_UNROLL
        for (int i = 0; i < 21; ++i) H[i] = 0.0;
        FBUS_UNROLL
        for (int i = 0; i < 6; ++i) gvec[i] = 0.0;
    }
    double cost = 0.0;
    FBUS_GN_UNROLL
    for (int i = 0; i < 4; ++i) {
        const double cx = (i == 1 || i == 2) ? g.size : 0.0, cy = (i >= 2) ? g.size : 0.0;  // corners (0,0),(s,0),(s,s),(0,s), z = 0
        const double XL[3] = {-(p[0] + Rm[0] * cx + Rm[1] * cy), -(p[1] + Rm[3] * cx + Rm[4] * cy), p[2] + Rm[6] * cx + Rm[7] * cy};  // un-flip: F = diag(-1,-1,1)
        // d XL / d(dp) = F ; d XL / d(dphi) = -F Rm [cm]x, and with cm = (cx, cy, 0):
        //   (Rm [cm]x)[r][:] = (-Rm[r][2] cy, Rm[r][2] cx, Rm[r][0] cy - Rm[r][1] cx)
        double Dr[9];  // rotation part of D (3 x 3); the translation part is F itself
        FBUS_UNROLL
        for (int r = 0; r < 3; ++r) {
            const double fs = (r < 2) ? -1.0 : 1.0;
            Dr[r * 3 + 0] = fs * (Rm[r * 3 + 2] * cy);
            Dr[r * 3 + 1] = -fs * (Rm[r * 3 + 2] * cx);
            Dr[r * 3 + 2] = -fs * (Rm[r * 3 + 0] * cy - Rm[r * 3 + 1] * cx);
        }
        FBUS_GN_UNROLL
        for (int cam = 0; cam < 2; ++cam) {
            double X[3];
            if (cam == 0) {
                FBUS_UNROLL
                for (int r = 0; r < 3; ++r) X[r] = XL[r];
            } else {
                const double dL[3] = {XL[0] - g.P_LR[0], XL[1] - g.P_LR[1], XL[2] - g.P_LR[2]};
                mat3_vec(g.R_RL_inv, dL, X);
            }
            double uv[2], Jp[6];
            project_refr<JAC, true>(g, X, uv, Jp, sw[cam * 4 + i]);
            const double ru = uv[0] - c[cam * 8 + 2 * i], rv = uv[1] - c[cam * 8 + 2 * i + 1];
            cost += ru * ru;
            cost += rv * rv;
            if (!JAC) continue;
            // G = d(uv)/d(XL) (2 x 3): Jp for the left camera, Jp R_RL^-1 for the right one
            double G[6];
            if (cam == 0) {
                FBUS_UNROLL
                for (int e = 0; e < 6; ++e) G[e] = Jp[e];
            } else {
                FBUS_UNROLL
                for (int r = 0; r < 2; ++r)
                    FBUS_UNROLL
                    for (int e = 0; e < 3; ++e) {
                        double t = Jp[r * 3] * g.R_RL_inv[e];
                        t += Jp[r * 3 + 1] * g.R_RL_inv[3 + e];
                        t += Jp[r * 3 + 2] * g.R_RL_inv[6 + e];
                        G[r * 3 + e] = t;
                    }
            }
            // J = G [F | Dr]
            double Ju[6], Jv[6];
            Ju[0] = -G[0]; Ju[1] = -G[1]; Ju[2] = G[2];
            Jv[0] = -G[3]; Jv[1] = -G[4]; Jv[2] = G[5];
            FBUS_UNROLL
            for (int e = 0; e < 3; ++e) {
                double tu = G[0] * Dr[e], tv = G[3] * Dr[e];
                tu += G[1] * Dr[3 + e]; tv += G[4] * Dr[3 + e];
                tu += G[2] * Dr[6 + e]; tv += G[5] * Dr[6 + e];
                Ju[3 + e] = tu; Jv[3 + e] = tv;
            }
            FBUS_UNROLL
            for (int a = 0; a < 6; ++a) {
                gvec[a] += Ju[a] * ru;
                gvec[a] += Jv[a] * rv;
                FBUS_UNROLL
                for (int b = 0; b <= a; ++b) {
                    H[a * (a + 1) / 2 + b] += Ju[a] * Ju[b];
                    H[a * (a + 1) / 2 + b] += Jv[a] * Jv[b];
                }
            }
        }
    }
    return cost;
}

FBUS_HD double gn_normal_eq(const GnConsts& g, const double* c, const double* Rm, const double* p, double* H, double* gvec) {
    double sw[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    return gn_normal_eq<true>(g, c, Rm, p, H, gvec, sw);
}

// Gauss-Newton iterations; Rm, p updated in place; returns the final cost (sum of squared residuals) when FINAL_COST
// (one more residual evaluation), else the cost at the start of the last iteration.
template <bool FINAL_COST = true>
FBUS_HD double gn_refine(const GnConsts& g, const double* c, double* Rm, double* p, int iters) {
    double cost = 0.0;
    // Newton warm starts: the seed pose reproduces the observed corners to ~the pixel noise, so the observed pixel's
    // own air angle sin(theta) = |uv| / sqrt(1 + |uv|^2) is within ~1e-4 of the root of the first projection
    double sw[8];
    FBUS_UNROLL
    for (int e = 0; e < 8; ++e) {
        const double r2 = c[2 * e] * c[2 * e] + c[2 * e + 1] * c[2 * e + 1];
        sw[e] = sqrt(r2) * rsqrt_d(1.0 + r2);
    }
    for (int it = 0; it < iters; ++it) {
        double H[21], gv[6], Li[6], d[6];
        cost = gn_normal_eq<true>(g, c, Rm, p, H, gv, sw);
        CholStep<6, 0>::run(H, Li);
        // solve H d = -g
        FBUS_UNROLL
        for (int i = 0; i < 6; ++i) {
            double s = -gv[i];
            FBUS_UNROLL
            for (int j = 0; j < i; ++j) s -= H[i * (i + 1) / 2 + j] * d[j];
            d[i] = s * Li[i];
        }
        FBUS_UNROLL
        for (int i = 5; i >= 0; --i) {
            double s = d[i];
            FBUS_UNROLL
            for (int j = i + 1; j < 6; ++j) s -= H[j * (j + 1) / 2 + i] * d[j];
            d[i] = s * Li[i];
        }
        p[0] += d[0]; p[1] += d[1]; p[2] += d[2];
        // Rm <- Rm Exp(dphi)  (Rodrigues)
        const double th2 = d[3] * d[3] + d[4] * d[4] + d[5] * d[5];
        const double th = sqrt(th2);
        double A, Bc;  // Exp = I + A [phi]x + Bc [phi]x^2
        if (th < 1e-8) { A = 1.0 - th2 / 6.0; Bc = 0.5 - th2 / 24.0; }
        else { double sn, cs; sincos(th, &sn, &cs); A = sn / th; Bc = (1.0 - cs) / th2; }
        const double x = d[3], y = d[4], z = d[5];
        const double E[9] = {1.0 - Bc * (y * y + z * z), -A * z + Bc * x * y, A * y + Bc * x * z,
                             A * z + Bc * x * y, 1.0 - Bc * (x * x + z * z), -A * x + Bc * y * z,
                             -A * y + Bc * x * z, A * x + Bc * y * z, 1.0 - Bc * (x * x + y * y)};
        double Rn[9];
        FBUS_UNROLL
        for (int r = 0; r < 3; ++r)
            FBUS_UNROLL
            for (int cc = 0; cc < 3; ++cc) Rn[r * 3 + cc] = Rm[r * 3] * E[cc] + Rm[r * 3 + 1] * E[3 + cc] + Rm[r * 3 + 2] * E[6 + cc];
        FBUS_UNROLL
        for (int e = 0; e < 9; ++e) Rm[e] = Rn[e];
        if (g.tol > 0.0) {  // converged: the step just applied is below the tolerance (a warp goes on until its last lane is)
            double dn = fabs(d[0]);
            FBUS_UNROLL
            for (int i = 1; i < 6; ++i) dn = fmax(dn, fabs(d[i]));
            if (dn < g.tol) break;
        }
    }
    if (FINAL_COST) cost = gn_normal_eq<false>(g, c, Rm, p, nullptr, nullptr, sw);
    return cost;
}

// closed-form seed as a rotation matrix + position (same algebra as marker_pose, which returns the quaternion)
FBUS_HD void quat_to_rotmat_unit(const double* q, double* R) {
    double qn[4] = {q[0], q[1], q[2], q[3]};
    qnormalize(qn);
    q2R(qn, R);
}

// Forward model of one marker (fbus_marker_project): pose[7] = p xyz, q wxyz of corner 0 in the flipped left-camera frame ->
// uv[16] = left (x,y) of corners 0..3, then right, the input layout of the solves.  Corner geometry and un-flip as in
// gn_normal_eq; underwater: right camera through R_RL_inv / P_LR and the exact (non-FAST) flat-port projection; in air: the
// pinhole geometry of VISION::NormalTriangulation, x_R ~ T_LR_air [X_L; 1].  Returns false, with all 16 outputs NaN, when a
// corner lies at or behind the port (Z <= d_air + d_glass underwater, Z <= 0 in air) in either camera's frame.
FBUS_HD bool project_marker(const DevConsts& k, const GnConsts& g, int underwater, const double* pose, double* uv) {
    double Rm[9];
    quat_to_rotmat_unit(pose + 3, Rm);
    const double zmin = underwater ? g.d0 + g.d1 : 0.0;
    bool ok = true;
    for (int i = 0; i < 4 && ok; ++i) {
        const double cx = (i == 1 || i == 2) ? g.size : 0.0, cy = (i >= 2) ? g.size : 0.0;
        const double XL[3] = {-(pose[0] + Rm[0] * cx + Rm[1] * cy), -(pose[1] + Rm[3] * cx + Rm[4] * cy), pose[2] + Rm[6] * cx + Rm[7] * cy};
        for (int cam = 0; cam < 2; ++cam) {
            double X[3];
            if (cam == 0) {
                X[0] = XL[0]; X[1] = XL[1]; X[2] = XL[2];
            } else if (underwater) {
                const double dL[3] = {XL[0] - g.P_LR[0], XL[1] - g.P_LR[1], XL[2] - g.P_LR[2]};
                mat3_vec(g.R_RL_inv, dL, X);
            } else {
                FBUS_UNROLL
                for (int r = 0; r < 3; ++r)
                    X[r] = k.T_LR_air[r * 4] * XL[0] + k.T_LR_air[r * 4 + 1] * XL[1] + k.T_LR_air[r * 4 + 2] * XL[2] + k.T_LR_air[r * 4 + 3];
            }
            if (!(X[2] > zmin)) { ok = false; break; }  // also catches a non-finite pose
            double* o = uv + cam * 8 + 2 * i;
            if (underwater) {
                double s = 0.0;
                project_refr<false, false>(g, X, o, nullptr, s);
            } else {
                o[0] = X[0] / X[2];
                o[1] = X[1] / X[2];
            }
        }
    }
    if (!ok) {
        FBUS_UNROLL
        for (int e = 0; e < 16; ++e) uv[e] = (double)NAN;
    }
    return ok;
}

}  // namespace fbus
