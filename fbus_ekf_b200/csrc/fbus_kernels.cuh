// fbus_kernels.cuh -- CUDA kernels of the batched FBUS-EKF hot path (sm_100a).
//
//   (K12, the fused window kernel ekf_window_split_kernel, lives in fbus_kernel_split.cuh; this header holds the
//   parameter block it shares with the host and every other kernel)
//   init_gravity_kernel K0 : FILTER::InitializeGravityAndBias (filter.cpp:256-285)
//   refract_kernel      K3+K4: RefractionTriangulation + ComputeMarkerPose (vision.cpp:472-759)
//   marker_pose_kernel  K4 alone
//   stats_kernel / stats_reduce_kernel, filter_errors_kernel, synth_kernel, fp64_peak_kernel: measurement support.
//
// Thread mapping: one thread per filter (or per marker); filter index fastest in every array, so a warp
// reads/writes 32 consecutive doubles (256 B) per field.
#pragma once

#include <cuda_runtime.h>

#include "fbus_math.cuh"
#include "fbus_refract.cuh"

namespace fbus {

constexpr int NOM_FIELDS = 37;  // t q4 R9 p3 v3 ba3 bg3 g3 pv3 qv4 + t_img (MATLAB-semantics mode: time of the previous image frame)
enum NomField { F_T = 0, F_Q = 1, F_R = 5, F_P = 14, F_V = 17, F_BA = 20, F_BG = 23, F_G = 26, F_PV = 29, F_QV = 32, F_TIMG = 36 };

enum WinMode { M_INIT = 1, M_RESET = 2, M_PROP = 4, M_UPDATE = 8, M_FUSED = 16 };

struct WinParams {
    double* nom;       // [36][B]
    double* P;         // [171][B]
    int32_t* prev_id;  // [B]
    int32_t* init;     // [B]
    int32_t* status;   // [B]
    size_t B;
    const double* imu_t;      // device [N]
    const double* imu;        // [N][6][B]  FBUS_IMU_F64_SI (nullptr when imu32 is set)
    const float* imu32;       // [N][6][B]  FBUS_IMU_F32_SENSOR: accel in g, gyro in deg/s, or nullptr
    const double* det_t;      // device [W]
    const int32_t* det_id;    // [W][m][B]
    const double* det_pose;   // [W][m][7][B]
    const uint32_t* win_off;  // device [W+1] (fused mode)
    const MarkerTable* tab;   // device: marker map
    double* trace;            // [w1-w0][17][B] or nullptr
    uint32_t w0, w1;
    int32_t m;     // marker slots per frame
    int32_t mode;  // WinMode mask
    // un-fused propagate
    uint32_t prop_first, prop_count;
    double prop_t_end;
    uint32_t n_imu_before;  // un-fused init
    uint32_t* cursor_io;      // [B] fused mode: index of the first IMU sample a filter has not consumed yet (written at the end)
    int32_t cursor_resume;    // fused mode: start from cursor_io (continuation of the same stream) instead of win_off[w0]
    uint32_t stagger_cycles;  // split kernel, 2 CTAs per SM: start delay of odd-ticket CTAs
    uint32_t* sm_ticket;      // split kernel: per-SM arrival counters [256] (device), or nullptr
    uint32_t lane_fpc;        // second-generation lane kernel: filters per CTA (1..32); the other slots of a CTA stay idle
};

// One IMU component (c = 0..2 accel, 3..5 gyro).  Float32 sensor samples are converted exactly as the reference's IMU callback
// does before it builds IMUData (main.cpp:254): accel = (double)a * g, gyro = (double)(w / 180.f) * M_PI with the reference's
// M_PI = 3.1415926 (common.hpp:14).  The float division is IEEE and the products are rounded on their own (__dmul_rn: the
// compiler must not contract them into an FMA with whatever consumes the sample), so the filter sees the same doubles as
// the reference.
__device__ __forceinline__ double imu_cvt(float f, int c, double imu_g) {
    return (c < 3) ? __dmul_rn((double)f, imu_g) : __dmul_rn((double)__fdiv_rn(f, 180.0f), 3.1415926);
}
// format decided at run time (one-off kernels)
__device__ __forceinline__ double imu_sample(const double* imu, const float* imu32, double imu_g, size_t i, int c, size_t B, size_t b) {
    const size_t idx = (i * 6 + (size_t)c) * B + b;
    return imu32 != nullptr ? imu_cvt(imu32[idx], c, imu_g) : imu[idx];
}
// format decided at compile time (the hot window kernels have one instantiation per format)
template <bool IMU32, class PRM>
__device__ __forceinline__ double imu_sample_t(const PRM& prm, double imu_g, size_t i, int c, size_t B, size_t b) {
    const size_t idx = (i * 6 + (size_t)c) * B + b;
    if constexpr (IMU32) return imu_cvt(prm.imu32[idx], c, imu_g);
    else return prm.imu[idx];
}

// FILTER::SetImuData's 1-pole IIR (filter.cpp:36-48): one thread per (channel, filter) walks the samples in order; the
// recurrence is two rounded products and a rounded sum per sample (no FMA contraction: the reference has none).  Loads do not
// depend on the recurrence, so the unrolled loop keeps several in flight.
__global__ void iir_prefilter_kernel(const double* imu, const float* imu32, double imu_g, size_t B, uint32_t first, uint32_t count, double* out) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= 6 * B || count == 0) return;
    const int c = (int)(idx / B);
    const size_t b = idx % B;
    const double keep = 1.0 - 0.1, gain = 0.1;  // (1 - filter_coeff), filter_coeff
    double prev = imu_sample(imu, imu32, imu_g, first, c, B, b);
    out[(size_t)c * B + b] = prev;
#pragma unroll 4
    for (uint32_t i = 1; i < count; ++i) {
        const double raw = imu_sample(imu, imu32, imu_g, (size_t)first + i, c, B, b);
        prev = __dadd_rn(__dmul_rn(prev, keep), __dmul_rn(raw, gain));
        out[((size_t)i * 6 + c) * B + b] = prev;
    }
}

// K0: FILTER::InitializeGravityAndBias (filter.cpp:256-285)
__global__ void init_gravity_kernel(double* nom, size_t B, const double* imu, const float* imu32, double imu_g, uint32_t first, uint32_t count) {
    const size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B || count == 0) return;
    double am[3] = {0, 0, 0}, gm[3] = {0, 0, 0};
    for (uint32_t i = first; i < first + count; ++i) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            am[c] = am[c] + imu_sample(imu, imu32, imu_g, i, c, B, b);
            gm[c] = gm[c] + imu_sample(imu, imu32, imu_g, i, 3 + c, B, b);
        }
    }
    const double nn = (double)count;
    double a[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        nom[(size_t)(F_BG + c) * B + b] = gm[c] / nn;
        a[c] = am[c] / nn;
    }
    nom[(size_t)(F_G + 0) * B + b] = 0.0;
    nom[(size_t)(F_G + 1) * B + b] = 0.0;
    nom[(size_t)(F_G + 2) * B + b] = -norm3(a);
}

// FILTER::FILTER (filter.hpp:63-137): P0 diagonal, identity quaternion, everything else zero
__global__ void ctor_kernel(double* nom, double* P, int32_t* prev_id, int32_t* init, int32_t* status, size_t B,
                            double p0, double p1, double p2, double p3, double p4, double p5) {
    const size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    for (int f = 0; f < NOM_FIELDS; ++f) nom[(size_t)f * B + b] = (f == F_Q || f == F_QV) ? 1.0 : 0.0;
    const double p0d[6] = {p0, p1, p2, p3, p4, p5};
    for (int i = 0; i < NX; ++i)
        for (int j = i; j < NX; ++j) P[(size_t)pidx_u(i, j) * B + b] = (i == j) ? p0d[i / 3] : 0.0;
    prev_id[b] = 0;
    init[b] = 0;
    status[b] = 0;
}

// K3+K4: one thread per marker.  corners [16][n] float32 -> pose [7][n], corners3d [12][n], valid [n]
#ifndef FBUS_REFRACT_MINB
#define FBUS_REFRACT_MINB 6  // measured: 9.72e9 solves/s with 6 CTAs/SM (80 regs) vs 9.39e9 with 5 (82 regs), 9.06e9 with 8 (64 regs, spills)
#endif
__global__ void __launch_bounds__(128, FBUS_REFRACT_MINB) refract_kernel(const __grid_constant__ DevConsts k, const float* __restrict__ corners, size_t n, size_t ld,
                                                      double* __restrict__ pose, double* __restrict__ c3d, int32_t* __restrict__ valid) {
    // n markers of arrays whose rows are ld apart (ld = n for a whole array; a chunk of a larger one otherwise)
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float c[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) c[e] = corners[(size_t)e * ld + i];
    double C[12];
    bool dead = false;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        double Pc[3];
        const double nrm = triangulate_corner(k, (double)c[2 * e], (double)c[2 * e + 1], (double)c[8 + 2 * e], (double)c[8 + 2 * e + 1], Pc);
        // the reference breaks out of the corner loop at the first out-of-range corner (vision.cpp:602-606)
        C[3 * e] = dead ? 0.0 : Pc[0];
        C[3 * e + 1] = dead ? 0.0 : Pc[1];
        C[3 * e + 2] = dead ? 0.0 : Pc[2];
        if (nrm > k.dect_thres) dead = true;
    }
    double p[3] = {0, 0, 0}, q[4] = {1, 0, 0, 0};
    if (!dead) marker_pose(C, k.rod_s, k.rod_c, p, q);
#pragma unroll
    for (int e = 0; e < 3; ++e) pose[(size_t)e * ld + i] = p[e];
#pragma unroll
    for (int e = 0; e < 4; ++e) pose[(size_t)(3 + e) * ld + i] = q[e];
    if (c3d) {
#pragma unroll
        for (int e = 0; e < 12; ++e) c3d[(size_t)e * ld + i] = C[e];
    }
    if (valid) valid[i] = dead ? 0 : 1;
}

// N4: fisheye undistortion of the detected corner pixels; one thread per marker (16 coordinates)
__global__ void __launch_bounds__(128) undistort_kernel(const __grid_constant__ DevConsts k, const float* __restrict__ px, size_t n,
                                                        float* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const int cam = e >> 2;
        float xo, yo;
        undistort_fisheye_point(k.cam_k[cam], k.cam_d[cam], (double)px[(size_t)(2 * e) * n + i], (double)px[(size_t)(2 * e + 1) * n + i], &xo, &yo);
        out[(size_t)(2 * e) * n + i] = xo;
        out[(size_t)(2 * e + 1) * n + i] = yo;
    }
}

// N3+K4: in-air stereo DLT triangulation (VISION::NormalTriangulation, vision.cpp:395-466) + ComputeMarkerPose
__global__ void __launch_bounds__(128) inair_kernel(const __grid_constant__ DevConsts k, const float* __restrict__ corners, size_t n, size_t ld,
                                                    double* __restrict__ pose, double* __restrict__ c3d, int32_t* __restrict__ valid) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float c[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) c[e] = corners[(size_t)e * ld + i];
    double C[12];
    bool dead = false;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        double Pc[3];
        const double nrm = triangulate_corner_inair(k, (double)c[2 * e], (double)c[2 * e + 1], (double)c[8 + 2 * e], (double)c[8 + 2 * e + 1], Pc);
        C[3 * e] = dead ? 0.0 : Pc[0];
        C[3 * e + 1] = dead ? 0.0 : Pc[1];
        C[3 * e + 2] = dead ? 0.0 : Pc[2];
        if (nrm > k.dect_thres) dead = true;  // break at the first out-of-range corner (vision.cpp:451-455)
    }
    double p[3] = {0, 0, 0}, q[4] = {1, 0, 0, 0};
    if (!dead) marker_pose(C, k.rod_s, k.rod_c, p, q);
#pragma unroll
    for (int e = 0; e < 3; ++e) pose[(size_t)e * ld + i] = p[e];
#pragma unroll
    for (int e = 0; e < 4; ++e) pose[(size_t)(3 + e) * ld + i] = q[e];
    if (c3d) {
#pragma unroll
        for (int e = 0; e < 12; ++e) c3d[(size_t)e * ld + i] = C[e];
    }
    if (valid) valid[i] = dead ? 0 : 1;
}

// K3+K4+K5: closed-form solve, then Gauss-Newton refinement of the pose on the stereo reprojection error (R3)
#ifndef FBUS_GN_MINB
#define FBUS_GN_MINB 4  // measured on B200: 4 CTAs/SM (128 regs, small spills) beats 2 CTAs/SM at 216 regs by 12 %
#endif
template <typename CT>
__global__ void __launch_bounds__(128, FBUS_GN_MINB) refract_gn_kernel(const __grid_constant__ DevConsts k, const __grid_constant__ GnConsts g,
                                                         const CT* __restrict__ corners, size_t n, int iters, double* __restrict__ pose,
                                                         double* __restrict__ cost_out, int32_t* __restrict__ valid) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double c[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) c[e] = (double)corners[(size_t)e * n + i];
    double C[12];
    bool dead = false;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        double Pc[3];
        const double nrm = triangulate_corner(k, c[2 * e], c[2 * e + 1], c[8 + 2 * e], c[8 + 2 * e + 1], Pc);
        C[3 * e] = Pc[0]; C[3 * e + 1] = Pc[1]; C[3 * e + 2] = Pc[2];
        if (nrm > k.dect_thres) dead = true;
    }
    double p[3] = {0, 0, 0}, q[4] = {1, 0, 0, 0}, cost = 0.0;
    if (!dead) {
        marker_pose(C, k.rod_s, k.rod_c, p, q);
        double Rm[9];
        quat_to_rotmat_unit(q, Rm);
        cost = gn_refine(g, c, Rm, p, iters);
        R2q(Rm, q);
    }
#pragma unroll
    for (int e = 0; e < 3; ++e) pose[(size_t)e * n + i] = p[e];
#pragma unroll
    for (int e = 0; e < 4; ++e) pose[(size_t)(3 + e) * n + i] = q[e];
    if (cost_out) cost_out[i] = cost;
    if (valid) valid[i] = dead ? 0 : 1;
}

// Vision front-end -> filter hand-off in one kernel (what VisionThreadFunction does between DetectArucoTag and
// SetDetectionResult, vision.cpp:60-139): triangulate (refractive or in-air), marker pose, optional GN refinement, and
// write the result straight into the detection-frame layout of fbus_det_frames: item i = (frame*m + slot)*B + filter,
// pose element e at ((i / B) * 7 + e) * B + i % B, id = marker id or -1 when the marker was rejected (only markers
// with isComputePose enter the DetectionResultList, vision.cpp:88-99).
__global__ void __launch_bounds__(128, FBUS_GN_MINB) solve_to_det_kernel(const __grid_constant__ DevConsts k, const __grid_constant__ GnConsts g,
                                                           const float* __restrict__ corners, const int32_t* __restrict__ ids_in, size_t n,
                                                           size_t B, int underwater, int iters, int32_t* __restrict__ det_id,
                                                           double* __restrict__ det_pose) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int id = ids_in[i];
    double c[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) c[e] = (double)corners[(size_t)e * n + i];
    double C[12];
    bool dead = id < 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        double Pc[3];
        const double nrm = underwater ? triangulate_corner(k, c[2 * e], c[2 * e + 1], c[8 + 2 * e], c[8 + 2 * e + 1], Pc)
                                      : triangulate_corner_inair(k, c[2 * e], c[2 * e + 1], c[8 + 2 * e], c[8 + 2 * e + 1], Pc);
        C[3 * e] = Pc[0]; C[3 * e + 1] = Pc[1]; C[3 * e + 2] = Pc[2];
        if (nrm > k.dect_thres) dead = true;
    }
    double p[3] = {0, 0, 0}, q[4] = {1, 0, 0, 0};
    if (!dead) {
        marker_pose(C, k.rod_s, k.rod_c, p, q);
        if (underwater && iters > 0) {
            double Rm[9];
            quat_to_rotmat_unit(q, Rm);
            gn_refine<false>(g, c, Rm, p, iters);
            R2q(Rm, q);
        }
    }
    det_id[i] = dead ? -1 : id;
    double* out = det_pose + (i / B) * 7 * B + (i % B);
#pragma unroll
    for (int e = 0; e < 3; ++e) out[(size_t)e * B] = p[e];
#pragma unroll
    for (int e = 0; e < 4; ++e) out[(size_t)(3 + e) * B] = q[e];
}

__global__ void __launch_bounds__(128) marker_pose_kernel(const __grid_constant__ DevConsts k, const double* __restrict__ c3d, size_t n,
                                                          double* __restrict__ pose) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double C[12], p[3], q[4];
#pragma unroll
    for (int e = 0; e < 12; ++e) C[e] = c3d[(size_t)e * n + i];
    marker_pose(C, k.rod_s, k.rod_c, p, q);
#pragma unroll
    for (int e = 0; e < 3; ++e) pose[(size_t)e * n + i] = p[e];
#pragma unroll
    for (int e = 0; e < 4; ++e) pose[(size_t)(3 + e) * n + i] = q[e];
}

// ---- statistics: per-block partial sums, then a fixed-order final reduce (deterministic) ----------
// Error of filter b against the truth, declared into the enclosing scope: ep2 = |p - p_true|^2, et2 = |dtheta|^2
// (dtheta = 2 sign(dq_w) dq_xyz of dq = conj(q) q_true), nees = e^T P6^-1 e over (p, theta) with 6 dof, ok = false when the
// (p, theta) block of P is not positive definite.  One definition for stats_kernel (which sums the terms) and
// filter_errors_kernel (which writes them per filter).  A macro, not an inline function: inlining the same code changed
// stats_kernel's register allocation and instruction schedule, and the statistics kernel is kept exactly as it was.
#define FBUS_FILTER_ERROR_TERMS(nom, P, B, b, truth_p, truth_q)    \
        double e[6], q[4], qt[4], dq[4]; \
_Pragma("unroll") \
        for (int c = 0; c < 3; ++c) e[c] = nom[(size_t)(F_P + c) * B + b] - truth_p[(size_t)c * B + b]; \
_Pragma("unroll") \
        for (int c = 0; c < 4; ++c) { q[c] = nom[(size_t)(F_Q + c) * B + b]; qt[c] = truth_q[(size_t)c * B + b]; } \
        const double cq[4] = {q[0], -q[1], -q[2], -q[3]}; \
        qmul(cq, qt, dq); \
        const double sg = dq[0] < 0 ? -1.0 : 1.0; \
_Pragma("unroll") \
        for (int c = 0; c < 3; ++c) e[3 + c] = 2.0 * sg * dq[1 + c]; \
        const int ix[6] = {0, 1, 2, 6, 7, 8}; \
        double L[36]; \
        bool ok = true; \
_Pragma("unroll") \
        for (int j = 0; j < 6; ++j) { \
            double s = P[(size_t)pidx(ix[j], ix[j]) * B + b]; \
_Pragma("unroll") \
            for (int c = 0; c < j; ++c) s -= L[j * 6 + c] * L[j * 6 + c]; \
            if (!(s > 0.0)) ok = false; \
            const double d = sqrt(s); \
            L[j * 6 + j] = d; \
_Pragma("unroll") \
            for (int i = j + 1; i < 6; ++i) { \
                double s2 = P[(size_t)pidx(ix[i], ix[j]) * B + b]; \
_Pragma("unroll") \
                for (int c = 0; c < j; ++c) s2 -= L[i * 6 + c] * L[j * 6 + c]; \
                L[i * 6 + j] = s2 / d; \
            } \
        } \
        double y[6], nees = 0.0; \
_Pragma("unroll") \
        for (int i = 0; i < 6; ++i) { \
            double s = e[i]; \
_Pragma("unroll") \
            for (int c = 0; c < i; ++c) s -= L[i * 6 + c] * y[c]; \
            y[i] = s / L[i * 6 + i]; \
            nees += y[i] * y[i]; \
        } \
        const double ep2 = e[0] * e[0] + e[1] * e[1] + e[2] * e[2]; \
        const double et2 = e[3] * e[3] + e[4] * e[4] + e[5] * e[5];
constexpr int STATS_BS = 128;
__global__ void __launch_bounds__(STATS_BS) stats_kernel(const double* nom, const double* P, size_t B, const double* truth_p,
                                                         const double* truth_q, double* partial /*[grid][8]*/) {
    __shared__ double red[STATS_BS][6];
    const size_t b = (size_t)blockIdx.x * STATS_BS + threadIdx.x;
    double v[6] = {0, 0, 0, 0, 0, 0};  // ep2, et2, nees, n_ok, n_bad, max_ep
    if (b < B) {
        FBUS_FILTER_ERROR_TERMS(nom, P, B, b, truth_p, truth_q)
        if (ok && isfinite(ep2) && isfinite(et2) && isfinite(nees)) {
            v[0] = ep2; v[1] = et2; v[2] = nees; v[3] = 1.0; v[5] = sqrt(ep2);
        } else {
            v[4] = 1.0;
        }
    }
#pragma unroll
    for (int c = 0; c < 6; ++c) red[threadIdx.x][c] = v[c];
    __syncthreads();
    for (int s = STATS_BS / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) {
#pragma unroll
            for (int c = 0; c < 5; ++c) red[threadIdx.x][c] += red[threadIdx.x + s][c];
            red[threadIdx.x][5] = fmax(red[threadIdx.x][5], red[threadIdx.x + s][5]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
#pragma unroll
        for (int c = 0; c < 6; ++c) partial[(size_t)blockIdx.x * 8 + c] = red[0][c];
    }
}
__global__ void stats_reduce_kernel(const double* partial, int nblk, double* out /*[8]*/) {
    __shared__ double red[256][6];
    double v[6] = {0, 0, 0, 0, 0, 0};
    for (int i = threadIdx.x; i < nblk; i += 256) {
#pragma unroll
        for (int c = 0; c < 5; ++c) v[c] += partial[(size_t)i * 8 + c];
        v[5] = fmax(v[5], partial[(size_t)i * 8 + 5]);
    }
#pragma unroll
    for (int c = 0; c < 6; ++c) red[threadIdx.x][c] = v[c];
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) {
#pragma unroll
            for (int c = 0; c < 5; ++c) red[threadIdx.x][c] += red[threadIdx.x + s][c];
            red[threadIdx.x][5] = fmax(red[threadIdx.x][5], red[threadIdx.x + s][5]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
#pragma unroll
        for (int c = 0; c < 6; ++c) out[c] = red[0][c];
        out[6] = 0.0; out[7] = 0.0;
    }
}

// the per-filter terms stats_kernel sums: out[0][b] = |p - p_true|^2, [1][b] = |dtheta|^2, [2][b] = NEES (6 dof), [3][b] = 1.0
// when all are finite and P6 is positive definite, else 0.0 (rows 0..2 then hold whatever was computed)
__global__ void __launch_bounds__(STATS_BS) filter_errors_kernel(const double* nom, const double* P, size_t B, const double* truth_p,
                                                                 const double* truth_q, double* out /*[4][B]*/) {
    const size_t b = (size_t)blockIdx.x * STATS_BS + threadIdx.x;
    if (b >= B) return;
    FBUS_FILTER_ERROR_TERMS(nom, P, B, b, truth_p, truth_q)
    out[b] = ep2;
    out[B + b] = et2;
    out[2 * B + b] = nees;
    out[3 * B + b] = (ok && isfinite(ep2) && isfinite(et2) && isfinite(nees)) ? 1.0 : 0.0;
}

// ---- synthetic Monte-Carlo streams: Philox4x32-10 counter RNG --------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
// two independent N(0,1) from one Philox call (Box-Muller on two 53-bit uniforms)
__device__ __forceinline__ void normal2(uint64_t seed, uint64_t filt, uint32_t idx, uint32_t stream, double* z0, double* z1) {
    uint32_t r[4];
    philox4x32_10((uint32_t)filt, (uint32_t)(filt >> 32), idx, stream, (uint32_t)seed, (uint32_t)(seed >> 32), r);
    const uint64_t a = ((uint64_t)r[0] << 32) | r[1], bb = ((uint64_t)r[2] << 32) | r[3];
    const double u1 = ((double)(a >> 11) + 1.0) * (1.0 / 9007199254740992.0);  // (0,1]
    const double u2 = (double)(bb >> 11) * (1.0 / 9007199254740992.0);        // [0,1)
    const double rad = sqrt(-2.0 * log(u1));
    double s, c;
    sincospi(2.0 * u2, &s, &c);
    *z0 = rad * c;
    *z1 = rad * s;
}
struct SynthParams {
    size_t B, N, W;
    const double* base_imu;   // device [N][6]
    const double* base_pose;  // device [W][7]
    double* imu;              // [N][6][B]
    int32_t* det_id;          // [W][1][B]
    double* det_pose;         // [W][1][7][B]
    double* bias_out;         // [6][B] or nullptr
    double s_acc, s_gyro, s_ba, s_bg, s_pos, s_quat;
    uint64_t seed, filter_offset;
    int32_t marker_id, pad;
};
__global__ void __launch_bounds__(128) synth_kernel(const __grid_constant__ SynthParams sp) {
    const size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= sp.B) return;
    const uint64_t gf = sp.filter_offset + b;
    double bias[6];
    {
        double z[6];
        normal2(sp.seed, gf, 0u, 0u, &z[0], &z[1]);
        normal2(sp.seed, gf, 0u, 1u, &z[2], &z[3]);
        normal2(sp.seed, gf, 0u, 2u, &z[4], &z[5]);
#pragma unroll
        for (int c = 0; c < 3; ++c) { bias[c] = sp.s_ba * z[c]; bias[3 + c] = sp.s_bg * z[3 + c]; }
        if (sp.bias_out) {
#pragma unroll
            for (int c = 0; c < 6; ++c) sp.bias_out[(size_t)c * sp.B + b] = bias[c];
        }
    }
    for (size_t i = 0; i < sp.N; ++i) {
        double z[6];
        normal2(sp.seed, gf, (uint32_t)i, 16u, &z[0], &z[1]);
        normal2(sp.seed, gf, (uint32_t)i, 17u, &z[2], &z[3]);
        normal2(sp.seed, gf, (uint32_t)i, 18u, &z[4], &z[5]);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            sp.imu[(i * 6 + c) * sp.B + b] = sp.base_imu[i * 6 + c] + bias[c] + sp.s_acc * z[c];
            sp.imu[(i * 6 + 3 + c) * sp.B + b] = sp.base_imu[i * 6 + 3 + c] + bias[3 + c] + sp.s_gyro * z[3 + c];
        }
    }
    for (size_t w = 0; w < sp.W; ++w) {
        double z[8];
        normal2(sp.seed, gf, (uint32_t)w, 32u, &z[0], &z[1]);
        normal2(sp.seed, gf, (uint32_t)w, 33u, &z[2], &z[3]);
        normal2(sp.seed, gf, (uint32_t)w, 34u, &z[4], &z[5]);
        normal2(sp.seed, gf, (uint32_t)w, 35u, &z[6], &z[7]);
        sp.det_id[w * sp.B + b] = sp.marker_id;
        double q[4];
#pragma unroll
        for (int c = 0; c < 3; ++c) sp.det_pose[(w * 7 + c) * sp.B + b] = sp.base_pose[w * 7 + c] + sp.s_pos * z[c];
#pragma unroll
        for (int c = 0; c < 4; ++c) q[c] = sp.base_pose[w * 7 + 3 + c] + sp.s_quat * z[3 + c];
        qnormalize(q);
#pragma unroll
        for (int c = 0; c < 4; ++c) sp.det_pose[(w * 7 + 3 + c) * sp.B + b] = q[c];
    }
}

// ---- forward model and per-filter stereo corner streams (fbus_marker_project, fbus_synth_corners) ----------------------
// One thread per marker: pose element e of marker i at pose[e * ld_e + i * ld_i] (ld_e = n, ld_i = 1: the [7][n] layout of
// fbus_marker_project; ld_e = 1, ld_i = 7: the [n][7] rows of fbus_corner_spec.base_pose) -> corners [16][n], valid [n] or null
__global__ void __launch_bounds__(128) marker_project_kernel(const __grid_constant__ DevConsts k, const __grid_constant__ GnConsts g,
                                                             const double* __restrict__ pose, size_t n, size_t ld_e, size_t ld_i, int underwater,
                                                             double* __restrict__ corners, int32_t* __restrict__ valid) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double ps[7], uv[16];
#pragma unroll
    for (int e = 0; e < 7; ++e) ps[e] = pose[(size_t)e * ld_e + i * ld_i];
    const bool ok = project_marker(k, g, underwater, ps, uv);
#pragma unroll
    for (int e = 0; e < 16; ++e) corners[(size_t)e * n + i] = uv[e];
    if (valid) valid[i] = ok ? 1 : 0;
}

// Philox streams of fbus_synth_corners: slot s draws from streams CORNER_STREAM0 + CORNER_STREAM_STRIDE * s + d, d = 0..7 the
// white noise (coordinates 2d, 2d+1), 8 the drop / outlier uniforms, 9..16 the outlier normals.  All >= 64: disjoint from
// synth_kernel's streams 0-2, 16-18 and 32-35, so one seed drives both generators independently.
constexpr uint32_t CORNER_STREAM0 = 64u, CORNER_STREAM_STRIDE = 32u;
struct CornerSynthParams {
    size_t B, m, n;              // n = (w1 - w0) * m * B items, item ((w - w0) * m + slot) * B + b
    size_t w0;                   // global index of the first frame (the Philox counter uses global frames)
    const double* base;          // device [16][(w1 - w0) * m]: noise-free corners of each (frame, slot)
    const int32_t* base_id;      // device [(w1 - w0) * m]: marker id, < 0 = empty slot
    const int32_t* base_valid;   // device [(w1 - w0) * m]: projection valid
    float* corners;              // [16][n]
    int32_t* ids;                // [n]
    double s_corner, p_drop, p_out, s_out;
    uint64_t seed, filter_offset;
};
__device__ __forceinline__ double uniform53(uint32_t hi, uint32_t lo) {  // [0,1)
    return (double)((((uint64_t)hi << 32) | lo) >> 11) * (1.0 / 9007199254740992.0);
}
__global__ void __launch_bounds__(128) synth_corners_kernel(const __grid_constant__ CornerSynthParams sp) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= sp.n) return;
    const size_t ws = i / sp.B, b = i % sp.B;  // (frame, slot) of this chunk; filter
    const uint32_t w = (uint32_t)(sp.w0 + ws / sp.m);
    const uint32_t st = CORNER_STREAM0 + CORNER_STREAM_STRIDE * (uint32_t)(ws % sp.m);
    const uint64_t gf = sp.filter_offset + b;
    const size_t nws = sp.n / sp.B;
    int32_t id = sp.base_valid[ws] ? sp.base_id[ws] : -1;
    bool outlier = false;
    if (id >= 0) {
        uint32_t r[4];
        philox4x32_10((uint32_t)gf, (uint32_t)(gf >> 32), w, st + 8u, (uint32_t)sp.seed, (uint32_t)(sp.seed >> 32), r);
        if (uniform53(r[0], r[1]) < sp.p_drop) id = -1;
        else outlier = uniform53(r[2], r[3]) < sp.p_out;
    }
    sp.ids[i] = id;
    if (id < 0) {
#pragma unroll
        for (int e = 0; e < 16; ++e) sp.corners[(size_t)e * sp.n + i] = 0.0f;
        return;
    }
    double c[16];
#pragma unroll
    for (int d = 0; d < 8; ++d) {
        double z0, z1;
        normal2(sp.seed, gf, w, st + (uint32_t)d, &z0, &z1);
        c[2 * d] = sp.base[(size_t)(2 * d) * nws + ws] + sp.s_corner * z0;
        c[2 * d + 1] = sp.base[(size_t)(2 * d + 1) * nws + ws] + sp.s_corner * z1;
    }
    if (outlier) {
#pragma unroll
        for (int d = 0; d < 8; ++d) {
            double z0, z1;
            normal2(sp.seed, gf, w, st + 9u + (uint32_t)d, &z0, &z1);
            c[2 * d] += sp.s_out * z0;
            c[2 * d + 1] += sp.s_out * z1;
        }
    }
#pragma unroll
    for (int e = 0; e < 16; ++e) sp.corners[(size_t)e * sp.n + i] = (float)c[e];
}

// ---- FP64 FMA peak microbenchmark: 8 independent DFMA chains per thread ----------------------------
__global__ void __launch_bounds__(256) fp64_peak_kernel(double* out, int iters, double seed) {
    double a0 = seed, a1 = seed + 1, a2 = seed + 2, a3 = seed + 3, a4 = seed + 4, a5 = seed + 5, a6 = seed + 6, a7 = seed + 7;
    const double m = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
            a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
        }
    }
    const double s = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (s == 123.456) out[blockIdx.x * blockDim.x + threadIdx.x] = s;  // never true; keeps the chain alive
}

}  // namespace fbus
