// fbus_kernel_lane.cuh -- K12 for SMALL batches: the fused window kernel with NINE LANES PER FILTER.
//
// Why: with one thread per filter a batch of a few thousand filters cannot fill 148 SMs -- 4 096 filters are 128 warps of
// covariance work, each a serial chain of ~660 dependent-ish FP64 instructions per IMU sample, and the throughput is the
// per-filter latency times the batch (0.47e6 filter-steps/s per filter whatever the CTA shape, profiles/probes/RESULTS.md).
// Here the covariance of ONE filter is spread over nine lanes of a warp (three filters per warp, 27 of 32 lanes busy):
//
//   lane l (0..8) of a filter owns the FULL columns l and l+9 of the symmetric 18x18 covariance in registers (36 doubles).
//
//   propagate  P <- F P F^T + Qbar   (FILTER::UpdateCovariance, filter.cpp:588-616) in two applications of the same
//     column operator  y = F x  (33 FMA: rows 0..8 change, F = I + the six small blocks of filter.cpp:598-604):
//       A.  M[:, j] = F P[:, j]            for both own columns                      (local)
//       T.  the top nine entries of both columns go to shared memory, lane l reads ROW l of M back   (18 st + 18 ld)
//       B.  P'[:, l] = F (row l of M)^T    -- by symmetry of P this is column l of F P F^T; its rows 9..17 are
//           copies of M[l][9..17], i.e. bit-identical to what the lanes owning columns 9..17 hold, and column l+9 of P'
//           is M[:, l+9] as it stands.
//     Only the top-left 9x9 is evaluated in two association orders (P'[i][j] by lane j, P'[j][i] by lane i); it is
//     symmetrised once per frame (the reference symmetrises after every step, filter.cpp:614-615; the difference is at the
//     rounding level and bounded by the window length).
//   update     (FILTER::ObservationUpdate, filter.cpp:622-739): the NOMINAL warp (one lane per filter, 32 filters) runs
//     the state-only prologue of the structured update (update_prologue in fbus_math.cuh: predicted measurement, Hs, S,
//     Cholesky, C = Hs^T S^-1 Hs = Lc Lc^T, y) from the 6x6 block P6 the lanes publish; the lanes then form their two
//     columns of Z = Lc^T G locally (G = rows {0,1,2,6,7,8} of P = six entries of each own column), exchange the Z
//     columns through shared memory and sweep  P -= Z^T Z  (exactly symmetric by construction) and  dx = Z^T y.
//
// The nominal warp is the one of the two-warp kernel (fbus_kernel_split.cuh, nominal_role<.., LANE = true>): detection scan,
// F6b / F5, F2, the streams, one IMU sample ahead of the covariance lanes through the same two-deep coefficient ring.
// CTA = 32 filters = 11 covariance warps + 1 nominal warp = 384 threads, every barrier CTA-wide.
//
// This is the layout north_star sketches ("one warp or warp-group per filter with P held in registers and shared memory");
// the thread-per-filter kernels stay for every batch that fills the GPU, where they execute 1.6x fewer FP64
// warp-instructions per filter-step.
#pragma once

#include "fbus_kernel_split.cuh"

namespace fbus {

constexpr int LANE_TS = 19;               // row stride of the per-filter transpose scratch (18 + 1: bank-conflict-free row reads)
constexpr int LANE_T = 9 * LANE_TS;       // doubles of transpose scratch per filter
constexpr size_t LANE_SMEM = (size_t)(LX_TOTAL * 32 + LANE_T * 32) * sizeof(double);

// y = F x on one column (rows 0..8 change):  filter.cpp:598-604 with A = -R[a]x dt, B = -R dt and W = F[theta,theta] - I in
// full (-[w]x dt for the C++ semantics, expm(-[w]x dt) - I for the MATLAB ones: the nominal warp decides, the lanes just apply it)
__device__ __forceinline__ void lane_apply_F(double* x, const double* A, const double* Bm, const double* W, double dt) {
    double y[9];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        double s = x[i];
        s += dt * x[3 + i];
        y[i] = s;
        double t = x[3 + i];
        t += dt * x[15 + i];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            t += A[i * 3 + c] * x[6 + c];
            t += Bm[i * 3 + c] * x[9 + c];
        }
        y[3 + i] = t;
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        double t = x[6 + i];
        t -= dt * x[12 + i];
#pragma unroll
        for (int c = 0; c < 3; ++c) t += W[i * 3 + c] * x[6 + c];
        y[6 + i] = t;
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) x[i] = y[i];
}

// y = F x on TWO columns at once with F[theta,theta] - I = -[w]x dt given by u = w dt (C++ semantics only: 30 FMA per column), written
// term by term across all eighteen results (the same products in the same order per result as lane_apply_F): with few warps per scheduler every dependent FP64 instruction costs its full 8-clock latency, and ptxas keeps the
// source order of independent chains, so the independent results are advanced together instead of one after the other
__device__ __forceinline__ void lane_apply_Fu2(double* x, double* z, const double* A, const double* Bm, double u0, double u1, double u2, double dt) {
    double px[3], pz[3], vx[3], vz[3], tx[3], tz[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        vx[i] = x[3 + i]; vz[i] = z[3 + i];
        px[i] = x[i];     pz[i] = z[i];
        tx[i] = x[6 + i]; tz[i] = z[6 + i];
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) { vx[i] += dt * x[15 + i]; vz[i] += dt * z[15 + i]; }
#pragma unroll
    for (int i = 0; i < 3; ++i) { px[i] += dt * x[3 + i]; pz[i] += dt * z[3 + i]; }
#pragma unroll
    for (int i = 0; i < 3; ++i) { tx[i] -= dt * x[12 + i]; tz[i] -= dt * z[12 + i]; }
#pragma unroll
    for (int i = 0; i < 3; ++i) { vx[i] += A[i * 3] * x[6]; vz[i] += A[i * 3] * z[6]; }
    tx[0] += u2 * x[7]; tz[0] += u2 * z[7]; tx[1] -= u2 * x[6]; tz[1] -= u2 * z[6]; tx[2] += u1 * x[6]; tz[2] += u1 * z[6];
#pragma unroll
    for (int i = 0; i < 3; ++i) { vx[i] += Bm[i * 3] * x[9]; vz[i] += Bm[i * 3] * z[9]; }
    tx[0] -= u1 * x[8]; tz[0] -= u1 * z[8]; tx[1] += u0 * x[8]; tz[1] += u0 * z[8]; tx[2] -= u0 * x[7]; tz[2] -= u0 * z[7];
#pragma unroll
    for (int i = 0; i < 3; ++i) { vx[i] += A[i * 3 + 1] * x[7]; vz[i] += A[i * 3 + 1] * z[7]; }
#pragma unroll
    for (int i = 0; i < 3; ++i) { vx[i] += Bm[i * 3 + 1] * x[10]; vz[i] += Bm[i * 3 + 1] * z[10]; }
#pragma unroll
    for (int i = 0; i < 3; ++i) { vx[i] += A[i * 3 + 2] * x[8]; vz[i] += A[i * 3 + 2] * z[8]; }
#pragma unroll
    for (int i = 0; i < 3; ++i) { vx[i] += Bm[i * 3 + 2] * x[11]; vz[i] += Bm[i * 3 + 2] * z[11]; }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        x[i] = px[i]; x[3 + i] = vx[i]; x[6 + i] = tx[i];
        z[i] = pz[i]; z[3 + i] = vz[i]; z[6 + i] = tz[i];
    }
}
// one column, term by term
__device__ __forceinline__ void lane_apply_Fu1(double* x, const double* A, const double* Bm, double u0, double u1, double u2, double dt) {
    double px[3], vx[3], tx[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) { vx[i] = x[3 + i]; px[i] = x[i]; tx[i] = x[6 + i]; }
#pragma unroll
    for (int i = 0; i < 3; ++i) vx[i] += dt * x[15 + i];
#pragma unroll
    for (int i = 0; i < 3; ++i) px[i] += dt * x[3 + i];
#pragma unroll
    for (int i = 0; i < 3; ++i) tx[i] -= dt * x[12 + i];
#pragma unroll
    for (int i = 0; i < 3; ++i) vx[i] += A[i * 3] * x[6];
    tx[0] += u2 * x[7]; tx[1] -= u2 * x[6]; tx[2] += u1 * x[6];
#pragma unroll
    for (int i = 0; i < 3; ++i) vx[i] += Bm[i * 3] * x[9];
    tx[0] -= u1 * x[8]; tx[1] += u0 * x[8]; tx[2] -= u0 * x[7];
#pragma unroll
    for (int i = 0; i < 3; ++i) vx[i] += A[i * 3 + 1] * x[7];
#pragma unroll
    for (int i = 0; i < 3; ++i) vx[i] += Bm[i * 3 + 1] * x[10];
#pragma unroll
    for (int i = 0; i < 3; ++i) vx[i] += A[i * 3 + 2] * x[8];
#pragma unroll
    for (int i = 0; i < 3; ++i) vx[i] += Bm[i * 3 + 2] * x[11];
#pragma unroll
    for (int i = 0; i < 3; ++i) { x[i] = px[i]; x[3 + i] = vx[i]; x[6 + i] = tx[i]; }
}

// COVARIANCE lanes: warp cw (0..10) holds filters 3cw .. 3cw+2 of the CTA, lane = 9*g + l
// NOISE: q0, q1 come from this filter's row of the [6][B] buffer `noise` (fbus_set_noise) instead of k.Qd
// ALL: FBUS_FLAG_ALL_MARKERS -- after the first update of a frame, further update rounds follow until no filter of the CTA
// requests one (nominal_role posts one marker per filter and round)
// GATE: the innovation gate -- after (c) a filter's request is read again, the nominal lane has withdrawn a rejected one
template <bool JOSEPH, bool NOISE = false, bool ALL = false, bool GATE = false>
__device__ __forceinline__ void lane_cov_role(const WinParams& prm, const DevConsts& k, double* smem, SplitShared& sh, int32_t (*sflag)[32],
                                              int cw, int lane, const double* noise = nullptr) {
    constexpr int NT = LANE_NT;
    const size_t B = prm.B;
    const int g = lane / 9, l = lane - 9 * g;
    const int f0 = cw * 3 + g;
    const bool act = (g < 3) && (f0 < 32);
    const int f = act ? f0 : 31;  // idle lanes shadow filter 31 for their (unused) reads and never write
    const size_t b0 = (size_t)blockIdx.x * 32 + f;
    const bool live = act && b0 < B;
    const size_t b = (b0 < B) ? b0 : B - 1;
    double* const X = smem + f;                                   // exchange area, entry stride 32
    double* const T = smem + (size_t)LX_TOTAL * 32 + (size_t)f * LANE_T;  // transpose scratch of this filter
    // own columns l and l + 9 (full 18 entries each) from the packed upper triangle
    double c0[18], c1[18];
#pragma unroll
    for (int i = 0; i < 18; ++i) {
        const int a0 = i < l ? i : l, b0i = i < l ? l : i;            // (min, max) of (i, l)
        const int a1 = i < l + 9 ? i : l + 9, b1i = i < l + 9 ? l + 9 : i;
        c0[i] = prm.P[(size_t)(a0 * NX - (a0 * (a0 - 1)) / 2 + (b0i - a0)) * B + b];
        c1[i] = prm.P[(size_t)(a1 * NX - (a1 * (a1 - 1)) / 2 + (b1i - a1)) * B + b];
    }
    // process noise on the own diagonal entries (GammaQGamma^T is diagonal, filter.hpp:108-125): column l gets it in row l,
    // column l+9 in row l+9
    double q0 = (l >= 3 && l < 6) ? k.Qd[0] : (l >= 6 ? k.Qd[1] : 0.0);
    double q1 = (l < 3) ? k.Qd[2] : (l < 6 ? k.Qd[3] : 0.0);
    if constexpr (NOISE) {  // this filter's own values
        q0 = (l >= 3 && l < 6) ? noise[b] : (l >= 6 ? noise[B + b] : 0.0);
        q1 = (l < 3) ? noise[2 * B + b] : (l < 6 ? noise[3 * B + b] : 0.0);
    }
    for (uint32_t w = prm.w0; w < prm.w1; ++w) {
        cta_bar<NT>();  // (a) the nominal warp has posted the IMU range
        const int fp = (int)((w - prm.w0) & 1u);
        const uint32_t lo = sh.lo_hi[fp][0][0], hi = sh.lo_hi[fp][1][0];
        bool touched = false;
        for (uint32_t i = lo; i < hi; ++i) {
            cta_bar<NT>();  // record (i) is complete; the nominal warp moves on to sample i+1
            const int slot = (int)((i - lo) & 1u);
            const bool valid = act && sflag[slot][f] != 0;
            const double* rec = X + (size_t)slot * LX_REC * 32;
            double A[9], Bm[9], Wm[9];
#pragma unroll
            for (int e = 0; e < 9; ++e) { A[e] = rec[(size_t)e * 32]; Bm[e] = rec[(size_t)(9 + e) * 32]; Wm[e] = rec[(size_t)(18 + e) * 32]; }
            const double dt = rec[(size_t)27 * 32];
            if (valid) {  // A: M = F P on both columns
                lane_apply_F(c0, A, Bm, Wm, dt);
                lane_apply_F(c1, A, Bm, Wm, dt);
#pragma unroll
                for (int r = 0; r < 9; ++r) {  // T: publish the rows of M that change
                    T[r * LANE_TS + l] = c0[r];
                    T[r * LANE_TS + 9 + l] = c1[r];
                }
            }
            __syncwarp();
            if (valid) {  // B: column l of F P F^T = F (row l of M)^T
#pragma unroll
                for (int c = 0; c < 18; ++c) c0[c] = T[l * LANE_TS + c];
                lane_apply_F(c0, A, Bm, Wm, dt);
#pragma unroll
                for (int r = 3; r < 9; ++r) c0[r] += (r == l) ? q0 : 0.0;
#pragma unroll
                for (int r = 9; r < 15; ++r) c1[r] += (r == l + 9) ? q1 : 0.0;
                touched = true;
            }
            __syncwarp();  // the row reads are done before the next sample's publish
        }
        if (__any_sync(0xffffffffu, touched)) {  // symmetrise the top-left 9x9 (the only part evaluated in two orders)
            if (touched) {
#pragma unroll
                for (int r = 0; r < 9; ++r) T[r * LANE_TS + l] = c0[r];
            }
            __syncwarp();
            if (touched) {
#pragma unroll
                for (int r = 0; r < 9; ++r) c0[r] = 0.5 * (c0[r] + T[l * LANE_TS + r]);
            }
            __syncwarp();
        }
        cta_bar<NT>();  // (r) update requests posted
        if (sh.any_upd[0]) {
            // ALL: one round per posted request (nominal_role), until a round without any
            do {
            const bool req = act && sflag[2][f] != 0;
            // the 6x6 block of the p / theta rows and columns for the prologue: lanes l in {0,1,2,6,7,8} own its columns
            if (req && (l < 3 || l >= 6)) {
                const int ci = l < 3 ? l : l - 3;
#pragma unroll
                for (int m = 0; m < 6; ++m) X[(size_t)(LX_P6 + m * 6 + ci) * 32] = c0[m < 3 ? m : m + 3];
            }
            cta_bar<NT>();  // (p) P6 published
            cta_bar<NT>();  // (c) the nominal warp has posted Lc and y
            bool upd = req;  // GATE: not withdrawn by the gate
            if constexpr (GATE) upd = req && sflag[2][f] != 0;
            // own columns of the factor Z with (I-KH)P = P - Z^T Z, dx = Z^T y:
            //   default  Z = X G   (7 x 18), X = L^-1 Hs, y = z = L^-1 r      (S = L L^T)
            //   Joseph   Z = Lc^T G (6 x 18), Lc Lc^T = C_J, y = Lc^-1 u       (update_prologue)
            constexpr int NZ = JOSEPH ? 6 : 7;
            double z0[NZ], z1[NZ];
            if (upd) {
                if constexpr (JOSEPH) {
                    double Cm[21];
#pragma unroll
                    for (int c = 0; c < 21; ++c) Cm[c] = X[(size_t)(LX_CM + c) * 32];
#pragma unroll
                    for (int kz = 0; kz < 6; ++kz) {
                        double s0 = Cm[kz * (kz + 1) / 2 + kz] * c0[kz < 3 ? kz : kz + 3];
                        double s1 = Cm[kz * (kz + 1) / 2 + kz] * c1[kz < 3 ? kz : kz + 3];
#pragma unroll
                        for (int m = kz + 1; m < 6; ++m) {
                            s0 += Cm[m * (m + 1) / 2 + kz] * c0[m < 3 ? m : m + 3];
                            s1 += Cm[m * (m + 1) / 2 + kz] * c1[m < 3 ? m : m + 3];
                        }
                        z0[kz] = s0;
                        z1[kz] = s1;
                    }
                } else {
#pragma unroll
                    for (int kz = 0; kz < 7; ++kz) {
                        double s0 = 0.0, s1 = 0.0;
#pragma unroll
                        for (int m = 0; m < 6; ++m) {
                            const double x = X[(size_t)(LX_SCR + kz * 6 + m) * 32];
                            s0 += x * c0[m < 3 ? m : m + 3];
                            s1 += x * c1[m < 3 ? m : m + 3];
                        }
                        z0[kz] = s0;
                        z1[kz] = s1;
                    }
                }
                double d0 = 0.0, d1 = 0.0;  // dx = Z^T y for the own columns
#pragma unroll
                for (int kz = 0; kz < NZ; ++kz) {
                    T[kz * LANE_TS + l] = z0[kz];
                    T[kz * LANE_TS + 9 + l] = z1[kz];
                    const double yk = X[(size_t)(LX_Y + kz) * 32];
                    d0 += yk * z0[kz];
                    d1 += yk * z1[kz];
                }
                X[(size_t)(LX_DX + l) * 32] = d0;
                X[(size_t)(LX_DX + 9 + l) * 32] = d1;
            }
            __syncwarp();  // the filter's Z columns are in its scratch
            if (upd) {
#pragma unroll
                for (int r = 0; r < 18; ++r) {  // P -= Z^T Z on both columns (exactly symmetric: the same products in the same order on both sides)
                    double v0 = c0[r], v1 = c1[r];
#pragma unroll
                    for (int kz = 0; kz < NZ; ++kz) {
                        const double zr = T[kz * LANE_TS + r];
                        v0 -= zr * z0[kz];
                        v1 -= zr * z1[kz];
                    }
                    c0[r] = v0;
                    c1[r] = v1;
                }
            }
            __syncwarp();
            cta_bar<NT>();  // (d) dx posted
            } while (ALL && (cta_bar<NT>(), sh.any_upd[0] != 0));  // (r) of the next round: does any filter request one?
        }
    }
    if (live) {  // upper triangle back: column j is stored by its owner for rows i <= j
#pragma unroll
        for (int i = 0; i < 18; ++i) {
            if (i <= l) prm.P[(size_t)(i * NX - (i * (i - 1)) / 2 + (l - i)) * B + b] = c0[i];
            if (i <= l + 9) prm.P[(size_t)(i * NX - (i * (i - 1)) / 2 + (l + 9 - i)) * B + b] = c1[i];
        }
    }
}

// NOISE: every filter has its own noise values, `noise` is the [6][B] buffer of fbus_set_noise (the other instantiations never
// read the parameter)
// ALL: FBUS_FLAG_ALL_MARKERS, every known marker of a frame updates the filter in turn (include/fbus_ekf.h)
// GATE: the innovation gate of fbus_set_gate, thresholds and counts in `gate` (the other instantiations never read the parameter)
template <bool JOSEPH, bool IMU32, bool MATLAB = false, bool NOISE = false, bool ALL = false, bool GATE = false>
__global__ void __launch_bounds__(LANE_NT, 1) ekf_window_lane_kernel(const __grid_constant__ WinParams prm, const __grid_constant__ DevConsts k,
                                                                     const double* __restrict__ noise, const GateBufs gate) {
    extern __shared__ double smem[];
    __shared__ SplitShared sh;
    __shared__ int32_t sflag[3][32];
    const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (wi < 11) {
        if constexpr (NOISE) lane_cov_role<JOSEPH, true, ALL, GATE>(prm, k, smem, sh, sflag, wi, lane, noise);
        else lane_cov_role<JOSEPH, false, ALL, GATE>(prm, k, smem, sh, sflag, wi, lane);
    } else {
        const size_t b0 = (size_t)blockIdx.x * 32 + lane;
        const bool live = b0 < prm.B;
        if constexpr (GATE)
            nominal_role<32, false, IMU32, true, JOSEPH, MATLAB, false, NOISE, ALL, true>(prm, k, smem, sh, sflag, lane, live ? b0 : prm.B - 1,
                                                                                          live, nullptr, nullptr, nullptr, noise, gate);
        else if constexpr (NOISE)
            nominal_role<32, false, IMU32, true, JOSEPH, MATLAB, false, true, ALL>(prm, k, smem, sh, sflag, lane, live ? b0 : prm.B - 1, live,
                                                                                   nullptr, nullptr, nullptr, noise);
        else nominal_role<32, false, IMU32, true, JOSEPH, MATLAB, false, false, ALL>(prm, k, smem, sh, sflag, lane, live ? b0 : prm.B - 1, live);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Second generation (C++ semantics; the MATLAB-semantics mode stays on the kernel above).
//
// What bounded the first generation was not the covariance lanes but the NOMINAL lane: F2 is a serial chain of ~380 instructions per
// sample (rsqrt, sincos, two quaternion products and normalisations, three rotation matrices), ~1 700 clk, and a filter-step could
// not be shorter.  Only a small part of that chain runs through the state: the increment quaternions depend on the sample, the biases
// and dt alone.  Here
//   * the covariance warps evaluate nominal_increment for a whole chunk of L2_CH samples at once (warp = sample slot, lane = filter)
//     before they start on the chunk's covariance steps,
//   * the nominal lane walks the remaining chain (two quaternion products, normalisations, rotation matrices, RK4 sums) and posts the
//     coefficients of F into a ring that holds the whole chunk, one named barrier per record (the nominal lanes arrive without waiting): no CTA-wide rendezvous per sample, the
//     covariance lanes of a filter follow their nominal lane at their own pace.
// Results are bit-identical to the first generation (the same expressions in the same order, split at values that are not contracted).
// ------------------------------------------------------------------------------------------------------------------
constexpr size_t LANE2_SMEM = (size_t)(L2_TOTAL * 32 + L2_RING + LANE_T * 32) * sizeof(double);

template <bool JOSEPH, bool IMU32, bool NOISE = false>  // NOISE: as lane_cov_role
__device__ __forceinline__ void lane2_cov_role(const WinParams& prm, const DevConsts& k, double* smem, SplitShared& sh, int32_t (*sflag)[32],
                                               Lane2Shared& l2, int cw, int lane, const double* noise = nullptr) {
    constexpr int NT = LANE_NT;
    const size_t B = prm.B;
    const int g = lane / 9, l = lane - 9 * g;
    const int f0 = cw * 3 + g;
    const bool act = (g < 3) && (f0 < 32);
    const int f = act ? f0 : 31;  // idle lanes shadow filter 31 for their (unused) reads and never write
    const size_t b0 = (size_t)blockIdx.x * prm.lane_fpc + f;
    const bool live = act && f < (int)prm.lane_fpc && b0 < B;
    const size_t b = (b0 < B) ? b0 : B - 1;
    double* const X = smem + f;                                   // exchange area, entry stride 32
    const double* const ring = smem + (size_t)L2_TOTAL * 32;                                  // [slot][filter][L2_RS]
    double* const T = smem + (size_t)L2_TOTAL * 32 + L2_RING + (size_t)f * LANE_T;            // transpose scratch of this filter
    // increment pass: this warp is sample slot cw of the chunk, this lane is filter `lane` of the CTA
    double* const XI = smem + lane;
    const size_t bi0 = (size_t)blockIdx.x * prm.lane_fpc + lane;
    const size_t bi = (bi0 < B) ? bi0 : B - 1;
    double c0[18], c1[18];
#pragma unroll
    for (int i = 0; i < 18; ++i) {
        const int a0 = i < l ? i : l, b0i = i < l ? l : i;            // (min, max) of (i, l)
        const int a1 = i < l + 9 ? i : l + 9, b1i = i < l + 9 ? l + 9 : i;
        c0[i] = prm.P[(size_t)(a0 * NX - (a0 * (a0 - 1)) / 2 + (b0i - a0)) * B + b];
        c1[i] = prm.P[(size_t)(a1 * NX - (a1 * (a1 - 1)) / 2 + (b1i - a1)) * B + b];
    }
    double q0 = (l >= 3 && l < 6) ? k.Qd[0] : (l >= 6 ? k.Qd[1] : 0.0);
    double q1 = (l < 3) ? k.Qd[2] : (l < 6 ? k.Qd[3] : 0.0);
    if constexpr (NOISE) {  // this filter's own values
        q0 = (l >= 3 && l < 6) ? noise[b] : (l >= 6 ? noise[B + b] : 0.0);
        q1 = (l < 3) ? noise[2 * B + b] : (l < 6 ? noise[3 * B + b] : 0.0);
    }
    // the sample this warp's slot will most likely hold in the NEXT chunk (the one right behind the current chunk), loaded a whole
    // chunk of covariance steps (and an update) ahead of its use
    const uint32_t imu_end = (prm.mode & M_FUSED) ? prm.win_off[prm.w1] : prm.prop_first + prm.prop_count;
    uint32_t pf_idx = 0xffffffffu;
    double pf[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (uint32_t w = prm.w0; w < prm.w1; ++w) {
        L2T(threadIdx.x == 0, 1, 1);
        cta_bar<NT>();  // (a) the nominal warp has posted the IMU range
        L2T(threadIdx.x == 0, 1, 2);
        const int fp = (int)((w - prm.w0) & 1u);
        const uint32_t lo = sh.lo_hi[fp][0][0], hi = sh.lo_hi[fp][1][0];
        bool touched = false;
        uint32_t cpar = 0;
        for (uint32_t cb = lo; cb < hi; cb += L2_CH, cpar ^= 1u) {
            const uint32_t ce = min(cb + (uint32_t)L2_CH, hi);
            cta_bar<NT>();  // (I) validity, dt and the biases of the chunk are posted
            L2T(threadIdx.x == 0, 1, 3);
            if (cw < (int)(ce - cb) && l2.sval[cpar][cw][lane]) {  // F2's sample-only half for (sample cb + cw, filter lane)
                double* ic = XI + (size_t)(L2_INC + cw * L2_NE) * 32;
                const double dt = ic[0];
                double wv[3], dqh[4], dq[4];
                if (pf_idx != cb + (uint32_t)cw) {
#pragma unroll
                    for (int c = 0; c < 6; ++c) pf[c] = imu_sample_t<IMU32>(prm, k.imu_g, (size_t)cb + cw, c, B, bi);
                }
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    ic[(size_t)(10 + c) * 32] = pf[c] - XI[(size_t)(L2_BIAS + c) * 32];
                    wv[c] = pf[3 + c] - XI[(size_t)(L2_BIAS + 3 + c) * 32];
                }
                nominal_increment(wv, dt, dqh, dq);
#pragma unroll
                for (int c = 0; c < 4; ++c) { ic[(size_t)(2 + c) * 32] = dqh[c]; ic[(size_t)(6 + c) * 32] = dq[c]; }
#pragma unroll
                for (int c = 0; c < 3; ++c) ic[(size_t)(13 + c) * 32] = wv[c] * dt;  // u of cov_coeffs
            }
            pf_idx = ce + (uint32_t)cw;
            if (cw < L2_CH && pf_idx < imu_end) {
#pragma unroll
                for (int c = 0; c < 6; ++c) pf[c] = imu_sample_t<IMU32>(prm, k.imu_g, (size_t)pf_idx, c, B, bi);
            } else {
                pf_idx = 0xffffffffu;
            }
            L2T(threadIdx.x == 0, 1, 4);
            cta_bar<NT>();  // (J) increments posted
            L2T(threadIdx.x == 0, 1, 5);
            for (uint32_t i = cb; i < ce; ++i) {
                const int slot = (int)(i - cb);
                slot_wait(slot);  // record (slot) is complete
                const bool valid = act && l2.sval[cpar][slot][f] != 0;
                const double2* rec2 = reinterpret_cast<const double2*>(ring + ((size_t)slot * 32 + (size_t)f) * L2_RS);
                double A[9], Bm[9], u0, u1, u2, dt;
                {
                    double rv[22];
#pragma unroll
                    for (int e = 0; e < 11; ++e) {
                        const double2 v = rec2[e];
                        rv[2 * e] = v.x;
                        rv[2 * e + 1] = v.y;
                    }
#pragma unroll
                    for (int e = 0; e < 9; ++e) { A[e] = rv[e]; Bm[e] = rv[9 + e]; }
                    u0 = rv[18]; u1 = rv[19]; u2 = rv[20]; dt = rv[21];
                }
                if (valid) {  // A: M = F P on both columns
                    lane_apply_Fu2(c0, c1, A, Bm, u0, u1, u2, dt);
#pragma unroll
                    for (int r = 0; r < 9; ++r) {  // T: publish the rows of M that change
                        T[r * LANE_TS + l] = c0[r];
                        T[r * LANE_TS + 9 + l] = c1[r];
                    }
                }
                __syncwarp();
                if (valid) {  // B: column l of F P F^T = F (row l of M)^T
#pragma unroll
                    for (int c = 0; c < 18; ++c) c0[c] = T[l * LANE_TS + c];
                    lane_apply_Fu1(c0, A, Bm, u0, u1, u2, dt);
#pragma unroll
                    for (int r = 3; r < 9; ++r) c0[r] += (r == l) ? q0 : 0.0;
#pragma unroll
                    for (int r = 9; r < 15; ++r) c1[r] += (r == l + 9) ? q1 : 0.0;
                    touched = true;
                }
                __syncwarp();  // the row reads are done before the next sample's publish
                L2T(threadIdx.x == 0, 1, 10 + slot);
            }
        }
        if (__any_sync(0xffffffffu, touched)) {  // symmetrise the top-left 9x9 (the only part evaluated in two orders)
            if (touched) {
#pragma unroll
                for (int r = 0; r < 9; ++r) T[r * LANE_TS + l] = c0[r];
            }
            __syncwarp();
            if (touched) {
#pragma unroll
                for (int r = 0; r < 9; ++r) c0[r] = 0.5 * (c0[r] + T[l * LANE_TS + r]);
            }
            __syncwarp();
        }
        L2T(threadIdx.x == 0, 1, 6);
        cta_bar<NT>();  // (r) update requests posted
        L2T(threadIdx.x == 0, 1, 7);
        if (sh.any_upd[0]) {
            const bool req = act && sflag[2][f] != 0;
            if (req && (l < 3 || l >= 6)) {
                const int ci = l < 3 ? l : l - 3;
#pragma unroll
                for (int m = 0; m < 6; ++m) X[(size_t)(L2_SHIFT + LX_P6 + m * 6 + ci) * 32] = c0[m < 3 ? m : m + 3];
            }
            cta_bar<NT>();  // (p) P6 published
            L2T(threadIdx.x == 0, 1, 8);
            cta_bar<NT>();  // (c) the nominal warp has posted the gain factors
            L2T(threadIdx.x == 0, 1, 9);
            constexpr int NZ = JOSEPH ? 6 : 7;
            double z0[NZ], z1[NZ];
            if (req) {
                if constexpr (JOSEPH) {
                    double Cm[21];
#pragma unroll
                    for (int c = 0; c < 21; ++c) Cm[c] = X[(size_t)(L2_SHIFT + LX_CM + c) * 32];
#pragma unroll
                    for (int kz = 0; kz < 6; ++kz) {
                        double s0 = Cm[kz * (kz + 1) / 2 + kz] * c0[kz < 3 ? kz : kz + 3];
                        double s1 = Cm[kz * (kz + 1) / 2 + kz] * c1[kz < 3 ? kz : kz + 3];
#pragma unroll
                        for (int m = kz + 1; m < 6; ++m) {
                            s0 += Cm[m * (m + 1) / 2 + kz] * c0[m < 3 ? m : m + 3];
                            s1 += Cm[m * (m + 1) / 2 + kz] * c1[m < 3 ? m : m + 3];
                        }
                        z0[kz] = s0;
                        z1[kz] = s1;
                    }
                } else {
#pragma unroll
                    for (int kz = 0; kz < 7; ++kz) z0[kz] = z1[kz] = 0.0;
#pragma unroll
                    for (int m = 0; m < 6; ++m) {  // term by term across the fourteen sums (see lane_apply_Fu2)
#pragma unroll
                        for (int kz = 0; kz < 7; ++kz) {
                            const double x = X[(size_t)(L2_SHIFT + LX_SCR + kz * 6 + m) * 32];
                            z0[kz] += x * c0[m < 3 ? m : m + 3];
                            z1[kz] += x * c1[m < 3 ? m : m + 3];
                        }
                    }
                }
                double d0 = 0.0, d1 = 0.0;  // dx = Z^T y for the own columns
#pragma unroll
                for (int kz = 0; kz < NZ; ++kz) {
                    T[kz * LANE_TS + l] = z0[kz];
                    T[kz * LANE_TS + 9 + l] = z1[kz];
                    const double yk = X[(size_t)(L2_SHIFT + LX_Y + kz) * 32];
                    d0 += yk * z0[kz];
                    d1 += yk * z1[kz];
                }
                X[(size_t)(L2_SHIFT + LX_DX + l) * 32] = d0;
                X[(size_t)(L2_SHIFT + LX_DX + 9 + l) * 32] = d1;
            }
            L2T(threadIdx.x == 0, 1, 20);
            cta_bar<NT>();  // (d) dx posted (also: the filter's Z columns are in its scratch)
            L2T(threadIdx.x == 0, 1, 21);
            if (req) {
#pragma unroll
                for (int kz = 0; kz < NZ; ++kz) {  // P -= Z^T Z on both columns (exactly symmetric: the same products in the same order on
#pragma unroll                                     // both sides), one row of Z at a time across all thirty-six entries
                    for (int r = 0; r < 18; ++r) {
                        const double zr = T[kz * LANE_TS + r];
                        c0[r] -= zr * z0[kz];
                        c1[r] -= zr * z1[kz];
                    }
                }
            }
            __syncwarp();
            L2T(threadIdx.x == 0, 1, 22);
        }
    }
    if (live) {  // upper triangle back: column j is stored by its owner for rows i <= j
#pragma unroll
        for (int i = 0; i < 18; ++i) {
            if (i <= l) prm.P[(size_t)(i * NX - (i * (i - 1)) / 2 + (l - i)) * B + b] = c0[i];
            if (i <= l + 9) prm.P[(size_t)(i * NX - (i * (i - 1)) / 2 + (l + 9 - i)) * B + b] = c1[i];
        }
    }
}

template <bool JOSEPH, bool IMU32, bool NOISE = false>  // NOISE: as ekf_window_lane_kernel
__global__ void __launch_bounds__(LANE_NT, 1) ekf_window_lane2_kernel(const __grid_constant__ WinParams prm, const __grid_constant__ DevConsts k,
                                                                      const double* __restrict__ noise) {
    extern __shared__ double smem[];
    __shared__ SplitShared sh;
    __shared__ int32_t sflag[3][32];
    __shared__ Lane2Shared l2;
    __shared__ MarkerTable s_tab;  // the marker map is read by every frame's plan and update: one copy per CTA in shared memory
    const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
    {
        static_assert(sizeof(MarkerTable) % sizeof(double) == 0, "MarkerTable is copied as doubles");
        const double* src = reinterpret_cast<const double*>(prm.tab);
        double* dst = reinterpret_cast<double*>(&s_tab);
        for (int i = threadIdx.x; i < (int)(sizeof(MarkerTable) / sizeof(double)); i += LANE_NT) dst[i] = src[i];
        __syncthreads();
    }
    if (wi < 11) {
        if constexpr (NOISE) lane2_cov_role<JOSEPH, IMU32, true>(prm, k, smem, sh, sflag, l2, wi, lane, noise);
        else lane2_cov_role<JOSEPH, IMU32>(prm, k, smem, sh, sflag, l2, wi, lane);
    } else {
        // a CTA serves lane_fpc filters (<= 32): batches that cannot fill the GPU are spread thin, because a filter-step is the
        // faster the fewer filters share the CTA's nominal warp, schedulers and shared-memory bandwidth
        const size_t b0 = (size_t)blockIdx.x * prm.lane_fpc + lane;
        const bool live = lane < (int)prm.lane_fpc && b0 < prm.B;
        if constexpr (NOISE)
            nominal_role<32, false, IMU32, true, JOSEPH, false, true, true>(prm, k, smem, sh, sflag, lane, live ? b0 : prm.B - 1, live, &l2,
                                                                            &s_tab, smem + (size_t)L2_TOTAL * 32, noise);
        else nominal_role<32, false, IMU32, true, JOSEPH, false, true>(prm, k, smem, sh, sflag, lane, live ? b0 : prm.B - 1, live, &l2, &s_tab,
                                                                       smem + (size_t)L2_TOTAL * 32);
    }
}

}  // namespace fbus
