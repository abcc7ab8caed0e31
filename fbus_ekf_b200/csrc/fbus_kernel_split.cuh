// fbus_kernel_split.cuh -- K12, warp-specialised: the fused window kernel with TWO warps per 32 filters.
//
// Why: the packed covariance (171 doubles = 1368 B per filter) caps residency at ~128-160 filters per SM, i.e. one
// warp per scheduler with one thread per filter.  A lone warp cannot overlap its shared-memory traffic, integer work
// and the serial sin/cos/sqrt/div chains of the nominal-state integration with the half-rate FP64 pipe (ncu: FP64 pipe
// ~33 % busy, "wait"/"short scoreboard" stalls, 1.0 warp per scheduler).  Here every group of 32 filters gets
//   * a COVARIANCE warp: F1 (P <- F P F^T + Q) and the measurement update's covariance work; P lives in TENSOR MEMORY
//                        (one TMEM lane per filter, fbus_tmem.cuh) in the 128-filter CTAs, in shared memory in the
//                        32-filter CTAs used for small batches;
//   * a NOMINAL warp:    detection scan, F6b init, F5 reset, F2 nominal integration (q,p,v + the carried rotmatI2G),
//                        the IMU/detection streams, and the error-state injection after an update.
// so each scheduler holds two warps with complementary instruction mixes.  The nominal warp runs one IMU sample AHEAD
// and hands the covariance warp the coefficients of F for that sample (A = -R[a]x dt, B = -R dt, w dt, dt: 22 doubles)
// through a 2-deep ring in shared memory; one named barrier per sample (private to the warp pair) orders the ring, one
// CTA-wide barrier per frame keeps all warps on the same instruction-cache lines.  For an update the nominal warp posts
// (marker, y, q, R, p), the covariance warp runs measurement_update and posts back the injected pose / state increments;
// meanwhile the nominal warp plans the next frame.  Variants that were measured and dropped (cooperative update, deeper
// mbarrier ring, register-resident blocks across frames, ...) are listed in DESIGN.md; the git history has their code.
//
#pragma once

#include "fbus_kernels.cuh"
#include "fbus_tmem.cuh"

// 1 (default): the 128-filter CTAs keep the covariance in TENSOR MEMORY (one TMEM lane per filter, fbus_tmem.cuh) instead
// of shared memory; the 32-filter CTAs of small batches (several per SM) always use shared memory
#ifndef FBUS_TMEM
#define FBUS_TMEM 1
#endif

namespace fbus {

// -DFBUS_L2_TRACE: phase time stamps of CTA 0 of the second-generation lane kernel (nominal lane 0 = role 0, covariance warp 0 =
// role 1) for profiles/probes/lane2_trace.py; compiled out of the library
#ifdef FBUS_L2_TRACE
__device__ long long g_l2_trace[2][16384];
__device__ int g_l2_trace_n[2];
#define L2T(cond, role, tag)                                                    \
    do {                                                                        \
        if (blockIdx.x == 0 && (cond)) {                                        \
            const int i_ = g_l2_trace_n[role]++;                                \
            if (i_ < 8192) {                                                    \
                g_l2_trace[role][2 * i_] = (tag);                               \
                g_l2_trace[role][2 * i_ + 1] = clock64();                       \
            }                                                                   \
        }                                                                       \
    } while (0)
#else
#define L2T(cond, role, tag) ((void)0)
#endif

constexpr int XCH = 54;  // doubles of exchange area per filter: ring 2 x 22 (+ request, results); the update parks 54 doubles of Z here

// CTA-wide named barrier used by both roles (the two roles run different code, so the barrier is issued from
// different program counters; whole warps take each path, and arrivals are counted per barrier id)
template <int NT>
__device__ __forceinline__ void cta_bar() { asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory"); }
// per-sample barrier, private to the covariance + nominal warp of one filter group (barrier ids 2..9); the CTA re-aligns
// once per frame with cta_bar
__device__ __forceinline__ void step_bar(int pair) { asm volatile("bar.sync %0, 64;" ::"r"(pair + 2) : "memory"); }
struct SplitShared {
    // per nominal warp: min first / max end of the candidate IMU range.  Double-buffered by frame parity: a nominal warp
    // posts frame w+1's range after passing only its pair-private barriers, while warps of OTHER pairs may still be
    // reading frame w's entries (they read after the CTA barrier (a) of frame w); with two copies the writer of frame w+2
    // -- which has passed barrier (a) of frame w+1, i.e. after every reader of frame w arrived there -- is the first to
    // touch frame w's copy again.
    uint32_t lo_hi[2][2][8];
    int32_t any_upd[8];     // per nominal warp: some filter requests an update (pair-private: written before (r), read after)
};

// ------------------------------------------------------------------------------------------------------------------
// Hand-off protocol per detection frame (barriers: (a) CTA-wide, the others private to the warp pair):
//   (a)      IMU ranges posted                      -> both roles know [lo, hi)
//   step(i)  ring record i published                 (one per IMU sample; the nominal warp is one sample ahead)
//   (r)      update request posted                   -- written into the ring slot that sample `hi` WOULD use, which is
//                                                       free while the covariance warp still works on sample hi-1, so the
//                                                       request is on the table when that warp leaves its last step
//   (d)      update results posted                   -- meanwhile the nominal warp has planned the NEXT frame (detection
//                                                       scan, marker lookup, F5/F6b vision pose: none depend on the state)
// The next frame's (a) doubles as "results consumed".
// ------------------------------------------------------------------------------------------------------------------
constexpr int RQ_EXTRA = 44;  // the request needs 23 doubles: 22 in the free ring slot + this one

// top-left 9x9 <-> registers, block-wise (six 3x3 blocks) for the tensor-memory accessor
template <bool TM, class CV>
__device__ __forceinline__ void tl_load_any(const CV P, double* TL) {
    if constexpr (TM) {
        FBUS_UNROLL
        for (int bj = 0; bj < 3; ++bj)
            FBUS_UNROLL
            for (int bi = 0; bi <= bj; ++bi) {
                double T[9];
                P.ldraw(bi, bj, T);
                tm_wait_ld();
                FBUS_UNROLL
                for (int r = 0; r < 3; ++r)
                    FBUS_UNROLL
                    for (int c = (bi == bj ? r : 0); c < 3; ++c) TL[tlidx(3 * bi + r, 3 * bj + c)] = T[r * 3 + c];
            }
    } else {
        tl_load<0>(P, TL);
    }
}
template <bool TM, class CV>
__device__ __forceinline__ void tl_store_any(const CV P, const double* TL) {
    if constexpr (TM) {
        FBUS_UNROLL
        for (int bj = 0; bj < 3; ++bj)
            FBUS_UNROLL
            for (int bi = 0; bi <= bj; ++bi) {
                double T[9];
                FBUS_UNROLL
                for (int r = 0; r < 3; ++r)
                    FBUS_UNROLL
                    for (int c = 0; c < 3; ++c) T[r * 3 + c] = TL[tlidx(3 * bi + r, 3 * bj + c)];
                P.straw(bi, bj, T);
            }
    } else {
        tl_store<0>(P, TL);
    }
}

__device__ __forceinline__ int pair_any(const SplitShared& sh, int wq) { return sh.any_upd[wq]; }

// ------------------------------------------------------------------------------------------------------------------
// COVARIANCE role: owns P (shared memory; top-left 9x9 in registers while propagating)
// ------------------------------------------------------------------------------------------------------------------
// Where the covariance warp of a NOISE instantiation keeps its filters' four process noise values: in shared memory (4 x BSF
// doubles next to the exchange area) when that still fits the 227 KB a CTA may have.  The 128-filter CTAs with the covariance in
// shared memory (FBUS_TMEM=0) already take 225 KB; they read the values from the noise buffer through the L1 cache per sample.
template <int BSF, bool TM>
constexpr bool noise_q_in_smem = (size_t)((TM ? 0 : NPK) + XCH + 4) * BSF * sizeof(double) + 2048 <= (size_t)227 * 1024;

// NOISE: the filters have their own noise values (fbus_set_noise): `noise` is the [6][B] buffer, `sq` this filter's four process
// noise values in shared memory (entry stride BSF; nullptr when noise_q_in_smem is false), read where Qv is built instead of being
// held in registers across the step loop
template <int BSF, bool JOSEPH, bool TM, bool NOISE = false>
__device__ __forceinline__ void cov_role(const WinParams& prm, const DevConsts& k, double* smem, SplitShared& sh, int32_t (*sflag)[BSF],
                                         int fl, size_t b, bool live, uint32_t tm_base, const double* noise = nullptr, double* sq = nullptr) {
    constexpr int NT = 2 * BSF, NW = BSF / 32;
    constexpr int NPS = TM ? 0 : NPK;  // doubles of P per filter in shared memory
    const size_t B = prm.B;
    using CV = typename std::conditional<TM, CovTM<false>, Cov<BSF>>::type;
    CV P;
    if constexpr (TM) {
        // lane 32*(warp%4) in bits 31..16; broadcast from lane 0 so that the compiler knows the address is warp-uniform and
        // keeps it (and the block offsets added to it) in uniform registers instead of converting for every tcgen05 access
        P.base = __shfl_sync(0xffffffffu, tm_base + ((uint32_t)((threadIdx.x >> 5) & 3) << 21), 0);
    }
    else P.s = smem + fl;
    double* const X = smem + (size_t)NPS * BSF + fl;
    const int wq = fl >> 5;
    if constexpr (NOISE && noise_q_in_smem<BSF, TM>) {  // written and read by this thread only
#pragma unroll
        for (int c = 0; c < 4; ++c) sq[(size_t)c * BSF] = noise[(size_t)c * B + b];
    }
    if constexpr (TM) {
        FBUS_UNROLL
        for (int bj = 0; bj < 6; ++bj)
            FBUS_UNROLL
            for (int bi = 0; bi <= bj; ++bi) {
                double T[9];
                FBUS_UNROLL
                for (int r = 0; r < 3; ++r)
                    FBUS_UNROLL
                    for (int c = 0; c < 3; ++c) T[r * 3 + c] = prm.P[(size_t)pidx(3 * bi + r, 3 * bj + c) * B + b];
                P.straw(bi, bj, T);
            }
        P.fence_st();
    } else {
        for (int e = 0; e < NPK; ++e) smem[e * BSF + fl] = prm.P[(size_t)e * B + b];
    }
    for (uint32_t w = prm.w0; w < prm.w1; ++w) {
        cta_bar<NT>();  // (a) the nominal warps have posted their IMU ranges
        const int fp = (int)((w - prm.w0) & 1u);
        uint32_t lo = sh.lo_hi[fp][0][0], hi = sh.lo_hi[fp][1][0];
#pragma unroll
        for (int q = 1; q < NW; ++q) { lo = min(lo, sh.lo_hi[fp][0][q]); hi = max(hi, sh.lo_hi[fp][1][q]); }
        int fs = 0;  // ring slot that carries the update request
        if (lo < hi) {
            fs = (int)((hi - lo) & 1u);
            double TL[NTL];  // top-left 9x9 of P lives in registers for the whole window
            tl_load_any<TM>(P, TL);
            for (uint32_t i = lo; i < hi; ++i) {
                step_bar(wq);  // record (i) is complete; the nominal warp moves on to sample i+1
                const int slot = (int)((i - lo) & 1u);
                const int valid = sflag[slot][fl];
                // tensor-memory accesses are warp-wide: a warp with any valid lane runs the step on all lanes, the
                // others with F = I and no process noise (every entry of P keeps its value)
                if (TM ? __any_sync(0xffffffffu, valid) : valid) {
                    const double* rec = X + (size_t)slot * 22 * BSF;
                    double A[9], Bm[9];
#pragma unroll
                    for (int e = 0; e < 9; ++e) { A[e] = rec[(size_t)e * BSF]; Bm[e] = rec[(size_t)(9 + e) * BSF]; }
                    const double u0 = rec[(size_t)18 * BSF], u1 = rec[(size_t)19 * BSF], u2 = rec[(size_t)20 * BSF];
                    const double dt = rec[(size_t)21 * BSF];
                    double Qv[4] = {k.Qd[0], k.Qd[1], k.Qd[2], k.Qd[3]};
                    if constexpr (NOISE && noise_q_in_smem<BSF, TM>) {
#pragma unroll
                        for (int c = 0; c < 4; ++c) Qv[c] = sq[(size_t)c * BSF];
                    } else if constexpr (NOISE) {
#pragma unroll
                        for (int c = 0; c < 4; ++c) Qv[c] = __ldg(noise + (size_t)c * B + b);
                    }
                    if (TM && !valid) Qv[0] = Qv[1] = Qv[2] = Qv[3] = 0.0;  // the record of an invalid sample is all zeros
                    P.fence_st();  // the previous step's stores
                    propagate_cov_core<BSF, true>(P, A, Bm, u0, u1, u2, dt, Qv, TL);
                }
            }
            tl_store_any<TM>(P, TL);
        }
        step_bar(wq);  // (r) update request posted (normally long before this warp gets here)
        if (pair_any(sh, wq)) {
            const int req = sflag[2][fl];
            if (TM ? true : (req != 0)) {  // tensor memory: all lanes, the ones without a request with zero gain
                const double* rq = X + (size_t)fs * 22 * BSF;
                Nominal t;
                double yP[3], yQ[4];
#pragma unroll
                for (int c = 0; c < 3; ++c) yP[c] = rq[(size_t)c * BSF];
#pragma unroll
                for (int c = 0; c < 4; ++c) { yQ[c] = rq[(size_t)(3 + c) * BSF]; t.q[c] = rq[(size_t)(7 + c) * BSF]; }
#pragma unroll
                for (int c = 0; c < 9; ++c) t.R[c] = rq[(size_t)(11 + c) * BSF];
                t.p[0] = rq[(size_t)20 * BSF]; t.p[1] = rq[(size_t)21 * BSF]; t.p[2] = X[(size_t)RQ_EXTRA * BSF];
#pragma unroll
                for (int c = 0; c < 3; ++c) { t.v[c] = 0.0; t.ba[c] = 0.0; t.bg[c] = 0.0; t.g[c] = 0.0; }
                t.t = 0.0;
                const MarkerConst mkc = prm.tab->mk[(req > 0 ? req : 1) - 1];
                P.fence_st();
                if constexpr (NOISE) {  // R of this filter, read at the update
                    const MeasNoise r{noise[4 * B + b], noise[5 * B + b]};
                    measurement_update<BSF, JOSEPH ? 1 : 0, BSF>(P, t, k, r, mkc, yP, yQ, X, req != 0);
                } else {
                    measurement_update<BSF, JOSEPH ? 1 : 0, BSF>(P, t, k, mkc, yP, yQ, X, req != 0);
                }
                P.fence_st();
                // hand back: corrected p, q and the increments of v, b_a, b_g, g
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    X[(size_t)(23 + c) * BSF] = t.p[c];
                    X[(size_t)(30 + c) * BSF] = t.v[c];
                    X[(size_t)(33 + c) * BSF] = t.ba[c];
                    X[(size_t)(36 + c) * BSF] = t.bg[c];
                    X[(size_t)(39 + c) * BSF] = t.g[c];
                }
#pragma unroll
                for (int c = 0; c < 4; ++c) X[(size_t)(26 + c) * BSF] = t.q[c];
            }
            step_bar(wq);  // (d) results posted
        }
    }
    if constexpr (TM) {
        P.fence_st();
        FBUS_UNROLL
        for (int bj = 0; bj < 6; ++bj)
            FBUS_UNROLL
            for (int bi = 0; bi <= bj; ++bi) {
                double T[9];
                P.ldraw(bi, bj, T);
                tm_wait_ld();
                if (live) {
                    FBUS_UNROLL
                    for (int r = 0; r < 3; ++r)
                        FBUS_UNROLL
                        for (int c = (bi == bj ? r : 0); c < 3; ++c) prm.P[(size_t)pidx(3 * bi + r, 3 * bj + c) * B + b] = T[r * 3 + c];
                }
            }
    } else {
        if (live)
            for (int e = 0; e < NPK; ++e) prm.P[(size_t)e * B + b] = smem[e * BSF + fl];
    }
}

// ------------------------------------------------------------------------------------------------------------------
// NOMINAL role: owns the nominal state (registers), the streams, and all per-frame decisions
// ------------------------------------------------------------------------------------------------------------------
// What a frame will do, decided from the detections alone (filter.cpp:329-341 / 418-430 / 639-675): nothing in here
// depends on the filter state except `inited`, `prev_id`, `cursor` and the nominal time, none of which the update changes,
// so the plan of frame w+1 is made while the covariance warp runs frame w's update.
struct FramePlan {
    bool do_prop, apply_init, apply_reset;
    int req;                 // marker index + 1 of the update, 0 = no update
    uint32_t p_first, p_end;
    uint32_t n_init_erase;   // F6b: imuCnt, the leading buffered samples not later than the frame (filter.cpp:299-305)
    double t_det, t_end;
    double y[7];             // measurement of the update (p, q of the chosen detection)
    double qv[4], pv[3];     // vision-only pose for init / reset
    // MATLAB-semantics mode only (dead in the other instantiations)
    double Rv[9];            // quaternion_to_rotmat of the un-normalised Q_IG (State.rotateMat after init / reset)
    double t_init;           // time of the last IMU sample not later than the initialising frame (preImuTime, FBUS_EKF.m:175)
    double t_img_new;        // preImgTime after this frame
    bool set_t_img;
    // FBUS_FLAG_ALL_MARKERS only (dead in the other instantiations): slots of the frame's further updates, bit s = slot s; their
    // poses are read again from the detection buffers when their round comes
    uint32_t extra;
};

// ALL: FBUS_FLAG_ALL_MARKERS -- pl.extra lists the frame's other known markers (max_markers <= 32, checked by the host)
template <int BSF, bool ALL = false>
__device__ __forceinline__ void plan_frame(const WinParams& prm, const DevConsts& k, const MarkerTable* tab, uint32_t w, size_t b, bool live,
                                           uint32_t cursor, double n_t, int inited, int& prev_id, int& status, FramePlan& pl) {
    const size_t B = prm.B;
    const int mode = prm.mode;
    const bool fused = (mode & M_FUSED) != 0;
    const bool uses_det = (mode & (M_INIT | M_RESET | M_UPDATE | M_FUSED)) != 0;
    pl.do_prop = pl.apply_init = pl.apply_reset = false;
    pl.req = 0;
    pl.p_first = pl.p_end = 0;
    pl.n_init_erase = 0;
    pl.t_det = pl.t_end = 0.0;
    bool do_update = false;
    int n_det = 0, idx_near = 0, idx_prev = 0;
    double md = 10.0, prev_dist = 0.0;
    // ---- scan this frame's detections (filter.cpp:329-341 / 418-430 / 639-658) ----------------
    if (uses_det) {
        pl.t_det = prm.det_t[w];
        for (int s = 0; s < prm.m; ++s) {
            const size_t slot = (size_t)w * prm.m + s;
            const int id = prm.det_id[slot * B + b];
            if (id < 0) continue;
            const double* pp = prm.det_pose + slot * 7 * B + b;
            const double px = pp[0], py = pp[B], pz = pp[2 * B];
            const double dist = sqrt_d(px * px + py * py + pz * pz);
            if (n_det == 0) { idx_near = s; idx_prev = s; }  // detectionResult_[0] defaults (min_dist_id = 0)
            if (dist < md) { md = dist; idx_near = s; }
            if (id == prev_id) { prev_dist = dist; idx_prev = s; }
            ++n_det;
        }
    }
    int idx_upd = idx_near;  // nearest, or the previously used marker within the switch threshold (filter.cpp:660-664)
    {
        const double dd = prev_dist - md;
        if ((dd < 0 ? -dd : dd) < k.switch_thres && prev_dist != 0) idx_upd = idx_prev;
    }
    bool do_init = false, do_reset = false;
    uint32_t n_before = prm.n_imu_before;
    if (fused) {
        if (n_det == 0) {
            status |= FBUS_ST_NO_DETECTION;  // filter thread not woken (vision.cpp:136-140)
        } else if (!inited) {
            do_init = true;
            n_before = 0;
            const uint32_t hi = prm.win_off[w + 1];
            for (uint32_t i = cursor; i < hi; ++i) {  // the reference's loop stops at the first later sample
                if (prm.imu_t[i] > pl.t_det) break;
                ++n_before;
            }
            pl.n_init_erase = n_before;
        } else {
            do_reset = pl.do_prop = do_update = true;
            pl.p_first = cursor;
            pl.p_end = prm.win_off[w + 1];
            pl.t_end = pl.t_det;
        }
    } else {
        do_init = (mode & M_INIT) != 0;
        do_reset = (mode & M_RESET) != 0;
        do_update = (mode & M_UPDATE) != 0;
        if (mode & M_PROP) {
            pl.do_prop = true;
            pl.p_first = prm.prop_first;
            pl.p_end = prm.prop_first + prm.prop_count;
            pl.t_end = prm.prop_t_end;
        }
        if ((mode & M_UPDATE) && n_det == 0) status |= FBUS_ST_NO_DETECTION;
    }
    // ---- F6b InitializePose (filter.cpp:291-399) / F5 ResetSystemState (filter.cpp:405-477) -------
    if ((do_init || do_reset) && n_det > 0) {
        bool ok = !(md > k.max_dist);
        if (do_init) ok = ok && (n_before > 0);
        int mk = -1;
        double dp[3], dq[4];
        if (ok) {
            const size_t slot = (size_t)w * prm.m + idx_near;
            const int did = prm.det_id[slot * B + b];
            const double* pp = prm.det_pose + slot * 7 * B + b;
#pragma unroll
            for (int c = 0; c < 3; ++c) dp[c] = pp[(size_t)c * B];
#pragma unroll
            for (int c = 0; c < 4; ++c) dq[c] = pp[(size_t)(3 + c) * B];
            mk = find_marker(k, tab, did);
            ok = mk >= 0;
        }
        if (ok) {
            double Rv[9];
            const MarkerConst mkc = tab->mk[mk];
            vision_pose(k, mkc, dp, dq, pl.qv, Rv, pl.pv);
            double t_now = n_t;
            int inited_now = inited;
            if (do_init) { pl.apply_init = true; t_now = pl.t_det; inited_now = 1; }
            if (do_reset) {
                if (live) {
#pragma unroll
                    for (int i = 0; i < 3; ++i) prm.nom[(size_t)(F_PV + i) * B + b] = pl.pv[i];
#pragma unroll
                    for (int i = 0; i < 4; ++i) prm.nom[(size_t)(F_QV + i) * B + b] = pl.qv[i];
                }
                if (pl.t_det - t_now > k.reset_gap && inited_now) {
                    pl.apply_reset = true;
                    status |= FBUS_ST_RESET_DONE;  // P, g and the carried R stay untouched
                }
            }
        } else {
            if (do_init) status |= FBUS_ST_INIT_FAILED;
            if (do_reset) status |= FBUS_ST_RESET_SKIPPED;
        }
    } else if (do_init) {
        status |= FBUS_ST_INIT_FAILED;
    }
    // ---- marker and measurement of this frame's update (filter.cpp:666-675) ---------------------------------
    if (do_update && n_det > 0) {
        const size_t slot = (size_t)w * prm.m + idx_upd;
        const int did = prm.det_id[slot * B + b];
        const int mk = find_marker(k, tab, did);
        if (mk >= 0) {
            prev_id = did;
            pl.req = mk + 1;
            const double* pp = prm.det_pose + slot * 7 * B + b;
#pragma unroll
            for (int c = 0; c < 7; ++c) pl.y[c] = pp[(size_t)c * B];
        } else {
            status |= FBUS_ST_UPDATE_SKIPPED;
        }
    }
    if constexpr (ALL) {  // every other slot with a known id, in slot order
        pl.extra = 0u;
        if (do_update && n_det > 0) {
            for (int s = 0; s < prm.m; ++s) {
                if (s == idx_upd) continue;
                const int id = prm.det_id[((size_t)w * prm.m + s) * B + b];
                if (id < 0) continue;
                if (find_marker(k, tab, id) >= 0) pl.extra |= 1u << s;
                else status |= FBUS_ST_UPDATE_SKIPPED;
            }
        }
        if (pl.req == 0 && pl.extra != 0u) {  // the chosen marker is unknown: the first other one takes its round (prev_id unchanged)
            const size_t slot = (size_t)w * prm.m + (__ffs(pl.extra) - 1);
            pl.extra &= pl.extra - 1u;
            pl.req = find_marker(k, tab, prm.det_id[slot * B + b]) + 1;
            const double* pp = prm.det_pose + slot * 7 * B + b;
#pragma unroll
            for (int c = 0; c < 7; ++c) pl.y[c] = pp[(size_t)c * B];
        }
    }
}

// MATLAB-semantics mode (FBUS_FLAG_MATLAB): what a frame does in matlab/FBUS_EKF.m:151-197.  Differences from plan_frame:
// nearest marker without hysteresis or range gate (MeasureUpdate.m:51-60); a gap between two IMAGE times resets and skips
// propagation and update (FBUS_EKF.m:168-171, ResetState.m); the initialising frame is processed by the main loop as well
// (FBUS_EKF.m:116-151: the loop starts again at the first image row); the vision-only pose of every frame is that of
// ComputeVisionOnlyResults.m (normalised Q_IG).  An unknown marker id, on which the MATLAB script would stop with an index error,
// skips the frame for that filter with a status bit, like the C++ path.
template <int BSF>
__device__ __forceinline__ void plan_frame_matlab(const WinParams& prm, const DevConsts& k, const MarkerTable* tab, uint32_t w, size_t b, bool live,
                                                  uint32_t cursor, double t_img, int inited, int& prev_id, int& status, FramePlan& pl) {
    const size_t B = prm.B;
    const int mode = prm.mode;
    const bool fused = (mode & M_FUSED) != 0;
    pl.do_prop = pl.apply_init = pl.apply_reset = pl.set_t_img = false;
    pl.req = 0;
    pl.p_first = pl.p_end = 0;
    pl.n_init_erase = 0;
    pl.t_det = pl.t_end = pl.t_init = pl.t_img_new = 0.0;
    if (!(mode & (M_INIT | M_RESET | M_UPDATE | M_FUSED))) {  // un-fused propagate
        pl.do_prop = true;
        pl.p_first = prm.prop_first;
        pl.p_end = prm.prop_first + prm.prop_count;
        pl.t_end = prm.prop_t_end;
        return;
    }
    pl.t_det = prm.det_t[w];
    int n_det = 0, idx_near = 0;
    double md = 10.0;
    for (int s = 0; s < prm.m; ++s) {
        const size_t slot = (size_t)w * prm.m + s;
        if (prm.det_id[slot * B + b] < 0) continue;
        const double* pp = prm.det_pose + slot * 7 * B + b;
        const double px = pp[0], py = pp[B], pz = pp[2 * B];
        const double dist = sqrt_d(px * px + py * py + pz * pz);
        if (n_det == 0) idx_near = s;
        if (dist < md) { md = dist; idx_near = s; }
        ++n_det;
    }
    if (n_det == 0) { status |= FBUS_ST_NO_DETECTION; return; }
    const size_t slot = (size_t)w * prm.m + idx_near;
    const int did = prm.det_id[slot * B + b];
    const int mk = find_marker(k, tab, did);
    if (mk < 0) {
        status |= inited ? (FBUS_ST_UPDATE_SKIPPED | FBUS_ST_RESET_SKIPPED) : FBUS_ST_INIT_FAILED;
        return;
    }
    const MarkerConst mkc = tab->mk[mk];
    const double* pp = prm.det_pose + slot * 7 * B + b;
#pragma unroll
    for (int c = 0; c < 7; ++c) pl.y[c] = pp[(size_t)c * B];
    vision_pose<true>(k, mkc, pl.y, pl.y + 3, pl.qv, pl.Rv, pl.pv);  // InitPositionAndQuaternion.m / ResetState.m
    if (live) {  // ComputeVisionOnlyResults.m: the same with Q_IG normalised first
        double qn[4] = {pl.qv[0], pl.qv[1], pl.qv[2], pl.qv[3]}, Rn[9], u[3], r1[3], r2[3];
        qnormalize(qn);
        q2R_matlab(qn, Rn);
        mat3t_vec(k.R_IL, pl.y, u);
        mat3_vec(Rn, k.P_IL, r1);
        mat3_vec(Rn, u, r2);
#pragma unroll
        for (int i = 0; i < 3; ++i) prm.nom[(size_t)(F_PV + i) * B + b] = (mkc.p[i] - r1[i]) - r2[i];
#pragma unroll
        for (int i = 0; i < 4; ++i) prm.nom[(size_t)(F_QV + i) * B + b] = qn[i];
    }
    bool run_frame = false;  // propagate + update
    if (fused) {
        if (!inited) {
            uint32_t n_before = 0;
            const uint32_t hi = prm.win_off[w + 1];
            for (uint32_t i = cursor; i < hi; ++i) {
                if (prm.imu_t[i] > pl.t_det) break;
                pl.t_init = prm.imu_t[i];
                ++n_before;
            }
            if (n_before == 0) { status |= FBUS_ST_INIT_FAILED; return; }
            pl.apply_init = true;
            pl.n_init_erase = n_before;
            cursor += n_before;
            run_frame = true;  // preImgTime is still 0: no reset, the (empty) IMU loop, then MeasureUpdate
        } else if (t_img != 0.0 && pl.t_det - t_img > k.reset_gap) {
            pl.apply_reset = true;
            status |= FBUS_ST_RESET_DONE;
        } else {
            run_frame = true;
        }
        pl.set_t_img = true;
        pl.t_img_new = pl.t_det;
        if (run_frame) {
            pl.do_prop = true;
            pl.p_first = cursor;
            pl.p_end = prm.win_off[w + 1];
            pl.t_end = pl.t_det;
        }
    } else {
        if (mode & M_INIT) {
            if (prm.n_imu_before == 0) { status |= FBUS_ST_INIT_FAILED; return; }
            pl.apply_init = true;
            pl.t_init = pl.t_det;  // the un-fused call has no IMU buffer to take preImuTime from
        }
        if (mode & M_RESET) { pl.apply_reset = true; status |= FBUS_ST_RESET_DONE; }  // ResetState.m is unconditional
        run_frame = (mode & M_UPDATE) != 0;
    }
    if (run_frame) {
        prev_id = did;
        pl.req = mk + 1;
    }
}

// exchange area of the lanes-per-filter kernel (fbus_kernel_lane.cuh), doubles per filter laid out [entry][32 filters]:
// ring 2 x 22 | P6 (6x6 of the p/theta rows and columns) | Lc (21, Joseph form only) | y (6) or z (7) | dx (18) |
// X = L^-1 Hs (42: scratch of the update prologue, and the 7-row factor the lanes read in the default form)
// (a ring slot has 28 doubles here: A 9, B 9, W = F[theta,theta] - I 9, dt -- the MATLAB-semantics mode needs the full W)
constexpr int LX_REC = 28, LX_P6 = 56, LX_CM = 92, LX_Y = 113, LX_DX = 120, LX_SCR = 138, LX_TOTAL = 180;
constexpr int LANE_NT = 384;  // 11 covariance warps (3 filters each, 9 lanes per filter) + the nominal warp
// Second generation of the lanes-per-filter kernel (ekf_window_lane2_kernel): the ring holds a whole CHUNK of L2_CH samples, the
// sample-only half of F2 (nominal_increment) is evaluated for all samples of the chunk in parallel by the covariance warps (warp =
// sample slot, lane = filter) before the nominal lane walks its now short chain, and each ring record is handed over through its own
// mbarrier instead of a CTA-wide barrier per sample.  Exchange area: ring L2_CH x 28 | the sections of the first generation, shifted |
// increments [L2_CH][L2_NE] | ba, bg of the frame.
constexpr int L2_CH = 8;
constexpr int L2_SHIFT = -LX_P6;  // the exchange sections of the first generation start at entry 0 (its two-slot ring is not used)
constexpr int L2_NE = 16;         // dt, t, dqh (4), dq (4), a = accel - b_a (3), u = (gyro - b_g) dt (3)
constexpr int L2_INC = LX_TOTAL + L2_SHIFT;
constexpr int L2_BIAS = L2_INC + L2_CH * L2_NE;
constexpr int L2_TOTAL = L2_BIAS + 6;
// ring of the second generation: [slot][filter][L2_RS doubles], a filter's record (A 9, B 9, u 3, dt = 22 doubles) contiguous so that
// it moves as eleven 16-byte accesses on both sides.  L2_RS = 30: the 32 nominal lanes' 16-byte stores at a stride of 240 bytes
// fall on eight distinct bank groups (four wavefronts for 512 bytes, the minimum), the three filters a covariance warp reads are
// conflict-free, and 240 is a multiple of 16.
constexpr int L2_RS = 30;
constexpr int L2_RING = L2_CH * 32 * L2_RS;  // doubles
struct Lane2Shared {
    int32_t sval[2][L2_CH][32];      // sample (slot) is processed by filter (lane); double-buffered by chunk parity: the nominal
                                     // lane posts chunk c+1 while the covariance lanes may still be working through chunk c
};
// hand-over of ring slot s: named barrier 2 + s, 32 producer threads (the nominal lanes) arrive without waiting, the 352 covariance
// threads wait.  A hardware barrier, not a polled flag: the waiting warps sleep and leave the issue slots to the nominal warp
// (a first version polled an mbarrier, and the eleven spinning warps slowed the nominal chain ~4x).
// (bar.arrive / bar.sync order the producer's earlier shared-memory writes before the consumers' later reads, as every barrier does;
// the arrive is executed by the whole, converged warp: the aligned form counts warps, not threads)
__device__ __forceinline__ void slot_arrive(int slot) { asm volatile("bar.arrive %0, %1;" ::"r"(slot + 2), "n"(LANE_NT) : "memory"); }
__device__ __forceinline__ void slot_wait(int slot) { asm volatile("bar.sync %0, %1;" ::"r"(slot + 2), "n"(LANE_NT) : "memory"); }

// the p/theta sub-matrix P6 = P[{0,1,2,6,7,8}, {0,1,2,6,7,8}] as the covariance lanes publish it: the only part of P the
// update prologue reads (accessor interface of update_prologue)
struct P6View {
    const double* s;  // [36][32] entries of this filter
    static constexpr bool kTLR = false;
    static constexpr bool kBlocked = false;
    static FBUS_HD constexpr int m6(int i) { return i < 3 ? i : i - 3; }  // rows 0,1,2 -> 0..2 ; 6,7,8 -> 3..5
    __device__ __forceinline__ double at(int a, int c) const { return s[(size_t)(a * 6 + c) * 32]; }
    __device__ __forceinline__ double ld(int i, int j) const { return at(m6(i), m6(j)); }
    __device__ __forceinline__ void lddiag(int bb, double* X) const {
        const int o = bb == 0 ? 0 : 3;
        FBUS_UNROLL
        for (int r = 0; r < 3; ++r)
            FBUS_UNROLL
            for (int c = 0; c < 3; ++c) X[r * 3 + c] = at(o + r, o + c);
    }
    __device__ __forceinline__ void ldblk(int bi, int bj, double* X) const {
        const int oi = bi == 0 ? 0 : 3, oj = bj == 0 ? 0 : 3;
        FBUS_UNROLL
        for (int r = 0; r < 3; ++r)
            FBUS_UNROLL
            for (int c = 0; c < 3; ++c) X[r * 3 + c] = at(oi + r, oj + c);
    }
};

// The innovation gate of fbus_set_gate (first-generation lanes-per-filter kernel): per-filter thresholds [B] and the per-filter
// counts of rejected updates [B]
struct GateBufs {
    const double* thr;
    int32_t* rejected;
};
// NIS = r^T S^-1 r = |z|^2 of z = L^-1 r (S = L L^T); the update is rejected iff thr > 0 and not NIS <= thr, so a non-finite NIS
// is rejected and a threshold <= 0 or NaN gates nothing
__device__ __forceinline__ bool gate_rejects(const double* z, double thr) {
    double nis = z[0] * z[0];
#pragma unroll
    for (int i = 1; i < 7; ++i) nis += z[i] * z[i];
    return thr > 0.0 && !(nis <= thr);
}

// LANE = true: the role runs inside the lanes-per-filter kernel (fbus_kernel_lane.cuh): every barrier is CTA-wide, invalid ring
// records need no neutral content, and the update is split differently -- this warp (one lane per filter) runs the
// state-only prologue (predicted measurement, Hs, S, the gain factors) from the published P6 and the error-state
// injection, the covariance lanes run the sweep P -= Z^T Z and dx = Z^T y.
// NOISE (LANE only): the update prologue takes this filter's R from rows 4, 5 of the [6][B] buffer `noise` (fbus_set_noise)
// ALL (first-generation LANE only): FBUS_FLAG_ALL_MARKERS -- the update hand-off (r) (p) (c) (d) repeats, one marker per filter and
// round (the planned one, then pl.extra in slot order), each at the state the previous injection left, until a round in which no
// filter of the CTA posts a request; the next frame's plan is made in the first round only
// GATE (first-generation LANE only): the innovation gate of fbus_set_gate -- after the prologue every update whose NIS fails the
// filter's threshold is withdrawn (sflag[2] cleared before (c), which the covariance lanes re-read) and not injected; the
// filter's count of rejections is kept in a register and written once at the end
template <int BSF, bool TM, bool IMU32 = false, bool LANE = false, bool JOSEPH = false, bool MATLAB = false, bool LANE2 = false,
          bool NOISE = false, bool ALL = false, bool GATE = false>
__device__ __forceinline__ void nominal_role(const WinParams& prm, const DevConsts& k, double* smem, SplitShared& sh,
                                             int32_t (*sflag)[BSF], int fl, size_t b, bool live, Lane2Shared* l2 = nullptr,
                                             const MarkerTable* tab_smem = nullptr, double* ring2 = nullptr, const double* noise = nullptr,
                                             GateBufs gt = GateBufs{nullptr, nullptr}) {
    const MarkerTable* const tab = tab_smem ? tab_smem : prm.tab;  // the second-generation lane kernel keeps a copy in shared memory
    constexpr int NT = LANE ? LANE_NT : 2 * BSF, NW = BSF / 32;
    static_assert(!LANE || BSF == 32, "the lanes-per-filter kernel has 32 filters per CTA");
    static_assert(!MATLAB || (LANE && !JOSEPH), "the MATLAB-semantics mode runs on the lanes-per-filter kernel, reference update form");
    static_assert(!LANE2 || (LANE && !MATLAB), "the second-generation lanes-per-filter kernel has the C++ semantics only");
    static_assert(!NOISE || LANE, "the warp-specialised kernel applies R in its covariance role");
    static_assert(!ALL || (LANE && !LANE2 && !MATLAB), "the all-markers mode runs on the first-generation lanes-per-filter kernel, C++ semantics");
    static_assert(!GATE || (LANE && !LANE2 && !MATLAB), "the innovation gate runs on the first-generation lanes-per-filter kernel, C++ semantics");
    constexpr int REC = LANE ? LX_REC : 22;  // doubles per ring slot
    constexpr int LXS = LANE2 ? L2_SHIFT : 0;  // shift of the exchange sections behind the ring
    const size_t B = prm.B;
    double* const X = smem + (size_t)((TM || LANE) ? 0 : NPK) * BSF + fl;
    auto sbar = [&](int pair) {
        if constexpr (LANE) cta_bar<NT>();
        else step_bar(pair);
    };
    const bool fused = (prm.mode & M_FUSED) != 0;
    const int wq = fl >> 5;  // nominal warp index
    Nominal n;
    n.t = prm.nom[(size_t)F_T * B + b];
#pragma unroll
    for (int i = 0; i < 4; ++i) n.q[i] = prm.nom[(size_t)(F_Q + i) * B + b];
#pragma unroll
    for (int i = 0; i < 9; ++i) n.R[i] = prm.nom[(size_t)(F_R + i) * B + b];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        n.p[i] = prm.nom[(size_t)(F_P + i) * B + b];
        n.v[i] = prm.nom[(size_t)(F_V + i) * B + b];
        n.ba[i] = prm.nom[(size_t)(F_BA + i) * B + b];
        n.bg[i] = prm.nom[(size_t)(F_BG + i) * B + b];
        n.g[i] = prm.nom[(size_t)(F_G + i) * B + b];
    }
    int prev_id = prm.prev_id[b];
    int inited = prm.init[b];
    int status = prm.status[b];
    double gthr = 0.0;    // GATE: this filter's threshold
    int32_t n_rej = 0;    // GATE: its count of rejected updates
    if constexpr (GATE) {
        gthr = gt.thr[b];
        n_rej = gt.rejected[b];
    }
    uint32_t cursor = fused ? (prm.cursor_resume ? prm.cursor_io[b] : prm.win_off[prm.w0]) : 0u;
    // first IMU sample of the NEXT window, prefetched while this warp waits for the covariance warp's update
    uint32_t pf_i = 0xffffffffu;
    double pf_st = 0.0, pf_sd[6];

    double t_img = MATLAB ? prm.nom[(size_t)F_TIMG * B + b] : 0.0;  // preImgTime (FBUS_EKF.m:144)
    auto plan = [&](uint32_t wf, FramePlan& out) {
        if constexpr (MATLAB) plan_frame_matlab<BSF>(prm, k, tab, wf, b, live, cursor, t_img, inited, prev_id, status, out);
        else plan_frame<BSF, ALL>(prm, k, tab, wf, b, live, cursor, n.t, inited, prev_id, status, out);
        if constexpr (LANE2) {
            // lanes past the batch mirror the last filter for their reads; in this kernel they neither propagate nor update, so
            // that a small batch (the live single-filter case) leaves the covariance warps of the unused slots asleep
            if (!live) {
                out.do_prop = out.apply_init = out.apply_reset = false;
                out.req = 0;
            }
        }
    };
    FramePlan pl;
    if (prm.w0 < prm.w1) plan(prm.w0, pl);

    for (uint32_t w = prm.w0; w < prm.w1; ++w) {
        L2T(LANE2 && fl == 0, 0, 1);
        // ---- apply the planned F6b InitializePose / F5 ResetSystemState --------------------------------------
        if (pl.apply_init) {
            n.t = MATLAB ? pl.t_init : pl.t_det;
#pragma unroll
            for (int i = 0; i < 4; ++i) n.q[i] = pl.qv[i];
            if constexpr (MATLAB) {
#pragma unroll
                for (int i = 0; i < 9; ++i) n.R[i] = pl.Rv[i];
            } else {
                q2R(pl.qv, n.R);
            }
#pragma unroll
            for (int i = 0; i < 3; ++i) n.p[i] = pl.pv[i];
            n.g[0] = 9.8; n.g[1] = 0.0; n.g[2] = 0.0;  // filter.cpp:387
            inited = 1;
            if (fused) cursor += pl.n_init_erase;  // only the samples not later than the frame are erased (filter.cpp:299-305,390)
        }
        if (pl.apply_reset) {
            if constexpr (MATLAB) {  // ResetState.m:70-79: rotateMat refreshed, b_g and the IMU time base kept
#pragma unroll
                for (int i = 0; i < 4; ++i) n.q[i] = pl.qv[i];
#pragma unroll
                for (int i = 0; i < 9; ++i) n.R[i] = pl.Rv[i];
#pragma unroll
                for (int i = 0; i < 3; ++i) { n.p[i] = pl.pv[i]; n.v[i] = 0.0; n.ba[i] = 0.0; }
            } else {
                n.t = pl.t_det;
#pragma unroll
                for (int i = 0; i < 4; ++i) n.q[i] = pl.qv[i];
#pragma unroll
                for (int i = 0; i < 3; ++i) { n.p[i] = pl.pv[i]; n.v[i] = 0.0; n.ba[i] = 0.0; n.bg[i] = 0.0; }
            }
        }
        const double t_img_frame = t_img;  // samples older than the PREVIOUS image time are skipped (FBUS_EKF.m:180-183)
        if (MATLAB && pl.set_t_img) t_img = pl.t_img_new;
        const bool do_prop = pl.do_prop;
        const uint32_t p_first = pl.p_first, p_end = pl.p_end;
        const double t_end = pl.t_end;
        int req = pl.req;  // marker index + 1 of this round's update (ALL: changes from round to round)

        // ---- F3 BatchImuProcessing (filter.cpp:483-531): one sample ahead of the covariance warp -------------
        const int fp = (int)((w - prm.w0) & 1u);  // copy of the range table this frame uses (see SplitShared)
        {
            const uint32_t vlo = __reduce_min_sync(0xffffffffu, do_prop ? p_first : 0xffffffffu);
            const uint32_t vhi = __reduce_max_sync(0xffffffffu, do_prop ? p_end : 0u);
            if ((fl & 31) == 0) { sh.lo_hi[fp][0][wq] = vlo; sh.lo_hi[fp][1][wq] = vhi; }
        }
        cta_bar<NT>();  // (a)
        L2T(LANE2 && fl == 0, 0, 2);
        uint32_t lo = sh.lo_hi[fp][0][0], hi = sh.lo_hi[fp][1][0];
#pragma unroll
        for (int q = 1; q < NW; ++q) { lo = min(lo, sh.lo_hi[fp][0][q]); hi = max(hi, sh.lo_hi[fp][1][q]); }
        int fs = 0;
        if constexpr (LANE2) {
            if (lo < hi) {
                const double start = n.t;
                bool open = do_prop;          // false once this filter hit a sample later than t_end (the reference's break)
                uint32_t consumed = p_first;  // samples erased afterwards (filter.cpp:492-503,520)
                double tprev = n.t;           // sysNominalState_.timeStamp as the sample loop sees it
                uint32_t cpar = 0;            // chunk parity (restarts with every frame, as in the covariance role)
#pragma unroll
                for (int c = 0; c < 3; ++c) {  // the biases are constant over the window: posted once for the increment pass
                    X[(size_t)(L2_BIAS + c) * BSF] = n.ba[c];
                    X[(size_t)(L2_BIAS + 3 + c) * BSF] = n.bg[c];
                }
                // R(q) of the current quaternion = rotmatI2GBeginTime of the next sample (filter.cpp:543).  It is the carried
                // rotmatI2G except right after an update or a reset, which change q and leave rotmatI2G alone (A.3-2).
                double Rq[9];
                q2R(n.q, Rq);
                // The velocity / position half of F2 runs ONE SAMPLE BEHIND the quaternion half: it is not part of the chain
                // through q, and in the same instruction stream it fills the latency gaps of that chain.  Pending operands
                // (dt = 0, a = 0: a no-op until the first processed sample).
                double pq[4] = {n.q[0], n.q[1], n.q[2], n.q[3]}, pdqh[4] = {1.0, 0.0, 0.0, 0.0}, pa[3] = {0.0, 0.0, 0.0}, pR0[9], pdt = 0.0;
#pragma unroll
                for (int c = 0; c < 9; ++c) pR0[c] = Rq[c];
                // the time stamps are shared by all filters: lane j loads the chunk's j-th, the loop below reads them by shuffle;
                // the next chunk's are in flight while this chunk is processed
                const int tl = fl & 31;
                double ts = (tl < L2_CH && lo + tl < hi) ? prm.imu_t[lo + tl] : 0.0;
                for (uint32_t c0 = lo; c0 < hi; c0 += L2_CH) {
                    const uint32_t c1 = min(c0 + (uint32_t)L2_CH, hi);
                    const double ts_next = (tl < L2_CH && c1 + tl < hi) ? prm.imu_t[c1 + tl] : 0.0;
                    // which samples of the chunk this filter processes, and their dt (the only part of the window logic that is a
                    // chain through the time stamps, filter.cpp:492-516).  Unrolled and branch-free: the shuffles and comparisons of
                    // all slots are independent, only open / tprev / consumed chain from slot to slot.
#pragma unroll
                    for (int j = 0; j < L2_CH; ++j) {
                        const uint32_t i = c0 + (uint32_t)j;
                        const double ti = __shfl_sync(0xffffffffu, ts, j);
                        const bool in = open && i < c1 && i >= p_first && i < p_end;
                        const bool early = ti < start, late = ti > t_end;
                        const bool valid = in && !early && !late;
                        if (in && !early && late) open = false;  // this sample stays buffered (the reference's break)
                        if (in && (early || !late)) consumed = i + 1;
                        const double dt = valid ? ti - tprev : 0.0;
                        if (valid) tprev = ti;
                        double* ic = X + (size_t)(L2_INC + j * L2_NE) * BSF;
                        ic[0] = dt;
                        ic[(size_t)BSF] = ti;
                        l2->sval[cpar][j][fl] = valid ? 1 : 0;
                    }
                    L2T(fl == 0, 0, 3);
                    cta_bar<NT>();  // (I) validity, dt and the biases are posted: the covariance warps evaluate the increments
                    cta_bar<NT>();  // (J) increments posted
                    L2T(fl == 0, 0, 4);
                    for (uint32_t i = c0; i < c1; ++i) {
                        const int slot = (int)(i - c0);
                        const bool valid = l2->sval[cpar][slot][fl] != 0;
                        const double* ic = X + (size_t)(L2_INC + slot * L2_NE) * BSF;
                        double dt = 0.0, dqh[4], dq[4], av[3];
                        if (valid) {
                            dt = ic[0];
                            double u[3];
#pragma unroll
                            for (int c = 0; c < 4; ++c) { dqh[c] = ic[(size_t)(2 + c) * BSF]; dq[c] = ic[(size_t)(6 + c) * BSF]; }
#pragma unroll
                            for (int c = 0; c < 3; ++c) { av[c] = ic[(size_t)(10 + c) * BSF]; u[c] = ic[(size_t)(13 + c) * BSF]; }
                            // coefficients of F from the CARRIED rotmatI2G (A.3-2,3), as cov_coeffs forms them
                            const double ndt = -dt;
                            const double s0 = av[0] * ndt, s1 = av[1] * ndt, s2 = av[2] * ndt;
                            double rv[22];
#pragma unroll
                            for (int r = 0; r < 3; ++r) {
                                rv[r * 3 + 0] = fma(n.R[r * 3 + 1], s2, -FBUS_PROD(n.R[r * 3 + 2], s1));
                                rv[r * 3 + 1] = fma(n.R[r * 3 + 2], s0, -FBUS_PROD(n.R[r * 3 + 0], s2));
                                rv[r * 3 + 2] = fma(n.R[r * 3 + 0], s1, -FBUS_PROD(n.R[r * 3 + 1], s0));
#pragma unroll
                                for (int c = 0; c < 3; ++c) rv[9 + r * 3 + c] = n.R[r * 3 + c] * ndt;
                            }
                            rv[18] = u[0]; rv[19] = u[1]; rv[20] = u[2];  // -[w]x dt by its three numbers
                            rv[21] = dt;
                            double2* rec2 = reinterpret_cast<double2*>(ring2 + ((size_t)slot * 32 + (size_t)fl) * L2_RS);
#pragma unroll
                            for (int e = 0; e < 11; ++e) rec2[e] = make_double2(rv[2 * e], rv[2 * e + 1]);
                        }
                        __syncwarp();
                        slot_arrive(slot);  // record (slot) is complete
                        if (valid) {
                            // F2 after F1's coefficients were taken (filter.cpp:509-513): q of this sample side by side with v, p of
                            // the previous one
                            double q0[4], R0[9];  // quaternion and R(q) before this sample's step: operands of its own v, p half
#pragma unroll
                            for (int c = 0; c < 4; ++c) q0[c] = n.q[c];
#pragma unroll
                            for (int c = 0; c < 9; ++c) R0[c] = Rq[c];
                            nominal_apply_dual(n, Rq, pdt, pq, pdqh, pa, pR0, dq);
                            pdt = dt;
#pragma unroll
                            for (int c = 0; c < 4; ++c) { pq[c] = q0[c]; pdqh[c] = dqh[c]; }
#pragma unroll
                            for (int c = 0; c < 3; ++c) pa[c] = av[c];
#pragma unroll
                            for (int c = 0; c < 9; ++c) pR0[c] = R0[c];
                            n.t = ic[(size_t)BSF];
                            L2T(fl == 0, 0, 10 + slot);
                        }
                    }
                    cpar ^= 1u;
                    ts = ts_next;
                }
                nominal_apply_vp(n, pdt, pq, pdqh, pa, pR0, Rq);  // the last sample's v, p
                if (fused && do_prop) cursor = consumed;
            }
        } else
        if (lo < hi) {
            fs = (int)((hi - lo) & 1u);
            const double start = MATLAB ? t_img_frame : n.t;
            bool open = do_prop;          // false once this filter hit a sample later than t_end (the reference's break)
            uint32_t consumed = p_first;  // samples erased afterwards (filter.cpp:492-503,520)
            const bool pfi = (pf_i == lo);
            double s_t = pfi ? pf_st : prm.imu_t[lo], s_d[6];
#pragma unroll
            for (int c = 0; c < 6; ++c) s_d[c] = pfi ? pf_sd[c] : imu_sample_t<IMU32>(prm, k.imu_g, lo, c, B, b);
            for (uint32_t i = lo; i < hi; ++i) {
                const double ti = s_t;
                double d[6];
#pragma unroll
                for (int c = 0; c < 6; ++c) d[c] = s_d[c];
                if (i + 1 < hi) {  // prefetch the next sample
                    s_t = prm.imu_t[i + 1];
#pragma unroll
                    for (int c = 0; c < 6; ++c) s_d[c] = imu_sample_t<IMU32>(prm, k.imu_g, (size_t)i + 1, c, B, b);
                }
                const int slot = (int)((i - lo) & 1u);
                int valid = 0;
                if (open && i >= p_first && i < p_end) {
                    if (ti < start) {
                        consumed = i + 1;
                        if (MATLAB) n.t = ti;  // preImuTime moves on (FBUS_EKF.m:181)
                    } else if (ti > t_end) {
                        open = false;  // this sample stays buffered
                    } else {
                        consumed = i + 1;
                        valid = 1;
                        const double dt = ti - n.t;
                        double wv[3], av[3], A[9], Bm[9], u[3];
#pragma unroll
                        for (int c = 0; c < 3; ++c) { av[c] = d[c] - n.ba[c]; wv[c] = d[3 + c] - n.bg[c]; }
                        cov_coeffs(n.R, av, wv, dt, A, Bm, u);  // F1 uses the CARRIED rotmatI2G (A.3-2,3)
                        double* rec = X + (size_t)slot * REC * BSF;
#pragma unroll
                        for (int e = 0; e < 9; ++e) { rec[(size_t)e * BSF] = A[e]; rec[(size_t)(9 + e) * BSF] = Bm[e]; }
                        if constexpr (LANE) {  // W = F[theta,theta] - I in full
                            double Wm[9];
                            if constexpr (MATLAB) {
                                expm_rot_minus_I(wv, dt, Wm);  // ImuUpdate.m:68
                            } else {                            // -[w]x dt, filter.cpp:603
                                Wm[0] = 0.0; Wm[1] = u[2]; Wm[2] = -u[1];
                                Wm[3] = -u[2]; Wm[4] = 0.0; Wm[5] = u[0];
                                Wm[6] = u[1]; Wm[7] = -u[0]; Wm[8] = 0.0;
                            }
#pragma unroll
                            for (int e = 0; e < 9; ++e) rec[(size_t)(18 + e) * BSF] = Wm[e];
                            rec[(size_t)27 * BSF] = dt;
                        } else {
                            rec[(size_t)18 * BSF] = u[0]; rec[(size_t)19 * BSF] = u[1]; rec[(size_t)20 * BSF] = u[2];
                            rec[(size_t)21 * BSF] = dt;
                        }
                        if constexpr (MATLAB) propagate_nominal_matlab(n, dt, d, d + 3);
                        else propagate_nominal(n, dt, d, d + 3);  // F2 after F1's coefficients were taken (filter.cpp:509-513)
                        n.t = ti;
                    }
                }
                if (TM && !LANE && !valid) {  // tensor-memory mode: the covariance warp runs every lane, invalid ones with F = I
                    double* rec = X + (size_t)slot * REC * BSF;
#pragma unroll
                    for (int e = 0; e < 22; ++e) rec[(size_t)e * BSF] = 0.0;
                }
                sflag[slot][fl] = valid;
                sbar(wq);  // publish record (i); also: the covariance warp has finished sample i-1
            }
            if (fused && do_prop) cursor = consumed;
        }

        FramePlan nx;
        nx.do_prop = nx.apply_init = nx.apply_reset = false;
        nx.req = 0;
        for (uint32_t round = 0;; ++round) {
        bool rej = false;  // GATE: this round's update of this filter failed the gate
        // ---- F4 ObservationUpdate (filter.cpp:622-739): post the request (into the ring slot the covariance warp is
        //      not reading), the covariance warp does the algebra ------------------------------------------------
        if (req && !LANE) {
            double* rq = X + (size_t)fs * 22 * BSF;
#pragma unroll
            for (int c = 0; c < 7; ++c) rq[(size_t)c * BSF] = pl.y[c];  // yP (3), yQ (4)
#pragma unroll
            for (int c = 0; c < 4; ++c) rq[(size_t)(7 + c) * BSF] = n.q[c];
#pragma unroll
            for (int c = 0; c < 9; ++c) rq[(size_t)(11 + c) * BSF] = n.R[c];
            rq[(size_t)20 * BSF] = n.p[0]; rq[(size_t)21 * BSF] = n.p[1]; X[(size_t)RQ_EXTRA * BSF] = n.p[2];
        }
        sflag[2][fl] = req;
        {
            const int wany = __any_sync(0xffffffffu, req != 0);
            if ((fl & 31) == 0) sh.any_upd[wq] = wany;
        }
        L2T(LANE2 && fl == 0, 0, 5);
        sbar(wq);  // (r)
        L2T(LANE2 && fl == 0, 0, 6);
        const int any = pair_any(sh, wq);
        if constexpr (LANE) {
            if (any) {
                sbar(wq);  // (p) the covariance lanes have published P6
                L2T(LANE2 && fl == 0, 0, 7);
                if (req) {
                    const MarkerConst mkc = tab->mk[req - 1];
                    if constexpr (JOSEPH) {  // 6-row factor Lc of the Joseph-form C_J and y = Lc^-1 u
                        double Cm[21], yv[6], zg[7];
                        if constexpr (NOISE) {
                            const MeasNoise r{noise[4 * B + b], noise[5 * B + b]};
                            update_prologue<BSF, BSF, true, P6View>(P6View{X + (size_t)(LXS + LX_P6) * BSF}, n, k, r, mkc, pl.y, pl.y + 3, Cm,
                                                                    yv, X + (size_t)(LXS + LX_SCR) * BSF, GATE ? zg : nullptr);
                        } else if constexpr (GATE) {
                            update_prologue<BSF, BSF, true, P6View>(P6View{X + (size_t)(LXS + LX_P6) * BSF}, n, k, k, mkc, pl.y, pl.y + 3, Cm,
                                                                    yv, X + (size_t)(LXS + LX_SCR) * BSF, zg);
                        } else {
                            update_prologue<BSF, BSF, true, P6View>(P6View{X + (size_t)(LXS + LX_P6) * BSF}, n, k, mkc, pl.y, pl.y + 3, Cm, yv,
                                                                    X + (size_t)(LXS + LX_SCR) * BSF);
                        }
                        if constexpr (GATE) rej = gate_rejects(zg, gthr);
#pragma unroll
                        for (int c = 0; c < 21; ++c) X[(size_t)(LXS + LX_CM + c) * BSF] = Cm[c];
#pragma unroll
                        for (int c = 0; c < 6; ++c) X[(size_t)(LXS + LX_Y + c) * BSF] = yv[c];
                    } else {  // 7-row factor X = L^-1 Hs (left in the scratch entries) and z = L^-1 r: no second factorisation
                        // (computing Hs and r before the barrier, while the lanes finish, measured slower: the 37 doubles held
                        // across the wait spill at this kernel's 168 registers)
                        double L[28], Li[7], zv[7];
                        UpdHs hh;
                        update_hs<MATLAB>(n, k, mkc, pl.y, pl.y + 3, hh);
                        if constexpr (NOISE) {
                            const MeasNoise r{noise[4 * B + b], noise[5 * B + b]};
                            update_prologue_sx<BSF, BSF, P6View>(P6View{X + (size_t)(LXS + LX_P6) * BSF}, r, hh, L, Li, zv, X + (size_t)(LXS + LX_SCR) * BSF);
                        } else {
                            update_prologue_sx<BSF, BSF, P6View>(P6View{X + (size_t)(LXS + LX_P6) * BSF}, k, hh, L, Li, zv, X + (size_t)(LXS + LX_SCR) * BSF);
                        }
#pragma unroll
                        for (int c = 0; c < 7; ++c) X[(size_t)(LXS + LX_Y + c) * BSF] = zv[c];
                        if constexpr (GATE) rej = gate_rejects(zv, gthr);
                    }
                    if (GATE && rej) {  // withdrawn: the covariance lanes re-read the request after (c)
                        sflag[2][fl] = 0;
                        status |= FBUS_ST_UPDATE_REJECTED;
                        ++n_rej;
                    }
                }
                L2T(LANE2 && fl == 0, 0, 8);
                sbar(wq);  // (c) gain factors posted
            }
        }
        // ---- while the update runs: the next window's first IMU sample and the next frame's plan ---------------
        if (w + 1 < prm.w1 && (!ALL || round == 0)) {
            if (!LANE2 && fused && cursor < prm.win_off[prm.w1]) {  // (the second-generation lane kernel loads the samples in its covariance warps)
                pf_i = cursor;
                pf_st = prm.imu_t[cursor];
#pragma unroll
                for (int c = 0; c < 6; ++c) pf_sd[c] = imu_sample_t<IMU32>(prm, k.imu_g, cursor, c, B, b);
            }
            plan(w + 1, nx);
        }
        L2T(LANE2 && fl == 0, 0, 9);
        if (any) {
            sbar(wq);  // (d) results posted
            L2T(LANE2 && fl == 0, 0, 20);
            if (req && !rej) {
                if constexpr (LANE) {
                    double dx[18];
#pragma unroll
                    for (int c = 0; c < 18; ++c) dx[c] = X[(size_t)(LXS + LX_DX + c) * BSF];
                    inject_error_state(n, dx);  // rotmatI2G deliberately NOT refreshed (A.3-2)
                } else {
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        n.p[c] = X[(size_t)(23 + c) * BSF];
                        n.v[c] += X[(size_t)(30 + c) * BSF];
                        n.ba[c] += X[(size_t)(33 + c) * BSF];
                        n.bg[c] += X[(size_t)(36 + c) * BSF];
                        n.g[c] += X[(size_t)(39 + c) * BSF];
                    }
#pragma unroll
                    for (int c = 0; c < 4; ++c) n.q[c] = X[(size_t)(26 + c) * BSF];  // rotmatI2G deliberately NOT refreshed (A.3-2)
                }
            }
        }
        if constexpr (!ALL) {
            break;
        } else {  // FBUS_FLAG_ALL_MARKERS: this filter's next marker of the frame, if any; a round nobody requested ends the frame
            if (!any) break;
            req = 0;
            if (pl.extra) {
                const size_t slot = (size_t)w * prm.m + (__ffs(pl.extra) - 1);
                pl.extra &= pl.extra - 1u;
                req = find_marker(k, tab, prm.det_id[slot * B + b]) + 1;
                const double* pp = prm.det_pose + slot * 7 * B + b;
#pragma unroll
                for (int c = 0; c < 7; ++c) pl.y[c] = pp[(size_t)c * B];
            }
        }
        }
        // ---- trace row: the data/fusion.txt record (filter.cpp:241-246) -------------------------
        if (prm.trace && live) {
            double* row = prm.trace + (size_t)(w - prm.w0) * 17 * B + b;
            row[0] = n.t;
#pragma unroll
            for (int c = 0; c < 3; ++c) row[(size_t)(1 + c) * B] = n.p[c];
#pragma unroll
            for (int c = 0; c < 4; ++c) row[(size_t)(4 + c) * B] = n.q[c];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                row[(size_t)(8 + c) * B] = n.v[c];
                row[(size_t)(11 + c) * B] = n.ba[c];
                row[(size_t)(14 + c) * B] = n.bg[c];
            }
        }
        pl = nx;
        L2T(LANE2 && fl == 0, 0, 21);
    }
    if (!live) return;
    bool fin = isfinite(n.t);
#pragma unroll
    for (int i = 0; i < 4; ++i) fin = fin && isfinite(n.q[i]);
#pragma unroll
    for (int i = 0; i < 3; ++i) fin = fin && isfinite(n.p[i]) && isfinite(n.v[i]);
    if (!fin) status |= FBUS_ST_NONFINITE;
    prm.nom[(size_t)F_T * B + b] = n.t;
#pragma unroll
    for (int i = 0; i < 4; ++i) prm.nom[(size_t)(F_Q + i) * B + b] = n.q[i];
#pragma unroll
    for (int i = 0; i < 9; ++i) prm.nom[(size_t)(F_R + i) * B + b] = n.R[i];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        prm.nom[(size_t)(F_P + i) * B + b] = n.p[i];
        prm.nom[(size_t)(F_V + i) * B + b] = n.v[i];
        prm.nom[(size_t)(F_BA + i) * B + b] = n.ba[i];
        prm.nom[(size_t)(F_BG + i) * B + b] = n.bg[i];
        prm.nom[(size_t)(F_G + i) * B + b] = n.g[i];
    }
    prm.prev_id[b] = prev_id;
    prm.init[b] = inited;
    if (fused) prm.cursor_io[b] = cursor;
    prm.status[b] = status;
    if constexpr (GATE) gt.rejected[b] = n_rej;
    if (MATLAB) prm.nom[(size_t)F_TIMG * B + b] = t_img;
}

// Two CTAs can share an SM when BSF = 64 (2 x 110 KB of shared memory, 2 x 128 threads x 255 registers).  Warp w of
// every CTA lands on scheduler w % 4, so with a fixed role order both CTAs would stack their covariance warps on the
// same two schedulers.  Each CTA therefore takes an arrival ticket per SM: odd tickets swap the role order (covariance
// warps on schedulers 2,3 instead of 0,1) and start half a frame period late, so that one CTA's update phase (one busy
// warp per filter group) overlaps the other's propagation phase.
// IMU32: the IMU stream holds float32 sensor samples (FBUS_IMU_F32_SENSOR) instead of doubles
// NOISE: every filter has its own noise values, `noise` is the [6][B] buffer of fbus_set_noise (the other instantiations never
// read the parameter)
template <int BSF, bool JOSEPH, bool IMU32 = false, bool NOISE = false>  // filters per CTA; the CTA has 2*BSF threads
__global__ void __launch_bounds__(2 * BSF) ekf_window_split_kernel(const __grid_constant__ WinParams prm, const __grid_constant__ DevConsts k,
                                                                   const double* __restrict__ noise) {
    extern __shared__ double smem[];
    __shared__ SplitShared sh;
    __shared__ int32_t sflag[3][BSF];  // [0],[1]: ring slot valid ; [2]: update requested (marker index + 1, 0 = none)
    __shared__ uint32_t s_ticket;
    static_assert(BSF % 32 == 0 && BSF / 32 <= 8, "BSF must be a multiple of the warp size, at most 256");
    constexpr int NW = BSF / 32;
    uint32_t parity = 0;
    if (BSF < 128 && prm.sm_ticket != nullptr) {
        if (threadIdx.x == 0) {
            uint32_t smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            s_ticket = atomicAdd(prm.sm_ticket + (smid & 255u), 1u);
        }
        __syncthreads();
        parity = s_ticket & 1u;
        if (parity && prm.stagger_cycles > 0) {
            const long long t0 = clock64();
            while (clock64() - t0 < (long long)prm.stagger_cycles) { }
        }
    }
    const int wi = threadIdx.x >> 5;
    const bool is_cov = ((wi < NW) ? 1u : 0u) != parity;
    const int fl = (wi % NW) * 32 + (threadIdx.x & 31);  // filter lane inside the CTA
    const size_t b0 = (size_t)blockIdx.x * BSF + fl;
    const bool live = b0 < prm.B;
    const size_t b = live ? b0 : prm.B - 1;  // threads past the batch mirror the last filter and never store
    constexpr bool TM = (FBUS_TMEM != 0) && BSF == 128;
    uint32_t tm_base = 0;
    if constexpr (TM) {
        __shared__ uint32_t tm_slot;
        tm_base = tm_alloc_cta(&tm_slot);
    }
    if constexpr (NOISE) {
        double* sq = nullptr;
        if constexpr (noise_q_in_smem<BSF, TM>) {
            __shared__ double s_noise_q[4 * BSF];  // process noise of the CTA's filters: accel_n, gyro_n, accel_b, gyro_b
            sq = s_noise_q + fl;
        }
        if (is_cov) cov_role<BSF, JOSEPH, TM, true>(prm, k, smem, sh, sflag, fl, b, live, tm_base, noise, sq);
        else nominal_role<BSF, TM, IMU32>(prm, k, smem, sh, sflag, fl, b, live);
    } else {
        if (is_cov) cov_role<BSF, JOSEPH, TM>(prm, k, smem, sh, sflag, fl, b, live, tm_base);
        else nominal_role<BSF, TM, IMU32>(prm, k, smem, sh, sflag, fl, b, live);
    }
    if constexpr (TM) tm_free_cta(tm_base);
}

}  // namespace fbus
