// fbus_capi.cu -- implementation of the C ABI declared in include/fbus_ekf.h.
//
// Host side: handle, device buffers, staging of caller-owned host arrays, kernel launches on the
// handle's stream.  There is no CPU compute path: every entry point that does arithmetic launches a
// kernel from fbus_kernels.cuh, and fbus_create fails when no CUDA device is usable.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/fbus_ekf.h"
#include "fbus_host_consts.hpp"
#include "fbus_kernels.cuh"
#include "fbus_kernel_split.cuh"
#include "fbus_kernel_lane.cuh"

using namespace fbus;

namespace {

#ifndef FBUS_WIN_BS
#define FBUS_WIN_BS 128
#endif
constexpr size_t PACK_MAX = (size_t)256 << 10;  // host-resident calls up to this many input bytes take the packed single-copy path
constexpr int WIN_BS = FBUS_WIN_BS;  // filters per CTA of the window kernel; the CTA has 2*WIN_BS threads (covariance + nominal warps)
// the 128-filter CTAs keep P in tensor memory (FBUS_TMEM): shared memory then only holds the exchange area
constexpr bool WIN_TMEM = (FBUS_TMEM != 0) && WIN_BS == 128;
constexpr size_t WIN_SMEM = (size_t)((WIN_TMEM ? 0 : NPK) + XCH) * WIN_BS * sizeof(double);

thread_local std::string g_last_error;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

}  // namespace

struct fbus_handle {
    int device = 0;
    cudaStream_t stream = nullptr;
    size_t B = 0;
    fbus_config cfg;
    DevConsts k;
    MarkerTable tab;
    GnConsts gn;
    MarkerTable* d_tab = nullptr;
    uint32_t* d_ticket = nullptr;
    uint32_t* d_cursor = nullptr;  // [B] first unconsumed IMU sample per filter after the last fused call
    // identity of the last fused call, for the continuation rule of fbus_step_windows
    const void* last_imu_data = nullptr;
    size_t last_n_samples = 0, last_w1 = 0;
    uint32_t stagger_cycles = 0;
    size_t pipeline_min_bytes = (size_t)64 << 20;  // host streams smaller than this are staged and processed in one go
    bool small_batch = false;
    bool lane_batch = false;  // batches that leave SMs idle even with 32-filter CTAs: nine lanes per filter (fbus_kernel_lane.cuh)
    int lane_gen = 2;         // generation of the lanes-per-filter kernel (FBUS_LANE_GEN=1: the first one, kept for the MATLAB-semantics mode)
    uint32_t lane_fpc = 32;   // second generation: filters per CTA (the batch is spread over all SMs)
    double* d_nom = nullptr;
    double* d_P = nullptr;
    int32_t* d_prev = nullptr;
    int32_t* d_init = nullptr;
    int32_t* d_status = nullptr;
    DevBuf imu_t, det_t, win_off, imu_data, det_id, det_pose, trace, scratch_in, scratch_out, scratch_aux, stats_partial, stats_out;
    DevBuf noise;             // [6][B] per-filter noise values of fbus_set_noise (FBUS_NOISE_FIELDS rows, fbus_config order)
    bool noise_on = false;    // the window kernels read `noise` instead of the config's values
    bool noise_smem_set = false;  // shared-memory limits of the NOISE instantiations set (on the first fbus_set_noise)
    DevBuf errors;            // [4][B] device result of fbus_filter_errors for a host output
    DevBuf gate, gate_rej;    // [B] thresholds of fbus_set_gate, [B] int32 counts of rejected updates
    bool gate_on = false;     // the window launches go to the gated instantiations of the first-generation lane kernel
    bool gate_set = false;    // fbus_set_gate was called with an array: the counts exist
    bool gate_smem_set = false;  // shared-memory limits of the GATE instantiations set (on the first fbus_set_gate)
    // second staging set + copy stream: host-resident streams are copied chunk c+1 while chunk c is computed
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
    // small host-resident calls (the live single-filter use: one frame, ~8 IMU samples per call): every input array is packed into
    // one pinned buffer and goes to the device in ONE copy instead of six pageable ones
    char* pack_host = nullptr;  // pinned, PACK_MAX bytes
    char* pack_dev = nullptr;
    cudaEvent_t ev_pack = nullptr;  // the last packed copy has left pack_host
    size_t pipeline_frames = 2;  // frames per chunk of the host-stream pipeline (FBUS_PIPELINE_FRAMES, 0 = off)
    std::string err;
};

namespace {

int fail(fbus_handle* h, int code, const std::string& msg) {
    g_last_error = msg;
    if (h) h->err = msg;
    return code;
}
#define CUDA_TRY(h, expr)                                                                            \
    do {                                                                                             \
        cudaError_t _e = (expr);                                                                     \
        if (_e != cudaSuccess)                                                                       \
            return fail(h, FBUS_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));         \
    } while (0)

// Every memory kind a caller passes is checked here, before the call has any effect; the code after the check holds it as `host`.
int check_mem(fbus_handle* h, int32_t mem, const char* call, bool* host) {
    if (mem != FBUS_MEM_HOST && mem != FBUS_MEM_DEVICE)
        return fail(h, FBUS_E_BADARG, std::string(call) + ": memory kind must be FBUS_MEM_HOST or FBUS_MEM_DEVICE");
    *host = mem == FBUS_MEM_HOST;
    return FBUS_OK;
}

// IMU samples of either element format: bytes per value and the (imu, imu32) pointer pair of the kernels
inline size_t imu_elem(const fbus_imu_stream* imu) { return imu->format == FBUS_IMU_F32_SENSOR ? sizeof(float) : sizeof(double); }
inline void set_imu_ptr(const fbus_imu_stream* imu, const void* base, const double** p64, const float** p32) {
    const bool f32 = imu->format == FBUS_IMU_F32_SENSOR;
    *p64 = f32 ? nullptr : (const double*)base;
    *p32 = f32 ? (const float*)base : nullptr;
}

// an IMU stream of which the call reads samples [first, first + count), and their timestamps if need_t
int check_imu(fbus_handle* h, const fbus_imu_stream* imu, size_t first, size_t count, bool need_t, const char* call, bool* host) {
    if (!h || !imu || imu->batch != h->B || first > imu->n_samples || count > imu->n_samples - first || !imu->data ||
        (need_t && !imu->t) || (imu->format != FBUS_IMU_F64_SI && imu->format != FBUS_IMU_F32_SENSOR))
        return fail(h, FBUS_E_BADARG, std::string(call) + ": bad imu stream");
    return check_mem(h, imu->mem, call, host);
}

// detection frames of which the call reads frames [w0, w1)
int check_det(fbus_handle* h, const fbus_det_frames* det, size_t w0, size_t w1, const char* call, bool* host) {
    if (!det || det->batch != h->B || w1 > det->n_frames || w0 > w1 || det->max_markers == 0 || !det->t || !det->id || !det->pose)
        return fail(h, FBUS_E_BADARG, std::string(call) + ": bad detection frames");
    // the kernel keeps a frame's update slots as a 32-bit mask
    if ((h->k.flags & FBUS_FLAG_ALL_MARKERS) && det->max_markers > 32)
        return fail(h, FBUS_E_BADARG, std::string(call) + ": FBUS_FLAG_ALL_MARKERS: max_markers > 32");
    return check_mem(h, det->mem, call, host);
}

// A caller's input array on the device: host memory is copied into `buf` on the handle's stream, device memory is used in place.
template <class T>
int stage(fbus_handle* h, DevBuf& buf, const T* src, size_t count, bool host, const T** out) {
    if (!host) {
        *out = src;
        return FBUS_OK;
    }
    CUDA_TRY(h, buf.reserve(count * sizeof(T)));
    CUDA_TRY(h, cudaMemcpyAsync(buf.p, src, count * sizeof(T), cudaMemcpyHostToDevice, h->stream));
    *out = (const T*)buf.p;
    return FBUS_OK;
}
// values [first, first + count) of the stream's bulk array (values, not samples) on the device, as the kernels' pointer pair
int stage_imu(fbus_handle* h, const fbus_imu_stream* imu, bool host, size_t first, size_t count, const double** p64, const float** p32) {
    const size_t es = imu_elem(imu);
    const char* d;
    int rc = stage(h, h->imu_data, (const char*)imu->data + first * es, count * es, host, &d);
    if (rc == FBUS_OK) set_imu_ptr(imu, d, p64, p32);
    return rc;
}

// The outputs of a one-shot call.  Device memory: the kernel writes the caller's arrays.  Host memory: it writes handle
// scratch, which finish() copies back to every array the caller passed before it waits for the stream once.
struct Outputs {
    fbus_handle* h;
    bool host;
    int n = 0;
    struct { void* dst; const void* src; size_t bytes; } copy[3];

    int reserve(DevBuf& buf, size_t bytes) {
        if (host) CUDA_TRY(h, buf.reserve(bytes));
        return FBUS_OK;
    }
    // the array the kernel writes `count` elements of `dst` to: `dst` itself, or `scratch` (reserved) for host memory
    template <class T>
    T* to(T* dst, void* scratch, size_t count) {
        if (!host) return dst;
        if (dst) copy[n++] = {dst, scratch, count * sizeof(T)};
        return (T*)scratch;
    }
    int finish() {
        if (!host) return FBUS_OK;
        for (int i = 0; i < n; ++i) CUDA_TRY(h, cudaMemcpyAsync(copy[i].dst, copy[i].src, copy[i].bytes, cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        return FBUS_OK;
    }
};

// the continuation rule of fbus_step_windows ends here: the next fused call starts with an empty IMU buffer at win_off[w0]
inline void forget_stream_position(fbus_handle* h) {
    h->last_imu_data = nullptr;
    h->last_n_samples = 0;
    h->last_w1 = 0;
}

// NOISE: the instantiations that take every filter's noise values from h->noise (fbus_set_noise); the others get a null
// pointer they never read
// GATE: the innovation gate (fbus_set_gate): the gated first-generation lanes-per-filter kernel at any batch size; the lane
// kernel's other instantiations get null pointers they never read
template <bool NOISE, bool GATE>
int launch_window_t(fbus_handle* h, WinParams& prm) {
    prm.nom = h->d_nom;
    prm.P = h->d_P;
    prm.prev_id = h->d_prev;
    prm.init = h->d_init;
    prm.status = h->d_status;
    prm.B = h->B;
    prm.tab = h->d_tab;
    prm.sm_ticket = h->d_ticket;
    prm.cursor_io = h->d_cursor;
    prm.stagger_cycles = (prm.mode & M_FUSED) ? h->stagger_cycles : 0u;
    const unsigned grid = (unsigned)((h->B + WIN_BS - 1) / WIN_BS);
    const bool jo = (h->k.flags & FBUS_FLAG_JOSEPH) != 0, f32 = prm.imu32 != nullptr;
    const double* const nz = NOISE ? (const double*)h->noise.p : nullptr;
    const GateBufs gt{GATE ? (const double*)h->gate.p : nullptr, GATE ? (int32_t*)h->gate_rej.p : nullptr};
    if (GATE) {  // (fbus_set_gate refuses a MATLAB-semantics handle)
        const unsigned g32 = (unsigned)((h->B + 31) / 32);
        if (h->k.flags & FBUS_FLAG_ALL_MARKERS) {
            if (f32) {
                if (jo) ekf_window_lane_kernel<true, true, false, NOISE, true, true><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
                else ekf_window_lane_kernel<false, true, false, NOISE, true, true><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
            } else if (jo) ekf_window_lane_kernel<true, false, false, NOISE, true, true><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
            else ekf_window_lane_kernel<false, false, false, NOISE, true, true><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
        } else if (f32) {
            if (jo) ekf_window_lane_kernel<true, true, false, NOISE, false, true><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
            else ekf_window_lane_kernel<false, true, false, NOISE, false, true><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
        } else if (jo) ekf_window_lane_kernel<true, false, false, NOISE, false, true><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
        else ekf_window_lane_kernel<false, false, false, NOISE, false, true><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
    } else if (h->k.flags & FBUS_FLAG_ALL_MARKERS) {  // every marker of a frame: the first-generation lanes-per-filter kernel at any batch size
        const unsigned g32 = (unsigned)((h->B + 31) / 32);
        if (f32) {
            if (jo) ekf_window_lane_kernel<true, true, false, NOISE, true><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
            else ekf_window_lane_kernel<false, true, false, NOISE, true><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
        } else if (jo) ekf_window_lane_kernel<true, false, false, NOISE, true><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
        else ekf_window_lane_kernel<false, false, false, NOISE, true><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
    } else if (h->k.flags & FBUS_FLAG_MATLAB) {  // MATLAB-semantics mode: the lanes-per-filter kernel at any batch size
        const unsigned g32 = (unsigned)((h->B + 31) / 32);
        if (f32) ekf_window_lane_kernel<false, true, true, NOISE><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
        else ekf_window_lane_kernel<false, false, true, NOISE><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
    } else if (h->lane_batch && h->lane_gen == 2) {
        prm.lane_fpc = h->lane_fpc;
        const unsigned g32 = (unsigned)((h->B + h->lane_fpc - 1) / h->lane_fpc);
        if (f32) {
            if (jo) ekf_window_lane2_kernel<true, true, NOISE><<<g32, LANE_NT, LANE2_SMEM, h->stream>>>(prm, h->k, nz);
            else ekf_window_lane2_kernel<false, true, NOISE><<<g32, LANE_NT, LANE2_SMEM, h->stream>>>(prm, h->k, nz);
        } else if (jo) ekf_window_lane2_kernel<true, false, NOISE><<<g32, LANE_NT, LANE2_SMEM, h->stream>>>(prm, h->k, nz);
        else ekf_window_lane2_kernel<false, false, NOISE><<<g32, LANE_NT, LANE2_SMEM, h->stream>>>(prm, h->k, nz);
    } else if (h->lane_batch) {
        const unsigned g32 = (unsigned)((h->B + 31) / 32);
        if (f32) {
            if (jo) ekf_window_lane_kernel<true, true, false, NOISE><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
            else ekf_window_lane_kernel<false, true, false, NOISE><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
        } else if (jo) ekf_window_lane_kernel<true, false, false, NOISE><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
        else ekf_window_lane_kernel<false, false, false, NOISE><<<g32, LANE_NT, LANE_SMEM, h->stream>>>(prm, h->k, nz, gt);
    } else if (h->small_batch) {
        // fewer 128-filter CTAs than SMs (e.g. BASELINE configs[2], 4 096 filters): 32-filter CTAs (one covariance + one
        // nominal warp) spread the batch over four times as many SMs
        const unsigned g32 = (unsigned)((h->B + 31) / 32);
        const size_t smem32 = (size_t)(NPK + XCH) * 32 * sizeof(double);
        if (f32) {
            if (jo) ekf_window_split_kernel<32, true, true, NOISE><<<g32, 64, smem32, h->stream>>>(prm, h->k, nz);
            else ekf_window_split_kernel<32, false, true, NOISE><<<g32, 64, smem32, h->stream>>>(prm, h->k, nz);
        } else if (jo) ekf_window_split_kernel<32, true, false, NOISE><<<g32, 64, smem32, h->stream>>>(prm, h->k, nz);
        else ekf_window_split_kernel<32, false, false, NOISE><<<g32, 64, smem32, h->stream>>>(prm, h->k, nz);
    } else if (f32) {
        if (jo) ekf_window_split_kernel<WIN_BS, true, true, NOISE><<<grid, 2 * WIN_BS, WIN_SMEM, h->stream>>>(prm, h->k, nz);
        else ekf_window_split_kernel<WIN_BS, false, true, NOISE><<<grid, 2 * WIN_BS, WIN_SMEM, h->stream>>>(prm, h->k, nz);
    } else if (jo) ekf_window_split_kernel<WIN_BS, true, false, NOISE><<<grid, 2 * WIN_BS, WIN_SMEM, h->stream>>>(prm, h->k, nz);
    else ekf_window_split_kernel<WIN_BS, false, false, NOISE><<<grid, 2 * WIN_BS, WIN_SMEM, h->stream>>>(prm, h->k, nz);
    CUDA_TRY(h, cudaGetLastError());
    return FBUS_OK;
}
int launch_window(fbus_handle* h, WinParams& prm) {
    if (h->gate_on) return h->noise_on ? launch_window_t<true, true>(h, prm) : launch_window_t<false, true>(h, prm);
    return h->noise_on ? launch_window_t<true, false>(h, prm) : launch_window_t<false, false>(h, prm);
}

// the largest dynamic shared memory of every window kernel of one NOISE flavour (the default is 48 KB)
template <bool NOISE>
cudaError_t set_window_smem_limits() {
    const int smem32 = (int)((NPK + XCH) * 32 * sizeof(double));
    cudaError_t e = cudaSuccess;
    auto set = [&](const void* fn, size_t bytes) {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    };
    set((const void*)ekf_window_split_kernel<WIN_BS, false, false, NOISE>, WIN_SMEM);
    set((const void*)ekf_window_split_kernel<WIN_BS, true, false, NOISE>, WIN_SMEM);
    set((const void*)ekf_window_split_kernel<WIN_BS, false, true, NOISE>, WIN_SMEM);
    set((const void*)ekf_window_split_kernel<WIN_BS, true, true, NOISE>, WIN_SMEM);
    set((const void*)ekf_window_split_kernel<32, false, false, NOISE>, smem32);
    set((const void*)ekf_window_split_kernel<32, true, false, NOISE>, smem32);
    set((const void*)ekf_window_split_kernel<32, false, true, NOISE>, smem32);
    set((const void*)ekf_window_split_kernel<32, true, true, NOISE>, smem32);
    set((const void*)ekf_window_lane_kernel<false, false, false, NOISE>, LANE_SMEM);
    set((const void*)ekf_window_lane_kernel<true, false, false, NOISE>, LANE_SMEM);
    set((const void*)ekf_window_lane_kernel<false, true, false, NOISE>, LANE_SMEM);
    set((const void*)ekf_window_lane_kernel<true, true, false, NOISE>, LANE_SMEM);
    set((const void*)ekf_window_lane_kernel<false, false, true, NOISE>, LANE_SMEM);
    set((const void*)ekf_window_lane_kernel<false, true, true, NOISE>, LANE_SMEM);
    set((const void*)ekf_window_lane_kernel<false, false, false, NOISE, true>, LANE_SMEM);
    set((const void*)ekf_window_lane_kernel<true, false, false, NOISE, true>, LANE_SMEM);
    set((const void*)ekf_window_lane_kernel<false, true, false, NOISE, true>, LANE_SMEM);
    set((const void*)ekf_window_lane_kernel<true, true, false, NOISE, true>, LANE_SMEM);
    set((const void*)ekf_window_lane2_kernel<false, false, NOISE>, LANE2_SMEM);
    set((const void*)ekf_window_lane2_kernel<true, false, NOISE>, LANE2_SMEM);
    set((const void*)ekf_window_lane2_kernel<false, true, NOISE>, LANE2_SMEM);
    set((const void*)ekf_window_lane2_kernel<true, true, NOISE>, LANE2_SMEM);
    return e;
}
// the same for the GATE instantiations of the first-generation lane kernel (both NOISE flavours)
cudaError_t set_gate_smem_limits() {
    cudaError_t e = cudaSuccess;
    auto set = [&](const void* fn) {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LANE_SMEM);
    };
    set((const void*)ekf_window_lane_kernel<false, false, false, false, false, true>);
    set((const void*)ekf_window_lane_kernel<true, false, false, false, false, true>);
    set((const void*)ekf_window_lane_kernel<false, true, false, false, false, true>);
    set((const void*)ekf_window_lane_kernel<true, true, false, false, false, true>);
    set((const void*)ekf_window_lane_kernel<false, false, false, false, true, true>);
    set((const void*)ekf_window_lane_kernel<true, false, false, false, true, true>);
    set((const void*)ekf_window_lane_kernel<false, true, false, false, true, true>);
    set((const void*)ekf_window_lane_kernel<true, true, false, false, true, true>);
    set((const void*)ekf_window_lane_kernel<false, false, false, true, false, true>);
    set((const void*)ekf_window_lane_kernel<true, false, false, true, false, true>);
    set((const void*)ekf_window_lane_kernel<false, true, false, true, false, true>);
    set((const void*)ekf_window_lane_kernel<true, true, false, true, false, true>);
    set((const void*)ekf_window_lane_kernel<false, false, false, true, true, true>);
    set((const void*)ekf_window_lane_kernel<true, false, false, true, true, true>);
    set((const void*)ekf_window_lane_kernel<false, true, false, true, true, true>);
    set((const void*)ekf_window_lane_kernel<true, true, false, true, true, true>);
    return e;
}

// fbus_init_position_quaternion (M_INIT), fbus_reset_state (M_RESET) and fbus_update (M_UPDATE): one un-fused step of the
// window kernel on one frame, staged re-based to index 0
int step_frame(fbus_handle* h, const fbus_det_frames* det, size_t frame, int32_t mode, size_t n_imu_before, const char* call) {
    if (!h) return FBUS_E_BADARG;
    CUDA_TRY(h, cudaSetDevice(h->device));
    bool host;
    int rc = check_det(h, det, frame, frame + 1, call, &host);
    if (rc) return rc;
    const size_t m = det->max_markers, B = h->B;
    WinParams prm;
    memset(&prm, 0, sizeof prm);
    // timestamps are always host memory
    if ((rc = stage(h, h->det_t, det->t + frame, 1, true, &prm.det_t))) return rc;
    if ((rc = stage(h, h->det_id, det->id + frame * m * B, m * B, host, &prm.det_id))) return rc;
    if ((rc = stage(h, h->det_pose, det->pose + frame * m * 7 * B, m * 7 * B, host, &prm.det_pose))) return rc;
    prm.m = (int32_t)m;
    prm.w0 = 0;
    prm.w1 = 1;
    prm.mode = mode;
    prm.n_imu_before = (uint32_t)n_imu_before;
    if (mode == M_INIT) forget_stream_position(h);  // the un-fused initialisation stands outside any fused call's IMU buffer
    return launch_window(h, prm);
}

}  // namespace

extern "C" {

int fbus_abi_version(void) { return FBUS_ABI_VERSION; }

#ifdef FBUS_L2_TRACE
// experiment builds only (profiles/probes/lane2_trace.py): (tag, clock) pairs of one role, resets the counters
int fbus_debug_l2_trace(long long* out, int role, int max_pairs) {
    int n[2];
    if (cudaMemcpyFromSymbol(n, g_l2_trace_n, sizeof(n)) != cudaSuccess) return -1;
    int cnt = n[role] < max_pairs ? n[role] : max_pairs;
    if (cnt > 8192) cnt = 8192;
    if (cudaMemcpyFromSymbol(out, g_l2_trace, sizeof(long long) * 2 * cnt, sizeof(long long) * 16384 * role) != cudaSuccess) return -1;
    int z[2] = {0, 0};
    if (role == 1) cudaMemcpyToSymbol(g_l2_trace_n, z, sizeof(z));
    return cnt;
}
#endif

int fbus_config_default(fbus_config* cfg) {
    if (!cfg) return FBUS_E_BADARG;
    config_default(cfg);
    return FBUS_OK;
}
int fbus_config_matlab(fbus_config* cfg) {
    if (!cfg) return FBUS_E_BADARG;
    config_matlab(cfg);
    return FBUS_OK;
}

void fbus_quat_from_rotmat(const double R[9], double q[4]) { R2q(R, q); }

const char* fbus_last_error(const fbus_handle* h) { return h ? h->err.c_str() : g_last_error.c_str(); }

int fbus_create(fbus_handle** out, const fbus_config* cfg, int device, size_t batch) {
    if (!out || !cfg || batch == 0) return fail(nullptr, FBUS_E_BADARG, "fbus_create: bad argument");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, FBUS_E_CUDA, std::string("fbus_create: no usable CUDA device (") + cudaGetErrorString(e) +
                                              "); this library has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(nullptr, FBUS_E_BADARG, "fbus_create: bad device index");
    fbus_handle* h = new fbus_handle;
    h->device = device;
    h->B = batch;
    h->cfg = *cfg;
    if ((cfg->flags & FBUS_FLAG_MATLAB) && (cfg->flags & FBUS_FLAG_JOSEPH)) {
        delete h;
        return fail(nullptr, FBUS_E_BADARG, "fbus_create: FBUS_FLAG_MATLAB and FBUS_FLAG_JOSEPH cannot be combined");
    }
    if ((cfg->flags & FBUS_FLAG_MATLAB) && (cfg->flags & FBUS_FLAG_ALL_MARKERS)) {
        delete h;
        return fail(nullptr, FBUS_E_BADARG, "fbus_create: FBUS_FLAG_MATLAB and FBUS_FLAG_ALL_MARKERS cannot be combined");
    }
    if (make_dev_consts(cfg, &h->k, &h->tab) != FBUS_OK) {
        delete h;
        return fail(nullptr, FBUS_E_BADARG, "fbus_create: bad config (n_markers)");
    }
    make_gn_consts(cfg, &h->k, &h->gn);
    auto bail = [&](const char* what, cudaError_t ce) {
        std::string msg = std::string("fbus_create: ") + what + ": " + cudaGetErrorString(ce);
        fbus_destroy(h);
        return fail(nullptr, ce == cudaErrorMemoryAllocation ? FBUS_E_NOMEM : FBUS_E_CUDA, msg);
    };
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
    if ((e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    if ((e = cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate(copy)", e);
    for (int i = 0; i < 2; ++i) {
        if ((e = cudaEventCreateWithFlags(&h->ev_copied[i], cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
        if ((e = cudaEventCreateWithFlags(&h->ev_done[i], cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    }
    if ((e = cudaEventCreateWithFlags(&h->ev_pack, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    if ((e = cudaMallocHost((void**)&h->pack_host, PACK_MAX)) != cudaSuccess) return bail("cudaMallocHost pack", e);
    if ((e = cudaMalloc((void**)&h->pack_dev, PACK_MAX)) != cudaSuccess) return bail("cudaMalloc pack", e);
    if (const char* pf = getenv("FBUS_PIPELINE_FRAMES")) h->pipeline_frames = (size_t)strtoul(pf, nullptr, 10);
    if (const char* pm = getenv("FBUS_PIPELINE_MIN_MB")) h->pipeline_min_bytes = (size_t)strtoul(pm, nullptr, 10) << 20;
    if ((e = cudaMalloc(&h->d_nom, sizeof(double) * NOM_FIELDS * batch)) != cudaSuccess) return bail("cudaMalloc nom", e);
    if ((e = cudaMalloc(&h->d_P, sizeof(double) * NPK * batch)) != cudaSuccess) return bail("cudaMalloc P", e);
    if ((e = cudaMalloc(&h->d_prev, sizeof(int32_t) * batch)) != cudaSuccess) return bail("cudaMalloc prev", e);
    if ((e = cudaMalloc(&h->d_init, sizeof(int32_t) * batch)) != cudaSuccess) return bail("cudaMalloc init", e);
    if ((e = cudaMalloc(&h->d_status, sizeof(int32_t) * batch)) != cudaSuccess) return bail("cudaMalloc status", e);
    if ((e = cudaMalloc(&h->d_ticket, 256 * sizeof(uint32_t))) != cudaSuccess) return bail("cudaMalloc tickets", e);
    if ((e = cudaMemset(h->d_ticket, 0, 256 * sizeof(uint32_t))) != cudaSuccess) return bail("cudaMemset tickets", e);
    if ((e = cudaMalloc(&h->d_cursor, batch * sizeof(uint32_t))) != cudaSuccess) return bail("cudaMalloc cursor", e);
    if ((e = cudaMemset(h->d_cursor, 0, batch * sizeof(uint32_t))) != cudaSuccess) return bail("cudaMemset cursor", e);
    {
        const char* sc = getenv("FBUS_STAGGER_CYCLES");
        h->stagger_cycles = sc ? (uint32_t)strtoul(sc, nullptr, 10) : 0u;  // measured: no benefit, off by default
    }
    if ((e = cudaMalloc(&h->d_tab, sizeof(MarkerTable))) != cudaSuccess) return bail("cudaMalloc marker table", e);
    if ((e = cudaMemcpy(h->d_tab, &h->tab, sizeof(MarkerTable), cudaMemcpyHostToDevice)) != cudaSuccess) return bail("marker table copy", e);
    if ((e = set_window_smem_limits<false>()) != cudaSuccess) return bail("cudaFuncSetAttribute", e);
    {
        cudaDeviceProp prop;
        if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return bail("cudaGetDeviceProperties", e);
        // 32-filter CTAs (covariance in shared memory) only while at most two of them land on an SM: measured with
        // profiles/probes/batch_sweep.py they beat the 128-filter tensor-memory CTAs by ~5 % up to 8 192 filters and fall
        // to ~3e9 filter-steps/s beyond (three small CTAs per SM), where the large CTAs keep scaling with the SMs they fill
        h->small_batch = WIN_BS > 32 && (batch + 31) / 32 <= 2 * (size_t)prop.multiProcessorCount;
        if (const char* sb = getenv("FBUS_SMALL_BATCH")) h->small_batch = atoi(sb) != 0;
        // one 32-filter lanes-per-filter CTA per SM at most: below that the batch is latency-bound and nine lanes per filter
        // cut the latency of a filter-step ~3x; an explicit FBUS_SMALL_BATCH choice keeps the thread-per-filter kernels
        // Measured (profiles/probes/lane_gen_sweep.py): with a full 32-filter CTA the lanes-per-filter kernels are no faster per
        // frame than the 32-filter thread-per-filter CTAs (the CTA's one nominal warp, its schedulers and its shared-memory
        // bandwidth are shared by 32 filters); with at most 16 filters per CTA the second generation is 13-24 % faster.  So the
        // lane kernel takes the batches that can be spread at <= 16 filters per SM, as thin as the SM count allows.
        const size_t nsm = (size_t)prop.multiProcessorCount;
        h->lane_fpc = (uint32_t)((batch + nsm - 1) / nsm);
        h->lane_batch = !getenv("FBUS_SMALL_BATCH") && h->lane_fpc <= 16;
        if (const char* lb = getenv("FBUS_LANE")) h->lane_batch = atoi(lb) != 0;
        if (h->lane_fpc > 32) h->lane_fpc = 32;
        if (const char* fp = getenv("FBUS_LANE_FPC")) {
            const int v = atoi(fp);
            if (v >= 1 && v <= 32) h->lane_fpc = (uint32_t)v;
        }
        if (const char* lg = getenv("FBUS_LANE_GEN")) h->lane_gen = atoi(lg);
    }
    if (getenv("FBUS_DEBUG")) {
        int nb = -1;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, ekf_window_split_kernel<WIN_BS, false>, 2 * WIN_BS, WIN_SMEM);
        fprintf(stderr, "[fbus] window kernel: %d filters/CTA, %zu B dynamic smem, %d CTA(s)/SM\n", WIN_BS, WIN_SMEM, nb);
    }
    const unsigned grid = (unsigned)((batch + 127) / 128);
    ctor_kernel<<<grid, 128, 0, h->stream>>>(h->d_nom, h->d_P, h->d_prev, h->d_init, h->d_status, batch, cfg->p0_diag[0],
                                             cfg->p0_diag[1], cfg->p0_diag[2], cfg->p0_diag[3], cfg->p0_diag[4], cfg->p0_diag[5]);
    if ((e = cudaGetLastError()) != cudaSuccess) return bail("ctor_kernel", e);
    if ((e = cudaStreamSynchronize(h->stream)) != cudaSuccess) return bail("ctor sync", e);
    *out = h;
    return FBUS_OK;
}

int fbus_destroy(fbus_handle* h) {
    if (!h) return FBUS_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    cudaFree(h->d_nom); cudaFree(h->d_P); cudaFree(h->d_prev); cudaFree(h->d_init); cudaFree(h->d_status); cudaFree(h->d_tab); cudaFree(h->d_ticket); cudaFree(h->d_cursor);
    if (h->copy_stream) { cudaStreamSynchronize(h->copy_stream); cudaStreamDestroy(h->copy_stream); }
    if (h->ev_pack) cudaEventDestroy(h->ev_pack);
    if (h->pack_host) cudaFreeHost(h->pack_host);
    cudaFree(h->pack_dev);
    for (int i = 0; i < 2; ++i) {
        if (h->ev_copied[i]) cudaEventDestroy(h->ev_copied[i]);
        if (h->ev_done[i]) cudaEventDestroy(h->ev_done[i]);
    }
    DevBuf* bufs[] = {&h->imu_t, &h->det_t, &h->win_off, &h->imu_data, &h->det_id, &h->det_pose, &h->trace,
                      &h->scratch_in, &h->scratch_out, &h->scratch_aux, &h->stats_partial, &h->stats_out, &h->noise, &h->errors,
                      &h->gate, &h->gate_rej};
    for (DevBuf* b : bufs) b->release();
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return FBUS_OK;
}

int fbus_synchronize(fbus_handle* h) {
    if (!h) return FBUS_E_BADARG;
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return FBUS_OK;
}
size_t fbus_batch(const fbus_handle* h) { return h ? h->B : 0; }
void* fbus_stream(fbus_handle* h) { return h ? (void*)h->stream : nullptr; }

int fbus_init_gravity_gyrobias(fbus_handle* h, const fbus_imu_stream* imu, size_t first, size_t count) {
    bool host;
    int rc = check_imu(h, imu, first, count, false, "fbus_init_gravity_gyrobias", &host);
    if (rc) return rc;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (count == 0) return FBUS_OK;
    forget_stream_position(h);  // InitializeGravityAndBias clears the IMU buffer (filter.cpp:279)
    const double* d64;
    const float* d32;
    if ((rc = stage_imu(h, imu, host, first * 6 * h->B, count * 6 * h->B, &d64, &d32))) return rc;
    const unsigned grid = (unsigned)((h->B + 127) / 128);
    init_gravity_kernel<<<grid, 128, 0, h->stream>>>(h->d_nom, h->B, d64, d32, h->k.imu_g, 0u, (uint32_t)count);
    CUDA_TRY(h, cudaGetLastError());
    return FBUS_OK;
}

int fbus_iir_prefilter(fbus_handle* h, const fbus_imu_stream* imu, size_t first, size_t count, double* out, int32_t out_mem) {
    static const char* const call = "fbus_iir_prefilter";
    bool host, out_host;
    int rc = check_imu(h, imu, first, count, false, call, &host);
    if (rc) return rc;
    if (!out) return fail(h, FBUS_E_BADARG, "fbus_iir_prefilter: bad argument");
    if ((rc = check_mem(h, out_mem, call, &out_host))) return rc;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (count == 0) return FBUS_OK;
    const size_t n = count * 6 * h->B;
    const double* d64;
    const float* d32;
    if ((rc = stage_imu(h, imu, host, first * 6 * h->B, n, &d64, &d32))) return rc;
    Outputs o{h, out_host};
    if ((rc = o.reserve(h->scratch_out, n * sizeof(double)))) return rc;
    double* dout = o.to(out, h->scratch_out.p, n);
    const unsigned grid = (unsigned)((6 * h->B + 127) / 128);
    iir_prefilter_kernel<<<grid, 128, 0, h->stream>>>(d64, d32, h->k.imu_g, h->B, 0u, (uint32_t)count, dout);
    CUDA_TRY(h, cudaGetLastError());
    return o.finish();
}

int fbus_init_position_quaternion(fbus_handle* h, const fbus_det_frames* det, size_t frame, size_t n_imu_before) {
    return step_frame(h, det, frame, M_INIT, n_imu_before, "fbus_init_position_quaternion");
}

int fbus_propagate(fbus_handle* h, const fbus_imu_stream* imu, size_t first, size_t count, double t_end) {
    bool host;
    int rc = check_imu(h, imu, first, count, true, "fbus_propagate", &host);
    if (rc) return rc;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (count == 0) return FBUS_OK;
    WinParams prm;
    memset(&prm, 0, sizeof prm);
    if ((rc = stage(h, h->imu_t, imu->t + first, count, true, &prm.imu_t))) return rc;
    if ((rc = stage_imu(h, imu, host, first * 6 * h->B, count * 6 * h->B, &prm.imu, &prm.imu32))) return rc;
    prm.mode = M_PROP;
    prm.prop_first = 0;
    prm.prop_count = (uint32_t)count;
    prm.prop_t_end = t_end;
    prm.w0 = 0;
    prm.w1 = 1;
    return launch_window(h, prm);
}

int fbus_reset_state(fbus_handle* h, const fbus_det_frames* det, size_t frame) {
    return step_frame(h, det, frame, M_RESET, 0, "fbus_reset_state");
}

int fbus_update(fbus_handle* h, const fbus_det_frames* det, size_t frame) {
    return step_frame(h, det, frame, M_UPDATE, 0, "fbus_update");
}

// Fused frames [w0, w1) of a stream.  The kernel indexes the stream with absolute sample / frame numbers (the small host arrays
// t, win_off, det_t are staged in full up to the end of the range; device-resident bulk arrays are used in place), so that a
// continuation can reach samples a filter has not consumed yet.
//   host-resident bulk arrays, one launch : samples [win_off[w0], win_off[w1]) and frames [w0, w1) are staged (no continuation)
//   host-resident, pipelined             : device buffers for the whole range, filled chunk by chunk on the copy stream while the
//                                          previous chunk is computed; chunks after the first continue (cursor_resume)
static int step_windows_range(fbus_handle* h, const fbus_imu_stream* imu, bool imu_host, const fbus_det_frames* det, bool det_host,
                              const uint32_t* win_off, size_t w0, size_t w1, double* trace, bool trace_host, bool resume,
                              size_t chunk_frames) {
    const size_t B = h->B, nw = w1 - w0, m = det->max_markers;
    const size_t s0 = win_off[w0], s1 = win_off[w1];
    WinParams prm;
    memset(&prm, 0, sizeof prm);
    const size_t es = imu_elem(imu);  // bytes per IMU value: double (SI) or float (sensor units)
    // Small host-resident call (the live use: one filter, one frame): all six input arrays travel in one pinned buffer and one copy.
    // Layout (16-byte aligned pieces): t[0, s1) | det_t[0, w1) | pose[w0, w1) | imu[s0, s1) | win_off[0, w1] | id[w0, w1)
    auto al16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
    const size_t nb_t = al16((s1 ? s1 : 1) * sizeof(double)), nb_dt = al16(w1 * sizeof(double)), nb_pose = al16(nw * m * 7 * B * sizeof(double));
    const size_t nb_imu = al16((s1 - s0) * 6 * B * es), nb_off = al16((w1 + 1) * sizeof(uint32_t)), nb_id = al16(nw * m * B * sizeof(int32_t));
    const size_t nb_all = nb_t + nb_dt + nb_pose + nb_imu + nb_off + nb_id;
    const bool packed = imu_host && det_host && chunk_frames == 0 && h->pack_host && nb_all <= PACK_MAX;
    // small host arrays, staged in full so that absolute indices work: t[0, s1), win_off[0, w1], det_t[0, w1)
    const double* dt;
    const double* ddt;
    const uint32_t* doff;
    int rc;
    // bulk arrays: device-resident ones in place; host-resident ones into buffers that hold the range [s0, s1) / [w0, w1),
    // addressed through base pointers shifted back to index 0 (never dereferenced below the range)
    const char* dimu = (const char*)imu->data;
    const int32_t* did = det->id;
    const double* dpose = det->pose;
    if (packed) {
        CUDA_TRY(h, cudaEventSynchronize(h->ev_pack));  // the previous packed copy has read the pinned buffer
        char* ph = h->pack_host;
        const size_t o_t = 0, o_dt = o_t + nb_t, o_pose = o_dt + nb_dt, o_imu = o_pose + nb_pose, o_off = o_imu + nb_imu, o_id = o_off + nb_off;
        if (s1) memcpy(ph + o_t, imu->t, s1 * sizeof(double));  // s1 == 0: nothing of imu->t is read (the kernel indexes no sample)
        memcpy(ph + o_dt, det->t, w1 * sizeof(double));
        memcpy(ph + o_pose, det->pose + w0 * m * 7 * B, nw * m * 7 * B * sizeof(double));
        if (s1 > s0) memcpy(ph + o_imu, (const char*)imu->data + s0 * 6 * B * es, (s1 - s0) * 6 * B * es);
        memcpy(ph + o_off, win_off, (w1 + 1) * sizeof(uint32_t));
        memcpy(ph + o_id, det->id + w0 * m * B, nw * m * B * sizeof(int32_t));
        CUDA_TRY(h, cudaMemcpyAsync(h->pack_dev, ph, nb_all, cudaMemcpyHostToDevice, h->stream));
        CUDA_TRY(h, cudaEventRecord(h->ev_pack, h->stream));
        dt = (const double*)(h->pack_dev + o_t);
        ddt = (const double*)(h->pack_dev + o_dt);
        doff = (const uint32_t*)(h->pack_dev + o_off);
        dimu = h->pack_dev + o_imu - s0 * 6 * B * es;
        did = (const int32_t*)(h->pack_dev + o_id) - w0 * m * B;
        dpose = (const double*)(h->pack_dev + o_pose) - w0 * m * 7 * B;
    } else {
        if (s1) {
            rc = stage(h, h->imu_t, imu->t, s1, true, &dt);
            if (rc) return rc;
        } else {  // an empty sample range: imu->t may be empty too, the kernel indexes no sample
            CUDA_TRY(h, h->imu_t.reserve(sizeof(double)));
            dt = (const double*)h->imu_t.p;
        }
        rc = stage(h, h->win_off, win_off, w1 + 1, true, &doff);
        if (rc) return rc;
        rc = stage(h, h->det_t, det->t, w1, true, &ddt);
        if (rc) return rc;
    }
    if (imu_host && !packed) {
        CUDA_TRY(h, h->imu_data.reserve((s1 - s0 ? s1 - s0 : 1) * 6 * B * es));
        dimu = (const char*)h->imu_data.p - s0 * 6 * B * es;
    }
    if (det_host && !packed) {
        CUDA_TRY(h, h->det_id.reserve(nw * m * B * sizeof(int32_t)));
        CUDA_TRY(h, h->det_pose.reserve(nw * m * 7 * B * sizeof(double)));
        did = (const int32_t*)h->det_id.p - w0 * m * B;
        dpose = (const double*)h->det_pose.p - w0 * m * 7 * B;
    }
    double* dtrace = nullptr;
    if (trace) {
        if (!trace_host) dtrace = trace;
        else {
            CUDA_TRY(h, h->trace.reserve(nw * 17 * B * sizeof(double)));
            dtrace = (double*)h->trace.p;
        }
    }
    prm.imu_t = dt;
    set_imu_ptr(imu, dimu, &prm.imu, &prm.imu32);
    prm.win_off = doff;
    prm.det_t = ddt;
    prm.det_id = did;
    prm.det_pose = dpose;
    prm.m = (int32_t)m;
    prm.mode = M_FUSED;
    const bool piped = chunk_frames > 0 && h->copy_stream != nullptr;
    cudaStream_t cs = piped ? h->copy_stream : h->stream;
    if (piped) {  // the range buffers may still be read by earlier work on the main stream
        CUDA_TRY(h, cudaEventRecord(h->ev_done[0], h->stream));
        CUDA_TRY(h, cudaStreamWaitEvent(cs, h->ev_done[0], 0));
    }
    const size_t step = piped ? chunk_frames : nw;
    int c = 0;
    for (size_t a = w0; a < w1; a += step, ++c) {
        const size_t e = (a + step < w1) ? a + step : w1;
        const size_t sa = win_off[a], se = win_off[e];
        if (imu_host && !packed && se > sa)
            CUDA_TRY(h, cudaMemcpyAsync((char*)h->imu_data.p + (sa - s0) * 6 * B * es, (const char*)imu->data + sa * 6 * B * es,
                                        (se - sa) * 6 * B * es, cudaMemcpyHostToDevice, cs));
        if (det_host && !packed) {
            CUDA_TRY(h, cudaMemcpyAsync((int32_t*)h->det_id.p + (a - w0) * m * B, det->id + a * m * B, (e - a) * m * B * sizeof(int32_t),
                                        cudaMemcpyHostToDevice, cs));
            CUDA_TRY(h, cudaMemcpyAsync((double*)h->det_pose.p + (a - w0) * m * 7 * B, det->pose + a * m * 7 * B,
                                        (e - a) * m * 7 * B * sizeof(double), cudaMemcpyHostToDevice, cs));
        }
        if (piped) {
            CUDA_TRY(h, cudaEventRecord(h->ev_copied[c & 1], cs));
            CUDA_TRY(h, cudaStreamWaitEvent(h->stream, h->ev_copied[c & 1], 0));
        }
        prm.w0 = (uint32_t)a;
        prm.w1 = (uint32_t)e;
        prm.cursor_resume = (resume || c > 0) ? 1 : 0;
        prm.trace = dtrace ? dtrace + (a - w0) * 17 * B : nullptr;
        rc = launch_window(h, prm);
        if (rc) return rc;
    }
    if (trace && trace_host) {
        CUDA_TRY(h, cudaMemcpyAsync(trace, dtrace, nw * 17 * B * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    }
    return FBUS_OK;
}

int fbus_step_windows(fbus_handle* h, const fbus_imu_stream* imu, const fbus_det_frames* det, const uint32_t* win_off,
                      size_t w0, size_t w1, double* trace, int32_t trace_mem) {
    static const char* const call = "fbus_step_windows";
    bool imu_host, det_host, trace_host;
    if (!det || !win_off) return fail(h, FBUS_E_BADARG, "fbus_step_windows: bad argument");
    // samples [0, win_off[w1]): the kernel indexes the stream with absolute sample numbers
    int rc = check_imu(h, imu, 0, w0 < w1 ? win_off[w1] : 0, true, call, &imu_host);
    if (rc) return rc;
    if ((rc = check_mem(h, trace_mem, call, &trace_host))) return rc;
    if (w0 >= w1) return (w0 == w1) ? FBUS_OK : fail(h, FBUS_E_BADARG, "fbus_step_windows: w0 > w1");
    CUDA_TRY(h, cudaSetDevice(h->device));
    for (size_t w = w0; w < w1; ++w)
        if (win_off[w + 1] < win_off[w]) return fail(h, FBUS_E_BADARG, "fbus_step_windows: win_off must be non-decreasing");
    if ((rc = check_det(h, det, w0, w1, call, &det_host))) {  // a bad detection descriptor ends the continuation
        forget_stream_position(h);
        return rc;
    }
    const size_t nw = w1 - w0, B = h->B;
    // Continuation (see the header): the call picks up where the previous one on this handle stopped -- same device-resident
    // IMU array, w0 equal to the previous w1 -- so samples a filter has not consumed yet stay buffered across the two calls.
    const bool device_streams = !imu_host && !det_host;
    const bool resume = device_streams && w0 > 0 && w0 == h->last_w1 && imu->data == h->last_imu_data && imu->n_samples == h->last_n_samples;
    // Host-resident streams that are large enough to matter: pipeline the frames in chunks so that the PCIe copy of
    // chunk c+1 runs while chunk c is computed (the state makes one extra HBM round trip per chunk).
    const size_t ch = h->pipeline_frames;
    const size_t bytes = (size_t)(win_off[w1] - win_off[w0]) * 6 * imu_elem(imu) * B;
    const bool piped = imu_host && det_host && ch > 0 && nw >= 2 * ch && bytes >= h->pipeline_min_bytes && h->copy_stream;
    rc = step_windows_range(h, imu, imu_host, det, det_host, win_off, w0, w1, trace, trace_host, resume, piped ? ch : 0);
    // a failed call leaves nothing to continue from
    h->last_imu_data = (device_streams && rc == FBUS_OK) ? (const void*)imu->data : nullptr;
    h->last_n_samples = imu->n_samples;
    h->last_w1 = (rc == FBUS_OK) ? w1 : 0;
    return rc;
}

static int stereo_solve(fbus_handle* h, const float* corners, size_t n, double* pose, double* corners3d, int32_t* valid, int32_t mem,
                        bool underwater);
int fbus_refract_solve(fbus_handle* h, const float* corners, size_t n, double* pose, double* corners3d, int32_t* valid, int32_t mem) {
    return stereo_solve(h, corners, n, pose, corners3d, valid, mem, true);
}
int fbus_inair_solve(fbus_handle* h, const float* corners, size_t n, double* pose, double* corners3d, int32_t* valid, int32_t mem) {
    return stereo_solve(h, corners, n, pose, corners3d, valid, mem, false);
}
static int stereo_solve(fbus_handle* h, const float* corners, size_t n, double* pose, double* corners3d, int32_t* valid, int32_t mem,
                        bool underwater) {
    const char* const call = underwater ? "fbus_refract_solve" : "fbus_inair_solve";
    if (!h || !corners || !pose) return fail(h, FBUS_E_BADARG, std::string(call) + ": bad argument");
    bool host;
    int rc = check_mem(h, mem, call, &host);
    if (rc) return rc;
    if (n == 0) return FBUS_OK;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (!host) {
        const unsigned grid = (unsigned)((n + 127) / 128);
        if (underwater) refract_kernel<<<grid, 128, 0, h->stream>>>(h->k, corners, n, n, pose, corners3d, valid);
        else inair_kernel<<<grid, 128, 0, h->stream>>>(h->k, corners, n, n, pose, corners3d, valid);
        CUDA_TRY(h, cudaGetLastError());
        return FBUS_OK;
    }
    // Host arrays: the [16][n] / [7][n] / [12][n] arrays are cut into column chunks; the H2D copy of chunk c+1 (second stream)
    // overlaps the kernel and the D2H copy of chunk c (PCIe is full duplex), so a call costs about one direction's transfer.
    CUDA_TRY(h, h->scratch_in.reserve(16 * n * sizeof(float)));
    CUDA_TRY(h, h->scratch_out.reserve((7 + 12) * n * sizeof(double)));
    CUDA_TRY(h, h->scratch_aux.reserve(n * sizeof(int32_t)));
    float* dc = (float*)h->scratch_in.p;
    double* dpose = (double*)h->scratch_out.p;
    double* dc3 = dpose + 7 * n;
    int32_t* dvalid = (int32_t*)h->scratch_aux.p;
    const bool piped = h->copy_stream != nullptr && n >= 65536;
    const size_t nch = piped ? 4 : 1;  // few chunks: at ~1 ms per call the API calls per chunk (~30 us) matter
    const size_t step = ((n + nch - 1) / nch + 127) / 128 * 128;
    cudaStream_t cs = piped ? h->copy_stream : h->stream;
    if (piped) {  // the staging buffers may still be read by earlier work on the main stream
        CUDA_TRY(h, cudaEventRecord(h->ev_done[0], h->stream));
        CUDA_TRY(h, cudaStreamWaitEvent(cs, h->ev_done[0], 0));
    }
    int c = 0;
    for (size_t a = 0; a < n; a += step, ++c) {
        const size_t m = (a + step <= n) ? step : n - a;
        CUDA_TRY(h, cudaMemcpy2DAsync(dc + a, n * sizeof(float), corners + a, n * sizeof(float), m * sizeof(float), 16, cudaMemcpyHostToDevice, cs));
        if (piped) {
            CUDA_TRY(h, cudaEventRecord(h->ev_copied[c & 1], cs));
            CUDA_TRY(h, cudaStreamWaitEvent(h->stream, h->ev_copied[c & 1], 0));
        }
        const unsigned grid = (unsigned)((m + 127) / 128);
        if (underwater) refract_kernel<<<grid, 128, 0, h->stream>>>(h->k, dc + a, m, n, dpose + a, dc3 + a, dvalid + a);
        else inair_kernel<<<grid, 128, 0, h->stream>>>(h->k, dc + a, m, n, dpose + a, dc3 + a, dvalid + a);
        CUDA_TRY(h, cudaGetLastError());
        CUDA_TRY(h, cudaMemcpy2DAsync(pose + a, n * sizeof(double), dpose + a, n * sizeof(double), m * sizeof(double), 7, cudaMemcpyDeviceToHost, h->stream));
        if (corners3d)
            CUDA_TRY(h, cudaMemcpy2DAsync(corners3d + a, n * sizeof(double), dc3 + a, n * sizeof(double), m * sizeof(double), 12, cudaMemcpyDeviceToHost,
                                          h->stream));
        if (valid) CUDA_TRY(h, cudaMemcpyAsync(valid + a, dvalid + a, m * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    }
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return FBUS_OK;
}

int fbus_solve_to_detections(fbus_handle* h, const float* corners, const int32_t* marker_ids, size_t n_frames, size_t max_markers,
                             int32_t underwater, int32_t gn_iters, int32_t* det_id, double* det_pose, int32_t mem) {
    if (!h || !corners || !marker_ids || !det_id || !det_pose || max_markers == 0 || gn_iters < 0 || gn_iters > 50)
        return fail(h, FBUS_E_BADARG, "fbus_solve_to_detections: bad argument");
    bool host;
    int rc = check_mem(h, mem, "fbus_solve_to_detections", &host);
    if (rc) return rc;
    const size_t n = n_frames * max_markers * h->B;
    if (n == 0) return FBUS_OK;
    CUDA_TRY(h, cudaSetDevice(h->device));
    const float* dc;
    const int32_t* di;
    if ((rc = stage(h, h->scratch_in, corners, 16 * n, host, &dc))) return rc;
    if ((rc = stage(h, h->scratch_aux, marker_ids, n, host, &di))) return rc;
    Outputs o{h, host};
    if ((rc = o.reserve(h->scratch_out, 7 * n * sizeof(double) + n * sizeof(int32_t)))) return rc;
    double* opose = o.to(det_pose, h->scratch_out.p, 7 * n);
    int32_t* oid = o.to(det_id, (double*)h->scratch_out.p + 7 * n, n);
    solve_to_det_kernel<<<(unsigned)((n + 127) / 128), 128, 0, h->stream>>>(h->k, h->gn, dc, di, n, h->B, underwater, gn_iters, oid, opose);
    CUDA_TRY(h, cudaGetLastError());
    return o.finish();
}

int fbus_undistort_fisheye(fbus_handle* h, const float* pixels, size_t n, float* normalised, int32_t mem) {
    if (!h || !pixels || !normalised) return fail(h, FBUS_E_BADARG, "fbus_undistort_fisheye: bad argument");
    bool host;
    int rc = check_mem(h, mem, "fbus_undistort_fisheye", &host);
    if (rc) return rc;
    if (n == 0) return FBUS_OK;
    CUDA_TRY(h, cudaSetDevice(h->device));
    const float* dp;
    if ((rc = stage(h, h->scratch_in, pixels, 16 * n, host, &dp))) return rc;
    Outputs o{h, host};
    if ((rc = o.reserve(h->scratch_out, 16 * n * sizeof(float)))) return rc;
    float* dout = o.to(normalised, h->scratch_out.p, 16 * n);
    undistort_kernel<<<(unsigned)((n + 127) / 128), 128, 0, h->stream>>>(h->k, dp, n, dout);
    CUDA_TRY(h, cudaGetLastError());
    return o.finish();
}

int fbus_refract_solve_gn(fbus_handle* h, const void* corners, int32_t corner_dtype, size_t n, int32_t iters, double* pose,
                          double* cost, int32_t* valid, int32_t mem) {
    if (!h || !corners || !pose || iters < 0 || iters > 50 || (corner_dtype != 0 && corner_dtype != 1))
        return fail(h, FBUS_E_BADARG, "fbus_refract_solve_gn: bad argument");
    bool host;
    int rc = check_mem(h, mem, "fbus_refract_solve_gn", &host);
    if (rc) return rc;
    if (n == 0) return FBUS_OK;
    CUDA_TRY(h, cudaSetDevice(h->device));
    const size_t esz = corner_dtype ? sizeof(double) : sizeof(float);
    const char* dc;
    if ((rc = stage(h, h->scratch_in, (const char*)corners, 16 * n * esz, host, &dc))) return rc;
    Outputs o{h, host};
    if ((rc = o.reserve(h->scratch_out, (7 + 1) * n * sizeof(double)))) return rc;
    if ((rc = o.reserve(h->scratch_aux, n * sizeof(int32_t)))) return rc;
    // for host memory the kernel writes cost and valid to scratch even when the caller does not want them
    double* dpose = o.to(pose, h->scratch_out.p, 7 * n);
    double* dcost = o.to(cost, (double*)h->scratch_out.p + 7 * n, n);
    int32_t* dvalid = o.to(valid, h->scratch_aux.p, n);
    const unsigned grid = (unsigned)((n + 127) / 128);
    if (corner_dtype) refract_gn_kernel<double><<<grid, 128, 0, h->stream>>>(h->k, h->gn, (const double*)dc, n, iters, dpose, dcost, dvalid);
    else refract_gn_kernel<float><<<grid, 128, 0, h->stream>>>(h->k, h->gn, (const float*)dc, n, iters, dpose, dcost, dvalid);
    CUDA_TRY(h, cudaGetLastError());
    return o.finish();
}

int fbus_marker_pose(fbus_handle* h, const double* corners3d, size_t n, double* pose, int32_t mem) {
    if (!h || !corners3d || !pose) return fail(h, FBUS_E_BADARG, "fbus_marker_pose: bad argument");
    bool host;
    int rc = check_mem(h, mem, "fbus_marker_pose", &host);
    if (rc) return rc;
    if (n == 0) return FBUS_OK;
    CUDA_TRY(h, cudaSetDevice(h->device));
    const double* dc;
    if ((rc = stage(h, h->scratch_in, corners3d, 12 * n, host, &dc))) return rc;
    Outputs o{h, host};
    if ((rc = o.reserve(h->scratch_out, 7 * n * sizeof(double)))) return rc;
    double* dpose = o.to(pose, h->scratch_out.p, 7 * n);
    const unsigned grid = (unsigned)((n + 127) / 128);
    marker_pose_kernel<<<grid, 128, 0, h->stream>>>(h->k, dc, n, dpose);
    CUDA_TRY(h, cudaGetLastError());
    return o.finish();
}

int fbus_get_state(fbus_handle* h, fbus_state_soa* out) {
    if (!h || !out || out->batch != h->B) return fail(h, FBUS_E_BADARG, "fbus_get_state: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->device));
    const size_t B = h->B;
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    struct { double* dst; int field; int n; } f[] = {{out->t, F_T, 1}, {out->q, F_Q, 4}, {out->R, F_R, 9}, {out->p, F_P, 3},
                                                     {out->v, F_V, 3}, {out->ba, F_BA, 3}, {out->bg, F_BG, 3}, {out->g, F_G, 3},
                                                     {out->pv, F_PV, 3}, {out->qv, F_QV, 4}};
    for (auto& x : f)
        if (x.dst) CUDA_TRY(h, cudaMemcpy(x.dst, h->d_nom + (size_t)x.field * B, sizeof(double) * x.n * B, cudaMemcpyDeviceToHost));
    if (out->prev_marker_id) CUDA_TRY(h, cudaMemcpy(out->prev_marker_id, h->d_prev, sizeof(int32_t) * B, cudaMemcpyDeviceToHost));
    if (out->initialised) CUDA_TRY(h, cudaMemcpy(out->initialised, h->d_init, sizeof(int32_t) * B, cudaMemcpyDeviceToHost));
    if (out->status) CUDA_TRY(h, cudaMemcpy(out->status, h->d_status, sizeof(int32_t) * B, cudaMemcpyDeviceToHost));
    if (out->P) {
        std::vector<double> pk((size_t)NPK * B);
        CUDA_TRY(h, cudaMemcpy(pk.data(), h->d_P, sizeof(double) * NPK * B, cudaMemcpyDeviceToHost));
        for (int i = 0; i < NX; ++i)
            for (int j = 0; j < NX; ++j) memcpy(out->P + (size_t)(i * NX + j) * B, pk.data() + (size_t)pidx(i, j) * B, sizeof(double) * B);
    }
    return FBUS_OK;
}

int fbus_set_state(fbus_handle* h, const fbus_state_soa* in) {
    if (!h || !in || in->batch != h->B) return fail(h, FBUS_E_BADARG, "fbus_set_state: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->device));
    forget_stream_position(h);  // an overwritten state does not continue the previous fused call's IMU buffer
    const size_t B = h->B;
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    struct { const double* src; int field; int n; } f[] = {{in->t, F_T, 1}, {in->q, F_Q, 4}, {in->R, F_R, 9}, {in->p, F_P, 3},
                                                           {in->v, F_V, 3}, {in->ba, F_BA, 3}, {in->bg, F_BG, 3}, {in->g, F_G, 3},
                                                           {in->pv, F_PV, 3}, {in->qv, F_QV, 4}};
    for (auto& x : f)
        if (x.src) CUDA_TRY(h, cudaMemcpy(h->d_nom + (size_t)x.field * B, x.src, sizeof(double) * x.n * B, cudaMemcpyHostToDevice));
    if (in->prev_marker_id) CUDA_TRY(h, cudaMemcpy(h->d_prev, in->prev_marker_id, sizeof(int32_t) * B, cudaMemcpyHostToDevice));
    if (in->initialised) CUDA_TRY(h, cudaMemcpy(h->d_init, in->initialised, sizeof(int32_t) * B, cudaMemcpyHostToDevice));
    if (in->status) CUDA_TRY(h, cudaMemcpy(h->d_status, in->status, sizeof(int32_t) * B, cudaMemcpyHostToDevice));
    if (in->P) {
        std::vector<double> pk((size_t)NPK * B);
        for (int i = 0; i < NX; ++i)
            for (int j = i; j < NX; ++j) memcpy(pk.data() + (size_t)pidx_u(i, j) * B, in->P + (size_t)(i * NX + j) * B, sizeof(double) * B);
        CUDA_TRY(h, cudaMemcpy(h->d_P, pk.data(), sizeof(double) * NPK * B, cudaMemcpyHostToDevice));
    }
    return FBUS_OK;
}

int fbus_clear_status(fbus_handle* h) {
    if (!h) return FBUS_E_BADARG;
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaMemsetAsync(h->d_status, 0, sizeof(int32_t) * h->B, h->stream));
    return FBUS_OK;
}

int fbus_stats_combine(const double* parts, size_t n_parts, double* out) {
    if (!parts || !out || n_parts == 0) {
        g_last_error = "fbus_stats_combine: bad argument";
        return FBUS_E_BADARG;
    }
    for (int i = 0; i < FBUS_NSTATS; ++i) out[i] = 0.0;
    for (size_t p = 0; p < n_parts; ++p) {
        const double* v = parts + p * FBUS_NSTATS;
        for (int i = 0; i < 5; ++i) out[i] += v[i];
        out[5] = (p == 0 || v[5] > out[5]) ? v[5] : out[5];
    }
    return FBUS_OK;
}

int fbus_stats(fbus_handle* h, const double* truth_p, const double* truth_q, int32_t mem, double* out_host, double* out_dev) {
    if (!h || !truth_p || !truth_q) return fail(h, FBUS_E_BADARG, "fbus_stats: bad argument");
    bool host;
    int rc = check_mem(h, mem, "fbus_stats", &host);
    if (rc) return rc;
    CUDA_TRY(h, cudaSetDevice(h->device));
    const size_t B = h->B;
    const double* tp;
    const double* tq;
    if ((rc = stage(h, h->scratch_in, truth_p, 3 * B, host, &tp))) return rc;
    if ((rc = stage(h, h->scratch_out, truth_q, 4 * B, host, &tq))) return rc;
    const int grid = (int)((B + STATS_BS - 1) / STATS_BS);
    CUDA_TRY(h, h->stats_partial.reserve((size_t)grid * 8 * sizeof(double)));
    CUDA_TRY(h, h->stats_out.reserve(FBUS_NSTATS * sizeof(double)));
    stats_kernel<<<grid, STATS_BS, 0, h->stream>>>(h->d_nom, h->d_P, B, tp, tq, (double*)h->stats_partial.p);
    CUDA_TRY(h, cudaGetLastError());
    double* dout = out_dev ? out_dev : (double*)h->stats_out.p;
    stats_reduce_kernel<<<1, 256, 0, h->stream>>>((const double*)h->stats_partial.p, grid, dout);
    CUDA_TRY(h, cudaGetLastError());
    if (out_host) {
        CUDA_TRY(h, cudaMemcpyAsync(out_host, dout, FBUS_NSTATS * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    }
    return FBUS_OK;
}

int fbus_set_noise(fbus_handle* h, const double* noise, int32_t mem) {
    if (!h) return fail(h, FBUS_E_BADARG, "fbus_set_noise: bad argument");
    bool host;
    int rc = check_mem(h, mem, "fbus_set_noise", &host);
    if (rc) return rc;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (!noise) {  // back to the config's values and the default kernels; the buffer is kept for a later call
        h->noise_on = false;
        return FBUS_OK;
    }
    if (!h->noise_smem_set) {  // the NOISE instantiations are prepared when first needed: creation only touches the default ones
        CUDA_TRY(h, set_window_smem_limits<true>());
        h->noise_smem_set = true;
    }
    const size_t bytes = (size_t)FBUS_NOISE_FIELDS * h->B * sizeof(double);
    CUDA_TRY(h, h->noise.reserve(bytes));  // allocated on the first call (the size is fixed by the batch)
    // stream-ordered: kernels enqueued before this call still read the previous values
    CUDA_TRY(h, cudaMemcpyAsync(h->noise.p, noise, bytes, host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, h->stream));
    h->noise_on = true;
    return FBUS_OK;
}

int fbus_set_gate(fbus_handle* h, const double* gate, int32_t mem) {
    if (!h) return fail(h, FBUS_E_BADARG, "fbus_set_gate: bad argument");
    bool host;
    int rc = check_mem(h, mem, "fbus_set_gate", &host);
    if (rc) return rc;
    if (h->k.flags & FBUS_FLAG_MATLAB) return fail(h, FBUS_E_BADARG, "fbus_set_gate: not available with FBUS_FLAG_MATLAB");
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (!gate) {  // back to the default kernels; thresholds and counts are kept
        h->gate_on = false;
        return FBUS_OK;
    }
    if (!h->gate_smem_set) {  // the GATE instantiations are prepared when first needed: creation only touches the default ones
        CUDA_TRY(h, set_gate_smem_limits());
        h->gate_smem_set = true;
    }
    const size_t B = h->B;
    CUDA_TRY(h, h->gate.reserve(B * sizeof(double)));  // allocated on the first call (the size is fixed by the batch)
    CUDA_TRY(h, h->gate_rej.reserve(B * sizeof(int32_t)));
    // stream-ordered: kernels enqueued before this call still read the previous thresholds and add to the previous counts
    CUDA_TRY(h, cudaMemcpyAsync(h->gate.p, gate, B * sizeof(double), host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(h->gate_rej.p, 0, B * sizeof(int32_t), h->stream));
    h->gate_on = true;
    h->gate_set = true;
    return FBUS_OK;
}

int fbus_rejected_updates(fbus_handle* h, int32_t* out, int32_t out_mem) {
    if (!h || !out) return fail(h, FBUS_E_BADARG, "fbus_rejected_updates: bad argument");
    bool out_host;
    int rc = check_mem(h, out_mem, "fbus_rejected_updates", &out_host);
    if (rc) return rc;
    if (!h->gate_set) return fail(h, FBUS_E_STATE, "fbus_rejected_updates: no gate was set on this handle");
    CUDA_TRY(h, cudaSetDevice(h->device));
    Outputs o{h, out_host};
    int32_t* dst = o.to(out, h->gate_rej.p, h->B);  // host: finish() copies the counts themselves back
    if (dst != h->gate_rej.p)
        CUDA_TRY(h, cudaMemcpyAsync(dst, h->gate_rej.p, h->B * sizeof(int32_t), cudaMemcpyDeviceToDevice, h->stream));
    return o.finish();
}

int fbus_filter_errors(fbus_handle* h, const double* truth_p, const double* truth_q, int32_t mem, double* out, int32_t out_mem) {
    static const char* const call = "fbus_filter_errors";
    if (!h || !truth_p || !truth_q || !out) return fail(h, FBUS_E_BADARG, "fbus_filter_errors: bad argument");
    bool host, out_host;
    int rc = check_mem(h, mem, call, &host);
    if (rc == FBUS_OK) rc = check_mem(h, out_mem, call, &out_host);
    if (rc) return rc;
    CUDA_TRY(h, cudaSetDevice(h->device));
    const size_t B = h->B;
    const double* tp;
    const double* tq;
    if ((rc = stage(h, h->scratch_in, truth_p, 3 * B, host, &tp))) return rc;
    if ((rc = stage(h, h->scratch_out, truth_q, 4 * B, host, &tq))) return rc;
    Outputs o{h, out_host};
    if ((rc = o.reserve(h->errors, 4 * B * sizeof(double)))) return rc;
    double* dout = o.to(out, h->errors.p, 4 * B);
    filter_errors_kernel<<<(unsigned)((B + STATS_BS - 1) / STATS_BS), STATS_BS, 0, h->stream>>>(h->d_nom, h->d_P, B, tp, tq, dout);
    CUDA_TRY(h, cudaGetLastError());
    return o.finish();
}

// ---- NCCL, loaded at run time: the library itself has no link-time dependency on it ------------------------------------
namespace {
// the few NCCL declarations used (nccl.h: ncclResult_t ncclSuccess = 0; ncclDataType_t ncclFloat64 = 8; ncclRedOp_t ncclSum = 0,
// ncclMax = 2); kept local so that the library builds on machines without the NCCL headers
typedef void* nccl_comm_t;
struct NcclApi {
    void* lib = nullptr;
    int (*CommInitAll)(nccl_comm_t*, int, const int*) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    std::string why;
};
constexpr int kNcclFloat64 = 8, kNcclSum = 0, kNcclMax = 2;

NcclApi& nccl_api() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* names[] = {getenv("FBUS_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char* nm : names) {
            if (!nm || !*nm) continue;
            api.lib = dlopen(nm, RTLD_NOW | RTLD_LOCAL);
            if (api.lib) break;
            api.why = dlerror();
        }
        if (!api.lib) return;
        api.CommInitAll = (int (*)(nccl_comm_t*, int, const int*))dlsym(api.lib, "ncclCommInitAll");
        api.AllReduce = (int (*)(const void*, void*, size_t, int, int, nccl_comm_t, cudaStream_t))dlsym(api.lib, "ncclAllReduce");
        api.GroupStart = (int (*)())dlsym(api.lib, "ncclGroupStart");
        api.GroupEnd = (int (*)())dlsym(api.lib, "ncclGroupEnd");
        api.GetErrorString = (const char* (*)(int))dlsym(api.lib, "ncclGetErrorString");
        if (!api.CommInitAll || !api.AllReduce || !api.GroupStart || !api.GroupEnd) {
            api.why = "libnccl lacks ncclCommInitAll / ncclAllReduce / ncclGroupStart / ncclGroupEnd";
            api.lib = nullptr;
        }
    });
    return api;
}
int nccl_fail(fbus_handle* h, const char* what, int rc) {
    NcclApi& a = nccl_api();
    return fail(h, FBUS_E_NCCL, std::string(what) + ": " + ((a.lib && a.GetErrorString) ? a.GetErrorString(rc) : "NCCL error"));
}
// sum of entries 0..4, maximum of entry 5, entries 6..7 zero: two all-reduces on the handle's stream (inside the caller's group)
int enqueue_stats_allreduce(fbus_handle* h, nccl_comm_t comm, double* v) {
    NcclApi& a = nccl_api();
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaMemsetAsync(v + 6, 0, 2 * sizeof(double), h->stream));
    int rc = a.AllReduce(v, v, 5, kNcclFloat64, kNcclSum, comm, h->stream);
    if (rc) return nccl_fail(h, "ncclAllReduce(sum)", rc);
    rc = a.AllReduce(v + 5, v + 5, 1, kNcclFloat64, kNcclMax, comm, h->stream);
    if (rc) return nccl_fail(h, "ncclAllReduce(max)", rc);
    return FBUS_OK;
}
std::mutex g_comm_mu;
std::map<std::vector<int>, std::vector<nccl_comm_t>> g_comms;  // one clique per device list, kept for the life of the process
}  // namespace

int fbus_stats_allreduce(fbus_handle* const* handles, int n, double* const* dev_vecs, double* out_host) {
    if (!handles || !dev_vecs || n <= 0) return fail(nullptr, FBUS_E_BADARG, "fbus_stats_allreduce: bad argument");
    for (int i = 0; i < n; ++i)
        if (!handles[i] || !dev_vecs[i]) return fail(nullptr, FBUS_E_BADARG, "fbus_stats_allreduce: null handle or vector");
    fbus_handle* h0 = handles[0];
    if (n > 1) {
        std::vector<int> devs(n);
        for (int i = 0; i < n; ++i) {
            devs[i] = handles[i]->device;
            for (int j = 0; j < i; ++j)
                if (devs[j] == devs[i]) return fail(h0, FBUS_E_BADARG, "fbus_stats_allreduce: two handles on the same device (combine those with fbus_stats_combine)");
        }
        NcclApi& a = nccl_api();
        if (!a.lib) return fail(h0, FBUS_E_NCCL, "fbus_stats_allreduce: NCCL not available (" + a.why + "); set FBUS_NCCL_LIB");
        std::vector<nccl_comm_t> comms;
        {
            std::lock_guard<std::mutex> lk(g_comm_mu);
            auto it = g_comms.find(devs);
            if (it == g_comms.end()) {
                std::vector<nccl_comm_t> c(n, nullptr);
                const int rc = a.CommInitAll(c.data(), n, devs.data());
                if (rc) return nccl_fail(h0, "ncclCommInitAll", rc);
                it = g_comms.emplace(devs, c).first;
            }
            comms = it->second;
        }
        int rc = a.GroupStart();
        if (rc) return nccl_fail(h0, "ncclGroupStart", rc);
        int frc = FBUS_OK;
        for (int i = 0; i < n && frc == FBUS_OK; ++i) frc = enqueue_stats_allreduce(handles[i], comms[i], dev_vecs[i]);
        rc = a.GroupEnd();
        if (frc != FBUS_OK) return frc;
        if (rc) return nccl_fail(h0, "ncclGroupEnd", rc);
    } else {
        CUDA_TRY(h0, cudaSetDevice(h0->device));
        CUDA_TRY(h0, cudaMemsetAsync(dev_vecs[0] + 6, 0, 2 * sizeof(double), h0->stream));
    }
    for (int i = 0; i < n; ++i) {  // every vector is final when the call returns
        CUDA_TRY(handles[i], cudaSetDevice(handles[i]->device));
        if (i == 0 && out_host)
            CUDA_TRY(h0, cudaMemcpyAsync(out_host, dev_vecs[0], FBUS_NSTATS * sizeof(double), cudaMemcpyDeviceToHost, h0->stream));
        CUDA_TRY(handles[i], cudaStreamSynchronize(handles[i]->stream));
    }
    return FBUS_OK;
}

int fbus_stats_allreduce_comm(fbus_handle* h, void* nccl_comm, double* dev_vec, double* out_host) {
    if (!h || !nccl_comm || !dev_vec) return fail(h, FBUS_E_BADARG, "fbus_stats_allreduce_comm: bad argument");
    NcclApi& a = nccl_api();
    if (!a.lib) return fail(h, FBUS_E_NCCL, "fbus_stats_allreduce_comm: NCCL not available (" + a.why + "); set FBUS_NCCL_LIB");
    int rc = a.GroupStart();
    if (rc) return nccl_fail(h, "ncclGroupStart", rc);
    const int frc = enqueue_stats_allreduce(h, (nccl_comm_t)nccl_comm, dev_vec);
    rc = a.GroupEnd();
    if (frc != FBUS_OK) return frc;
    if (rc) return nccl_fail(h, "ncclGroupEnd", rc);
    if (out_host) {
        CUDA_TRY(h, cudaMemcpyAsync(out_host, dev_vec, FBUS_NSTATS * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    }
    return FBUS_OK;
}

int fbus_synth_streams(fbus_handle* h, const fbus_synth_spec* spec, double* imu_data, int32_t* det_id, double* det_pose, double* bias_out) {
    if (!h || !spec || !imu_data || !det_id || !det_pose || !spec->base_imu || !spec->base_pose)
        return fail(h, FBUS_E_BADARG, "fbus_synth_streams: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->device));
    SynthParams sp;
    memset(&sp, 0, sizeof sp);
    const double* bi;
    const double* bp;
    int rc = stage(h, h->scratch_in, spec->base_imu, spec->n_samples * 6, true, &bi);
    if (rc) return rc;
    rc = stage(h, h->scratch_out, spec->base_pose, spec->n_frames * 7, true, &bp);
    if (rc) return rc;
    sp.B = h->B; sp.N = spec->n_samples; sp.W = spec->n_frames;
    sp.base_imu = bi; sp.base_pose = bp;
    sp.imu = imu_data; sp.det_id = det_id; sp.det_pose = det_pose; sp.bias_out = bias_out;
    sp.s_acc = spec->sigma_acc; sp.s_gyro = spec->sigma_gyro; sp.s_ba = spec->sigma_ba; sp.s_bg = spec->sigma_bg;
    sp.s_pos = spec->sigma_pos; sp.s_quat = spec->sigma_quat;
    sp.seed = spec->seed; sp.filter_offset = spec->filter_offset; sp.marker_id = spec->marker_id;
    const unsigned grid = (unsigned)((h->B + 127) / 128);
    synth_kernel<<<grid, 128, 0, h->stream>>>(sp);
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));  // base arrays staged from caller memory: make reuse safe
    return FBUS_OK;
}

int fbus_marker_project(fbus_handle* h, const double* pose, size_t n, int32_t underwater, double* corners, int32_t* valid, int32_t mem) {
    if (!h || !pose || !corners || (underwater != 0 && underwater != 1)) return fail(h, FBUS_E_BADARG, "fbus_marker_project: bad argument");
    bool host;
    int rc = check_mem(h, mem, "fbus_marker_project", &host);
    if (rc) return rc;
    if (n == 0) return FBUS_OK;
    CUDA_TRY(h, cudaSetDevice(h->device));
    const double* dp;
    if ((rc = stage(h, h->scratch_in, pose, 7 * n, host, &dp))) return rc;
    Outputs o{h, host};
    if ((rc = o.reserve(h->scratch_out, 16 * n * sizeof(double)))) return rc;
    if ((rc = o.reserve(h->scratch_aux, n * sizeof(int32_t)))) return rc;
    double* dc = o.to(corners, h->scratch_out.p, 16 * n);
    int32_t* dv = valid ? o.to(valid, h->scratch_aux.p, n) : nullptr;
    marker_project_kernel<<<(unsigned)((n + 127) / 128), 128, 0, h->stream>>>(h->k, h->gn, dp, n, n, 1, underwater, dc, dv);
    CUDA_TRY(h, cudaGetLastError());
    return o.finish();
}

int fbus_synth_corners(fbus_handle* h, const fbus_corner_spec* spec, size_t w0, size_t w1, float* corners, int32_t* ids) {
    if (!h || !spec || !corners || !ids || !spec->base_pose || !spec->base_id) return fail(h, FBUS_E_BADARG, "fbus_synth_corners: bad argument");
    const size_t m = spec->max_markers, W = spec->n_frames;
    if (w0 > w1 || w1 > W || m == 0) return fail(h, FBUS_E_BADARG, "fbus_synth_corners: need w0 <= w1 <= n_frames and max_markers > 0");
    // Philox counters: the global frame index is one 32-bit word, the slot's streams must stay below 2^32
    if (W > 0xFFFFFFFFull || m > (0xFFFFFFFFull - CORNER_STREAM0) / CORNER_STREAM_STRIDE)
        return fail(h, FBUS_E_BADARG, "fbus_synth_corners: n_frames or max_markers too large");
    if (spec->underwater != 0 && spec->underwater != 1) return fail(h, FBUS_E_BADARG, "fbus_synth_corners: underwater must be 0 or 1");
    if (!(spec->sigma_corner >= 0.0) || !(spec->sigma_outlier >= 0.0)) return fail(h, FBUS_E_BADARG, "fbus_synth_corners: negative sigma");
    if (!(spec->p_drop >= 0.0 && spec->p_drop <= 1.0) || !(spec->p_outlier >= 0.0 && spec->p_outlier <= 1.0))
        return fail(h, FBUS_E_BADARG, "fbus_synth_corners: probability outside [0, 1]");
    const size_t nws = (w1 - w0) * m, n = nws * h->B;
    if (n == 0) return FBUS_OK;
    CUDA_TRY(h, cudaSetDevice(h->device));
    // the noise-free corners of each (frame, slot) of the range, projected once for all filters
    CUDA_TRY(h, h->scratch_in.reserve(nws * 7 * sizeof(double)));
    CUDA_TRY(h, h->scratch_out.reserve(nws * 16 * sizeof(double)));
    CUDA_TRY(h, h->scratch_aux.reserve(nws * 2 * sizeof(int32_t)));
    double* dpose = (double*)h->scratch_in.p;
    double* dbase = (double*)h->scratch_out.p;
    int32_t* did = (int32_t*)h->scratch_aux.p;
    int32_t* dvalid = did + nws;
    CUDA_TRY(h, cudaMemcpyAsync(dpose, spec->base_pose + w0 * m * 7, nws * 7 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(did, spec->base_id + w0 * m, nws * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    marker_project_kernel<<<(unsigned)((nws + 127) / 128), 128, 0, h->stream>>>(h->k, h->gn, dpose, nws, 1, 7, spec->underwater, dbase, dvalid);
    CUDA_TRY(h, cudaGetLastError());
    CornerSynthParams sp;
    memset(&sp, 0, sizeof sp);
    sp.B = h->B; sp.m = m; sp.n = n; sp.w0 = w0;
    sp.base = dbase; sp.base_id = did; sp.base_valid = dvalid;
    sp.corners = corners; sp.ids = ids;
    sp.s_corner = spec->sigma_corner; sp.p_drop = spec->p_drop; sp.p_out = spec->p_outlier; sp.s_out = spec->sigma_outlier;
    sp.seed = spec->seed; sp.filter_offset = spec->filter_offset;
    synth_corners_kernel<<<(unsigned)((n + 127) / 128), 128, 0, h->stream>>>(sp);
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));  // base arrays staged from caller memory: make reuse safe
    return FBUS_OK;
}

int fbus_measure_fp64_peak(fbus_handle* h, double* flops) {
    if (!h || !flops) return fail(h, FBUS_E_BADARG, "fbus_measure_fp64_peak: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->device));
    cudaDeviceProp prop;
    CUDA_TRY(h, cudaGetDeviceProperties(&prop, h->device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    CUDA_TRY(h, h->scratch_aux.reserve((size_t)blocks * threads * sizeof(double)));
    cudaEvent_t e0, e1;
    CUDA_TRY(h, cudaEventCreate(&e0));
    CUDA_TRY(h, cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 6; ++rep) {
        CUDA_TRY(h, cudaEventRecord(e0, h->stream));
        fp64_peak_kernel<<<blocks, threads, 0, h->stream>>>((double*)h->scratch_aux.p, iters, 1.0 + rep);
        CUDA_TRY(h, cudaEventRecord(e1, h->stream));
        CUDA_TRY(h, cudaEventSynchronize(e1));
        float ms = 0.f;
        CUDA_TRY(h, cudaEventElapsedTime(&ms, e0, e1));
        const double fl = 2.0 * 64.0 * (double)iters * (double)blocks * threads / (ms * 1e-3);
        if (rep > 0 && fl > best) best = fl;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    CUDA_TRY(h, cudaGetLastError());
    *flops = best;
    return FBUS_OK;
}

}  // extern "C"
