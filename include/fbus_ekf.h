/*
 * fbus_ekf.h -- C ABI of the B200-native batched FBUS-EKF hot path.
 *
 * This header is the drop-in boundary (SURVEY.md section 8b).  The reference has no FFI; the seam
 * it replaces is the public surface of FBUSEKF::FILTER (C++/include/filter.hpp:143-178) and, with
 * identical meaning, the MATLAB pure-function API (matlab/InitGravityAndGyrobias.m,
 * InitPositionAndQuaternion.m, ImuUpdate.m, MeasureUpdate.m, ResetState.m,
 * ComputeVisionOnlyResults.m) plus the two vision functions VISION::RefractionTriangulation /
 * VISION::ComputeMarkerPose (C++/src/vision.cpp:472-759).  Every entry point below names the
 * reference function (file:line) it stands in for.
 *
 * Conventions
 *   - plain C types only; no torch / STL / Eigen types cross this boundary;
 *   - every batched array is structure-of-arrays with the FILTER INDEX FASTEST:  x[field][B];
 *   - quaternions are scalar-first Hamilton (w,x,y,z) as in every log of the reference;
 *   - matrices crossing the boundary are row-major;
 *   - all arithmetic is IEEE FP64 (the reference uses Eigen doubles); corners are float32 because
 *     the reference holds them as cv::Point2f (vision.cpp:492-494);
 *   - every call returns 0 on success or a negative FBUS_E_* code; fbus_last_error() gives text;
 *   - a handle is bound to one CUDA device and one stream and is not internally locked;
 *   - work is asynchronous: caller-owned buffers (host or device) must stay valid and unchanged until
 *     fbus_synchronize() / a synchronising call (fbus_get_state, fbus_stats with a host output);
 *     pinned host memory is read by DMA after the call returns, and large host-resident streams are
 *     copied in frame chunks on a second stream so that the PCIe copy overlaps the kernels;
 *   - there is NO CPU fallback: if no CUDA device is usable fbus_create fails with FBUS_E_CUDA.
 */
#ifndef FBUS_EKF_H
#define FBUS_EKF_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FBUS_ABI_VERSION 3 /* 2: fbus_config.imu_g / gn_tol, fbus_imu_stream.format, fbus_iir_prefilter; 3: fbus_stats_allreduce*, FBUS_E_NCCL;
                              added within 3 (no struct changed): fbus_set_noise, fbus_filter_errors, fbus_marker_project,
                              fbus_synth_corners with the new fbus_corner_spec, fbus_set_gate, fbus_rejected_updates,
                              FBUS_ST_UPDATE_REJECTED */

/* error codes */
#define FBUS_OK 0
#define FBUS_E_BADARG (-1)
#define FBUS_E_CUDA (-2)
#define FBUS_E_NOMEM (-3)
#define FBUS_E_STATE (-4)
#define FBUS_E_NCCL (-5) /* NCCL missing (libnccl.so.2 could not be loaded) or an NCCL call failed */

/* where a caller-owned data pointer lives (the mem / out_mem / trace_mem arguments and the mem fields of fbus_imu_stream and
   fbus_det_frames); a call given any other value returns FBUS_E_BADARG without any effect */
#define FBUS_MEM_HOST 0
#define FBUS_MEM_DEVICE 1

/* element format of fbus_imu_stream.data */
#define FBUS_IMU_F64_SI 0     /* double, accel in m/s^2 and gyro in rad/s: the fields of IMUData (common.hpp:176-193) */
#define FBUS_IMU_F32_SENSOR 1 /* float, accel in g and gyro in deg/s: the fields of the IMSEE SDK's ImuData
                                 (driver/IMSEE-SDK/include/types.h:122-127) as the IMU callback receives them.  The
                                 kernels convert every sample exactly as main.cpp:254 does before building IMUData --
                                 accel = (double)a * imu_g, gyro = (double)(w / 180.f) * M_PI with the reference's
                                 M_PI = 3.1415926 (common.hpp:14) -- so the filter sees bit-identical doubles while a
                                 host-resident stream needs half the bytes on the way to the device */

/* dimensions of the reference filter (filter.hpp:82-125): 18 error states, 12 noise terms, 7 rows */
#define FBUS_NX 18
#define FBUS_NW 12
#define FBUS_NZ 7
#define FBUS_NP_PACKED 171 /* upper triangle of the 18x18 covariance */
#define FBUS_MAX_MARKERS 16 /* marker map capacity (markersetup.yml has 12) */

/* per-filter status bits (written by the kernels instead of the reference's LOG(WARNING)+return) */
#define FBUS_ST_INIT_FAILED 0x1      /* InitializePose returned false (filter.cpp:308-358) */
#define FBUS_ST_RESET_SKIPPED 0x2    /* ResetSystemState early return (filter.cpp:432-447) */
#define FBUS_ST_RESET_DONE 0x4       /* gap > reset_gap: state overwritten (filter.cpp:462-474) */
#define FBUS_ST_UPDATE_SKIPPED 0x8   /* marker not in server: no update (filter.cpp:671-673) */
#define FBUS_ST_NONFINITE 0x10       /* a state entry became NaN/Inf */
#define FBUS_ST_NO_DETECTION 0x20    /* empty detection list for this filter/frame */
#define FBUS_ST_MARKER_REJECTED 0x40 /* refractive solve: a corner beyond makrer_dect_dist_thres */
#define FBUS_ST_UPDATE_REJECTED 0x80 /* an update was rejected by the innovation gate (fbus_set_gate) */

/* flags in fbus_config.flags */
#define FBUS_FLAG_JOSEPH 0x1 /* opt-in Joseph-form covariance update (north_star); default is the
                                reference's (I-KH)P form, filter.cpp:735 */
#define FBUS_FLAG_MATLAB 0x2 /* MATLAB-semantics mode: the numerics of the matlab/ .m files where they differ from filter.cpp (SURVEY A.4):
                                  ImuUpdate.m       always the axis-angle quaternion increment; rotation matrices of the
                                                    UN-normalised products (quaternion_to_rotmat.m form); R0 of the Runge-Kutta
                                                    step = the carried State.rotateMat; Fx(7:9,7:9) = expm(-[w]x dt);
                                  MeasureUpdate.m   position-only residual (quaternion rows zeroed, :88); nearest marker, no
                                                    hysteresis, no range gate;
                                  rotmat_to_quaternion.m  unit eigen-quaternions for Q_IL and the marker map;
                                  FBUS_EKF.m        dt between consecutive IMU samples; a gap > reset_gap between two IMAGE
                                                    times resets (ResetState.m: p, q, rotateMat from vision, v = b_a = 0, b_g kept)
                                                    and SKIPS propagation and update for that frame (:168-171); the frame that
                                                    initialises the pose also gets a measurement update (:116-151).
                                fbus_config_matlab() also sets the script's P0 and measurement noise.  Runs on the
                                lanes-per-filter window kernel at any batch size; not combinable with FBUS_FLAG_JOSEPH.
                                Checked against oracle/fbus_oracle_matlab.py (a NumPy restatement of the .m files; "parity
                                unpinned": no MATLAB here). */
#define FBUS_FLAG_ALL_MARKERS 0x4 /* opt-in: every detected marker of a frame updates the filter, not only the nearest one.
    1. Every frame that gets a measurement update in the reference's path (the fused path of fbus_step_windows after reset
       and propagation; fbus_update) gets a SEQUENCE of 7-row updates.  The first uses exactly the marker the reference
       chooses (nearest, with the marker_switch_thres hysteresis against prev_marker_id; prev_marker_id is updated as
       always); if that marker is known, this step is bit-for-bit the default update.
    2. Every other slot of the frame follows in slot order if its id is >= 0 and in the marker map: a separate 7-row update
       with the reference's measurement model and quaternion sign choice, linearised at the state the previous update left
       (sequential updates with injection in between).  Covariance form (I-KH)P, or the reduced Joseph form under
       FBUS_FLAG_JOSEPH; R is the config's or, under fbus_set_noise, the filter's own.
    3. A slot whose id is unknown is skipped and sets FBUS_ST_UPDATE_SKIPPED.  If the chosen marker is unknown, the other
       known markers are still applied and prev_marker_id stays unchanged, as in the reference.
    4. Init, reset and the vision-only pose still use the nearest marker only; trace rows, status bits and the continuation
       rule of fbus_step_windows are unchanged.
    5. With at most one known detection per frame the results equal the default mode's.
    6. Not combinable with FBUS_FLAG_MATLAB (fbus_create returns FBUS_E_BADARG); combines with FBUS_FLAG_JOSEPH,
       fbus_set_noise and both IMU element formats.
    7. The kernel keeps a frame's update slots as a 32-bit mask: with this flag the stepping calls reject
       max_markers > 32 with FBUS_E_BADARG (the default mode takes any max_markers).
    Runs on the first-generation lanes-per-filter window kernel at any batch size. */

/*
 * Per-run constants.  Mirrors EkfParam / RefractInfo / CameraInfo.T_SC / MarkerPoseServer
 * (C++/include/common.hpp:19-103) and the #defines of filter.hpp:25-34.
 */
typedef struct fbus_config {
    double tsc_left[16];  /* RAW left  T_SC, row-major 4x4 (camerainfo*.yml "TSC").  The filter path
                             premultiplies diag(-1,-1,1,1) itself (filter.hpp:67-70); the vision path
                             uses it raw (vision.hpp:83-84). */
    double tsc_right[16]; /* RAW right T_SC */
    /* EkfParam (paramconfig.yml:44-57) */
    double accel_n_cov, gyro_n_cov, accel_b_cov, gyro_b_cov;
    double pos_n_cov, quat_n_cov;
    double marker_max_dist;     /* fcpMarkerMaxDist */
    double marker_switch_thres; /* fcpMarkerSwitchThres */
    /* initial covariance per 3-block: p, v, theta, b_a, b_g, g (filter.hpp:29-34) */
    double p0_diag[6];
    double reset_gap; /* 0.1 s, filter.cpp:462 */
    /* RefractInfo (paramconfig.yml:30-42) */
    double n_air, n_glass, n_water;
    double d_air, d_glass;
    double normal[3];
    double marker_dect_dist_thres; /* makrer_dect_dist_thres, vision.cpp:602 */
    double marker_size;            /* marker side length, 0.28 m (vision.hpp:114); used only by the GN refinement */
    /* fisheye intrinsics of the left [0] and right [1] camera (camerainfo*.yml K and D): fx, fy, cx, cy and the four
       Kannala-Brandt coefficients; used only by fbus_undistort_fisheye */
    double cam_k[2][4];
    double cam_d[2][4];
    /* marker map (markersetup.yml / main.cpp:192-203); rotations are converted to quaternions with
       the Eigen Quaterniond(Matrix3d) rule exactly as main.cpp:201 does */
    int32_t n_markers;
    int32_t marker_id[FBUS_MAX_MARKERS];
    double marker_pos[FBUS_MAX_MARKERS * 3];
    double marker_rot[FBUS_MAX_MARKERS * 9];
    int32_t flags;
    int32_t reserved;
    double imu_g; /* IMUInfo.g (camerainfo*.yml "g": 9.802): scale of FBUS_IMU_F32_SENSOR accelerations, main.cpp:252-254 */
    double gn_tol; /* Gauss-Newton refinement (fbus_refract_solve_gn, gn_iters of fbus_solve_to_detections): 0 (default) runs
                      exactly the requested number of iterations; > 0 stops a marker as soon as an applied step is smaller than
                      this in every component (metres / radians).  The iteration contracts by ~1e-2 per step at the
                      logs' corner noise (~0.2 at ten times that noise), so the result agrees with the fixed count to well
                      below gn_tol */
} fbus_config;

/* Fill *cfg with the values the bundled logs were recorded with: C++/config/camerainfo1.yml,
   paramconfig.yml, markersetup.yml, filter.hpp:29-34. */
int fbus_config_default(fbus_config* cfg);
/* The same with the constants of matlab/FBUS_EKF.m:28-41,83-112 (P0, measurement noise) and FBUS_FLAG_MATLAB set. */
int fbus_config_matlab(fbus_config* cfg);

/*
 * IMU stream (IMUData, common.hpp:176-193).  Timestamps are shared by the batch (one time base,
 * B independent noise realisations); the six measurement fields are per filter.
 */
typedef struct fbus_imu_stream {
    size_t n_samples;   /* N */
    size_t batch;       /* B, must equal the handle's batch */
    const double* t;    /* [N]        HOST pointer, seconds */
    const double* data; /* [N][6][B]  accel xyz (m/s^2) then gyro xyz (rad/s); host or device.
                           With format = FBUS_IMU_F32_SENSOR the pointer is a `const float*` in disguise:
                           [N][6][B] floats, accel xyz (g) then gyro xyz (deg/s) */
    int32_t mem;        /* FBUS_MEM_HOST / FBUS_MEM_DEVICE for `data` */
    int32_t format;     /* FBUS_IMU_F64_SI (0) / FBUS_IMU_F32_SENSOR */
} fbus_imu_stream;

/*
 * Detection frames (DetectionResultList, filter.hpp:39-57): per frame up to max_markers marker
 * poses in the flipped left-camera frame, exactly the rows of data/image.txt (vision.cpp:104-106).
 */
typedef struct fbus_det_frames {
    size_t n_frames;    /* W */
    size_t max_markers; /* m slots per frame */
    size_t batch;       /* B */
    const double* t;    /* [W]            HOST pointer: frame timestamps */
    const int32_t* id;  /* [W][m][B]      marker id, < 0 = empty slot; host or device */
    const double* pose; /* [W][m][7][B]   p xyz, q wxyz; host or device */
    int32_t mem;
    int32_t reserved;
} fbus_det_frames;

/*
 * State view for get/set (NominalState + ErrorState.stateCovariance, common.hpp:205-247).
 * Any pointer may be NULL (field skipped).  All pointers are HOST memory.
 */
typedef struct fbus_state_soa {
    size_t batch;
    double* t;    /* [B]       nominal timeStamp */
    double* q;    /* [4][B]    quaternionI2G w,x,y,z */
    double* R;    /* [9][B]    rotmatI2G, CARRIED state (may be stale, SURVEY A.3-2) */
    double* p;    /* [3][B]    positionAtG */
    double* v;    /* [3][B]    velocityAtG */
    double* ba;   /* [3][B]    accelBias */
    double* bg;   /* [3][B]    gyroBias */
    double* g;    /* [3][B]    gravityAtG */
    double* pv;   /* [3][B]    positionOnlyVisual */
    double* qv;   /* [4][B]    quaternionOnlyVisual */
    double* P;    /* [324][B]  full 18x18 covariance, row-major */
    int32_t* prev_marker_id; /* [B] preUsedMarkerID_ */
    int32_t* initialised;    /* [B] isInitializePose_ */
    int32_t* status;         /* [B] OR of FBUS_ST_* since the last fbus_clear_status */
} fbus_state_soa;

typedef struct fbus_handle fbus_handle;

/* ---- lifetime ---------------------------------------------------------------------------- */

/* FILTER::FILTER (filter.hpp:63-137): allocates the state of `batch` filters on CUDA device
   `device`, sets P0, Q, R, Gamma, prev marker id 0, not initialised. */
int fbus_create(fbus_handle** out, const fbus_config* cfg, int device, size_t batch);
int fbus_destroy(fbus_handle* h);
const char* fbus_last_error(const fbus_handle* h); /* h may be NULL: last create/global error */
int fbus_abi_version(void);
int fbus_synchronize(fbus_handle* h);
size_t fbus_batch(const fbus_handle* h);
/* the CUDA stream all work of this handle is enqueued on (cudaStream_t as void*) */
void* fbus_stream(fbus_handle* h);

/* ---- F6: initialisation ------------------------------------------------------------------- */

/* FILTER::InitializeGravityAndBias (filter.cpp:256-285) == InitGravityAndGyrobias.m:
   b_g = mean(gyro), g = (0,0,-|mean(accel)|) over samples [first, first+count). */
int fbus_init_gravity_gyrobias(fbus_handle* h, const fbus_imu_stream* imu, size_t first, size_t count);

/* FILTER::InitializePose (filter.cpp:291-399) == InitPositionAndQuaternion.m, from frame `frame`.
   n_imu_before = number of buffered IMU samples not later than the frame (imuCnt, filter.cpp:299-312);
   0 makes the initialisation fail exactly as the reference does. */
int fbus_init_position_quaternion(fbus_handle* h, const fbus_det_frames* det, size_t frame, size_t n_imu_before);

/* ---- F1-F5: stepping ---------------------------------------------------------------------- */

/* FILTER::BatchImuProcessing (filter.cpp:483-531) == the ImuUpdate.m loop: for samples
   [first, first+count) in order: skip t < nominal.t, stop at t > t_end; dt = t - nominal.t;
   UpdateCovariance (filter.cpp:588-616) THEN UpdateNominalState (filter.cpp:533-582). */
int fbus_propagate(fbus_handle* h, const fbus_imu_stream* imu, size_t first, size_t count, double t_end);

/* FILTER::ResetSystemState (filter.cpp:405-477) == ResetState.m + ComputeVisionOnlyResults.m. */
int fbus_reset_state(fbus_handle* h, const fbus_det_frames* det, size_t frame);

/* FILTER::ObservationUpdate (filter.cpp:622-739) == MeasureUpdate.m (C++ numerics). */
int fbus_update(fbus_handle* h, const fbus_det_frames* det, size_t frame);

/*
 * Fused window kernel: the body of FILTER::FilterThreadFunction (filter.cpp:207-235) for frames
 * [w0, w1): per filter, if not initialised try InitializePose and go to the next frame; else
 * ResetSystemState, BatchImuProcessing over IMU samples [win_off[w], win_off[w+1]) with
 * t_end = det->t[w], ObservationUpdate.  State stays on chip for all the frames of one call.
 * win_off is a HOST array of n_frames+1 sample indices.
 * IMU buffer semantics (filter.cpp:390,493-520): a frame in which a filter does nothing (no detection for it, failed
 * initialisation) leaves that filter's IMU samples buffered for its next frame; within one call this is exact for any
 * memory kind (large host-resident streams are copied and processed in frame chunks, which is invisible in the results).
 * Across calls: a call starts with an empty buffer at win_off[w0], EXCEPT when it continues the previous call on this
 * handle -- device-resident streams, the same imu->data pointer and n_samples, w0 equal to the previous w1 -- in which case
 * the unconsumed samples carry over, exactly as if the two frame ranges had been one call.
 * trace (optional, HOST or DEVICE per trace_mem): [w1-w0][17][B] rows
 *   t p(3) q(wxyz) v(3) b_a(3) b_g(3)  -- the data/fusion.txt row (filter.cpp:241-246) after each frame.
 */
int fbus_step_windows(fbus_handle* h, const fbus_imu_stream* imu, const fbus_det_frames* det,
                      const uint32_t* win_off, size_t w0, size_t w1, double* trace, int32_t trace_mem);

/* ---- R1-R2: refractive flat-port marker-pose solve ---------------------------------------- */

/*
 * VISION::RefractionTriangulation (vision.cpp:472-618) followed by VISION::ComputeMarkerPose
 * (vision.cpp:624-759) for n independent markers.
 *   corners [16][n] float32: left (x,y) of corners 0..3 then right (x,y) of corners 0..3, the
 *                            column order of the water data/corners.txt (vision.cpp:111-119);
 *   pose    [7][n]  double : p xyz, q wxyz of corner 0 (positionAtCL, quaternionM2CL);
 *   corners3d [12][n] double or NULL: the four triangulated corners (cornerPositionAtCL);
 *   valid   [n] int32 or NULL: 1 = pose computed, 0 = rejected (a corner farther than the threshold).
 * mem applies to all four pointers.
 */
int fbus_refract_solve(fbus_handle* h, const float* corners, size_t n, double* pose, double* corners3d,
                       int32_t* valid, int32_t mem);

/*
 * Vision front-end -> filter hand-off (VisionThreadFunction between DetectArucoTag and SetDetectionResult,
 * vision.cpp:60-139) for a whole batch: corners [16][W*m*B] float32 (item index (frame*m + slot)*B + filter) and the
 * detected marker ids [W][m][B] (< 0 = empty slot) -> detection frames in the layout of fbus_det_frames:
 * det_id [W][m][B] (-1 where the marker was rejected by the range gate) and det_pose [W][m][7][B].
 * underwater: 1 = RefractionTriangulation, 0 = NormalTriangulation; gn_iters > 0 adds the Gauss-Newton refinement (R3).
 */
int fbus_solve_to_detections(fbus_handle* h, const float* corners, const int32_t* marker_ids, size_t n_frames, size_t max_markers,
                             int32_t underwater, int32_t gn_iters, int32_t* det_id, double* det_pose, int32_t mem);

/*
 * N4: cv::fisheye::undistortPoints(distorted, undistorted, K, D) as VISION::DetectArucoTag applies it to the detected
 * corner pixels (vision.cpp:203,253,318,369): Kannala-Brandt inverse by Newton iterations on theta.
 *   pixels [16][n] float32 (left xy x4, right xy x4; left rows use cam 0, right rows cam 1) -> normalised [16][n] float32,
 *   the input layout of fbus_refract_solve / fbus_inair_solve.
 */
int fbus_undistort_fisheye(fbus_handle* h, const float* pixels, size_t n, float* normalised, int32_t mem);

/* VISION::NormalTriangulation (vision.cpp:395-466: homogeneous DLT per stereo corner pair, land mode) followed by
   VISION::ComputeMarkerPose; same layouts and meaning as fbus_refract_solve. */
int fbus_inair_solve(fbus_handle* h, const float* corners, size_t n, double* pose, double* corners3d,
                     int32_t* valid, int32_t mem);

/*
 * R3 (north_star; NOT in the reference, "parity unpinned"): the closed-form solve above followed by `iters`
 * Gauss-Newton iterations on the stereo reprojection error through the flat port (16 residuals, 6 parameters,
 * analytic Jacobians; SURVEY.md A.6).  corner_dtype: 0 = float32 corners (as the reference holds them), 1 = float64.
 *   pose [7][n]: refined p xyz, q wxyz of corner 0;  cost [n] or NULL: final sum of squared residuals;
 *   valid [n] or NULL as fbus_refract_solve.  Checked against oracle/fbus_oracle_np.py and synthetic ground truth.
 */
int fbus_refract_solve_gn(fbus_handle* h, const void* corners, int32_t corner_dtype, size_t n, int32_t iters, double* pose,
                          double* cost, int32_t* valid, int32_t mem);

/* VISION::ComputeMarkerPose alone (vision.cpp:624-759) from 3-D corners [12][n] (the land
   data/corners.txt layout, vision.cpp:120-124). */
int fbus_marker_pose(fbus_handle* h, const double* corners3d, size_t n, double* pose, int32_t mem);

/* FILTER::SetImuData's 1-pole pre-filter (filter.cpp:36-48) over samples [first, first + count) of a stream, per filter and
   channel: out[0] = in[first] (the reference pushes the first sample of an empty buffer unfiltered), then
   out[i] = out[i-1] * (1 - 0.1) + in[first + i] * 0.1 -- two rounded products and one rounded sum, as the Eigen expression
   evaluates; nothing is contracted into an FMA.  `in` may be of either element format; `out` is [count][6][B] doubles in SI
   units (host or device; for a device-resident FBUS_IMU_F64_SI stream it may alias the input samples: in place).
   A caller restarts the recurrence wherever the live buffer was empty (after InitializeGravityAndBias: one call per
   stretch). */
int fbus_iir_prefilter(fbus_handle* h, const fbus_imu_stream* in, size_t first, size_t count, double* out, int32_t out_mem);

/* ---- per-filter noise values ------------------------------------------------------------- */

/* rows of a per-filter noise array, in fbus_config order */
#define FBUS_NOISE_FIELDS 6 /* accel_n_cov, gyro_n_cov, accel_b_cov, gyro_b_cov, pos_n_cov, quat_n_cov */
/* Gives every filter its own noise covariances: noise is [FBUS_NOISE_FIELDS][B] doubles (mem as given), row f holding the
   fbus_config field f of each filter.  The array is copied into a handle-owned device buffer (allocated on the first call,
   freed by fbus_destroy), and from the next stepping call on (fbus_step_windows, fbus_propagate, fbus_update,
   fbus_reset_state, the init calls) filter b uses column b in place of the config's six values, used as given like
   fbus_config's.  noise = NULL returns the handle to the config's values.  State, status and the continuation rule of
   fbus_step_windows are untouched: a call between two continued calls takes effect from the next call on. */
int fbus_set_noise(fbus_handle* h, const double* noise, int32_t mem);

/* ---- innovation gate (chi-square test of every measurement update) --------------------------- */

/* gate[B] doubles (mem as given) or NULL.  Copied into a handle-owned device buffer, like fbus_set_noise.
    1. Every 7-row measurement update -- the reference's update in the fused path of fbus_step_windows and in fbus_update, and
       each further update under FBUS_FLAG_ALL_MARKERS -- forms the normalised innovation squared NIS = r^T S^-1 r: r is the
       7-row residual after the quaternion sign choice, S = H P H^T + R at that update's own linearisation state, R the config's
       value or, under fbus_set_noise, the filter's own.
    2. With g = gate[b] the update of filter b is rejected iff g > 0 && !(NIS <= g): a non-finite NIS is rejected, and g <= 0 or
       NaN means no gate for that filter.
    3. A rejected update leaves the nominal state and the covariance bit-for-bit unchanged, sets FBUS_ST_UPDATE_REJECTED and adds
       1 to the filter's count (fbus_rejected_updates).
    4. Marker selection comes before the gate and is unchanged: prev_marker_id is updated as always.
    5. Not gated and unchanged: init, reset, the vision-only pose (pv, qv), trace rows, the other status bits and the
       continuation rule of fbus_step_windows.
    6. Under FBUS_FLAG_ALL_MARKERS each update of the sequence is gated on its own; a rejected chosen marker does not stop the
       further slots.
    7. Combines with FBUS_FLAG_JOSEPH, FBUS_FLAG_ALL_MARKERS, fbus_set_noise and both IMU element formats.  On a FBUS_FLAG_MATLAB
       handle the call returns FBUS_E_BADARG.  gate = NULL turns the gate off (the window kernels are the default ones again;
       the counts stay readable).  A call between two continued fbus_step_windows calls takes effect from the next call on.
    Thresholds: the quaternion rows carry about 3 degrees of freedom plus a second-order component along hQ, so the NIS of a
    consistent filter lies between chi-square with 6 and with 7 degrees of freedom:
                     0.95    0.99    0.999
        chi2(6)     12.59   16.81   22.46
        chi2(7)     14.07   18.48   24.32
    Runs on the first-generation lanes-per-filter window kernel at any batch size while a gate is set. */
int fbus_set_gate(fbus_handle* h, const double* gate, int32_t mem);
/* out[B] int32 (out_mem as given): updates rejected per filter since the last fbus_set_gate with a non-NULL array.
   Returns FBUS_E_STATE if the gate was never set on this handle; synchronises for a HOST output. */
int fbus_rejected_updates(fbus_handle* h, int32_t* out, int32_t out_mem);

/* ---- state access ------------------------------------------------------------------------- */

int fbus_get_state(fbus_handle* h, fbus_state_soa* out); /* synchronises */
int fbus_set_state(fbus_handle* h, const fbus_state_soa* in);
int fbus_clear_status(fbus_handle* h);

/* ---- statistics (new; the reference has no ground truth) ---------------------------------- */

#define FBUS_NSTATS 8
/* out[0]=sum |p-p_true|^2, [1]=sum |dtheta|^2, [2]=sum NEES over (p,theta) (6 dof),
   [3]=count of finite filters, [4]=count of non-finite filters, [5]=max |p-p_true|, [6..7] reserved.
   truth_p [3][B], truth_q [4][B] (mem as given).  out_dev (optional) is a DEVICE buffer of
   FBUS_NSTATS doubles that receives the same vector so the caller can hand it to an NCCL allreduce
   without a host round trip; out_host (optional) is HOST. */
int fbus_stats(fbus_handle* h, const double* truth_p, const double* truth_q, int32_t mem,
               double* out_host, double* out_dev);
/* Per-filter error terms, the ones fbus_stats sums: out is [4][B] (out_mem as given) with
   out[0][b] = |p - p_true|^2, out[1][b] = |dtheta|^2, out[2][b] = NEES over (p,theta) (6 dof), out[3][b] = 1.0 when the three
   are finite and the (p,theta) block of P is positive definite, else 0.0 (rows 0..2 then hold whatever was computed).
   fbus_stats entries 0..4 are the sums of rows 0..2 over filters with flag 1 and the counts of flags 1 and 0 (up to
   summation order); entry 5 is exactly the maximum of sqrt(row 0) over filters with flag 1.  truth_p [3][B], truth_q [4][B]
   (mem as given).  Synchronises when out is HOST. */
int fbus_filter_errors(fbus_handle* h, const double* truth_p, const double* truth_q, int32_t mem, double* out, int32_t out_mem);
/* Combine rule of the per-shard vectors (SURVEY 8e: what the multi-GPU driver applies with its all-reduce; here for callers
   that gather the vectors themselves -- several handles in one process, MPI): parts is [n_parts][FBUS_NSTATS] on the HOST;
   out[0..4] = sums over the parts, out[5] = maximum, out[6..7] = 0.  Pure host code, needs no handle. */
int fbus_stats_combine(const double* parts, size_t n_parts, double* out);

/*
 * The one collective of the multi-GPU path (SURVEY 8e; north_star: "only a final NCCL allreduce of RMSE/NEES statistics
 * over NVLink"): filters are independent, every device works on its own shard with no hot-path traffic, and at the end the
 * FBUS_NSTATS-double vectors of fbus_stats are combined with ncclAllReduce -- entries 0..4 with ncclSum, entry 5 with ncclMax,
 * entries 6..7 zeroed -- over NVLink / NVSwitch.  NCCL is loaded at run time (libnccl.so.2, or the path in FBUS_NCCL_LIB);
 * without it the calls return FBUS_E_NCCL, nothing else of the library needs it.
 *
 * One process, one handle per device (the C++ host of north_star): handles[0..n) live on n DIFFERENT devices; dev_vecs[i]
 * is the DEVICE vector on handles[i]'s device that fbus_stats(.., out_dev) wrote.  After the call every dev_vecs[i] holds the
 * combined vector, and out_host (optional, HOST, FBUS_NSTATS doubles) too.  The communicators are created on first use
 * (ncclCommInitAll) and cached per device list.  n = 1 needs no NCCL.
 */
int fbus_stats_allreduce(fbus_handle* const* handles, int n, double* const* dev_vecs, double* out_host);
/* One rank per process (torchrun, MPI): nccl_comm is an ncclComm_t the caller owns whose rank on this process uses the
   handle's device; dev_vec as above.  Enqueued on the handle's stream; synchronises when out_host is given. */
int fbus_stats_allreduce_comm(fbus_handle* h, void* nccl_comm, double* dev_vec, double* out_host);

/* ---- synthetic Monte-Carlo streams (benchmark workload generator, SURVEY 8d config 3/5) ---- */

typedef struct fbus_synth_spec {
    size_t n_samples; /* N IMU samples */
    size_t n_frames;  /* W detection frames */
    const double* base_imu;  /* [N][6] HOST: noise-free body accel + gyro of the shared trajectory */
    const double* base_pose; /* [W][7] HOST: noise-free marker pose (p, q) seen from the camera */
    int32_t marker_id;       /* id of the single marker */
    int32_t reserved;
    double sigma_acc, sigma_gyro;       /* white noise std */
    double sigma_ba, sigma_bg;          /* per-filter constant bias std */
    double sigma_pos, sigma_quat;       /* marker pose noise std */
    uint64_t seed;
    uint64_t filter_offset; /* global index of this handle's filter 0 (multi-GPU shards) */
} fbus_synth_spec;

/* Generates per-filter noisy streams ON THE DEVICE (Philox4x32-10 keyed by seed, counter = global
   filter index / sample / field) into caller-provided DEVICE buffers laid out as fbus_imu_stream.data
   [N][6][B], fbus_det_frames.id [W][1][B] and .pose [W][1][7][B].  bias_out (optional, DEVICE,
   [6][B]) receives the drawn b_a, b_g. */
int fbus_synth_streams(fbus_handle* h, const fbus_synth_spec* spec, double* imu_data, int32_t* det_id,
                       double* det_pose, double* bias_out);

/*
 * Forward model of the stereo front end (not in the reference; the exact inverse of fbus_refract_solve / fbus_inair_solve):
 *   pose    [7][n]  double: p xyz, q wxyz of corner 0 in the flipped left-camera frame (the layout the solves write); the
 *                           quaternion is normalised before use;
 *   corners [16][n] double: left (x,y) of corners 0..3, then right, normalised coordinates (the solves' input layout);
 *   valid   [n] int32 or NULL: 1, or 0 when one of the 8 corner points lies at or behind the port in its camera's frame
 *                           (Z <= d_air + d_glass underwater, Z <= 0 in air); that item's 16 outputs are then NaN.
 * Corners (0,0,0), (s,0,0), (s,s,0), (0,s,0) of the marker (s = marker_size) are un-flipped into the left camera frame.
 * underwater = 1: the right camera through the true inverse of R_RL and P_LR, and the flat-port projection air -> glass ->
 * water solved by Newton iterations to 4.5e-16 relative (the one the Gauss-Newton refinement uses, with its paraxial branch);
 * underwater = 0: the pinhole geometry of VISION::NormalTriangulation, x_R ~ [R_IR R_IL^T | P_LI - R P_RI] [X_L; 1].
 * mem applies to all three pointers.
 */
int fbus_marker_project(fbus_handle* h, const double* pose, size_t n, int32_t underwater, double* corners, int32_t* valid,
                        int32_t mem);

typedef struct fbus_corner_spec {
    size_t n_frames, max_markers;    /* W, m */
    const double* base_pose;         /* [W][m][7] HOST: noise-free marker pose per slot (flipped left-camera frame) */
    const int32_t* base_id;          /* [W][m]    HOST: marker id per slot, < 0 = empty */
    int32_t underwater, reserved;    /* 1: flat-port projection, 0: in air (fbus_marker_project) */
    double sigma_corner;             /* std of the white noise on every normalised coordinate */
    double p_drop;                   /* probability that a (frame, slot, filter) detection is missing */
    double p_outlier, sigma_outlier; /* probability of a gross error; its extra std on all 16 coordinates of the marker */
    uint64_t seed, filter_offset;    /* as fbus_synth_spec */
} fbus_corner_spec;

/*
 * Per-filter stereo corner streams of the marker map, generated ON THE DEVICE for frames [w0, w1) into caller-provided DEVICE
 * buffers laid out as the input of fbus_solve_to_detections: corners [16][(w1-w0)*m*B] float32 with item
 * ((w - w0)*m + slot)*B + b, and ids [(w1-w0)][m][B].
 *   1. The noise-free corners of a (frame, slot) are fbus_marker_project of its base pose, computed once for all filters.
 *   2. A slot with base id < 0, or whose projection is not valid, gets id -1 and zero corners in every filter.
 *   3. Otherwise a uniform draw u_drop < p_drop drops the detection (id -1, zero corners).  A second uniform draw
 *      u_out < p_outlier makes it an outlier: it keeps its id and every coordinate gets an extra sigma_outlier * z' from
 *      independent normals.
 *   4. Each coordinate is base + sigma_corner * z (+ sigma_outlier * z'), summed in double and rounded once to float32 (the
 *      reference holds corners as cv::Point2f).
 * Randomness: the Philox4x32-10 / Box-Muller generator of fbus_synth_streams, key = seed, counter = (global filter index
 * filter_offset + b as two words, GLOBAL frame index w, stream 64 + 32*slot + d): d = 0..7 the normals of coordinates 2d and
 * 2d+1, d = 8 the two uniforms (53 bits each, in [0,1)), d = 9..16 the outlier normals.  These streams are disjoint from those of
 * fbus_synth_streams, so one seed drives both calls independently; frame ranges split over several calls, and batches split
 * into shards with filter_offset, give bit-for-bit the output of one call.
 * FBUS_E_BADARG: NULL outputs or base arrays, w0 > w1, w1 > n_frames, max_markers == 0, a negative sigma, a probability outside
 * [0, 1], underwater not 0 or 1.  Synchronises (the base arrays are staged from host memory).
 */
int fbus_synth_corners(fbus_handle* h, const fbus_corner_spec* spec, size_t w0, size_t w1, float* corners, int32_t* ids);

/* ---- helpers with no device work (usable without a GPU) ----------------------------------- */

/* Eigen Quaterniond(Matrix3d) rule (main.cpp:201, filter.cpp:370): R row-major -> q wxyz, not normalised */
void fbus_quat_from_rotmat(const double R[9], double q[4]);

/* FP64 FMA peak microbenchmark: runs a DFMA-saturating kernel on the handle's device and returns
   the measured FLOP/s (FMA = 2) in *flops; used as the roofline denominator (SURVEY 8d). */
int fbus_measure_fp64_peak(fbus_handle* h, double* flops);

#ifdef __cplusplus
}
#endif
#endif /* FBUS_EKF_H */
