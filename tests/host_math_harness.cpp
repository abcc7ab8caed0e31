// tests/host_math_harness.cpp -- TEST-ONLY: compiles the device math header for the host so the
// structured kernels' arithmetic can be compared with the oracle on a machine without a GPU.
// Not part of the product; the product has no CPU path.
#include "../fbus_ekf_b200/csrc/fbus_host_consts.hpp"

using namespace fbus;

static void nom_from(const double* a, Nominal& n) {
    n.t = a[0];
    for (int i = 0; i < 4; ++i) n.q[i] = a[1 + i];
    for (int i = 0; i < 9; ++i) n.R[i] = a[5 + i];
    for (int i = 0; i < 3; ++i) { n.p[i] = a[14 + i]; n.v[i] = a[17 + i]; n.ba[i] = a[20 + i]; n.bg[i] = a[23 + i]; n.g[i] = a[26 + i]; }
}
static void nom_to(const Nominal& n, double* a) {
    a[0] = n.t;
    for (int i = 0; i < 4; ++i) a[1 + i] = n.q[i];
    for (int i = 0; i < 9; ++i) a[5 + i] = n.R[i];
    for (int i = 0; i < 3; ++i) { a[14 + i] = n.p[i]; a[17 + i] = n.v[i]; a[20 + i] = n.ba[i]; a[23 + i] = n.bg[i]; a[26 + i] = n.g[i]; }
}

extern "C" {
void hm_config_default(fbus_config* c) { config_default(c); }

int hm_propagate(const fbus_config* cfg, double* P171, double* nom, const double* accel, const double* gyro, double dt) {
    DevConsts k;
    MarkerTable tab;
    if (make_dev_consts(cfg, &k, &tab)) return -1;
    Nominal n;
    nom_from(nom, n);
    double w[3], a[3];
    for (int i = 0; i < 3; ++i) { w[i] = gyro[i] - n.bg[i]; a[i] = accel[i] - n.ba[i]; }
    Cov<1> P{P171};
    propagate_cov<1>(P, n.R, a, w, dt, k.Qd);
    propagate_nominal(n, dt, accel, gyro);
    n.t += dt;
    nom_to(n, nom);
    return 0;
}

int hm_update(const fbus_config* cfg, double* P171, double* nom, int marker_id, const double* yP, const double* yQ) {
    DevConsts k;
    MarkerTable tab;
    if (make_dev_consts(cfg, &k, &tab)) return -1;
    const int m = find_marker(k, &tab, marker_id);
    if (m < 0) return -2;
    Nominal n;
    nom_from(nom, n);
    Cov<1> P{P171};
    measurement_update<1>(P, n, k, tab.mk[m], yP, yQ);
    nom_to(n, nom);
    return 0;
}

// the Joseph-form instantiation (FBUS_FLAG_JOSEPH) whatever cfg->flags says
int hm_update_joseph(const fbus_config* cfg, double* P171, double* nom, int marker_id, const double* yP, const double* yQ) {
    DevConsts k;
    MarkerTable tab;
    if (make_dev_consts(cfg, &k, &tab)) return -1;
    const int m = find_marker(k, &tab, marker_id);
    if (m < 0) return -2;
    Nominal n;
    nom_from(nom, n);
    Cov<1> P{P171};
    measurement_update<1, 1>(P, n, k, tab.mk[m], yP, yQ);
    nom_to(n, nom);
    return 0;
}
}

extern "C" int hm_update_coop(const fbus_config* cfg, double* P171, double* nom, int marker_id, const double* yP, const double* yQ) {
    DevConsts k;
    MarkerTable tab;
    if (make_dev_consts(cfg, &k, &tab)) return -1;
    const int m = find_marker(k, &tab, marker_id);
    if (m < 0) return -2;
    Nominal n;
    nom_from(nom, n);
    Cov<1> P{P171};
    measurement_update_coop<1>(P, n, k, tab.mk[m], yP, yQ);
    nom_to(n, nom);
    return 0;
}

#include "../fbus_ekf_b200/csrc/fbus_refract.cuh"
extern "C" {
// corners16: Lxy x4, Rxy x4 (float32) -> corners3d[12], pose[7]; returns valid flag
int hm_refract(const fbus_config* cfg, const float* c16, double* c3d, double* pose) {
    DevConsts k;
    MarkerTable tab;
    if (make_dev_consts(cfg, &k, &tab)) return -1;
    int ok = 1;
    for (int i = 0; i < 4; ++i) {
        const double nrm = triangulate_corner(k, c16[2 * i], c16[2 * i + 1], c16[8 + 2 * i], c16[8 + 2 * i + 1], c3d + 3 * i);
        if (nrm > k.dect_thres) ok = 0;
    }
    marker_pose(c3d, k.rod_s, k.rod_c, pose, pose + 3);
    return ok;
}
int hm_marker_pose(const fbus_config* cfg, const double* c3d, double* pose) {
    DevConsts k;
    MarkerTable tab;
    if (make_dev_consts(cfg, &k, &tab)) return -1;
    marker_pose(c3d, k.rod_s, k.rod_c, pose, pose + 3);
    return 0;
}
}

extern "C" {
// R3: closed form + GN on one marker; c16 double; returns valid flag; pose[7], cost
int hm_refract_gn(const fbus_config* cfg, const double* c16, int iters, double* pose, double* cost) {
    DevConsts k;
    MarkerTable tab;
    if (make_dev_consts(cfg, &k, &tab)) return -1;
    GnConsts g;
    make_gn_consts(cfg, &k, &g);
    double C[12];
    int ok = 1;
    for (int i = 0; i < 4; ++i)
        if (triangulate_corner(k, c16[2 * i], c16[2 * i + 1], c16[8 + 2 * i], c16[8 + 2 * i + 1], C + 3 * i) > k.dect_thres) ok = 0;
    marker_pose(C, k.rod_s, k.rod_c, pose, pose + 3);
    double Rm[9];
    quat_to_rotmat_unit(pose + 3, Rm);
    *cost = gn_refine(g, c16, Rm, pose, iters);
    R2q(Rm, pose + 3);
    return ok;
}
// projection + Jacobian of one point (for finite-difference checks)
void hm_project_refr(const fbus_config* cfg, const double* X, double* uv, double* J) {
    DevConsts k;
    MarkerTable tab;
    make_dev_consts(cfg, &k, &tab);
    GnConsts g;
    make_gn_consts(cfg, &k, &g);
    project_refr(g, X, uv, J);
}
}

extern "C" int hm_inair(const fbus_config* cfg, const float* c16, double* c3d, double* pose) {
    DevConsts k;
    MarkerTable tab;
    if (make_dev_consts(cfg, &k, &tab)) return -1;
    int ok = 1;
    for (int i = 0; i < 4; ++i)
        if (triangulate_corner_inair(k, c16[2 * i], c16[2 * i + 1], c16[8 + 2 * i], c16[8 + 2 * i + 1], c3d + 3 * i) > k.dect_thres) ok = 0;
    marker_pose(c3d, k.rod_s, k.rod_c, pose, pose + 3);
    return ok;
}

// MATLAB-semantics mode pieces (FBUS_FLAG_MATLAB): the host build of the same inlines the kernels use
extern "C" {
void hm_rotmat_to_quat_eig(const double* R, double* q) { rotmat_to_quat_eig(R, q); }
void hm_expm_rot_minus_I(const double* w, double dt, double* W) { expm_rot_minus_I(w, dt, W); }
void hm_propagate_nominal_matlab(double* nom, const double* accel, const double* gyro, double dt) {
    Nominal n;
    nom_from(nom, n);
    propagate_nominal_matlab(n, dt, accel, gyro);
    nom_to(n, nom);
}
}
