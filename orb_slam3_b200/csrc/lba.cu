// Local bundle adjustment LM engine for B200 (sm_100a) behind include/orb_b200.h
// (lba_solve): the g2o loop that Optimizer::LocalBundleAdjustment runs
// (reference src/Optimizer.cc:1410-1411 -> Thirdparty/g2o optimization_algorithm_
// levenberg.cpp:61-169, block_solver.hpp:354-604), all in fp64.
//
// Data layout (HBM, SoA, fp64): poses K x 7 (quaternion xyzw + t), points L x 3,
// edges sorted by landmark (CSR lm_ptr) so one thread owns a landmark and its
// H_ll / b_l sums are deterministic; a second CSR (by free pose) and a pair list
// (pose i1 <= i2 -> the landmarks they share) are built once per solve on the
// host -- the analogue of g2o's buildStructure (block_solver.hpp:143-295).
//
// Kernels per LM trial:
//   lin_edge_kernel     residuals, Huber weights, Jacobians, W (6x3 per edge); lm_gather_kernel sums H_ll, b_l
//   pose_reduce_kernel  H_pp, b_p per free pose (fixed-order tree sum)
//   lm_prepare_kernel   (H_ll + lambda I)^-1, D^-1 b_l; y_edge_kernel Y = W D^-1
//   schur_pairs_kernel  S_{i1 i2} = [H_pp] - sum_l Y_{i1 l} W_{i2 l}^T : the dense contraction,
//                       on the tensor cores as fp64 DMMA (mma.sync.m8n8k4.f64), one CTA per pose pair
//   bschur_kernel       b_s = b_p - sum W D^-1 b_l          (stored as an extra row of S)
//   [ncclAllReduce of (S | b_s) when landmarks are sharded over GPUs]
//   ldlt_kernel         blocked right-looking LDL^T of S (+rhs row), all SMs, own grid barrier
//   backsub_kernel      L^T x_p = z
//   lm_update_kernel    x_l = D^-1 (b_l - W^T x_p), state backup, oplus (SE3 exp), scale terms
//   chi_kernel          robust chi2 of the trial state
// The LM control law (lambda, rho, accept/reject, stop rules) runs on the host
// between trials, reading three doubles back per trial; *stop is polled there.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <float.h>
#include <limits.h>
#include <stdlib.h>
#include <math.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <string>
#include <thread>
#include <vector>

#include "../../include/orb_b200.h"
#include "se3_dev.cuh"
#include "orb_engine.h"
#include "ldlt_plan.h"

namespace orbb200 {

#define CUDA_TRYL(expr)                                                                \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      set_last_error(std::string(#expr) + ": " + cudaGetErrorString(_e));              \
      return ORB_E_CUDA;                                                               \
    }                                                                                  \
  } while (0)

struct LbaDev {
  int n_kf, n_free, n_mp, n_edges, n;  // n = 6*n_free
  // graph (edges sorted by landmark)
  const int* lm_ptr; const int* e_kf; const int* e_free; const uint8_t* e_stereo;
  const double* e_obs; const float* e_is2; const float* kf_cam; const int* free_kf;
  const int* pose_ptr; const int* pose_edges;
  const int* pair_i1; const int* pair_i2; const int* pair_ptr; const int* pair_ea; const int* pair_eb;
  int n_pairs;
  // rig extension (all null unless the graph has a KannalaBrandt8 camera or second-camera edges)
  const uint8_t* kf_model;  // bit 0: mpCamera is KannalaBrandt8, bit 1: mpCamera2 is
  const float* kf_dist;     // n_kf x 4: k0..k3 of mpCamera
  const float* kf_cam2;     // n_kf x 8: fx fy cx cy k0..k3 of mpCamera2
  const double* kf_trl;     // n_kf x 7: SE3Quat(Trl)
  // state
  double* pose; double* pts; double* pose_bak; double* pts_bak;
  // system
  double *Hll, *bl, *W, *Y, *Hpp_e, *bp_e, *Hpp, *bp, *Dinv, *db, *S, *x, *chi_lm, *chi2_e, *scale_part;
  double* scalars;  // [0] chi, [1] scale, [2] maxdiag, [3] pivot_fail
  HuberD hm, hs;
};

constexpr int HPE_STRIDE = 22;  // doubles per edge in Hpp_e: the 21 upper-triangle entries + 1 pad (16-byte records)

// GeometricCamera::project / projectJac(Eigen::Vector3d) of the two camera models on their float parameters
// p = fx fy cx cy, k = k0..k3: Pinhole.cpp:42-48, 71-81; KannalaBrandt8.cpp:46-65 (theta and psi through the float
// atan2f / sqrtf, as the reference writes them), :145-175.
__device__ __forceinline__ void cam_project(bool kb8, const float* p, const float* k, const double* X, double* uv) {
  if (kb8) {
    const double x2_plus_y2 = X[0] * X[0] + X[1] * X[1];
    // atan2f of float arguments: evaluated in fp64 and rounded once (equal to glibc's float routine except where
    // either is an ulp off the exact value; the difference is ~1e-5 px, far inside the 1e-4 bar of the LM deltas)
    const double theta = (double)(float)atan2((double)__fsqrt_rn((float)x2_plus_y2), (double)(float)X[2]);
    const double psi = (double)(float)atan2((double)(float)X[1], (double)(float)X[0]);
    const double theta2 = theta * theta, theta3 = theta * theta2, theta5 = theta3 * theta2, theta7 = theta5 * theta2,
                 theta9 = theta7 * theta2;
    const double r = theta + (double)k[0] * theta3 + (double)k[1] * theta5 + (double)k[2] * theta7 + (double)k[3] * theta9;
    double sn, cs;
    sincos(psi, &sn, &cs);
    uv[0] = (double)p[0] * r * cs + (double)p[2];
    uv[1] = (double)p[1] * r * sn + (double)p[3];
  } else {
    uv[0] = (double)p[0] * X[0] / X[2] + (double)p[2];
    uv[1] = (double)p[1] * X[1] / X[2] + (double)p[3];
  }
}
__device__ __forceinline__ void cam_project_jac(bool kb8, const float* p, const float* k, const double* X, double* J) {
  const double fx = p[0], fy = p[1];
  if (kb8) {
    const double x2 = X[0] * X[0], y2 = X[1] * X[1], z2 = X[2] * X[2];
    const double r2 = x2 + y2, r = sqrt(r2), r3 = r2 * r;
    const double theta = atan2(r, X[2]);
    const double theta2 = theta * theta, theta3 = theta2 * theta, theta4 = theta2 * theta2, theta5 = theta4 * theta,
                 theta6 = theta2 * theta4, theta7 = theta6 * theta, theta8 = theta4 * theta4, theta9 = theta8 * theta;
    const double k0 = k[0], k1 = k[1], k2 = k[2], k3 = k[3];
    const double f = theta + theta3 * k0 + theta5 * k1 + theta7 * k2 + theta9 * k3;
    const double fd = 1 + 3 * k0 * theta2 + 5 * k1 * theta4 + 7 * k2 * theta6 + 9 * k3 * theta8;
    const double den = r2 * (r2 + z2);
    J[0] = fx * (fd * X[2] * x2 / den + f * y2 / r3);
    J[3] = fy * (fd * X[2] * X[1] * X[0] / den - f * X[1] * X[0] / r3);
    J[1] = fx * (fd * X[2] * X[1] * X[0] / den - f * X[1] * X[0] / r3);
    J[4] = fy * (fd * X[2] * y2 / den + f * x2 / r3);
    J[2] = -fx * fd * X[0] / (r2 + z2);
    J[5] = -fy * fd * X[1] / (r2 + z2);
  } else {
    J[0] = fx / X[2]; J[1] = 0.; J[2] = -fx * X[0] / (X[2] * X[2]);
    J[3] = 0.; J[4] = fy / X[2]; J[5] = -fy * X[1] / (X[2] * X[2]);
  }
}
// e->pCamera of a 2-D edge of a rig graph: mpCamera (mono, Optimizer.cc:1326) or mpCamera2 (body, :1387)
struct EdgeCam { bool kb8; const float* p; const float* k; };
__device__ __forceinline__ EdgeCam edge_cam(const LbaDev& D, int k, bool body) {
  const uint8_t m = D.kf_model[k];
  if (body) return EdgeCam{(m & 2) != 0, D.kf_cam2 + 8 * (size_t)k, D.kf_cam2 + 8 * (size_t)k + 4};
  return EdgeCam{(m & 1) != 0, D.kf_cam + 5 * (size_t)k, D.kf_dist + 4 * (size_t)k};
}
// (mTrl * Tcw) of a body edge: SE3Quat::operator* (se3quat.h:104-110)
__device__ __forceinline__ void body_pose(const LbaDev& D, int k, const DQuat& q, const double* t, DQuat& qrw, double* trw) {
  const double* T = D.kf_trl + 7 * (size_t)k;
  const DQuat qrl = {T[0], T[1], T[2], T[3]};
  q_rot(qrl, t, trw);
  trw[0] += T[4]; trw[1] += T[5]; trw[2] += T[6];
  qrw = q_mul(qrl, q);
  q_normalize(qrw);
}

// residual of one edge; returns chi2 (r^T Omega r).  RIG: the graph carries the rig extension (KannalaBrandt8 cameras
// and / or EdgeSE3ProjectXYZToBody edges); P = the keyframe's pose (only read for body edges), X = the landmark
template <bool RIG>
__device__ __forceinline__ double edge_residual(const LbaDev& D, int e, const double* Xc, double* r, const double* P = nullptr,
                                                const double* X = nullptr) {
  const float* cam = D.kf_cam + 5 * D.e_kf[e];
  const double* obs = D.e_obs + 3 * (size_t)e;
  const double s = (double)D.e_is2[e];
  if (RIG && D.e_stereo[e] != LBA_EDGE_STEREO) {
    // OptimizableTypes.h:99-104 / :126-133: obs - pCamera->project(T.map(Xw)), T = Tcw or mTrl * Tcw
    const bool body = D.e_stereo[e] == LBA_EDGE_BODY;
    const EdgeCam c = edge_cam(D, D.e_kf[e], body);
    double Xe[3] = {Xc[0], Xc[1], Xc[2]}, uv[2];
    if (body) {
      DQuat qrw; double trw[3];
      const DQuat q = {P[0], P[1], P[2], P[3]};
      body_pose(D, D.e_kf[e], q, P + 4, qrw, trw);
      q_rot(qrw, X, Xe);
      Xe[0] += trw[0]; Xe[1] += trw[1]; Xe[2] += trw[2];
    }
    cam_project(c.kb8, c.p, c.k, Xe, uv);
    r[0] = obs[0] - uv[0]; r[1] = obs[1] - uv[1]; r[2] = 0;
    return r[0] * (s * r[0]) + r[1] * (s * r[1]);
  }
  if (D.e_stereo[e]) {
    // types_six_dof_expmap.cpp:190-197: invz = 1.0f/trans_xyz[2] is the DOUBLE quotient rounded to float; bf*invz a float product
    const double fx = cam[0], fy = cam[1], cx = cam[2], cy = cam[3];
    const float bf = cam[4];
    const float invz = __double2float_rn(__ddiv_rn(1.0, Xc[2]));
    const double u = Xc[0] * (double)invz * fx + cx;
    const double v = Xc[1] * (double)invz * fy + cy;
    r[0] = obs[0] - u; r[1] = obs[1] - v; r[2] = obs[2] - (u - (double)__fmul_rn(bf, invz));
    return r[0] * (s * r[0]) + r[1] * (s * r[1]) + r[2] * (s * r[2]);
  }
  r[0] = obs[0] - ((double)cam[0] * Xc[0] / Xc[2] + (double)cam[2]);
  r[1] = obs[1] - ((double)cam[1] * Xc[1] / Xc[2] + (double)cam[3]);
  r[2] = 0;
  return r[0] * (s * r[0]) + r[1] * (s * r[1]);
}

// Jacobians of one edge at camera-frame point Xc (pose P = quaternion q + t, landmark X): A = d r / d X (d x 3),
// B = d r / d pose (d x 6), rows padded to three (base_binary_edge.hpp:55-120 calls linearizeOplus of the edge type).
template <bool RIG>
__device__ __forceinline__ void edge_jacobians(const LbaDev& D, int e, int k, const DQuat& q, const double* P, const double* Xc,
                                               double* A, double* B) {
  const int d = D.e_stereo[e] == LBA_EDGE_STEREO ? 3 : 2;
  const float* cam = D.kf_cam + 5 * k;
  double R[9];
  q_to_R(q, R);
  const double x = Xc[0], y = Xc[1], z = Xc[2];
  if (RIG && d == 2) {
    // EdgeSE3ProjectXYZ::linearizeOplus (OptimizableTypes.cpp:139-160) with either camera model:
    //   Xi = -projectJac(Xc) R,  Xj = -projectJac(Xc) SE3deriv(Xc);
    // EdgeSE3ProjectXYZToBody::linearizeOplus (:192-213):
    //   Xi = -projectJac(X_r) (Trl Tlw).rotation(),  Xj = -projectJac(X_r) Rrl SE3deriv(X_l)
    const bool body = D.e_stereo[e] == LBA_EDGE_BODY;
    const EdgeCam c = edge_cam(D, k, body);
    double J[6], Jm[6];
    if (body) {
      const double* T = D.kf_trl + 7 * (size_t)k;
      const DQuat qrl = {T[0], T[1], T[2], T[3]};
      double Xr[3], Rrl[9], trw[3];
      q_rot(qrl, Xc, Xr);
      Xr[0] += T[4]; Xr[1] += T[5]; Xr[2] += T[6];
      cam_project_jac(c.kb8, c.p, c.k, Xr, J);
      q_to_R(qrl, Rrl);
      DQuat qrw;
      body_pose(D, k, q, P + 4, qrw, trw);
      q_to_R(qrw, R);  // the landmark Jacobian rotates with the second camera
#pragma unroll
      for (int rr = 0; rr < 2; rr++)
#pragma unroll
        for (int cc = 0; cc < 3; cc++)
          Jm[rr * 3 + cc] = -(J[rr * 3] * Rrl[cc] + J[rr * 3 + 1] * Rrl[3 + cc] + J[rr * 3 + 2] * Rrl[6 + cc]);
    } else {
      cam_project_jac(c.kb8, c.p, c.k, Xc, J);
#pragma unroll
      for (int i = 0; i < 6; i++) Jm[i] = -J[i];
    }
#pragma unroll
    for (int rr = 0; rr < 2; rr++) {
#pragma unroll
      for (int cc = 0; cc < 3; cc++)
        A[rr * 3 + cc] = -(J[rr * 3] * R[cc] + J[rr * 3 + 1] * R[3 + cc] + J[rr * 3 + 2] * R[6 + cc]);
      const double j0 = Jm[rr * 3], j1 = Jm[rr * 3 + 1], j2 = Jm[rr * 3 + 2];
      // SE3deriv rows: (0,z,-y,1,0,0) (-z,0,x,0,1,0) (y,-x,0,0,0,1)
      B[rr * 6 + 0] = -j1 * z + j2 * y; B[rr * 6 + 1] = j0 * z - j2 * x; B[rr * 6 + 2] = -j0 * y + j1 * x;
      B[rr * 6 + 3] = j0; B[rr * 6 + 4] = j1; B[rr * 6 + 5] = j2;
    }
#pragma unroll
    for (int cc = 0; cc < 3; cc++) A[6 + cc] = 0;
#pragma unroll
    for (int cc = 12; cc < 18; cc++) B[cc] = 0;
  } else if (d == 3) {  // types_six_dof_expmap.cpp:228-274
    const double fx = cam[0], fy = cam[1], bf = cam[4];
    const double z_2 = z * z;
#pragma unroll
    for (int c = 0; c < 3; c++) {
      A[c] = -fx * R[c] / z + fx * x * R[6 + c] / z_2;
      A[3 + c] = -fy * R[3 + c] / z + fy * y * R[6 + c] / z_2;
      A[6 + c] = A[c] - bf * R[6 + c] / z_2;
    }
    B[0] = x * y / z_2 * fx; B[1] = -(1 + (x * x / z_2)) * fx; B[2] = y / z * fx;
    B[3] = -1. / z * fx; B[4] = 0; B[5] = x / z_2 * fx;
    B[6] = (1 + y * y / z_2) * fy; B[7] = -x * y / z_2 * fy; B[8] = -x / z * fy;
    B[9] = 0; B[10] = -1. / z * fy; B[11] = y / z_2 * fy;
    B[12] = B[0] - bf * y / z_2; B[13] = B[1] + bf * x / z_2; B[14] = B[2];
    B[15] = B[3]; B[16] = 0; B[17] = B[5] - bf / z_2;
  } else {  // OptimizableTypes.cpp:139-160 with Pinhole::projectJac
    const double fx = cam[0], fy = cam[1];
    const double J0 = -(fx / z), J2 = fx * x / (z * z), J4 = -(fy / z), J5 = fy * y / (z * z);
#pragma unroll
    for (int c = 0; c < 3; c++) {
      A[c] = J0 * R[c] + J2 * R[6 + c];
      A[3 + c] = J4 * R[3 + c] + J5 * R[6 + c];
      A[6 + c] = 0;
    }
    // SE3deriv rows: (0,z,-y,1,0,0) (-z,0,x,0,1,0) (y,-x,0,0,0,1)
    B[0] = J2 * y;          B[1] = J0 * z - J2 * x; B[2] = -J0 * y; B[3] = J0; B[4] = 0;  B[5] = J2;
    B[6] = -J4 * z + J5 * y; B[7] = -J5 * x;        B[8] = J4 * x;  B[9] = 0;  B[10] = J4; B[11] = J5;
#pragma unroll
    for (int c = 12; c < 18; c++) B[c] = 0;
  }
}

// Per-edge pose-side records (16-byte aligned: 22 / 6 / 18 doubles) written as 16-byte stores: a thread owns a whole
// record, so every store of a warp is its own sector -- halving the store count halves the LSU traffic
__device__ __forceinline__ void store_pose_records(const LbaDev& D, int e, const double* A, const double* B, double ws,
                                                   const double* orr) {
  double he[HPE_STRIDE], bev[6], we[18];
  int t = 0;
#pragma unroll
  for (int i = 0; i < 6; i++) {
#pragma unroll
    for (int j = i; j < 6; j++) he[t++] = ws * (B[i] * B[j] + B[6 + i] * B[6 + j] + B[12 + i] * B[12 + j]);
    bev[i] = B[i] * orr[0] + B[6 + i] * orr[1] + B[12 + i] * orr[2];
#pragma unroll
    for (int j = 0; j < 3; j++) we[i * 3 + j] = ws * (B[i] * A[j] + B[6 + i] * A[3 + j] + B[12 + i] * A[6 + j]);
  }
  he[21] = 0.0;
  double2* He2 = reinterpret_cast<double2*>(D.Hpp_e + HPE_STRIDE * (size_t)e);
  double2* be2 = reinterpret_cast<double2*>(D.bp_e + 6 * (size_t)e);
  double2* We2 = reinterpret_cast<double2*>(D.W + 18 * (size_t)e);
#pragma unroll
  for (int i = 0; i < HPE_STRIDE / 2; i++) He2[i] = make_double2(he[2 * i], he[2 * i + 1]);
#pragma unroll
  for (int i = 0; i < 3; i++) be2[i] = make_double2(bev[2 * i], bev[2 * i + 1]);
#pragma unroll
  for (int i = 0; i < 9; i++) We2[i] = make_double2(we[2 * i], we[2 * i + 1]);
}

// Robust chi2 of a trial state, one thread per landmark: all its edges (base_binary_edge.hpp:55-120).  The
// linearising pass runs one thread per EDGE instead (lin_edge_kernel + lm_gather_kernel below).
template <bool RIG>
__global__ void __launch_bounds__(128) chi_kernel(LbaDev D) {
  const int l = blockIdx.x * 128 + threadIdx.x;
  if (l >= D.n_mp) return;
  const double X[3] = {D.pts[3 * (size_t)l], D.pts[3 * (size_t)l + 1], D.pts[3 * (size_t)l + 2]};
  double chi = 0;
  // the keyframe index -> pose hop is two dependent global loads: the pose of the NEXT edge is fetched while this
  // edge is evaluated (ncu: long-scoreboard stalls were 60 % of all samples at 16 warps per SM)
  const int e_begin = D.lm_ptr[l], e_end = D.lm_ptr[l + 1];
  int k_next = e_begin < e_end ? D.e_kf[e_begin] : 0;
  double Pn[7];
#pragma unroll
  for (int c = 0; c < 7; c++) Pn[c] = D.pose[7 * (size_t)k_next + c];
  for (int e = e_begin; e < e_end; e++) {
    double P[7];
#pragma unroll
    for (int c = 0; c < 7; c++) P[c] = Pn[c];
    if (e + 1 < e_end) {
      k_next = D.e_kf[e + 1];
#pragma unroll
      for (int c = 0; c < 7; c++) Pn[c] = D.pose[7 * (size_t)k_next + c];
    }
    DQuat q = {P[0], P[1], P[2], P[3]};
    double Xc[3], r[3];
    q_rot(q, X, Xc);
    Xc[0] += P[4]; Xc[1] += P[5]; Xc[2] += P[6];
    const double e2 = edge_residual<RIG>(D, e, Xc, r, P, X);
    D.chi2_e[e] = e2;
    double rho0, rho1;
    robustify(D.e_stereo[e] == LBA_EDGE_STEREO ? D.hs : D.hm, e2, rho0, rho1);  // body edges: thHuberMono (:1380-1382)
    chi += rho0;
  }
  D.chi_lm[l] = chi;
}

// The linearising pass, one thread per EDGE: a landmark has ~6.5 edges, so a thread per landmark (as in chi_kernel) runs
// 6.5 x fewer threads, each a serial loop of dependent loads (edge -> keyframe -> pose) -- ncu: 12 % of the DRAM
// throughput, 13 % of the issue slots.  Here every edge is its own thread; its contribution to the landmark block
// (H_ll upper triangle, b_l, robust chi2: 10 doubles) goes to a per-edge record that lm_gather_kernel adds up per
// landmark in edge order -- the same order of additions as the serial loop.
constexpr int LMC_STRIDE = 10;
template <bool RIG>
__global__ void __launch_bounds__(128) lin_edge_kernel(LbaDev D, double* __restrict__ lmc) {
  const int e = blockIdx.x * 128 + threadIdx.x;
  if (e >= D.n_edges) return;
  const int k = D.e_kf[e], l = D.e_free[D.n_edges + e];
  double P[7], X[3];
#pragma unroll
  for (int c = 0; c < 7; c++) P[c] = D.pose[7 * (size_t)k + c];
#pragma unroll
  for (int c = 0; c < 3; c++) X[c] = D.pts[3 * (size_t)l + c];
  DQuat q = {P[0], P[1], P[2], P[3]};
  double Xc[3], r[3];
  q_rot(q, X, Xc);
  Xc[0] += P[4]; Xc[1] += P[5]; Xc[2] += P[6];
  const double e2 = edge_residual<RIG>(D, e, Xc, r, P, X);
  D.chi2_e[e] = e2;
  double rho0, rho1;
  robustify(D.e_stereo[e] == LBA_EDGE_STEREO ? D.hs : D.hm, e2, rho0, rho1);
  double A[9], B[18];
  edge_jacobians<RIG>(D, e, k, q, P, Xc, A, B);
  const double s = (double)D.e_is2[e];
  const double ws = rho1 * s;
  double orr[3];
#pragma unroll
  for (int i = 0; i < 3; i++) orr[i] = -(s * r[i]) * rho1;
  double rec[LMC_STRIDE];
  int t = 0;
#pragma unroll
  for (int i = 0; i < 3; i++) {
#pragma unroll
    for (int j = i; j < 3; j++) rec[t++] = ws * (A[i] * A[j] + A[3 + i] * A[3 + j] + A[6 + i] * A[6 + j]);
    rec[6 + i] = A[i] * orr[0] + A[3 + i] * orr[1] + A[6 + i] * orr[2];
  }
  rec[9] = rho0;
  double2* o2 = reinterpret_cast<double2*>(lmc + LMC_STRIDE * (size_t)e);
#pragma unroll
  for (int i = 0; i < LMC_STRIDE / 2; i++) o2[i] = make_double2(rec[2 * i], rec[2 * i + 1]);
  if (D.e_free[e] >= 0) store_pose_records(D, e, A, B, ws, orr);
}
__global__ void __launch_bounds__(128) lm_gather_kernel(LbaDev D, const double* __restrict__ lmc) {
  const int l = blockIdx.x * 128 + threadIdx.x;
  if (l >= D.n_mp) return;
  double acc[LMC_STRIDE];
#pragma unroll
  for (int i = 0; i < LMC_STRIDE; i++) acc[i] = 0;
  for (int e = D.lm_ptr[l]; e < D.lm_ptr[l + 1]; e++) {
    const double2* r2 = reinterpret_cast<const double2*>(lmc + LMC_STRIDE * (size_t)e);
#pragma unroll
    for (int i = 0; i < LMC_STRIDE / 2; i++) { const double2 v = r2[i]; acc[2 * i] += v.x; acc[2 * i + 1] += v.y; }
  }
  double* H = D.Hll + 6 * (size_t)l;
#pragma unroll
  for (int i = 0; i < 6; i++) H[i] = acc[i];
  D.bl[3 * (size_t)l] = acc[6]; D.bl[3 * (size_t)l + 1] = acc[7]; D.bl[3 * (size_t)l + 2] = acc[8];
  D.chi_lm[l] = acc[9];
}

__device__ __forceinline__ double block_sum(double v, double* sm) {
  // fixed-order reduction: warp shuffles then warp partials in order
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) sm[warp] = v;
  __syncthreads();
  double t = 0;
  for (int w = 0; w < nw; w++) t += sm[w];
  return t;
}

// The same reduction for NV values per thread with two barriers instead of 2 NV (same order of additions as NV calls
// of block_sum: shuffle tree inside a warp, then the warp partials in warp order); totals valid in threads 0..NV-1.
template <int NV, int NW>
__device__ __forceinline__ double block_sum_many(double* v, double (*sm)[NV]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < NV; k++)
    for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_down_sync(0xffffffffu, v[k], o);
  __syncthreads();
  if (lane == 0)
#pragma unroll
    for (int k = 0; k < NV; k++) sm[warp][k] = v[k];
  __syncthreads();
  double t = 0;
  if (threadIdx.x < NV)
    for (int w = 0; w < NW; w++) t += sm[w][threadIdx.x];
  return t;
}

// One CTA per free pose: H_pp (full symmetric 6x6) and b_p.
constexpr int POSE_THREADS = 512;  // a free pose has a few thousand edges at config 5: 128 threads left the gather latency exposed
__global__ void __launch_bounds__(POSE_THREADS) pose_reduce_kernel(LbaDev D) {
  __shared__ double sm[POSE_THREADS / 32][27];
  const int f = blockIdx.x;
  double acc[27];
#pragma unroll
  for (int i = 0; i < 27; i++) acc[i] = 0;
  for (int p = D.pose_ptr[f] + threadIdx.x; p < D.pose_ptr[f + 1]; p += POSE_THREADS) {
    const int e = D.pose_edges[p];
    const double2* He2 = reinterpret_cast<const double2*>(D.Hpp_e + HPE_STRIDE * (size_t)e);  // 16-byte records
    const double2* be2 = reinterpret_cast<const double2*>(D.bp_e + 6 * (size_t)e);
#pragma unroll
    for (int i = 0; i < 10; i++) { const double2 v = He2[i]; acc[2 * i] += v.x; acc[2 * i + 1] += v.y; }
    acc[20] += He2[10].x;
#pragma unroll
    for (int i = 0; i < 3; i++) { const double2 v = be2[i]; acc[21 + 2 * i] += v.x; acc[22 + 2 * i] += v.y; }
  }
  const double tot = block_sum_many<27, POSE_THREADS / 32>(acc, sm);  // thread k < 27 holds total k
  if (threadIdx.x < 21) {
    // upper-triangle index k -> (i, j), row-major over i <= j
    int i = 0, k = (int)threadIdx.x;
    while (k >= 6 - i) { k -= 6 - i; i++; }
    const int j = i + k;
    D.Hpp[36 * (size_t)f + i * 6 + j] = tot;
    D.Hpp[36 * (size_t)f + j * 6 + i] = tot;
  } else if (threadIdx.x < 27) {
    D.bp[6 * (size_t)f + (threadIdx.x - 21)] = tot;
  }
}

// Deterministic sum of an array by one CTA; optional max of |diag| entries.
__global__ void __launch_bounds__(1024) reduce_kernel(const double* a, int n, double* out) {
  __shared__ double sm[32];
  double v = 0;
  for (int i = threadIdx.x; i < n; i += 1024) v += a[i];
  const double t = block_sum(v, sm);
  if (threadIdx.x == 0) *out = t;
}
__global__ void __launch_bounds__(1024) maxdiag_kernel(LbaDev D, const double* Hpp, int with_landmarks, double* out) {
  __shared__ double sm[32];
  double m = 0;
  if (Hpp)
    for (int i = threadIdx.x; i < D.n_free * 6; i += 1024) m = fmax(m, fabs(Hpp[36 * (size_t)(i / 6) + (i % 6) * 7]));
  for (int l = threadIdx.x; with_landmarks && l < D.n_mp; l += 1024) {
    const double* H = D.Hll + 6 * (size_t)l;
    m = fmax(m, fmax(fabs(H[0]), fmax(fabs(H[3]), fabs(H[5]))));
  }
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_down_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) { for (int w = 0; w < 32; w++) m = fmax(m, sm[w]); *out = m; }
}

// Per landmark: D^-1 = (H_ll + lambda I)^-1 (cofactors), D^-1 b_l; y_edge_kernel then forms Y one thread per edge.
__global__ void __launch_bounds__(128) lm_prepare_kernel(LbaDev D, double lambda) {
  const int l = blockIdx.x * 128 + threadIdx.x;
  if (l >= D.n_mp) return;
  const double* H = D.Hll + 6 * (size_t)l;
  const double m0 = H[0] + lambda, m1 = H[1], m2 = H[2], m4 = H[3] + lambda, m5 = H[4], m8 = H[5] + lambda;
  const double c00 = m4 * m8 - m5 * m5, c01 = m5 * m2 - m1 * m8, c02 = m1 * m5 - m4 * m2;
  const double id = 1.0 / (m0 * c00 + m1 * c01 + m2 * c02);
  double Di[9];
  Di[0] = c00 * id; Di[1] = (m2 * m5 - m1 * m8) * id; Di[2] = (m1 * m5 - m2 * m4) * id;
  Di[3] = c01 * id; Di[4] = (m0 * m8 - m2 * m2) * id; Di[5] = (m2 * m1 - m0 * m5) * id;
  Di[6] = c02 * id; Di[7] = (m1 * m2 - m0 * m5) * id; Di[8] = (m0 * m4 - m1 * m1) * id;
  double* Do = D.Dinv + 9 * (size_t)l;
#pragma unroll
  for (int i = 0; i < 9; i++) Do[i] = Di[i];
  const double* b = D.bl + 3 * (size_t)l;
#pragma unroll
  for (int i = 0; i < 3; i++) D.db[3 * (size_t)l + i] = Di[i * 3] * b[0] + Di[i * 3 + 1] * b[1] + Di[i * 3 + 2] * b[2];
}

// Y_e = W_e D_l^-1, one thread per edge (the edges of a landmark are neighbours: its D^-1 comes from L1 / L2).
// 144-byte records, 16-byte aligned: nine 16-byte loads / stores instead of eighteen 8-byte ones.
__global__ void __launch_bounds__(128) y_edge_kernel(LbaDev D) {
  const int e = blockIdx.x * 128 + threadIdx.x;
  if (e >= D.n_edges || D.e_free[e] < 0) return;
  const double* Di = D.Dinv + 9 * (size_t)D.e_free[D.n_edges + e];
  double Dl[9];
#pragma unroll
  for (int i = 0; i < 9; i++) Dl[i] = Di[i];
  const double2* We2 = reinterpret_cast<const double2*>(D.W + 18 * (size_t)e);
  double2* Ye2 = reinterpret_cast<double2*>(D.Y + 18 * (size_t)e);
  double We[18], Ye[18];
#pragma unroll
  for (int i = 0; i < 9; i++) { const double2 v = We2[i]; We[2 * i] = v.x; We[2 * i + 1] = v.y; }
#pragma unroll
  for (int i = 0; i < 6; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) Ye[i * 3 + j] = We[i * 3] * Dl[j] + We[i * 3 + 1] * Dl[3 + j] + We[i * 3 + 2] * Dl[6 + j];
#pragma unroll
  for (int i = 0; i < 9; i++) Ye2[i] = make_double2(Ye[2 * i], Ye[2 * i + 1]);
}

// The Schur contraction on the tensor cores: one CTA (4 warps) per pose pair
// (i1 <= i2); every shared landmark contributes a 6x3 * 3x6 product, issued as an
// fp64 DMMA m8n8k4 (A = Y_{i1,l} padded to 8x4, B = W_{i2,l}^T padded to 4x8).
__global__ void __launch_bounds__(256) schur_pairs_kernel(LbaDev D) {
  __shared__ double part[8][64];
  const int p = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const bool live = (g < 6) && (t < 3);
  const int off = g * 3 + t;
  // two accumulator pairs so consecutive DMMAs do not serialise on the C operand
  double c0 = 0, c1 = 0, e0 = 0, e1 = 0;
  const int beg = D.pair_ptr[p], end = D.pair_ptr[p + 1];
  for (int i0 = beg + warp * 4; i0 < end; i0 += 8 * 4) {
    // 4 entries per trip: all index loads, then all operand loads, then the DMMAs (the loop is a
    // chain of dependent L2 accesses otherwise)
    int ea[4], eb[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int i = i0 + u;
      ea[u] = i < end ? D.pair_ea[i] : -1;
      eb[u] = i < end ? D.pair_eb[i] : -1;
    }
    double a[4], b[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      a[u] = (live && ea[u] >= 0) ? D.Y[18 * (size_t)ea[u] + off] : 0.0;
      b[u] = (live && eb[u] >= 0) ? D.W[18 * (size_t)eb[u] + off] : 0.0;
    }
#pragma unroll
    for (int u = 0; u < 4; u += 2) {
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                   : "+d"(c0), "+d"(c1)
                   : "d"(a[u]), "d"(b[u]));
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                   : "+d"(e0), "+d"(e1)
                   : "d"(a[u + 1]), "d"(b[u + 1]));
    }
  }
  part[warp][g * 8 + 2 * t] = c0 + e0;
  part[warp][g * 8 + 2 * t + 1] = c1 + e1;
  __syncthreads();
  if (threadIdx.x < 36) {
    const int r = threadIdx.x / 6, c = threadIdx.x % 6;  // r: dims of pose i1, c: dims of pose i2
    double v = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) v += part[w][r * 8 + c];
    const int i1 = D.pair_i1[p], i2 = D.pair_i2[p];
    double out = -v;
    if (i1 == i2) out += D.Hpp[36 * (size_t)i1 + r * 6 + c];
    // lower triangle of S: block row i2, block column i1
    D.S[(size_t)(6 * i2 + c) * D.n + 6 * i1 + r] = out;
  }
}

// b_s = b_p - sum_e W_e (D^-1 b_l): row n of the S buffer.  One CTA per free pose.
__global__ void __launch_bounds__(POSE_THREADS) bschur_kernel(LbaDev D) {
  __shared__ double sm[POSE_THREADS / 32][6];
  const int f = blockIdx.x;
  double acc[6] = {0, 0, 0, 0, 0, 0};
  for (int p = D.pose_ptr[f] + threadIdx.x; p < D.pose_ptr[f + 1]; p += POSE_THREADS) {
    const int e = D.pose_edges[p];
    // landmark of edge e: binary search in lm_ptr is avoided by storing db per edge landmark via e_mp
    const double* We = D.W + 18 * (size_t)e;
    const double* d = D.db + 3 * (size_t)D.e_free[D.n_edges + e];  // second half of e_free = landmark id
#pragma unroll
    for (int i = 0; i < 6; i++) acc[i] += We[i * 3] * d[0] + We[i * 3 + 1] * d[1] + We[i * 3 + 2] * d[2];
  }
  const double t = block_sum_many<6, POSE_THREADS / 32>(acc, sm);
  if (threadIdx.x < 6) D.S[(size_t)D.n * D.n + 6 * f + threadIdx.x] = D.bp[6 * (size_t)f + threadIdx.x] - t;
}

// Landmark shards exchange only the row envelope of (S | b_s): rows are packed back to back for the
// ncclAllReduce (dir 0) and scattered into the dense buffer again afterwards (dir 1).  Row n = rhs.
__global__ void __launch_bounds__(256) env_pack_kernel(double* __restrict__ S, int n, const int* __restrict__ first,
                                                       const long long* __restrict__ rowp, double* __restrict__ buf, int dir) {
  const int i = blockIdx.x;
  const int f = i < n ? first[i] : 0, len = i < n ? i - f + 1 : n;
  double* row = S + (size_t)i * n + f;
  double* b = buf + rowp[i];
  for (int j = threadIdx.x; j < len; j += 256) {
    if (dir == 0) b[j] = row[j];
    else row[j] = b[j];
  }
}

__global__ void add_lambda_kernel(LbaDev D, double lambda) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < D.n) D.S[(size_t)i * D.n + i] += lambda;
}

// ---------------------------------------------------------------- dense LDL^T
// (n+1) x n row-major buffer, lower triangle of S in rows 0..n-1, rhs in row n.
// Blocked right-looking LDL^T over all SMs; every CTA factors the 32x32 diagonal
// block redundantly in shared memory (saves a grid barrier), owns a slice of the
// rows below for the panel solve, then a slice of the trailing tiles.
constexpr int NB = 32;

__device__ __forceinline__ void grid_barrier(unsigned* bar, unsigned nblocks, unsigned& gen) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned target = (++gen) * nblocks;
    atomicAdd(bar, 1u);
    while (*(volatile unsigned*)bar < target) { }
    __threadfence();
  }
  __syncthreads();
}

__global__ void __launch_bounds__(256) ldlt_kernel(double* __restrict__ M, int n, unsigned* bar, double* fail) {
  __shared__ double L11[NB][NB + 1];
  __shared__ double Dd[NB];
  __shared__ double Ti[NB][NB + 1];
  __shared__ double Tj[NB][NB + 1];
  const int rows = n + 1;  // including the rhs row
  unsigned gen = 0;
  const unsigned nblk = gridDim.x;
  for (int k0 = 0; k0 < n; k0 += NB) {
    const int nb = min(NB, n - k0);
    // ---- diagonal block (redundant per CTA)
    for (int i = threadIdx.x; i < NB * NB; i += 256) {
      const int r = i / NB, c = i % NB;
      L11[r][c] = (r < nb && c <= r) ? M[(size_t)(k0 + r) * n + k0 + c] : 0.0;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
      // right-looking LDL^T of the 32x32 block by one warp: lane r keeps row r in registers, the
      // scaled column is broadcast through shared memory.  The serial chain per column is one
      // reciprocal + one FMA (the left-looking form chained a whole dot product: 12.8 us / panel).
      const int r = threadIdx.x;
      double* colbuf = &Ti[0][0];
      double a[NB];
#pragma unroll
      for (int m = 0; m < NB; m++) a[m] = L11[r][m];
#pragma unroll
      for (int c = 0; c < NB; c++) {
        if (c < nb) {  // uniform
          const double d = __shfl_sync(0xffffffffu, a[c], c);
          if (r == c) { Dd[c] = d; if (d == 0.0) *fail = 1.0; }
          // 1/d: fp32 seed + two Newton steps in fp64 (~1 ulp) instead of the slow IEEE division
          double inv = (double)__frcp_rn((float)d);
          inv = inv * (2.0 - d * inv);
          inv = inv * (2.0 - d * inv);
          const double ld = a[c];  // (L*D)[r][c] for r > c
          colbuf[r] = ld;
          __syncwarp();
          if (r > c) {
            const double l = ld * inv;
#pragma unroll
            for (int m = c + 1; m < NB; m++)
              if (m <= r) a[m] -= l * colbuf[m];
            a[c] = l;
          }
          __syncwarp();
        }
      }
#pragma unroll
      for (int m = 0; m < NB; m++)
        if (m < r) L11[r][m] = a[m];
    }
    __syncthreads();
    // ---- panel: rows below the block, one warp per row (lane j owns column j of the row);
    //      forward substitution with the running value broadcast by shuffle
    const int r0 = k0 + nb;
    {
      const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
      for (int i = r0 + blockIdx.x * 8 + warp; i < rows; i += 8 * nblk) {
        double* Mi = M + (size_t)i * n + k0;
        double a = (lane < nb) ? Mi[lane] : 0.0;
        for (int m = 0; m < nb; m++) {
          const double ldm = __shfl_sync(0xffffffffu, a, m);  // (L*D)_im is final once m steps are done
          if (lane > m) a -= ldm * L11[lane][m];
        }
        if (lane < nb) Mi[lane] = a / Dd[lane];
      }
    }
    grid_barrier(bar, nblk, gen);
    // every CTA has loaded the diagonal block by now: publish its factor
    if (blockIdx.x == 0) {
      for (int i = threadIdx.x; i < nb * nb; i += 256) {
        const int r = i / nb, c = i % nb;
        if (c < r) M[(size_t)(k0 + r) * n + k0 + c] = L11[r][c];
        else if (c == r) M[(size_t)(k0 + r) * n + k0 + c] = Dd[r];
      }
    }
    // ---- trailing update, 32x32 tiles (bi >= bj), rhs row is the last partial tile row
    const int T = (rows - r0 + NB - 1) / NB;
    const int ntiles = T * (T + 1) / 2;
    for (int tile = blockIdx.x; tile < ntiles; tile += nblk) {
      // tile -> (bi, bj), bi >= bj
      int bi = (int)((sqrt(8.0 * tile + 1.0) - 1.0) * 0.5);
      while ((bi + 1) * (bi + 2) / 2 <= tile) bi++;
      while (bi * (bi + 1) / 2 > tile) bi--;
      const int bj = tile - bi * (bi + 1) / 2;
      const int i0 = r0 + bi * NB, j0 = r0 + bj * NB;
      if (j0 >= n) continue;  // column block beyond the matrix (only the rhs row exists there)
      __syncthreads();
      for (int i = threadIdx.x; i < NB * NB; i += 256) {
        const int r = i / NB, c = i % NB;
        Ti[r][c] = (i0 + r < rows && c < nb) ? M[(size_t)(i0 + r) * n + k0 + c] : 0.0;
        Tj[r][c] = (j0 + r < n && c < nb) ? M[(size_t)(j0 + r) * n + k0 + c] * Dd[c] : 0.0;
      }
      __syncthreads();
      for (int i = threadIdx.x; i < NB * NB; i += 256) {
        const int r = i / NB, c = i % NB;
        const int gi = i0 + r, gj = j0 + c;
        if (gi >= rows || gj >= n || gj > gi) continue;
        double s = 0;
#pragma unroll 8
        for (int m = 0; m < NB; m++) s += Ti[r][m] * Tj[c][m];
        M[(size_t)gi * n + gj] -= s;
      }
    }
    grid_barrier(bar, nblk, gen);
  }
}

// L^T x = z  (z = row n of M after ldlt_kernel).  Single CTA, right-looking: solve the last
// 32 unknowns from a shared-memory copy of their diagonal block, then subtract their
// contribution from every earlier right-hand side (rows of L are contiguous: coalesced).
__global__ void __launch_bounds__(1024) backsub_kernel(const double* __restrict__ M, int n, double* __restrict__ x) {
  extern __shared__ double acc[];  // n entries
  __shared__ double xb[NB];
  __shared__ double Lb[NB][NB + 1];
  for (int i = threadIdx.x; i < n; i += 1024) acc[i] = M[(size_t)n * n + i];
  const int nblocks = (n + NB - 1) / NB;
  for (int b = nblocks - 1; b >= 0; b--) {
    const int k0 = b * NB, nb = min(NB, n - k0);
    {
      const int r = threadIdx.x >> 5, c = threadIdx.x & 31;  // 1024 threads = 32 x 32
      Lb[r][c] = (r < nb && c < r) ? M[(size_t)(k0 + r) * n + k0 + c] : 0.0;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
      // unit upper-triangular solve inside the block, last row first
      const int r = threadIdx.x;
      double v = (r < nb) ? acc[k0 + r] : 0.0;
      for (int c = nb - 1; c >= 0; c--) {
        const double xc = __shfl_sync(0xffffffffu, v, c);
        if (r < c) v -= Lb[c][r] * xc;
      }
      if (r < nb) { xb[r] = v; x[k0 + r] = v; }
    }
    __syncthreads();
    // acc[j] -= sum_{i in block} L[i][j] x_i for j < k0
    for (int j = threadIdx.x; j < k0; j += 1024) {
      const double* col = M + (size_t)k0 * n + j;
      double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
      int i = 0;
      for (; i + 4 <= nb; i += 4) {  // four independent loads in flight
        s0 += col[(size_t)i * n] * xb[i];
        s1 += col[(size_t)(i + 1) * n] * xb[i + 1];
        s2 += col[(size_t)(i + 2) * n] * xb[i + 2];
        s3 += col[(size_t)(i + 3) * n] * xb[i + 3];
      }
      for (; i < nb; i++) s0 += col[(size_t)i * n] * xb[i];
      acc[j] -= (s0 + s1) + (s2 + s3);
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------- envelope (skyline) LDL^T
// The reduced system of a local window is block-banded once the keyframes are ordered along the
// covisibility chain (g2o hands Eigen's SimplicialLDLT a sparse matrix for the same reason,
// linear_solver_eigen.h:94-124): without pivoting the factor never leaves the row envelope of S.  This
// kernel factors S inside its envelope with ONE CTA -- no grid barriers -- and solves for x in the same
// launch.  Per 32-column panel: (1) the 32x32 diagonal block by the 1024 threads (one register each, the
// pivot column broadcast through shared memory: ~32 x (barrier + reciprocal) on the critical path),
// (2) the rows of the envelope below it (<= SKY_WMAX, one warp per row, forward substitution by shuffles),
// their L and L*D kept in shared memory, (3) the trailing update of the window's lower triangle in 4x4
// register micro-tiles straight from those two shared arrays.  `reach[c]` = last row whose envelope
// contains a column <= c (prefix maximum, host-built from the pose-pair list); row n is the right-hand side.
constexpr int SKY_THREADS = 1024;
constexpr int SKY_WMAX = 320;  // rows of one panel window incl. the rhs row (dynamic shared memory: 2 x 32 x WMAX doubles)

__global__ void __launch_bounds__(SKY_THREADS) ldlt_sky_kernel(double* __restrict__ M, int n, const int* __restrict__ reach,
                                                             const int* __restrict__ first, double* fail,
                                                             double* __restrict__ x) {
  extern __shared__ __align__(16) double sky_dyn[];
  double* Alt = sky_dyn;                         // [32][SKY_WMAX]  L   of the window rows, transposed (m major)
  double* Aldt = sky_dyn + 32 * SKY_WMAX;        // [32][SKY_WMAX]  L*D of the window rows
  __shared__ double L11[NB][NB + 1];
  __shared__ double colb[NB];
  __shared__ double Dd[NB], Di[NB];
  __shared__ double xb[NB];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int k0 = 0; k0 < n; k0 += NB) {
    const int nb = min(NB, n - k0);
    // ---- (1) diagonal block: thread (r, c) owns a[r][c], r = warp, c = lane
    {
      const int r = warp, c = lane;
      double a = (r < nb && c <= r) ? M[(size_t)(k0 + r) * n + k0 + c] : 0.0;
      for (int k = 0; k < nb; k++) {
        if (c == k && r >= k) colb[r] = a;  // column k of L*D (pivot included)
        __syncthreads();
        const double d = colb[k];
        // 1/d: fp32 seed + two Newton steps in fp64 (~1 ulp), redundantly per thread
        double inv = (double)__frcp_rn((float)d);
        inv = inv * (2.0 - d * inv);
        inv = inv * (2.0 - d * inv);
        if (r == k && c == k) { Dd[k] = d; Di[k] = inv; if (d == 0.0) *fail = 1.0; }
        if (r > k && c > k && c <= r) a -= (colb[r] * inv) * colb[c];
        if (c == k && r > k) a = colb[r] * inv;  // L[r][k]
        __syncthreads();
      }
      L11[r][c] = a;  // strictly lower part = L, diagonal = D
      if (r < nb && c <= r) M[(size_t)(k0 + r) * n + k0 + c] = a;
    }
    __syncthreads();
    // ---- (2) panel rows: the envelope rows below the block, then the rhs row (window index w)
    const int r0 = k0 + nb;
    const int rend = min(max(reach[k0 + nb - 1] + 1, r0), n);  // envelope rows are [r0, rend)
    const int nw = rend - r0 + 1;                               // + rhs
    for (int w = warp; w < nw; w += SKY_THREADS / 32) {
      const int i = (w < nw - 1) ? r0 + w : n;
      double* Mi = M + (size_t)i * n + k0;
      double a = (lane < nb) ? Mi[lane] : 0.0;
      for (int m = 0; m < nb; m++) {
        const double ldm = __shfl_sync(0xffffffffu, a, m);  // (L*D)_im is final once m steps are done
        if (lane > m) a -= ldm * L11[lane][m];
      }
      const double l = (lane < nb) ? a * Di[lane] : 0.0;
      if (lane < nb) Mi[lane] = l;
      Alt[lane * SKY_WMAX + w] = l;
      Aldt[lane * SKY_WMAX + w] = (lane < nb) ? a : 0.0;
    }
    __syncthreads();
    // ---- (3) trailing update inside the window: M[i][j] -= sum_m L[i][m] (L*D)[j][m], j <= i, 4x4 micro-tiles
    {
      const int T = (nw + 3) >> 2;           // micro-tile rows
      const int ntile = T * (T + 1) / 2;
      for (int t = tid; t < ntile; t += SKY_THREADS) {
        int ti = (int)((sqrtf(8.f * (float)t + 1.f) - 1.f) * 0.5f);
        while ((ti + 1) * (ti + 2) / 2 <= t) ti++;
        while (ti * (ti + 1) / 2 > t) ti--;
        const int tj = t - ti * (ti + 1) / 2;
        double acc[4][4];
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
          for (int b = 0; b < 4; b++) acc[a][b] = 0.0;
#pragma unroll 4
        for (int m = 0; m < NB; m++) {
          const double2 li0 = *reinterpret_cast<const double2*>(&Alt[m * SKY_WMAX + 4 * ti]);
          const double2 li1 = *reinterpret_cast<const double2*>(&Alt[m * SKY_WMAX + 4 * ti + 2]);
          const double2 lj0 = *reinterpret_cast<const double2*>(&Aldt[m * SKY_WMAX + 4 * tj]);
          const double2 lj1 = *reinterpret_cast<const double2*>(&Aldt[m * SKY_WMAX + 4 * tj + 2]);
          const double li[4] = {li0.x, li0.y, li1.x, li1.y}, lj[4] = {lj0.x, lj0.y, lj1.x, lj1.y};
#pragma unroll
          for (int a = 0; a < 4; a++)
#pragma unroll
            for (int b = 0; b < 4; b++) acc[a][b] += li[a] * lj[b];
        }
#pragma unroll
        for (int a = 0; a < 4; a++) {
          const int wi = 4 * ti + a;
          if (wi >= nw) continue;
          const int gi = (wi < nw - 1) ? r0 + wi : n;
#pragma unroll
          for (int b = 0; b < 4; b++) {
            const int wj = 4 * tj + b;
            if (wj >= nw - 1 || wj > wi) continue;  // the rhs row has no column; lower triangle only
            M[(size_t)gi * n + r0 + wj] -= acc[a][b];
          }
        }
      }
    }
    __syncthreads();
  }
  // ---- L^T x = z, z = row n (already scaled by 1/D).  Blocks from the last to the first; the running
  //      right-hand side lives in shared memory (Alt is free now), contributions of a solved block are
  //      gathered row-wise (coalesced) into Aldt and summed per column.
  double* acc = Alt;  // n <= 32 * SKY_WMAX
  for (int i = tid; i < n; i += SKY_THREADS) acc[i] = M[(size_t)n * n + i];
  __syncthreads();
  const int nblocks = (n + NB - 1) / NB;
  for (int b = nblocks - 1; b >= 0; b--) {
    const int k0 = b * NB, nb = min(NB, n - k0);
    L11[warp][lane] = (warp < nb && lane < warp) ? M[(size_t)(k0 + warp) * n + k0 + lane] : 0.0;
    __syncthreads();
    if (warp == 0) {
      double v = (lane < nb) ? acc[k0 + lane] : 0.0;
      for (int c = nb - 1; c >= 0; c--) {
        const double xc = __shfl_sync(0xffffffffu, v, c);
        if (lane < c) v -= L11[c][lane] * xc;
      }
      if (lane < nb) { xb[lane] = v; x[k0 + lane] = v; }
    }
    __syncthreads();
    // columns [jmin, k0) can hold non-zeros of the block's rows
    int jmin = k0;
    for (int r = 0; r < nb; r++) jmin = min(jmin, first[k0 + r]);
    const int wcols = k0 - jmin;  // <= SKY_WMAX - 1 (host-checked)
    if (wcols > 0) {
      if (warp < nb) {
        const double xi = xb[warp];
        const double* Li = M + (size_t)(k0 + warp) * n + jmin;
        for (int j = lane; j < wcols; j += 32) Aldt[warp * SKY_WMAX + j] = Li[j] * xi;
      }
      __syncthreads();
      for (int j = tid; j < wcols; j += SKY_THREADS) {
        double s = 0;
        for (int r = 0; r < nb; r++) s += Aldt[r * SKY_WMAX + j];
        acc[jmin + j] -= s;
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------- window-resident envelope LDL^T
// Third formulation of the reduced solve, for narrow envelopes (a keyframe chain: <= WIN_ROWS rows under a
// pivot).  What bounded ldlt_sky_kernel was not arithmetic but a chain of ~1200 pivots at ~1 us each: every
// 32-column panel paid global-memory round trips (diagonal block in, panel rows in/out, trailing tiles in/out)
// and 64 block-wide barriers.  Here the active part of the matrix -- the rows of the envelope under the current
// pivots, a (<= 120)^2 lower triangle -- LIVES in shared memory as a ring (row i, column j at [i % WIN][j % WIN]);
// rows enter it once, from global memory, when the envelope first reaches them (independent loads, off the
// critical path), are updated in place panel after panel, and leave as finished columns of L.  Panels are 8
// columns wide: the 8x8 pivot block is factored by one thread entirely in registers (no communication on the
// chain), the panel rows on the tensor pipe through the inverse of the pivot block, the rank-8 update of the window
// in 8x8 DMMA tiles; two barriers per 8 pivots instead of 64 per 32.  The back-substitution runs in the same launch,
// 8 unknowns per step, with the next step's rows of L already in flight.
constexpr int WIN = 128, WIN_P = WIN + 1, WIN_ROWS = WIN - 8, WPB = 8, WIN_THREADS = 512;
constexpr int WIN_LP = 132;  // row pitch of the m-major L / L*D panels: the four k-rows of a DMMA fragment fall into different banks

// Asynchronous 8-byte copies global -> shared (LDGSTS): unlike a load into registers they are not waited for by
// bar.sync, so a copy issued in one phase of ldlt_win_kernel can be in flight across the barriers of the next ones
// (measured: with register loads every barrier paid the full global-memory round trip of the loads before it).
// `valid == false` writes zeros without reading.
__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gsrc, bool valid) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int sz = valid ? 8 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ int wmod(int v) { return v & (WIN - 1); }  // v % WIN for v >= 0 (ring indices)
static_assert((WIN & (WIN - 1)) == 0, "ring size must be a power of two");

// One side of a solve: the matrix (its own (n+1) x n buffer), its envelope tables, and -- for the two-sided solve --
// where the side stops.  WinArgs.mode: 0 = factor everything and back-substitute (one CTA, side 0);
// 1 = factor panels [0, pend) and write the window that is left (the separator rows with this side's Schur
// update applied, + their right-hand side entries) to `dump` (row pitch wd = esep - ksep, rhs at dump[wd * wd]);
// 2 = back-substitute columns [0, ksep) given the separator's solution xs.  Modes 1 and 2 run one CTA per side.
struct WinSide {
  double* M; const int* reach; const int* first; double* dump;
  int n, pend, ksep, esep;
};
struct WinArgs {
  WinSide s[2];
  double* fail; double* x; const double* xs;
  int mode, msep;  // msep: first separator column in the caller's numbering (side 1 runs in reversed numbering)
};

// __grid_constant__: wa.s[blockIdx.x] is read in place from the parameter space; without it the compiler may copy
// the whole struct to local memory to index it
__global__ void __launch_bounds__(WIN_THREADS) ldlt_win_kernel(const __grid_constant__ WinArgs wa) {
  const WinSide& sd = wa.s[blockIdx.x];
  double* __restrict__ M = sd.M;
  const int n = sd.n, mode = wa.mode;
  const int* __restrict__ reach = sd.reach;
  const int* __restrict__ first_g = sd.first;
  double* fail = wa.fail;
  double* __restrict__ x = wa.x;
  extern __shared__ __align__(16) double win_dyn[];
  double* A = win_dyn;                       // [WIN][WIN_P] ring of the trailing window
  double* zr = A + WIN * WIN_P;              // [WIN] right-hand side entries of the window columns
  double* Lt = zr + WIN;                     // [8][WIN_LP] L of the panel rows, m-major; slot nr = rhs row
  double* LDt = Lt + WPB * WIN_LP;           // [8][WIN_LP] L*D of the panel rows
  int* first = reinterpret_cast<int*>(LDt + WPB * WIN_LP);  // [n] envelope starts (read at every step: keep them on chip)
  int* rlast = first + n;                    // [ceil(n/8)] last window row of every panel
  double* stg = reinterpret_cast<double*>(rlast + ((((n + WPB - 1) / WPB) + 1) & ~1));  // [12][WIN + 8] rows on their way into the window (n = 6 x poses is even)
  __shared__ double Lb[WPB][WPB];            // pivot block: strict lower = L, diagonal = D
  __shared__ double Dib[WPB];                // 1 / D
  __shared__ double Gi[WPB][WPB];            // inverse of the unit lower-triangular pivot block (phase (A) on the tensor pipe)
  __shared__ unsigned short tile_ij[(WIN / 8) * (WIN / 8 + 1) / 2];  // lower-triangle tile number -> (ti << 8) | tj
  const int lane = threadIdx.x & 31;
  const int warp = (int)(threadIdx.x >> 5), tid = warp * 32 + lane;
  const int npan = (n + WPB - 1) / WPB;
  for (int i = tid; i < n; i += WIN_THREADS) first[i] = first_g[i];
  for (int p = tid; p < npan; p += WIN_THREADS) {
    const int k0 = p * WPB, nb = min(WPB, n - k0);
    rlast[p] = min(max(reach[k0 + nb - 1], k0 + nb - 1), n - 1);
  }
  for (int ti = tid; ti < WIN / 8; ti += WIN_THREADS)
    for (int tj = 0; tj <= ti; tj++) tile_ij[ti * (ti + 1) / 2 + tj] = (unsigned short)((ti << 8) | tj);
  __syncthreads();
  // rows [lo, hi] enter the window: columns [c0, i], zero left of the envelope (the ring slot is stale).
  // Called by warps w0.. of the CTA; all loads of a call are independent.
  auto load_rows = [&](int lo, int hi, int c0, int w0, int nwarps) {
    for (int i = lo + (warp - w0); i <= hi; i += nwarps) {
      const int f = first[i];
      const double* Mi = M + (size_t)i * n;
      double* Ai = A + (wmod(i)) * WIN_P;
      // a row of the window has at most WIN columns: four loads per lane, all in flight together
      double v[4];
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const int j = c0 + lane + 32 * q;
        v[q] = (j <= i && j >= f) ? Mi[j] : 0.0;
      }
      const double zv = lane == 0 ? M[(size_t)n * n + i] : 0.0;
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const int j = c0 + lane + 32 * q;
        if (j <= i) Ai[wmod(j)] = v[q];
      }
      if (lane == 0) zr[wmod(i)] = zv;
    }
  };
  // pivot block of panel p, one thread, registers only: factors rows/cols [k0, k0+nb) of the ring, leaves L (strict
  // lower) and D in Lb, 1/D in Dib; another warp writes them to M during the next phase (pivot_store)
  auto pivot = [&](int p) {
    const int k0 = p * WPB, nb = min(WPB, n - k0);
    double a[WPB][WPB];
#pragma unroll
    for (int r = 0; r < WPB; r++) {
      const double* Ar = A + (wmod(k0 + r)) * WIN_P;
#pragma unroll
      for (int c = 0; c < WPB; c++) a[r][c] = (r < nb && c <= r) ? Ar[wmod(k0 + c)] : (r == c ? 1.0 : 0.0);
    }
#pragma unroll
    for (int k = 0; k < WPB; k++) {
      const double d = a[k][k];
      if (d == 0.0) *fail = 1.0;
      // 1/d: the hardware's fp64 reciprocal seed (MUFU.RCP64H, ~20 bits, no float round trip) + two Newton steps
      double inv;
      asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(inv) : "d"(d));
      inv = inv * (2.0 - d * inv);
      inv = inv * (2.0 - d * inv);
      Dib[k] = inv;
      double l[WPB];
#pragma unroll
      for (int r = k + 1; r < WPB; r++) l[r] = a[r][k] * inv;
#pragma unroll
      for (int r = k + 1; r < WPB; r++)
#pragma unroll
        for (int m = k + 1; m <= r; m++) a[r][m] -= l[r] * a[m][k];
#pragma unroll
      for (int r = k + 1; r < WPB; r++) a[r][k] = l[r];
    }
#pragma unroll
    for (int r = 0; r < WPB; r++)
#pragma unroll
      for (int c = 0; c <= r; c++) Lb[r][c] = a[r][c];
  };
  // G = L_bb^-1 (unit lower triangular) after pivot(): lane r of the pivot's warp forms column r,
  // g[c] = -sum_{m<c} L[c][m] g[m] below the diagonal (L[c][c] = 1), one uniform instruction stream for the eight
  // lanes.  Phase (A) multiplies the panel rows by G^T on the tensor pipe.
  auto pivot_inverse = [&]() {
    __syncwarp();
    if (lane < WPB) {
      double g[WPB];
      g[0] = lane == 0 ? 1.0 : 0.0;
#pragma unroll
      for (int c = 1; c < WPB; c++) {
        double t = 0.0;
#pragma unroll
        for (int m = 0; m < c; m++) t += Lb[c][m] * g[m];
        g[c] = c > lane ? -t : (c == lane ? 1.0 : 0.0);
      }
#pragma unroll
      for (int c = 0; c < WPB; c++) Gi[c][lane] = g[c];
    }
  };
  auto pivot_store = [&](int p) {  // one warp, in phase (A) of panel p (Lb is stable until the barrier)
    const int k0 = p * WPB, nb = min(WPB, n - k0);
    for (int e = lane; e < WPB * WPB; e += 32) {
      const int r = e >> 3, c = e & 7;
      if (r < nb && c <= r) M[(size_t)(k0 + r) * n + k0 + c] = Lb[r][c];  // L below, D on the diagonal
    }
  };
  // 8x8 tiles of the rank-nb update of panel (r0, nr): C -= L_i (8x8) * (L*D)_j^T, two fp64 DMMA m8n8k4 each;
  // fragment layout A[g][t], B[t][g], C[g][2t], C[g][2t+1] with g = lane / 4, t = lane % 4.  A warp owns a run of
  // consecutive tiles (row-major over the lower triangle) and handles TG at a time: the operands of all of them are
  // fetched before the first DMMA, so TG accumulator chains are in flight instead of one (the kernel is bound by
  // the latency of its dependent chains, not by throughput).
  const int fg = lane >> 2, ft = lane & 3;
  constexpr int ZR_OFF = WIN * WIN_P;  // zr follows the ring: one index space for matrix rows and the rhs row
  constexpr int TG = 4;  // interior tiles in flight per warp
  auto mma2 = [&](double& c0, double& c1, double a0, double a1, double b0, double b1) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(c0), "+d"(c1) : "d"(a0), "d"(b0));
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(c0), "+d"(c1) : "d"(a1), "d"(b1));
  };
  auto update_run = [&](int t_begin, int t_end, int r0, int nr) {
    if (t_begin >= t_end) return;
    const int tt = tile_ij[t_begin];
    int ti = tt >> 8, tj = tt & 255, t = t_begin;
    while (t < t_end) {
      const int wi = 8 * ti + fg;
      const double a0 = -Lt[ft * WIN_LP + wi], a1 = -Lt[(ft + 4) * WIN_LP + wi];
      const int rowoff = (wi >= nr) ? ZR_OFF : (wmod(r0 + wi)) * WIN_P;  // the rhs row has no column of its own
      // tiles strictly below the diagonal in a row block that lies inside the window need no element predicates
      // and share the row operands: TG of them at a time, all loads before the first DMMA
      if (8 * ti + 7 <= nr) {
        while (tj + TG <= ti && t + TG <= t_end) {
          int i0[TG], i1[TG];
          double b0[TG], b1[TG], c0[TG], c1[TG];
#pragma unroll
          for (int u = 0; u < TG; u++) {
            const int cj = 8 * (tj + u);
            b0[u] = LDt[ft * WIN_LP + cj + fg]; b1[u] = LDt[(ft + 4) * WIN_LP + cj + fg];
            i0[u] = rowoff + wmod(r0 + cj + 2 * ft);
            i1[u] = rowoff + wmod(r0 + cj + 2 * ft + 1);
            c0[u] = A[i0[u]]; c1[u] = A[i1[u]];
          }
#pragma unroll
          for (int u = 0; u < TG; u++) mma2(c0[u], c1[u], a0, a1, b0[u], b1[u]);
#pragma unroll
          for (int u = 0; u < TG; u++) { A[i0[u]] = c0[u]; A[i1[u]] = c1[u]; }
          tj += TG; t += TG;
        }
        if (t >= t_end) break;
      }
      // one tile, fully predicated (diagonal tiles, the last row block, the tail of a run)
      {
        const int wj = 8 * tj + 2 * ft;
        const double b0 = LDt[ft * WIN_LP + 8 * tj + fg], b1 = LDt[(ft + 4) * WIN_LP + 8 * tj + fg];
        const bool ok0 = wi <= nr && wj < nr && wj <= wi, ok1 = wi <= nr && wj + 1 < nr && wj + 1 <= wi;
        const int i0 = rowoff + wmod(r0 + wj), i1 = rowoff + wmod(r0 + wj + 1);
        double c0 = ok0 ? A[i0] : 0.0, c1 = ok1 ? A[i1] : 0.0;
        mma2(c0, c1, a0, a1, b0, b1);
        if (ok0) A[i0] = c0;
        if (ok1) A[i1] = c1;
        if (tj == ti) { ti++; tj = 0; } else tj++;
        t++;
      }
    }
  };
  // the tile of the next pivot block, on the critical path: no tile bookkeeping at all
  auto update_tile0 = [&](int r0, int nr) {
    const int wj = 2 * ft;
    const double a0 = -Lt[ft * WIN_LP + fg], a1 = -Lt[(ft + 4) * WIN_LP + fg];
    const double b0 = LDt[ft * WIN_LP + fg], b1 = LDt[(ft + 4) * WIN_LP + fg];
    const int rowoff = (fg >= nr) ? ZR_OFF : (wmod(r0 + fg)) * WIN_P;
    const bool ok0 = fg <= nr && wj < nr && wj <= fg, ok1 = fg <= nr && wj + 1 < nr && wj + 1 <= fg;
    const int i0 = rowoff + wmod(r0 + wj), i1 = rowoff + wmod(r0 + wj + 1);
    double c0 = ok0 ? A[i0] : 0.0, c1 = ok1 ? A[i1] : 0.0;
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(c0), "+d"(c1) : "d"(a0), "d"(b0));
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(c0), "+d"(c1) : "d"(a1), "d"(b1));
    if (ok0) A[i0] = c0;
    if (ok1) A[i1] = c1;
  };
  // warps of phase (A): four 8-row blocks per warp (WIN / 32 warps cover a whole window); the other warps bring rows
  // into the window
  // (measured: eight forward warps + eight loaders is 6 % slower than four + twelve -- 4.06 vs 3.81 ms per optimize(10)
  // at config 5 -- although phase (A) itself gets shorter)
  constexpr int FWD_WARPS = WIN / 32;
  constexpr int LD_WARPS = WIN_THREADS / 32 - FWD_WARPS;  // the other warps bring rows into the window
  // A row that panel p+2 adds to the window is copied asynchronously into a staging row during phase (A) of panel
  // p and moved into the ring during phase (A) of panel p+1 (when its slot is free): a whole panel of time for the
  // round trip to global memory instead of a wait inside the phase.  One row per loader warp and panel; a panel that adds more
  // rows than there are loader warps (irregular envelopes) loads the rest directly.
  int pf_row = -1, pf_c0 = 0;
  double* my_stg = stg + (warp >= FWD_WARPS ? warp - FWD_WARPS : 0) * (WIN + 8);
  auto prefetch_row = [&](int i, int c0) {
    const int f = first[i];
    const double* Mi = M + (size_t)i * n;
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const int j = c0 + lane + 32 * q;
      const bool valid = j <= i && j >= f;
      cp_async8(my_stg + lane + 32 * q, valid ? Mi + j : M, valid);
    }
    if (lane == 0) cp_async8(my_stg + WIN, M + (size_t)n * n + i, true);
    cp_async_commit();
    pf_row = i; pf_c0 = c0;
  };
  auto commit_row = [&]() {
    if (pf_row < 0) return;
    cp_async_wait<0>();
    double* Ai = A + (wmod(pf_row)) * WIN_P;
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const int j = pf_c0 + lane + 32 * q;
      if (j <= pf_row) Ai[wmod(j)] = my_stg[lane + 32 * q];
    }
    if (lane == 0) zr[wmod(pf_row)] = my_stg[WIN];
    pf_row = -1;
  };
  // first new row of panel q's window (q >= 1), as phase (A) of panel q-1 computes it
  auto new_rows_lo = [&](int q) {
    const int r0q = q * WPB;  // = k0 + nb of panel q-1 (only the last panel is short)
    const int preq = min(r0q + WPB - 1, n - 1);
    return max(rlast[q - 1], preq) + 1;
  };
  const int pend = mode == 1 ? sd.pend : (mode == 2 ? 0 : npan);  // panels this CTA eliminates
  if (pend > 0) {
    load_rows(0, rlast[0], 0, 0, WIN_THREADS / 32);
    if (warp >= FWD_WARPS && pend > 1) {
      const int i = new_rows_lo(1) + (warp - FWD_WARPS);
      if (i <= rlast[1]) prefetch_row(i, WPB);
    }
    __syncthreads();
    if (warp == 0) {
      if (tid == 0) pivot(0);
      pivot_inverse();
    }
  }
  __syncthreads();
  for (int p = 0; p < pend; p++) {
    const int k0 = p * WPB, nb = min(WPB, n - k0);
    const int R = rlast[p];  // last row of the window; rows [k0, R] are resident, the pivot block is factored
    const bool more = p + 1 < pend;
    // rows of the next pivot block that are not resident yet (narrow or ending envelope) are loaded by warp 0 in (B)
    const int r0 = k0 + nb, nr = R - r0 + 1;  // nr rows under the pivot block; slot nr = rhs
    const int pre = more ? min(r0 + WPB - 1, n - 1) : R;
    // ---- (A) panel rows [k0+nb, R] and the rhs row: forward substitution on the tensor pipe.  The other warps
    //      bring in the rows the NEXT panel adds to the window (their ring slots are free: the window of panel p+1
    //      starts at r0), so the global-memory latency is off the chain.
    // (L*D) rows = A_rows * L_bb^-T: one 8-row block per warp trip, two fp64 DMMA m8n8k4 (A[g][t] = window row
    // g, panel column t / t+4; B[t][g] = G[g][t] / G[g][t+4]; C[g][2t], C[g][2t+1]); L = (L*D) / D.  The rhs row
    // is row nr of the window (zr).  Blocks of a warp are independent: all operand loads first.
    if (warp < FWD_WARPS) {
      const int nblk = (nr + 1 + 7) >> 3;
      const double g0 = Gi[fg][ft], g1 = Gi[fg][ft + 4];
      const double di0 = Dib[2 * ft], di1 = Dib[2 * ft + 1];
      constexpr int FB = (WIN / 8 + FWD_WARPS - 1) / FWD_WARPS;  // row blocks per forward warp
      double a0[FB], a1[FB], c0[FB], c1[FB];
#pragma unroll
      for (int u = 0; u < FB; u++) {
        const int wi = 8 * (warp + u * FWD_WARPS) + fg;
        const bool valid = warp + u * FWD_WARPS < nblk && wi <= nr;
        const int rowoff = (wi >= nr) ? ZR_OFF : (wmod(r0 + wi)) * WIN_P;
        a0[u] = (valid && ft < nb) ? A[rowoff + wmod(k0 + ft)] : 0.0;
        a1[u] = (valid && ft + 4 < nb) ? A[rowoff + wmod(k0 + ft + 4)] : 0.0;
        c0[u] = 0.0; c1[u] = 0.0;
      }
#pragma unroll
      for (int u = 0; u < FB; u++)
        if (warp + u * FWD_WARPS < nblk) mma2(c0[u], c1[u], a0[u], a1[u], g0, g1);
#pragma unroll
      for (int u = 0; u < FB; u++) {
        if (warp + u * FWD_WARPS >= nblk) continue;
        const int wi = 8 * (warp + u * FWD_WARPS) + fg;
        const double l0 = c0[u] * di0, l1 = c1[u] * di1;   // columns >= nb: c = 0 (a = 0 there and G is triangular)
        Lt[(2 * ft) * WIN_LP + wi] = l0; Lt[(2 * ft + 1) * WIN_LP + wi] = l1;
        LDt[(2 * ft) * WIN_LP + wi] = c0[u]; LDt[(2 * ft + 1) * WIN_LP + wi] = c1[u];
        if (wi <= nr) {
          double* dst = M + (size_t)(wi == nr ? n : r0 + wi) * n + k0 + 2 * ft;
          if (2 * ft + 1 < nb) *reinterpret_cast<double2*>(dst) = make_double2(l0, l1);  // n even, k0 % 8 == 0: 16-byte aligned
          else if (2 * ft < nb) dst[0] = l0;
        }
      }
    }
    if (warp >= FWD_WARPS) {
      commit_row();  // the row of panel p+1 fetched one panel ago
      if (warp == FWD_WARPS) pivot_store(p);
      if (more) {
        const int lo1 = max(R, pre) + 1 + LD_WARPS;  // rows beyond one per loader warp: directly
        if (lo1 <= rlast[p + 1]) load_rows(lo1, rlast[p + 1], r0, FWD_WARPS, LD_WARPS);
        if (p + 2 < pend) {
          const int i = new_rows_lo(p + 2) + (warp - FWD_WARPS);
          if (i <= rlast[p + 2]) prefetch_row(i, r0 + WPB);
        }
      }
    }
    __syncthreads();
    // ---- (B) rank-nb update of the window on the tensor pipe, with look-ahead: warp 0 updates the tile that
    //      holds the NEXT pivot block first and then factors it (one thread) while the other warps update the
    //      rest of the window
    {
      const int T8 = (nr + 1 + 7) >> 3;
      const int ntile = T8 * (T8 + 1) / 2;
      // warp 0 shares its scheduler with warps 4, 8, 12: they take what is left after the other twelve warps got
      // seven tiles each (a 96-row window: 90 tiles = 12 x 7 + 3 x 2), so the pivot chain issues almost alone
      if (warp == 0) {
        if (pre > R) load_rows(R + 1, pre, r0, 0, 1);
        update_tile0(r0, nr);
        __syncwarp();
        if (tid == 0 && more) pivot(p + 1);
        if (more) pivot_inverse();
      } else {
        const int T = ntile - 1;
        const int light = T / 22, heavy = (T - 3 * light + 11) / 12;
        int tb, te;
        if (warp & 3) { tb = 1 + (warp - 1 - (warp >> 2)) * heavy; te = tb + heavy; }
        else { const int rest = max(T - 12 * heavy, 0), per = (rest + 2) / 3; tb = 1 + 12 * heavy + ((warp >> 2) - 1) * per; te = tb + per; }
        update_run(min(tb, ntile), min(te, ntile), r0, nr);
      }
    }
    __syncthreads();
  }
  // ---- L^T x = z (z = row n of M, already scaled by 1/D), 8 unknowns per step, four warps, one named barrier per
  //      step.  With G = L_bb^-T (the inverse of the step's unit-triangular pivot block) the step is
  //        x_b = G acc_b,   acc_j -= sum_c P[j][c] acc_b[c],   P = L_panel^T G,
  //      so the chain from one step to the next is: read acc_b, 8 multiply-adds, write acc_j, barrier.  A warp
  //      issues roughly one instruction every four cycles here (one warp per scheduler, dependent code), so the
  //      step is as fast as its instruction count: the inverses of all pivot blocks and the window start of every
  //      block are formed up front (one thread per block, staged in the dead ring), x_b = G acc_b is evaluated for
  //      all blocks after the loop (acc_b is final once its step is done), the rows of L are fetched two steps
  //      ahead through a running pointer and turned into the thread's row of P while it waits.
  if (mode == 1) {
    // the window that is left: rows [ks, R] x columns [ks, row] of the ring (entries left of a row's envelope were
    // zeroed when the row came in) and their rhs entries -- the separator block with this side's update applied
    const int ks = pend * WPB, R = rlast[pend - 1], wd = sd.esep - sd.ksep;
    for (int i = ks + warp; i <= R; i += WIN_THREADS / 32) {
      const double* Ai = A + wmod(i) * WIN_P;
      for (int j = ks + lane; j <= i; j += 32) sd.dump[(size_t)(i - ks) * wd + (j - ks)] = Ai[wmod(j)];
    }
    for (int j = ks + tid; j <= R; j += WIN_THREADS) sd.dump[(size_t)wd * wd + (j - ks)] = zr[wmod(j)];
    return;
  }
  // mode 2: columns >= ksep are solved (the separator, xs) or belong to the other side (zero here): their blocks
  // enter the loop below with an identity pivot block and only update columns < ksep
  const int ksep = mode == 2 ? sd.ksep : n, esep = mode == 2 ? sd.esep : n;
  double* acc = A;            // [n]
  double* pblk = A + n;       // [npan][28]: Linv[c][r], r < c, at c(c-1)/2 + r   (n + 29 npan <= WIN * WIN_P: host-checked)
  int* jmb = reinterpret_cast<int*>(pblk + (size_t)npan * 28);  // [npan] first column of the block's row window
  for (int i = tid; i < n; i += WIN_THREADS) {
    double v = 0.0;
    if (i < ksep) v = M[(size_t)n * n + i];
    else if (i < esep) v = wa.xs[(blockIdx.x ? n - 1 - i : i) - wa.msep];  // side 1 counts from the other end
    acc[i] = v;
  }
  for (int bq = tid; bq < npan; bq += WIN_THREADS) {
    const int k0 = bq * WPB, nb = min(WPB, n - k0);
    int jmv = k0;
    for (int r = 0; r < nb; r++) jmv = min(jmv, first[k0 + r]);
    double Lq[WPB][WPB], Li[WPB][WPB];
#pragma unroll
    for (int c = 1; c < WPB; c++)
#pragma unroll
      for (int r = 0; r < c; r++) Lq[c][r] = (k0 + c < n && k0 < ksep) ? M[(size_t)(k0 + c) * n + k0 + r] : 0.0;
    // inverse of the unit lower triangle, row by row: Li[c][r] = -(L[c][r] + sum_{r<m<c} L[c][m] Li[m][r])
#pragma unroll
    for (int c = 1; c < WPB; c++)
#pragma unroll
      for (int r = 0; r < c; r++) {
        double t = Lq[c][r];
#pragma unroll
        for (int m = r + 1; m < c; m++) t += Lq[c][m] * Li[m][r];
        Li[c][r] = -t;
      }
#pragma unroll
    for (int c = 1; c < WPB; c++)
#pragma unroll
      for (int r = 0; r < c; r++) pblk[bq * 28 + c * (c - 1) / 2 + r] = Li[c][r];
    jmb[bq] = jmv;  // (after the reads of `first`: jmb may alias nothing, it lives in the ring)
  }
  __syncthreads();
  constexpr int BS_THREADS = WIN;  // one thread per window column (WIN_ROWS < WIN)
  if (tid < BS_THREADS) {
    double Pc[WPB];
    double* bsr = reinterpret_cast<double*>(jmb + ((npan + 1) & ~1));  // [4][WPB][WIN]: rows of L, four blocks in flight
    auto fetch = [&](int bq) {
      const int k0 = bq * WPB, nb = min(WPB, n - k0), j = jmb[bq] + tid;
      const double* src = M + (size_t)k0 * n + j;
      double* dst = bsr + (bq & 3) * (WPB * WIN) + tid;
#pragma unroll
      for (int r = 0; r < WPB; r++) {
        const bool valid = r < nb && j < min(k0, ksep);
        cp_async8(dst + r * WIN, valid ? src + (size_t)r * n : M, valid);
      }
      cp_async_commit();
    };
    // P[j][c] = sum_{r <= c} L[k0+r][j] G[r][c],  G[r][c] = Linv[c][r], G[c][c] = 1
    auto transform = [&](int bq) {
      const double* pb = pblk + bq * 28;
      const double* rp = bsr + (bq & 3) * (WPB * WIN) + tid;
      double rows[WPB];
#pragma unroll
      for (int r = 0; r < WPB; r++) rows[r] = rp[r * WIN];
#pragma unroll
      for (int c = 0; c < WPB; c++) {
        double t = rows[c];
#pragma unroll
        for (int r = 0; r < c; r++) t += rows[r] * pb[c * (c - 1) / 2 + r];
        Pc[c] = t;
      }
    };
    const int b0 = (esep + WPB - 1) / WPB - 1;  // = npan - 1 unless the blocks beyond the separator are skipped
    fetch(b0);
    if (b0 > 0) fetch(b0 - 1); else cp_async_commit();
    cp_async_wait<1>();
    transform(b0);
    if (b0 > 1) fetch(b0 - 2); else cp_async_commit();
    for (int bq = b0; bq >= 0; bq--) {
      const int k0 = bq * WPB;
      const int j = jmb[bq] + tid;
      // ---- the chain (only the last block can be short: its missing slots read as zero)
      if (j < min(k0, ksep)) {
        double ab[WPB];
#pragma unroll
        for (int c = 0; c < WPB; c++) ab[c] = (k0 + c < n) ? acc[k0 + c] : 0.0;
        const double s0 = Pc[0] * ab[0] + Pc[1] * ab[1] + Pc[2] * ab[2] + Pc[3] * ab[3];
        const double s1 = Pc[4] * ab[4] + Pc[5] * ab[5] + Pc[6] * ab[6] + Pc[7] * ab[7];
        acc[j] -= s0 + s1;
      }
      // ---- off the chain: the next step's row of P (its rows arrived two steps ago), the copies of the step after
      //      the next.  One group is committed per step so that wait_group counts steps.
      if (bq > 0) {
        cp_async_wait<1>();
        transform(bq - 1);
        if (bq > 2) fetch(bq - 3); else cp_async_commit();
      }
      asm volatile("bar.sync 1, %0;" ::"n"(BS_THREADS) : "memory");
    }
    cp_async_wait<0>();
  }
  __syncthreads();
  // x_b = G acc_b for every block at once: G[r][c] = Linv[c][r] (c > r), 1 on the diagonal
  for (int i = tid; i < ksep; i += WIN_THREADS) {
    const int bq = i / WPB, r = i - bq * WPB, k0 = bq * WPB, nb = min(WPB, n - k0);
    const double* pb = pblk + bq * 28;
    double xv = acc[i];
    for (int c = r + 1; c < nb; c++) xv += pb[c * (c - 1) / 2 + r] * acc[k0 + c];
    x[blockIdx.x ? n - 1 - i : i] = xv;
  }
  if (mode == 2 && blockIdx.x == 0)
    for (int i = ksep + tid; i < esep; i += WIN_THREADS) x[i] = wa.xs[i - ksep];
}

// ---- two-sided reduced solve ("burn at both ends")
// The pivot chain of ldlt_win_kernel is sequential, but an envelope matrix can be eliminated from both ends at once:
// the first m columns top-down by one CTA, the last n - e columns bottom-up by a second CTA (= top-down on the matrix
// with rows and columns in reverse order, P S P), where [m, e) -- the separator -- is wide enough that no row >= e
// reaches a column < m.  Each side leaves its Schur update of the separator block; the updates add up, the separator
// (a dense block of <= WIN_ROWS - 8 unknowns) is factored and solved by one CTA, and the two sides back-substitute
// in parallel.  Same arithmetic per pivot as the one-sided kernel, half the chain; the order of the operations is
// fixed, so a solve stays bitwise reproducible.
//
// rev_gather_kernel: side 1's matrix M1 = P S P inside its (monotone) row envelope first1, rows [0, e1); the
// separator block and the separator's rhs entries start from zero there, so that side 1's window ends up holding
// only its update (-Delta_B).  One CTA per row of M1 (+ one for the rhs row).
__global__ void __launch_bounds__(128) rev_gather_kernel(const double* __restrict__ S, double* __restrict__ M1, int n,
                                                         const int* __restrict__ first1, int m1, int e1) {
  const int a = blockIdx.x;
  if (a == e1) {  // rhs row
    for (int b = threadIdx.x; b < e1; b += 128) M1[(size_t)n * n + b] = b >= m1 ? 0.0 : S[(size_t)n * n + (n - 1 - b)];
    return;
  }
  const int j = n - 1 - a;
  for (int b = first1[a] + threadIdx.x; b <= a; b += 128) {
    const int i = n - 1 - b;  // i >= j: S[i][j] is a lower-triangle entry
    M1[(size_t)a * n + b] = (a >= m1 && b >= m1) ? 0.0 : S[(size_t)i * n + j];
  }
}
// sep_merge_kernel: the separator system (w unknowns, dense lower triangle + rhs row, row pitch w) =
// side 0's window (S - Delta_T on rows <= R0, the untouched S below) + side 1's window (-Delta_B, in reversed
// numbering, rows <= R1).  One CTA per separator row (+ one for the rhs).
__global__ void __launch_bounds__(128) sep_merge_kernel(const double* __restrict__ S, int n, int m, int w, int R0, int m1, int R1,
                                                        const double* __restrict__ dump0, const double* __restrict__ dump1,
                                                        double* __restrict__ Msep) {
  const int si = blockIdx.x;
  if (si == w) {
    for (int t = threadIdx.x; t < w; t += 128) {
      const int i = m + t, a = n - 1 - i;
      double v = i <= R0 ? dump0[(size_t)w * w + t] : S[(size_t)n * n + i];
      if (a <= R1) v += dump1[(size_t)w * w + (a - m1)];
      Msep[(size_t)w * w + t] = v;
    }
    return;
  }
  const int i = m + si;
  for (int sj = threadIdx.x; sj <= si; sj += 128) {
    const int j = m + sj;
    double v = i <= R0 ? dump0[(size_t)si * w + sj] : S[(size_t)i * n + j];
    const int a = n - 1 - j, b = n - 1 - i;  // the same entry in side 1's numbering (a >= b)
    if (a <= R1) v += dump1[(size_t)(a - m1) * w + (b - m1)];
    Msep[(size_t)si * w + sj] = v;
  }
}

// x_l = D^-1 (b_l - W^T x_p); scale terms x.(lambda x + b); backup + update points.
__global__ void __launch_bounds__(128) lm_update_points_kernel(LbaDev D, double lambda) {
  const int l = blockIdx.x * 128 + threadIdx.x;
  if (l >= D.n_mp) return;
  const double* b = D.bl + 3 * (size_t)l;
  double c[3] = {b[0], b[1], b[2]};
  for (int e = D.lm_ptr[l]; e < D.lm_ptr[l + 1]; e++) {
    const int f = D.e_free[e];
    if (f < 0) continue;
    const double* We = D.W + 18 * (size_t)e;
    const double* xp = D.x + 6 * (size_t)f;
#pragma unroll
    for (int i = 0; i < 6; i++) {
      c[0] -= We[i * 3] * xp[i]; c[1] -= We[i * 3 + 1] * xp[i]; c[2] -= We[i * 3 + 2] * xp[i];
    }
  }
  const double* Di = D.Dinv + 9 * (size_t)l;
  double sc = 0;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const double xl = Di[i * 3] * c[0] + Di[i * 3 + 1] * c[1] + Di[i * 3 + 2] * c[2];
    D.x[(size_t)D.n + 3 * (size_t)l + i] = xl;
    sc += xl * (lambda * xl + b[i]);
    const double old = D.pts[3 * (size_t)l + i];
    D.pts_bak[3 * (size_t)l + i] = old;
    D.pts[3 * (size_t)l + i] = old + xl;
  }
  D.scale_part[D.n_free + l] = sc;
}

// VertexSE3Expmap::oplusImpl: T <- exp(delta) * T   (se3quat.h:223-257)
__global__ void __launch_bounds__(64) lm_update_poses_kernel(LbaDev D, double lambda) {
  const int f = blockIdx.x * 64 + threadIdx.x;
  if (f >= D.n_free) return;
  const int k = D.free_kf[f];
  double* P = D.pose + 7 * (size_t)k;
  double* Pb = D.pose_bak + 7 * (size_t)k;
  const double* u = D.x + 6 * (size_t)f;
  double sc = 0;
  for (int i = 0; i < 6; i++) sc += u[i] * (lambda * u[i] + D.bp[6 * (size_t)f + i]);
  D.scale_part[f] = sc;
  for (int i = 0; i < 7; i++) Pb[i] = P[i];
  const double w0 = u[0], w1 = u[1], w2 = u[2];
  const double theta = sqrt(w0 * w0 + w1 * w1 + w2 * w2);
  const double Om[9] = {0, -w2, w1, w2, 0, -w0, -w1, w0, 0};
  double Om2[9];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) Om2[i * 3 + j] = Om[i * 3] * Om[j] + Om[i * 3 + 1] * Om[3 + j] + Om[i * 3 + 2] * Om[6 + j];
  double R[9], V[9];
  if (theta < 0.00001) {
    for (int i = 0; i < 9; i++) { R[i] = ((i % 4 == 0) ? 1.0 : 0.0) + Om[i] + Om2[i]; V[i] = R[i]; }
  } else {
    const double a = sin(theta) / theta, b = (1 - cos(theta)) / (theta * theta);
    const double c = (theta - sin(theta)) / pow(theta, 3.0);
    for (int i = 0; i < 9; i++) {
      const double I = (i % 4 == 0) ? 1.0 : 0.0;
      R[i] = I + a * Om[i] + b * Om2[i];
      V[i] = I + b * Om[i] + c * Om2[i];
    }
  }
  DQuat qe = R_to_q(R);
  q_normalize(qe);
  double te[3];
  for (int i = 0; i < 3; i++) te[i] = V[i * 3] * u[3] + V[i * 3 + 1] * u[4] + V[i * 3 + 2] * u[5];
  DQuat q0 = {P[0], P[1], P[2], P[3]};
  const double t0[3] = {P[4], P[5], P[6]};
  double rt[3];
  q_rot(qe, t0, rt);
  DQuat qn = q_mul(qe, q0);
  q_normalize(qn);
  P[0] = qn.x; P[1] = qn.y; P[2] = qn.z; P[3] = qn.w;
  P[4] = te[0] + rt[0]; P[5] = te[1] + rt[1]; P[6] = te[2] + rt[2];
}

__global__ void restore_kernel(LbaDev D) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 3 * D.n_mp) D.pts[i] = D.pts_bak[i];
  if (i < D.n_free * 7) {
    const int k = D.free_kf[i / 7];
    D.pose[7 * (size_t)k + i % 7] = D.pose_bak[7 * (size_t)k + i % 7];
  }
}

__global__ void normalize_poses_kernel(LbaDev D) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= D.n_kf) return;
  double* P = D.pose + 7 * (size_t)k;
  DQuat q = {P[0], P[1], P[2], P[3]};
  q_normalize(q);  // SE3Quat(q, t) constructor (Optimizer.cc:1217)
  P[0] = q.x; P[1] = q.y; P[2] = q.z; P[3] = q.w;
}

__global__ void depth_kernel(LbaDev D, uint8_t* out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= D.n_edges) return;
  const int l = D.e_free[D.n_edges + e];
  const double* P = D.pose + 7 * (size_t)D.e_kf[e];
  DQuat q = {P[0], P[1], P[2], P[3]};
  double Xc[3];
  if (D.kf_trl && D.e_stereo[e] == LBA_EDGE_BODY) {  // OptimizableTypes.h:135-139: depth in the second camera
    DQuat qrw; double trw[3];
    body_pose(D, D.e_kf[e], q, P + 4, qrw, trw);
    q_rot(qrw, D.pts + 3 * (size_t)l, Xc);
    out[e] = (Xc[2] + trw[2]) > 0.0;
    return;
  }
  q_rot(q, D.pts + 3 * (size_t)l, Xc);
  out[e] = (Xc[2] + P[6]) > 0.0;
}

// ------------------------------------------------------------------- fp64 tensor-pipe peak (measurement)
// The denominator of the Schur roofline (SURVEY.md 8d: "record the fp64 peak measured the same way" as
// MEASURED_PEAKS.json): every warp of a full grid issues independent DMMA m8n8k4 chains from registers, best of
// `reps` launches between CUDA events.  2 * 8 * 8 * 4 = 512 flop per instruction.
__global__ void __launch_bounds__(256) dmma_peak_kernel(double* out, int iters) {
  double c[8][2];
#pragma unroll
  for (int i = 0; i < 8; i++) { c[i][0] = 0.0; c[i][1] = 0.0; }
  const double a = 1.0 + 1e-9 * threadIdx.x, b = 1.0 - 1e-9 * threadIdx.x;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 8; i++)
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                   : "+d"(c[i][0]), "+d"(c[i][1])
                   : "d"(a), "d"(b));
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) s += c[i][0] + c[i][1];
  if (s == 12345.678) out[0] = s;  // keep the chains alive
}

int measure_fp64_mma_peak(int device, int reps, double* tflops_out) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_last_error("no CUDA device: orb_slam3_b200 has no CPU path");
    return ORB_E_NODEVICE;
  }
  CUDA_TRYL(cudaSetDevice(device));
  int sms = 0;
  CUDA_TRYL(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  double* d = nullptr;
  CUDA_TRYL(cudaMalloc(&d, 64));
  cudaEvent_t e0, e1;
  CUDA_TRYL(cudaEventCreate(&e0));
  CUDA_TRYL(cudaEventCreate(&e1));
  const int iters = 20000, grid = sms * 8;
  double best = 0;
  for (int r = 0; r < reps + 2; r++) {
    cudaEventRecord(e0);
    dmma_peak_kernel<<<grid, 256>>>(d, iters);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    const double tf = 512.0 * 8 * iters * (256 / 32) * (double)grid / (ms * 1e-3) / 1e12;
    if (r >= 2) best = std::max(best, tf);
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
  CUDA_TRYL(cudaGetLastError());
  *tflops_out = best;
  return 0;
}

// ------------------------------------------------------------------- NCCL (dlopen)
struct Uid { char internal[128]; };
struct Nccl {
  void* lib = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, /*ncclUniqueId by value*/ Uid, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
static Nccl g_nccl;

static int nccl_load() {
  if (g_nccl.lib) return 0;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* nm : names) {
    g_nccl.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (g_nccl.lib) break;
  }
  if (!g_nccl.lib) { set_last_error(std::string("dlopen libnccl.so.2: ") + dlerror()); return ORB_E_NCCL; }
  *(void**)&g_nccl.GetUniqueId = dlsym(g_nccl.lib, "ncclGetUniqueId");
  *(void**)&g_nccl.CommInitRank = dlsym(g_nccl.lib, "ncclCommInitRank");
  *(void**)&g_nccl.AllReduce = dlsym(g_nccl.lib, "ncclAllReduce");
  *(void**)&g_nccl.CommDestroy = dlsym(g_nccl.lib, "ncclCommDestroy");
  *(void**)&g_nccl.GetErrorString = dlsym(g_nccl.lib, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce) {
    set_last_error("libnccl: missing symbols");
    return ORB_E_NCCL;
  }
  return 0;
}

// ------------------------------------------------------------------- solver
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes) {
    if (bytes <= cap) return 0;
    if (p) cudaFree(p);
    p = nullptr;
    cap = bytes + bytes / 8 + 256;
    CUDA_TRYL(cudaMalloc(&p, cap));
    return 0;
  }
};

struct Solver {
  int device = 0;
  bool initialized = false;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[8];
  DevBuf graph, work;
  // Host side of the structure build: the landmark-sorted edge arrays and the pair lists (tens of MB at config 5) are
  // written straight into one persistent pinned block -- fresh std::vectors cost a page fault per 4 KB on every call
  // and their cudaMemcpyAsync goes through the driver's pageable staging path.
  uint8_t* pin_base = nullptr;
  size_t pin_cap = 0, pin_off = 0;
  int pin_reserve(size_t bytes) {
    pin_off = 0;
    if (bytes <= pin_cap) return 0;
    if (pin_base) cudaFreeHost(pin_base);
    pin_base = nullptr; pin_cap = 0;
    const size_t want = bytes + bytes / 4;
    if (cudaHostAlloc((void**)&pin_base, want, cudaHostAllocDefault) != cudaSuccess) {
      set_last_error("lba_solve: cudaHostAlloc of the structure arena");
      return ORB_E_CUDA;
    }
    pin_cap = want;
    return 0;
  }
  template <class T>
  T* pin_take(size_t count) {
    T* r = (T*)(pin_base + pin_off);
    pin_off += (count * sizeof(T) + 255) & ~(size_t)255;
    return r;
  }
  double* h_scalars = nullptr;  // pinned
  unsigned* d_bar = nullptr;
  int sm_count = 0, ldlt_blocks = 0;
  long long launches = 0;
  void* comm = nullptr;
  int rank = 0, world = 1;

  int init() {
    if (initialized) return 0;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
      set_last_error("no CUDA device: orb_slam3_b200 has no CPU path");
      return ORB_E_NODEVICE;
    }
    CUDA_TRYL(cudaSetDevice(device));
    CUDA_TRYL(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    for (auto& e : ev) CUDA_TRYL(cudaEventCreate(&e));
    CUDA_TRYL(cudaHostAlloc((void**)&h_scalars, 8 * sizeof(double), cudaHostAllocDefault));
    CUDA_TRYL(cudaMalloc((void**)&d_bar, 256));
    cudaDeviceProp prop;
    CUDA_TRYL(cudaGetDeviceProperties(&prop, device));
    sm_count = prop.multiProcessorCount;
    int per_sm = 0;
    CUDA_TRYL(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ldlt_kernel, 256, 0));
    ldlt_blocks = sm_count * std::max(1, std::min(per_sm, 1));
    initialized = true;
    return 0;
  }
  ~Solver() {
    if (!initialized) return;
    cudaSetDevice(device);
    if (comm && g_nccl.CommDestroy) g_nccl.CommDestroy(comm);
    if (graph.p) cudaFree(graph.p);
    if (work.p) cudaFree(work.p);
    cudaFreeHost(h_scalars);
    if (pin_base) cudaFreeHost(pin_base);
    cudaFree(d_bar);
    for (auto& e : ev) cudaEventDestroy(e);
    cudaStreamDestroy(stream);
  }
};

template <class T>
struct PinView {  // the slice of Solver's pinned arena that stands in for a std::vector
  T* p; size_t n;
  T& operator[](size_t i) { return p[i]; }
  const T& operator[](size_t i) const { return p[i]; }
  T* data() { return p; }
  size_t size() const { return n; }
};

template <class T>
static T* carve(uint8_t*& p, size_t count) {
  T* r = (T*)p;
  p += (count * sizeof(T) + 255) & ~(size_t)255;
  return r;
}

static int solve_impl(Solver& S, const lba_graph_view* g, const volatile uint8_t* stop, int max_iters,
                      double lambda_init, double* kf_pose_out, double* mp_pos_out, double* chi2_out,
                      uint8_t* depth_pos_out, lba_stats* stats) {
  if (!g || !kf_pose_out || !mp_pos_out || g->n_kf <= 0 || g->n_mp < 0 || g->n_edges < 0) {
    set_last_error("lba_solve: bad argument");
    return ORB_E_ARG;
  }
  int rc = S.init();
  if (rc) return rc;
  CUDA_TRYL(cudaSetDevice(S.device));
  const int K = g->n_kf, L = g->n_mp, E = g->n_edges;
  // ---- structure (host): free poses, landmark CSR, pose CSR, pose-pair lists
  const auto t_host0 = std::chrono::steady_clock::now();
  // The analogue of g2o's buildStructure (block_solver.hpp:143-295), rebuilt for every call because every local
  // window is a new graph.  The passes over the landmarks (pattern / pair counts, edge gather, pair fill) run on
  // PREP_T host threads over contiguous landmark ranges; every list keeps ascending landmark order, so the result
  // does not depend on the thread count.
  constexpr int PREP_T = 8;
  auto parallel = [&](auto&& fn) {
    std::vector<std::thread> th;
    for (int t = 1; t < PREP_T; t++) th.emplace_back([&, t] { fn(t); });
    fn(0);
    for (auto& x : th) x.join();
  };
  std::vector<int> nat_idx(K, -1), nat_kf;  // free poses in the caller's order
  for (int k = 0; k < K; k++)
    if (!g->kf_fixed[k]) { nat_idx[k] = (int)nat_kf.size(); nat_kf.push_back(k); }
  const int nf = (int)nat_kf.size(), n = 6 * nf;
  if (nf == 0) { set_last_error("lba_solve: no free keyframe"); return ORB_E_ARG; }
  std::vector<int> lm_ptr(L + 1, 0);
  bool any_body = false;
  for (int e = 0; e < E; e++) {
    if (g->e_mp[e] < 0 || g->e_mp[e] >= L || g->e_kf[e] < 0 || g->e_kf[e] >= K) { set_last_error("edge index"); return ORB_E_ARG; }
    if (g->e_stereo[e] > LBA_EDGE_BODY) { set_last_error("lba_solve: unknown edge type"); return ORB_E_ARG; }
    any_body |= g->e_stereo[e] == LBA_EDGE_BODY;
    lm_ptr[g->e_mp[e] + 1]++;
  }
  // rig extension of the view: KannalaBrandt8 cameras and / or second-camera (EdgeSE3ProjectXYZToBody) edges take the
  // general-camera instantiations of the edge kernels; plain Pinhole windows keep the specialised ones
  bool any_kb8 = false;
  for (int k = 0; k < K && g->kf_cam_model; k++) any_kb8 |= g->kf_cam_model[k] == ORB_CAM_KB8;
  if (any_kb8 && !g->kf_cam_dist) { set_last_error("lba_solve: kf_cam_model names a KannalaBrandt8 camera but kf_cam_dist is NULL"); return ORB_E_ARG; }
  if (any_body && (!g->kf_cam2 || !g->kf_trl)) { set_last_error("lba_solve: LBA_EDGE_BODY edges need kf_cam2 and kf_trl"); return ORB_E_ARG; }
  for (int k = 0; k < K; k++)
    if ((g->kf_cam_model && g->kf_cam_model[k] > ORB_CAM_KB8) || (any_body && g->kf_cam2_model && g->kf_cam2_model[k] > ORB_CAM_KB8)) {
      set_last_error("lba_solve: unknown camera model"); return ORB_E_ARG;
    }
  const bool rig = any_kb8 || any_body;
  for (int l = 0; l < L; l++) lm_ptr[l + 1] += lm_ptr[l];
  std::vector<int> perm(E), cursor(lm_ptr.begin(), lm_ptr.end() - 1);
  for (int e = 0; e < E; e++) perm[cursor[g->e_mp[e]]++] = e;   // sorted position -> original edge
  int lm_lo[PREP_T + 1];  // landmark ranges with about the same number of edges
  {
    lm_lo[0] = 0;
    for (int t = 1; t <= PREP_T; t++) {
      const long long want = (long long)E * t / PREP_T;
      lm_lo[t] = t == PREP_T ? L : (int)(std::lower_bound(lm_ptr.begin(), lm_ptr.end(), (int)want) - lm_ptr.begin());
      lm_lo[t] = std::min(std::max(lm_lo[t], lm_lo[t - 1]), L);
    }
  }
  // ---- pass A: per thread, how often every unordered pair of free poses shares a landmark (caller's numbering;
  //      a pose pairs with itself once per edge), and the useful Schur flops
  const size_t nf2 = (size_t)nf * nf;
  std::vector<std::vector<int>> cntT(PREP_T, std::vector<int>(nf2, 0));
  double flopsT[PREP_T];
  parallel([&](int t) {
    std::vector<int>& cnt = cntT[t];
    std::vector<int> fl;
    double fsum = 0;
    for (int l = lm_lo[t]; l < lm_lo[t + 1]; l++) {
      fl.clear();
      for (int s = lm_ptr[l]; s < lm_ptr[l + 1]; s++) {
        const int f = nat_idx[g->e_kf[perm[s]]];
        if (f >= 0) fl.push_back(f);
      }
      const double m = (double)fl.size();
      fsum += 50 + m * (108 + 36) + m * (m + 1) / 2 * 216;
      // two edges of one landmark on the SAME pose (left + right camera of a rig) contribute both cross terms
      // Y_a W_b^T and Y_b W_a^T to the pose's diagonal block (g2o adds both edges into one H_pl block)
      for (size_t a = 0; a < fl.size(); a++)
        for (size_t b = a; b < fl.size(); b++)
          cnt[(size_t)std::min(fl[a], fl[b]) * nf + std::max(fl[a], fl[b])] += (a != b && fl[a] == fl[b]) ? 2 : 1;
    }
    flopsT[t] = fsum;
  });
  double schur_flops = 0;
  for (int t = 0; t < PREP_T; t++) schur_flops += flopsT[t];
  std::vector<int> tot(nf2, 0);
  for (int t = 0; t < PREP_T; t++)
    for (size_t i = 0; i < nf2; i++) tot[i] += cntT[t][i];
  // covisibility pattern of the free poses (block pattern of S); with landmark shards every rank only sees
  // its own landmarks, so the patterns are OR-ed over the ranks: ordering, envelope and the choice of the
  // solver kernel must be identical everywhere (all ranks factor the same matrix)
  std::vector<uint8_t> adj(nf2, 0);
  for (int a = 0; a < nf; a++) {
    adj[(size_t)a * nf + a] = 1;
    for (int b = a + 1; b < nf; b++)
      if (tot[(size_t)a * nf + b]) adj[(size_t)a * nf + b] = adj[(size_t)b * nf + a] = 1;
  }
  if (S.world > 1) {
    if (S.graph.reserve(adj.size() + 256)) return ORB_E_CUDA;
    CUDA_TRYL(cudaMemcpyAsync(S.graph.p, adj.data(), adj.size(), cudaMemcpyHostToDevice, S.stream));
    const int r = g_nccl.AllReduce(S.graph.p, S.graph.p, adj.size(), /*ncclUint8*/ 1, /*ncclMax*/ 2, S.comm, S.stream);
    if (r) { set_last_error("ncclAllReduce(covisibility pattern)"); return ORB_E_NCCL; }
    CUDA_TRYL(cudaMemcpyAsync(adj.data(), S.graph.p, adj.size(), cudaMemcpyDeviceToHost, S.stream));
    CUDA_TRYL(cudaStreamSynchronize(S.stream));
  }
  // Elimination order of the free poses.  The envelope solver's cost is the profile of S, so when the
  // caller's keyframe order is not already chain-like (Optimizer.cc:1135-1160 lists the current keyframe
  // first, then its covisibles) the poses are renumbered by reverse Cuthill-McKee on the covisibility
  // pattern; the natural order is kept when it is at least as good (what Eigen's AMD ordering does for g2o).
  std::vector<int> pos(nf);  // pos[natural free index] = free index used from here on
  for (int i = 0; i < nf; i++) pos[i] = i;
  if (nf > 2) {
    auto profile = [&](const std::vector<int>& q) {  // q[f] = position of pose f
      long long p = 0;
      std::vector<int> lo(nf);
      for (int i = 0; i < nf; i++) lo[i] = i;
      for (int a = 0; a < nf; a++)
        for (int b = 0; b < nf; b++)
          if (adj[(size_t)a * nf + b] && q[b] < q[a]) lo[q[a]] = std::min(lo[q[a]], q[b]);
      for (int i = 0; i < nf; i++) p += i - lo[i] + 1;
      return p;
    };
    std::vector<int> deg(nf, 0), order, rpos(nf, -1);
    for (int a = 0; a < nf; a++)
      for (int b = 0; b < nf; b++) deg[a] += adj[(size_t)a * nf + b] && a != b;
    std::vector<uint8_t> seen(nf, 0);
    while ((int)order.size() < nf) {
      int start = -1;  // lowest-degree unvisited node of the next component
      for (int a = 0; a < nf; a++)
        if (!seen[a] && (start < 0 || deg[a] < deg[start])) start = a;
      seen[start] = 1;
      size_t head = order.size();
      order.push_back(start);
      while (head < order.size()) {
        const int a = order[head++];
        std::vector<int> nb;
        for (int b = 0; b < nf; b++)
          if (adj[(size_t)a * nf + b] && !seen[b]) { nb.push_back(b); seen[b] = 1; }
        std::stable_sort(nb.begin(), nb.end(), [&](int x, int y) { return deg[x] < deg[y]; });
        order.insert(order.end(), nb.begin(), nb.end());
      }
    }
    std::reverse(order.begin(), order.end());
    for (int i = 0; i < nf; i++) rpos[order[i]] = i;
    if (profile(rpos) * 10 < profile(pos) * 9) {  // renumber only for a >= 10 % smaller profile
      pos = rpos;
      std::vector<uint8_t> adj2(nf2, 0);  // the pattern in the new numbering
      for (int a = 0; a < nf; a++)
        for (int b = 0; b < nf; b++)
          if (adj[(size_t)a * nf + b]) adj2[(size_t)pos[a] * nf + pos[b]] = 1;
      adj.swap(adj2);
    }
  }
  std::vector<int> free_idx(K, -1), free_kf(nf);
  for (int i = 0; i < nf; i++) { free_kf[pos[i]] = nat_kf[i]; free_idx[nat_kf[i]] = pos[i]; }
  // ---- pose pairs (i1 <= i2 in the final numbering): slots, list offsets, per-thread fill cursors
  std::vector<int> pair_i1, pair_i2, pair_ptr(1, 0);
  std::vector<int> inv(nf);
  for (int i = 0; i < nf; i++) inv[pos[i]] = i;
  auto nat_key = [&](int i1, int i2) {  // final (i1, i2) -> index into the caller-numbered count tables
    const int a = inv[i1], b = inv[i2];
    return (size_t)std::min(a, b) * nf + std::max(a, b);
  };
  std::vector<int> slot_of(nf2, -1);  // by caller-numbered key
  for (int a = 0; a < nf; a++)
    for (int b = a; b < nf; b++) {
      const size_t key = nat_key(a, b);
      const int c = tot[key];
      if (c == 0 && a != b) continue;
      slot_of[key] = (int)pair_i1.size();
      pair_i1.push_back(a); pair_i2.push_back(b);
      pair_ptr.push_back(pair_ptr.back() + c);
    }
  const int n_pairs = (int)pair_i1.size();
  // cntT[t][key] <- first list position thread t writes for that pair (prefix over the threads)
  {
    std::vector<int> run(nf2, 0);
    for (size_t key = 0; key < nf2; key++)
      if (slot_of[key] >= 0) run[key] = pair_ptr[slot_of[key]];
    for (int t = 0; t < PREP_T; t++)
      for (size_t key = 0; key < nf2; key++) {
        const int c = cntT[t][key];
        cntT[t][key] = run[key];
        run[key] += c;
      }
  }
  // ---- pass B: edge gather (landmark-sorted arrays), pose CSR counts and the pair lists
  const size_t n_pair_entries = (size_t)pair_ptr.back();
  if (S.pin_reserve(256 * 8 + (size_t)E * (4 + 8 + 1 + 24 + 4 + 4) + 8 * n_pair_entries)) return ORB_E_CUDA;
  PinView<int> se_kf{S.pin_take<int>(E), (size_t)E}, se_free{S.pin_take<int>(2 * (size_t)E), 2 * (size_t)E};
  PinView<uint8_t> se_st{S.pin_take<uint8_t>(E), (size_t)E};
  PinView<double> se_obs{S.pin_take<double>(3 * (size_t)E), 3 * (size_t)E};
  PinView<float> se_is2{S.pin_take<float>(E), (size_t)E};
  PinView<int> pair_ea{S.pin_take<int>(n_pair_entries), n_pair_entries}, pair_eb{S.pin_take<int>(n_pair_entries), n_pair_entries};
  std::vector<std::vector<int>> poseT(PREP_T, std::vector<int>(nf, 0));
  parallel([&](int t) {
    std::vector<int>& cur = cntT[t];
    std::vector<int>& pc = poseT[t];
    std::vector<int> tmp;
    for (int l = lm_lo[t]; l < lm_lo[t + 1]; l++) {
      tmp.clear();
      for (int s = lm_ptr[l]; s < lm_ptr[l + 1]; s++) {
        const int e = perm[s];
        se_kf[s] = g->e_kf[e];
        se_free[s] = free_idx[g->e_kf[e]];
        se_free[(size_t)E + s] = g->e_mp[e];
        se_st[s] = g->e_stereo[e];
        memcpy(&se_obs[3 * (size_t)s], g->e_obs + 3 * (size_t)e, 3 * sizeof(double));
        se_is2[s] = g->e_inv_sigma2[e];
        if (se_free[s] >= 0) { pc[se_free[s]]++; tmp.push_back(s); }
      }
      for (size_t a = 0; a < tmp.size(); a++)
        for (size_t b = a; b < tmp.size(); b++) {
          const int fa = se_free[tmp[a]], fb = se_free[tmp[b]];
          const int p2 = cur[nat_key(std::min(fa, fb), std::max(fa, fb))]++;
          pair_ea[p2] = fa <= fb ? tmp[a] : tmp[b];
          pair_eb[p2] = fa <= fb ? tmp[b] : tmp[a];
          if (a != b && fa == fb) {  // same pose twice: the transposed cross term as well (see pass A)
            const int p3 = cur[nat_key(fa, fa)]++;
            pair_ea[p3] = tmp[b];
            pair_eb[p3] = tmp[a];
          }
        }
    }
  });
  std::vector<int> pose_ptr(nf + 1, 0);
  for (int f = 0; f < nf; f++) {
    int c = 0;
    for (int t = 0; t < PREP_T; t++) { const int v = poseT[t][f]; poseT[t][f] = c; c += v; }  // -> per-thread offsets
    pose_ptr[f + 1] = pose_ptr[f] + c;
  }
  PinView<int> pose_edges{S.pin_take<int>((size_t)pose_ptr[nf]), (size_t)pose_ptr[nf]};  // <= E entries (reserved above)
  parallel([&](int t) {
    std::vector<int>& off = poseT[t];
    for (int s = lm_ptr[lm_lo[t]]; s < lm_ptr[lm_lo[t + 1]]; s++)
      if (se_free[s] >= 0) pose_edges[pose_ptr[se_free[s]] + off[se_free[s]]++] = s;
  });
  // ---- row envelope of S (scalar rows): first[i] = first non-zero column, reach[c] = last row whose
  //      envelope holds a column <= c; feasibility / cost of the single-CTA envelope solver
  std::vector<int> env_first(n), env_reach(n, 0);
  {
    std::vector<int> bfirst(nf);
    for (int i = 0; i < nf; i++) {
      bfirst[i] = i;
      for (int j = 0; j < i; j++)
        if (adj[(size_t)i * nf + j]) { bfirst[i] = j; break; }
    }
    for (int i = 0; i < n; i++) env_first[i] = 6 * bfirst[i / 6];
    for (int i = 0; i < n; i++) env_reach[env_first[i]] = std::max(env_reach[env_first[i]], i);
    for (int c = 1; c < n; c++) env_reach[c] = std::max(env_reach[c], env_reach[c - 1]);
  }
  std::vector<long long> env_rowp(n + 2, 0);
  for (int i = 0; i < n; i++) env_rowp[i + 1] = env_rowp[i] + (i - env_first[i] + 1);
  env_rowp[n + 1] = env_rowp[n] + n;
  const size_t env_total = (size_t)env_rowp[n + 1];
  int sky_rows_max = 0;
  double sky_flops = 0;
  for (int k0 = 0; k0 < n; k0 += NB) {
    const int nb = std::min(NB, n - k0), r0 = k0 + nb;
    const int rend = std::min(std::max(env_reach[k0 + nb - 1] + 1, r0), n);
    const int nw = rend - r0 + 1;
    int jmin = k0;
    for (int r = 0; r < nb; r++) jmin = std::min(jmin, env_first[k0 + r]);
    sky_rows_max = std::max(sky_rows_max, std::max(nw, k0 - jmin));
    sky_flops += (double)nw * nw * nb;
  }
  int win_rows_max = 0;  // 8-column panels of the window-resident kernel
  for (int k0 = 0; k0 < n; k0 += WPB) {
    const int nb = std::min(WPB, n - k0);
    const int R = std::min(std::max(env_reach[k0 + nb - 1], k0 + nb - 1), n - 1);
    int jmin = k0;
    for (int r = 0; r < nb; r++) jmin = std::min(jmin, env_first[k0 + r]);
    win_rows_max = std::max(win_rows_max, std::max(R - k0 + 1, k0 - jmin + nb));
  }
  // envelope tables (4.5 bytes per unknown) share the shared memory; the back-substitution keeps n + 29 n / 8 + 4096 doubles in the ring
  const bool win_ok = win_rows_max <= WIN_ROWS && n <= 2600;
  static const char* ldlt_env = getenv("ORB_B200_LDLT");  // "dense" | "sky" | "win" | unset = automatic
  bool use_sky = sky_rows_max <= SKY_WMAX - 4 && n <= 32 * SKY_WMAX && sky_flops <= 6.0e7;
  if (ldlt_env && !strcmp(ldlt_env, "dense")) use_sky = false;
  if (ldlt_env && !strcmp(ldlt_env, "sky")) use_sky = sky_rows_max <= SKY_WMAX - 4 && n <= 32 * SKY_WMAX;
  bool use_win = win_ok && !(ldlt_env && (!strcmp(ldlt_env, "sky") || !strcmp(ldlt_env, "dense")));
  // ---- two-sided plan (see rev_gather_kernel): side 0 eliminates the panels [0, ts_p0), side 1 -- in reversed
  //      numbering -- the panels [0, ts_p1) = the last 8 ts_p1 columns; separator [ts_m, ts_e2).  ORB_B200_LDLT=win
  //      pins the one-sided kernel, =win2 takes the two-sided one whenever a separator exists; automatic: from 50
  //      panels on (the separator's own dense factorisation and the four extra launches cost about 15 panels).
  bool use_two = false;
  int ts_m = 0, ts_e2 = 0, ts_p0 = 0, ts_p1 = 0, ts_w = 0, ts_R0 = 0, ts_R1 = 0;
  std::vector<int> first1, reach1;
  if (use_win && !(ldlt_env && !strcmp(ldlt_env, "win")) && ((ldlt_env && !strcmp(ldlt_env, "win2")) || n >= 50 * WPB)) {
    TwoSidedPlan plan = plan_two_sided(n, env_reach, WPB, WIN_ROWS);  // csrc/ldlt_plan.h (held on the CPU by tests/test_ldlt_plan.py)
    if (plan.ok) {
      use_two = true;
      ts_m = plan.m; ts_e2 = plan.e2; ts_p0 = plan.p0; ts_p1 = plan.p1; ts_w = plan.w; ts_R0 = plan.R0; ts_R1 = plan.R1;
      first1.swap(plan.first1); reach1.swap(plan.reach1);
    }
  }
  // ---- device memory
  size_t gbytes = 256 * 24 + sizeof(int) * 2 * (size_t)n + sizeof(long long) * ((size_t)n + 2) + sizeof(int) * ((size_t)L + 1 + 3 * (size_t)E + nf + (nf + 1) + pose_edges.size() +
                                            2 * (size_t)n_pairs + pair_ptr.size() + 2 * pair_ea.size()) +
                  (size_t)E * (1 + 24 + 4) + (size_t)K * 20 + (rig ? 256 * 4 + (size_t)K * (1 + 16 + 32 + 56) : 0) +
                  (use_two ? 256 * 4 + sizeof(int) * (2 * (size_t)n + 2 * (size_t)ts_w) : 0);
  if (S.graph.reserve(gbytes)) return ORB_E_CUDA;
  uint8_t* gp = (uint8_t*)S.graph.p;
  LbaDev D;
  memset(&D, 0, sizeof(D));
  D.n_kf = K; D.n_free = nf; D.n_mp = L; D.n_edges = E; D.n = n; D.n_pairs = n_pairs;
  cudaStream_t st = S.stream;
#define UPLOAD(field, type, vec, count)                                                              \
  do {                                                                                               \
    type* dptr = carve<type>(gp, std::max<size_t>(count, 1));                                        \
    if ((count) > 0) CUDA_TRYL(cudaMemcpyAsync(dptr, (vec), sizeof(type) * (count), cudaMemcpyHostToDevice, st)); \
    D.field = dptr;                                                                                  \
  } while (0)
  UPLOAD(lm_ptr, int, lm_ptr.data(), (size_t)L + 1);
  UPLOAD(e_kf, int, se_kf.data(), (size_t)E);
  UPLOAD(e_free, int, se_free.data(), 2 * (size_t)E);
  UPLOAD(e_stereo, uint8_t, se_st.data(), (size_t)E);
  UPLOAD(e_obs, double, se_obs.data(), 3 * (size_t)E);
  UPLOAD(e_is2, float, se_is2.data(), (size_t)E);
  UPLOAD(kf_cam, float, g->kf_cam, 5 * (size_t)K);
  std::vector<uint8_t> model;  // (function scope: the copies below are asynchronous)
  std::vector<float> dist, cam2;
  std::vector<double> trl;
  if (rig) {
    model.assign(K, 0);
    dist.assign(4 * (size_t)K, 0.f); cam2.assign(8 * (size_t)K, 0.f);
    trl.assign(7 * (size_t)K, 0.0);
    for (int k = 0; k < K; k++) {
      if (g->kf_cam_model && g->kf_cam_model[k] == ORB_CAM_KB8) { model[k] |= 1; memcpy(&dist[4 * (size_t)k], g->kf_cam_dist + 4 * (size_t)k, 16); }
      if (any_body) {
        if (g->kf_cam2_model && g->kf_cam2_model[k] == ORB_CAM_KB8) model[k] |= 2;
        memcpy(&cam2[8 * (size_t)k], g->kf_cam2 + 8 * (size_t)k, 32);
        memcpy(&trl[7 * (size_t)k], g->kf_trl + 7 * (size_t)k, 56);
      } else trl[7 * (size_t)k + 3] = 1.0;
    }
    UPLOAD(kf_model, uint8_t, model.data(), (size_t)K);
    UPLOAD(kf_dist, float, dist.data(), 4 * (size_t)K);
    UPLOAD(kf_cam2, float, cam2.data(), 8 * (size_t)K);
    UPLOAD(kf_trl, double, trl.data(), 7 * (size_t)K);
  }
  UPLOAD(free_kf, int, free_kf.data(), (size_t)nf);
  UPLOAD(pose_ptr, int, pose_ptr.data(), (size_t)nf + 1);
  UPLOAD(pose_edges, int, pose_edges.data(), pose_edges.size());
  UPLOAD(pair_i1, int, pair_i1.data(), (size_t)n_pairs);
  UPLOAD(pair_i2, int, pair_i2.data(), (size_t)n_pairs);
  UPLOAD(pair_ptr, int, pair_ptr.data(), pair_ptr.size());
  UPLOAD(pair_ea, int, pair_ea.data(), pair_ea.size());
  UPLOAD(pair_eb, int, pair_eb.data(), pair_eb.size());
  const int *d_env_first = nullptr, *d_env_reach = nullptr;
  {
    int* dptr = carve<int>(gp, (size_t)n);
    CUDA_TRYL(cudaMemcpyAsync(dptr, env_first.data(), sizeof(int) * n, cudaMemcpyHostToDevice, st));
    d_env_first = dptr;
    dptr = carve<int>(gp, (size_t)n);
    CUDA_TRYL(cudaMemcpyAsync(dptr, env_reach.data(), sizeof(int) * n, cudaMemcpyHostToDevice, st));
    d_env_reach = dptr;
  }
  const int *d_first1 = nullptr, *d_reach1 = nullptr, *d_sep_first = nullptr, *d_sep_reach = nullptr;
  std::vector<int> sep_first, sep_reach;
  if (use_two) {
    sep_first.assign(ts_w, 0); sep_reach.assign(ts_w, ts_w - 1);  // the separator block is dense
    int* dptr = carve<int>(gp, (size_t)n);
    CUDA_TRYL(cudaMemcpyAsync(dptr, first1.data(), sizeof(int) * n, cudaMemcpyHostToDevice, st));
    d_first1 = dptr;
    dptr = carve<int>(gp, (size_t)n);
    CUDA_TRYL(cudaMemcpyAsync(dptr, reach1.data(), sizeof(int) * n, cudaMemcpyHostToDevice, st));
    d_reach1 = dptr;
    dptr = carve<int>(gp, (size_t)ts_w);
    CUDA_TRYL(cudaMemcpyAsync(dptr, sep_first.data(), sizeof(int) * ts_w, cudaMemcpyHostToDevice, st));
    d_sep_first = dptr;
    dptr = carve<int>(gp, (size_t)ts_w);
    CUDA_TRYL(cudaMemcpyAsync(dptr, sep_reach.data(), sizeof(int) * ts_w, cudaMemcpyHostToDevice, st));
    d_sep_reach = dptr;
  }
  const long long* d_env_rowp = nullptr;
  {
    long long* dptr = carve<long long>(gp, (size_t)n + 2);
    CUDA_TRYL(cudaMemcpyAsync(dptr, env_rowp.data(), sizeof(long long) * (n + 2), cudaMemcpyHostToDevice, st));
    d_env_rowp = dptr;
  }
#undef UPLOAD
  const size_t nS = (size_t)(n + 1) * n;
  size_t wbytes = 256 * 32 + sizeof(double) * (14 * (size_t)K + 6 * (size_t)L + (size_t)L * (6 + 3 + 9 + 3 + 1) +
                                               (size_t)E * (18 + 18 + HPE_STRIDE + 6 + 1) + (size_t)nf * 42 + nS + (S.world > 1 ? env_total : 1) +
                                               (size_t)n + 3 * (size_t)L + (size_t)nf + L + 16) + (size_t)E +
                  (use_two ? 256 * 5 + sizeof(double) * (nS + 3 * ((size_t)ts_w + 1) * ts_w + WIN) : 0) +
                  256 + sizeof(double) * (LMC_STRIDE * (size_t)E + 2);
  if (S.work.reserve(wbytes)) return ORB_E_CUDA;
  uint8_t* wp = (uint8_t*)S.work.p;
  D.pose = carve<double>(wp, 7 * (size_t)K); D.pose_bak = carve<double>(wp, 7 * (size_t)K);
  D.pts = carve<double>(wp, 3 * (size_t)L + 1); D.pts_bak = carve<double>(wp, 3 * (size_t)L + 1);
  D.Hll = carve<double>(wp, 6 * (size_t)L + 1); D.bl = carve<double>(wp, 3 * (size_t)L + 1);
  D.Dinv = carve<double>(wp, 9 * (size_t)L + 1); D.db = carve<double>(wp, 3 * (size_t)L + 1);
  D.chi_lm = carve<double>(wp, (size_t)L + 1);
  D.W = carve<double>(wp, 18 * (size_t)E + 1); D.Y = carve<double>(wp, 18 * (size_t)E + 1);
  D.Hpp_e = carve<double>(wp, HPE_STRIDE * (size_t)E + 2); D.bp_e = carve<double>(wp, 6 * (size_t)E + 1);
  D.chi2_e = carve<double>(wp, (size_t)E + 1);
  D.Hpp = carve<double>(wp, 36 * (size_t)nf); D.bp = carve<double>(wp, 6 * (size_t)nf);
  D.S = carve<double>(wp, nS);
  double* d_env_pack = carve<double>(wp, S.world > 1 ? env_total : 1);
  D.x = carve<double>(wp, (size_t)n + 3 * (size_t)L + 1);
  D.scale_part = carve<double>(wp, (size_t)nf + L + 1);
  D.scalars = carve<double>(wp, 16);
  uint8_t* d_depth = carve<uint8_t>(wp, (size_t)E + 1);
  double* d_lmc = carve<double>(wp, LMC_STRIDE * (size_t)E + 2);  // per-edge landmark-block records of lin_edge_kernel
  double *d_M1 = nullptr, *d_dump0 = nullptr, *d_dump1 = nullptr, *d_Msep = nullptr, *d_xs = nullptr;
  if (use_two) {
    d_M1 = carve<double>(wp, nS);
    d_dump0 = carve<double>(wp, ((size_t)ts_w + 1) * ts_w); d_dump1 = carve<double>(wp, ((size_t)ts_w + 1) * ts_w);
    d_Msep = carve<double>(wp, ((size_t)ts_w + 1) * ts_w);
    d_xs = carve<double>(wp, WIN);
    // outside its envelope the reversed matrix is never written: zero once per solve (its back-substitution reads
    // whole 8-row blocks from the leftmost envelope start of the block)
    CUDA_TRYL(cudaMemsetAsync(d_M1, 0, sizeof(double) * nS, st));
  }
  const float thm = (float)sqrt(5.991), ths = (float)sqrt(7.815);  // Optimizer.cc:1275-1276
  D.hm.delta = thm; D.hm.dsqr = (double)(float)((double)thm * (double)thm);
  D.hs.delta = ths; D.hs.dsqr = (double)(float)((double)ths * (double)ths);
  CUDA_TRYL(cudaMemcpyAsync(D.pose, g->kf_pose, sizeof(double) * 7 * (size_t)K, cudaMemcpyHostToDevice, st));
  if (L) CUDA_TRYL(cudaMemcpyAsync(D.pts, g->mp_pos, sizeof(double) * 3 * (size_t)L, cudaMemcpyHostToDevice, st));
  CUDA_TRYL(cudaMemsetAsync(D.chi2_e, 0, sizeof(double) * ((size_t)E + 1), st));
  CUDA_TRYL(cudaMemsetAsync(D.x, 0, sizeof(double) * ((size_t)n + 3 * (size_t)L + 1), st));
  CUDA_TRYL(cudaMemsetAsync(D.scalars, 0, sizeof(double) * 16, st));
  CUDA_TRYL(cudaMemsetAsync(D.W, 0, sizeof(double) * (18 * (size_t)E + 1), st));
  const double ms_host_prep = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_host0).count();
  if (S.world > 1) {
    // The ranks finish their host-side structure build (and the uploads queued above) at different times; the first
    // collective of the solve would make the early ones wait, and that wait would be booked as device time of the
    // first linearisation (measured: ms_linearize grew from 1.28 ms on two GPUs to 1.63 ms on four).  One tiny
    // all-reduce + synchronisation lines the ranks up before the timed region starts; the wait is part of ms_wall.
    CUDA_TRYL(cudaMemsetAsync(D.scalars + 8, 0, sizeof(double), st));
    int r = g_nccl.AllReduce(D.scalars + 8, D.scalars + 8, 1, /*ncclFloat64*/ 8, /*ncclSum*/ 0, S.comm, st);
    if (r) { set_last_error("ncclAllReduce(start barrier)"); return ORB_E_NCCL; }
    CUDA_TRYL(cudaStreamSynchronize(st));
  }
  CUDA_TRYL(cudaEventRecord(S.ev[0], st));
  normalize_poses_kernel<<<(K + 127) / 128, 128, 0, st>>>(D);
  S.launches++;

  const int lm_blocks = (L + 127) / 128;
  auto terminate = [&]() { return stop && *stop; };
  auto allreduce = [&](double* buf, size_t count) -> int {
    if (S.world <= 1) return 0;
    int r = g_nccl.AllReduce(buf, buf, count, /*ncclFloat64*/ 8, /*ncclSum*/ 0, S.comm, st);
    if (r != 0) { set_last_error(std::string("ncclAllReduce: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?")); return ORB_E_NCCL; }
    return 0;
  };
  // chi (robust) of the current state -> h_scalars[0]; all ranks see the global value
  auto eval_chi = [&](bool linearize) -> int {
    // rig: KannalaBrandt8 cameras / second-camera edges take the general-camera instantiations
    if (L) {
      if (linearize) {  // one thread per edge + a per-landmark gather
        if (rig) lin_edge_kernel<true><<<(E + 127) / 128, 128, 0, st>>>(D, d_lmc);
        else lin_edge_kernel<false><<<(E + 127) / 128, 128, 0, st>>>(D, d_lmc);
        lm_gather_kernel<<<lm_blocks, 128, 0, st>>>(D, d_lmc);
        S.launches += 1;
      } else if (rig) chi_kernel<true><<<lm_blocks, 128, 0, st>>>(D);
      else chi_kernel<false><<<lm_blocks, 128, 0, st>>>(D);
    }
    reduce_kernel<<<1, 1024, 0, st>>>(D.chi_lm, L, D.scalars);
    S.launches += 2;
    return 0;
  };
  double lambda = -1, ni = 2, chi_first = 0, currentChi = 0;
  int nBad = 0, trials = 0, iters = 0;
  float ms_lin = 0, ms_schur = 0, ms_solve = 0, ms_upd = 0;
  bool lin_pending = false;
  auto lap = [&](int a, int b, float& acc) {
    float t = 0;
    if (cudaEventElapsedTime(&t, S.ev[a], S.ev[b]) == cudaSuccess) acc += t;
  };
  for (int it = 0; it < max_iters && !terminate(); it++) {
    CUDA_TRYL(cudaEventRecord(S.ev[1], st));
    eval_chi(true);
    pose_reduce_kernel<<<nf, POSE_THREADS, 0, st>>>(D);
    S.launches++;
    // From the second iteration on the host already knows the robust chi2 of this state: it is the chi2 of the trial
    // that was just accepted (or, after a rejected trial, of the restored state) -- g2o's activeRobustChi2() at the top
    // of an iteration (optimization_algorithm_levenberg.cpp:69-70) re-evaluates the same edges at the same estimates.
    // No read-back, no stream synchronisation and no all-reduce there: the linearisation is queued behind the trial.
    const bool need_chi = it == 0;
    if (need_chi && S.world > 1 && (rc = allreduce(D.scalars, 1))) return rc;  // global robust chi2
    if (it == 0 && !(lambda_init > 0)) {
      // computeLambdaInit: max |diag| over all free vertices of the *global* Hessian
      if (S.world == 1) {
        maxdiag_kernel<<<1, 1024, 0, st>>>(D, D.Hpp, 1, D.scalars + 2);
      } else {
        maxdiag_kernel<<<1, 1024, 0, st>>>(D, nullptr, 1, D.scalars + 2);
        int r = g_nccl.AllReduce(D.scalars + 2, D.scalars + 2, 1, 8, /*ncclMax*/ 2, S.comm, st);
        if (r) { set_last_error("ncclAllReduce(max)"); return ORB_E_NCCL; }
        CUDA_TRYL(cudaMemcpyAsync(D.S, D.Hpp, sizeof(double) * 36 * (size_t)nf, cudaMemcpyDeviceToDevice, st));
        if ((rc = allreduce(D.S, 36 * (size_t)nf))) return rc;
        maxdiag_kernel<<<1, 1024, 0, st>>>(D, D.S, 0, D.scalars + 4);
      }
      S.launches++;
    }
    CUDA_TRYL(cudaEventRecord(S.ev[2], st));
    if (need_chi) {
      CUDA_TRYL(cudaMemcpyAsync(S.h_scalars, D.scalars, 5 * sizeof(double), cudaMemcpyDeviceToHost, st));
      CUDA_TRYL(cudaStreamSynchronize(st));
      lap(1, 2, ms_lin);
      currentChi = S.h_scalars[0];
    } else {
      lin_pending = true;  // ev[1] -> ev[2] is read after the trial's synchronisation
    }
    double tempChi = currentChi;
    const double iniChi = currentChi;
    if (it == 0) {
      chi_first = currentChi;
      if (lambda_init > 0) lambda = lambda_init;
      else lambda = 1e-5 * std::max(S.h_scalars[2], S.world > 1 ? S.h_scalars[4] : 0.0);  // tau = 1e-5
      ni = 2; nBad = 0;
    }
    double rho = 0;
    int qmax = 0;
    do {
      CUDA_TRYL(cudaEventRecord(S.ev[3], st));
      // Schur complement
      CUDA_TRYL(cudaMemsetAsync(D.S, 0, sizeof(double) * nS, st));
      if (L) {
        lm_prepare_kernel<<<lm_blocks, 128, 0, st>>>(D, lambda);
        y_edge_kernel<<<(E + 127) / 128, 128, 0, st>>>(D);
        S.launches += 1;
      }
      schur_pairs_kernel<<<n_pairs, 256, 0, st>>>(D);
      bschur_kernel<<<nf, POSE_THREADS, 0, st>>>(D);
      S.launches += 3;
      // landmark shards: every rank holds its partial H_pp, b_p and Schur terms; one sum gives (S | b_s)
      if (S.world > 1) {
        env_pack_kernel<<<n + 1, 256, 0, st>>>(D.S, n, d_env_first, d_env_rowp, d_env_pack, 0);
        if ((rc = allreduce(d_env_pack, env_total))) return rc;
        env_pack_kernel<<<n + 1, 256, 0, st>>>(D.S, n, d_env_first, d_env_rowp, d_env_pack, 1);
        S.launches += 2;
      }
      add_lambda_kernel<<<(n + 255) / 256, 256, 0, st>>>(D, lambda);
      CUDA_TRYL(cudaEventRecord(S.ev[4], st));
      // reduced solve
      CUDA_TRYL(cudaMemsetAsync(S.d_bar, 0, 256, st));
      CUDA_TRYL(cudaMemsetAsync(D.scalars + 3, 0, sizeof(double), st));
      if (use_win) {
        const size_t smem = sizeof(double) * (WIN * WIN_P + WIN + 2 * WPB * WIN_LP + (WIN_THREADS / 32 - WIN / 32) * (WIN + 8)) +
                            sizeof(int) * ((size_t)n + (n + WPB - 1) / WPB + 4);
        const void* kfn = (const void*)ldlt_win_kernel;
        CUDA_TRYL(raise_dynamic_smem(kfn, smem, S.device));
        WinArgs wa;
        memset(&wa, 0, sizeof(wa));
        wa.fail = D.scalars + 3;
        void* args[] = {&wa};
        if (!use_two) {
          wa.s[0] = WinSide{D.S, d_env_reach, d_env_first, nullptr, n, 0, 0, 0};
          wa.x = D.x; wa.mode = 0;
          CUDA_TRYL(cudaLaunchKernel(kfn, dim3(1), dim3(WIN_THREADS), args, smem, st));
          S.launches += 1;
        } else {
          const int m1 = WPB * ts_p1, e1 = n - ts_m;
          rev_gather_kernel<<<e1 + 1, 128, 0, st>>>(D.S, d_M1, n, d_first1, m1, e1);
          wa.s[0] = WinSide{D.S, d_env_reach, d_env_first, d_dump0, n, ts_p0, ts_m, ts_e2};
          wa.s[1] = WinSide{d_M1, d_reach1, d_first1, d_dump1, n, ts_p1, m1, e1};
          wa.mode = 1;
          CUDA_TRYL(cudaLaunchKernel(kfn, dim3(2), dim3(WIN_THREADS), args, smem, st));
          sep_merge_kernel<<<ts_w + 1, 128, 0, st>>>(D.S, n, ts_m, ts_w, ts_R0, m1, ts_R1, d_dump0, d_dump1, d_Msep);
          WinArgs ws;
          memset(&ws, 0, sizeof(ws));
          ws.fail = D.scalars + 3; ws.mode = 0; ws.x = d_xs;
          ws.s[0] = WinSide{d_Msep, d_sep_reach, d_sep_first, nullptr, ts_w, 0, 0, 0};
          void* sargs[] = {&ws};
          CUDA_TRYL(cudaLaunchKernel(kfn, dim3(1), dim3(WIN_THREADS), sargs, smem, st));
          wa.mode = 2; wa.xs = d_xs; wa.x = D.x; wa.msep = ts_m;
          CUDA_TRYL(cudaLaunchKernel(kfn, dim3(2), dim3(WIN_THREADS), args, smem, st));
          S.launches += 5;
        }
      } else if (use_sky) {
        const size_t smem = sizeof(double) * 2 * 32 * SKY_WMAX;
        CUDA_TRYL(raise_dynamic_smem((const void*)ldlt_sky_kernel, smem, S.device));
        ldlt_sky_kernel<<<1, SKY_THREADS, smem, st>>>(D.S, n, d_env_reach, d_env_first, D.scalars + 3, D.x);
        S.launches += 1;
      } else {
        double* Mp = D.S;
        int nn = n;
        unsigned* bar = S.d_bar;
        double* failp = D.scalars + 3;
        void* args[] = {&Mp, &nn, &bar, &failp};
        const int blocks = std::min(S.ldlt_blocks, std::max(1, (n + 1 + NB - 1) / NB * ((n + 1 + NB - 1) / NB)));
        CUDA_TRYL(cudaLaunchCooperativeKernel((void*)ldlt_kernel, dim3(blocks), dim3(256), args, 0, st));
        backsub_kernel<<<1, 1024, sizeof(double) * n, st>>>(D.S, n, D.x);
        S.launches += 2;
      }
      S.launches += 1;
      CUDA_TRYL(cudaEventRecord(S.ev[5], st));
      // update + evaluate
      if (L) lm_update_points_kernel<<<lm_blocks, 128, 0, st>>>(D, lambda);
      lm_update_poses_kernel<<<(nf + 63) / 64, 64, 0, st>>>(D, S.rank == 0 ? lambda : 0.0);
      eval_chi(false);
      reduce_kernel<<<1, 1024, 0, st>>>(D.scale_part, nf + L, D.scalars + 1);
      S.launches += 3;
      if (S.world > 1) {
        if ((rc = allreduce(D.scalars, 2))) return rc;
      }
      CUDA_TRYL(cudaMemcpyAsync(S.h_scalars, D.scalars, 4 * sizeof(double), cudaMemcpyDeviceToHost, st));
      CUDA_TRYL(cudaEventRecord(S.ev[6], st));
      CUDA_TRYL(cudaStreamSynchronize(st));
      if (lin_pending) { lap(1, 2, ms_lin); lin_pending = false; }
      lap(3, 4, ms_schur); lap(4, 5, ms_solve); lap(5, 6, ms_upd);
      const bool ok2 = S.h_scalars[3] == 0.0;
      tempChi = S.h_scalars[0];
      if (!ok2) tempChi = DBL_MAX;
      rho = currentChi - tempChi;
      double scale = S.h_scalars[1];
      scale += 1e-3;
      rho /= scale;
      if (rho > 0 && std::isfinite(tempChi)) {
        double alpha = 1. - pow((2 * rho - 1), 3);
        alpha = std::min(alpha, 2. / 3.);
        const double scaleFactor = std::max(1. / 3., alpha);
        lambda *= scaleFactor;
        ni = 2;
        currentChi = tempChi;
      } else {
        lambda *= ni;
        ni *= 2;
        restore_kernel<<<(std::max(3 * L, 7 * nf) + 255) / 256, 256, 0, st>>>(D);  // pop
        S.launches++;
      }
      qmax++;
      trials++;
    } while (rho < 0 && qmax < 10 && !terminate());
    iters++;
    if (qmax == 10 || rho == 0) break;
    if ((iniChi - currentChi) * 1e3 < iniChi) nBad++;
    else nBad = 0;
    if (nBad >= 3) break;
  }
  // ---- outputs
  if (E) depth_kernel<<<(E + 255) / 256, 256, 0, st>>>(D, d_depth);
  S.launches++;
  CUDA_TRYL(cudaEventRecord(S.ev[7], st));
  std::vector<double> chi_sorted(E);
  std::vector<uint8_t> dep_sorted(E);
  CUDA_TRYL(cudaMemcpyAsync(kf_pose_out, D.pose, sizeof(double) * 7 * (size_t)K, cudaMemcpyDeviceToHost, st));
  if (L) CUDA_TRYL(cudaMemcpyAsync(mp_pos_out, D.pts, sizeof(double) * 3 * (size_t)L, cudaMemcpyDeviceToHost, st));
  if (E) {
    CUDA_TRYL(cudaMemcpyAsync(chi_sorted.data(), D.chi2_e, sizeof(double) * E, cudaMemcpyDeviceToHost, st));
    CUDA_TRYL(cudaMemcpyAsync(dep_sorted.data(), d_depth, E, cudaMemcpyDeviceToHost, st));
  }
  CUDA_TRYL(cudaStreamSynchronize(st));
  for (int s = 0; s < E; s++) {
    if (chi2_out) chi2_out[perm[s]] = chi_sorted[s];
    if (depth_pos_out) depth_pos_out[perm[s]] = dep_sorted[s];
  }
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    stats->iterations = iters; stats->trials = trials; stats->stopped = terminate() ? 1 : 0;
    stats->chi2_initial = chi_first; stats->chi2_final = currentChi; stats->lambda_final = lambda;
    float tot = 0;
    cudaEventElapsedTime(&tot, S.ev[0], S.ev[7]);
    stats->ms_total = tot; stats->ms_linearize = ms_lin; stats->ms_schur = ms_schur; stats->ms_solve = ms_solve;
    stats->ms_update = ms_upd; stats->n_free_kf = nf; stats->n_pairs = n_pairs; stats->schur_flops = schur_flops;
    stats->solver_kind = use_win ? (use_two ? 3 : 2) : (use_sky ? 1 : 0); stats->envelope_rows_max = use_win ? win_rows_max : sky_rows_max;
    stats->ms_host_prep = ms_host_prep;
    stats->ms_wall = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_host0).count();
    stats->allreduce_bytes_per_trial = S.world > 1 ? (double)env_total * sizeof(double) : 0.0;
  }
  return iters;
}

}  // namespace orbb200

using orbb200::Solver;
struct lba_solver { Solver s; };

extern "C" {

int lba_create(int device, lba_solver** out) {
  if (!out || device < 0) return ORB_E_ARG;
  *out = new lba_solver();
  (*out)->s.device = device;
  return ORB_OK;
}
void lba_destroy(lba_solver* s) { delete s; }

int lba_nccl_unique_id(void* out128) {
  if (!out128) return ORB_E_ARG;
  int rc = orbb200::nccl_load();
  if (rc) return rc;
  orbb200::Uid id;
  memset(&id, 0, sizeof(id));
  if (orbb200::g_nccl.GetUniqueId(&id) != 0) { orbb200::set_last_error("ncclGetUniqueId failed"); return ORB_E_NCCL; }
  memcpy(out128, &id, 128);
  return ORB_OK;
}

int lba_comm_init(lba_solver* s, int rank, int world, const void* unique_id128) {
  if (!s || !unique_id128 || world < 1 || rank < 0 || rank >= world) return ORB_E_ARG;
  int rc = s->s.init();
  if (rc) return rc;
  if (world == 1) { s->s.rank = 0; s->s.world = 1; return ORB_OK; }
  rc = orbb200::nccl_load();
  if (rc) return rc;
  cudaSetDevice(s->s.device);
  orbb200::Uid id;
  memcpy(&id, unique_id128, 128);
  void* comm = nullptr;
  int r = orbb200::g_nccl.CommInitRank(&comm, world, id, rank);
  if (r != 0) {
    orbb200::set_last_error(std::string("ncclCommInitRank: ") +
                            (orbb200::g_nccl.GetErrorString ? orbb200::g_nccl.GetErrorString(r) : "?"));
    return ORB_E_NCCL;
  }
  s->s.comm = comm; s->s.rank = rank; s->s.world = world;
  return ORB_OK;
}

int lba_solve(lba_solver* s, const lba_graph_view* g, const volatile uint8_t* stop, int max_iters,
              double lambda_init, double* kf_pose_out, double* mp_pos_out, double* chi2_out,
              uint8_t* depth_pos_out, lba_stats* stats) {
  if (!s) return ORB_E_ARG;
  return orbb200::solve_impl(s->s, g, stop, max_iters, lambda_init, kf_pose_out, mp_pos_out, chi2_out,
                             depth_pos_out, stats);
}

long long lba_kernel_launches(const lba_solver* s) { return s ? s->s.launches : 0; }

// Host-only: the two-sided plan for a row envelope (env_reach as lba_solve builds it), for the CPU test of the scheme.
int lba_debug_two_sided_plan(int n, const int* env_reach, int* out9, int* first1_out, int* reach1_out) {
  if (n <= 0 || !env_reach || !out9) { orbb200::set_last_error("lba_debug_two_sided_plan: bad argument"); return ORB_E_ARG; }
  const std::vector<int> reach(env_reach, env_reach + n);
  const orbb200::TwoSidedPlan P = orbb200::plan_two_sided(n, reach, orbb200::WPB, orbb200::WIN_ROWS);
  const int o[9] = {P.ok ? 1 : 0, P.m, P.e2, P.p0, P.p1, P.w, P.R0, P.R1, orbb200::WIN_ROWS};
  memcpy(out9, o, sizeof(o));
  if (first1_out) memcpy(first1_out, P.first1.data(), sizeof(int) * n);
  if (reach1_out) memcpy(reach1_out, P.reach1.data(), sizeof(int) * n);
  return ORB_OK;
}

int lba_measure_fp64_mma_peak(int device, int reps, double* tflops_out) {
  if (!tflops_out || reps < 1) return ORB_E_ARG;
  return orbb200::measure_fp64_mma_peak(device, reps, tflops_out);
}

}  // extern "C"
