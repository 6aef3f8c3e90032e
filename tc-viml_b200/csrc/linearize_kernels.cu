// linearize_kernels.cu — residual/Jacobian evaluation of ProjectionFactor and LineProjectionFactor,
// loss correction, J^T J / J^T r assembly and the landmark Schur complement, for batches of windows.
//
// Reference semantics (paths relative to /root/reference/vins_estimator/src):
//   factor/projection_factor.cpp:21-124, factor/line_projection_factor.cpp:19-120,
//   factor/marginalization_factor.cpp:37-68 (loss), :141-172 (ThreadsConstructA), :267-282 (Schur).
// The arithmetic is re-organised for the GPU (shared sub-products, reciprocal instead of repeated
// division, FMA); parity with the oracle is to 1e-9 relative, not bit-exact.
#include <cstdlib>
#include <vector>

#include "common.cuh"

namespace {

__device__ __forceinline__ void quat_to_rot(double w, double x, double y, double z, double* R) {
  const double tx = 2.0 * x, ty = 2.0 * y, tz = 2.0 * z;
  const double twx = tx * w, twy = ty * w, twz = tz * w;
  const double txx = tx * x, txy = ty * x, txz = tz * x;
  const double tyy = ty * y, tyz = tz * y, tzz = tz * z;
  R[0] = 1.0 - (tyy + tzz);
  R[1] = txy - twz;
  R[2] = txz + twy;
  R[3] = txy + twz;
  R[4] = 1.0 - (txx + tzz);
  R[5] = tyz - twx;
  R[6] = txz - twy;
  R[7] = tyz + twx;
  R[8] = 1.0 - (txx + tyy);
}

// C = A^T * B^T  (3x3 row-major)
__device__ __forceinline__ void mul_AtBt(const double* A, const double* B, double* C) {
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) C[3 * r + c] = A[r] * B[3 * c] + A[3 + r] * B[3 * c + 1] + A[6 + r] * B[3 * c + 2];
}

// Observation table -> per-factor pairs (viml.h, viml_window_batch): one CTA per window; pts_i of a factor is its feature's
// entry of feat_obs (every factor of a feature is built from feature_per_frame[0].point, estimator.cpp:1747-1766), pts_j its own.
template <typename T2>   // double2, or float2 (observations the caller still holds as the tracker's float32: widened here, exactly)
__global__ void expand_obs_kernel(LinearizeArgs a, const T2* __restrict__ feat_obs, const T2* __restrict__ pf_obs_j) {
  const int w = blockIdx.x;
  const int k0 = a.pf_window_offset[w], k1 = a.pf_window_offset[w + 1];
  const T2* fo = feat_obs + (size_t)w * a.F;
  double4* dst = reinterpret_cast<double4*>(const_cast<double*>(a.pf_obs));
  for (int k = k0 + threadIdx.x; k < k1; k += blockDim.x) {
    const uint32_t feat = a.pf_idx[k] >> 16;
    const T2 pj = pf_obs_j[k];
    double pix = 0.0, piy = 0.0;   // never read out of range; valid indices are the caller's to keep (viml.h, viml_window_batch)
    if (feat < (uint32_t)a.F) pix = (double)fo[feat].x, piy = (double)fo[feat].y;
    dst[k] = make_double4(pix, piy, (double)pj.x, (double)pj.y);
  }
}

// Line table -> lf_geom (viml.h, viml_window_batch): ptr = Rbw * map line end point + Tbw as Eigen evaluates it (row dot product
// left to right, then the translation; estimator.cpp:1832-1833) and (A, B, C) of Line2D(Vector4d) on the widened float32 end points
// (feature_manager.cpp:11-13).  Explicit round-to-nearest multiplies and adds: this file is compiled with FMA contraction.
struct MapFrame { double R[9], T[3]; };
__global__ void expand_lines_kernel(LinearizeArgs a, const double* __restrict__ map, int64_t N, MapFrame mf,
                                    const int32_t* __restrict__ idx, const float4* __restrict__ seg) {
  const int64_t k = a.lf_begin + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= a.lf_begin + a.NL) return;
  double* __restrict__ g = const_cast<double*>(a.lf_geom);
  int64_t j = idx[k];
  j = j < 0 ? 0 : (j >= N ? N - 1 : j);   // validated on the host-pointer path; clamped here for device-pointer callers
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const double x = map[(3 * e) * N + j], y = map[(3 * e + 1) * N + j], z = map[(3 * e + 2) * N + j];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const double d = __dadd_rn(__dadd_rn(__dmul_rn(mf.R[3 * r], x), __dmul_rn(mf.R[3 * r + 1], y)), __dmul_rn(mf.R[3 * r + 2], z));
      g[(size_t)(3 * e + r) * a.NL_stride + k] = __dadd_rn(d, mf.T[r]);
    }
  }
  const float4 s = seg[k];
  const double sx = s.x, sy = s.y, ex = s.z, ey = s.w;
  g[(size_t)6 * a.NL_stride + k] = __dsub_rn(ey, sy);
  g[(size_t)7 * a.NL_stride + k] = __dsub_rn(sx, ex);
  g[(size_t)8 * a.NL_stride + k] = __dsub_rn(__dmul_rn(ex, sy), __dmul_rn(sx, ey));
}

// One thread per pose (and one per window for the extrinsic): fills the cache described in common.cuh.
__global__ void prep_windows_kernel(LinearizeArgs a) {
  const int stride = a.P * kPoseCache + kExCache;
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)a.W * (a.P + 1);
  if (t >= total) return;
  const int w = (int)(t / (a.P + 1)), p = (int)(t % (a.P + 1));
  const double* ex = a.ex_pose + (size_t)w * 7;
  double ric[9];
  quat_to_rot(ex[6], ex[3], ex[4], ex[5], ric);
  double* cw = a.cache + (size_t)w * stride;
  if (p == a.P) {
    double* ec = cw + a.P * kPoseCache;
    const double n2 = ex[3] * ex[3] + ex[4] * ex[4] + ex[5] * ex[5] + ex[6] * ex[6];
    double ricinv[9];
    quat_to_rot(ex[6] / n2, -ex[3] / n2, -ex[4] / n2, -ex[5] / n2, ricinv);
#pragma unroll
    for (int k = 0; k < 3; ++k) ec[EC_TIC + k] = ex[k];
#pragma unroll
    for (int k = 0; k < 9; ++k) ec[EC_RIC + k] = ric[k], ec[EC_RICINV + k] = ricinv[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) ec[EC_RTT + k] = ric[k] * ex[0] + ric[3 + k] * ex[1] + ric[6 + k] * ex[2];
    return;
  }
  const double* q = a.poses + ((size_t)w * a.P + p) * 7;
  double* pc = cw + p * kPoseCache;
  double R[9], Rinv[9], M[9];
  quat_to_rot(q[6], q[3], q[4], q[5], R);
  const double n2 = q[3] * q[3] + q[4] * q[4] + q[5] * q[5] + q[6] * q[6];
  quat_to_rot(q[6] / n2, -q[3] / n2, -q[4] / n2, -q[5] / n2, Rinv);
  mul_AtBt(ric, R, M);
#pragma unroll
  for (int k = 0; k < 3; ++k) pc[PC_P + k] = q[k];
#pragma unroll
  for (int k = 0; k < 9; ++k) pc[PC_R + k] = R[k], pc[PC_RINV + k] = Rinv[k], pc[PC_M + k] = M[k];
  // line-factor transform: normalised quaternions (line_projection_factor.cpp:31-40, estimator.cpp:1777-1781)
  const double nq = sqrt(n2), ne = sqrt(ex[3] * ex[3] + ex[4] * ex[4] + ex[5] * ex[5] + ex[6] * ex[6]);
  double Rn[9], ricn[9], Rl[9];
  quat_to_rot(q[6] / nq, q[3] / nq, q[4] / nq, q[5] / nq, Rn);
  quat_to_rot(ex[6] / ne, ex[3] / ne, ex[4] / ne, ex[5] / ne, ricn);
  mul_AtBt(ricn, Rn, Rl);
#pragma unroll
  for (int k = 0; k < 9; ++k) pc[PC_RL + k] = Rl[k];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double rt = Rl[3 * k] * q[0] + Rl[3 * k + 1] * q[1] + Rl[3 * k + 2] * q[2];
    const double ct = ricn[k] * ex[0] + ricn[3 + k] * ex[1] + ricn[6 + k] * ex[2];
    pc[PC_TL + k] = -rt - ct;
  }
}

// 1/x and 1/sqrt(x) from the hardware approximations (2^-23) plus two Newton steps: relative error ~2e-16, a
// third of the instructions (and of the dependent latency) of the IEEE-rounded division / sqrt sequences.  The
// parity bar on this path is 1e-9 relative, not bit equality.
__device__ __forceinline__ double fast_rcp(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  r = fma(r, fma(-x, r, 1.0), r);
  r = fma(r, fma(-x, r, 1.0), r);
  return r;
}
__device__ __forceinline__ double fast_rsqrt(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  y = y * fma(-0.5 * x * y, y, 1.5);
  y = y * fma(-0.5 * x * y, y, 1.5);
  return y;
}

__device__ __forceinline__ int find_window(const int32_t* __restrict__ off, int W, int64_t k) {
  int lo = 0, hi = W;  // off[lo] <= k < off[hi]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (off[mid] <= k) lo = mid; else hi = mid;
  }
  return lo;
}

// Window of factor k for a warp of consecutive factors: lane 0's binary search is shared, the other lanes walk
// forward (a warp of 32 consecutive factors spans one or two windows).
__device__ __forceinline__ int find_window_warp(const int32_t* __restrict__ off, int W, int64_t k, int64_t k_warp) {
  int w = 0;
  if ((threadIdx.x & 31) == 0) w = find_window(off, W, k_warp);
  w = __shfl_sync(0xffffffffu, w, 0);
  while (w + 1 < W && off[w + 1] <= k) ++w;
  return w;
}

__device__ __forceinline__ void mat3_vec(const double* __restrict__ M, double x, double y, double z, double& ox,
                                         double& oy, double& oz) {
  ox = M[0] * x + M[1] * y + M[2] * z;
  oy = M[3] * x + M[4] * y + M[5] * z;
  oz = M[6] * x + M[7] * y + M[8] * z;
}

// Local Jacobian of a ProjectionFactor: a = d r/d pose_i (2x6), b = pose_j, c = extrinsic, d = inv depth.
struct PointJac {
  double r[2];
  double a[2][6], b[2][6], c[2][6], d[2];
};

__device__ __forceinline__ void eval_point(const LinearizeArgs& A, const double* __restrict__ cw, int i, int j,
                                           double lam, double pix, double piy, double piz, double pjx, double pjy,
                                           PointJac& J) {
  const double* __restrict__ ci = cw + i * kPoseCache;
  const double* __restrict__ cj = cw + j * kPoseCache;
  const double* __restrict__ ce = cw + A.P * kPoseCache;
  const double inv_l = fast_rcp(lam);
  const double cx_ = pix * inv_l, cy_ = piy * inv_l, cz_ = piz * inv_l;  // pts_camera_i (:35)
  double ix, iy, iz;                                                        // pts_imu_i (:36)
  mat3_vec(ce + EC_RIC, cx_, cy_, cz_, ix, iy, iz);
  ix += ce[EC_TIC], iy += ce[EC_TIC + 1], iz += ce[EC_TIC + 2];
  double wx, wy, wz;                                                        // pts_w (:37)
  mat3_vec(ci + PC_R, ix, iy, iz, wx, wy, wz);
  wx += ci[PC_P], wy += ci[PC_P + 1], wz += ci[PC_P + 2];
  const double dx = wx - cj[PC_P], dy = wy - cj[PC_P + 1], dz = wz - cj[PC_P + 2];
  double jx, jy, jz;                                                        // pts_imu_j (:38)
  mat3_vec(cj + PC_RINV, dx, dy, dz, jx, jy, jz);
  double qx, qy, qz;                                                        // pts_camera_j (:39)
  mat3_vec(ce + EC_RICINV, jx - ce[EC_TIC], jy - ce[EC_TIC + 1], jz - ce[EC_TIC + 2], qx, qy, qz);
  const double invz = fast_rcp(qz);
  const double s = A.sqrt_info;
  double r0 = s * (qx * invz - pjx), r1 = s * (qy * invz - pjy);           // :46-49
  double sc = 1.0;
  if (A.flags & VIML_LOSS_CAUCHY) {                                         // marginalization_factor.cpp:37-67
    // rho[2] < 0 always for Cauchy => residual_scaling = sqrt(rho1) = 1/sqrt(1 + s/a^2), alpha = 0
    // (the max(DBL_MIN, .) guard of ceres::CauchyLoss only matters for s > 1e308)
    sc = fast_rsqrt(fma(r0 * r0 + r1 * r1, A.inv_cauchy_a2, 1.0));
  }
  J.r[0] = sc * r0, J.r[1] = sc * r1;
  // reduce (:72-75) scaled by sqrt_info and the loss factor
  const double g = s * sc * invz;
  const double red0z = -g * qx * invz, red1z = -g * qy * invz;
  // A_ = reduce * M_j ; M_j = ric^T Rj^T
  const double* __restrict__ M = cj + PC_M;
  double A0[3], A1[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    A0[k] = g * M[k] + red0z * M[6 + k];
    A1[k] = g * M[3 + k] + red1z * M[6 + k];
  }
  // B = A_ * Ri
  const double* __restrict__ Ri = ci + PC_R;
  double B0[3], B1[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    B0[k] = A0[0] * Ri[k] + A0[1] * Ri[3 + k] + A0[2] * Ri[6 + k];
    B1[k] = A1[0] * Ri[k] + A1[1] * Ri[3 + k] + A1[2] * Ri[6 + k];
  }
  // C = reduce * ric^T
  const double* __restrict__ ric = ce + EC_RIC;
  double C0[3], C1[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    C0[k] = g * ric[3 * k] + red0z * ric[3 * k + 2];
    C1[k] = g * ric[3 * k + 1] + red1z * ric[3 * k + 2];
  }
  // D = B * ric  (= reduce * ric^T Rj^T Ri ric)
  double D0[3], D1[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    D0[k] = B0[0] * ric[k] + B0[1] * ric[3 + k] + B0[2] * ric[6 + k];
    D1[k] = B1[0] * ric[k] + B1[1] * ric[3 + k] + B1[2] * ric[6 + k];
  }
  // v = ric^T (Rj^T (pts_w - Pj) - tic) = M (pts_w - Pj) - ric^T tic   (:105-106 collapsed)
  double vx, vy, vz;
  mat3_vec(M, dx, dy, dz, vx, vy, vz);
  vx -= ce[EC_RTT], vy -= ce[EC_RTT + 1], vz -= ce[EC_RTT + 2];
  // pose_i (:81-85): [A_ | B * -skew(pts_imu_i)]  ; row b: b^T(-[p]x) = (p x b)^T
#pragma unroll
  for (int k = 0; k < 3; ++k) J.a[0][k] = A0[k], J.a[1][k] = A1[k];
  J.a[0][3] = iy * B0[2] - iz * B0[1], J.a[0][4] = iz * B0[0] - ix * B0[2], J.a[0][5] = ix * B0[1] - iy * B0[0];
  J.a[1][3] = iy * B1[2] - iz * B1[1], J.a[1][4] = iz * B1[0] - ix * B1[2], J.a[1][5] = ix * B1[1] - iy * B1[0];
  // pose_j (:93-97): [-A_ | C * skew(pts_imu_j)] ; row c: c^T [p]x = (c x p)^T.  The reference's pts_imu_j
  // is the quaternion-rotated one (:38).
#pragma unroll
  for (int k = 0; k < 3; ++k) J.b[0][k] = -A0[k], J.b[1][k] = -A1[k];
  J.b[0][3] = C0[1] * jz - C0[2] * jy, J.b[0][4] = C0[2] * jx - C0[0] * jz, J.b[0][5] = C0[0] * jy - C0[1] * jx;
  J.b[1][3] = C1[1] * jz - C1[2] * jy, J.b[1][4] = C1[2] * jx - C1[0] * jz, J.b[1][5] = C1[0] * jy - C1[1] * jx;
  // extrinsic (:103-108): [B - C | -D skew(pc_i) + reduce skew(v)] ; rows: pc_i x d + red x v
#pragma unroll
  for (int k = 0; k < 3; ++k) J.c[0][k] = B0[k] - C0[k], J.c[1][k] = B1[k] - C1[k];
  J.c[0][3] = (cy_ * D0[2] - cz_ * D0[1]) + (0.0 * vz - red0z * vy);
  J.c[0][4] = (cz_ * D0[0] - cx_ * D0[2]) + (red0z * vx - g * vz);
  J.c[0][5] = (cx_ * D0[1] - cy_ * D0[0]) + (g * vy - 0.0 * vx);
  J.c[1][3] = (cy_ * D1[2] - cz_ * D1[1]) + (g * vz - red1z * vy);
  J.c[1][4] = (cz_ * D1[0] - cx_ * D1[2]) + (red1z * vx - 0.0 * vz);
  J.c[1][5] = (cx_ * D1[1] - cy_ * D1[0]) + (0.0 * vy - g * vx);
  // inverse depth (:115): reduce * T * pts_i * -1/lambda^2
  const double nl2 = -inv_l * inv_l;
  J.d[0] = (D0[0] * pix + D0[1] * piy + D0[2] * piz) * nl2;
  J.d[1] = (D1[0] * pix + D1[1] * piy + D1[2] * piz) * nl2;
}

struct LineJac {
  double r[2];
  double a[2][6];
};

__device__ __forceinline__ void eval_line(const LinearizeArgs& A, const double* __restrict__ cw, int frame,
                                          const double* g9, LineJac& J) {
  const double* __restrict__ cf = cw + frame * kPoseCache;
  const double* __restrict__ R = cf + PC_RL;
  double sx, sy, sz, ex, ey, ez;
  mat3_vec(R, g9[0], g9[1], g9[2], sx, sy, sz);
  mat3_vec(R, g9[3], g9[4], g9[5], ex, ey, ez);
  sx += cf[PC_TL], sy += cf[PC_TL + 1], sz += cf[PC_TL + 2];
  ex += cf[PC_TL], ey += cf[PC_TL + 1], ez += cf[PC_TL + 2];
  const double isz = fast_rcp(sz), iez = fast_rcp(ez);
  // (K*pc).x/(K*pc).z = (fx*X + cx*Z)/Z                                (line_projection_factor.cpp:45-51)
  const double us = (A.fx * sx + A.cx * sz) * isz, vs = (A.fy * sy + A.cy * sz) * isz;
  const double ue = (A.fx * ex + A.cx * ez) * iez, ve = (A.fy * ey + A.cy * ez) * iez;
  const double a = g9[6], b = g9[7], c = g9[8];
  const double d = a * a + b * b, id = fast_rcp(d);
  const double mus = (b * b * us - a * b * vs - a * c) * id, mvs = (a * a * vs - a * b * us - b * c) * id;
  const double mue = (b * b * ue - a * b * ve - a * c) * id, mve = (a * a * ve - a * b * ue - b * c) * id;
  const double dus = mus - us, dvs = mvs - vs, due = mue - ue, dve = mve - ve;
  double r0 = sqrt(dus * dus + dvs * dvs), r1 = sqrt(due * due + dve * dve);   // :68-69
  double sc = 1.0;
  if (A.flags & VIML_LOSS_CAUCHY) {
    sc = fast_rsqrt(fma(r0 * r0 + r1 * r1, A.inv_cauchy_a2, 1.0));
  }
  J.r[0] = sc * r0, J.r[1] = sc * r1;
  const double m2d = -2.0 * id * sc;
  const double e1s = m2d * (dus * a * a + a * b * dvs), e2s = m2d * (dus * a * b + b * b * dvs);   // :76-80
  const double e1e = m2d * (due * a * a + a * b * dve), e2e = m2d * (due * a * b + b * b * dve);
  // w = e_p * d(pi)/d(pc)  (:93-100), then [I | skew(pc)] (:104-113): rot part = w x pc ... as coded:
  // (w^T skew(pc))_c = sum_r w_r S(r,c)  with S = [[0,-z,y],[z,0,-x],[-y,x,0]]
  {
    const double w0 = e1s * A.fx * isz, w1 = e2s * A.fy * isz;
    const double w2 = -(e1s * A.fx * sx + e2s * A.fy * sy) * isz * isz;
    J.a[0][0] = w0, J.a[0][1] = w1, J.a[0][2] = w2;
    J.a[0][3] = w1 * sz - w2 * sy;
    J.a[0][4] = w2 * sx - w0 * sz;
    J.a[0][5] = w0 * sy - w1 * sx;
  }
  {
    const double w0 = e1e * A.fx * iez, w1 = e2e * A.fy * iez;
    const double w2 = -(e1e * A.fx * ex + e2e * A.fy * ey) * iez * iez;
    J.a[1][0] = w0, J.a[1][1] = w1, J.a[1][2] = w2;
    J.a[1][3] = w1 * ez - w2 * ey;
    J.a[1][4] = w2 * ex - w0 * ez;
    J.a[1][5] = w0 * ey - w1 * ex;
  }
}

__device__ __forceinline__ void store_jac7(double* __restrict__ dst, const double (*J)[6]) {
  // row-major 2x7, column 6 zero; 112 B = 7 x 16 B, 16-byte aligned
  double2* d2 = reinterpret_cast<double2*>(dst);
  d2[0] = make_double2(J[0][0], J[0][1]);
  d2[1] = make_double2(J[0][2], J[0][3]);
  d2[2] = make_double2(J[0][4], J[0][5]);
  d2[3] = make_double2(0.0, J[1][0]);
  d2[4] = make_double2(J[1][1], J[1][2]);
  d2[5] = make_double2(J[1][3], J[1][4]);
  d2[6] = make_double2(J[1][5], 0.0);
}

// Warp-cooperative version: the 32 rows of a warp (32 x 112 B, contiguous in the output array) are first laid out
// in shared memory (STS.128 at a 7 x 16 B lane stride is conflict-free), then written with fully coalesced
// 512-byte STG.128 instructions.  Direct per-lane stores touch 32 different lines per instruction and write every
// sector in two halves; this halves the LSU sector work and gives L2 whole sectors.
// `stage` is this warp's 3584-byte buffer, `dst` the output row of the warp's first lane, nvalid its live lanes.
__device__ __forceinline__ void store_jac7_coalesced(double2* __restrict__ stage, double* __restrict__ dst,
                                                     const double (*J)[6], int lane, int nvalid) {
  double2* mine = stage + 7 * lane;
  mine[0] = make_double2(J[0][0], J[0][1]);
  mine[1] = make_double2(J[0][2], J[0][3]);
  mine[2] = make_double2(J[0][4], J[0][5]);
  mine[3] = make_double2(0.0, J[1][0]);
  mine[4] = make_double2(J[1][1], J[1][2]);
  mine[5] = make_double2(J[1][3], J[1][4]);
  mine[6] = make_double2(J[1][5], 0.0);
  __syncwarp();
  double2* d2 = reinterpret_cast<double2*>(dst);
  const int n16 = 7 * nvalid;  // 16-byte units to copy
#pragma unroll
  for (int q = 0; q < 7; ++q) {
    const int e = q * 32 + lane;
    if (e < n16) d2[e] = stage[e];
  }
  __syncwarp();
}

// H(rows r0.., cols c0..) += X^T Y and its mirror, X,Y 2x6, via global atomics (generic path: used for
// windows too large for the shared-memory assembly kernel and as the simple reference device path).
__device__ __forceinline__ void atomic_block(double* __restrict__ H, int D, int r0, int c0, const double (*X)[6],
                                             const double (*Y)[6], bool diag) {
#pragma unroll
  for (int r = 0; r < 6; ++r)
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      const double v = X[0][r] * Y[0][c] + X[1][r] * Y[1][c];
      atomicAdd(H + (size_t)(r0 + r) * D + c0 + c, v);
      if (!diag) atomicAdd(H + (size_t)(c0 + c) * D + r0 + r, v);
    }
}

// Generic accumulation of one point factor into the zero-initialised blocks of its window.  Every point factor of a window adds
// to the same extrinsic block and b_ex: when the 32 factors of the warp belong to one window (`warp_window`: always, for one huge
// window) those 27 sums are reduced over the warp first and lane 0 adds them once — 57 K factors no longer queue on 42 addresses.
__device__ __forceinline__ void point_atomics(const LinearizeArgs& A, int w, int i, int j, int f, const PointJac& J, bool live,
                                              bool warp_window) {
  const int D = A.D;
  double* H = A.out.H_pp + (size_t)w * D * D;
  double* bp = A.out.b_p + (size_t)w * D;
  const int oi = 6 * i, oj = 6 * j, oe = 6 * A.P;
  if (warp_window) {
    double v[27];
    int n = 0;
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
      for (int c = r; c < 6; ++c) v[n++] = live ? J.c[0][r] * J.c[0][c] + J.c[1][r] * J.c[1][c] : 0.0;
#pragma unroll
    for (int r = 0; r < 6; ++r) v[21 + r] = live ? J.c[0][r] * J.r[0] + J.c[1][r] * J.r[1] : 0.0;
#pragma unroll
    for (int e = 0; e < 27; ++e)
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) v[e] += __shfl_xor_sync(0xffffffffu, v[e], d);
    if ((threadIdx.x & 31) == 0) {
      n = 0;
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int c = r; c < 6; ++c) {
          atomicAdd(H + (size_t)(oe + r) * D + oe + c, v[n]);
          if (c != r) atomicAdd(H + (size_t)(oe + c) * D + oe + r, v[n]);
          ++n;
        }
#pragma unroll
      for (int r = 0; r < 6; ++r) atomicAdd(bp + oe + r, v[21 + r]);
    }
  }
  if (!live) return;
  double* Hl = A.out.H_lp + ((size_t)w * A.F + f) * D;
  atomic_block(H, D, oi, oi, J.a, J.a, true);
  atomic_block(H, D, oi, oj, J.a, J.b, false);
  atomic_block(H, D, oi, oe, J.a, J.c, false);
  atomic_block(H, D, oj, oj, J.b, J.b, true);
  atomic_block(H, D, oj, oe, J.b, J.c, false);
  if (!warp_window) atomic_block(H, D, oe, oe, J.c, J.c, true);
#pragma unroll
  for (int r = 0; r < 6; ++r) {
    atomicAdd(bp + oi + r, J.a[0][r] * J.r[0] + J.a[1][r] * J.r[1]);
    atomicAdd(bp + oj + r, J.b[0][r] * J.r[0] + J.b[1][r] * J.r[1]);
    if (!warp_window) atomicAdd(bp + oe + r, J.c[0][r] * J.r[0] + J.c[1][r] * J.r[1]);
    atomicAdd(Hl + oi + r, J.a[0][r] * J.d[0] + J.a[1][r] * J.d[1]);
    atomicAdd(Hl + oj + r, J.b[0][r] * J.d[0] + J.b[1][r] * J.d[1]);
    atomicAdd(Hl + oe + r, J.c[0][r] * J.d[0] + J.c[1][r] * J.d[1]);
  }
  atomicAdd(A.out.H_ll + (size_t)w * A.F + f, J.d[0] * J.d[0] + J.d[1] * J.d[1]);
  atomicAdd(A.out.b_l + (size_t)w * A.F + f, J.d[0] * J.r[0] + J.d[1] * J.r[1]);
}

// Generic accumulation of one line factor: (frame, frame) block and b.
__device__ __forceinline__ void line_atomics(const LinearizeArgs& A, int w, int frame, const LineJac& J) {
  const int D = A.D;
  double* H = A.out.H_pp + (size_t)w * D * D;
  double* bp = A.out.b_p + (size_t)w * D;
  const int of = 6 * frame;
  atomic_block(H, D, of, of, J.a, J.a, true);
#pragma unroll
  for (int r = 0; r < 6; ++r) atomicAdd(bp + of + r, J.a[0][r] * J.r[0] + J.a[1][r] * J.r[1]);
}

template <bool MODE_A, bool MODE_B>
#ifndef VIML_POINTS_MINB
#define VIML_POINTS_MINB 4
#endif
// mode A alone streams (4 CTAs per SM hide the store latency); with the atomic H/b accumulation of the generic path the Jacobians
// stay live across ~190 atomics and 128 registers spill (70 LDL/STL in round 1): two CTAs per SM, up to 255 registers (at 168 it still spills 100 bytes)
__global__ void __launch_bounds__(128, MODE_B ? 2 : VIML_POINTS_MINB) points_kernel(LinearizeArgs A) {
  __shared__ double2 stage[MODE_A ? 4 * 7 * 32 : 1];
  const int64_t k_raw = A.pf_begin + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t k_end = A.pf_begin + A.NP;
  const int lane = threadIdx.x & 31;
  const int64_t k_warp = k_raw - lane;
  if (k_warp >= k_end) return;                       // whole warp out of range
  const int nvalid = (int)min((int64_t)32, k_end - k_warp);
  const int64_t k = min(k_raw, k_end - 1);           // idle tail lanes recompute the last factor, they store nothing
  const bool live = k_raw < k_end;
  const int w = find_window_warp(A.pf_window_offset, A.W, k, k_warp);
  const uint32_t pk = A.pf_idx[k];
  const int i = pk & 0xff, j = (pk >> 8) & 0xff, f = pk >> 16;
  const double4 ob = reinterpret_cast<const double4*>(A.pf_obs)[k];
  const double piz = A.pf_pts_i_z ? A.pf_pts_i_z[k] : 1.0;
  const double lam = A.inv_depth[(size_t)w * A.F + f];
  const double* cw = A.cache + (size_t)w * (A.P * kPoseCache + kExCache);
  PointJac J;
  eval_point(A, cw, i, j, lam, ob.x, ob.y, piz, ob.z, ob.w, J);
  if (MODE_A) {
    double2* st = stage + (threadIdx.x >> 5) * 7 * 32;
    if (live && A.out.pf_residual) reinterpret_cast<double2*>(A.out.pf_residual)[k] = make_double2(J.r[0], J.r[1]);
    if (A.out.pf_jac_pose_i) store_jac7_coalesced(st, A.out.pf_jac_pose_i + 14 * k_warp, J.a, lane, nvalid);
    if (A.out.pf_jac_pose_j) store_jac7_coalesced(st, A.out.pf_jac_pose_j + 14 * k_warp, J.b, lane, nvalid);
    if (A.out.pf_jac_ex) store_jac7_coalesced(st, A.out.pf_jac_ex + 14 * k_warp, J.c, lane, nvalid);
    if (live && A.out.pf_jac_feat) reinterpret_cast<double2*>(A.out.pf_jac_feat)[k] = make_double2(J.d[0], J.d[1]);
  }
  if (MODE_B) {
    const bool warp_window = __all_sync(0xffffffffu, w == __shfl_sync(0xffffffffu, w, 0));
    point_atomics(A, w, i, j, f, J, live, warp_window);
  }
}

template <bool MODE_A, bool MODE_B>
__global__ void __launch_bounds__(128) lines_kernel(LinearizeArgs A) {
  __shared__ double2 stage[MODE_A ? 4 * 7 * 32 : 1];
  const int64_t k_raw = A.lf_begin + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t k_end = A.lf_begin + A.NL;
  const int lane = threadIdx.x & 31;
  const int64_t k_warp = k_raw - lane;
  if (k_warp >= k_end) return;
  const int nvalid = (int)min((int64_t)32, k_end - k_warp);
  const int64_t k = min(k_raw, k_end - 1);
  const bool live = k_raw < k_end;
  const int w = find_window_warp(A.lf_window_offset, A.W, k, k_warp);
  const int frame = A.lf_frame[k];
  double g9[9];
#pragma unroll
  for (int c = 0; c < 9; ++c) g9[c] = A.lf_geom[(size_t)c * A.NL_stride + k];
  const double* cw = A.cache + (size_t)w * (A.P * kPoseCache + kExCache);
  LineJac J;
  eval_line(A, cw, frame, g9, J);
  if (MODE_A) {
    if (live && A.out.lf_residual) reinterpret_cast<double2*>(A.out.lf_residual)[k] = make_double2(J.r[0], J.r[1]);
    if (A.out.lf_jac_pose)
      store_jac7_coalesced(stage + (threadIdx.x >> 5) * 7 * 32, A.out.lf_jac_pose + 14 * k_warp, J.a, lane, nvalid);
  }
  if (MODE_B && live) line_atomics(A, w, frame, J);
}

// VIML_S_PACKED: upper triangle of every window's S, row r = columns r..D-1.  grid = (windows, slices of the window's entries):
// one CTA per window for the sliding-window size, many for a long window (D = 1212: 1.5 M entries)
__global__ void __launch_bounds__(256) pack_upper_kernel(int D, const double* __restrict__ S, double* __restrict__ Sp) {
  const double* __restrict__ s = S + (size_t)blockIdx.x * D * D;
  double* __restrict__ o = Sp + (size_t)blockIdx.x * ((size_t)D * (D + 1) / 2);
  for (int e = blockIdx.y * blockDim.x + threadIdx.x; e < D * D; e += gridDim.y * blockDim.x) {
    const int r = e / D, c = e - r * D;
    if (c >= r) o[(size_t)r * D - ((size_t)r * (r - 1)) / 2 + c - r] = s[e];
  }
}

#include "assemble2.cuh"
#include "gn_kernels.cuh"

}  // namespace

int viml_launch_linearize(viml_ctx* ctx, const LinearizeArgs& a) {
  cudaStream_t st = ctx->stream;
  const bool modeA = (a.flags & VIML_OUT_RESIDUAL_JACOBIAN) != 0;
  const bool modeB = (a.flags & (VIML_OUT_HB | VIML_OUT_SCHUR)) != 0;
  // fused path: plan_kernel + assemble_kernel (assemble2.cuh); anything outside its static limits goes through the
  // generic atomic kernels
  const size_t plan_smem = (size_t)a.F * 8 + ((size_t)a.F + 1) * 4 + (((size_t)a.F + 1) & ~(size_t)1) * 2 + (size_t)a.F * a.P * 2 + 16;
  const bool fast = modeB && a.P <= stream::PMAX && a.F <= stream::FMAXP && plan_smem <= 200 * 1024 && !ctx->force_generic;
  stream::PlanPtrs PL{};
  if (fast) {
    const size_t n_tasks = (size_t)a.NP / 64 + (size_t)a.W * (a.F / stream::TASK_F + stream::PMAX + 4) + 2;
    auto pad = [](size_t b) { return DeviceArena::padded(b); };
    VIML_TRY_CUDA(ctx, ctx->scratch3.reserve(pad((size_t)a.W * 16) + pad(n_tasks * 16) + pad((size_t)a.NP * 8 + 8) +
                                             pad((size_t)a.W * a.F * 4 + 4) + pad((size_t)a.NL * 8 + 8) + pad(4)));
    PL.hdr = ctx->scratch3.take<int4>((size_t)a.W);
    PL.tasks = ctx->scratch3.take<int4>(n_tasks);
    PL.slots = ctx->scratch3.take<uint32_t>((size_t)a.NP * 2 + 2);
    PL.finfo = ctx->scratch3.take<uint32_t>((size_t)a.W * a.F + 1);
    PL.lslots = ctx->scratch3.take<uint32_t>((size_t)a.NL * 2 + 2);
    PL.any_irregular = ctx->scratch3.take<int>(1);
    // the plan depends on the factor indices only, the pose cache (prep_windows_kernel) on the states only: the two
    // short kernels run side by side on two streams and meet before the fused kernel
    VIML_TRY_CUDA(ctx, cudaEventRecord(ctx->ev_fork, st));
    VIML_TRY_CUDA(ctx, cudaStreamWaitEvent(ctx->aux_stream, ctx->ev_fork, 0));
    VIML_TRY_CUDA(ctx, cudaMemsetAsync(PL.any_irregular, 0, 4, ctx->aux_stream));
    VIML_TRY_CUDA(ctx, cudaFuncSetAttribute(stream::plan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan_smem));
    {
      LaunchScope ls(ctx, K_PLAN, ctx->aux_stream);
      stream::plan_kernel<<<a.W, a.F > 512 ? stream::PT_MAX : stream::PT, plan_smem, ctx->aux_stream>>>(a, PL);
    }
    VIML_TRY_CUDA(ctx, cudaEventRecord(ctx->ev_join, ctx->aux_stream));
  }
  {
    const int64_t total = (int64_t)a.W * (a.P + 1);
    LaunchScope ls(ctx, K_PREP);
    prep_windows_kernel<<<(unsigned)((total + 127) / 128), 128, 0, st>>>(a);
  }
  if (fast) {
    VIML_TRY_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_join, 0));
    // one CTA (4 warps) per window, three CTAs per SM; every H/b entry is written exactly once (no memset)
    const int NB = a.P + 1, nblk = NB * (NB + 1) / 2;
    const size_t smem = ((size_t)((nblk * 36 + a.D + 1) & ~1) + (size_t)a.P * kPoseCache + kExCache + (size_t)stream::AW * stream::WORK_D) * 8;
    const int use_tma = ((((uintptr_t)a.out.H_pp) | ((uintptr_t)a.out.b_p)) & 15) == 0 ? 1 : 0;
    // the attribute is per device: set on every call (a process may hold contexts on several devices)
    VIML_TRY_CUDA(ctx, cudaFuncSetAttribute(stream::assemble_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VIML_TRY_CUDA(ctx, cudaFuncSetAttribute(stream::assemble_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    {
      LaunchScope ls(ctx, K_ASSEMBLE);
      if (modeA) stream::assemble_kernel<true><<<a.W, stream::AW * 32, smem, st>>>(a, PL, use_tma);
      else stream::assemble_kernel<false><<<a.W, stream::AW * 32, smem, st>>>(a, PL, use_tma);
    }
    {
      const int grid = a.W < 4 * ctx->sm_count ? a.W : 4 * ctx->sm_count;
      LaunchScope ls(ctx, K_IRREGULAR);
      if (modeA) stream::irregular_kernel<true><<<grid, 128, 0, st>>>(a, PL);
      else stream::irregular_kernel<false><<<grid, 128, 0, st>>>(a, PL);
    }
  } else {
    if (modeB) {
      const size_t W = a.W, D = a.D, F = a.F;
      VIML_TRY_CUDA(ctx, cudaMemsetAsync(a.out.H_pp, 0, W * D * D * sizeof(double), st));
      VIML_TRY_CUDA(ctx, cudaMemsetAsync(a.out.H_lp, 0, W * F * D * sizeof(double), st));
      VIML_TRY_CUDA(ctx, cudaMemsetAsync(a.out.H_ll, 0, W * F * sizeof(double), st));
      VIML_TRY_CUDA(ctx, cudaMemsetAsync(a.out.b_p, 0, W * D * sizeof(double), st));
      VIML_TRY_CUDA(ctx, cudaMemsetAsync(a.out.b_l, 0, W * F * sizeof(double), st));
    }
    if (a.NP > 0) {
      const unsigned grid = (unsigned)((a.NP + 127) / 128);
      LaunchScope ls(ctx, K_POINTS);
      if (modeA && modeB) points_kernel<true, true><<<grid, 128, 0, st>>>(a);
      else if (modeA) points_kernel<true, false><<<grid, 128, 0, st>>>(a);
      else if (modeB) points_kernel<false, true><<<grid, 128, 0, st>>>(a);
    }
    if (a.NL > 0) {
      const unsigned grid = (unsigned)((a.NL + 127) / 128);
      LaunchScope ls(ctx, K_LINES);
      if (modeA && modeB) lines_kernel<true, true><<<grid, 128, 0, st>>>(a);
      else if (modeA) lines_kernel<true, false><<<grid, 128, 0, st>>>(a);
      else if (modeB) lines_kernel<false, true><<<grid, 128, 0, st>>>(a);
    }
  }
  if (a.flags & VIML_OUT_SCHUR) {
    const double eps = 1e-8;  // MarginalizationInfo::eps (marginalization_factor.h:70)
    double* S = a.out.S;
    if (a.flags & VIML_S_PACKED) {   // full S into scratch, its upper triangle to the caller
      VIML_TRY_CUDA(ctx, ctx->s_full.reserve(DeviceArena::padded((size_t)a.W * a.D * a.D * 8)));
      S = ctx->s_full.take<double>((size_t)a.W * a.D * a.D);
    }
    viml_launch_schur(ctx, a.W, a.F, a.D, a.out.H_pp, a.out.H_lp, a.out.H_ll, a.out.b_p, a.out.b_l, S, a.out.g, eps);
    if (a.flags & VIML_S_PACKED) {
      LaunchScope ls(ctx, K_SCHUR);
      const unsigned slices = (unsigned)std::min<int64_t>(((int64_t)a.D * a.D + 256 * 32 - 1) / (256 * 32), 1024);
      pack_upper_kernel<<<dim3((unsigned)a.W, slices), 256, 0, st>>>(a.D, S, a.out.S);
    }
  }
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  return VIML_OK;
}

int viml_launch_expand_obs(viml_ctx* ctx, const LinearizeArgs& a, const void* feat_obs, const void* pf_obs_j, bool f32) {
  if (a.NP == 0) return VIML_OK;
  LaunchScope ls(ctx, K_PREP);
  if (f32) expand_obs_kernel<float2><<<a.W, 128, 0, ctx->stream>>>(a, (const float2*)feat_obs, (const float2*)pf_obs_j);
  else expand_obs_kernel<double2><<<a.W, 128, 0, ctx->stream>>>(a, (const double2*)feat_obs, (const double2*)pf_obs_j);
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  return VIML_OK;
}

int viml_launch_expand_lines(viml_ctx* ctx, const LinearizeArgs& a, const int32_t* lf_map_index, const float* lf_seg2d) {
  if (a.NL == 0) return VIML_OK;
  if (!ctx->map_set || ctx->n_map <= 0) {
    ctx->err = "line factors given by map index need a map (viml_set_map)";
    return VIML_ERR_NOMAP;
  }
  MapFrame mf;
  for (int k = 0; k < 9; ++k) mf.R[k] = ctx->cfg.Rbw[k];
  for (int k = 0; k < 3; ++k) mf.T[k] = ctx->cfg.Tbw[k];
  LaunchScope ls(ctx, K_PREP);
  expand_lines_kernel<<<(unsigned)((a.NL + 127) / 128), 128, 0, ctx->stream>>>(a, ctx->d_map, ctx->n_map, mf, lf_map_index,
                                                                             reinterpret_cast<const float4*>(lf_seg2d));
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  return VIML_OK;
}

int viml_launch_prep(viml_ctx* ctx, const LinearizeArgs& a) {
  const int64_t total = (int64_t)a.W * (a.P + 1);
  LaunchScope ls(ctx, K_PREP);
  prep_windows_kernel<<<(unsigned)((total + 127) / 128), 128, 0, ctx->stream>>>(a);
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  return VIML_OK;
}

int viml_launch_reduced(viml_ctx* ctx, int W, int D, const DenseArgs& dn, const double* S, const double* g, double* Sx, double* gx) {
  LaunchScope ls(ctx, K_GN);
  const int smem = gn::kReducedStage * (int)sizeof(double);
  VIML_TRY_CUDA(ctx, cudaFuncSetAttribute(gn::reduced_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  gn::reduced_kernel<<<W, 256, smem, ctx->stream>>>(D, dn, S, g, Sx, gx);
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  return VIML_OK;
}

int viml_launch_gn_solve(viml_ctx* ctx, int W, int Dx, double lambda, const double* Sx, const double* gx, double* dx, int32_t* solved,
                         double* cost, const double* lambda_w, const int32_t* running) {
  const size_t smem = gn_solve_smem(Dx);
  LaunchScope ls(ctx, K_GN);
  VIML_TRY_CUDA(ctx, cudaFuncSetAttribute(gn::solve_tiled_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  gn::solve_tiled_kernel<false><<<W, 256, smem, ctx->stream>>>(Dx, lambda, Sx, gx, dx, solved, cost, 0, DenseArgs{}, nullptr, nullptr,
                                                                lambda_w, running);
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  return VIML_OK;
}

int viml_launch_gn_reduced_solve(viml_ctx* ctx, int W, int D, const DenseArgs& dn, const double* S, const double* g, double lambda,
                                 double* dx, int32_t* solved, double* cost, const double* lambda_w, const int32_t* running) {
  const int Dx = D + dn.X;
  const size_t smem = gn_fused_solve_smem(Dx);
  LaunchScope ls(ctx, K_GN);
  VIML_TRY_CUDA(ctx, cudaFuncSetAttribute(gn::solve_tiled_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  gn::solve_tiled_kernel<true><<<W, 256, smem, ctx->stream>>>(Dx, lambda, nullptr, nullptr, dx, solved, cost, D, dn, S, g, lambda_w,
                                                               running);
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  return VIML_OK;
}

int viml_launch_gn_update(viml_ctx* ctx, const LinearizeArgs& a, int X, const double* extra_in, const double* dx, const int32_t* solved,
                          double* o_poses, double* o_ex, double* o_dep, double* o_extra, const int32_t* running) {
  LaunchScope ls(ctx, K_GN);
  gn::update_kernel<<<a.W, 128, 0, ctx->stream>>>(a, X, extra_in, dx, solved, o_poses, o_ex, o_dep, o_extra, running);
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  return VIML_OK;
}

int viml_launch_cost(viml_ctx* ctx, const LinearizeArgs& a, const DenseArgs& dn, const double* dx, const int32_t* solved, int slot,
                     double* cost, const int32_t* running) {
  LaunchScope ls(ctx, K_GN);
  gn::cost_kernel<<<a.W, 128, 0, ctx->stream>>>(a, dn, dx, solved, slot, cost, running);
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  return VIML_OK;
}

int viml_launch_solve_policy(viml_ctx* ctx, int W, const SolveArgs& s, int round) {
  LaunchScope ls(ctx, K_GN);
  gn::policy_kernel<<<W, 128, 0, ctx->stream>>>(s, round);
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  return VIML_OK;
}
