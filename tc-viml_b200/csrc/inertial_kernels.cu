// inertial_kernels.cu — the window's IMU factors and the prior of the last marginalisation, evaluated on the device at a state.
//
// Reference: IMUFactor::Evaluate (vins_estimator/src/factor/imu_factor.h:19-181) with IntegrationBase::evaluate
// (factor/integration_base.h), MarginalizationFactor::Evaluate (factor/marginalization_factor.cpp:335-384).  Quaternion arithmetic
// is Eigen's (SURVEY.md Appendix A): Quaterniond(p[6], p[3], p[4], p[5]), inverse() divides by the squared norm, no normalisation;
// Utility::positify is the identity (utility.h:41-48).  Pre-integration (push_back, midPointIntegration, repropagate) and
// sqrt_info stay with the host: their outputs are inputs here.
//
// Three kernels:
//   csr_offsets_kernel  one CTA: scan over the windows of (factors, rows, columns, Jacobian entries) -> the dense-factor CSR
//                       offsets (per window the prior first, then its IMU factors), so that the device flavour needs no readback;
//   prior_kernel        one CTA per window: dx per kept block, r = linearized_residuals + J dx, J copied into the CSR;
//   imu_kernel          one warp per factor: lane c < 30 builds raw Jacobian column c of the 15 x 30 block
//                       [pose_i(6) | sb_i(9) | pose_j(6) | sb_j(9)], lane 30 the raw residual; every lane premultiplies its
//                       column by sqrt_info (staged in shared memory, read by broadcast) and writes its entries of both layouts.
#include "common.cuh"

namespace inertial {

struct Q {
  double w, x, y, z;
};
struct V {
  double x, y, z;
};

__device__ __forceinline__ Q qmul(Q a, Q b) {
  return {a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z, a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y,
          a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z, a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x};
}
__device__ __forceinline__ Q qinv(Q q) {
  const double n2 = q.w * q.w + q.x * q.x + q.y * q.y + q.z * q.z;
  return {q.w / n2, -q.x / n2, -q.y / n2, -q.z / n2};
}
__device__ __forceinline__ V cross(V a, V b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
// Eigen's _transformVector: uv = q.vec x v; uv += uv; v + w uv + q.vec x uv
__device__ __forceinline__ V rot(Q q, V v) {
  const V u{q.x, q.y, q.z};
  V uv = cross(u, v);
  uv = {uv.x + uv.x, uv.y + uv.y, uv.z + uv.z};
  const V c = cross(u, uv);
  return {v.x + q.w * uv.x + c.x, v.y + q.w * uv.y + c.y, v.z + q.w * uv.z + c.z};
}
// column k of toRotationMatrix(q)
__device__ __forceinline__ V rotcol(Q q, int k) {
  const double tx = 2 * q.x, ty = 2 * q.y, tz = 2 * q.z;
  const double twx = tx * q.w, twy = ty * q.w, twz = tz * q.w, txx = tx * q.x, txy = ty * q.x, txz = tz * q.x;
  const double tyy = ty * q.y, tyz = tz * q.y, tzz = tz * q.z;
  if (k == 0) return {1 - (tyy + tzz), txy + twz, txz - twy};
  if (k == 1) return {txy - twz, 1 - (txx + tzz), tyz + twx};
  return {txz + twy, tyz - twx, 1 - (txx + tyy)};
}
__device__ __forceinline__ double comp(V v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : v.z); }
__device__ __forceinline__ V unit(int k) { return {k == 0 ? 1.0 : 0.0, k == 1 ? 1.0 : 0.0, k == 2 ? 1.0 : 0.0}; }
// column k of skewSymmetric(v) (utility.h:31-38) = v x e_k
__device__ __forceinline__ V skewcol(V v, int k) { return cross(v, unit(k)); }
__device__ __forceinline__ Q quat(const double* p) { return {p[6], p[3], p[4], p[5]}; }
__device__ __forceinline__ V vec(const double* p) { return {p[0], p[1], p[2]}; }
// column c of the 3 x 3 block (r0, c0) of a row-major 15 x 15 matrix
__device__ __forceinline__ V jcol(const double* J, int r0, int c0) {
  return {J[r0 * 15 + c0], J[(r0 + 1) * 15 + c0], J[(r0 + 2) * 15 + c0]};
}
__device__ __forceinline__ V mul3(const double* J, int r0, int c0, V v) {   // block (r0, c0) times v
  V o;
  o.x = J[r0 * 15 + c0] * v.x + J[r0 * 15 + c0 + 1] * v.y + J[r0 * 15 + c0 + 2] * v.z;
  o.y = J[(r0 + 1) * 15 + c0] * v.x + J[(r0 + 1) * 15 + c0 + 1] * v.y + J[(r0 + 1) * 15 + c0 + 2] * v.z;
  o.z = J[(r0 + 2) * 15 + c0] * v.x + J[(r0 + 2) * 15 + c0 + 1] * v.y + J[(r0 + 2) * 15 + c0 + 2] * v.z;
  return o;
}

constexpr int O_P = 0, O_R = 3, O_V = 6, O_BA = 9, O_BG = 12;

__global__ void __launch_bounds__(1024) csr_offsets_kernel(InertialArgs v, InertialCsr csr) {
  __shared__ long long s_tot[32][4];
  __shared__ long long s_carry[4];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < 4) s_carry[tid] = 0;
  __syncthreads();
  for (int base = 0; base < v.W; base += 1024) {
    const int w = base + tid;
    int nw = 0, ni = 0;
    long long q[4] = {0, 0, 0, 0};
    if (w < v.W) {
      nw = v.n_max > 0 ? min(max(v.prior_n[w], 0), v.n_max) : 0;
      ni = v.NI > 0 ? max(v.imu_window_offset[w + 1] - v.imu_window_offset[w], 0) : 0;   // null offsets when NI == 0
      q[0] = (nw > 0) + ni, q[1] = nw + 15LL * ni, q[2] = nw + 30LL * ni, q[3] = (long long)nw * nw + 450LL * ni;
    }
    long long inc[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      inc[u] = q[u];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const long long t = __shfl_up_sync(0xffffffffu, inc[u], o);
        if (lane >= o) inc[u] += t;
      }
    }
    if (lane == 31)
#pragma unroll
      for (int u = 0; u < 4; ++u) s_tot[warp][u] = inc[u];
    __syncthreads();
    if (warp == 0) {
      for (int u = 0; u < 4; ++u) {
        long long t = s_tot[lane][u];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const long long s = __shfl_up_sync(0xffffffffu, t, o);
          if (lane >= o) t += s;
        }
        s_tot[lane][u] = t;   // inclusive over warps
      }
    }
    __syncthreads();
    long long ex[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) ex[u] = s_carry[u] + (warp > 0 ? s_tot[warp - 1][u] : 0) + inc[u] - q[u];
    if (w < v.W) {
      const long long fb = ex[0], rb = ex[1], cb = ex[2], jb = ex[3];
      csr.window_offset[w] = (int32_t)fb;
      int k = (int)fb;
      if (nw > 0) {
        csr.row_offset[k] = rb, csr.col_offset[k] = cb, csr.jac_offset[k] = jb;
        ++k;
      }
      for (int t = 0; t < ni; ++t, ++k) {
        csr.row_offset[k] = rb + nw + 15LL * t;
        csr.col_offset[k] = cb + nw + 30LL * t;
        csr.jac_offset[k] = jb + (long long)nw * nw + 450LL * t;
      }
      if (w == v.W - 1) {   // the terminating entries
        csr.window_offset[v.W] = k;
        csr.row_offset[k] = rb + q[1], csr.col_offset[k] = cb + q[2], csr.jac_offset[k] = jb + q[3];
      }
    }
    __syncthreads();
    if (tid < 4) s_carry[tid] += s_tot[31][tid];
    __syncthreads();
  }
}

// MarginalizationFactor::Evaluate (marginalization_factor.cpp:335-384) of window w's prior.
__global__ void __launch_bounds__(128) prior_kernel(InertialArgs v, viml_inertial_out out, InertialCsr csr, bool offsets) {
  extern __shared__ double s_dx[];
  const int w = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = min(max(v.prior_n[w], 0), v.n_max);
  if (n == 0) return;
  const int nb = min(max(v.prior_n_blocks[w], 0), v.max_blocks), Dx = v.D + v.X;
  const bool to_csr = csr.row_offset != nullptr;
  const int k = to_csr ? csr.window_offset[w] : 0;
  const int64_t r0 = to_csr ? csr.row_offset[k] : 0, c0 = to_csr ? csr.col_offset[k] : 0, j0 = to_csr ? csr.jac_offset[k] : 0;
  for (int c = tid; c < n; c += blockDim.x) {
    s_dx[c] = 0.0;
    if (to_csr && offsets) csr.col_index[c0 + c] = min(c, Dx - 1);   // in range even for an invalid block list (device flavour)
  }
  __syncthreads();
  for (int b = tid; b < nb; b += blockDim.x) {
    const int32_t* blk = v.prior_block + ((size_t)w * v.max_blocks + b) * 4;
    const double* x0 = v.prior_x0 + ((size_t)w * v.max_blocks + b) * VIML_PRIOR_X0_STRIDE;
    const int kind = blk[0];
    const double* x;
    int tcol, size;
    if (kind == VIML_BLOCK_POSE) {
      const int idx = min(max(blk[1], 0), v.P - 1);
      x = v.poses + ((size_t)w * v.P + idx) * 7, tcol = 6 * idx, size = 7;
    } else if (kind == VIML_BLOCK_EX) {
      x = v.ex_pose + (size_t)w * 7, tcol = 6 * v.P, size = 7;
    } else {
      size = min(max(blk[2], 1), min(max(v.X, 1), VIML_PRIOR_X0_STRIDE));
      if (v.X == 0) continue;
      const int idx = min(max(blk[1], 0), v.X - size);
      x = v.extra + (size_t)w * v.X + idx, tcol = v.D + idx;
    }
    const int local = size == 7 ? 6 : size;
    const int first = min(max(blk[3], 0), n - local);
    if (first < 0) continue;
    if (size != 7) {
      for (int t = 0; t < size; ++t) s_dx[first + t] = x[t] - x0[t];                                   // :356
    } else {
      for (int t = 0; t < 3; ++t) s_dx[first + t] = x[t] - x0[t];                                      // :359
      const Q dq = qmul(qinv(quat(x0)), quat(x));                                                      // :360
      const double sg = (dq.w >= 0) ? 2.0 : -2.0;                                                      // :361-364
      s_dx[first + 3] = sg * dq.x, s_dx[first + 4] = sg * dq.y, s_dx[first + 5] = sg * dq.z;
    }
    if (to_csr && offsets)
      for (int t = 0; t < local; ++t) csr.col_index[c0 + first + t] = tcol + t;
  }
  __syncthreads();
  const double* __restrict__ J = v.prior_jacobian + (size_t)w * v.n_max * v.n_max;
  for (int r = warp; r < n; r += blockDim.x / 32) {   // :366  r = linearized_residuals + linearized_jacobians dx
    double s = 0.0;
    for (int c = lane; c < n; c += 32) s = fma(J[(size_t)r * v.n_max + c], s_dx[c], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
      const double res = v.prior_residual[(size_t)w * v.n_max + r] + s;
      if (out.prior_residual) out.prior_residual[(size_t)w * v.n_max + r] = res;
      if (to_csr) csr.residual[r0 + r] = res;
    }
  }
  if (to_csr && csr.jacobian)   // :371-380: the Jacobian is linearized_jacobians itself
    for (int e = tid; e < n * n; e += blockDim.x) {
      const int r = e / n, c = e - r * n;
      csr.jacobian[j0 + e] = J[(size_t)r * v.n_max + c];
    }
}

constexpr int kImuWarps = 4;

// IMUFactor::Evaluate (imu_factor.h:19-181) of factor f = one warp.
__global__ void __launch_bounds__(32 * kImuWarps) imu_kernel(InertialArgs v, viml_inertial_out out, InertialCsr csr, bool offsets,
                                                             bool want_jac) {
  __shared__ double s_info[kImuWarps][225];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t f = (int64_t)blockIdx.x * kImuWarps + warp;
  if (f >= v.NI) return;   // warp-uniform; only warp-level synchronisation below
  const double* __restrict__ info = v.imu_sqrt_info + f * 225;
  for (int e = lane; e < 225; e += 32) s_info[warp][e] = info[e];
  __syncwarp();
  if (!want_jac && lane != 30) return;
  // window of the factor: the last w with imu_window_offset[w] <= f
  int lo = 0, hi = v.W;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (v.imu_window_offset[mid] <= f) lo = mid;
    else hi = mid;
  }
  const int w = lo;
  const int pi = min(max(v.imu_pose[2 * f], 0), v.P - 1), pj = min(max(v.imu_pose[2 * f + 1], 0), v.P - 1);
  const int bi = min(max(v.imu_sb[2 * f], 0), max(v.X - 9, 0)), bj = min(max(v.imu_sb[2 * f + 1], 0), max(v.X - 9, 0));
  const double* __restrict__ xi = v.poses + ((size_t)w * v.P + pi) * 7;
  const double* __restrict__ xj = v.poses + ((size_t)w * v.P + pj) * 7;
  const double* __restrict__ si = v.extra + (size_t)w * v.X + bi;
  const double* __restrict__ sj = v.extra + (size_t)w * v.X + bj;
  const double* __restrict__ pre = v.imu_preint + f * 17;
  const double* __restrict__ jac = v.imu_jacobian + f * 225;
  const double dt = pre[0];
  const V Pi = vec(xi), Pj = vec(xj), Vi = vec(si), Vj = vec(sj);
  const Q Qi = quat(xi), Qj = quat(xj), Qii = qinv(Qi);
  const Q dq{pre[7], pre[4], pre[5], pre[6]};
  const V G{v.G[0], v.G[1], v.G[2]};
  const V dbg{si[6] - pre[14], si[7] - pre[15], si[8] - pre[16]};
  const int g = lane / 3, k = lane - 3 * (lane / 3);
  double col[15];
#pragma unroll
  for (int r = 0; r < 15; ++r) col[r] = 0.0;
  auto put = [&](int r0, V a) { col[r0] = a.x, col[r0 + 1] = a.y, col[r0 + 2] = a.z; };
  auto negv = [](V a) { return V{-a.x, -a.y, -a.z}; };
  // corrected_delta_q = delta_q * Utility::deltaQ(dq_dbg * dbg)   (integration_base.h evaluate)
  auto corrected_dq = [&]() {
    const V th = mul3(jac, O_R, O_BG, dbg);
    return qmul(dq, Q{1.0, 0.5 * th.x, 0.5 * th.y, 0.5 * th.z});
  };
  switch (g) {
    case 0:   // pose_i, position: [P] = -Ri^T
      put(O_P, negv(rotcol(Qii, k)));
      break;
    case 1: { // pose_i, rotation
      const V a = rot(Qii, V{0.5 * G.x * dt * dt + Pj.x - Pi.x - Vi.x * dt, 0.5 * G.y * dt * dt + Pj.y - Pi.y - Vi.y * dt,
                             0.5 * G.z * dt * dt + Pj.z - Pi.z - Vi.z * dt});
      put(O_P, skewcol(a, k));
      // -BR(Qleft(Qj^-1 Qi) Qright(cdq)) e_k = -(p_w u + p_v x u - p_v (q_v . e_k)),  u = q_w e_k - q_v x e_k
      const Q p = qmul(qinv(Qj), Qi), q = corrected_dq();
      const V qv{q.x, q.y, q.z}, pv{p.x, p.y, p.z}, ek = unit(k), qe = cross(qv, ek);
      const V u{q.w * ek.x - qe.x, q.w * ek.y - qe.y, q.w * ek.z - qe.z};
      const V pu = cross(pv, u);
      const double qk = comp(qv, k);
      put(O_R, V{-(p.w * u.x + pu.x - pv.x * qk), -(p.w * u.y + pu.y - pv.y * qk), -(p.w * u.z + pu.z - pv.z * qk)});
      const V b = rot(Qii, V{G.x * dt + Vj.x - Vi.x, G.y * dt + Vj.y - Vi.y, G.z * dt + Vj.z - Vi.z});
      put(O_V, skewcol(b, k));
      break;
    }
    case 2: { // sb_i, velocity: [P] = -Ri^T dt, [V] = -Ri^T
      const V c = rotcol(Qii, k);
      put(O_P, V{-c.x * dt, -c.y * dt, -c.z * dt});
      put(O_V, negv(c));
      break;
    }
    case 3:   // sb_i, Ba: [P] = -dp_dba, [V] = -dv_dba, [BA] = -I
      put(O_P, negv(jcol(jac, O_P, O_BA + k)));
      put(O_V, negv(jcol(jac, O_V, O_BA + k)));
      put(O_BA, negv(unit(k)));
      break;
    case 4: { // sb_i, Bg: [P] = -dp_dbg, [R] = -BR(Qleft(Qj^-1 Qi delta_q)) dq_dbg, [V] = -dv_dbg, [BG] = -I
      put(O_P, negv(jcol(jac, O_P, O_BG + k)));
      const Q s = qmul(qmul(qinv(Qj), Qi), dq);
      const V sv{s.x, s.y, s.z}, d = jcol(jac, O_R, O_BG + k), sd = cross(sv, d);
      put(O_R, V{-(s.w * d.x + sd.x), -(s.w * d.y + sd.y), -(s.w * d.z + sd.z)});
      put(O_V, negv(jcol(jac, O_V, O_BG + k)));
      put(O_BG, negv(unit(k)));
      break;
    }
    case 5:   // pose_j, position: [P] = Ri^T
      put(O_P, rotcol(Qii, k));
      break;
    case 6: { // pose_j, rotation: [R] = BR(Qleft(cdq^-1 Qi^-1 Qj))
      const Q s = qmul(qmul(qinv(corrected_dq()), Qii), Qj);
      const V sv{s.x, s.y, s.z}, ek = unit(k), se = cross(sv, ek);
      put(O_R, V{s.w * ek.x + se.x, s.w * ek.y + se.y, s.w * ek.z + se.z});
      break;
    }
    case 7:   // sb_j, velocity: [V] = Ri^T
      put(O_V, rotcol(Qii, k));
      break;
    case 8:
      put(O_BA, unit(k));   // constant row offsets only: col[] stays in registers
      break;
    case 9:
      put(O_BG, unit(k));
      break;
    default:
      if (lane == 30) {   // IntegrationBase::evaluate
        const V dba{si[3] - pre[11], si[4] - pre[12], si[5] - pre[13]};
        const V Bai{si[3], si[4], si[5]}, Bgi{si[6], si[7], si[8]}, Baj{sj[3], sj[4], sj[5]}, Bgj{sj[6], sj[7], sj[8]};
        const Q cdq = corrected_dq();
        const V a1 = mul3(jac, O_V, O_BA, dba), a2 = mul3(jac, O_V, O_BG, dbg);
        const V cdv{pre[8] + a1.x + a2.x, pre[9] + a1.y + a2.y, pre[10] + a1.z + a2.z};
        const V b1 = mul3(jac, O_P, O_BA, dba), b2 = mul3(jac, O_P, O_BG, dbg);
        const V cdp{pre[1] + b1.x + b2.x, pre[2] + b1.y + b2.y, pre[3] + b1.z + b2.z};
        const V rp = rot(Qii, V{0.5 * G.x * dt * dt + Pj.x - Pi.x - Vi.x * dt, 0.5 * G.y * dt * dt + Pj.y - Pi.y - Vi.y * dt,
                                0.5 * G.z * dt * dt + Pj.z - Pi.z - Vi.z * dt});
        put(O_P, V{rp.x - cdp.x, rp.y - cdp.y, rp.z - cdp.z});
        const Q e = qmul(qinv(cdq), qmul(Qii, Qj));
        put(O_R, V{2 * e.x, 2 * e.y, 2 * e.z});
        const V rv = rot(Qii, V{G.x * dt + Vj.x - Vi.x, G.y * dt + Vj.y - Vi.y, G.z * dt + Vj.z - Vi.z});
        put(O_V, V{rv.x - cdv.x, rv.y - cdv.y, rv.z - cdv.z});
        put(O_BA, V{Baj.x - Bai.x, Baj.y - Bai.y, Baj.z - Bai.z});
        put(O_BG, V{Bgj.x - Bgi.x, Bgj.y - Bgi.y, Bgj.z - Bgi.z});
      }
      break;
  }
  const double* __restrict__ S = s_info[warp];
  const bool to_csr = csr.row_offset != nullptr;
  int64_t ro = 0, co = 0, jo = 0;
  if (to_csr) {
    const int kf = csr.window_offset[w] + (v.n_max > 0 && v.prior_n[w] > 0 ? 1 : 0) + (int)(f - v.imu_window_offset[w]);
    ro = csr.row_offset[kf], co = csr.col_offset[kf], jo = csr.jac_offset[kf];
    if (offsets && lane < 30) {
      const int c = lane < 6 ? 6 * pi + lane : lane < 15 ? v.D + bi + lane - 6 : lane < 21 ? 6 * pj + lane - 15 : v.D + bj + lane - 21;
      csr.col_index[co + lane] = c;
    }
  }
  if (lane == 31) {   // column 6 of both pose blocks
    for (int r = 0; r < 15; ++r) {
      if (out.imu_jac_pose_i) out.imu_jac_pose_i[f * 105 + r * 7 + 6] = 0.0;
      if (out.imu_jac_pose_j) out.imu_jac_pose_j[f * 105 + r * 7 + 6] = 0.0;
    }
    return;
  }
  double* dst = nullptr;   // this lane's Ceres column
  int ld = 0;
  if (lane < 6) dst = out.imu_jac_pose_i ? out.imu_jac_pose_i + f * 105 + lane : nullptr, ld = 7;
  else if (lane < 15) dst = out.imu_jac_sb_i ? out.imu_jac_sb_i + f * 135 + lane - 6 : nullptr, ld = 9;
  else if (lane < 21) dst = out.imu_jac_pose_j ? out.imu_jac_pose_j + f * 105 + lane - 15 : nullptr, ld = 7;
  else if (lane < 30) dst = out.imu_jac_sb_j ? out.imu_jac_sb_j + f * 135 + lane - 21 : nullptr, ld = 9;
  else dst = out.imu_residual ? out.imu_residual + f * 15 : nullptr, ld = 1;
  double* cdst = !to_csr ? nullptr : lane < 30 ? (csr.jacobian ? csr.jacobian + jo + lane : nullptr) : csr.residual + ro;
  const int cld = lane < 30 ? 30 : 1;
#pragma unroll
  for (int r = 0; r < 15; ++r) {   // sqrt_info * column
    double s = 0.0;
#pragma unroll
    for (int q = 0; q < 15; ++q) s = fma(S[r * 15 + q], col[q], s);
    if (dst) dst[r * ld] = s;
    if (cdst) cdst[r * cld] = s;
  }
}

}  // namespace inertial

int viml_launch_inertial(viml_ctx* ctx, const InertialArgs& v, const viml_inertial_out& out, const InertialCsr& csr, bool offsets) {
  if (v.W == 0) return VIML_OK;
  const bool to_csr = csr.row_offset != nullptr;
  if (to_csr && offsets) {
    LaunchScope ls(ctx, K_GN);
    inertial::csr_offsets_kernel<<<1, 1024, 0, ctx->stream>>>(v, csr);
    VIML_TRY_CUDA(ctx, cudaGetLastError());
  }
  if (v.n_max > 0) {
    LaunchScope ls(ctx, K_GN);
    const int smem = v.n_max * (int)sizeof(double);
    if (smem > 48 * 1024)
      VIML_TRY_CUDA(ctx, cudaFuncSetAttribute(inertial::prior_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    inertial::prior_kernel<<<v.W, 128, smem, ctx->stream>>>(v, out, csr, offsets);
    VIML_TRY_CUDA(ctx, cudaGetLastError());
  }
  if (v.NI > 0) {
    const bool want_jac = (to_csr && csr.jacobian) || out.imu_jac_pose_i || out.imu_jac_sb_i || out.imu_jac_pose_j || out.imu_jac_sb_j ||
                          (to_csr && offsets);
    LaunchScope ls(ctx, K_GN);
    inertial::imu_kernel<<<(unsigned)((v.NI + inertial::kImuWarps - 1) / inertial::kImuWarps), 32 * inertial::kImuWarps, 0, ctx->stream>>>(
        v, out, csr, offsets, want_jac);
    VIML_TRY_CUDA(ctx, cudaGetLastError());
  }
  return VIML_OK;
}
