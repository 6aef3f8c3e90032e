// gn_kernels.cuh — the reduced system of the whole window and one Gauss-Newton / Levenberg-Marquardt iteration on it.
// Included by linearize_kernels.cu (uses eval_point / eval_line for the cost).
//
// Reference: what ceres::Solve(SPARSE_SCHUR) does per iteration with the problem Estimator::OptimizationWithLine builds
// (estimator.cpp:1677-1905): normal equations of all residual blocks, Schur elimination of the landmarks, a dense solve of
// the reduced camera system, PoseLocalParameterization::Plus (pose_local_parameterization.cpp:3-19).  The prior and the IMU
// factors enter as evaluated dense blocks (marginalization_factor.cpp:335-384, imu_factor.h:19-181), accumulated by the
// ThreadsConstructA rule (marginalization_factor.cpp:141-172): A += J_i^T J_j over the tangent columns, b += J_i^T r.
#pragma once

namespace gn {

// Factor k of a DenseArgs: n rows x c columns, its Jacobian (row-major), residual and tangent columns.
struct DenseFactor {
  int n, c;
  const double* J;
  const double* r;
  const int32_t* ci;
};
__device__ __forceinline__ DenseFactor dense_factor(const DenseArgs& dn, int k) {
  return {(int)(dn.row_offset[k + 1] - dn.row_offset[k]), (int)(dn.col_offset[k + 1] - dn.col_offset[k]), dn.jacobian + dn.jac_offset[k],
          dn.residual + dn.row_offset[k], dn.col_index + dn.col_offset[k]};
}

// Adds J_k^T J_k and J_k^T r_k of window w's dense-block factors, one factor after the other (two factors may share columns), by a
// CTA of 256 threads.  A factor's Jacobian is staged in sJ with a row stride of c_pad + 4 doubles (conflict-free fragment loads) and
// J^T J is formed as 8 x 8 tiles on the FP64 tensor pipe: the upper-triangle tiles dealt round-robin to the warps, ceil(n / 4) DMMA
// steps each.  A factor that does not fit the stage (cap doubles) takes the entry-by-entry loop, which counts as one diagonal tile.
// add(i, j, v, diag) adds entry (i, j) = (ci[a], ci[b]) of J^T J, the tile of column a at or left of b's, diag for a diagonal tile;
// LOWER: a diagonal tile hands over only its a >= b half.  J^T r is added into b.  kq = lane & 3, mq = lane >> 2: the thread's
// place in a DMMA fragment (the fused kernel has them at hand for its factorisation).
template <bool LOWER, class Add>
__device__ __forceinline__ void add_dense_factors(const DenseArgs& dn, int w, int cap, double* __restrict__ sJ, double* __restrict__ b,
                                                  int kq, int mq, Add add) {
  if (dn.ND == 0) return;
  const int tid = threadIdx.x, warp = tid >> 5;
  for (int k = dn.window_offset[w]; k < dn.window_offset[w + 1]; ++k) {
    const DenseFactor f = dense_factor(dn, k);
    const int n = f.n, c = f.c;
    const double* __restrict__ J = f.J;
    const double* __restrict__ r = f.r;
    const int32_t* __restrict__ ci = f.ci;
    const int np = (n + 3) & ~3, cp = (c + 7) & ~7, ld = cp + 4;
    if (np * ld + np <= cap) {
      double* __restrict__ sr = sJ + np * ld;   // the residual behind the Jacobian
      for (int e = tid; e < np * ld; e += 256) {
        const int q = e / ld, a = e - q * ld;
        sJ[e] = (q < n && a < c) ? J[(size_t)q * c + a] : 0.0;
      }
      for (int q = tid; q < np; q += 256) sr[q] = q < n ? r[q] : 0.0;
      __syncthreads();
      const int nt = cp >> 3, ntile = nt * (nt + 1) / 2;
      for (int t = warp; t < ntile; t += 8) {      // t-th tile of the upper triangle, row-major: row ta holds nt - ta tiles
        int rem = t, ta = 0;
        while (rem >= nt - ta) rem -= nt - ta, ++ta;
        const int tb = ta + rem;
        double c0 = 0.0, c1 = 0.0;
        const double* __restrict__ pa = sJ + kq * ld + 8 * ta + mq;
        const double* __restrict__ pb = sJ + kq * ld + 8 * tb + mq;
        for (int s4 = 0; s4 < np; s4 += 4) stream::dmma(c0, c1, pa[s4 * ld], pb[s4 * ld]);
        const int a = 8 * ta + mq, bb = 8 * tb + 2 * kq;
        if (a < c) {
          if (bb < c && (!LOWER || ta != tb || a >= bb)) add(ci[a], ci[bb], c0, ta == tb);
          if (bb + 1 < c && (!LOWER || ta != tb || a >= bb + 1)) add(ci[a], ci[bb + 1], c1, ta == tb);
        }
      }
      for (int a = tid; a < c; a += 256) {
        double v = 0.0;
        for (int q = 0; q < n; ++q) v = fma(sJ[q * ld + a], sr[q], v);
        b[ci[a]] += v;
      }
    } else {
      for (int e = tid; e < c * c; e += 256) {
        const int a = e / c, bb = e - a * c;
        if (LOWER && a < bb) continue;
        double v = 0.0;
        for (int q = 0; q < n; ++q) v = fma(J[(size_t)q * c + a], J[(size_t)q * c + bb], v);
        add(ci[a], ci[bb], v, true);
      }
      for (int a = tid; a < c; a += 256) {
        double v = 0.0;
        for (int q = 0; q < n; ++q) v = fma(J[(size_t)q * c + a], r[q], v);
        b[ci[a]] += v;
      }
    }
    __syncthreads();
  }
}

// Sx = embed(S) + sum_k J_k^T J_k,  gx = embed(g) + sum_k J_k^T r_k.  One CTA per window; an entry of an off-diagonal tile is added
// with its mirror.
constexpr int kReducedStage = 12288;   // doubles of dynamic shared memory (96 KB): a 76 x 75 prior needs 76 x 84

__global__ void __launch_bounds__(256) reduced_kernel(int D, DenseArgs dn, const double* __restrict__ S, const double* __restrict__ g,
                                                      double* __restrict__ Sx, double* __restrict__ gx) {
  extern __shared__ __align__(16) double sJ[];
  const int w = blockIdx.x, tid = threadIdx.x, lane = tid & 31, Dx = D + dn.X;
  double* __restrict__ A = Sx + (size_t)w * Dx * Dx;
  double* __restrict__ b = gx + (size_t)w * Dx;
  const double* __restrict__ Sw = S + (size_t)w * D * D;
  for (int e = tid; e < Dx * Dx; e += blockDim.x) {
    const int r = e / Dx, c = e - r * Dx;
    A[e] = (r < D && c < D) ? Sw[r * D + c] : 0.0;
  }
  for (int e = tid; e < Dx; e += blockDim.x) b[e] = e < D ? g[(size_t)w * D + e] : 0.0;
  __syncthreads();
  add_dense_factors<false>(dn, w, kReducedStage, sJ, b, lane & 3, lane >> 2, [=](int i, int j, double v, bool diag) {
    A[(size_t)i * Dx + j] += v;
    if (!diag) A[(size_t)j * Dx + i] += v;
  });
}

// ---- tiled Cholesky solve ---------------------------------------------------------------------------------------------------------
// solve_tiled_kernel: (Sx + lambda diag Sx) dx = -gx, one CTA (8 warps) per window, the matrix held in shared memory as the lower
// triangle of 8 x 8 tiles (tile (I, J), J <= I, at (I (I + 1) / 2 + J) * 64; Dx padded to a multiple of 8 with an identity
// diagonal).  Right-looking blocked factorisation: per tile column K (1) warp 0 factors the diagonal tile, (2) one thread per row
// solves the panel rows against it, (3) the trailing tiles take A[I][J] -= L[I][K] L[J][K]^T as two DMMA steps each, dealt
// round-robin to warps 1..7 while warp 0 updates and factors the next diagonal tile (look-ahead).  22 tile columns and ~44 barriers
// for Dx = 171, and the O(n^3) part runs on the FP64 tensor pipe.  Forward / backward substitution tile by tile.
// solved[w] = 0 when a pivot is not positive (dx = 0 then).  cost[3w + 2] = -gx.dx - 1/2 dx.Sx.dx (undamped model).
// FUSED: the matrix is not read from Sx but built in place — embed(S) plus the window's dense-block factors through
// add_dense_factors, like reduced_kernel, with a stage of kFusedStage doubles — so that Sx never makes its 234 KB round trip through
// HBM; the model decrease then uses A x = -g:  x^T Sx x = -g.x - lambda sum d_i x_i^2  with d the undamped diagonal.  A step takes
// the fused kernel where its shared memory fits (gn_fused_takes in common.cuh: Dx <= 200) and the caller does not want Sx / gx;
// otherwise reduced_kernel writes Sx / gx and the unfused kernel solves them.
constexpr int kTile = 8;
__device__ __forceinline__ int tile_at(int I, int J) { return (I * (I + 1) / 2 + J) * 64; }

// lambda_w (nullable): a damping per window instead of `lambda`; running (nullable): a window with running[w] == 0 is skipped
// (its CTA returns at once and writes nothing); damp (nullable): (Sx + diag(damp_w)) dx = -gx, an additive damping per column
// instead of lambda diag(Sx).
template <bool FUSED>
__global__ void __launch_bounds__(256) solve_tiled_kernel(int Dx, double lambda, const double* __restrict__ Sx, const double* __restrict__ gx,
                                                          double* __restrict__ dx, int32_t* __restrict__ solved, double* __restrict__ cost,
                                                          int D, DenseArgs dn, const double* __restrict__ S, const double* __restrict__ g,
                                                          const double* __restrict__ lambda_w, const int32_t* __restrict__ running,
                                                          const double* __restrict__ damp) {
  extern __shared__ __align__(16) double sm[];
  __shared__ int s_ok;
  __shared__ double s_red[8], s_dinv[kTile];
  const int w = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (running && !running[w]) return;
  if (lambda_w) lambda = lambda_w[w];
  const double* __restrict__ dmp = damp ? damp + (size_t)w * Dx : nullptr;
  const int NB = (Dx + kTile - 1) / kTile, Dp = NB * kTile;
  double* __restrict__ L = sm;                                   // NB (NB + 1) / 2 tiles
  double* __restrict__ y = sm + (size_t)NB * (NB + 1) / 2 * 64;  // [Dp]
  double* __restrict__ gv = y + Dp;                              // FUSED: [Dp] the right-hand side's g, [Dp] the undamped diagonal,
  double* __restrict__ dv = gv + Dp;                             //        then the Jacobian stage
  double* __restrict__ sJ = dv + Dp;
  const double* __restrict__ A = FUSED ? nullptr : Sx + (size_t)w * Dx * Dx;
  for (int e = tid; e < Dp * Dp; e += 256) {   // padding rows: identity; everything else starts at zero
    const int i = e / Dp, j = e - i * Dp;
    if (j <= i) L[tile_at(i >> 3, j >> 3) + (i & 7) * 8 + (j & 7)] = (i >= Dx && i == j) ? 1.0 : 0.0;
  }
  __syncthreads();
  const int kq = lane & 3, mq = lane >> 2;
  if (FUSED) {
    // embed(S): the landmark Schur complement of the window is exactly symmetric (every tile is written with its mirror)
    const double* __restrict__ Sw = S + (size_t)w * D * D;
    for (int e0 = tid; e0 < D * D; e0 += 4 * 256) {
      double v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = e0 + u * 256 < D * D ? Sw[e0 + u * 256] : 0.0;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = e0 + u * 256;
        if (e >= D * D) break;
        const int i = e / D, j = e - i * D;
        if (j <= i) L[tile_at(i >> 3, j >> 3) + (i & 7) * 8 + (j & 7)] = v[u];
      }
    }
    for (int e = tid; e < Dp; e += 256) gv[e] = e < D ? g[(size_t)w * D + e] : 0.0;
    __syncthreads();
    // entry (i, j) and its mirror land on the same lower-triangle slot: off-diagonal tiles add once, a diagonal tile (which holds
    // both) the a >= b half
    add_dense_factors<true>(dn, w, kFusedStage, sJ, gv, kq, mq, [=](int i, int j, double v, bool) {
      const int hi = max(i, j), lo = min(i, j);
      L[tile_at(hi >> 3, lo >> 3) + (hi & 7) * 8 + (lo & 7)] += v;
    });
    for (int i = tid; i < Dp; i += 256) {
      double& d = L[tile_at(i >> 3, i >> 3) + (i & 7) * 8 + (i & 7)];
      dv[i] = d;
      if (i < Dx) {
        if (dmp) d += dmp[i];
        else d *= 1.0 + lambda;
      }
      y[i] = -gv[i];
    }
  } else {
    // (A + A^T) / 2 into the tiles with row-wise (coalesced) reads only: the lower entries first, then every upper entry adds
    // its half to its mirror (one writer per entry in either pass); four independent loads in flight per thread and pass
    for (int pass = 0; pass < 2; ++pass) {
      for (int e0 = tid; e0 < Dx * Dx; e0 += 4 * 256) {
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = e0 + u * 256 < Dx * Dx ? A[e0 + u * 256] : 0.0;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int e = e0 + u * 256;
          if (e >= Dx * Dx) break;
          const int i = e / Dx, j = e - i * Dx;
          if (pass == 0 && j <= i)
            L[tile_at(i >> 3, j >> 3) + (i & 7) * 8 + (j & 7)] = (i == j) ? (dmp ? v[u] + dmp[i] : v[u] * (1.0 + lambda)) : 0.5 * v[u];
          if (pass == 1 && j > i) L[tile_at(j >> 3, i >> 3) + (j & 7) * 8 + (i & 7)] += 0.5 * v[u];
        }
      }
      __syncthreads();
    }
    for (int e = tid; e < Dp; e += 256) y[e] = e < Dx ? -gx[(size_t)w * Dx + e] : 0.0;
  }
  __syncthreads();
  // the strictly upper part of the diagonal tiles is never read as data but is multiplied in the DMMA steps: zero it
  for (int e = tid; e < NB * 64; e += 256) {
    const int I = e >> 6, r = (e >> 3) & 7, c = e & 7;
    if (c > r) L[tile_at(I, I) + r * 8 + c] = 0.0;
  }
  if (tid == 0) s_ok = 1;
  __syncthreads();
  // 8 x 8 Cholesky of a diagonal tile by one warp: column by column, lane = row for the scaling, lanes over the 64 entries for
  // the update; leaves 1 / L[j][j] in s_dinv.  Clears s_ok on a non-positive pivot.
  auto factor_diag = [&](double* __restrict__ Dk) {
    for (int j = 0; j < kTile; ++j) {
      const double d = Dk[j * 8 + j];
      const bool good = d > 0.0 && isfinite(d);
      const double sd = good ? sqrt(d) : 1.0, inv = good ? rsqrt(d) : 1.0;
      __syncwarp();
      if (!good && lane == 0) s_ok = 0;
      if (lane < kTile && lane >= j) Dk[lane * 8 + j] = (lane == j) ? sd : Dk[lane * 8 + j] * inv;
      if (lane == 0) s_dinv[j] = inv;
      __syncwarp();
      for (int e = lane; e < 64; e += 32) {
        const int r = e >> 3, c = e & 7;
        if (c > j && r >= c) Dk[r * 8 + c] -= Dk[r * 8 + j] * Dk[c * 8 + j];
      }
      __syncwarp();
    }
  };
  if (warp == 0) factor_diag(L + tile_at(0, 0));
  __syncthreads();
  for (int K = 0; K < NB && s_ok; ++K) {   // s_ok is only written between the barriers below: uniform
    const double* __restrict__ Dk = L + tile_at(K, K);
    // panel: row `tid` of the tiles below the diagonal one solves x L_KK^T = a (forward substitution over the 8 columns)
    const int nrows = (NB - K - 1) * kTile;
    if (tid < nrows) {
      double* __restrict__ a = L + tile_at(K + 1 + (tid >> 3), K) + (tid & 7) * 8;
      double x[kTile];
#pragma unroll
      for (int c = 0; c < kTile; ++c) {
        double v = a[c];
#pragma unroll
        for (int k = 0; k < c; ++k) v -= x[k] * Dk[c * 8 + k];
        x[c] = v * s_dinv[c];
      }
#pragma unroll
      for (int c = 0; c < kTile; ++c) a[c] = x[c];
    }
    __syncthreads();
    // trailing update on the tensor pipe: tile (I, J), K < J <= I, of the m x m lower triangle (row-major index t).  Warp 0 takes
    // tile 0 — the next diagonal tile — and factors it at once (look-ahead: the serial 8-column factorisation runs beside the
    // other warps' tiles instead of in front of a barrier); warps 1..7 share the rest.
    {
      const int m = NB - K - 1;
      auto update = [&](int I, int J) {
        const double* __restrict__ Li = L + tile_at(K + 1 + I, K);
        const double* __restrict__ Lj = L + tile_at(K + 1 + J, K);
        double2* cptr = reinterpret_cast<double2*>(L + tile_at(K + 1 + I, K + 1 + J) + mq * 8 + 2 * kq);
        double2 c = *cptr;
        stream::dmma(c.x, c.y, -Li[mq * 8 + kq], Lj[mq * 8 + kq]);
        stream::dmma(c.x, c.y, -Li[mq * 8 + 4 + kq], Lj[mq * 8 + 4 + kq]);
        *cptr = c;
      };
      if (warp == 0) {
        if (m > 0) {
          update(0, 0);
          __syncwarp();
          factor_diag(L + tile_at(K + 1, K + 1));
        }
      } else {
        int t = warp, I = 0;                 // tiles 1, 2, ...: t = 1 + (warp - 1), step 7
        while (I < m && t >= I + 1) t -= I + 1, ++I;
        int J = t;
        while (I < m) {
          update(I, J);
          J += 7;
          while (I < m && J > I) J -= I + 1, ++I;
        }
      }
    }
    __syncthreads();
  }
  const bool ok = s_ok != 0;
  if (ok) {
    // forward L z = y: diagonal tile by warp 0 (serial over its 8 rows), then one thread per row below
    for (int K = 0; K < NB; ++K) {
      const double* __restrict__ Dk = L + tile_at(K, K);
      if (tid == 0) {
#pragma unroll
        for (int r = 0; r < kTile; ++r) {
          double v = y[K * 8 + r];
          for (int k = 0; k < r; ++k) v -= Dk[r * 8 + k] * y[K * 8 + k];
          y[K * 8 + r] = v / Dk[r * 8 + r];
        }
      }
      __syncthreads();
      const int nrows = (NB - K - 1) * kTile;
      if (tid < nrows) {
        const double* __restrict__ a = L + tile_at(K + 1 + (tid >> 3), K) + (tid & 7) * 8;
        double v = y[(K + 1) * 8 + tid];
#pragma unroll
        for (int c = 0; c < kTile; ++c) v -= a[c] * y[K * 8 + c];
        y[(K + 1) * 8 + tid] = v;
      }
      __syncthreads();
    }
    // backward L^T x = z: diagonal tile, then every entry above takes its share of this tile row
    for (int K = NB - 1; K >= 0; --K) {
      const double* __restrict__ Dk = L + tile_at(K, K);
      if (tid == 0) {
#pragma unroll
        for (int r = kTile - 1; r >= 0; --r) {
          double v = y[K * 8 + r];
          for (int k = r + 1; k < kTile; ++k) v -= Dk[k * 8 + r] * y[K * 8 + k];
          y[K * 8 + r] = v / Dk[r * 8 + r];
        }
      }
      __syncthreads();
      if (tid < K * kTile) {   // y[8 J + c] -= sum_r L[K][J][r][c] y[8 K + r]
        const double* __restrict__ a = L + tile_at(K, tid >> 3) + (tid & 7);
        double v = y[tid];
#pragma unroll
        for (int r = 0; r < kTile; ++r) v -= a[r * 8] * y[K * 8 + r];
        y[tid] = v;
      }
      __syncthreads();
    }
  }
  // model decrease with the undamped Sx: -g.x - x.Sx x / 2 (exactly 0 for a window that was not solved, even when its system
  // holds a NaN or an infinity)
  double part = 0.0;
  if (FUSED) {   // (Sx + lambda diag d) x = -g  =>  x.Sx x = -g.x - lambda sum d_i x_i^2  (damp_i in place of lambda d_i)
    for (int i = tid; i < Dx; i += 256) {
      const double xi = ok ? y[i] : 0.0;
      if (ok) part += -0.5 * gv[i] * xi + 0.5 * (dmp ? dmp[i] : lambda * dv[i]) * xi * xi;
      dx[(size_t)w * Dx + i] = xi;
    }
  } else {       // a warp per row of Sx (coalesced), lanes over the columns
    for (int i = warp; i < Dx; i += 8) {
      double sx = 0.0;
      if (ok)
        for (int c = lane; c < Dx; c += 32) sx = fma(A[(size_t)i * Dx + c], y[c], sx);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sx += __shfl_xor_sync(0xffffffffu, sx, o);
      const double xi = ok ? y[i] : 0.0;
      if (lane == 0) {
        if (ok) part += -gx[(size_t)w * Dx + i] * xi - 0.5 * xi * sx;
        dx[(size_t)w * Dx + i] = xi;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  if (lane == 0) s_red[warp] = part;
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int k = 0; k < 8; ++k) t += s_red[k];
    cost[3 * (size_t)w + 2] = t;
    solved[w] = ok ? 1 : 0;
  }
}

__device__ __forceinline__ void pose_plus(const double* __restrict__ x, const double* __restrict__ d, double* __restrict__ o) {
  // PoseLocalParameterization::Plus: p = _p + dp; q = (_q * Utility::deltaQ(dtheta)).normalized()
  o[0] = x[0] + d[0], o[1] = x[1] + d[1], o[2] = x[2] + d[2];
  const double ax = x[3], ay = x[4], az = x[5], aw = x[6];
  const double bx = 0.5 * d[3], by = 0.5 * d[4], bz = 0.5 * d[5], bw = 1.0;   // deltaQ: (1, theta/2), not normalised
  const double w = aw * bw - ax * bx - ay * by - az * bz;
  const double qx = aw * bx + ax * bw + ay * bz - az * by;
  const double qy = aw * by + ay * bw + az * bx - ax * bz;
  const double qz = aw * bz + az * bw + ax * by - ay * bx;
  const double n = sqrt(qx * qx + qy * qy + qz * qz + w * w);
  o[3] = qx / n, o[4] = qy / n, o[5] = qz / n, o[6] = w / n;
}

// New state of every window: poses / extrinsic by Plus, landmarks by back-substitution (or by the increments dl_in when given),
// extra state by addition.  running (nullable): windows with running[w] == 0 are skipped.
__global__ void __launch_bounds__(128) update_kernel(LinearizeArgs A, int X, const double* __restrict__ extra_in, const double* __restrict__ dx,
                                                     const int32_t* __restrict__ solved, double* __restrict__ o_poses,
                                                     double* __restrict__ o_ex, double* __restrict__ o_dep, double* __restrict__ o_extra,
                                                     const int32_t* __restrict__ running, const double* __restrict__ dl_in) {
  const int w = blockIdx.x, tid = threadIdx.x, P = A.P, F = A.F, D = A.D, Dx = D + X;
  if (running && !running[w]) return;
  const bool ok = solved[w] != 0;
  const double* __restrict__ d = dx + (size_t)w * Dx;
  for (int p = tid; p <= P; p += blockDim.x) {
    const double* x = p < P ? A.poses + ((size_t)w * P + p) * 7 : A.ex_pose + (size_t)w * 7;
    double* o = p < P ? o_poses + ((size_t)w * P + p) * 7 : o_ex + (size_t)w * 7;
    if (ok) {
      pose_plus(x, d + 6 * p, o);
    } else {
      for (int k = 0; k < 7; ++k) o[k] = x[k];
    }
  }
  for (int l = tid; l < F; l += blockDim.x) {
    const double lam = A.inv_depth[(size_t)w * F + l];
    double dl = 0.0;
    const double hll = dl_in ? 0.0 : A.out.H_ll[(size_t)w * F + l];
    if (ok && dl_in) {
      dl = dl_in[(size_t)w * F + l];
    } else if (ok && hll > 1e-8) {
      const double* __restrict__ row = A.out.H_lp + ((size_t)w * F + l) * D;
      double s = A.out.b_l[(size_t)w * F + l];
      for (int c = 0; c < D; ++c) s = fma(row[c], d[c], s);
      dl = -s / hll;
    }
    o_dep[(size_t)w * F + l] = ok ? lam + dl : lam;   // not lam + 0.0, which turns -0.0 into +0.0
  }
  if (o_extra)
    for (int e = tid; e < X; e += blockDim.x) {
      const double x = extra_in ? extra_in[(size_t)w * X + e] : 0.0;
      o_extra[(size_t)w * X + e] = ok ? x + d[D + e] : x;
    }
}

// cost[3w + slot] = 1/2 sum rho(|r|^2) over the window's point and line factors at the state of A (pose cache ready)
// + 1/2 sum |r_k + J_k dx|^2 over its dense-block factors (dx == nullptr, or a window the step did not solve: at the
// linearisation point, so that cost[1] == cost[0] even when a Jacobian holds a NaN).  running (nullable): windows with
// running[w] == 0 are skipped.
__global__ void __launch_bounds__(128) cost_kernel(LinearizeArgs A, DenseArgs dn, const double* __restrict__ dx,
                                                   const int32_t* __restrict__ solved, int slot, double* __restrict__ cost,
                                                   const int32_t* __restrict__ running) {
  __shared__ double s_red[4];
  const int w = blockIdx.x, tid = threadIdx.x, Dx = A.D + dn.X;
  if (running && !running[w]) return;
  const bool moved = dx != nullptr && solved[w] != 0;
  const bool cauchy = (A.flags & VIML_LOSS_CAUCHY) != 0;
  LinearizeArgs R = A;
  R.flags &= ~VIML_LOSS_CAUCHY;   // raw residuals: rho is applied here, not the Jacobian correction
  const double a2 = A.cauchy_a * A.cauchy_a;
  const double* cw = A.cache + (size_t)w * (A.P * kPoseCache + kExCache);
  double acc = 0.0;
  for (int64_t k = A.pf_window_offset[w] + tid; k < A.pf_window_offset[w + 1]; k += blockDim.x) {
    const uint32_t pk = A.pf_idx[k];
    const int i = pk & 0xff, j = (pk >> 8) & 0xff, f = pk >> 16;
    if (i >= A.P || j >= A.P || f >= A.F) continue;
    const double4 ob = reinterpret_cast<const double4*>(A.pf_obs)[k];
    PointJac J;
    eval_point(R, cw, i, j, A.inv_depth[(size_t)w * A.F + f], ob.x, ob.y, A.pf_pts_i_z ? A.pf_pts_i_z[k] : 1.0, ob.z, ob.w, J);
    const double s = J.r[0] * J.r[0] + J.r[1] * J.r[1];
    acc += cauchy ? a2 * log(1.0 + s / a2) : s;
  }
  if (A.NL > 0)
    for (int64_t k = A.lf_window_offset[w] + tid; k < A.lf_window_offset[w + 1]; k += blockDim.x) {
      const int frame = A.lf_frame[k];
      if (frame < 0 || frame >= A.P) continue;
      double g9[9];
#pragma unroll
      for (int c = 0; c < 9; ++c) g9[c] = A.lf_geom[(size_t)c * A.NL_stride + k];
      LineJac J;
      eval_line(R, cw, frame, g9, J);
      const double s = J.r[0] * J.r[0] + J.r[1] * J.r[1];
      acc += cauchy ? a2 * log(1.0 + s / a2) : s;
    }
  if (dn.ND > 0)
    for (int k = dn.window_offset[w]; k < dn.window_offset[w + 1]; ++k) {
      const DenseFactor f = dense_factor(dn, k);
      for (int q = tid; q < f.n; q += blockDim.x) {
        double v = f.r[q];
        if (moved)
          for (int a = 0; a < f.c; ++a) v = fma(f.J[(size_t)q * f.c + a], dx[(size_t)w * Dx + f.ci[a]], v);
        acc += v * v;
      }
    }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((tid & 31) == 0) s_red[tid >> 5] = acc;
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int k = 0; k < (int)blockDim.x / 32; ++k) t += s_red[k];
    cost[3 * (size_t)w + slot] = 0.5 * t;
  }
}

// ---- the dogleg strategy of viml_solve_vi (VIML_SOLVE_DOGLEG, viml.h) -----------------------------------------------------------
// The full problem has N = Dx + F columns; H is the loss-corrected visual J^T J (H_pp, H_lp, diagonal H_ll) plus the dense-block
// factors' J^T J, g = J^T r.  A landmark with H_ll <= 1e-8 takes no part (the Schur step's eps rule): its entries are 0 throughout.
// Every reduction below has a fixed order (per thread, then the warp's shuffle tree, then the warps in order), so a window's result
// depends on nothing but its own inputs.
constexpr double kDoglegEps = 1e-8;

// The sum over the CTA of one value per thread (NW warps), in a fixed order; every thread gets it.
template <int NW>
__device__ __forceinline__ double cta_sum(double v, double* s_red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if (lane == 0) s_red[warp] = v;
  __syncthreads();
  double t = 0.0;
#pragma unroll
  for (int k = 0; k < NW; ++k) t += s_red[k];
  return t;
}

__device__ __forceinline__ double dogleg_d(double s, double h) {   // Ceres' D-space diagonal of the scaled column
  return sqrt(fmin(fmax(s * s * h, 1e-6), 1e32));
}

// Kernel A, fresh windows, after the assembly and the inertial evaluation at x and before the Schur step: diag(H), g, s (round 0),
// d, gamma, w, |gamma|^2, w^T H w, the damping of the reduced columns, and the damping of the landmark columns added to H_ll (whose
// undamped values are kept in g.hll).
__global__ void __launch_bounds__(256) dogleg_prepare_kernel(LinearizeArgs A, DenseArgs dn, DoglegArgs G, const SolveState* __restrict__ state,
                                                             int round) {
  __shared__ double s_h[kMaxDx], s_g[kMaxDx], s_w[kMaxDx], s_red[8];
  const int w = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (round > 0 && !G.fresh[w]) return;
  const int D = A.D, F = A.F, Dx = G.Dx, N = Dx + F;
  const double mu = round > 0 ? state[w].mu : kDoglegMinMu;
  const double* __restrict__ Hpp = A.out.H_pp + (size_t)w * D * D;
  const double* __restrict__ Hlp = A.out.H_lp + (size_t)w * F * D;
  double* __restrict__ Hll = A.out.H_ll + (size_t)w * F;
  const double* __restrict__ bl = A.out.b_l + (size_t)w * F;
  double *sw = G.s + (size_t)w * N, *dw = G.d + (size_t)w * N, *gw = G.gamma + (size_t)w * N, *ww = G.w + (size_t)w * N;
  for (int i = tid; i < Dx; i += 256) {
    s_h[i] = i < D ? Hpp[(size_t)i * D + i] : 0.0;
    s_g[i] = i < D ? A.out.b_p[(size_t)w * D + i] : 0.0;
  }
  __syncthreads();
  if (dn.ND > 0)   // one factor after the other; inside a factor every column is a different one
    for (int k = dn.window_offset[w]; k < dn.window_offset[w + 1]; ++k) {
      const DenseFactor f = dense_factor(dn, k);
      for (int a = tid; a < f.c; a += 256) {
        double hh = 0.0, gg = 0.0;
        for (int q = 0; q < f.n; ++q) {
          const double j = f.J[(size_t)q * f.c + a];
          hh = fma(j, j, hh);
          gg = fma(j, f.r[q], gg);
        }
        s_h[f.ci[a]] += hh;
        s_g[f.ci[a]] += gg;
      }
      __syncthreads();
    }
  double gg = 0.0, whw = 0.0;
  for (int i = tid; i < Dx; i += 256) {
    const double h = s_h[i];
    if (round == 0) sw[i] = 1.0 / (1.0 + sqrt(h));
    const double si = sw[i], di = dogleg_d(si, h);
    const double gam = si * s_g[i] / di, wi = si * gam / di;
    dw[i] = di, gw[i] = gam, ww[i] = wi, s_w[i] = wi;
    G.damp[(size_t)w * Dx + i] = mu * (di * di) / (si * si);
    gg += gam * gam;
  }
  for (int l = tid; l < F; l += 256) {
    const double h = Hll[l];
    G.hll[(size_t)w * F + l] = h;
    if (round == 0) sw[Dx + l] = 1.0 / (1.0 + sqrt(h));
    double di = 0.0, gam = 0.0, wl = 0.0;
    if (h > kDoglegEps) {
      const double si = sw[Dx + l];
      di = dogleg_d(si, h);
      gam = si * bl[l] / di, wl = si * gam / di;
      Hll[l] = h + mu * (di * di) / (si * si);
      gg += gam * gam;
      whw += h * wl * wl;
    }
    dw[Dx + l] = di, gw[Dx + l] = gam, ww[Dx + l] = wl;
  }
  __syncthreads();
  for (int i = warp; i < D; i += 8) {   // w_p^T H_pp w_p: a warp per row
    double t = 0.0;
    for (int c = lane; c < D; c += 32) t = fma(Hpp[(size_t)i * D + c], s_w[c], t);
    whw += t * s_w[i];
  }
  for (int l = warp; l < F; l += 8) {   // 2 w_l (H_lp w_p)_l
    const double wl = ww[Dx + l];
    if (wl == 0.0) continue;
    double t = 0.0;
    for (int c = lane; c < D; c += 32) t = fma(Hlp[(size_t)l * D + c], s_w[c], t);
    whw += 2.0 * wl * t;
  }
  if (dn.ND > 0)   // |J_k w|^2
    for (int k = dn.window_offset[w]; k < dn.window_offset[w + 1]; ++k) {
      const DenseFactor f = dense_factor(dn, k);
      for (int q = tid; q < f.n; q += 256) {
        double v = 0.0;
        for (int a = 0; a < f.c; ++a) v = fma(f.J[(size_t)q * f.c + a], s_w[f.ci[a]], v);
        whw += v * v;
      }
    }
  gg = cta_sum<8>(gg, s_red);
  whw = cta_sum<8>(whw, s_red);
  if (tid == 0) G.scal[(size_t)w * kDoglegScal + 0] = gg, G.scal[(size_t)w * kDoglegScal + 3] = whw;
}

// Kernel B, fresh windows, after the solve of the damped reduced system (dx): the landmarks back-substituted with the damped H_ll
// (still in A.out.H_ll), the Gauss-Newton step dgn stored, n = d dgn / s, and n.n, gamma.n, w^T H dgn, dgn^T H dgn, valid.
__global__ void __launch_bounds__(256) dogleg_finish_kernel(LinearizeArgs A, DenseArgs dn, DoglegArgs G, const SolveState* __restrict__ state,
                                                            int round, const double* __restrict__ dx, const int32_t* __restrict__ solved) {
  __shared__ double s_d[kMaxDx], s_w[kMaxDx], s_red[8];
  const int w = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (round > 0 && !G.fresh[w]) return;
  const int D = A.D, F = A.F, Dx = G.Dx, N = Dx + F;
  const double mu = round > 0 ? state[w].mu : kDoglegMinMu;
  const double* __restrict__ Hpp = A.out.H_pp + (size_t)w * D * D;
  const double* __restrict__ Hlp = A.out.H_lp + (size_t)w * F * D;
  const double* __restrict__ Hd = A.out.H_ll + (size_t)w * F;
  const double* __restrict__ bl = A.out.b_l + (size_t)w * F;
  const double* __restrict__ h0 = G.hll + (size_t)w * F;
  const double *sw = G.s + (size_t)w * N, *dw = G.d + (size_t)w * N, *gw = G.gamma + (size_t)w * N, *ww = G.w + (size_t)w * N;
  double* __restrict__ gn = G.gn + (size_t)w * N;
  double nn = 0.0, gnn = 0.0, whd = 0.0, dhd = 0.0;
  for (int i = tid; i < Dx; i += 256) {
    const double v = dx[(size_t)w * Dx + i];
    s_d[i] = v, s_w[i] = ww[i], gn[i] = v;
    const double n = dw[i] * v / sw[i];
    nn += n * n;
    gnn += gw[i] * n;
  }
  __syncthreads();
  for (int i = warp; i < D; i += 8) {   // (H_pp dgn_p)_i against w_i and dgn_i
    double t = 0.0;
    for (int c = lane; c < D; c += 32) t = fma(Hpp[(size_t)i * D + c], s_d[c], t);
    whd += s_w[i] * t, dhd += s_d[i] * t;   // the lanes' partial sums
  }
  for (int l = warp; l < F; l += 8) {
    double td = 0.0, tw = 0.0;
    for (int c = lane; c < D; c += 32) {
      const double h = Hlp[(size_t)l * D + c];
      td = fma(h, s_d[c], td);
      tw = fma(h, s_w[c], tw);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) td += __shfl_xor_sync(0xffffffffu, td, o), tw += __shfl_xor_sync(0xffffffffu, tw, o);
    if (lane == 0) {
      const double h = h0[l];
      double v = 0.0;
      if (h > kDoglegEps) {
        v = -(bl[l] + td) / Hd[l];
        const double wl = ww[Dx + l], n = dw[Dx + l] * v / sw[Dx + l];
        nn += n * n;
        gnn += gw[Dx + l] * n;
        whd += wl * td + v * tw + h * wl * v;
        dhd += 2.0 * v * td + h * v * v;
      }
      gn[Dx + l] = v;
    }
  }
  if (dn.ND > 0)   // (J_k w) . (J_k dgn) and |J_k dgn|^2
    for (int k = dn.window_offset[w]; k < dn.window_offset[w + 1]; ++k) {
      const DenseFactor f = dense_factor(dn, k);
      for (int q = tid; q < f.n; q += 256) {
        double jw = 0.0, jd = 0.0;
        for (int a = 0; a < f.c; ++a) {
          const double j = f.J[(size_t)q * f.c + a];
          jw = fma(j, s_w[f.ci[a]], jw);
          jd = fma(j, s_d[f.ci[a]], jd);
        }
        whd += jw * jd;
        dhd += jd * jd;
      }
    }
  nn = cta_sum<8>(nn, s_red);
  gnn = cta_sum<8>(gnn, s_red);
  whd = cta_sum<8>(whd, s_red);
  dhd = cta_sum<8>(dhd, s_red);
  if (tid == 0) {
    double* sc = G.scal + (size_t)w * kDoglegScal;
    sc[1] = nn, sc[2] = gnn, sc[4] = whd, sc[5] = dhd;
    sc[6] = (solved[w] && mu < kDoglegMaxMu) ? 1.0 : 0.0;
  }
}

// Kernel C, running windows: Ceres' traditional dogleg step at the current radius from the stored scalars (scalar __d*_rn arithmetic,
// restated by tests/dogleg_policy.py), as a w + b dgn: its reduced part into dx, its landmark part into G.dl, its model decrease
// -(g.step + step^T H step / 2) into cost[3w + 2], its D-space norm into scal[7] and its validity into solved.
__global__ void __launch_bounds__(128) dogleg_step_kernel(DoglegArgs G, const SolveState* __restrict__ state, double initial_radius, int round,
                                                          const int32_t* __restrict__ running, double* __restrict__ dx,
                                                          double* __restrict__ cost, int32_t* __restrict__ solved) {
  __shared__ double s_ab[2];
  const int w = blockIdx.x, tid = threadIdx.x, Dx = G.Dx, F = G.F, N = Dx + F;
  if (running && !running[w]) return;
  double* __restrict__ sc = G.scal + (size_t)w * kDoglegScal;
  if (tid == 0) {
    const double radius = round > 0 ? state[w].radius : initial_radius;
    const double gg = sc[0], nn = sc[1], gnn = sc[2], whw = sc[3], whd = sc[4], dhd = sc[5];
    const bool valid = sc[6] != 0.0;
    double a = 0.0, b = 0.0, norm = 0.0, m = 0.0;
    if (valid) {
      const double gnorm = sqrt(gg), nnorm = sqrt(nn);
      const double alpha = (gg == 0.0 && whw == 0.0) ? 0.0 : __ddiv_rn(gg, whw);
      if (nnorm <= radius) {                               // 1. the Gauss-Newton step
        b = 1.0, norm = nnorm;
      } else if (__dmul_rn(alpha, gnorm) >= radius) {     // 2. along the gradient to the boundary
        a = -__ddiv_rn(radius, gnorm), norm = radius;
      } else {                                             // 3. from the Cauchy point towards the Gauss-Newton step
        const double ag = __dmul_rn(alpha, gnorm), a2 = __dmul_rn(ag, ag);
        const double ba = -__dmul_rn(alpha, gnn);
        const double c = __dsub_rn(ba, a2);
        const double bma = __dadd_rn(__dsub_rn(a2, __dmul_rn(2.0, ba)), nn);
        const double r2a = __dsub_rn(__dmul_rn(radius, radius), a2);
        const double dd = sqrt(__dadd_rn(__dmul_rn(c, c), __dmul_rn(bma, r2a)));
        const double beta = c <= 0.0 ? __ddiv_rn(__dsub_rn(dd, c), bma) : __ddiv_rn(r2a, __dadd_rn(dd, c));
        a = -__dmul_rn(alpha, __dsub_rn(1.0, beta)), b = beta;
        norm = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(__dmul_rn(a, a), gg), __dmul_rn(__dmul_rn(2.0, __dmul_rn(a, b)), gnn)),
                              __dmul_rn(__dmul_rn(b, b), nn)));
      }
      const double lin = __dadd_rn(__dmul_rn(a, gg), __dmul_rn(b, gnn));
      const double quad = __dadd_rn(__dadd_rn(__dmul_rn(__dmul_rn(a, a), whw), __dmul_rn(__dmul_rn(2.0, __dmul_rn(a, b)), whd)),
                                    __dmul_rn(__dmul_rn(b, b), dhd));
      m = -__dadd_rn(lin, __dmul_rn(0.5, quad));
    }
    sc[7] = norm;
    cost[3 * (size_t)w + 2] = m;
    solved[w] = valid ? 1 : 0;
    s_ab[0] = valid ? a : 0.0, s_ab[1] = valid ? b : 0.0;
  }
  __syncthreads();
  const double a = s_ab[0], b = s_ab[1];
  const bool any = a != 0.0 || b != 0.0;
  const double *ww = G.w + (size_t)w * N, *gn = G.gn + (size_t)w * N;
  for (int i = tid; i < N; i += 128) {
    const double v = any ? __dadd_rn(__dmul_rn(a, ww[i]), __dmul_rn(b, gn[i])) : 0.0;
    if (i < Dx) dx[(size_t)w * Dx + i] = v;
    else G.dl[(size_t)w * F + i - Dx] = v;
  }
}

// ---- the trust-region policy of viml_solve_vi (viml.h) -------------------------------------------------------------------------
// One CTA per window after each round's step.  A stopped window only writes a NaN trace row.  A running one reduces |dx| (the
// reduced step and the landmark increments x+ - x) and |x|, then thread 0 applies the policy; the scalar arithmetic goes through
// __d*_rn so that no multiply-add is fused, and an IEEE restatement (tests/solve_policy.py) reproduces the radius, the decisions and
// the trace bit for bit.  The CTA then moves x+ into x on acceptance and, at the window's last step, x into the outputs.
// s.dogleg != null: the strategy updates are the dogleg's (viml.h, VIML_SOLVE_DOGLEG; tests/dogleg_policy.py restates them).
__global__ void __launch_bounds__(128) policy_kernel(SolveArgs s, int round) {
  __shared__ double s_red[2][4];
  __shared__ int s_accept, s_stop;
  const int w = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int P = s.P, F = s.F, X = s.X, Dx = s.Dx, M = s.opt.max_iterations;
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  double* __restrict__ trow = s.out.trace ? s.out.trace + ((size_t)w * M + round) * 4 : nullptr;
  if (round > 0 && !s.running[w]) {
    if (trow && tid < 4) trow[tid] = nan;
    return;
  }
  double dd = 0.0, xx = 0.0;
  for (int i = tid; i < Dx; i += 128) {
    const double v = s.dx[(size_t)w * Dx + i];
    dd += v * v;
  }
  for (int l = tid; l < F; l += 128) {
    const double v = s.x_dep[(size_t)w * F + l], e = s.p_dep[(size_t)w * F + l] - v;
    dd += e * e;
    xx += v * v;
  }
  for (int i = tid; i < 7 * P + 7 + X; i += 128) {
    const double v = i < 7 * P ? s.x_poses[(size_t)w * 7 * P + i] : i < 7 * P + 7 ? s.x_ex[(size_t)w * 7 + i - 7 * P]
                                                                                     : s.x_extra[(size_t)w * X + i - 7 * P - 7];
    xx += v * v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    dd += __shfl_xor_sync(0xffffffffu, dd, o);
    xx += __shfl_xor_sync(0xffffffffu, xx, o);
  }
  if (lane == 0) s_red[0][warp] = dd, s_red[1][warp] = xx;
  __syncthreads();
  if (tid == 0) {
    const viml_solve_options& o = s.opt;
    const bool dogleg = s.dogleg != nullptr;
    SolveState st = s.state[w];
    const double f = s.cost[3 * (size_t)w], fp = s.cost[3 * (size_t)w + 1], m = s.cost[3 * (size_t)w + 2];
    int accept = 0, status = -1;
    if (round == 0) {   // f(x0) is this round's f(x)
      st.radius = o.initial_radius, st.decrease_factor = 2.0, st.f0 = f, st.f = f;
      st.consecutive_invalid = st.iterations = st.accepted = 0;
      st.mu = kDoglegMinMu, st.reuse = 0;
      if (!isfinite(f)) status = VIML_SOLVE_FAILURE;
    }
    if (status >= 0) {
      if (trow) trow[0] = trow[1] = trow[2] = trow[3] = nan;
    } else {
      if (trow) trow[0] = f, trow[1] = fp, trow[2] = m, trow[3] = dogleg ? st.radius : __ddiv_rn(1.0, st.radius);
      st.f = f;
      if (!s.solved[w] || !isfinite(fp) || !(m > 0.0)) {
        st.consecutive_invalid += 1;
        if (dogleg) {   // the radius stays; a new Gauss-Newton step with ten times the damping
          st.mu = __dmul_rn(st.mu, 10.0);
          st.reuse = 0;
        } else {
          st.radius = __ddiv_rn(st.radius, st.decrease_factor);
          st.decrease_factor = __dmul_rn(st.decrease_factor, 2.0);
        }
        if (st.consecutive_invalid > o.max_consecutive_invalid) status = VIML_SOLVE_FAILURE;
      } else {
        st.consecutive_invalid = 0;
        const double dnorm = sqrt(s_red[0][0] + s_red[0][1] + s_red[0][2] + s_red[0][3]);
        const double xnorm = sqrt(s_red[1][0] + s_red[1][1] + s_red[1][2] + s_red[1][3]);
        if (dnorm <= __dmul_rn(o.parameter_tolerance, __dadd_rn(xnorm, o.parameter_tolerance))) {
          status = VIML_SOLVE_PARAMETER_TOL;
        } else if (fabs(__dsub_rn(f, fp)) <= __dmul_rn(o.function_tolerance, f)) {
          status = VIML_SOLVE_FUNCTION_TOL;
        } else {
          const double rho = __ddiv_rn(__dsub_rn(f, fp), m);
          if (rho > o.min_relative_decrease) {
            accept = 1;
            st.accepted += 1;
            st.f = fp;
            if (dogleg) {
              if (rho < 0.25) {
                st.radius = __dmul_rn(st.radius, 0.5);
              } else if (rho > 0.75) {
                const double r3 = __dmul_rn(3.0, s.dogleg[(size_t)w * kDoglegScal + 7]);
                const double r = st.radius > r3 ? st.radius : r3;
                st.radius = r < o.max_radius ? r : o.max_radius;
              }
              const double mu = __ddiv_rn(__dmul_rn(2.0, st.mu), 10.0);
              st.mu = mu > kDoglegMinMu ? mu : kDoglegMinMu;
              st.reuse = 0;
            } else {
              const double t = __dsub_rn(__dmul_rn(2.0, rho), 1.0);
              const double c = __dsub_rn(1.0, __dmul_rn(__dmul_rn(t, t), t)), third = 1.0 / 3.0;
              const double r = __ddiv_rn(st.radius, c > third ? c : third);
              st.radius = r < o.max_radius ? r : o.max_radius;
              st.decrease_factor = 2.0;
            }
          } else if (dogleg) {   // the next round reuses the Gauss-Newton step and the Cauchy point at half the radius
            st.radius = __dmul_rn(st.radius, 0.5);
            st.reuse = 1;
          } else {
            st.radius = __ddiv_rn(st.radius, st.decrease_factor);
            st.decrease_factor = __dmul_rn(st.decrease_factor, 2.0);
          }
        }
      }
      st.iterations += 1;
      if (status < 0) {
        if (st.radius < o.min_radius) status = VIML_SOLVE_MIN_RADIUS;
        else if (st.iterations == M) status = VIML_SOLVE_NO_CONVERGENCE;
      }
    }
    st.status = status;
    s.state[w] = st;
    if (status >= 0) {
      s.running[w] = 0;
      if (dogleg) s.fresh[w] = 0;
      s.out.status[w] = status, s.out.iterations[w] = st.iterations, s.out.accepted[w] = st.accepted;
      s.out.cost[2 * (size_t)w] = st.f0, s.out.cost[2 * (size_t)w + 1] = st.f;
      if (s.out.radius) s.out.radius[w] = st.radius;
    } else {
      s.running[w] = 1;
      if (dogleg) s.fresh[w] = !st.reuse;
      else s.lambda_w[w] = __ddiv_rn(1.0, st.radius);
    }
    s_accept = accept, s_stop = status >= 0;
  }
  __syncthreads();
  const bool acc = s_accept != 0, stop = s_stop != 0;
  if (!acc && !stop) return;
  auto move = [&](double* __restrict__ x, const double* __restrict__ xp, double* __restrict__ out, size_t base, int n) {
    for (int i = tid; i < n; i += 128) {
      const double v = acc ? xp[base + i] : x[base + i];
      if (acc) x[base + i] = v;
      if (stop) out[base + i] = v;
    }
  };
  move(s.x_poses, s.p_poses, s.out.poses, (size_t)w * 7 * P, 7 * P);
  move(s.x_ex, s.p_ex, s.out.ex_pose, (size_t)w * 7, 7);
  if (F > 0) move(s.x_dep, s.p_dep, s.out.inv_depth, (size_t)w * F, F);
  if (X > 0) move(s.x_extra, s.p_extra, s.out.extra, (size_t)w * X, X);
}

}  // namespace gn
