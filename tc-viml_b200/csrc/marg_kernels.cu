// marg_kernels.cu — dense numeric core of MarginalizationInfo::marginalize, batched: one CTA per problem.
//
// Reference: /root/reference/vins_estimator/src/factor/marginalization_factor.cpp:264-293
//   Amm <- (Amm + Amm^T)/2; Amm^+ = V diag(l > eps ? 1/l : 0) V^T (SelfAdjointEigenSolver);
//   A = Arr - Arm Amm^+ Amr; b = brr - Arm Amm^+ bmm; eig(A) -> linearized_jacobians = sqrt(S) V^T,
//   linearized_residuals = sqrt(S^+) V^T b.
// The eigen-decomposition is a parallel two-sided cyclic Jacobi (round-robin pair ordering, n/2 disjoint
// rotations per round); eigen pairs are sorted ascending like Eigen.  Work matrices live in a per-CTA slice
// of device scratch (L1/L2 resident: <= 6 * 256^2 doubles).
// Also the per-window kernels of viml_marginalize_vi (selection, gather) and of viml_slide_vi (the state slide and the depth
// re-anchoring that follow the marginalisation).
#include "common.cuh"

namespace {

constexpr int kMargThreads = 256;

// Jacobi on the symmetric n x n matrix a (row-major, fully populated), eigenvectors in the columns of v.
__device__ void block_jacobi(double* __restrict__ a, double* __restrict__ v, int n, double* red, int* pq,
                             double* cs) {
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int e = tid; e < n * n; e += nt) v[e] = (e / n == e % n) ? 1.0 : 0.0;
  const int ne = (n + 1) & ~1;  // players in the round-robin tournament (one dummy if n is odd)
  const int half = ne / 2;
  __syncthreads();
  for (int sweep = 0; sweep < 40; ++sweep) {
    // convergence: off(A)^2 <= 1e-30 * ||A||_F^2
    double off = 0.0, all = 0.0;
    for (int e = tid; e < n * n; e += nt) {
      const double x = a[e] * a[e];
      all += x;
      if (e / n != e % n) off += x;
    }
    for (int d = 16; d > 0; d >>= 1) {
      off += __shfl_xor_sync(0xffffffffu, off, d);
      all += __shfl_xor_sync(0xffffffffu, all, d);
    }
    if ((tid & 31) == 0) red[tid >> 5] = off, red[32 + (tid >> 5)] = all;
    __syncthreads();
    if (tid == 0) {
      double o = 0.0, s = 0.0;
      for (int k = 0; k < (nt >> 5); ++k) o += red[k], s += red[32 + k];
      red[64] = (o <= 1e-30 * s || o == 0.0) ? 1.0 : 0.0;
    }
    __syncthreads();
    const bool done = red[64] != 0.0;
    __syncthreads();
    if (done) break;
    for (int round = 0; round < ne - 1; ++round) {
      // circle method: player ne-1 fixed, the others rotate
      for (int k = tid; k < half; k += nt) {
        int p = (k == 0) ? ne - 1 : (round + k) % (ne - 1);
        int q = (round + (ne - 1) - k) % (ne - 1);
        if (p > q) { const int t = p; p = q; q = t; }
        double c = 1.0, s = 0.0;
        if (q < n) {
          const double apq = a[p * n + q];
          if (apq != 0.0) {
            const double theta = (a[q * n + q] - a[p * n + p]) / (2.0 * apq);
            const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
            c = 1.0 / sqrt(t * t + 1.0);
            s = t * c;
          }
        } else {
          p = q = -1;
        }
        pq[2 * k] = p, pq[2 * k + 1] = q;
        cs[2 * k] = c, cs[2 * k + 1] = s;
      }
      __syncthreads();
      // columns: A <- A J, V <- V J
      for (int e = tid; e < n * half; e += nt) {
        const int i = e / half, k = e % half;
        const int p = pq[2 * k], q = pq[2 * k + 1];
        if (p < 0) continue;
        const double c = cs[2 * k], s = cs[2 * k + 1];
        const double aip = a[i * n + p], aiq = a[i * n + q];
        a[i * n + p] = c * aip - s * aiq;
        a[i * n + q] = s * aip + c * aiq;
        const double vip = v[i * n + p], viq = v[i * n + q];
        v[i * n + p] = c * vip - s * viq;
        v[i * n + q] = s * vip + c * viq;
      }
      __syncthreads();
      // rows: A <- J^T A
      for (int e = tid; e < n * half; e += nt) {
        const int k = e / n, j = e % n;
        const int p = pq[2 * k], q = pq[2 * k + 1];
        if (p < 0) continue;
        const double c = cs[2 * k], s = cs[2 * k + 1];
        const double apj = a[p * n + j], aqj = a[q * n + j];
        a[p * n + j] = c * apj - s * aqj;
        a[q * n + j] = s * apj + c * aqj;
      }
      __syncthreads();
    }
  }
}

// rank[k] = position of eigenvalue k in ascending order (ties by index)
__device__ void ascending_rank(const double* __restrict__ a, int n, int* rank) {
  for (int k = threadIdx.x; k < n; k += blockDim.x) {
    const double lk = a[k * n + k];
    int r = 0;
    for (int j = 0; j < n; ++j) {
      const double lj = a[j * n + j];
      r += (lj < lk) || (lj == lk && j < k);
    }
    rank[k] = r;
  }
  __syncthreads();
}

// sizes == nullptr: every problem is pos x pos with m0 marginalised, outputs [K][n][n] / [K][n] (ld = n = pos - m0).  Otherwise
// problem k is sizes[k] = {pos_k, m_k} (pos_k - m_k <= 0: skipped) in the leading part of a pos x pos slot of A / b, and its outputs
// fill the leading n_k x n_k of an ld x ld slot (per_cta sized for the largest m_k and n_k).
__global__ void __launch_bounds__(kMargThreads) marg_kernel(int K, int pos, int m0, double eps,
                                                            const double* __restrict__ A, const double* __restrict__ b,
                                                            double* __restrict__ A_schur, double* __restrict__ b_schur,
                                                            double* __restrict__ lin_jac, double* __restrict__ lin_res,
                                                            double* __restrict__ scratch, size_t per_cta,
                                                            const int2* __restrict__ sizes, int ld) {
  __shared__ double red[65];
  __shared__ int pq[256];
  __shared__ double cs[256];
  __shared__ int rank[256];
  __shared__ double lam[256];
  const int tid = threadIdx.x, nt = blockDim.x;
  double* ws = scratch + (size_t)blockIdx.x * per_cta;
  for (int k = blockIdx.x; k < K; k += gridDim.x) {
    const int m = sizes ? sizes[k].y : m0, n = (sizes ? sizes[k].x : pos) - m;
    if (n <= 0) continue;                     // CTA-uniform
    double* Wm = ws;                          // m*m   work / eigenvalues on the diagonal
    double* Vm = Wm + (size_t)m * m;          // m*m
    double* Inv = Vm + (size_t)m * m;         // m*m
    double* T = Inv + (size_t)m * m;          // n*m
    double* Wn = T + (size_t)n * m;           // n*n
    double* Vn = Wn + (size_t)n * n;          // n*n
    double* br = Vn + (size_t)n * n;          // n
    const double* Ak = A + (size_t)k * pos * pos;
    const double* bk = b + (size_t)k * pos;
    __syncthreads();
    if (m > 0) {
      for (int e = tid; e < m * m; e += nt) {
        const int r = e / m, c = e % m;
        Wm[e] = 0.5 * (Ak[(size_t)r * pos + c] + Ak[(size_t)c * pos + r]);                 // :267
      }
      __syncthreads();
      block_jacobi(Wm, Vm, m, red, pq, cs);                                                // :268
      for (int e = tid; e < m; e += nt) {
        const double l = Wm[e * m + e];
        lam[e] = l > eps ? 1.0 / l : 0.0;                                                  // :272
      }
      __syncthreads();
      for (int e = tid; e < m * m; e += nt) {
        const int r = e / m, c = e % m;
        double s = 0.0;
        for (int j = 0; j < m; ++j) s += Vm[r * m + j] * lam[j] * Vm[c * m + j];
        Inv[e] = s;
      }
      __syncthreads();
      for (int e = tid; e < n * m; e += nt) {                                              // Arm * Amm_inv
        const int r = e / m, c = e % m;
        double s = 0.0;
        for (int j = 0; j < m; ++j) s += Ak[(size_t)(m + r) * pos + j] * Inv[j * m + c];
        T[e] = s;
      }
      __syncthreads();
    }
    for (int e = tid; e < n * n + n; e += nt) {                                            // :281-282
      if (e < n * n) {
        const int r = e / n, c = e % n;
        double s = 0.0;
        for (int j = 0; j < m; ++j) s += T[r * m + j] * Ak[(size_t)j * pos + m + c];
        const double val = Ak[(size_t)(m + r) * pos + m + c] - s;
        Wn[e] = val;
        if (A_schur) A_schur[(size_t)k * ld * ld + (size_t)r * ld + c] = val;
      } else {
        const int r = e - n * n;
        double s = 0.0;
        for (int j = 0; j < m; ++j) s += T[r * m + j] * bk[j];
        const double val = bk[m + r] - s;
        br[r] = val;
        if (b_schur) b_schur[(size_t)k * ld + r] = val;
      }
    }
    __syncthreads();
    if (!lin_jac && !lin_res) continue;
    // SelfAdjointEigenSolver reads the lower triangle (:284)
    for (int e = tid; e < n * n; e += nt) {
      const int r = e / n, c = e % n;
      if (r < c) Wn[e] = Wn[c * n + r];
    }
    __syncthreads();
    // the mirrored copy above reads entries other threads may be writing: redo from A_schur semantics
    // (upper <- lower) is idempotent because only r < c entries are written and only r > c are read.
    block_jacobi(Wn, Vn, n, red, pq, cs);
    ascending_rank(Wn, n, rank);
    for (int e = tid; e < n; e += nt) lam[e] = Wn[e * n + e];
    __syncthreads();
    for (int e = tid; e < n * n + n; e += nt) {
      if (e < n * n) {
        if (!lin_jac) continue;
        const int kk = e / n, c = e % n;  // source eigenpair kk -> output row rank[kk]
        const double S = lam[kk] > eps ? lam[kk] : 0.0;                                    // :285
        lin_jac[(size_t)k * ld * ld + (size_t)rank[kk] * ld + c] = sqrt(S) * Vn[c * n + kk];  // :292
      } else {
        if (!lin_res) continue;
        const int kk = e - n * n;
        const double Sinv = lam[kk] > eps ? 1.0 / lam[kk] : 0.0;                           // :286
        const double sq = sqrt(Sinv);
        double s = 0.0;
        for (int c = 0; c < n; ++c) s += (sq * Vn[c * n + kk]) * br[c];                     // :293
        lin_res[(size_t)k * ld + rank[kk]] = s;
      }
    }
  }
}

// ---- viml_marginalize_vi: which factors and blocks of each window take part, and the dense problem they give -------------------
// Block slots of a window: pose p -> p, the extrinsic -> P, the speed-bias of pose q (extra offset 9q) -> P + 1 + q.
__device__ __forceinline__ bool imu_selected(const InertialArgs& v, int64_t f, bool old) {   // est.cpp:1916-1930
  return old && min(max(v.imu_pose[2 * f], 0), v.P - 1) == 0 && v.imu_preint[f * 17] < 10.0;
}

// Point factors with i == 0 of every MARGIN_OLD window (est.cpp:1933-1966).
__global__ void __launch_bounds__(128) marg_count_kernel(MargViArgs g) {
  __shared__ int s_cnt;
  const int w = blockIdx.x, tid = threadIdx.x;
  if (tid == 0) s_cnt = 0;
  __syncthreads();
  if (g.margin[w] == VIML_MARGIN_OLD) {
    int c = 0;
    for (int64_t k = g.pf_window_offset[w] + tid; k < g.pf_window_offset[w + 1]; k += blockDim.x) c += (g.pf_idx[k] & 0xffu) == 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((tid & 31) == 0) atomicAdd(&s_cnt, c);
  }
  __syncthreads();
  if (tid == 0) g.cnt[w] = s_cnt;
}

// One CTA per window: the window's selected point factors, in input order, into the CSR sel_* (the window's offset is the sum of the
// counts before it), and the IMU factors that take no part zeroed in the dense-factor CSR (their J^T J and J^T r add exact zeros).
__global__ void __launch_bounds__(128) marg_select_kernel(MargViArgs g) {
  __shared__ int s_part[4];
  __shared__ int s_base;
  const int w = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int c = 0;
  for (int u = tid; u < w; u += blockDim.x) c += g.cnt[u];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane == 0) s_part[warp] = c;
  __syncthreads();
  if (tid == 0) {
    s_base = s_part[0] + s_part[1] + s_part[2] + s_part[3];
    g.sel_offset[w] = s_base;
    if (w == g.W - 1) g.sel_offset[g.W] = s_base + g.cnt[w];
  }
  __syncthreads();
  const bool old = g.margin[w] == VIML_MARGIN_OLD;
  int at = s_base;
  if (old) {
    for (int64_t k0 = g.pf_window_offset[w]; k0 < g.pf_window_offset[w + 1]; k0 += blockDim.x) {
      const int64_t k = k0 + tid;
      const bool sel = k < g.pf_window_offset[w + 1] && (g.pf_idx[k] & 0xffu) == 0;
      const unsigned mask = __ballot_sync(0xffffffffu, sel);
      __syncthreads();   // s_part of the previous chunk has been read
      if (lane == 0) s_part[warp] = __popc(mask);
      __syncthreads();
      int before = 0, total = 0;
      for (int u = 0; u < 4; ++u) before += u < warp ? s_part[u] : 0, total += s_part[u];
      if (sel) {
        const int64_t d = at + before + __popc(mask & ((1u << lane) - 1u));
        g.sel_idx[d] = g.pf_idx[k];
        reinterpret_cast<double4*>(g.sel_obs)[d] = reinterpret_cast<const double4*>(g.pf_obs)[k];
        if (g.sel_z) g.sel_z[d] = g.pf_pts_i_z[k];
      }
      at += total;
    }
  }
  const InertialArgs& v = g.v;
  if (v.NI == 0) return;
  const bool prior = v.n_max > 0 && v.prior_n[w] > 0;   // imu_kernel's CSR slot of factor f
  for (int64_t f = v.imu_window_offset[w]; f < v.imu_window_offset[w + 1]; ++f) {
    if (imu_selected(v, f, old)) continue;
    const int kf = g.csr.window_offset[w] + (prior ? 1 : 0) + (int)(f - v.imu_window_offset[w]);
    for (int e = tid; e < 15; e += blockDim.x) g.csr.residual[g.csr.row_offset[kf] + e] = 0.0;
    for (int e = tid; e < 450; e += blockDim.x) g.csr.jacobian[g.csr.jac_offset[kf] + e] = 0.0;
  }
}

// One CTA per window: the blocks the selected factors touch, their columns in A = [marginalised | kept] gathered from Sx / gx, the
// problem size {pos, m}, and the output prior's n, block list and x0 (marg_kernel writes its Jacobian and residual).  A MARGIN_SECOND_NEW
// window whose prior does not hold pose P-2 gets its input prior copied.
__global__ void __launch_bounds__(256) marg_gather_kernel(MargViArgs g) {
  __shared__ int s_touch[2 * 255 + 1];
  __shared__ int s_col[kMaxDx];          // tangent column of each row of A
  __shared__ int s_blk[2 * 255 + 1][3];  // kept block: slot, output index, first column
  __shared__ int s_has, s_pos, s_m, s_nb;
  const InertialArgs& v = g.v;
  const viml_prior_out& o = g.out;
  const int w = blockIdx.x, tid = threadIdx.x, nt = blockDim.x, P = g.P, D = g.D, X = g.X, Dx = D + X, NS = 2 * P + 1;
  const int QS = min(P, X / 9);           // speed-bias slots inside the extra state
  const bool old = g.margin[w] == VIML_MARGIN_OLD;
  const int n_in = v.n_max > 0 ? min(max(v.prior_n[w], 0), v.n_max) : 0;
  const int nb_in = n_in > 0 ? min(max(v.prior_n_blocks[w], 0), v.max_blocks) : 0;
  auto prior_slot = [&](int b) {          // -1: an extra block outside the speed-bias slots
    const int32_t* blk = v.prior_block + ((size_t)w * v.max_blocks + b) * 4;
    if (blk[0] == VIML_BLOCK_POSE) return min(max(blk[1], 0), P - 1);
    if (blk[0] == VIML_BLOCK_EX) return P;
    return QS > 0 ? P + 1 + min(max(blk[1] / 9, 0), QS - 1) : -1;
  };
  for (int s = tid; s < NS; s += nt) s_touch[s] = 0;
  if (tid == 0) s_has = 0;
  __syncthreads();
  for (int b = tid; b < nb_in; b += nt)
    if (prior_slot(b) == P - 2) s_has = 1;
  __syncthreads();
  double* pj = o.prior_jacobian + (size_t)w * o.prior_n_max * o.prior_n_max;
  double* pr = o.prior_residual + (size_t)w * o.prior_n_max;
  int32_t* pb = o.prior_block + (size_t)w * o.prior_max_blocks * 4;
  double* px = o.prior_x0 + (size_t)w * o.prior_max_blocks * VIML_PRIOR_X0_STRIDE;
  if (!old && !s_has) {   // est.cpp:2047-2049: last_marginalization_info is kept
    const bool fits = n_in <= o.prior_n_max && nb_in <= o.prior_max_blocks;
    if (tid == 0) {
      o.prior_n[w] = fits ? n_in : 0, o.prior_n_blocks[w] = fits ? nb_in : 0;
      g.sizes[w] = make_int2(0, 0);
    }
    if (!fits) return;
    const double* J = v.prior_jacobian + (size_t)w * v.n_max * v.n_max;
    for (int e = tid; e < n_in * n_in; e += nt) pj[(size_t)(e / n_in) * o.prior_n_max + e % n_in] = J[(size_t)(e / n_in) * v.n_max + e % n_in];
    for (int e = tid; e < n_in; e += nt) pr[e] = v.prior_residual[(size_t)w * v.n_max + e];
    for (int e = tid; e < nb_in * 4; e += nt) pb[e] = v.prior_block[(size_t)w * v.max_blocks * 4 + e];
    for (int e = tid; e < nb_in * VIML_PRIOR_X0_STRIDE; e += nt) px[e] = v.prior_x0[(size_t)w * v.max_blocks * VIML_PRIOR_X0_STRIDE + e];
    return;
  }
  for (int b = tid; b < nb_in; b += nt) {
    const int s = prior_slot(b);
    if (s >= 0) s_touch[s] = 1;
  }
  if (old) {
    for (int64_t k = g.sel_offset[w] + tid; k < g.sel_offset[w + 1]; k += nt) {   // pose 0, pose j, extrinsic
      s_touch[0] = 1, s_touch[P] = 1;
      s_touch[min(max((int)((g.sel_idx[k] >> 8) & 0xffu), 0), P - 1)] = 1;
    }
    if (v.NI > 0 && QS > 0)
      for (int64_t f = v.imu_window_offset[w] + tid; f < v.imu_window_offset[w + 1]; f += nt) {
        if (!imu_selected(v, f, true)) continue;
        s_touch[0] = 1;
        s_touch[min(max(v.imu_pose[2 * f + 1], 0), P - 1)] = 1;
        s_touch[P + 1 + min(max(v.imu_sb[2 * f] / 9, 0), QS - 1)] = 1;
        s_touch[P + 1 + min(max(v.imu_sb[2 * f + 1] / 9, 0), QS - 1)] = 1;
      }
  }
  __syncthreads();
  if (tid == 0) {
    // marginalised: MARGIN_OLD pose 0 then speed-bias 0 (est.cpp:1922, :1950); MARGIN_SECOND_NEW pose P-2 (:2064)
    const int dp = old ? 0 : P - 2, ds = old ? P + 1 : -1;
    int pos = 0, nb = 0;
    if (s_touch[dp])
      for (int t = 0; t < 6; ++t) s_col[pos++] = 6 * dp + t;
    if (ds >= 0 && s_touch[ds])
      for (int t = 0; t < 9; ++t) s_col[pos++] = D + t;
    const int m = pos;
    for (int s = 0; s < NS; ++s) {   // kept, in output order: poses ascending, the extrinsic, speed-biases ascending
      if (!s_touch[s] || s == dp || s == ds) continue;
      const int local = s <= P ? 6 : 9, t0 = s < P ? 6 * s : s == P ? 6 * P : D + 9 * (s - P - 1);
      const int q = s < P ? s : s - P - 1;   // addr_shift (est.cpp:2030-2040, :2098-2108)
      const int slid = old ? q - 1 : q == P - 1 ? P - 2 : q;
      s_blk[nb][0] = s, s_blk[nb][1] = s == P ? 0 : s < P ? slid : 9 * slid, s_blk[nb][2] = pos - m;
      ++nb;
      for (int t = 0; t < local; ++t) s_col[pos++] = t0 + t;
    }
    const bool fits = pos - m <= o.prior_n_max && nb <= o.prior_max_blocks && pos <= g.pm;
    s_pos = fits && pos > m ? pos : 0, s_m = m, s_nb = fits && pos > m ? nb : 0;
    o.prior_n[w] = s_pos ? pos - m : 0, o.prior_n_blocks[w] = s_nb;
    g.sizes[w] = make_int2(s_pos, m);
  }
  __syncthreads();
  const int pos = s_pos, nb = s_nb;
  for (int e = tid; e < nb * 4; e += nt) {
    const int b = e >> 2, c = e & 3, s = s_blk[b][0];
    pb[e] = c == 0 ? (s < P ? VIML_BLOCK_POSE : s == P ? VIML_BLOCK_EX : VIML_BLOCK_EXTRA) : c == 1 ? s_blk[b][1] : c == 2 ? (s <= P ? 7 : 9)
                                                                                                                   : s_blk[b][2];
  }
  for (int e = tid; e < nb * VIML_PRIOR_X0_STRIDE; e += nt) {   // keep_block_data: the values at the linearisation point
    const int b = e / VIML_PRIOR_X0_STRIDE, t = e % VIML_PRIOR_X0_STRIDE, s = s_blk[b][0];
    const double* x = s < P ? v.poses + ((size_t)w * P + s) * 7 : s == P ? v.ex_pose + (size_t)w * 7 : v.extra + (size_t)w * X + 9 * (s - P - 1);
    px[e] = t < (s <= P ? 7 : 9) ? x[t] : 0.0;
  }
  const double* Sx = g.Sx + (size_t)w * Dx * Dx;
  double* A = g.A + (size_t)w * g.pm * g.pm;
  for (int e = tid; e < pos * pos; e += nt) {
    const int r = e / pos, c = e - r * pos;
    A[(size_t)r * g.pm + c] = Sx[(size_t)s_col[r] * Dx + s_col[c]];
  }
  for (int r = tid; r < pos; r += nt) g.b[(size_t)w * g.pm + r] = g.gx[(size_t)w * Dx + s_col[r]];
}

// ---- viml_slide_vi: the window slide (est.cpp:2121-2218) and removeBackShiftDepth, plain IEEE binary64 without fused multiply-adds --
constexpr int kSlideThreads = 256;
constexpr int kSlideChunk = 4096;   // features counted per pass over the window's point factors (F <= 65535: up to 16 passes)

__device__ __forceinline__ double dot3_rn(double a0, double a1, double a2, double b0, double b1, double b2) {
  return __dadd_rn(__dadd_rn(__dmul_rn(a0, b0), __dmul_rn(a1, b1)), __dmul_rn(a2, b2));
}

// normalized(q).toRotationMatrix() of a [p, q] block, Eigen's order (double2vector forms Rs so)
__device__ void slide_rot(const double* p7, double* R) {
  const double qx = p7[3], qy = p7[4], qz = p7[5], qw = p7[6];
  const double n = __dsqrt_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(qx, qx), __dmul_rn(qy, qy)), __dmul_rn(qz, qz)), __dmul_rn(qw, qw)));
  const double w = __ddiv_rn(qw, n), x = __ddiv_rn(qx, n), y = __ddiv_rn(qy, n), z = __ddiv_rn(qz, n);
  const double tx = __dmul_rn(2.0, x), ty = __dmul_rn(2.0, y), tz = __dmul_rn(2.0, z);
  const double twx = __dmul_rn(tx, w), twy = __dmul_rn(ty, w), twz = __dmul_rn(tz, w);
  const double txx = __dmul_rn(tx, x), txy = __dmul_rn(ty, x), txz = __dmul_rn(tz, x);
  const double tyy = __dmul_rn(ty, y), tyz = __dmul_rn(tz, y), tzz = __dmul_rn(tz, z);
  R[0] = __dsub_rn(1.0, __dadd_rn(tyy, tzz)), R[1] = __dsub_rn(txy, twz), R[2] = __dadd_rn(txz, twy);
  R[3] = __dadd_rn(txy, twz), R[4] = __dsub_rn(1.0, __dadd_rn(txx, tzz)), R[5] = __dsub_rn(tyz, twx);
  R[6] = __dsub_rn(txz, twy), R[7] = __dadd_rn(tyz, twx), R[8] = __dsub_rn(1.0, __dadd_rn(txx, tyy));
}

// The camera of a pose: R = R(q) R(q_ex) (cam[0..8], row-major), P = p + R(q) t_ex (cam[9..11])
__device__ void slide_camera(const double* pose, const double* ex, double* cam) {
  double Rb[9], Re[9];
  slide_rot(pose, Rb);
  slide_rot(ex, Re);
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) cam[3 * r + c] = dot3_rn(Rb[3 * r], Rb[3 * r + 1], Rb[3 * r + 2], Re[c], Re[3 + c], Re[6 + c]);
    cam[9 + r] = __dadd_rn(pose[r], dot3_rn(Rb[3 * r], Rb[3 * r + 1], Rb[3 * r + 2], ex[0], ex[1], ex[2]));
  }
}

// removeBackShiftDepth for one feature: the inverse depth of the point seen from camera c0 along (ux, uy, uz) at 1 / inv, in camera c1
__device__ double slide_reanchor(double inv, double ux, double uy, double uz, const double* c0, const double* c1, double init_depth) {
  const double d = __ddiv_rn(1.0, inv);
  const double a0 = __dmul_rn(ux, d), a1 = __dmul_rn(uy, d), a2 = __dmul_rn(uz, d);
  double v[3];
  for (int r = 0; r < 3; ++r)   // w - P1, w = R0 (uv_i d) + P0
    v[r] = __dsub_rn(__dadd_rn(dot3_rn(c0[3 * r], c0[3 * r + 1], c0[3 * r + 2], a0, a1, a2), c0[9 + r]), c1[9 + r]);
  const double zj = dot3_rn(c1[2], c1[5], c1[8], v[0], v[1], v[2]);   // row 2 of R1^T
  return zj > 0.0 ? __ddiv_rn(1.0, zj) : __ddiv_rn(1.0, init_depth);
}

// One CTA per window: the state copied with the slide (coalesced over the window's P*7 + 7 + X + F values), then for MARGIN_OLD the
// anchor-0 factors counted per feature (a shared-memory counter and the first factor of each feature in a chunk of kSlideChunk
// features), and every feature with two or more re-anchored by one thread from its first factor.
__global__ void __launch_bounds__(kSlideThreads) slide_kernel(SlideArgs s) {
  __shared__ int s_cnt[kSlideChunk];
  __shared__ int s_first[kSlideChunk];
  __shared__ double s_cam[24];   // the cameras of the old poses 0 and 1
  const int w = blockIdx.x, tid = threadIdx.x, nt = blockDim.x, P = s.P, F = s.F, X = s.X;
  const bool old = s.margin[w] == VIML_MARGIN_OLD;
  const double* pin = s.poses + (size_t)w * P * 7;
  const double* ein = s.ex_pose + (size_t)w * 7;
  const double* xin = s.extra + (size_t)w * X;
  const double* din = s.inv_depth + (size_t)w * F;
  double* dout = s.out.inv_depth + (size_t)w * F;
  const int np = 7 * P, n = np + 7 + X + F;
  auto from = [&](int q) { return old ? min(q + 1, P - 1) : q == P - 2 ? P - 1 : q; };   // the slot that moves into slot q
  for (int e = tid; e < n; e += nt) {
    if (e < np) {
      const int p = e / 7;
      s.out.poses[(size_t)w * np + e] = pin[7 * from(p) + e - 7 * p];
    } else if (e < np + 7) {
      s.out.ex_pose[(size_t)w * 7 + e - np] = ein[e - np];
    } else if (e < np + 7 + X) {
      const int x = e - np - 7, q = x / 9;
      s.out.extra[(size_t)w * X + x] = xin[q < P ? 9 * from(q) + x - 9 * q : x];
    } else {
      dout[e - np - 7 - X] = din[e - np - 7 - X];
    }
  }
  if (!old) return;   // CTA-uniform
  if (tid == 0) slide_camera(pin, ein, s_cam);
  if (tid == 32) slide_camera(pin + 7, ein, s_cam + 12);
  const int k0 = s.pf_window_offset[w], k1 = s.pf_window_offset[w + 1];
  for (int f0 = 0; f0 < F; f0 += kSlideChunk) {
    const int nf = min(kSlideChunk, F - f0);
    for (int f = tid; f < nf; f += nt) s_cnt[f] = 0, s_first[f] = 0x7fffffff;
    __syncthreads();   // orders the copy of the depths above before their re-anchored values below, and publishes s_cam
    for (int k = k0 + tid; k < k1; k += nt) {
      const uint32_t ix = s.pf_idx[k];
      const int f = (int)(ix >> 16) - f0;
      if ((ix & 0xffu) == 0 && f >= 0 && f < nf) {
        atomicAdd(&s_cnt[f], 1);
        atomicMin(&s_first[f], k);
      }
    }
    __syncthreads();
    for (int f = tid; f < nf; f += nt) {
      if (s_cnt[f] < 2) continue;   // one anchor-0 factor: the reference erases the feature
      const int k = s_first[f];
      const double* ob = s.pf_obs + (size_t)4 * k;
      const double z = s.pf_pts_i_z ? s.pf_pts_i_z[k] : 1.0;
      dout[f0 + f] = slide_reanchor(din[f0 + f], ob[0], ob[1], z, s_cam, s_cam + 12, s.init_depth);
    }
    __syncthreads();   // s_cnt / s_first are read before the next chunk resets them
  }
}

}  // namespace

int viml_launch_marg_select(viml_ctx* ctx, const MargViArgs& g) {
  {
    LaunchScope ls(ctx, K_MARG);
    marg_count_kernel<<<g.W, 128, 0, ctx->stream>>>(g);
  }
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  {
    LaunchScope ls(ctx, K_MARG);
    marg_select_kernel<<<g.W, 128, 0, ctx->stream>>>(g);
  }
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  return VIML_OK;
}

int viml_launch_marg_gather(viml_ctx* ctx, const MargViArgs& g) {
  {
    LaunchScope ls(ctx, K_MARG);
    marg_gather_kernel<<<g.W, 256, 0, ctx->stream>>>(g);
  }
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  return VIML_OK;
}

int viml_launch_slide(viml_ctx* ctx, const SlideArgs& s) {
  {
    LaunchScope ls(ctx, K_MARG);
    slide_kernel<<<s.W, kSlideThreads, 0, ctx->stream>>>(s);
  }
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  return VIML_OK;
}

int viml_launch_marginalize(viml_ctx* ctx, int K, int pos, int m, double eps, const double* A, const double* b,
                            double* A_schur, double* b_schur, double* lin_jac, double* lin_res, const int2* sizes, int m_max,
                            int n_max) {
  // sized: n_k <= pos bounds the work matrices, n_max is the output's leading dimension
  const int mm = sizes ? m_max : m, n = sizes ? std::min(n_max, pos) : pos - m, ld = sizes ? n_max : pos - m;
  const size_t per_cta = (size_t)3 * mm * mm + (size_t)n * mm + (size_t)2 * n * n + n + 32;
  const int grid = K < 2 * ctx->sm_count ? K : 2 * ctx->sm_count;
  VIML_TRY_CUDA(ctx, ctx->scratch.reserve(per_cta * grid * sizeof(double) + 256));
  double* scratch = ctx->scratch.take<double>(per_cta * grid);
  {
    LaunchScope ls(ctx, K_MARG);
    marg_kernel<<<grid, kMargThreads, 0, ctx->stream>>>(K, pos, m, eps, A, b, A_schur, b_schur, lin_jac, lin_res,
                                                        scratch, per_cta, sizes, ld);
  }
  VIML_TRY_CUDA(ctx, cudaGetLastError());
  return VIML_OK;
}
