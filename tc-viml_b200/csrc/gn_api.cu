// gn_api.cu — C-ABI entry points for the reduced system of the whole window (dense-block factors: prior, IMU) and one
// Gauss-Newton / Levenberg-Marquardt iteration on it, plus the line_3d.txt map reader.  See include/viml.h.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

#include "common.cuh"

namespace {

// viml_inertial_factors: null checks always, index / size validation on the host-pointer path (the device path reads nothing back).
int check_inertial(viml_ctx* ctx, const viml_inertial_factors* vi, int W, int P, bool dev) {
  if (!vi) return fail(ctx, VIML_ERR_INVALID, "null inertial factors");
  const int X = vi->extra_dim, D = 6 * (P + 1), n_max = vi->prior_n_max, mb = vi->prior_max_blocks;
  const int64_t NI = vi->n_imu;
  if (X < 0 || D + X > kMaxDx) return fail(ctx, VIML_ERR_INVALID, "inertial factors: extra_dim out of range (D + extra_dim <= 232)");
  if (NI < 0 || n_max < 0 || mb < 0) return fail(ctx, VIML_ERR_INVALID, "inertial factors: negative size");
  if (NI > 0 && (!vi->imu_window_offset || !vi->imu_pose || !vi->imu_sb || !vi->imu_preint || !vi->imu_jacobian || !vi->imu_sqrt_info))
    return fail(ctx, VIML_ERR_INVALID, "inertial factors: null IMU array");
  if (n_max > 0 && (!vi->prior_n || !vi->prior_jacobian || !vi->prior_residual || !vi->prior_n_blocks || (mb > 0 && (!vi->prior_block || !vi->prior_x0))))
    return fail(ctx, VIML_ERR_INVALID, "inertial factors: null prior array");
  // read from the struct alone, so both flavours check it: an IMU factor reads two 9-value speed-bias blocks of the extra state
  if (NI > 0 && X < 9) return fail(ctx, VIML_ERR_INVALID, "IMU factors need extra_dim >= 9 (two speed-bias blocks of 9 values)");
  if (dev || W == 0) return VIML_OK;
  if (NI > 0) {
    const int32_t* off = vi->imu_window_offset;
    if (off[0] != 0 || off[W] != NI) return fail(ctx, VIML_ERR_INVALID, "IMU factors: imu_window_offset is not a CSR of the factor list");
    for (int w = 0; w < W; ++w)
      if (off[w + 1] < off[w]) return fail(ctx, VIML_ERR_INVALID, "IMU factors: imu_window_offset decreases");
    for (int64_t k = 0; k < NI; ++k) {
      const int i = vi->imu_pose[2 * k], j = vi->imu_pose[2 * k + 1], si = vi->imu_sb[2 * k], sj = vi->imu_sb[2 * k + 1];
      if (i < 0 || i >= P || j < 0 || j >= P || i == j) return fail(ctx, VIML_ERR_INVALID, "IMU factor: pose index outside [0, P) or i == j");
      if (si < 0 || si + 9 > X || sj < 0 || sj + 9 > X) return fail(ctx, VIML_ERR_INVALID, "IMU factor: speed-bias block outside the extra state (sb + 9 <= X)");
      if (si + 9 > sj && sj + 9 > si) return fail(ctx, VIML_ERR_INVALID, "IMU factor: speed-bias blocks i and j overlap");
    }
  }
  if (n_max > 0) {
    std::vector<int> col_mark, tan_mark(D + X);
    for (int w = 0; w < W; ++w) {
      const int n = vi->prior_n[w];
      if (n < 0 || n > n_max) return fail(ctx, VIML_ERR_INVALID, "prior: n_w outside [0, prior_n_max]");
      if (n == 0) continue;
      const int nb = vi->prior_n_blocks[w];
      if (nb < 0 || nb > mb) return fail(ctx, VIML_ERR_INVALID, "prior: block count outside [0, prior_max_blocks]");
      col_mark.assign(n, 0);
      std::fill(tan_mark.begin(), tan_mark.end(), 0);
      for (int b = 0; b < nb; ++b) {
        const int32_t* blk = vi->prior_block + ((size_t)w * mb + b) * 4;
        const int kind = blk[0], idx = blk[1], size = blk[2], first = blk[3];
        int tcol;
        if (kind == VIML_BLOCK_POSE || kind == VIML_BLOCK_EX) {
          if (size != 7) return fail(ctx, VIML_ERR_INVALID, "prior: a pose / extrinsic block must have size 7");
          if (kind == VIML_BLOCK_POSE && (idx < 0 || idx >= P)) return fail(ctx, VIML_ERR_INVALID, "prior: pose index outside [0, P)");
          tcol = kind == VIML_BLOCK_POSE ? 6 * idx : 6 * P;
        } else if (kind == VIML_BLOCK_EXTRA) {
          if (size < 1 || size == 7 || size > VIML_PRIOR_X0_STRIDE || idx < 0 || idx + size > X)
            return fail(ctx, VIML_ERR_INVALID, "prior: extra block outside the extra state (or of size 7, or above VIML_PRIOR_X0_STRIDE)");
          tcol = D + idx;
        } else {
          return fail(ctx, VIML_ERR_INVALID, "prior: unknown block kind");
        }
        const int local = size == 7 ? 6 : size;
        if (first < 0 || first + local > n) return fail(ctx, VIML_ERR_INVALID, "prior: block columns outside [0, n_w)");
        for (int t = 0; t < local; ++t) {
          if (col_mark[first + t]++ || tan_mark[tcol + t]++) return fail(ctx, VIML_ERR_INVALID, "prior: blocks overlap");
        }
      }
      for (int c = 0; c < n; ++c)
        if (!col_mark[c]) return fail(ctx, VIML_ERR_INVALID, "prior: the blocks do not cover [0, n_w)");
    }
  }
  return VIML_OK;
}

// Stages viml_inertial_factors into *out (the Stager keeps the addresses of its fields: commit() fills them in); the state
// pointers are left to the caller.
void stage_inertial(Stager& st, const viml_inertial_factors* vi, int W, int P, InertialArgs* out) {
  InertialArgs& v = *out;
  v = InertialArgs{};
  v.W = W, v.P = P, v.D = 6 * (P + 1), v.X = vi->extra_dim, v.NI = vi->n_imu;
  for (int k = 0; k < 3; ++k) v.G[k] = vi->gravity[k];
  v.n_max = vi->prior_n_max, v.max_blocks = vi->prior_max_blocks;
  const size_t NI = (size_t)v.NI, n_max = (size_t)v.n_max, mb = (size_t)v.max_blocks;
  st.in(NI ? vi->imu_window_offset : nullptr, NI ? (size_t)W + 1 : 0, &v.imu_window_offset);
  st.in(vi->imu_pose, NI * 2, &v.imu_pose);
  st.in(vi->imu_sb, NI * 2, &v.imu_sb);
  st.in(vi->imu_preint, NI * 17, &v.imu_preint);
  st.in(vi->imu_jacobian, NI * 225, &v.imu_jacobian);
  st.in(vi->imu_sqrt_info, NI * 225, &v.imu_sqrt_info);
  if (n_max) {
    st.in(vi->prior_n, (size_t)W, &v.prior_n);
    st.in(vi->prior_jacobian, (size_t)W * n_max * n_max, &v.prior_jacobian);
    st.in(vi->prior_residual, (size_t)W * n_max, &v.prior_residual);
    st.in(vi->prior_n_blocks, (size_t)W, &v.prior_n_blocks);
    st.in(vi->prior_block, (size_t)W * mb * 4, &v.prior_block);
    st.in(vi->prior_x0, (size_t)W * mb * VIML_PRIOR_X0_STRIDE, &v.prior_x0);
  }
}

// Scratch of the dense-factor CSR of the evaluated IMU / prior factors (bounds in common.cuh).
void stage_inertial_csr(Stager& st, const InertialArgs& v, InertialCsr* csr, double** residual_plus) {
  const size_t W = (size_t)v.W, NI = (size_t)v.NI, n_max = (size_t)v.n_max;
  st.out((int32_t*)nullptr, W + 1, &csr->window_offset);
  st.out((int64_t*)nullptr, W + NI + 1, &csr->row_offset);
  st.out((int64_t*)nullptr, W + NI + 1, &csr->col_offset);
  st.out((int64_t*)nullptr, W + NI + 1, &csr->jac_offset);
  st.out((int32_t*)nullptr, W * n_max + 30 * NI + 1, &csr->col_index);
  st.out((double*)nullptr, W * n_max + 15 * NI + 1, &csr->residual);
  st.out((double*)nullptr, W * n_max * n_max + 450 * NI + 1, &csr->jacobian);
  st.out((double*)nullptr, W * n_max + 15 * NI + 1, residual_plus);
}

// viml_dense_factors of W windows over Dx tangent columns: ND and the arrays of *dn (the Stager keeps the addresses of its fields).
// The kernels index row_offset, jac_offset, the Jacobian and the Sx columns through window_offset, the offsets and col_index: the
// host flavour checks all of them; the device flavour reads back the three totals, which size the staged arrays.
int stage_dense(viml_ctx* ctx, Stager& st, const viml_dense_factors* dense, int W, int Dx, DenseArgs* dn) {
  const int64_t ND = dense ? dense->n_factors : 0;
  dn->ND = ND;
  if (ND == 0) return VIML_OK;
  if (!dense->window_offset || !dense->row_offset || !dense->col_offset || !dense->jac_offset || !dense->col_index || !dense->residual ||
      !dense->jacobian)
    return fail(ctx, VIML_ERR_INVALID, "dense factors: null array");
  int64_t n_rows = 0, n_cols = 0, n_jac = 0;
  if (st.dev) {   // totals are the last prefix entries: three 8-byte reads from the device
    int64_t t[3];
    VIML_TRY_CUDA(ctx, cudaMemcpyAsync(&t[0], dense->row_offset + ND, 8, cudaMemcpyDeviceToHost, ctx->stream));
    VIML_TRY_CUDA(ctx, cudaMemcpyAsync(&t[1], dense->col_offset + ND, 8, cudaMemcpyDeviceToHost, ctx->stream));
    VIML_TRY_CUDA(ctx, cudaMemcpyAsync(&t[2], dense->jac_offset + ND, 8, cudaMemcpyDeviceToHost, ctx->stream));
    VIML_TRY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    n_rows = t[0], n_cols = t[1], n_jac = t[2];
  } else {
    const int32_t* off = dense->window_offset;
    if (off[0] != 0 || off[W] != ND) return fail(ctx, VIML_ERR_INVALID, "dense factors: window_offset is not a CSR of the factor list");
    for (int w = 0; w < W; ++w)
      if (off[w + 1] < off[w]) return fail(ctx, VIML_ERR_INVALID, "dense factors: window_offset decreases");
    if (dense->row_offset[0] != 0 || dense->col_offset[0] != 0 || dense->jac_offset[0] != 0)
      return fail(ctx, VIML_ERR_INVALID, "dense factors: row_offset, col_offset and jac_offset must start at 0");
    n_rows = dense->row_offset[ND], n_cols = dense->col_offset[ND], n_jac = dense->jac_offset[ND];
    for (int64_t k = 0; k < n_cols; ++k)
      if (dense->col_index[k] < 0 || dense->col_index[k] >= Dx) return fail(ctx, VIML_ERR_INVALID, "dense factors: col_index out of range");
    for (int64_t k = 0; k < ND; ++k) {
      const int64_t n = dense->row_offset[k + 1] - dense->row_offset[k], c = dense->col_offset[k + 1] - dense->col_offset[k];
      if (n < 0 || c < 0 || dense->row_offset[k + 1] > n_rows || dense->col_offset[k + 1] > n_cols)
        return fail(ctx, VIML_ERR_INVALID, "dense factors: row_offset and col_offset must be non-decreasing up to their totals");
      if (dense->jac_offset[k + 1] - dense->jac_offset[k] != n * c)
        return fail(ctx, VIML_ERR_INVALID, "dense factors: jac_offset does not match rows x columns");
    }
    // only now that every factor's columns lie inside [0, n_cols): the fused kernel keeps the lower triangle only and adds a
    // diagonal tile's a >= b half, so a column repeated inside a factor would count once there and twice in reduced_kernel
    std::vector<int64_t> seen(Dx, -1);
    for (int64_t k = 0; k < ND; ++k)
      for (int64_t a = dense->col_offset[k]; a < dense->col_offset[k + 1]; ++a) {
        if (seen[dense->col_index[a]] == k) return fail(ctx, VIML_ERR_INVALID, "dense factors: col_index repeats a column inside a factor");
        seen[dense->col_index[a]] = k;
      }
  }
  st.in(dense->window_offset, (size_t)W + 1, &dn->window_offset);
  st.in(dense->row_offset, (size_t)ND + 1, &dn->row_offset);
  st.in(dense->col_offset, (size_t)ND + 1, &dn->col_offset);
  st.in(dense->jac_offset, (size_t)ND + 1, &dn->jac_offset);
  st.in(dense->col_index, (size_t)n_cols, &dn->col_index);
  st.in(dense->residual, (size_t)n_rows, &dn->residual);
  st.in(dense->jacobian, (size_t)n_jac, &dn->jacobian);
  return VIML_OK;
}

// The extra tangent columns of a step: the inertial factors' when given, else the dense factors'.
int step_extra_dim(const viml_dense_factors* dense, const viml_inertial_factors* vi) {
  return vi ? vi->extra_dim : dense ? dense->extra_dim : 0;
}

// Device scratch of the H/b blocks and the Schur step of W windows (VIML_OUT_HB | VIML_OUT_SCHUR) into *o.
void stage_hb_scratch(Stager& st, int W, int D, int F, viml_linearize_out* o) {
  st.out((double*)nullptr, (size_t)W * D * D, &o->H_pp);
  st.out((double*)nullptr, (size_t)W * F * D, &o->H_lp);
  st.out((double*)nullptr, (size_t)W * F, &o->H_ll);
  st.out((double*)nullptr, (size_t)W * D, &o->b_p);
  st.out((double*)nullptr, (size_t)W * F, &o->b_l);
  st.out((double*)nullptr, (size_t)W * D * D, &o->S);
  st.out((double*)nullptr, (size_t)W * D, &o->g);
}

// The batch without its line factors (form: check_window_batch's): the marginalisation and the slide read the point factors only.
void stage_point_batch(viml_ctx* ctx, Stager& st, const viml_window_batch* in, BatchForm form, uint32_t flags, StagedBatch* b) {
  viml_window_batch pts = *in;
  pts.n_line_factors = 0;
  form.line_table = false;
  stage_batch(ctx, st, &pts, form, flags, b);
}

// The dense-block factors every kernel reads, over the CSR `c` of the IMU / prior factors of `v`.  ND = W + NI is an upper bound:
// the kernels read ND only as "any dense factors".
DenseArgs dense_view(const InertialArgs& v, const InertialCsr& c) {
  return DenseArgs{v.X, (int64_t)v.W + v.NI, c.window_offset, c.row_offset, c.col_offset, c.jac_offset, c.col_index, c.residual, c.jacobian};
}

// Evaluates the IMU / prior factors of `v` at (poses, ex_pose, extra), kept in `v`, into `csr`; csr.jacobian null: residuals only.
int enqueue_inertial_at(viml_ctx* ctx, InertialArgs& v, const double* poses, const double* ex_pose, const double* extra,
                        const InertialCsr& csr) {
  v.poses = poses, v.ex_pose = ex_pose, v.extra = extra;
  return viml_launch_inertial(ctx, v, viml_inertial_out{}, csr, csr.jacobian != nullptr);
}

// Everything one Gauss-Newton step enqueues (device pointers), staged once: viml_gn_step / viml_gn_step_vi enqueue one step,
// viml_solve_vi one per round.  The state the step starts from is b.a.poses, b.a.ex_pose, b.a.inv_depth and extra; x+ goes to o_*.
struct StepPlan {
  int W, X, Dx;
  bool vi;            // the dense-block factors are the IMU / prior factors
  bool fused;         // a step that builds and solves the reduced system in one kernel: Sx / gx are neither wanted nor staged
  StagedBatch b;      // the window batch and its observation / line tables
  DenseArgs dn;
  InertialArgs va;
  InertialCsr csr;
  double* res_plus;   // residuals of the IMU / prior factors at x+
  const double* extra;
  double *Sx, *gx, *dx, *cost;
  int32_t* solved;
  double *o_poses, *o_ex, *o_dep, *o_extra;
};

// Stages the inputs of viml_reduced_system / viml_gn_step / viml_gn_step_vi / viml_solve_vi (checked by check_step_inputs, which
// gave `form`), their scratch and the outputs of `rout` / `gout` (null fields: device scratch) into `st`.  The caller commits `st`,
// then calls expand_tables().
int stage_step(viml_ctx* ctx, Stager& st, const viml_window_batch* in, const BatchForm& form, const viml_dense_factors* dense,
               const double* extra_state, const viml_reduced_out* rout, const viml_gn_out* gout, uint32_t flags,
               const viml_inertial_factors* vi, StepPlan* s) {
  const int W = in->n_windows, P = in->poses_per_window, F = in->feats_per_window, D = 6 * (P + 1);
  *s = StepPlan{};
  s->W = W, s->X = step_extra_dim(dense, vi), s->Dx = D + s->X;
  const int X = s->X, Dx = s->Dx;
  s->vi = vi != nullptr, s->fused = gout && !(rout && (rout->Sx || rout->gx)) && gn_fused_takes(Dx);
  s->dn.X = X;
  int rc = stage_dense(ctx, st, dense, W, Dx, &s->dn);
  if (rc != VIML_OK) return rc;
  stage_batch(ctx, st, in, form, (flags & VIML_LOSS_CAUCHY) | VIML_OUT_HB | VIML_OUT_SCHUR, &s->b);
  st.in(extra_state, extra_state ? (size_t)W * X : 0, &s->extra);
  if (vi) {
    stage_inertial(st, vi, W, P, &s->va);
    stage_inertial_csr(st, s->va, &s->csr, &s->res_plus);
  }
  // scratch (host == nullptr) and outputs
  stage_hb_scratch(st, W, D, F, &s->b.a.out);
  if (!s->fused) {
    st.out(rout ? rout->Sx : nullptr, (size_t)W * Dx * Dx, &s->Sx);
    st.out(rout ? rout->gx : nullptr, (size_t)W * Dx, &s->gx);
  }
  if (gout) {
    st.out(gout->dx, (size_t)W * Dx, &s->dx);
    st.out(gout->cost, (size_t)W * 3, &s->cost);
    st.out(gout->solved, (size_t)W, &s->solved);
    st.out(gout->poses, (size_t)W * P * 7, &s->o_poses);
    st.out(gout->ex_pose, (size_t)W * 7, &s->o_ex);
    st.out(gout->inv_depth, (size_t)W * F, &s->o_dep);
    if (X > 0) st.out(gout->extra, (size_t)W * X, &s->o_extra);
  }
  return VIML_OK;
}

// One dogleg round of viml_solve_vi (VIML_SOLVE_DOGLEG): the per-window storage, the trust-region state it reads and the round.
struct DoglegRound {
  const DoglegArgs* g;
  const SolveState* state;
  double initial_radius;
  int round;
};

// The solve of a step: the system built and solved in one kernel where s.fused, else reduced_kernel into s.Sx / s.gx and the
// unfused solve.  lambda, lambda_w, gate (the windows solved), damp: see viml_launch_gn_reduced_solve.
int enqueue_solve(viml_ctx* ctx, const StepPlan& s, const DenseArgs& dn, double lambda, const double* lambda_w, const int32_t* gate,
                  const double* damp) {
  const LinearizeArgs& a = s.b.a;
  if (s.fused) return viml_launch_gn_reduced_solve(ctx, s.W, a.D, dn, a.out.S, a.out.g, lambda, s.dx, s.solved, s.cost, lambda_w, gate, damp);
  const int rc = viml_launch_reduced(ctx, s.W, a.D, dn, a.out.S, a.out.g, s.Sx, s.gx);
  if (rc != VIML_OK) return rc;
  return viml_launch_gn_solve(ctx, s.W, s.Dx, lambda, s.Sx, s.gx, s.dx, s.solved, s.cost, lambda_w, gate, damp);
}

// One step at the state of s.b.a / s.extra: without s.cost the reduced system Sx, gx alone; with it the cost at x, the solve (the
// system built in the solve kernel when s.fused), the update into s.o_* and the cost at x+.  lambda_w / running: see
// viml_launch_gn_reduced_solve (nullptr: `lambda`, every window).
// dg (nullable): the step is the dogleg step of viml.h instead.  The round linearises without the Schur step, forms the damping
// (dogleg_prepare) and runs the Schur step itself on the damped H_ll; the solve and dogleg_finish run where dg->g->fresh is set
// (round 0: every window), dogleg_step and everything after it where `running` is.
// With s.vi the dense-block factors are the window's prior and IMU factors, evaluated on the device at x (system, cost[0]) and at
// x+ (cost[1], exactly); s.dn is then replaced by their CSR.
int enqueue_step(viml_ctx* ctx, const StepPlan& s, double lambda, const double* lambda_w, const int32_t* running,
                 const DoglegRound* dg = nullptr) {
  const LinearizeArgs& a = s.b.a;
  const int W = s.W, D = a.D;
  const DoglegArgs* g = dg ? dg->g : nullptr;
  LinearizeArgs al = a;
  if (dg) al.flags &= ~VIML_OUT_SCHUR;
  int rc = viml_launch_linearize(ctx, al);
  InertialArgs va = s.va;
  if (rc == VIML_OK && s.vi) rc = enqueue_inertial_at(ctx, va, a.poses, a.ex_pose, s.extra, s.csr);
  if (rc != VIML_OK) return rc;
  const DenseArgs dn = s.vi ? dense_view(va, s.csr) : s.dn;
  if (!s.cost) return viml_launch_reduced(ctx, W, D, dn, a.out.S, a.out.g, s.Sx, s.gx);
  rc = viml_launch_cost(ctx, a, dn, nullptr, nullptr, 0, s.cost, running);
  const int32_t* gate = running;
  const double* damp = nullptr;
  if (rc == VIML_OK && g) {   // the dogleg's damping array instead of lambda diag(Sx); a new Gauss-Newton step where fresh is set
    rc = viml_launch_dogleg_prepare(ctx, a, dn, *g, dg->state, dg->round);
    // MarginalizationInfo::eps, as in viml_launch_linearize
    if (rc == VIML_OK)
      rc = viml_launch_schur(ctx, W, a.F, D, a.out.H_pp, a.out.H_lp, a.out.H_ll, a.out.b_p, a.out.b_l, a.out.S, a.out.g, 1e-8);
    lambda = 0.0, lambda_w = nullptr, gate = dg->round ? g->fresh : nullptr, damp = g->damp;
  }
  if (rc == VIML_OK) rc = enqueue_solve(ctx, s, dn, lambda, lambda_w, gate, damp);
  if (rc == VIML_OK && g) rc = viml_launch_dogleg_finish(ctx, a, dn, *g, dg->state, dg->round, s.dx, s.solved);
  if (rc == VIML_OK && g)
    rc = viml_launch_dogleg_step(ctx, W, *g, dg->state, dg->initial_radius, dg->round, running, s.dx, s.cost, s.solved);
  if (rc == VIML_OK)
    rc = viml_launch_gn_update(ctx, a, s.X, s.extra, s.dx, s.solved, s.o_poses, s.o_ex, s.o_dep, s.o_extra, running, g ? g->dl : nullptr);
  if (rc != VIML_OK) return rc;
  LinearizeArgs a2 = a;
  a2.poses = s.o_poses, a2.ex_pose = s.o_ex, a2.inv_depth = s.o_dep;
  rc = viml_launch_prep(ctx, a2);
  if (rc != VIML_OK) return rc;
  if (!s.vi) return viml_launch_cost(ctx, a2, dn, s.dx, s.solved, 1, s.cost, running);
  // f(x+): the IMU / prior residuals re-evaluated at x+ (same CSR structure), 1/2 |r|^2 without the linear model
  InertialCsr cp = s.csr;
  cp.residual = s.res_plus, cp.jacobian = nullptr;
  rc = enqueue_inertial_at(ctx, va, s.o_poses, s.o_ex, s.o_extra, cp);
  DenseArgs dp = dn;
  dp.residual = s.res_plus;
  if (rc == VIML_OK) rc = viml_launch_cost(ctx, a2, dp, nullptr, nullptr, 1, s.cost, running);
  return rc;
}

// The window batch (*form: how it carries its observations and line factors), with host pointers its indices too.
int check_batch(viml_ctx* ctx, const viml_window_batch* in, bool dev, BatchForm* form) {
  const int rc = check_window_batch(ctx, in, dev, form);
  if (rc != VIML_OK || dev || in->n_windows == 0) return rc;
  return check_batch_indices(ctx, in, *form, 0, in->n_point_factors, 0, in->n_line_factors);
}

// Checks shared by viml_reduced_system / viml_gn_step / viml_gn_step_vi / viml_solve_vi / viml_marginalize_vi: the batch, and with
// `vi` the inertial factors and the extra state.
int check_step_inputs(viml_ctx* ctx, const viml_window_batch* in, const viml_dense_factors* dense, const double* extra_state,
                      uint32_t flags, const viml_inertial_factors* vi, const char* who, BatchForm* form) {
  const bool dev = (flags & VIML_PTRS_DEVICE) != 0;
  int rc = check_batch(ctx, in, dev, form);
  if (rc != VIML_OK) return rc;
  const int P = in->poses_per_window, D = 6 * (P + 1);
  if (vi) {
    rc = check_inertial(ctx, vi, in->n_windows, P, dev);
    if (rc != VIML_OK) return rc;
    if (vi->extra_dim > 0 && !extra_state) {
      ctx->err = std::string(who) + ": extra_dim > 0 needs extra_state";
      return VIML_ERR_INVALID;
    }
  }
  const int X = step_extra_dim(dense, vi);
  const int64_t ND = dense && !vi ? dense->n_factors : 0;
  if (X < 0 || ND < 0 || D + X > kMaxDx) return fail(ctx, VIML_ERR_INVALID, "dense factors: extra_dim out of range (D + extra_dim <= 232)");
  return VIML_OK;
}

// viml_reduced_system / viml_gn_step / viml_gn_step_vi: one step (or the reduced system alone).
int run(viml_ctx* ctx, const viml_window_batch* in, const viml_dense_factors* dense, const double* extra_state,
        const viml_gn_options* opt, const viml_reduced_out* rout, const viml_gn_out* gout, uint32_t flags,
        const viml_inertial_factors* vi = nullptr) {
  if (vi) dense = nullptr;
  BatchForm form;
  int rc = check_step_inputs(ctx, in, dense, extra_state, flags, vi, "viml_gn_step_vi", &form);
  if (rc != VIML_OK) return rc;
  const int W = in->n_windows, F = in->feats_per_window, X = step_extra_dim(dense, vi);
  const bool step = gout != nullptr;
  if (step && !(gout->poses && gout->ex_pose && (F == 0 || gout->inv_depth) && gout->cost && gout->solved))
    return fail(ctx, VIML_ERR_INVALID, "viml_gn_step needs poses, ex_pose, inv_depth, cost and solved outputs");
  if (step && X > 0 && !gout->extra) return fail(ctx, VIML_ERR_INVALID, "viml_gn_step: extra_dim > 0 needs the extra output");
  if (!step && !(rout && rout->Sx && rout->gx)) return fail(ctx, VIML_ERR_INVALID, "viml_reduced_system needs Sx and gx");
  if (W == 0) return VIML_OK;
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  Stager st{ctx, (flags & VIML_PTRS_DEVICE) != 0};
  StepPlan s;
  rc = stage_step(ctx, st, in, form, dense, extra_state, rout, gout, flags, vi, &s);
  if (rc == VIML_OK) rc = st.commit();
  if (rc == VIML_OK) rc = expand_tables(ctx, s.b);
  if (rc == VIML_OK) rc = enqueue_step(ctx, s, opt ? opt->lambda : 0.0, nullptr, nullptr);
  if (rc != VIML_OK) return rc;
  return st.finish();
}

int check_solve_options(viml_ctx* ctx, const viml_solve_options* o) {
  if (!o) return fail(ctx, VIML_ERR_INVALID, "viml_solve_vi: null options");
  if (o->max_iterations <= 0 || o->max_consecutive_invalid < 0)
    return fail(ctx, VIML_ERR_INVALID, "viml_solve_vi: max_iterations must be > 0 and max_consecutive_invalid >= 0");
  if (!(std::isfinite(o->min_radius) && std::isfinite(o->initial_radius) && std::isfinite(o->max_radius) && o->min_radius > 0.0 &&
        o->min_radius <= o->initial_radius && o->initial_radius <= o->max_radius))
    return fail(ctx, VIML_ERR_INVALID, "viml_solve_vi: radii must be finite with 0 < min_radius <= initial_radius <= max_radius");
  if (!(o->min_relative_decrease >= 0.0 && o->function_tolerance >= 0.0 && o->parameter_tolerance >= 0.0))
    return fail(ctx, VIML_ERR_INVALID, "viml_solve_vi: min_relative_decrease and the tolerances must be >= 0");
  return VIML_OK;
}

// The host-pointer preconditions viml_marginalize_vi and viml_slide_vi share (viml.h), after the batch's indices are checked: every
// margin[w] is 0 or 1, and no feature has point factors with both i == 0 and i != 0 (the outgoing frame anchors all of a feature's
// factors or none).
int check_margin_and_anchors(viml_ctx* ctx, const viml_window_batch* in, const int32_t* margin, const char* who) {
  const int W = in->n_windows, F = in->feats_per_window;
  for (int w = 0; w < W; ++w)
    if (margin[w] != VIML_MARGIN_OLD && margin[w] != VIML_MARGIN_SECOND_NEW) {
      ctx->err = std::string(who) + ": margin[w] must be 0 or 1";
      return VIML_ERR_INVALID;
    }
  std::vector<uint8_t> feat(F);
  for (int w = 0; w < W; ++w) {
    std::fill(feat.begin(), feat.end(), 0);
    for (int64_t k = in->pf_window_offset[w]; k < in->pf_window_offset[w + 1]; ++k) {
      const uint32_t ix = in->pf_idx[k];
      const int f = ix >> 16;
      feat[f] |= (ix & 0xffu) == 0 ? 1 : 2;
      if (feat[f] == 3) {
        ctx->err = std::string(who) + ": a feature has factors with both i == 0 and i != 0";
        return VIML_ERR_INVALID;
      }
    }
  }
  return VIML_OK;
}

// viml_marginalize_vi's preconditions on host pointers (viml.h), after check_step_inputs.  The kept dimension and block count of every
// window follow marg_gather_kernel's selection.
int check_marginalize_vi(viml_ctx* ctx, const viml_window_batch* in, const viml_inertial_factors* vi, const int32_t* margin,
                         const viml_prior_out* out) {
  const int W = in->n_windows, P = in->poses_per_window;
  int rc = check_margin_and_anchors(ctx, in, margin, "viml_marginalize_vi");
  if (rc != VIML_OK) return rc;
  for (int64_t k = 0; k < vi->n_imu; ++k)
    if (vi->imu_sb[2 * k] != 9 * vi->imu_pose[2 * k] || vi->imu_sb[2 * k + 1] != 9 * vi->imu_pose[2 * k + 1])
      return fail(ctx, VIML_ERR_INVALID, "viml_marginalize_vi: the speed-bias of pose p must sit at extra offset 9p (imu_sb == {9i, 9j})");
  const int NS = 2 * P + 1;
  std::vector<uint8_t> touch(NS);
  for (int w = 0; w < W; ++w) {
    const bool old = margin[w] == VIML_MARGIN_OLD;
    const int n_in = vi->prior_n_max > 0 ? vi->prior_n[w] : 0, nb_in = n_in > 0 ? vi->prior_n_blocks[w] : 0;
    std::fill(touch.begin(), touch.end(), 0);
    bool has = false;
    for (int b = 0; b < nb_in; ++b) {
      const int32_t* blk = vi->prior_block + ((size_t)w * vi->prior_max_blocks + b) * 4;
      int s = P;
      if (blk[0] == VIML_BLOCK_POSE) {
        s = blk[1];
      } else if (blk[0] == VIML_BLOCK_EXTRA) {
        if (blk[2] != 9 || blk[1] % 9 != 0 || blk[1] / 9 >= P)
          return fail(ctx, VIML_ERR_INVALID, "viml_marginalize_vi: an extra block of the prior must be the 9-block of a speed-bias (offset 9p, p < P)");
        s = P + 1 + blk[1] / 9;
        if (!old && blk[1] / 9 == P - 2)
          return fail(ctx, VIML_ERR_INVALID, "viml_marginalize_vi: MARGIN_SECOND_NEW with the speed-bias of pose P-2 in the prior");
      }
      has = has || s == P - 2;
      touch[s] = 1;
    }
    for (int64_t k = in->pf_window_offset[w]; old && k < in->pf_window_offset[w + 1]; ++k) {
      const uint32_t ix = in->pf_idx[k];
      if ((ix & 0xffu) == 0) touch[0] = touch[(ix >> 8) & 0xffu] = touch[P] = 1;
    }
    int n = 0, nb = 0;
    if (!old && !has) {
      n = n_in, nb = nb_in;
    } else {
      if (old && vi->n_imu > 0)
        for (int64_t f = vi->imu_window_offset[w]; f < vi->imu_window_offset[w + 1]; ++f)
          if (vi->imu_pose[2 * f] == 0 && vi->imu_preint[f * 17] < 10.0) {
            const int j = vi->imu_pose[2 * f + 1];
            touch[0] = touch[j] = touch[P + 1] = touch[P + 1 + j] = 1;
          }
      const int dp = old ? 0 : P - 2, ds = old ? P + 1 : -1;
      for (int s = 0; s < NS; ++s)
        if (touch[s] && s != dp && s != ds) n += s <= P ? 6 : 9, ++nb;
    }
    if (n > out->prior_n_max || nb > out->prior_max_blocks)
      return fail(ctx, VIML_ERR_INVALID, "viml_marginalize_vi: a window's kept dimension or block count exceeds the output's prior_n_max / prior_max_blocks");
  }
  return VIML_OK;
}

}  // namespace

extern "C" {

int viml_marginalize_vi(viml_ctx* ctx, const viml_window_batch* in, const viml_inertial_factors* vi, const double* extra_state,
                        const int32_t* margin, const viml_prior_out* out, uint32_t flags) {
  if (!ctx) return VIML_ERR_INVALID;
  if (!out) return fail(ctx, VIML_ERR_INVALID, "null output struct");
  if (!vi) return fail(ctx, VIML_ERR_INVALID, "null inertial factors");
  const bool dev = (flags & VIML_PTRS_DEVICE) != 0;
  BatchForm form;
  int rc = check_step_inputs(ctx, in, nullptr, extra_state, flags, vi, "viml_marginalize_vi", &form);
  if (rc != VIML_OK) return rc;
  const int W = in->n_windows, P = in->poses_per_window, F = in->feats_per_window, D = 6 * (P + 1), X = vi->extra_dim, Dx = D + X;
  const int64_t NP = in->n_point_factors;
  if (P < 2) return fail(ctx, VIML_ERR_INVALID, "viml_marginalize_vi: needs P >= 2");
  if (W == 0) return VIML_OK;
  const int n_max = out->prior_n_max, mb = out->prior_max_blocks;
  if (!margin || n_max < 0 || mb < 0 || !out->prior_n || !out->prior_n_blocks ||
      (n_max > 0 && (!out->prior_jacobian || !out->prior_residual)) || (mb > 0 && (!out->prior_block || !out->prior_x0)))
    return fail(ctx, VIML_ERR_INVALID, "viml_marginalize_vi: null margin or output array, or negative output sizes");
  if (!dev) {
    rc = check_marginalize_vi(ctx, in, vi, margin, out);
    if (rc != VIML_OK) return rc;
  }
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  Stager st{ctx, dev};
  StagedBatch b;   // line factors take no part (est.cpp:1911-2046 adds none)
  stage_point_batch(ctx, st, in, form, (flags & VIML_LOSS_CAUCHY) | VIML_OUT_HB | VIML_OUT_SCHUR, &b);
  LinearizeArgs& a = b.a;
  MargViArgs g{};
  g.W = W, g.P = P, g.D = D, g.X = X;
  g.pm = std::min(Dx, 15 + n_max);   // m <= 15: pose 0 and speed-bias 0
  const double* extra = nullptr;
  st.in(extra_state, extra_state ? (size_t)W * X : 0, &extra);
  st.in(margin, (size_t)W, &g.margin);
  stage_inertial(st, vi, W, P, &g.v);
  double* res_plus = nullptr;
  stage_inertial_csr(st, g.v, &g.csr, &res_plus);
  st.out((int32_t*)nullptr, (size_t)W, &g.cnt);
  st.out((int32_t*)nullptr, (size_t)W + 1, &g.sel_offset);
  st.out((uint32_t*)nullptr, (size_t)NP, &g.sel_idx);
  st.out((double*)nullptr, (size_t)NP * 4, &g.sel_obs);
  if (in->pf_pts_i_z) st.out((double*)nullptr, (size_t)NP, &g.sel_z);
  stage_hb_scratch(st, W, D, F, &a.out);
  double *Sx = nullptr, *gx = nullptr;
  st.out((double*)nullptr, (size_t)W * Dx * Dx, &Sx);
  st.out((double*)nullptr, (size_t)W * Dx, &gx);
  st.out((double*)nullptr, (size_t)W * g.pm * g.pm, &g.A);
  st.out((double*)nullptr, (size_t)W * g.pm, &g.b);
  st.out((int2*)nullptr, (size_t)W, &g.sizes);
  // entries past n / n_blocks keep the caller's content
  g.out.prior_n_max = n_max, g.out.prior_max_blocks = mb;
  st.out(out->prior_n, (size_t)W, &g.out.prior_n);
  st.out(out->prior_n_blocks, (size_t)W, &g.out.prior_n_blocks);
  st.inout(out->prior_jacobian, (size_t)W * n_max * n_max, &g.out.prior_jacobian);
  st.inout(out->prior_residual, (size_t)W * n_max, &g.out.prior_residual);
  st.inout(out->prior_block, (size_t)W * mb * 4, &g.out.prior_block);
  st.inout(out->prior_x0, (size_t)W * mb * VIML_PRIOR_X0_STRIDE, &g.out.prior_x0);
  rc = st.commit();
  if (rc == VIML_OK) rc = expand_tables(ctx, b);
  if (rc != VIML_OK) return rc;
  // the IMU factors and the prior at x, into the dense-factor CSR
  rc = enqueue_inertial_at(ctx, g.v, a.poses, a.ex_pose, extra, g.csr);
  if (rc != VIML_OK) return rc;
  g.pf_window_offset = a.pf_window_offset, g.pf_idx = a.pf_idx, g.pf_obs = a.pf_obs, g.pf_pts_i_z = a.pf_pts_i_z;
  rc = viml_launch_marg_select(ctx, g);
  if (rc != VIML_OK) return rc;
  // the selected point factors: S, g of the window with their features eliminated (NP is an upper bound of their number)
  a.pf_window_offset = g.sel_offset, a.pf_idx = g.sel_idx, a.pf_obs = g.sel_obs, a.pf_pts_i_z = g.sel_z;
  rc = viml_launch_linearize(ctx, a);
  if (rc != VIML_OK) return rc;
  rc = viml_launch_reduced(ctx, W, D, dense_view(g.v, g.csr), a.out.S, a.out.g, Sx, gx);
  if (rc != VIML_OK) return rc;
  g.Sx = Sx, g.gx = gx;
  rc = viml_launch_marg_gather(ctx, g);
  if (rc == VIML_OK && n_max > 0)   // MarginalizationInfo::eps (marginalization_factor.h:70)
    rc = viml_launch_marginalize(ctx, W, g.pm, 0, 1e-8, g.A, g.b, nullptr, nullptr, g.out.prior_jacobian, g.out.prior_residual, g.sizes,
                                 15, n_max);
  if (rc != VIML_OK) return rc;
  return st.finish();
}

int viml_slide_vi(viml_ctx* ctx, const viml_window_batch* in, const double* extra_state, int32_t extra_dim, const int32_t* margin,
                  double init_depth, const viml_slide_out* out, uint32_t flags) {
  if (!ctx) return VIML_ERR_INVALID;
  if (!out) return fail(ctx, VIML_ERR_INVALID, "null output struct");
  const bool dev = (flags & VIML_PTRS_DEVICE) != 0;
  BatchForm form;
  int rc = check_batch(ctx, in, dev, &form);
  if (rc != VIML_OK) return rc;
  const int W = in->n_windows, P = in->poses_per_window, F = in->feats_per_window, X = extra_dim;
  if (P < 2) return fail(ctx, VIML_ERR_INVALID, "viml_slide_vi: needs P >= 2");
  if (X < 9 * P) return fail(ctx, VIML_ERR_INVALID, "viml_slide_vi: extra_dim must hold the P speed-bias blocks (X >= 9P)");
  if (!(std::isfinite(init_depth) && init_depth > 0.0)) return fail(ctx, VIML_ERR_INVALID, "viml_slide_vi: init_depth must be finite and > 0");
  if (W == 0) return VIML_OK;
  if (!margin || !extra_state || !out->poses || !out->ex_pose || (F > 0 && !out->inv_depth) || !out->extra)
    return fail(ctx, VIML_ERR_INVALID, "viml_slide_vi: null margin, extra_state or output array");
  if (!dev) {
    rc = check_margin_and_anchors(ctx, in, margin, "viml_slide_vi");
    if (rc != VIML_OK) return rc;
  }
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  Stager st{ctx, dev};
  StagedBatch b;
  stage_point_batch(ctx, st, in, form, 0, &b);
  SlideArgs s{};
  s.W = W, s.P = P, s.F = F, s.X = X, s.init_depth = init_depth;
  st.in(margin, (size_t)W, &s.margin);
  st.in(extra_state, (size_t)W * X, &s.extra);
  st.out(out->poses, (size_t)W * P * 7, &s.out.poses);
  st.out(out->ex_pose, (size_t)W * 7, &s.out.ex_pose);
  st.out(out->inv_depth, (size_t)W * F, &s.out.inv_depth);
  st.out(out->extra, (size_t)W * X, &s.out.extra);
  rc = st.commit();
  if (rc == VIML_OK) rc = expand_tables(ctx, b);
  if (rc != VIML_OK) return rc;
  const LinearizeArgs& a = b.a;
  s.poses = a.poses, s.ex_pose = a.ex_pose, s.inv_depth = a.inv_depth;
  s.pf_window_offset = a.pf_window_offset, s.pf_idx = a.pf_idx, s.pf_obs = a.pf_obs, s.pf_pts_i_z = a.pf_pts_i_z;
  rc = viml_launch_slide(ctx, s);
  if (rc != VIML_OK) return rc;
  return st.finish();
}

int viml_reduced_system(viml_ctx* ctx, const viml_window_batch* in, const viml_dense_factors* dense, const viml_reduced_out* out,
                        uint32_t flags) {
  if (!ctx) return VIML_ERR_INVALID;
  return run(ctx, in, dense, nullptr, nullptr, out, nullptr, flags);
}

int viml_reduced_from_schur(viml_ctx* ctx, int32_t W, int32_t D, const double* S, const double* g, const viml_dense_factors* dense,
                            const viml_reduced_out* out, uint32_t flags) {
  if (!ctx) return VIML_ERR_INVALID;
  const int X = dense ? dense->extra_dim : 0, Dx = D + X;
  const int64_t ND = dense ? dense->n_factors : 0;
  if (W < 0 || D < 1 || X < 0 || ND < 0 || !S || !g || !out || !out->Sx || !out->gx)
    return fail(ctx, VIML_ERR_INVALID, "viml_reduced_from_schur: bad arguments");
  if (W == 0) return VIML_OK;
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  Stager st{ctx, (flags & VIML_PTRS_DEVICE) != 0};
  const double *dS = nullptr, *dg = nullptr;
  st.in(S, (size_t)W * D * D, &dS);
  st.in(g, (size_t)W * D, &dg);
  DenseArgs dn{};
  dn.X = X;
  int rc = stage_dense(ctx, st, dense, W, Dx, &dn);
  if (rc != VIML_OK) return rc;
  double *Sx = nullptr, *gx = nullptr;
  st.out(out->Sx, (size_t)W * Dx * Dx, &Sx);
  st.out(out->gx, (size_t)W * Dx, &gx);
  rc = st.commit();
  if (rc != VIML_OK) return rc;
  rc = viml_launch_reduced(ctx, W, D, dn, dS, dg, Sx, gx);
  if (rc != VIML_OK) return rc;
  return st.finish();
}

int viml_gn_step(viml_ctx* ctx, const viml_window_batch* in, const viml_dense_factors* dense, const double* extra_state,
                 const viml_gn_options* opt, const viml_gn_out* out, uint32_t flags) {
  if (!ctx) return VIML_ERR_INVALID;
  if (!out) return fail(ctx, VIML_ERR_INVALID, "null output struct");
  return run(ctx, in, dense, extra_state, opt, nullptr, out, flags);
}

int viml_gn_step_vi(viml_ctx* ctx, const viml_window_batch* in, const viml_inertial_factors* vi, const double* extra_state,
                    const viml_gn_options* opt, const viml_gn_out* out, uint32_t flags) {
  if (!ctx) return VIML_ERR_INVALID;
  if (!out) return fail(ctx, VIML_ERR_INVALID, "null output struct");
  if (!vi) return fail(ctx, VIML_ERR_INVALID, "null inertial factors");
  return run(ctx, in, nullptr, extra_state, opt, nullptr, out, flags, vi);
}

int viml_solve_vi(viml_ctx* ctx, const viml_window_batch* in, const viml_inertial_factors* vi, const double* extra_state,
                  const viml_solve_options* opt, const viml_solve_out* out, uint32_t flags) {
  if (!ctx) return VIML_ERR_INVALID;
  if (!out) return fail(ctx, VIML_ERR_INVALID, "null output struct");
  if (!vi) return fail(ctx, VIML_ERR_INVALID, "null inertial factors");
  BatchForm form;
  int rc = check_step_inputs(ctx, in, nullptr, extra_state, flags, vi, "viml_solve_vi", &form);
  if (rc == VIML_OK) rc = check_solve_options(ctx, opt);
  if (rc != VIML_OK) return rc;
  const int W = in->n_windows, P = in->poses_per_window, F = in->feats_per_window, X = vi->extra_dim, M = opt->max_iterations;
  if (!(out->poses && out->ex_pose && (F == 0 || out->inv_depth) && (X == 0 || out->extra) && out->status && out->iterations &&
        out->accepted && out->cost))
    return fail(ctx, VIML_ERR_INVALID, "viml_solve_vi needs poses, ex_pose, inv_depth (F > 0), extra (X > 0), status, iterations, "
                                       "accepted and cost outputs");
  if (W == 0) return VIML_OK;
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  Stager st{ctx, (flags & VIML_PTRS_DEVICE) != 0};
  StepPlan s;
  const viml_gn_out scratch{};   // x+, dx, cost and solved of every round stay on the device
  rc = stage_step(ctx, st, in, form, nullptr, extra_state, nullptr, &scratch, flags, vi, &s);
  if (rc != VIML_OK) return rc;
  SolveArgs sa{};
  sa.opt = *opt;
  sa.P = P, sa.F = F, sa.X = X, sa.Dx = s.Dx;
  st.out((SolveState*)nullptr, (size_t)W, &sa.state);
  st.out((int32_t*)nullptr, (size_t)W, &sa.running);
  st.out((double*)nullptr, (size_t)W, &sa.lambda_w);
  st.out((double*)nullptr, (size_t)W * P * 7, &sa.x_poses);
  st.out((double*)nullptr, (size_t)W * 7, &sa.x_ex);
  st.out((double*)nullptr, (size_t)W * F, &sa.x_dep);
  st.out((double*)nullptr, (size_t)W * X, &sa.x_extra);
  st.out(out->poses, (size_t)W * P * 7, &sa.out.poses);
  st.out(out->ex_pose, (size_t)W * 7, &sa.out.ex_pose);
  st.out(out->inv_depth, (size_t)W * F, &sa.out.inv_depth);
  st.out(out->extra, (size_t)W * X, &sa.out.extra);
  st.out(out->status, (size_t)W, &sa.out.status);
  st.out(out->iterations, (size_t)W, &sa.out.iterations);
  st.out(out->accepted, (size_t)W, &sa.out.accepted);
  st.out(out->cost, (size_t)W * 2, &sa.out.cost);
  st.out(out->radius, out->radius ? (size_t)W : 0, &sa.out.radius);
  st.out(out->trace, out->trace ? (size_t)W * M * 4 : 0, &sa.out.trace);
  const bool dogleg = (flags & VIML_SOLVE_DOGLEG) != 0;
  DoglegArgs g{};
  if (dogleg) {
    const size_t N = (size_t)s.Dx + F;
    g.Dx = s.Dx, g.F = F;
    for (double** p : {&g.s, &g.d, &g.gamma, &g.w, &g.gn}) st.out((double*)nullptr, (size_t)W * N, p);
    st.out((double*)nullptr, (size_t)W * F, &g.hll);
    st.out((double*)nullptr, (size_t)W * F, &g.dl);
    st.out((double*)nullptr, (size_t)W * s.Dx, &g.damp);
    st.out((double*)nullptr, (size_t)W * kDoglegScal, &g.scal);
    st.out((int32_t*)nullptr, (size_t)W, &g.fresh);
  }
  rc = st.commit();
  if (rc == VIML_OK) rc = expand_tables(ctx, s.b);
  if (rc != VIML_OK) return rc;
  // the rounds work on a copy of the initial state: the inputs stay untouched
  const size_t n_pose = (size_t)W * P * 7, n_ex = (size_t)W * 7, n_dep = (size_t)W * F, n_extra = (size_t)W * X;
  VIML_TRY_CUDA(ctx, cudaMemcpyAsync(sa.x_poses, s.b.a.poses, n_pose * 8, cudaMemcpyDeviceToDevice, ctx->stream));
  VIML_TRY_CUDA(ctx, cudaMemcpyAsync(sa.x_ex, s.b.a.ex_pose, n_ex * 8, cudaMemcpyDeviceToDevice, ctx->stream));
  if (n_dep) VIML_TRY_CUDA(ctx, cudaMemcpyAsync(sa.x_dep, s.b.a.inv_depth, n_dep * 8, cudaMemcpyDeviceToDevice, ctx->stream));
  if (n_extra) VIML_TRY_CUDA(ctx, cudaMemcpyAsync(sa.x_extra, s.extra, n_extra * 8, cudaMemcpyDeviceToDevice, ctx->stream));
  s.b.a.poses = sa.x_poses, s.b.a.ex_pose = sa.x_ex, s.b.a.inv_depth = sa.x_dep, s.extra = sa.x_extra;
  sa.p_poses = s.o_poses, sa.p_ex = s.o_ex, sa.p_dep = s.o_dep, sa.p_extra = s.o_extra;
  sa.dx = s.dx, sa.cost = s.cost, sa.solved = s.solved;
  if (dogleg) sa.dogleg = g.scal, sa.fresh = g.fresh;
  // round 0 runs every window at lambda = 1 / initial_radius; policy_kernel then starts each window's state from that step and
  // hands the next round its running flags and lambdas
  // (dogleg: round 0 forms every window's step at initial_radius and mu = 1e-8)
  for (int r = 0; r < M && rc == VIML_OK; ++r) {
    const DoglegRound dg{&g, sa.state, opt->initial_radius, r};
    rc = enqueue_step(ctx, s, 1.0 / opt->initial_radius, r ? sa.lambda_w : nullptr, r ? sa.running : nullptr, dogleg ? &dg : nullptr);
    if (rc == VIML_OK) rc = viml_launch_solve_policy(ctx, W, sa, r);
  }
  if (rc != VIML_OK) return rc;
  return st.finish();
}

int viml_inertial_evaluate(viml_ctx* ctx, const viml_window_batch* state, const double* extra_state, const viml_inertial_factors* vi,
                           const viml_inertial_out* out, uint32_t flags) {
  if (!ctx) return VIML_ERR_INVALID;
  if (!state || !out) return fail(ctx, VIML_ERR_INVALID, "viml_inertial_evaluate: null arguments");
  const int W = state->n_windows, P = state->poses_per_window;
  if (W < 0 || P < 1 || P > 255) return fail(ctx, VIML_ERR_INVALID, "window batch sizes out of range");
  const bool dev = (flags & VIML_PTRS_DEVICE) != 0;
  int rc = check_inertial(ctx, vi, W, P, dev);
  if (rc != VIML_OK) return rc;
  if (W > 0 && (!state->poses || !state->ex_pose)) return fail(ctx, VIML_ERR_INVALID, "null input array");
  if (vi->extra_dim > 0 && !extra_state) return fail(ctx, VIML_ERR_INVALID, "viml_inertial_evaluate: extra_dim > 0 needs extra_state");
  if (W == 0) return VIML_OK;
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  Stager st{ctx, dev};
  InertialArgs v;
  stage_inertial(st, vi, W, P, &v);
  st.in(state->poses, (size_t)W * P * 7, &v.poses);
  st.in(state->ex_pose, (size_t)W * 7, &v.ex_pose);
  st.in(extra_state, extra_state ? (size_t)W * v.X : 0, &v.extra);
  const size_t NI = (size_t)v.NI;
  viml_inertial_out o{};
  st.out(out->imu_residual, out->imu_residual ? NI * 15 : 0, &o.imu_residual);
  st.out(out->imu_jac_pose_i, out->imu_jac_pose_i ? NI * 105 : 0, &o.imu_jac_pose_i);
  st.out(out->imu_jac_sb_i, out->imu_jac_sb_i ? NI * 135 : 0, &o.imu_jac_sb_i);
  st.out(out->imu_jac_pose_j, out->imu_jac_pose_j ? NI * 105 : 0, &o.imu_jac_pose_j);
  st.out(out->imu_jac_sb_j, out->imu_jac_sb_j ? NI * 135 : 0, &o.imu_jac_sb_j);
  // in-out: rows past n_w keep the caller's content
  st.inout(out->prior_residual, out->prior_residual ? (size_t)W * v.n_max : 0, &o.prior_residual);
  rc = st.commit();
  if (rc == VIML_OK) rc = viml_launch_inertial(ctx, v, o, InertialCsr{}, false);
  if (rc != VIML_OK) return rc;
  return st.finish();
}

int viml_triangulate_batch(viml_ctx* ctx, const viml_triangulate_in* in, double init_depth, double* depth, uint32_t flags) {
  if (!ctx) return VIML_ERR_INVALID;
  if (!in || !depth) return fail(ctx, VIML_ERR_INVALID, "viml_triangulate_batch: null arguments");
  const int W = in->n_windows, P = in->poses_per_window;
  const int64_t NF = in->n_features;
  if (W < 0 || P < 1 || NF < 0) return fail(ctx, VIML_ERR_INVALID, "viml_triangulate_batch: sizes out of range");
  if (NF == 0) return VIML_OK;
  if (!in->poses || !in->ex_pose || !in->feat_window || !in->start_frame || !in->obs_offset || !in->points)
    return fail(ctx, VIML_ERR_INVALID, "viml_triangulate_batch: null input array");
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  const bool dev = (flags & VIML_PTRS_DEVICE) != 0;
  int64_t nobs = 0;
  if (dev) {
    VIML_TRY_CUDA(ctx, cudaMemcpyAsync(&nobs, in->obs_offset + NF, 8, cudaMemcpyDeviceToHost, ctx->stream));
    VIML_TRY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  } else {
    nobs = in->obs_offset[NF];
    for (int64_t l = 0; l < NF; ++l)
      if (in->feat_window[l] < 0 || in->feat_window[l] >= W) return fail(ctx, VIML_ERR_INVALID, "viml_triangulate_batch: feat_window out of range");
  }
  Stager st{ctx, dev};
  const double *dp = nullptr, *de = nullptr, *dpts = nullptr;
  const int32_t *dw = nullptr, *ds = nullptr;
  const int64_t* doff = nullptr;
  st.in(in->poses, (size_t)W * P * 7, &dp);
  st.in(in->ex_pose, (size_t)W * 7, &de);
  st.in(in->feat_window, (size_t)NF, &dw);
  st.in(in->start_frame, (size_t)NF, &ds);
  st.in(in->obs_offset, (size_t)NF + 1, &doff);
  st.in(in->points, (size_t)nobs * 3, &dpts);
  double* dd = nullptr;
  st.out(depth, (size_t)NF, &dd);
  int rc = st.commit();
  if (rc != VIML_OK) return rc;
  rc = viml_launch_triangulate(ctx, P, NF, dp, de, dw, ds, doff, dpts, init_depth, dd);
  if (rc != VIML_OK) return rc;
  return st.finish();
}

int viml_load_line_map(viml_ctx* ctx, const char* path, int64_t* n_lines) {
  if (!ctx) return VIML_ERR_INVALID;
  if (!path) return fail(ctx, VIML_ERR_INVALID, "null map path");
  std::ifstream f(path);
  if (!f.is_open()) return fail(ctx, VIML_ERR_INVALID, "cannot open the line map file");
  std::vector<double> rows;
  std::string fline;
  while (std::getline(f, fline)) {   // parameters.cpp:53-59: one Vector6d per text line
    std::istringstream iss(fline);
    double v[6] = {0, 0, 0, 0, 0, 0};
    for (int k = 0; k < 6; ++k)
      if (!(iss >> v[k])) {   // fields after a failed extraction: 0 here, uninitialised in the reference
        for (int q = k; q < 6; ++q) v[q] = 0.0;
        break;
      }
    rows.insert(rows.end(), v, v + 6);
  }
  if (n_lines) *n_lines = (int64_t)(rows.size() / 6);
  return viml_set_map(ctx, rows.data(), (int64_t)(rows.size() / 6));
}

}  // extern "C"
