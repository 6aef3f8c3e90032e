// viml_api.cu — the C-ABI of include/viml.h: context lifetime, host<->device staging, entry points.
// No CPU fallback anywhere: every compute path ends in a kernel launch on the context's device.
#include <dlfcn.h>

#include <cmath>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <numeric>
#include <vector>

#include "common.cuh"

namespace {

thread_local std::string g_create_error;

// c* = min{ c in [0,1] : acos(c) <= angle_th } with the host libm (the reference's acos, estimator.cpp:608).
double cos_threshold(double angle_th) {
  if (!(std::acos(1.0) <= angle_th)) return INFINITY;
  if (std::acos(0.0) <= angle_th) return 0.0;
  uint64_t lo, hi;
  double dlo = 0.0, dhi = 1.0;
  std::memcpy(&lo, &dlo, 8);
  std::memcpy(&hi, &dhi, 8);
  while (hi - lo > 1) {
    const uint64_t mid = lo + (hi - lo) / 2;
    double dm;
    std::memcpy(&dm, &mid, 8);
    if (std::acos(dm) <= angle_th) hi = mid; else lo = mid;
  }
  double r;
  std::memcpy(&r, &hi, 8);
  return r;
}

}  // namespace

static void drop_prof_events(viml_ctx* ctx) {
  for (auto& v : ctx->prof_events) {
    for (auto& pr : v) {
      cudaEventDestroy(pr.first);
      cudaEventDestroy(pr.second);
    }
    v.clear();
  }
}

extern "C" {

int viml_abi_version(void) { return VIML_ABI_VERSION; }

int viml_create(viml_ctx** out, const viml_config* cfg, int device) {
  if (!out || !cfg) return VIML_ERR_INVALID;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return VIML_ERR_NO_DEVICE;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return VIML_ERR_NO_DEVICE;
  if (prop.major != 10) return VIML_ERR_NO_DEVICE;  // the library only carries sm_100a code
  if (cudaSetDevice(device) != cudaSuccess) return VIML_ERR_NO_DEVICE;
  viml_ctx* ctx = new viml_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  ctx->cfg = *cfg;
  ctx->cos_th = cos_threshold(cfg->angle_th);
  ctx->nan_angle_passes = !(3.1415926 > cfg->angle_th);
  if (const char* e = getenv("VIML_FORCE_GENERIC")) ctx->force_generic = e[0] == '1';  // test hook
  if (const char* e = getenv("VIML_BRUTE_CULL")) ctx->brute_cull = e[0] == '1';
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->copy_stream2, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_a, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_b, cudaEventDisableTiming) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming) != cudaSuccess) {
    delete ctx;
    return VIML_ERR_CUDA;
  }
  *out = ctx;
  return VIML_OK;
}

void viml_destroy(viml_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  drop_prof_events(ctx);
  ctx->in_arena.release();
  ctx->out_arena.release();
  if (ctx->h_stage_in) cudaFreeHost(ctx->h_stage_in);
  if (ctx->h_stage_out) cudaFreeHost(ctx->h_stage_out);
  ctx->scratch.release();
  ctx->scratch2.release();
  ctx->scratch3.release();
  ctx->s_full.release();
  if (ctx->d_map) cudaFree(ctx->d_map);
  if (ctx->d_map_sorted) cudaFree(ctx->d_map_sorted);
  if (ctx->d_map_orig) cudaFree(ctx->d_map_orig);
  if (ctx->d_tile_sphere) cudaFree(ctx->d_tile_sphere);
  if (ctx->d_group_sphere) cudaFree(ctx->d_group_sphere);
  if (ctx->d_assoc_stats) cudaFree(ctx->d_assoc_stats);
  if (ctx->d_fov_slots) cudaFree(ctx->d_fov_slots);
  if (ctx->d_fov_slot_count) cudaFree(ctx->d_fov_slot_count);
  if (ctx->ev_a) cudaEventDestroy(ctx->ev_a);
  if (ctx->ev_b) cudaEventDestroy(ctx->ev_b);
  if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->copy_stream2) cudaStreamDestroy(ctx->copy_stream2);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->nccl_lib) dlclose(ctx->nccl_lib);
  delete ctx;
}

const char* viml_last_error(const viml_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int viml_sync(viml_ctx* ctx) {
  if (!ctx) return VIML_ERR_INVALID;
  VIML_TRY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return VIML_OK;
}

void* viml_stream(viml_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int viml_host_alloc(void** p, size_t bytes) {
  if (!p) return VIML_ERR_INVALID;
  return cudaHostAlloc(p, bytes, cudaHostAllocDefault) == cudaSuccess ? VIML_OK : VIML_ERR_CUDA;
}
int viml_host_free(void* p) { return cudaFreeHost(p) == cudaSuccess ? VIML_OK : VIML_ERR_CUDA; }

int viml_device_alloc(viml_ctx* ctx, void** p, size_t bytes) {
  if (!ctx || !p) return VIML_ERR_INVALID;
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  VIML_TRY_CUDA(ctx, cudaMalloc(p, bytes));
  return VIML_OK;
}
int viml_device_free(viml_ctx* ctx, void* p) {
  if (!ctx) return VIML_ERR_INVALID;
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  VIML_TRY_CUDA(ctx, cudaFree(p));
  return VIML_OK;
}
int viml_memcpy_h2d(viml_ctx* ctx, void* dst, const void* src, size_t bytes) {
  if (!ctx) return VIML_ERR_INVALID;
  VIML_TRY_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return VIML_OK;
}
int viml_memcpy_d2h(viml_ctx* ctx, void* dst, const void* src, size_t bytes) {
  if (!ctx) return VIML_ERR_INVALID;
  VIML_TRY_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  return VIML_OK;
}

int64_t viml_kernel_launches(const viml_ctx* ctx) { return ctx ? ctx->launches : 0; }


int viml_profile_begin(viml_ctx* ctx) {
  if (!ctx) return VIML_ERR_INVALID;
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  drop_prof_events(ctx);
  ctx->prof = true;
  return VIML_OK;
}

int viml_profile_end(viml_ctx* ctx, double* ms, int64_t* n) {
  if (!ctx) return VIML_ERR_INVALID;
  ctx->prof = false;
  VIML_TRY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int k = 0; k < VIML_NUM_KERNELS; ++k) {
    double tot = 0.0;
    for (auto& pr : ctx->prof_events[k]) {
      float t = 0.f;
      if (cudaEventElapsedTime(&t, pr.first, pr.second) == cudaSuccess) tot += t;
    }
    if (ms) ms[k] = tot;
    if (n) n[k] = (int64_t)ctx->prof_events[k].size();
  }
  drop_prof_events(ctx);
  return VIML_OK;
}

const char* viml_kernel_name(int id) {
  static const char* names[VIML_NUM_KERNELS] = {"prep_windows", "linearize_points", "linearize_lines", "assemble_hb",
                                                "schur_landmarks", "assoc_cam_pose", "assoc_cull", "assoc_scan",
                                                "assoc_fill_list", "assoc_project", "assoc_match", "marginalize_dense",
                                                "microbench", "plan_windows", "assemble_irregular", "gn_step"};
  return (id >= 0 && id < VIML_NUM_KERNELS) ? names[id] : "";
}

// ---- map -------------------------------------------------------------------------------------
int viml_set_map(viml_ctx* ctx, const double* lines, int64_t n) {
  if (!ctx || n < 0 || (n > 0 && !lines)) return VIML_ERR_INVALID;
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  VIML_TRY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  auto drop = [&](auto*& ptr) {
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
  };
  drop(ctx->d_map), drop(ctx->d_map_sorted), drop(ctx->d_map_orig), drop(ctx->d_tile_sphere), drop(ctx->d_group_sphere);
  drop(ctx->d_fov_slots), drop(ctx->d_fov_slot_count);   // the cached FoV lists index the old map
  ctx->fov_words = 0;
  ctx->n_map = 0, ctx->n_tiles = 0;
  ctx->map_set = true;
  if (n == 0) return VIML_OK;
  // AoS rows [sx sy sz ex ey ez] (parameters.cpp:50-59) -> six SoA planes
  std::vector<double> soa((size_t)6 * n);
  for (int64_t j = 0; j < n; ++j)
    for (int c = 0; c < 6; ++c) soa[(size_t)c * n + j] = lines[6 * j + c];
  VIML_TRY_CUDA(ctx, cudaMalloc((void**)&ctx->d_map, soa.size() * sizeof(double)));
  VIML_TRY_CUDA(ctx, cudaMemcpy(ctx->d_map, soa.data(), soa.size() * sizeof(double), cudaMemcpyHostToDevice));
  // Morton order of the segment mid-points (21 bits per axis over the bounding box); one-time ingest cost.
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int64_t j = 0; j < n; ++j)
    for (int c = 0; c < 3; ++c) {
      const double m = 0.5 * (lines[6 * j + c] + lines[6 * j + 3 + c]);
      if (std::isfinite(m)) lo[c] = std::min(lo[c], m), hi[c] = std::max(hi[c], m);
    }
  auto spread = [](uint64_t v) {  // 21 bits -> every third bit
    v &= 0x1fffff;
    v = (v | v << 32) & 0x1f00000000ffffull;
    v = (v | v << 16) & 0x1f0000ff0000ffull;
    v = (v | v << 8) & 0x100f00f00f00f00full;
    v = (v | v << 4) & 0x10c30c30c30c30c3ull;
    v = (v | v << 2) & 0x1249249249249249ull;
    return v;
  };
  // one scale for the three axes: cubic cells, so a flat map (x, y extent >> z extent) is split in x and y first
  double span = 0.0;
  for (int c = 0; c < 3; ++c)
    if (hi[c] > lo[c]) span = std::max(span, hi[c] - lo[c]);
  if (!(span > 0.0)) span = 1.0;
  std::vector<uint64_t> key(n);
  for (int64_t j = 0; j < n; ++j) {
    uint64_t k = 0;
    for (int c = 0; c < 3; ++c) {
      const double m = 0.5 * (lines[6 * j + c] + lines[6 * j + 3 + c]);
      double t = std::isfinite(m) ? (m - lo[c]) / span : 0.0;
      t = std::min(1.0, std::max(0.0, t));
      k |= spread((uint64_t)(t * 2097151.0)) << c;
    }
    key[j] = k;
  }
  std::vector<int32_t> order(n);
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return key[a] < key[b]; });
  std::vector<double> sorted((size_t)6 * n);
  for (int64_t k = 0; k < n; ++k)
    for (int c = 0; c < 6; ++c) sorted[(size_t)c * n + k] = lines[6 * (int64_t)order[k] + c];
  const int64_t nt = (n + kMapTile - 1) / kMapTile;
  std::vector<double> sph((size_t)nt * 4);
  for (int64_t t = 0; t < nt; ++t) {
    const int64_t k0 = t * kMapTile, k1 = std::min<int64_t>(n, k0 + kMapTile);
    double blo[3] = {INFINITY, INFINITY, INFINITY}, bhi[3] = {-INFINITY, -INFINITY, -INFINITY};
    bool finite = true;
    for (int64_t k = k0; k < k1; ++k)
      for (int c = 0; c < 6; ++c) {
        const double v = sorted[(size_t)c * n + k];
        finite &= std::isfinite(v);
        blo[c % 3] = std::min(blo[c % 3], v), bhi[c % 3] = std::max(bhi[c % 3], v);
      }
    double ctr[3], r2 = 0.0;
    for (int c = 0; c < 3; ++c) ctr[c] = 0.5 * (blo[c] + bhi[c]);
    for (int64_t k = k0; k < k1; ++k)
      for (int e = 0; e < 2; ++e) {
        double d2 = 0.0;
        for (int c = 0; c < 3; ++c) {
          const double d = sorted[(size_t)(3 * e + c) * n + k] - ctr[c];
          d2 += d * d;
        }
        r2 = std::max(r2, d2);
      }
    // a tile with a non-finite coordinate is never rejected (radius = +inf): the exact test decides
    sph[4 * t] = ctr[0], sph[4 * t + 1] = ctr[1], sph[4 * t + 2] = ctr[2];
    sph[4 * t + 3] = finite ? std::sqrt(r2) * (1.0 + 1e-12) : INFINITY;
  }
  VIML_TRY_CUDA(ctx, cudaMalloc((void**)&ctx->d_map_sorted, sorted.size() * sizeof(double)));
  VIML_TRY_CUDA(ctx, cudaMemcpy(ctx->d_map_sorted, sorted.data(), sorted.size() * sizeof(double), cudaMemcpyHostToDevice));
  VIML_TRY_CUDA(ctx, cudaMalloc((void**)&ctx->d_map_orig, (size_t)n * sizeof(int32_t)));
  VIML_TRY_CUDA(ctx, cudaMemcpy(ctx->d_map_orig, order.data(), (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice));
  VIML_TRY_CUDA(ctx, cudaMalloc((void**)&ctx->d_tile_sphere, sph.size() * sizeof(double)));
  VIML_TRY_CUDA(ctx, cudaMemcpy(ctx->d_tile_sphere, sph.data(), sph.size() * sizeof(double), cudaMemcpyHostToDevice));
  // second level: one sphere around every 16 consecutive tile spheres (consecutive Morton tiles are neighbours)
  const int64_t ngrp = (nt + 15) / 16;
  std::vector<double> gsp((size_t)std::max<int64_t>(ngrp, 1) * 4, 0.0);
  for (int64_t gq = 0; gq < ngrp; ++gq) {
    const int64_t ta = gq * 16, tb = std::min<int64_t>(nt, ta + 16);
    double c[3] = {0, 0, 0}, r = 0.0;
    bool fin = true;
    for (int64_t t = ta; t < tb; ++t) {
      fin &= std::isfinite(sph[4 * t + 3]) && std::isfinite(sph[4 * t]) && std::isfinite(sph[4 * t + 1]) && std::isfinite(sph[4 * t + 2]);
      for (int k = 0; k < 3; ++k) c[k] += sph[4 * t + k] / (double)(tb - ta);
    }
    for (int64_t t = ta; t < tb && fin; ++t) {
      double d2 = 0.0;
      for (int k = 0; k < 3; ++k) d2 += (sph[4 * t + k] - c[k]) * (sph[4 * t + k] - c[k]);
      r = std::max(r, std::sqrt(d2) * (1.0 + 1e-12) + sph[4 * t + 3]);
    }
    gsp[4 * gq] = fin ? c[0] : 0.0, gsp[4 * gq + 1] = fin ? c[1] : 0.0, gsp[4 * gq + 2] = fin ? c[2] : 0.0;
    gsp[4 * gq + 3] = fin ? r * (1.0 + 1e-12) : INFINITY;   // never rejected when a member is not finite
  }
  VIML_TRY_CUDA(ctx, cudaMalloc((void**)&ctx->d_group_sphere, gsp.size() * sizeof(double)));
  VIML_TRY_CUDA(ctx, cudaMemcpy(ctx->d_group_sphere, gsp.data(), gsp.size() * sizeof(double), cudaMemcpyHostToDevice));
  ctx->n_map = n;
  ctx->n_tiles = nt;
  return VIML_OK;
}

}  // extern "C"

// ---- linearisation -----------------------------------------------------------------------------
int check_window_batch(viml_ctx* ctx, const viml_window_batch* in, bool dev, BatchForm* form) {
  *form = BatchForm{};
  if (!in) return fail(ctx, VIML_ERR_INVALID, "null window batch");
  const int W = in->n_windows, P = in->poses_per_window, F = in->feats_per_window;
  const int64_t NP = in->n_point_factors, NL = in->n_line_factors;
  if (W < 0 || P < 1 || P > 255 || F < 0 || F > 65535 || NP < 0 || NL < 0)
    return fail(ctx, VIML_ERR_INVALID, "window batch sizes out of range");
  if (W == 0) return VIML_OK;
  const bool f64_table = in->feat_obs && in->pf_obs_j, f32_table = in->feat_obs_f32 && in->pf_obs_j_f32;
  form->obs_table = NP > 0 && !in->pf_obs && (f64_table || f32_table);
  form->obs_f32 = form->obs_table && !f64_table;
  form->feat_obs = !form->obs_table ? nullptr : form->obs_f32 ? (const void*)in->feat_obs_f32 : (const void*)in->feat_obs;
  form->pf_obs_j = !form->obs_table ? nullptr : form->obs_f32 ? (const void*)in->pf_obs_j_f32 : (const void*)in->pf_obs_j;
  form->obs_bytes = form->obs_f32 ? 8 : 16;
  form->line_table = NL > 0 && !in->lf_geom && in->lf_map_index && in->lf_seg2d_f32;
  if (!in->poses || !in->ex_pose || (F > 0 && !in->inv_depth) || !in->pf_window_offset ||
      (NP > 0 && (!in->pf_idx || (!in->pf_obs && !form->obs_table))) ||
      (NL > 0 && (!in->lf_window_offset || !in->lf_frame || (!in->lf_geom && !form->line_table))))
    return fail(ctx, VIML_ERR_INVALID, "null input array");
  if (form->line_table && (!ctx->map_set || ctx->n_map <= 0))
    return fail(ctx, VIML_ERR_NOMAP, "line factors given by map index need a map (viml_set_map)");
  if (dev) return VIML_OK;   // device pointers cannot be read here: their offsets and indices are the caller's to keep (viml.h)
  const int32_t* po = in->pf_window_offset;
  bool ok = po[0] == 0 && po[W] == NP;
  for (int w = 0; w < W && ok; ++w) ok = po[w] <= po[w + 1];
  if (NL > 0) {
    const int32_t* lo = in->lf_window_offset;
    ok = ok && lo[0] == 0 && lo[W] == NL;
    for (int w = 0; w < W && ok; ++w) ok = lo[w] <= lo[w + 1];
  }
  if (!ok) return fail(ctx, VIML_ERR_INVALID, "window offsets are not a CSR of the factor arrays (offset[0] == 0, non-decreasing, offset[W] == n_factors)");
  return VIML_OK;
}

int check_batch_indices(viml_ctx* ctx, const viml_window_batch* in, const BatchForm& form, int64_t pa, int64_t pb, int64_t la,
                        int64_t lb) {
  uint32_t bad = 0;
  const uint32_t uP = (uint32_t)in->poses_per_window, uF = (uint32_t)in->feats_per_window;
  for (int64_t k = pa; k < pb; ++k) {
    const uint32_t ix = in->pf_idx[k];
    bad |= (uint32_t)((ix & 0xffu) >= uP) | (uint32_t)(((ix >> 8) & 0xffu) >= uP) | (uint32_t)((ix >> 16) >= uF);
  }
  for (int64_t k = la; k < lb; ++k) bad |= (uint32_t)((uint32_t)in->lf_frame[k] >= uP);
  if (form.line_table)
    for (int64_t k = la; k < lb; ++k) bad |= (uint32_t)((uint64_t)(int64_t)in->lf_map_index[k] >= (uint64_t)ctx->n_map);
  if (bad) return fail(ctx, VIML_ERR_INVALID, "factor index out of range (pose index >= poses_per_window, feature >= feats_per_window, line frame >= poses_per_window or map index outside the map)");
  return VIML_OK;
}

LinearizeArgs linearize_args(const viml_ctx* ctx, const viml_window_batch* in, uint32_t flags) {
  LinearizeArgs a{};
  a.W = in->n_windows, a.P = in->poses_per_window, a.F = in->feats_per_window, a.D = 6 * (a.P + 1);
  a.NP = in->n_point_factors, a.NL = in->n_line_factors;
  a.pf_begin = 0, a.lf_begin = 0, a.NL_stride = a.NL;
  a.sqrt_info = ctx->cfg.sqrt_info, a.cauchy_a = ctx->cfg.cauchy_a;
  a.inv_cauchy_a2 = 1.0 / (ctx->cfg.cauchy_a * ctx->cfg.cauchy_a);
  a.fx = ctx->cfg.fx, a.fy = ctx->cfg.fy, a.cx = ctx->cfg.cx, a.cy = ctx->cfg.cy;
  a.flags = flags;
  return a;
}

void stage_batch(viml_ctx* ctx, Stager& st, const viml_window_batch* in, const BatchForm& form, uint32_t flags, StagedBatch* b) {
  const int W = in->n_windows, P = in->poses_per_window, F = in->feats_per_window;
  const int64_t NP = in->n_point_factors, NL = in->n_line_factors;
  *b = StagedBatch{};
  b->form = form;
  LinearizeArgs& a = b->a = linearize_args(ctx, in, flags);
  st.in(in->poses, (size_t)W * P * 7, &a.poses);
  st.in(in->ex_pose, (size_t)W * 7, &a.ex_pose);
  st.in(in->inv_depth, (size_t)W * F, &a.inv_depth);
  st.in(in->pf_window_offset, (size_t)W + 1, &a.pf_window_offset);
  st.in(in->pf_idx, (size_t)NP, &a.pf_idx, {kAxPf, 1});
  if (form.obs_table) {
    st.in((const char*)form.feat_obs, (size_t)W * F * form.obs_bytes, &b->fobs, {kAxWindow, (size_t)F * form.obs_bytes});
    st.in((const char*)form.pf_obs_j, (size_t)NP * form.obs_bytes, &b->obsj, {kAxPf, form.obs_bytes});
  } else {
    st.in(in->pf_obs, (size_t)NP * 4, &a.pf_obs, {kAxPf, 4});
  }
  st.in(in->pf_pts_i_z, in->pf_pts_i_z ? (size_t)NP : 0, &a.pf_pts_i_z, {kAxPf, 1});
  st.in(in->lf_window_offset, NL > 0 ? (size_t)W + 1 : 0, &a.lf_window_offset);
  st.in(in->lf_frame, (size_t)NL, &a.lf_frame);
  if (form.line_table) {
    st.in(in->lf_map_index, (size_t)NL, &b->lidx, {kAxLf, 1});
    st.in(in->lf_seg2d_f32, (size_t)NL * 4, &b->lseg, {kAxLf, 4});
  } else {
    st.in(in->lf_geom, (size_t)NL * 9, &a.lf_geom, {kAxLf, 1, 9});   // [9][NL]
  }
  st.out((double*)nullptr, (size_t)W * (P * kPoseCache + kExCache), &a.cache);
  if (form.obs_table) st.out((double*)nullptr, (size_t)NP * 4, &b->obs);
  if (form.line_table) st.out((double*)nullptr, (size_t)NL * 9, &b->geom);
}

int expand_tables(viml_ctx* ctx, StagedBatch& b) {
  if (b.form.obs_table) {
    b.a.pf_obs = b.obs;
    const int rc = viml_launch_expand_obs(ctx, b.a, b.fobs, b.obsj, b.form.obs_f32);
    if (rc != VIML_OK) return rc;
  }
  if (b.form.line_table) {
    b.a.lf_geom = b.geom;
    return viml_launch_expand_lines(ctx, b.a, b.lidx, b.lseg);
  }
  return VIML_OK;
}

extern "C" {

int viml_linearize_batch(viml_ctx* ctx, const viml_window_batch* in, const viml_linearize_out* out, uint32_t flags) {
  if (!ctx) return VIML_ERR_INVALID;
  if (!in || !out) return fail(ctx, VIML_ERR_INVALID, "null batch or output struct");
  const bool dev = (flags & VIML_PTRS_DEVICE) != 0;
  BatchForm form;
  int rc = check_window_batch(ctx, in, dev, &form);
  if (rc != VIML_OK) return rc;
  if (!(flags & (VIML_OUT_RESIDUAL_JACOBIAN | VIML_OUT_HB | VIML_OUT_SCHUR)))
    return fail(ctx, VIML_ERR_INVALID, "no output mode requested");
  const int W = in->n_windows, P = in->poses_per_window, F = in->feats_per_window, D = 6 * (P + 1);
  const int64_t NP = in->n_point_factors, NL = in->n_line_factors;
  if (W == 0) return VIML_OK;
  const bool wantA = (flags & VIML_OUT_RESIDUAL_JACOBIAN) != 0;
  const bool wantHB = (flags & VIML_OUT_HB) != 0, wantS = (flags & VIML_OUT_SCHUR) != 0;
  if (wantHB && !(out->H_pp && out->H_lp && out->H_ll && out->b_p && out->b_l))
    return fail(ctx, VIML_ERR_INVALID, "VIML_OUT_HB needs H_pp, H_lp, H_ll, b_p and b_l");
  if (wantS && !(out->S && out->g)) return fail(ctx, VIML_ERR_INVALID, "VIML_OUT_SCHUR needs S and g");
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  Stager st{ctx, dev};
  StagedBatch b;
  stage_batch(ctx, st, in, form, flags, &b);
  viml_linearize_out& o = b.a.out;
  if (wantA) {
    auto a_out = [&](double* host, size_t per, int axis, double** slot) {
      st.out(host, host ? per * (size_t)(axis == kAxPf ? NP : NL) : 0, slot, {axis, per});
    };
    a_out(out->pf_residual, 2, kAxPf, &o.pf_residual);
    a_out(out->pf_jac_pose_i, 14, kAxPf, &o.pf_jac_pose_i);
    a_out(out->pf_jac_pose_j, 14, kAxPf, &o.pf_jac_pose_j);
    a_out(out->pf_jac_ex, 14, kAxPf, &o.pf_jac_ex);
    a_out(out->pf_jac_feat, 2, kAxPf, &o.pf_jac_feat);
    a_out(out->lf_residual, 2, kAxLf, &o.lf_residual);
    a_out(out->lf_jac_pose, 14, kAxLf, &o.lf_jac_pose);
  }
  // the per-window outputs, elements per window: H_pp, H_lp, H_ll, b_p, b_l, S, g
  const size_t n_pp = (size_t)D * D, n_lp = (size_t)F * D, n_S = (flags & VIML_S_PACKED) ? (size_t)D * (D + 1) / 2 : n_pp;
  auto w_out = [&](double* host, size_t per, double** slot) { st.out(host, (size_t)W * per, slot, {kAxWindow, per}); };
  if (wantHB || wantS) {   // with VIML_OUT_SCHUR alone the H blocks are scratch
    w_out(wantHB ? out->H_pp : nullptr, n_pp, &o.H_pp);
    w_out(wantHB ? out->H_lp : nullptr, n_lp, &o.H_lp);
    w_out(wantHB ? out->H_ll : nullptr, F, &o.H_ll);
    w_out(wantHB ? out->b_p : nullptr, D, &o.b_p);
    w_out(wantHB ? out->b_l : nullptr, F, &o.b_l);
  }
  if (wantS) {
    w_out(out->S, n_S, &o.S);
    w_out(out->g, D, &o.g);
  }
  if (dev || (W < 512 && st.one_copy())) {
    // host pointers: check_window_batch has checked the offsets, the packed indices are checked before any kernel reads them
    if (!dev) rc = check_batch_indices(ctx, in, form, 0, NP, 0, NL);
    if (rc == VIML_OK) rc = st.commit();
    if (rc == VIML_OK) rc = expand_tables(ctx, b);
    if (rc == VIML_OK) rc = viml_launch_linearize(ctx, b.a);
    if (rc != VIML_OK) return rc;
    return st.finish();
  }
  // Host pointers, W >= 512 or more than Stager::kOneCopyBytes: chunks of windows.  A chunk's kernels run on a view of the batch
  // (per-window pointers advanced to its first window, per-factor arrays absolute: they are indexed by the global factor id).
  // check_window_batch has checked the offsets; the packed indices are checked chunk by chunk before the chunk's kernels (the host
  // runs ahead of the asynchronous copies and kernels, so the ~1 ms scan of a 2.3 M-factor batch hides behind the transfers).
  auto at = [&](int w) -> Stager::Units { return {w, in->pf_window_offset[w], NL > 0 ? in->lf_window_offset[w] : 0}; };
  auto chunk = [&](const Stager::Units& lo, const Stager::Units& hi) {
    const int w0 = (int)lo[kAxWindow];
    int rc = check_batch_indices(ctx, in, form, lo[kAxPf], hi[kAxPf], lo[kAxLf], hi[kAxLf]);
    if (rc != VIML_OK) return rc;   // bad indices never reach a kernel: this chunk and the following ones are not launched
    StagedBatch v = b;
    LinearizeArgs& va = v.a;
    va.W = (int)hi[kAxWindow] - w0, va.NP = hi[kAxPf] - lo[kAxPf], va.NL = hi[kAxLf] - lo[kAxLf];
    va.pf_begin = lo[kAxPf], va.lf_begin = lo[kAxLf];
    va.poses += (size_t)w0 * P * 7, va.ex_pose += (size_t)w0 * 7, va.inv_depth += (size_t)w0 * F, va.pf_window_offset += w0;
    if (NL > 0) va.lf_window_offset += w0;
    va.cache += (size_t)w0 * (P * kPoseCache + kExCache);
    if (v.fobs) v.fobs += (size_t)w0 * F * form.obs_bytes;
    auto advance = [&](double*& p, size_t per) { if (p) p += (size_t)w0 * per; };
    viml_linearize_out& vo = va.out;
    advance(vo.H_pp, n_pp), advance(vo.H_lp, n_lp), advance(vo.H_ll, F), advance(vo.b_p, D), advance(vo.b_l, F);
    advance(vo.S, n_S), advance(vo.g, D);
    rc = expand_tables(ctx, v);
    return rc != VIML_OK ? rc : viml_launch_linearize(ctx, v.a);
  };
  return st.run_chunked(W, at, [] { return VIML_OK; }, chunk);
}

// ---- dense marginalisation -----------------------------------------------------------------------
int viml_marginalize_batch(viml_ctx* ctx, const viml_marg_batch* in, const viml_marg_out* out, uint32_t flags) {
  if (!ctx) return VIML_ERR_INVALID;
  if (!in || !out) return fail(ctx, VIML_ERR_INVALID, "null marg batch");
  const int K = in->n_problems, pos = in->pos, m = in->m, n = pos - m;
  if (K < 0 || pos < 1 || pos > 256 || m < 0 || n < 1 || !in->A || !in->b)
    return fail(ctx, VIML_ERR_INVALID, "marg batch sizes out of range (pos <= 256, n >= 1)");
  if (K == 0) return VIML_OK;
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t szA = (size_t)K * pos * pos, szb = (size_t)K * pos, szS = (size_t)K * n * n, szs = (size_t)K * n;
  Stager st{ctx, (flags & VIML_PTRS_DEVICE) != 0};
  const double *dA = nullptr, *db = nullptr;
  double *dS = nullptr, *ds = nullptr, *dJ = nullptr, *dr = nullptr;
  st.in(in->A, szA, &dA);
  st.in(in->b, szb, &db);
  // an output the caller did not ask for is null: the kernel skips it
  st.out(out->A_schur, out->A_schur ? szS : 0, &dS);
  st.out(out->b_schur, out->b_schur ? szs : 0, &ds);
  st.out(out->linearized_jacobians, out->linearized_jacobians ? szS : 0, &dJ);
  st.out(out->linearized_residuals, out->linearized_residuals ? szs : 0, &dr);
  int rc = st.commit();
  if (rc == VIML_OK) rc = viml_launch_marginalize(ctx, K, pos, m, in->eps, dA, db, dS, ds, dJ, dr);
  if (rc != VIML_OK) return rc;
  return st.finish();
}

// ---- association -----------------------------------------------------------------------------------
int viml_line_associate(viml_ctx* ctx, const viml_assoc_query* q, const viml_assoc_out* out, uint32_t flags) {
  if (!ctx) return VIML_ERR_INVALID;
  if (!q || !out) return fail(ctx, VIML_ERR_INVALID, "null query or output struct");
  if (!ctx->map_set) return fail(ctx, VIML_ERR_NOMAP, "viml_line_associate before viml_set_map (an empty map is legal, but it must be set)");
  const int Pq = q->n_poses, L = q->lines_per_pose;
  const bool cached = (flags & VIML_FOV_CACHED) != 0;
  if (Pq < 0 || L < 0 || (!cached && !q->cull_poses) || !q->ex_pose || (L > 0 && !q->lines2d))
    return fail(ctx, VIML_ERR_INVALID, "bad association query");
  if (cached) {
    if (Pq > VIML_FOV_SLOTS && !q->fov_slot) return fail(ctx, VIML_ERR_INVALID, "VIML_FOV_CACHED: more poses than window slots and no fov_slot map");
    if (!q->match_poses && !q->cull_poses) return fail(ctx, VIML_ERR_INVALID, "VIML_FOV_CACHED needs match_poses");
    for (int p = 0; p < Pq && q->fov_slot; ++p)
      if (q->fov_slot[p] < 0 || q->fov_slot[p] >= VIML_FOV_SLOTS) return fail(ctx, VIML_ERR_INVALID, "fov_slot out of range");
  }
  if (Pq == 0) return VIML_OK;
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int64_t N = ctx->n_map, words = (N + 31) / 32;
  const bool dev = (flags & VIML_PTRS_DEVICE) != 0;
  AssocArgs a{};
  a.Pq = Pq, a.L = L, a.N = N, a.map = ctx->d_map, a.words = words;
  a.cached = cached;
  // cached lists: the slots' mask rows and counts gathered into [Pq][words] / [Pq] behind the pose order of this query
  uint32_t* cmask = nullptr;
  int32_t* ccount = nullptr;
  if (cached) {
    VIML_TRY_CUDA(ctx, ctx->s_full.reserve(DeviceArena::padded((size_t)Pq * words * 4 + 4) + DeviceArena::padded((size_t)Pq * 4)));
    cmask = ctx->s_full.take<uint32_t>((size_t)Pq * words + 1);
    ccount = ctx->s_full.take<int32_t>((size_t)Pq);
    for (int p = 0; p < Pq; ++p) {
      const int sl = q->fov_slot ? q->fov_slot[p] : p;
      if (ctx->d_fov_slots && ctx->fov_words == words) {
        if (words) VIML_TRY_CUDA(ctx, cudaMemcpyAsync(cmask + (size_t)p * words, ctx->d_fov_slots + (size_t)sl * words, (size_t)words * 4, cudaMemcpyDeviceToDevice, st));
        VIML_TRY_CUDA(ctx, cudaMemcpyAsync(ccount + p, ctx->d_fov_slot_count + sl, 4, cudaMemcpyDeviceToDevice, st));
      } else {   // no slot was ever updated for this map: empty lists
        if (words) VIML_TRY_CUDA(ctx, cudaMemsetAsync(cmask + (size_t)p * words, 0, (size_t)words * 4, st));
        VIML_TRY_CUDA(ctx, cudaMemsetAsync(ccount + p, 0, 4, st));
      }
    }
  }
  if (!ctx->d_assoc_stats) VIML_TRY_CUDA(ctx, cudaMalloc((void**)&ctx->d_assoc_stats, 32));
  VIML_TRY_CUDA(ctx, cudaMemsetAsync(ctx->d_assoc_stats, 0, 32, st));
  a.stats = ctx->d_assoc_stats;
  a.map_sorted = ctx->d_map_sorted, a.map_orig = ctx->d_map_orig, a.tile_sphere = ctx->d_tile_sphere, a.group_sphere = ctx->d_group_sphere, a.n_tiles = ctx->n_tiles;
  a.fov_capacity = out->fov_index ? out->fov_capacity : 0;
  const size_t nq = (size_t)Pq * L, cap = a.fov_capacity;
  // Every output is per pose; the kernels always write match_index, err, projected, fov_count and fov_mask (scratch where the
  // caller did not ask).  Host pointers: entries past fov_count keep the caller's fov_index, and ragged queries past n_lines2d keep
  // the caller's match_index, err and projected.
  Stager s{ctx, dev};
  auto per_pose = [](size_t n) { return Stager::Split{0, n}; };
  s.in(q->cull_poses ? q->cull_poses : q->match_poses, (size_t)Pq * 7, &a.cull_poses);
  s.in(q->match_poses, (size_t)Pq * 7, &a.match_poses);
  s.in(q->ex_pose, (size_t)Pq * 7, &a.ex_pose);
  s.in(q->cull_ex_pose, (size_t)Pq * 7, &a.cull_ex_pose);
  s.in(q->n_lines2d, (size_t)Pq, &a.n_lines2d);
  s.in(q->lines2d, nq * 4, &a.lines2d, per_pose((size_t)L * 4));
  const bool ragged = out->match_index && q->n_lines2d;   // in-out
  s.out(out->match_index, nq, &a.match_index, per_pose(L), ragged);
  s.out(out->err, nq * 3, &a.err, per_pose((size_t)L * 3), ragged);
  s.out(out->projected, nq * 4, &a.projected, per_pose((size_t)L * 4), ragged);
  s.out(out->fov_count, (size_t)Pq, &a.fov_count, per_pose(1));
  s.inout(out->fov_index, (size_t)Pq * cap, &a.fov_index, per_pose(cap));
  s.out(out->fov_mask, (size_t)Pq * words, &a.fov_mask, per_pose((size_t)words));
  // once the slots are placed: the poses the query did not give separately, and the cached lists
  auto prepare = [&]() -> int {
    if (!q->match_poses) a.match_poses = a.cull_poses;
    if (!q->cull_ex_pose) a.cull_ex_pose = a.ex_pose;
    if (cached) {
      if (words) VIML_TRY_CUDA(ctx, cudaMemcpyAsync(a.fov_mask, cmask, (size_t)Pq * words * 4, cudaMemcpyDeviceToDevice, st));
      VIML_TRY_CUDA(ctx, cudaMemcpyAsync(a.fov_count, ccount, (size_t)Pq * 4, cudaMemcpyDeviceToDevice, st));
    }
    return VIML_OK;
  };
  if (dev) {
    int rc = s.commit();
    if (rc == VIML_OK) rc = prepare();
    return rc != VIML_OK ? rc : viml_launch_associate(ctx, a);
  }
  // Host pointers: poses are independent, so the query runs in chunks of poses.  Phase 1 (camera poses, FoV cull, list offsets)
  // runs once for all poses as soon as the small arrays are up -- it does not need the detected lines, whose upload it overlaps --
  // and holds the call's only synchronisation; phase 2 (list fill, projection, match) then runs chunk by chunk.
  AssocPlan plan;
  auto phase1 = [&] {
    const int rc = prepare();
    return rc != VIML_OK ? rc : viml_assoc_phase1(ctx, a, &plan);
  };
  auto chunk = [&](const Stager::Units& lo, const Stager::Units& hi) {
    const int p0 = (int)lo[0], p1 = (int)hi[0];
    AssocArgs v = a;   // view of poses [p0, p1)
    v.Pq = p1 - p0;
    v.cull_poses = a.cull_poses + (size_t)p0 * 7, v.match_poses = a.match_poses + (size_t)p0 * 7;
    v.ex_pose = a.ex_pose + (size_t)p0 * 7, v.cull_ex_pose = a.cull_ex_pose + (size_t)p0 * 7;
    v.lines2d = a.lines2d + (size_t)p0 * L * 4, v.n_lines2d = a.n_lines2d ? a.n_lines2d + p0 : nullptr;
    v.match_index = a.match_index + (size_t)p0 * L, v.err = a.err + (size_t)p0 * L * 3, v.projected = a.projected + (size_t)p0 * L * 4;
    v.fov_count = a.fov_count + p0, v.fov_index = a.fov_index ? a.fov_index + (size_t)p0 * cap : nullptr;
    v.fov_mask = a.fov_mask + (size_t)p0 * words;
    return viml_assoc_phase2(ctx, v, plan, p0, p1);
  };
  return s.run_chunked(Pq, [](int p) { return Stager::Units{p, 0, 0}; }, phase1, chunk);
}

// ---- FoV cache ---------------------------------------------------------------------------------------
static int fov_cache_ready(viml_ctx* ctx) {
  const int64_t words = (ctx->n_map + 31) / 32;
  if (ctx->d_fov_slots && ctx->fov_words == words) return VIML_OK;
  if (ctx->d_fov_slots) cudaFree(ctx->d_fov_slots);
  ctx->d_fov_slots = nullptr;
  VIML_TRY_CUDA(ctx, cudaMalloc((void**)&ctx->d_fov_slots, (size_t)VIML_FOV_SLOTS * std::max<int64_t>(words, 1) * 4));
  if (!ctx->d_fov_slot_count) VIML_TRY_CUDA(ctx, cudaMalloc((void**)&ctx->d_fov_slot_count, VIML_FOV_SLOTS * 4));
  VIML_TRY_CUDA(ctx, cudaMemsetAsync(ctx->d_fov_slots, 0, (size_t)VIML_FOV_SLOTS * std::max<int64_t>(words, 1) * 4, ctx->stream));
  VIML_TRY_CUDA(ctx, cudaMemsetAsync(ctx->d_fov_slot_count, 0, VIML_FOV_SLOTS * 4, ctx->stream));
  ctx->fov_words = words;
  return VIML_OK;
}

int viml_fov_update(viml_ctx* ctx, int32_t slot, const double* pose, const double* ex_pose, int32_t* count) {
  if (!ctx) return VIML_ERR_INVALID;
  if (slot < 0 || slot >= VIML_FOV_SLOTS || !pose || !ex_pose) return fail(ctx, VIML_ERR_INVALID, "viml_fov_update: bad slot or null pose");
  if (!ctx->map_set) return fail(ctx, VIML_ERR_NOMAP, "viml_fov_update before viml_set_map");
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  int rc = fov_cache_ready(ctx);
  if (rc != VIML_OK) return rc;
  cudaStream_t st = ctx->stream;
  VIML_TRY_CUDA(ctx, ctx->in_arena.reserve(2 * DeviceArena::padded(56)));
  double* dp = ctx->in_arena.take<double>(7);
  double* de = ctx->in_arena.take<double>(7);
  VIML_TRY_CUDA(ctx, cudaMemcpyAsync(dp, pose, 56, cudaMemcpyHostToDevice, st));
  VIML_TRY_CUDA(ctx, cudaMemcpyAsync(de, ex_pose, 56, cudaMemcpyHostToDevice, st));
  AssocArgs a{};
  a.Pq = 1, a.L = 0, a.N = ctx->n_map, a.map = ctx->d_map, a.words = ctx->fov_words;
  a.map_sorted = ctx->d_map_sorted, a.map_orig = ctx->d_map_orig, a.tile_sphere = ctx->d_tile_sphere, a.group_sphere = ctx->d_group_sphere, a.n_tiles = ctx->n_tiles;
  if (!ctx->d_assoc_stats) VIML_TRY_CUDA(ctx, cudaMalloc((void**)&ctx->d_assoc_stats, 32));
  a.stats = ctx->d_assoc_stats;
  a.cull_poses = a.match_poses = dp, a.ex_pose = a.cull_ex_pose = de;
  a.fov_mask = ctx->d_fov_slots + (size_t)slot * ctx->fov_words;
  a.fov_count = ctx->d_fov_slot_count + slot;
  rc = viml_launch_associate(ctx, a);
  if (rc != VIML_OK) return rc;
  if (count) {
    VIML_TRY_CUDA(ctx, cudaMemcpyAsync(count, a.fov_count, 4, cudaMemcpyDeviceToHost, st));
    VIML_TRY_CUDA(ctx, cudaStreamSynchronize(st));
  }
  return VIML_OK;
}

int viml_fov_slide(viml_ctx* ctx, int32_t marginalize_old) {
  if (!ctx) return VIML_ERR_INVALID;
  if (!ctx->map_set) return fail(ctx, VIML_ERR_NOMAP, "viml_fov_slide before viml_set_map");
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  const int rc = fov_cache_ready(ctx);
  if (rc != VIML_OK) return rc;
  cudaStream_t st = ctx->stream;
  const size_t wb = (size_t)ctx->fov_words * 4;
  const int last = VIML_FOV_SLOTS - 1;
  auto row = [&](int s) { return ctx->d_fov_slots + (size_t)s * ctx->fov_words; };
  if (marginalize_old) {
    // estimator.cpp:2148 swaps slot i with i+1 for i = 0..WINDOW_SIZE-1 and :2160 then copies slot WINDOW_SIZE-1 into the
    // newest one: net effect slot i <- old slot i+1 (i < WINDOW_SIZE), newest slot unchanged.  Stream-ordered copies,
    // ascending, each reading a row that has not been overwritten yet.
    for (int i = 0; i < last; ++i) {
      if (wb) VIML_TRY_CUDA(ctx, cudaMemcpyAsync(row(i), row(i + 1), wb, cudaMemcpyDeviceToDevice, st));
      VIML_TRY_CUDA(ctx, cudaMemcpyAsync(ctx->d_fov_slot_count + i, ctx->d_fov_slot_count + i + 1, 4, cudaMemcpyDeviceToDevice, st));
    }
  } else {
    if (wb) VIML_TRY_CUDA(ctx, cudaMemcpyAsync(row(last - 1), row(last), wb, cudaMemcpyDeviceToDevice, st));   // :2218
    VIML_TRY_CUDA(ctx, cudaMemcpyAsync(ctx->d_fov_slot_count + last - 1, ctx->d_fov_slot_count + last, 4, cudaMemcpyDeviceToDevice, st));
  }
  return VIML_OK;
}

int viml_track_gate(viml_ctx* ctx, int32_t n_tracks, const int32_t* track_offset, const int32_t* line_index, uint8_t* credible_line,
                    uint8_t* credible_matching, uint32_t flags) {
  if (!ctx) return VIML_ERR_INVALID;
  if (n_tracks < 0 || (n_tracks > 0 && (!track_offset || !credible_matching))) return fail(ctx, VIML_ERR_INVALID, "viml_track_gate: bad arguments");
  if (!ctx->map_set) return fail(ctx, VIML_ERR_NOMAP, "viml_track_gate before viml_set_map");
  if (n_tracks == 0) return VIML_OK;
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  Stager st{ctx, (flags & VIML_PTRS_DEVICE) != 0};
  int64_t nobs = 0;   // device pointers pass through: the observation count is not needed
  if (!st.dev) {
    nobs = track_offset[n_tracks];
    if (nobs < 0 || (nobs > 0 && (!line_index || !credible_line))) return fail(ctx, VIML_ERR_INVALID, "viml_track_gate: null observation arrays");
  }
  const int32_t *doff = nullptr, *didx = nullptr;
  uint8_t *dcl = nullptr, *dcm = nullptr;
  st.in(track_offset, (size_t)n_tracks + 1, &doff);
  st.in(line_index, (size_t)nobs, &didx);
  st.out(credible_line, (size_t)nobs, &dcl);
  st.out(credible_matching, (size_t)n_tracks, &dcm);
  int rc = st.commit();
  if (rc == VIML_OK) rc = viml_launch_track_gate(ctx, n_tracks, doff, didx, dcl, dcm);
  if (rc != VIML_OK) return rc;
  return st.finish();
}

int viml_selftest_division(viml_ctx* ctx, const double* a, const double* b, int64_t n, int64_t* mismatches) {
  if (!ctx) return VIML_ERR_INVALID;
  if (n < 0 || (n > 0 && (!a || !b)) || !mismatches) return fail(ctx, VIML_ERR_INVALID, "bad division self-test arguments");
  VIML_TRY_CUDA(ctx, cudaSetDevice(ctx->device));
  Stager st{ctx, false};
  const double *da = nullptr, *db = nullptr;
  unsigned long long h = 0, *dm = nullptr;
  st.in(a, (size_t)n, &da);
  st.in(b, (size_t)n, &db);
  st.out(&h, 1, &dm);
  int rc = st.commit();
  if (rc != VIML_OK) return rc;
  VIML_TRY_CUDA(ctx, cudaMemsetAsync(dm, 0, 8, ctx->stream));
  rc = viml_launch_divcheck(ctx, da, db, n, dm);
  if (rc == VIML_OK) rc = st.finish();
  if (rc != VIML_OK) return rc;
  *mismatches = (int64_t)h;
  return VIML_OK;
}

int viml_assoc_stats(viml_ctx* ctx, int64_t* gate_tests, int64_t* gated, int64_t* overlap_scored,
                     int64_t* distance_scored) {
  if (!ctx) return VIML_ERR_INVALID;
  unsigned long long h[4] = {0, 0, 0, 0};
  if (ctx->d_assoc_stats) {
    VIML_TRY_CUDA(ctx, cudaMemcpyAsync(h, ctx->d_assoc_stats, 32, cudaMemcpyDeviceToHost, ctx->stream));
    VIML_TRY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  if (gate_tests) *gate_tests = (int64_t)h[0];
  if (gated) *gated = (int64_t)h[1];
  if (overlap_scored) *overlap_scored = (int64_t)h[2];
  if (distance_scored) *distance_scored = (int64_t)h[3];
  return VIML_OK;
}

// ---- multi-GPU: partial H/b all-reduce for the single huge window ----------------------------------
int viml_allreduce_hb(viml_ctx* ctx, void* nccl_comm, double* buf, int64_t count) {
  if (!ctx) return VIML_ERR_INVALID;
  if (!nccl_comm || !buf || count < 0) return fail(ctx, VIML_ERR_INVALID, "bad all-reduce arguments");
  if (!ctx->nccl_lib) {
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nme : names) {
      ctx->nccl_lib = dlopen(nme, RTLD_NOW | RTLD_GLOBAL);
      if (ctx->nccl_lib) break;
    }
    if (!ctx->nccl_lib) return fail(ctx, VIML_ERR_UNSUPPORTED, "libnccl.so.2 not loadable");
  }
  // ncclResult_t ncclAllReduce(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t)
  using allreduce_t = int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t);
  auto fn = (allreduce_t)dlsym(ctx->nccl_lib, "ncclAllReduce");
  if (!fn) return fail(ctx, VIML_ERR_UNSUPPORTED, "ncclAllReduce not found");
  const int ncclFloat64 = 8, ncclSum = 0;
  const int rc = fn(buf, buf, (size_t)count, ncclFloat64, ncclSum, nccl_comm, ctx->stream);
  if (rc != 0) return fail(ctx, VIML_ERR_CUDA, "ncclAllReduce failed");
  return VIML_OK;
}

}  // extern "C"
