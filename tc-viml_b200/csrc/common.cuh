// common.cuh — context, error handling and launch declarations shared by the CUDA translation units.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "viml.h"

#define VIML_TRY_CUDA(ctx, expr)                                                              \
  do {                                                                                        \
    cudaError_t e__ = (expr);                                                                 \
    if (e__ != cudaSuccess) {                                                                 \
      (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(e__);                      \
      return VIML_ERR_CUDA;                                                                   \
    }                                                                                         \
  } while (0)

// Growable device buffer; contents are not preserved across grow().
struct DeviceArena {
  char* base = nullptr;
  size_t cap = 0, used = 0;
  cudaError_t reserve(size_t bytes) {
    used = 0;
    if (bytes <= cap) return cudaSuccess;
    if (base) cudaFree(base);
    base = nullptr;
    cap = 0;
    const size_t want = bytes + bytes / 8 + (1u << 20);
    cudaError_t e = cudaMalloc((void**)&base, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  template <class T>
  T* take(size_t count) {
    const size_t bytes = (count * sizeof(T) + 255) & ~size_t(255);
    T* p = (T*)(base + used);
    used += bytes;
    return p;
  }
  static size_t padded(size_t bytes) { return (bytes + 255) & ~size_t(255); }
  void release() {
    if (base) cudaFree(base);
    base = nullptr;
    cap = used = 0;
  }
};

struct viml_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;
  cudaStream_t copy_stream2 = nullptr;
  cudaEvent_t ev_a = nullptr, ev_b = nullptr;
  cudaStream_t aux_stream = nullptr;            // plan_kernel runs here, beside prep_windows_kernel
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  viml_config cfg{};
  std::string err;
  int64_t launches = 0;
  // association decision threshold: angle > angle_th  <=>  |dot| < cos_th  (SURVEY.md §7)
  double cos_th = 0.0;
  int nan_angle_passes = 0;  // !(3.1415926 > angle_th)
  // prior map, six SoA planes of n_map doubles
  double* d_map = nullptr;
  int64_t n_map = 0;
  bool map_set = false;   // viml_set_map was called (an empty map is legal)
  // spatially sorted copy for the hierarchical cull: Morton order of segment mid-points, tiles of kMapTile
  // lines with a bounding sphere each (centre xyz + radius), and the original index of every sorted line
  double* d_map_sorted = nullptr;   // [6][n_map]
  int32_t* d_map_orig = nullptr;    // [n_map]
  double* d_tile_sphere = nullptr;  // [n_tiles][4]
  double* d_group_sphere = nullptr; // [ceil(n_tiles / 16)][4]: one sphere around 16 consecutive tile spheres
  int64_t n_tiles = 0;
  // FoV cache: one mask row per window slot (viml_fov_update / viml_fov_slide), sized for the current map
  uint32_t* d_fov_slots = nullptr;     // [VIML_FOV_SLOTS][fov_words]
  int32_t* d_fov_slot_count = nullptr; // [VIML_FOV_SLOTS]
  int64_t fov_words = 0;
  unsigned long long* d_assoc_stats = nullptr;  // {gate tests, gated pairs, overlap-scored, distance-scored} of the last association call
  DeviceArena in_arena, out_arena, scratch, scratch2, scratch3, s_full;
  // pinned blocks of Stager's one-copy path (one H2D, one D2H per call)
  char *h_stage_in = nullptr, *h_stage_out = nullptr;
  size_t h_stage_in_cap = 0, h_stage_out_cap = 0;
  void* nccl_lib = nullptr;
  // profiling (viml_profile_begin/end): event pairs per kernel id
  bool brute_cull = false;     // VIML_BRUTE_CULL=1: the literal all-pairs FoV sweep (roofline accounting, cross-check)
  bool force_generic = false;  // tests: route everything through the generic atomic kernels
  bool prof = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events[VIML_NUM_KERNELS];
};

inline int fail(viml_ctx* ctx, int code, const char* msg) {
  if (ctx) ctx->err = msg;
  return code;
}

// Host <-> device staging of an entry point: where a host call's arrays live on the device, and how they get there and back.
// in() slots are placed in ctx->in_arena and copied up, out() slots in ctx->out_arena and copied back.  An out() with a null host
// pointer is device scratch; an inout() is an out() whose device slot first receives the caller's buffer (entries the kernels do
// not write keep the caller's content).  With host pointers a slot whose count is 0 is null.  With VIML_PTRS_DEVICE the caller's
// pointers pass through unchanged and only scratch is placed.
// Host pointers are copied in one of three modes:
//  - one copy: commit() / finish() of a call whose staged bytes total at most kOneCopyBytes.  Every cudaMemcpyAsync costs 5-10 us
//    of driver and DMA set-up whatever its size (more from pageable memory), and a step stages some 30 arrays, so the inputs are
//    gathered into the pinned ctx->h_stage_in laid out like in_arena (one H2D), and the device range that holds every output comes
//    back into ctx->h_stage_out (one D2H) and is handed out from there.
//  - per array: commit() / finish() of a larger call, one copy per array on the context stream.
//  - chunked: run_chunked(), a pipeline of chunks over three streams for the large calls whose work splits into independent units
//    (windows, poses).  A slot given a Split goes up / comes back chunk by chunk; the other slots are whole.
// commit() and finish() synchronise nothing but the context stream at the end of finish(); run_chunked() returns synchronised.
struct Stager {
  static constexpr size_t kOneCopyBytes = size_t(4) << 20;
  // Positions on the unit axes of a chunked run (up to three: the linearisation's windows, point factors and line factors).
  using Units = std::array<int64_t, 3>;
  // How a slot splits into chunks: `per` elements for each unit of axis `axis`, in each of `planes` planes of an SoA array
  // ([planes][n] with n = count / planes: a chunk is one 2D copy of its range of every plane).  axis < 0: whole.
  struct Split { int axis = -1; size_t per = 0; int planes = 1; };
  viml_ctx* ctx;
  bool dev;
  struct In { const void* host; size_t bytes; const void** slot; Split sp; char* d; };   // sp.per in bytes; d: the placed slot
  struct Out { void* host; size_t bytes; void** slot; Split sp; bool inout; char* d; };
  std::vector<In> ins;
  std::vector<Out> outs;
  Stager(viml_ctx* c, bool d) : ctx(c), dev(d) {   // room for the arrays of any call: no reallocation while staging
    ins.reserve(32);
    outs.reserve(32);
  }
  template <class T>
  void in(const T* host, size_t count, const T** slot, Split sp = {}) {
    *slot = dev ? host : nullptr;
    sp.per *= sizeof(T);
    if (!dev && host && count) ins.push_back({host, count * sizeof(T), reinterpret_cast<const void**>(slot), sp, nullptr});
  }
  template <class T>
  void inout(T* host, size_t count, T** slot, Split sp = {}) { out(host, count, slot, sp, true); }
  template <class T>
  void out(T* host, size_t count, T** slot, Split sp = {}, bool inout = false) {
    *slot = dev ? host : nullptr;
    sp.per *= sizeof(T);
    if ((!dev || !host) && count)
      outs.push_back({dev ? nullptr : host, count * sizeof(T), reinterpret_cast<void**>(slot), sp, inout && !dev && host, nullptr});
  }
  size_t in_bytes() const {
    size_t b = 0;
    for (auto& e : ins) b += DeviceArena::padded(e.bytes);
    return b;
  }
  size_t out_bytes() const {
    size_t b = 0;
    for (auto& e : outs) b += DeviceArena::padded(e.bytes);
    return b;
  }
  bool one_copy() const { return !dev && in_bytes() + out_bytes() <= kOneCopyBytes; }
  // a pinned block of the one-copy path: grown, never shrunk
  static cudaError_t grow(char** buf, size_t* cap, size_t need) {
    if (need <= *cap) return cudaSuccess;
    if (*buf) cudaFreeHost(*buf);
    *buf = nullptr, *cap = 0;
    const cudaError_t e = cudaHostAlloc((void**)buf, need + need / 2 + 4096, cudaHostAllocDefault);
    if (e == cudaSuccess) *cap = need + need / 2 + 4096;
    return e;
  }
  // places every slot in the arenas
  int place() {
    VIML_TRY_CUDA(ctx, ctx->in_arena.reserve(in_bytes()));
    VIML_TRY_CUDA(ctx, ctx->out_arena.reserve(out_bytes()));
    for (auto& e : ins) *e.slot = e.d = ctx->in_arena.take<char>(e.bytes);
    for (auto& e : outs) *e.slot = e.d = ctx->out_arena.take<char>(e.bytes);
    return VIML_OK;
  }
  // Copies the units [lo, hi) of a slot of `bytes` (all of it when it is whole): one copy, or one 2D copy of its planes.
  static cudaError_t copy(void* dst, const void* src, size_t bytes, const Split& s, const Units& lo, const Units& hi,
                          cudaMemcpyKind kind, cudaStream_t st) {
    const size_t off = s.axis < 0 ? 0 : s.per * (size_t)lo[s.axis];
    const size_t n = s.axis < 0 ? bytes / s.planes : s.per * (size_t)(hi[s.axis] - lo[s.axis]);
    if (!n) return cudaSuccess;
    if (s.planes == 1) return cudaMemcpyAsync((char*)dst + off, (const char*)src + off, n, kind, st);
    const size_t pitch = bytes / s.planes;
    return cudaMemcpy2DAsync((char*)dst + off, pitch, (const char*)src + off, pitch, n, s.planes, kind, st);
  }
  // One copy or per array: places the slots and queues the uploads on the context stream, in-out slots after the inputs.
  int commit() {
    const size_t ib = in_bytes(), ob = out_bytes();
    const bool one = one_copy();
    const int rc = place();
    if (rc != VIML_OK) return rc;
    if (one) {
      VIML_TRY_CUDA(ctx, grow(&ctx->h_stage_in, &ctx->h_stage_in_cap, ib));
      VIML_TRY_CUDA(ctx, grow(&ctx->h_stage_out, &ctx->h_stage_out_cap, ob));
      for (auto& e : ins) memcpy(ctx->h_stage_in + (e.d - ctx->in_arena.base), e.host, e.bytes);
      if (ib) VIML_TRY_CUDA(ctx, cudaMemcpyAsync(ctx->in_arena.base, ctx->h_stage_in, ib, cudaMemcpyHostToDevice, ctx->stream));
    } else {
      for (auto& e : ins) VIML_TRY_CUDA(ctx, cudaMemcpyAsync(e.d, e.host, e.bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    for (auto& e : outs)
      if (e.inout) VIML_TRY_CUDA(ctx, cudaMemcpyAsync(e.d, e.host, e.bytes, cudaMemcpyHostToDevice, ctx->stream));
    return VIML_OK;
  }
  int finish() {
    if (dev) return VIML_OK;
    if (one_copy()) {
      char *lo = nullptr, *hi = nullptr;
      for (auto& e : outs)
        if (e.host) {
          char* b = (char*)*e.slot;
          lo = lo ? std::min(lo, b) : b, hi = hi ? std::max(hi, b + e.bytes) : b + e.bytes;
        }
      if (lo) VIML_TRY_CUDA(ctx, cudaMemcpyAsync(ctx->h_stage_out, lo, (size_t)(hi - lo), cudaMemcpyDeviceToHost, ctx->stream));
      VIML_TRY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
      for (auto& e : outs)
        if (e.host) memcpy(e.host, ctx->h_stage_out + ((char*)*e.slot - lo), e.bytes);
    } else {
      for (auto& e : outs)
        if (e.host) VIML_TRY_CUDA(ctx, cudaMemcpyAsync(e.host, *e.slot, e.bytes, cudaMemcpyDeviceToHost, ctx->stream));
      VIML_TRY_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    VIML_TRY_CUDA(ctx, cudaGetLastError());
    return VIML_OK;
  }
  // Chunked (host pointers only): H2D(c + 1) | kernels(c) | D2H(c - 1) on copy_stream, the context stream and copy_stream2.  PCIe
  // is full duplex, so with pinned host memory a call approaches max(H2D, D2H) time.  `n` units make C chunks, chunk c the units
  // [n c / C, n (c + 1) / C); at(u) gives the position of unit boundary u on every axis.
  //  1. copy_stream waits for the context stream: work queued there may still read the arenas.
  //  2. Whole inputs and in-out uploads go up; the context stream waits for them.
  //  3. Every chunk's inputs go up, each chunk followed by its event.
  //  4. step() runs: work over all units, which may synchronise the host (the uploads of step 3 overlap it).
  //  5. Per chunk: the context stream waits for its event, chunk(lo, hi) builds its view and launches, and copy_stream2 brings back
  //     the chunk's range of every host-backed output (whole outputs after the last chunk).
  // The three streams are synchronised and the events destroyed on every exit; the first error is returned.  An error of chunk()
  // launches no later chunk; the outputs of the chunks before it may already be written.
  template <class At, class Step, class Chunk>
  int run_chunked(int n, At at, Step step, Chunk chunk) {
    // measured on the 4096-window linearisation with the float32 table (75 MB up, 88 MB down): 2, 3, 4, 5, 6, 8, 12, 16 chunks ->
    // 2.96, 2.81, 2.67, 2.75, 2.70, 2.79, 2.93, 2.96 ms; on the cfg-3 association sweep: 2, 4, 6, 8, 12, 16 -> 2.32, 2.19, 2.30,
    // 2.36, 2.79, 2.76 ms
    const int C = n >= 512 ? 4 : 1;
    std::vector<Units> b(C + 1);
    for (int c = 0; c <= C; ++c) b[c] = at((int)((int64_t)n * c / C));
    std::vector<cudaEvent_t> ev;   // the C upload events, then one per launched chunk
    auto event = [&](cudaStream_t s) {
      cudaEvent_t e;
      cudaError_t r = cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
      if (r == cudaSuccess) ev.push_back(e), r = cudaEventRecord(e, s);
      return r;
    };
    auto run = [&]() -> int {
      cudaStream_t s_k = ctx->stream, s_in = ctx->copy_stream, s_out = ctx->copy_stream2;
      int rc = place();
      if (rc != VIML_OK) return rc;
      VIML_TRY_CUDA(ctx, cudaEventRecord(ctx->ev_a, s_k));
      VIML_TRY_CUDA(ctx, cudaStreamWaitEvent(s_in, ctx->ev_a, 0));
      for (auto& e : ins)
        if (e.sp.axis < 0) VIML_TRY_CUDA(ctx, copy(e.d, e.host, e.bytes, e.sp, b[0], b[C], cudaMemcpyHostToDevice, s_in));
      for (auto& e : outs)
        if (e.inout) VIML_TRY_CUDA(ctx, cudaMemcpyAsync(e.d, e.host, e.bytes, cudaMemcpyHostToDevice, s_in));
      VIML_TRY_CUDA(ctx, cudaEventRecord(ctx->ev_b, s_in));
      VIML_TRY_CUDA(ctx, cudaStreamWaitEvent(s_k, ctx->ev_b, 0));
      for (int c = 0; c < C; ++c) {
        for (auto& e : ins)
          if (e.sp.axis >= 0) VIML_TRY_CUDA(ctx, copy(e.d, e.host, e.bytes, e.sp, b[c], b[c + 1], cudaMemcpyHostToDevice, s_in));
        VIML_TRY_CUDA(ctx, event(s_in));
      }
      rc = step();
      for (int c = 0; c < C && rc == VIML_OK; ++c) {
        VIML_TRY_CUDA(ctx, cudaStreamWaitEvent(s_k, ev[c], 0));
        rc = chunk(b[c], b[c + 1]);
        if (rc != VIML_OK) break;
        VIML_TRY_CUDA(ctx, event(s_k));
        VIML_TRY_CUDA(ctx, cudaStreamWaitEvent(s_out, ev.back(), 0));
        for (auto& e : outs)
          if (e.host && (e.sp.axis >= 0 || c == C - 1))
            VIML_TRY_CUDA(ctx, copy(e.host, e.d, e.bytes, e.sp, b[c], b[c + 1], cudaMemcpyDeviceToHost, s_out));
      }
      return rc;
    };
    const int rc = run();
    const cudaError_t e1 = cudaStreamSynchronize(ctx->copy_stream2), e2 = cudaStreamSynchronize(ctx->stream),
                      e3 = cudaStreamSynchronize(ctx->copy_stream);
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
    if (rc != VIML_OK) return rc;
    VIML_TRY_CUDA(ctx, e1);
    VIML_TRY_CUDA(ctx, e2);
    VIML_TRY_CUDA(ctx, e3);
    VIML_TRY_CUDA(ctx, cudaGetLastError());
    return VIML_OK;
  }
};

enum KernelId {
  K_PREP = 0, K_POINTS, K_LINES, K_ASSEMBLE, K_SCHUR, K_CAMPOSE, K_CULL, K_SCAN, K_FILL, K_PROJECT, K_MATCH,
  K_MARG, K_MICRO, K_PLAN, K_IRREGULAR, K_GN, K_COUNT
};
static_assert(K_COUNT <= VIML_NUM_KERNELS, "raise VIML_NUM_KERNELS");

// Brackets one kernel launch with profiling events when enabled and counts it.
struct LaunchScope {
  viml_ctx* ctx;
  cudaEvent_t stop = nullptr;
  cudaStream_t on;
  LaunchScope(viml_ctx* c, int id, cudaStream_t st = nullptr) : ctx(c), on(st ? st : c->stream) {
    ctx->launches++;
    if (ctx->prof) {
      cudaEvent_t a, b;
      cudaEventCreate(&a);
      cudaEventCreate(&b);
      cudaEventRecord(a, on);
      ctx->prof_events[id].emplace_back(a, b);
      stop = b;
    }
  }
  ~LaunchScope() {
    if (stop) cudaEventRecord(stop, on);
  }
};

// Per-pose cache written by prep_windows_kernel and read by the factor kernels (42 doubles):
//   P[3]      position
//   R[9]      toRotationMatrix(q)               un-normalised (projection_factor.cpp:56-57)
//   Rinv[9]   toRotationMatrix(q.inverse())      == the map v -> Qj.inverse()*v (projection_factor.cpp:38)
//   M[9]      ric^T * R^T                        (projection_factor.cpp:81, :93)
//   Rl[9]     Ricn^T * Rn^T, Rn = toRotationMatrix(normalized(q))   (line_projection_factor.cpp:31-39)
//   tl[3]     -Rl*P - Ricn^T*Tic                 (line_projection_factor.cpp:40)
// Per-window extrinsic cache (24 doubles): tic[3], ric[9], ricinv[9], rtt[3] = ric^T*tic
constexpr int kMapTile = 64;   // lines per tile of the Morton-sorted map copy (measured on the cfg-3 sweep: 256 -> 0.234 ms, 64 -> 0.207, 32 -> 0.307)
constexpr int kPoseCache = 42;
constexpr int kExCache = 24;
constexpr int PC_P = 0, PC_R = 3, PC_RINV = 12, PC_M = 21, PC_RL = 30, PC_TL = 39;
constexpr int EC_TIC = 0, EC_RIC = 3, EC_RICINV = 12, EC_RTT = 21;

struct LinearizeArgs {  // device pointers only
  int W, P, F, D;
  int64_t NP, NL;          // factors covered by this launch
  int64_t pf_begin, lf_begin;  // first factor covered (chunked launches view a window range of one batch)
  int64_t NL_stride;       // plane stride of lf_geom (total line factors of the batch)
  const double* poses;
  const double* ex_pose;
  const double* inv_depth;
  const int32_t* pf_window_offset;
  const uint32_t* pf_idx;
  const double* pf_obs;
  const double* pf_pts_i_z;
  const int32_t* lf_window_offset;
  const int32_t* lf_frame;
  const double* lf_geom;
  double* cache;  // [W][P*kPoseCache + kExCache]
  viml_linearize_out out;
  double sqrt_info, cauchy_a, inv_cauchy_a2, fx, fy, cx, cy;
  uint32_t flags;
};

// How a viml_window_batch carries its observations and line factors (viml.h), decided once by check_window_batch.
struct BatchForm {
  bool obs_table, obs_f32;            // observations as the per-feature table (only when NP > 0), in float32
  bool line_table;                    // line factors as (map index, 2D segment)
  const void *feat_obs, *pf_obs_j;    // the arrays of the chosen table form
  size_t obs_bytes;                   // bytes of one {x, y} of the table: 16 or 8
};
// viml_api.cu: what every entry point that takes a viml_window_batch checks.  Sizes, null arrays, the form, VIML_ERR_NOMAP for a line
// table without a map; with host pointers (dev == false) also that both window offsets are CSRs of the factor arrays.
int check_window_batch(viml_ctx* ctx, const viml_window_batch* in, bool dev, BatchForm* form);
// Host pointers: the pose, feature, frame and map indices of point factors [pa, pb) and line factors [la, lb) (VIML_ERR_INVALID).
int check_batch_indices(viml_ctx* ctx, const viml_window_batch* in, const BatchForm& form, int64_t pa, int64_t pb, int64_t la,
                        int64_t lb);
// The LinearizeArgs of the whole batch with the context's camera and loss constants; the pointers are left null.
LinearizeArgs linearize_args(const viml_ctx* ctx, const viml_window_batch* in, uint32_t flags);
// A viml_window_batch staged for the device: its arrays in `a` (outputs left to the caller), and the observation / line tables
// with the scratch they are expanded into.
struct StagedBatch {
  LinearizeArgs a;
  BatchForm form;
  const char *fobs, *obsj;
  const float* lseg;
  const int32_t* lidx;
  double *obs, *geom;   // their expansions
};
// The unit axes of a window batch in a chunked run: windows, point factors, line factors.
constexpr int kAxWindow = 0, kAxPf = 1, kAxLf = 2;
// Stages the batch (checked by check_window_batch, which gave `form`) into `st`: the inputs of linearize_args(ctx, in, flags), the
// table sources, the expansion targets and the pose cache.  The per-factor inputs and the per-window observation table are split
// by factor / window; the rest is whole.  The Stager keeps the addresses of *b's fields; after st.commit() the caller calls
// expand_tables().
void stage_batch(viml_ctx* ctx, Stager& st, const viml_window_batch* in, const BatchForm& form, uint32_t flags, StagedBatch* b);
// The observation and line tables of the batch, expanded into the per-factor arrays every kernel reads.
int expand_tables(viml_ctx* ctx, StagedBatch& b);

// Largest reduced system a Gauss-Newton step takes, Dx = D + extra_dim (viml.h): its tiled Cholesky keeps the lower triangle in
// shared memory.
constexpr int kMaxDx = 232;
// Dynamic shared memory (bytes) of the tiled Cholesky solves of a Dx x Dx system (gn_kernels.cuh): the lower triangle of 8 x 8
// tiles and the right-hand side; the fused kernel, which builds the system in place, also keeps g, the undamped diagonal and a
// stage of kFusedStage doubles for a dense-factor Jacobian and residual (a 76 x 75 prior: 6460).
constexpr int kFusedStage = 6656;
constexpr size_t kSolveSmemMax = 224 * 1024;   // of the 227 KB a block may opt in to, beside the kernels' static shared memory
constexpr size_t gn_solve_smem(int Dx) {
  const size_t NB = (Dx + 7) / 8;
  return (NB * (NB + 1) / 2 * 64 + NB * 8) * sizeof(double);
}
constexpr size_t gn_fused_solve_smem(int Dx) {
  return gn_solve_smem(Dx) + (2 * (size_t)((Dx + 7) / 8) * 8 + kFusedStage) * sizeof(double);
}
// A Gauss-Newton step whose caller does not ask for Sx / gx builds and solves the system in the fused kernel where it fits,
// Dx <= 200; above, reduced_kernel writes Sx / gx and the unfused kernel solves it.
constexpr bool gn_fused_takes(int Dx) { return gn_fused_solve_smem(Dx) <= kSolveSmemMax; }
static_assert(gn_solve_smem(kMaxDx) <= kSolveSmemMax, "the unfused tiled Cholesky must take the largest reduced system");
static_assert(gn_fused_takes(200) && !gn_fused_takes(201), "the fused kernel takes Dx <= 200 (DESIGN.md 4.4)");

struct DenseArgs {  // device pointers only; viml_dense_factors
  int X;          // extra tangent columns behind the D pose / extrinsic columns
  int64_t ND;
  const int32_t* window_offset;
  const int64_t* row_offset;
  const int64_t* col_offset;
  const int64_t* jac_offset;
  const int32_t* col_index;
  const double* residual;
  const double* jacobian;
};

struct InertialArgs {  // device pointers only; viml_inertial_factors plus the state they are evaluated at
  int W, P, D, X;
  int64_t NI;
  double G[3];
  const int32_t* imu_window_offset;
  const int32_t* imu_pose;
  const int32_t* imu_sb;
  const double* imu_preint;
  const double* imu_jacobian;
  const double* imu_sqrt_info;
  int n_max, max_blocks;
  const int32_t* prior_n;
  const double* prior_jacobian;
  const double* prior_residual;
  const int32_t* prior_n_blocks;
  const int32_t* prior_block;
  const double* prior_x0;
  const double* poses;    // [W][P][7]
  const double* ex_pose;  // [W][7]
  const double* extra;    // [W][X] (may be null when X == 0)
};

// The dense-factor CSR of the evaluated IMU / prior factors (per window: the prior, then the IMU factors).  Sized on the host from
// NI, W and n_max alone: factors <= W + NI, rows <= W n_max + 15 NI, columns <= W n_max + 30 NI, Jacobian <= W n_max^2 + 450 NI.
struct InertialCsr {
  int32_t* window_offset;  // [W+1]
  int64_t *row_offset, *col_offset, *jac_offset;   // [W+NI+1]
  int32_t* col_index;
  double* residual;
  double* jacobian;        // null: residuals only
};

// inertial_kernels.cu.  offsets = true builds window_offset / *_offset / col_index of `csr` (the structure does not depend on the
// state); the residuals (and the Jacobian when csr.jacobian is set) are written for the state of `v`.  `out` (nullable fields) takes
// the Ceres layouts.
int viml_launch_inertial(viml_ctx* ctx, const InertialArgs& v, const viml_inertial_out& out, const InertialCsr& csr, bool offsets);

// linearize_kernels.cu
int viml_launch_linearize(viml_ctx* ctx, const LinearizeArgs& a);
int viml_launch_prep(viml_ctx* ctx, const LinearizeArgs& a);   // pose cache of the state in `a` only
// observation table -> per-factor pairs for the windows / factor range of `a` (a.pf_obs is the destination, absolute factor ids)
int viml_launch_expand_obs(viml_ctx* ctx, const LinearizeArgs& a, const void* feat_obs, const void* pf_obs_j, bool f32);
// line table -> the nine lf_geom planes for the line-factor range of `a` (a.lf_geom is the destination, absolute factor ids)
int viml_launch_expand_lines(viml_ctx* ctx, const LinearizeArgs& a, const int32_t* lf_map_index, const float* lf_seg2d);
int viml_launch_reduced(viml_ctx* ctx, int W, int D, const DenseArgs& dn, const double* S, const double* g, double* Sx, double* gx);
// lambda_w (nullable): a damping per window instead of `lambda`; running (nullable): only windows with running[w] != 0 are solved,
// updated and costed (the others are left untouched).  viml_launch_gn_reduced_solve builds and solves the system in one kernel
// (Dx = D + dn.X with gn_fused_takes(Dx)); viml_launch_gn_solve solves the Sx / gx of viml_launch_reduced.
int viml_launch_gn_reduced_solve(viml_ctx* ctx, int W, int D, const DenseArgs& dn, const double* S, const double* g, double lambda,
                                 double* dx, int32_t* solved, double* cost, const double* lambda_w = nullptr,
                                 const int32_t* running = nullptr);
int viml_launch_gn_solve(viml_ctx* ctx, int W, int Dx, double lambda, const double* Sx, const double* gx, double* dx, int32_t* solved,
                         double* cost, const double* lambda_w = nullptr, const int32_t* running = nullptr);
int viml_launch_gn_update(viml_ctx* ctx, const LinearizeArgs& a, int X, const double* extra_in, const double* dx, const int32_t* solved,
                          double* o_poses, double* o_ex, double* o_dep, double* o_extra, const int32_t* running = nullptr);
int viml_launch_cost(viml_ctx* ctx, const LinearizeArgs& a, const DenseArgs& dn, const double* dx, const int32_t* solved, int slot,
                     double* cost, const int32_t* running = nullptr);

// viml_solve_vi: the trust-region state of one window between rounds (written by policy_kernel only).
struct SolveState {
  double radius, decrease_factor;
  double f0, f;                 // f(x0), f at the current state x
  int32_t consecutive_invalid, iterations, accepted, status;
};
struct SolveArgs {  // device pointers only
  viml_solve_options opt;
  int P, F, X, Dx;
  SolveState* state;            // [W]
  int32_t* running;             // [W] read by the gated kernels of the next round
  double* lambda_w;             // [W] 1 / radius for the next round
  double *x_poses, *x_ex, *x_dep, *x_extra;              // the current state x
  const double *p_poses, *p_ex, *p_dep, *p_extra;        // x+ of this round
  const double* dx;             // [W][Dx] this round's reduced step
  const double* cost;           // [W][3]  this round's f(x), f(x+), model decrease
  const int32_t* solved;        // [W]
  viml_solve_out out;           // device pointers (radius, trace nullable)
};
// One CTA per window: applies the policy of viml.h to this round's step (round 0 also starts the state from the options).
int viml_launch_solve_policy(viml_ctx* ctx, int W, const SolveArgs& s, int round);
// schur_kernels.cu
int viml_launch_schur(viml_ctx* ctx, int W, int F, int D, const double* H_pp, const double* H_lp, const double* H_ll,
                      const double* b_p, const double* b_l, double* S, double* g, double eps);
double viml_dmma_peak_tflops(viml_ctx* ctx);
// marg_kernels.cu
int viml_launch_marginalize(viml_ctx* ctx, int K, int pos, int m, double eps, const double* A, const double* b,
                            double* A_schur, double* b_schur, double* lin_jac, double* lin_res);

struct AssocArgs {  // device pointers only
  int Pq, L;
  int64_t N;
  const double* map;  // [6][N] original order
  const double* map_sorted;  // [6][N] Morton order
  const int32_t* map_orig;   // [N]
  const double* tile_sphere; // [n_tiles][4]
  const double* group_sphere;// [ceil(n_tiles / 16)][4]
  int64_t n_tiles;
  const double* cull_poses;
  const double* match_poses;  // may alias cull_poses
  const double* ex_pose;
  const double* cull_ex_pose;  // may alias ex_pose
  const double* lines2d;
  const int32_t* n_lines2d;  // nullable
  int32_t* match_index;
  float* err;
  double* projected;
  int32_t* fov_count;   // always valid (scratch if the caller did not ask)
  int32_t* fov_index;   // nullable
  int32_t fov_capacity;
  uint32_t* fov_mask;   // always valid
  int64_t words;        // ceil(N/32)
  unsigned long long* stats;  // {gate tests, gated, overlap-scored, distance-scored}
  bool cached;                // VIML_FOV_CACHED: fov_mask / fov_count are given (cached lists), no cull
};
// associate_kernels.cu (compiled with -fmad=false)
int viml_launch_associate(viml_ctx* ctx, const AssocArgs& a);
// The same in two phases, so that a host can pipeline pose chunks without a synchronisation per chunk: phase 1 (camera poses, FoV
// cull, list offsets for ALL poses of `a`; one device->host read of the offsets), phase 2 (list fill, projection, match) for the
// poses [p0, p1) of a view `v` of `a` whose per-pose pointers are advanced to pose p0.
struct AssocPlan {
  void *cull = nullptr, *match = nullptr;   // camera poses [Pq]
  int64_t* off = nullptr;                   // device list offsets [Pq + 1]
  std::vector<int64_t> h_off;               // the same on the host
  int32_t* list = nullptr;
  void *seg = nullptr, *abc = nullptr, *aux = nullptr, *dir = nullptr, *len = nullptr, *rec = nullptr, *flen = nullptr;
  int Pq = 0;
};
int viml_assoc_phase1(viml_ctx* ctx, const AssocArgs& a, AssocPlan* plan);
int viml_assoc_phase2(viml_ctx* ctx, const AssocArgs& v, const AssocPlan& plan, int p0, int p1);
// triangulate_kernels.cu
int viml_launch_triangulate(viml_ctx* ctx, int P, int64_t NF, const double* poses, const double* ex, const int32_t* fwin,
                            const int32_t* start, const int64_t* off, const double* pts, double init_depth, double* depth);
int viml_launch_track_gate(viml_ctx* ctx, int n_tracks, const int32_t* track_offset, const int32_t* line_index, uint8_t* credible_line,
                           uint8_t* credible_matching);
int viml_launch_divcheck(viml_ctx* ctx, const double* a, const double* b, int64_t n, unsigned long long* mismatches);
