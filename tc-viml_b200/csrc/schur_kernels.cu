// schur_kernels.cu — landmark Schur complement with FP64 tensor-core tiles (DMMA, mma.sync m8n8k4.f64).
//
//   S = H_pp - sum_l W_l^T W_l / L_l ,   g = b_p - sum_l W_l^T b_l / L_l ,   W_l = H_lp[l][:],  L_l = H_ll[l]
//   landmarks with L_l <= eps are dropped (MarginalizationInfo::eps, marginalization_factor.h:70; the reference
//   inverts Amm through an eigen pseudo-inverse, marginalization_factor.cpp:267-282, which for the diagonal
//   landmark block is exactly this).
//
// It is a SYRK: D x D output, contraction over the F landmarks — the one GEMM-shaped piece of the hot path
// (2 D^2 F flop over D F 8 bytes, ~18 flop/B at D = 72), so it goes to the FP64 tensor pipe.  tcgen05 has no
// FP64 kind; on sm_100a the FP64 MMA is still mma.sync (DMMA in SASS).
// Two kernels: schur_tma_kernel (D <= 72, the sliding window: TMA + mbarrier producer/consumer pipeline, warps own output tiles)
// and schur_dmma_kernel (D > 72: one CTA per (72 x 72 output tile, window), 8 warps share the 81 8x8 sub-tiles — 45 on the
// diagonal, where only the upper triangle is computed and mirrored; W staged through shared memory in chunks of 32 landmarks with
// a row stride of 76 doubles, conflict-free fragment loads; with the band plan of extent_kernel / order_kernel a tile only visits
// the landmarks that touch it).
#include "common.cuh"

namespace {

constexpr int TS = 72;        // CTA tile edge (9 sub-tiles of 8)
constexpr int KC = 32;        // landmarks per staged chunk
constexpr int LDW = 76;       // padded row stride in doubles
constexpr int SWARPS = 8;

__device__ __forceinline__ void dmma(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(SWARPS * 32) schur_dmma_kernel(int F, int D, const double* __restrict__ H_pp,
                                                                 const double* __restrict__ H_lp,
                                                                 const double* __restrict__ H_ll,
                                                                 const double* __restrict__ b_p,
                                                                 const double* __restrict__ b_l, double* __restrict__ S,
                                                                 double* __restrict__ g, double eps, int ntile,
                                                                 const int* __restrict__ order, const int* __restrict__ tstart,
                                                                 const int* __restrict__ span) {
  __shared__ double sR[KC * LDW];   // W[l][row-tile columns]
  __shared__ double sC[KC * LDW];   // W[l][col-tile columns]
  __shared__ double sInv[KC], sB[KC];
  // upper-triangular tile index -> (ty, tx), ty <= tx
  int t = blockIdx.x, ty = 0;
  while (t >= ntile - ty) t -= ntile - ty, ++ty;
  const int tx = ty + t;
  const bool diag = tx == ty;
  const int w = blockIdx.y;
  const int r0 = ty * TS, c0 = tx * TS;
  const int nr = min(TS, D - r0), nc = min(TS, D - c0);
  const double* __restrict__ Hl = H_lp + (size_t)w * F * D;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int kq = lane & 3, mq = lane >> 2;
  // this warp's sub-tiles: the valid 8x8 sub-tiles form an nbr x nbc rectangle (its upper triangle on a diagonal tile), dealt
  // round-robin to the warps in row-major order; the i-th one of this warp is found arithmetically so that the per-warp list
  // stays in registers (indexing it in a runtime-filled array put it in local memory: 44 LDL in round 1)
  constexpr int MAXT = 11;
  const int nbr = (nr + 7) >> 3, nbc = (nc + 7) >> 3;
  const int nsub = diag ? nbr * (nbr + 1) / 2 : nbr * nbc;
  int nt = 0;
  int str[MAXT], stc[MAXT];
#pragma unroll
  for (int i = 0; i < MAXT; ++i) {
    const int k = warp + i * SWARPS;
    int a = 0, b = 0;
    if (k < nsub) {
      nt = i + 1;
      if (diag) {
        int t2 = k;
        while (t2 >= nbr - a) t2 -= nbr - a, ++a;
        b = a + t2;
      } else {
        a = k / nbc, b = k - a * nbc;
      }
    }
    str[i] = a, stc[i] = b;
  }
  double acc[MAXT][2];
#pragma unroll
  for (int i = 0; i < MAXT; ++i) acc[i][0] = acc[i][1] = 0.0;
  double gacc = 0.0;  // threads 0..71 of a diagonal tile own g[r0 + tid]
  // Landmarks that can contribute to this tile.  With the band plan (order != nullptr: landmarks sorted by the first pose
  // tile they touch, `span` = the widest tile extent of a landmark) a landmark touches row tile ty and column tile tx only if
  // its first tile lies in [tx - span, ty]; the extrinsic columns (last tile) are touched by every landmark, so for tx = last
  // the condition is on the rows alone.  Rows outside the range are structural zeros
  // in these columns: skipping them changes nothing but the work (a 201-pose window: ~10x fewer tile-landmark products).
  int lb = 0, le = F;
  const int* __restrict__ ord = nullptr;
  if (order) {
    ord = order + (size_t)w * F;
    const int* ts = tstart + (size_t)w * (ntile + 2);
    const int sp = span[w], last = ntile - 1;
    // (the (extrinsic, extrinsic) block and g_ex need every landmark: ex_block_kernel writes them after this kernel)
    const int lo_t = max(0, (tx == last ? ty : tx) - sp), hi_t = ty;
    lb = lo_t <= hi_t ? ts[lo_t] : 0;
    le = lo_t <= hi_t ? ts[hi_t + 1] : 0;
  }
  for (int l0 = lb; l0 < le; l0 += KC) {
    const int nl = min(KC, le - l0);
    __syncthreads();
    for (int e = tid; e < KC * TS; e += SWARPS * 32) {
      const int l = e / TS, c = e % TS;
      const size_t row = l < nl ? (size_t)(ord ? ord[l0 + l] : l0 + l) : 0;
      sR[l * LDW + c] = (l < nl && c < nr) ? Hl[row * D + r0 + c] : 0.0;
      if (!diag) sC[l * LDW + c] = (l < nl && c < nc) ? Hl[row * D + c0 + c] : 0.0;
    }
    if (tid < KC) {
      const size_t row = tid < nl ? (size_t)(ord ? ord[l0 + tid] : l0 + tid) : 0;
      const double L = tid < nl ? H_ll[(size_t)w * F + row] : 0.0;
      sInv[tid] = (L > eps) ? 1.0 / L : 0.0;
      sB[tid] = tid < nl ? b_l[(size_t)w * F + row] : 0.0;
    }
    __syncthreads();
    const double* cs = diag ? sR : sC;
#pragma unroll 2
    for (int kk = 0; kk < KC; kk += 4) {
      const double inv = sInv[kk + kq];
#pragma unroll
      for (int i = 0; i < MAXT; ++i)
        if (i < nt) {
          const double a = sR[(kk + kq) * LDW + 8 * str[i] + mq] * inv;
          const double b = cs[(kk + kq) * LDW + 8 * stc[i] + mq];
          dmma(acc[i][0], acc[i][1], a, b);
        }
    }
    if (diag && tid < nr) {
      double s = 0.0;
      for (int l = 0; l < KC; ++l) s = fma(sR[l * LDW + tid] * sInv[l], sB[l], s);
      gacc += s;
    }
  }
  const double* __restrict__ Hp = H_pp + (size_t)w * D * D;
  double* __restrict__ So = S + (size_t)w * D * D;
#pragma unroll
  for (int i = 0; i < MAXT; ++i)
    if (i < nt) {
      const int r = r0 + 8 * str[i] + mq;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int c = c0 + 8 * stc[i] + 2 * kq + h;
        if (r < D && c < D) {
          const double v = Hp[(size_t)r * D + c] - acc[i][h];
          So[(size_t)r * D + c] = v;
          // mirror: lower triangle of a diagonal tile's off-diagonal sub-tiles, and the transposed tile
          if (!diag || str[i] != stc[i]) So[(size_t)c * D + r] = Hp[(size_t)c * D + r] - acc[i][h];
        }
      }
    }
  if (diag && tid < nr) g[(size_t)w * D + r0 + tid] = b_p[(size_t)w * D + r0 + tid] - gacc;
}

// ---- band plan for long windows (D > 2 tiles) ----------------------------------------------------------------------
// extent_kernel: warp per landmark row, first and last 72-column pose tile with a non-zero entry (the extrinsic's six
// columns, which every landmark touches, are left out).  order_kernel: landmarks ordered by first tile (stable: warp k
// compacts the landmarks of key k in index order, so the summation order is fixed), tile start offsets, widest extent.
__global__ void __launch_bounds__(256) extent_kernel(int F, int D, const double* __restrict__ H_lp, int* __restrict__ tmin,
                                                     int* __restrict__ tmax, int ntile) {
  const int w = blockIdx.y, lane = threadIdx.x & 31, l = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (l >= F) return;
  const double* __restrict__ row = H_lp + ((size_t)w * F + l) * D;
  int lo = ntile, hi = -1;
  for (int c = lane; c < D - 6; c += 32)
    if (row[c] != 0.0) lo = min(lo, c / TS), hi = max(hi, c / TS);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o)), hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  if (lane == 0) tmin[(size_t)w * F + l] = lo, tmax[(size_t)w * F + l] = hi;
}

__global__ void __launch_bounds__(1024) order_kernel(int F, int ntile, const int* __restrict__ tmin, const int* __restrict__ tmax,
                                                     int* __restrict__ order, int* __restrict__ tstart, int* __restrict__ span) {
  __shared__ int cnt[34], base[35], s_span;
  const int w = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int* __restrict__ tm = tmin + (size_t)w * F;
  const int* __restrict__ tM = tmax + (size_t)w * F;
  if (tid < 34) cnt[tid] = 0;
  if (tid == 0) s_span = 0;
  __syncthreads();
  int sp = 0;
  for (int l = tid; l < F; l += blockDim.x) {
    atomicAdd(&cnt[tm[l]], 1);
    if (tM[l] >= 0) sp = max(sp, tM[l] - tm[l]);
  }
  atomicMax(&s_span, sp);
  __syncthreads();
  if (tid == 0) {
    int run = 0;
    for (int k = 0; k <= ntile; ++k) base[k] = run, run += cnt[k];
    base[ntile + 1] = run;
    for (int k = 0; k <= ntile + 1; ++k) tstart[(size_t)w * (ntile + 2) + k] = base[k];
    span[w] = s_span;
  }
  __syncthreads();
  if (warp <= ntile) {   // keys 0..ntile (ntile = landmarks without any pose entry), one warp per key
    int pos = base[warp];
    for (int l0 = 0; l0 < F; l0 += 32) {
      const int l = l0 + lane;
      const bool mine = l < F && tm[l] == warp;
      const unsigned m = __ballot_sync(0xffffffffu, mine);
      if (mine) order[(size_t)w * F + pos + __popc(m & ((1u << lane) - 1u))] = l;
      pos += __popc(m);
    }
  }
}

// The one block every landmark contributes to: S[ex, ex] = H_pp[ex, ex] - sum_l w_l w_l^T / L_l, g_ex = b_ex - sum_l w_l b_l / L_l
// with w_l the six extrinsic entries of landmark row l.  Runs after the band-limited tile kernel and overwrites its partial
// values for these 42 entries.
__global__ void __launch_bounds__(256) ex_block_kernel(int F, int D, const double* __restrict__ H_pp, const double* __restrict__ H_lp,
                                                       const double* __restrict__ H_ll, const double* __restrict__ b_p,
                                                       const double* __restrict__ b_l, double* __restrict__ S, double* __restrict__ g,
                                                       double eps) {
  __shared__ double red[8][42];
  const int w = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, e0 = D - 6;
  double acc[42];
#pragma unroll
  for (int k = 0; k < 42; ++k) acc[k] = 0.0;
  for (int l = tid; l < F; l += 256) {
    const double L = H_ll[(size_t)w * F + l];
    if (!(L > eps)) continue;
    const double inv = 1.0 / L, bl = b_l[(size_t)w * F + l];
    const double* __restrict__ row = H_lp + ((size_t)w * F + l) * D + e0;
    double v[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) v[k] = row[k];
#pragma unroll
    for (int r = 0; r < 6; ++r) {
#pragma unroll
      for (int c = 0; c < 6; ++c) acc[r * 6 + c] = fma(v[r] * inv, v[c], acc[r * 6 + c]);
      acc[36 + r] = fma(v[r] * inv, bl, acc[36 + r]);
    }
  }
#pragma unroll
  for (int k = 0; k < 42; ++k) {
    double t = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) red[warp][k] = t;
  }
  __syncthreads();
  if (tid < 42) {
    double t = 0.0;
    for (int q = 0; q < 8; ++q) t += red[q][tid];
    if (tid < 36) {
      const int r = e0 + tid / 6, c = e0 + tid % 6;
      S[(size_t)w * D * D + (size_t)r * D + c] = H_pp[(size_t)w * D * D + (size_t)r * D + c] - t;
    } else {
      g[(size_t)w * D + e0 + tid - 36] = b_p[(size_t)w * D + e0 + tid - 36] - t;
    }
  }
}

// ---- DMMA peak (for the roofline denominator of this kernel) ----
__global__ void __launch_bounds__(256) dmma_peak_kernel(double* out, double a, double b, int iters) {
  double c[8][2];
#pragma unroll
  for (int i = 0; i < 8; ++i) c[i][0] = threadIdx.x, c[i][1] = i;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 8; ++i) dmma(c[i][0], c[i][1], a, b);
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += c[i][0] + c[i][1];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}


// ---- sliding-window Schur with a TMA pipeline (D <= 72) ---------------------------------------------------------------------
// schur_tma_kernel: persistent CTAs of 9 consumer warps + 1 producer warp.  The producer streams the windows' landmark rows
// through a ring of shared-memory stages with cp.async.bulk (TMA bulk copy, one 8*D-byte row per copy into a stride of 76
// doubles: conflict-free fragment loads) completing on mbarriers; 1/L and b come from a small pre-pass (schur_inv_kernel,
// rows padded to whole stages).  The consumers OWN output sub-tiles, so the contraction over the landmarks needs no cross-warp
// reduction and no CTA-wide barrier: S is a symmetric 9 x 9 grid of 8x8 tiles, and on the torus every unordered pair of tile
// indices is (w, (w + d) mod 9) for exactly one w in 0..8 and d in 0..4 — warp w computes those five tiles (one A fragment, five
// B fragments, five DMMA per step of four landmarks; every warp runs the same code) and writes each with its mirror.  g[8w..8w+7]
// rides along on the A fragment: one FMA per step and lane, summed over the four k-lanes at the end of the window.  Without
// landmarks (F = 0) there are no chunks: the producer issues nothing and the consumers write S = H_pp, g = b_p.
constexpr int kTmaStageL = 32;                         // landmarks per stage
constexpr int kTmaStageD = kTmaStageL * LDW + 2 * kTmaStageL;   // doubles per stage: rows + 1/L + b
constexpr int kTmaStages = 4;
constexpr int kTmaWarps = 9;                           // consumer warps
constexpr int kTmaThreads = (kTmaWarps + 1) * 32;

__global__ void __launch_bounds__(256) schur_inv_kernel(int W, int F, int Fp, const double* __restrict__ H_ll, const double* __restrict__ b_l,
                                                        double eps, double* __restrict__ invp, double* __restrict__ bp) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= (int64_t)W * Fp) return;
  const int w = (int)(e / Fp), l = (int)(e % Fp);
  double inv = 0.0, b = 0.0;
  if (l < F) {
    const double L = H_ll[(size_t)w * F + l];
    inv = (L > eps) ? 1.0 / L : 0.0;
    b = b_l[(size_t)w * F + l];
  }
  invp[e] = inv, bp[e] = b;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred P1;\n\tWAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\tbra WAIT_LOOP;\n\tDONE:\n\t}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
               "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__global__ void __launch_bounds__(kTmaThreads, 2) schur_tma_kernel(int W, int F, int Fp, int D, const double* __restrict__ H_pp,
                                                                   const double* __restrict__ H_lp, const double* __restrict__ invp,
                                                                   const double* __restrict__ blp, const double* __restrict__ b_p,
                                                                   double* __restrict__ S, double* __restrict__ g) {
  extern __shared__ __align__(128) double tsm[];
  double* stages = tsm;                                             // [kTmaStages][kTmaStageD]
  uint64_t* full = reinterpret_cast<uint64_t*>(stages + (size_t)kTmaStages * kTmaStageD);
  uint64_t* empty = full + kTmaStages;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // columns D..75 of a stage row are never written by the copies (a row copy is D doubles) and rows beyond a window's last
  // landmark keep what the previous user of the stage left: everything starts as zero
  for (int e = tid; e < kTmaStages * kTmaStageD; e += kTmaThreads) tsm[e] = 0.0;
  if (tid == 0) {
    for (int s2 = 0; s2 < kTmaStages; ++s2) mbar_init(&full[s2], 32), mbar_init(&empty[s2], kTmaWarps * 32);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the zero fill (generic proxy) before the bulk copies (async proxy)
  __syncthreads();
  const int nchunk = (F + kTmaStageL - 1) / kTmaStageL;
  uint32_t it = 0;
  if (warp == kTmaWarps) {   // producer
    const uint32_t row_bytes = (uint32_t)D * 8u;
    for (int w = blockIdx.x; w < W; w += gridDim.x) {
      const double* __restrict__ Hl = H_lp + (size_t)w * F * D;
      for (int ch = 0; ch < nchunk; ++ch, ++it) {
        const int stg = it % kTmaStages;
        double* sw = stages + (size_t)stg * kTmaStageD;
        const int l0 = ch * kTmaStageL, nl = min(kTmaStageL, F - l0);
        mbar_wait(&empty[stg], ((it / kTmaStages) & 1) ^ 1);
        // every producer lane arrives with the byte count of its own copies, then issues them (the stage's full barrier counts
        // 32 arrivals): the canonical arrive.expect_tx + copy pair per issuing thread
        const int my_rows = lane < nl ? (nl - lane + 31) / 32 : 0;
        mbar_expect_tx(&full[stg], (uint32_t)my_rows * row_bytes + (lane == 0 ? 2u * kTmaStageL * 8u : 0u));
        for (int r = lane; r < nl; r += 32) bulk_g2s(sw + r * LDW, Hl + (size_t)(l0 + r) * D, row_bytes, &full[stg]);
        if (lane == 0) {
          bulk_g2s(sw + kTmaStageL * LDW, invp + (size_t)w * Fp + l0, kTmaStageL * 8u, &full[stg]);
          bulk_g2s(sw + kTmaStageL * LDW + kTmaStageL, blp + (size_t)w * Fp + l0, kTmaStageL * 8u, &full[stg]);
        }
      }
    }
    return;
  }
  // consumer warp `warp`: tiles (warp, ct[d]), d = 0..4
  const int kq = lane & 3, mq = lane >> 2;
  int coff[5];
#pragma unroll
  for (int d = 0; d < 5; ++d) coff[d] = 8 * ((warp + d) % 9);
  const int r = 8 * warp + mq;
  for (int w = blockIdx.x; w < W; w += gridDim.x) {
    // H_pp entries of this warp's tiles and of their mirrors are read in the epilogue; they are pulled into L2 now, while the
    // landmarks stream (holding them in registers across the loop costs the second CTA per SM)
    const double* __restrict__ Hp = H_pp + (size_t)w * D * D;
#pragma unroll
    for (int d = 0; d < 5; ++d) {
      const int c = coff[d] + 2 * kq;
      if (r < D && c < D) {
        asm volatile("prefetch.global.L2 [%0];" ::"l"(Hp + (size_t)r * D + c));
        if (d > 0) {
          asm volatile("prefetch.global.L2 [%0];" ::"l"(Hp + (size_t)c * D + r));
          asm volatile("prefetch.global.L2 [%0];" ::"l"(Hp + (size_t)(c + 1) * D + r));
        }
      }
    }
    double acc[5][2];
#pragma unroll
    for (int i = 0; i < 5; ++i) acc[i][0] = acc[i][1] = 0.0;
    double gacc = 0.0;
    for (int ch = 0; ch < nchunk; ++ch, ++it) {
      const int stg = it % kTmaStages;
      const double* sw = stages + (size_t)stg * kTmaStageD;
      const double* sinv = sw + kTmaStageL * LDW;
      const double* sb = sinv + kTmaStageL;
      const int nl = min(kTmaStageL, F - ch * kTmaStageL);
      mbar_wait(&full[stg], (it / kTmaStages) & 1);
      const int nk = (nl + 3) >> 2;   // rows nl.. of a last stage hold finite leftovers and meet 1/L = 0 from the padded pre-pass
#pragma unroll 2
      for (int k4 = 0; k4 < nk; ++k4) {
        const int l = 4 * k4 + kq;
        const double* row = sw + l * LDW + mq;
        const double fb0 = row[coff[0]];
        const double fa = fb0 * sinv[l];
        gacc = fma(fa, sb[l], gacc);
        dmma(acc[0][0], acc[0][1], fa, fb0);
#pragma unroll
        for (int d = 1; d < 5; ++d) dmma(acc[d][0], acc[d][1], fa, row[coff[d]]);
      }
      mbar_arrive(&empty[stg]);   // every consumer thread releases the stage itself (288 arrivals per phase)
    }
    // S = H_pp - acc on the owned tiles and their mirrors; g = b_p - sum over the k-lanes
    double* __restrict__ So = S + (size_t)w * D * D;
    double2 hu[5];
    double hm[5][2];
#pragma unroll
    for (int d = 0; d < 5; ++d) {
      const int c = coff[d] + 2 * kq;
      const bool in = r < D && c < D;   // D is even: c + 1 < D too
      hu[d] = in ? *reinterpret_cast<const double2*>(Hp + (size_t)r * D + c) : make_double2(0.0, 0.0);
      hm[d][0] = (in && d > 0) ? Hp[(size_t)c * D + r] : 0.0;
      hm[d][1] = (in && d > 0) ? Hp[(size_t)(c + 1) * D + r] : 0.0;
    }
    const double bpr = (kq == 0 && r < D) ? b_p[(size_t)w * D + r] : 0.0;
#pragma unroll
    for (int d = 0; d < 5; ++d) {
      const int c = coff[d] + 2 * kq;
      if (r < D && c < D) {
        *reinterpret_cast<double2*>(So + (size_t)r * D + c) = make_double2(hu[d].x - acc[d][0], hu[d].y - acc[d][1]);
        if (d > 0) {
          So[(size_t)c * D + r] = hm[d][0] - acc[d][0];
          So[(size_t)(c + 1) * D + r] = hm[d][1] - acc[d][1];
        }
      }
    }
    gacc += __shfl_xor_sync(0xffffffffu, gacc, 1);
    gacc += __shfl_xor_sync(0xffffffffu, gacc, 2);
    if (kq == 0 && r < D) g[(size_t)w * D + r] = bpr - gacc;
  }
}

}  // namespace

int viml_launch_schur(viml_ctx* ctx, int W, int F, int D, const double* H_pp, const double* H_lp, const double* H_ll,
                      const double* b_p, const double* b_l, double* S, double* g, double eps) {
  const int ntile = (D + TS - 1) / TS;
  if (ntile == 1) {   // sliding-window case: TMA-pipelined kernel, warps own output tiles
    const int Fp = (F + kTmaStageL - 1) / kTmaStageL * kTmaStageL;
    VIML_TRY_CUDA(ctx, ctx->scratch2.reserve(2 * DeviceArena::padded((size_t)W * Fp * 8)));
    double* invp = ctx->scratch2.take<double>((size_t)W * Fp);
    double* blp = ctx->scratch2.take<double>((size_t)W * Fp);
    if (Fp > 0) {   // F == 0: nothing to pad, and a grid of 0 blocks is a launch error
      LaunchScope ls(ctx, K_SCHUR);
      schur_inv_kernel<<<(unsigned)(((size_t)W * Fp + 255) / 256), 256, 0, ctx->stream>>>(W, F, Fp, H_ll, b_l, eps, invp, blp);
    }
    const int smem = kTmaStages * kTmaStageD * (int)sizeof(double) + 2 * kTmaStages * 8;
    VIML_TRY_CUDA(ctx, cudaFuncSetAttribute(schur_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const int grid = W < 2 * ctx->sm_count ? W : 2 * ctx->sm_count;
    LaunchScope ls(ctx, K_SCHUR);
    schur_tma_kernel<<<(unsigned)grid, kTmaThreads, smem, ctx->stream>>>(W, F, Fp, D, H_pp, H_lp, invp, blp, b_p, S, g);
    return VIML_OK;
  }
  dim3 grid((unsigned)(ntile * (ntile + 1) / 2), (unsigned)W);
  int *order = nullptr, *tstart = nullptr, *span = nullptr;
  if (ntile >= 3 && ntile <= 31 && F > 0) {   // long window: band plan (a landmark's row is non-zero in a few neighbouring tiles only)
    auto pad = [](size_t b) { return DeviceArena::padded(b); };
    VIML_TRY_CUDA(ctx, ctx->scratch2.reserve(3 * pad((size_t)W * F * 4) + pad((size_t)W * (ntile + 2) * 4) + pad((size_t)W * 4)));
    int* tmin = ctx->scratch2.take<int>((size_t)W * F);
    int* tmax = ctx->scratch2.take<int>((size_t)W * F);
    order = ctx->scratch2.take<int>((size_t)W * F);
    tstart = ctx->scratch2.take<int>((size_t)W * (ntile + 2));
    span = ctx->scratch2.take<int>((size_t)W);
    {
      LaunchScope ls(ctx, K_SCHUR);
      extent_kernel<<<dim3((unsigned)((F + 7) / 8), (unsigned)W), 256, 0, ctx->stream>>>(F, D, H_lp, tmin, tmax, ntile);
    }
    {
      LaunchScope ls(ctx, K_SCHUR);
      order_kernel<<<(unsigned)W, 1024, 0, ctx->stream>>>(F, ntile, tmin, tmax, order, tstart, span);
    }
  }
  {
    LaunchScope ls(ctx, K_SCHUR);
    schur_dmma_kernel<<<grid, SWARPS * 32, 0, ctx->stream>>>(F, D, H_pp, H_lp, H_ll, b_p, b_l, S, g, eps, ntile, order, tstart, span);
  }
  if (order) {
    LaunchScope ls(ctx, K_SCHUR);
    ex_block_kernel<<<(unsigned)W, 256, 0, ctx->stream>>>(F, D, H_pp, H_lp, H_ll, b_p, b_l, S, g, eps);
  }
  return VIML_OK;
}

double viml_dmma_peak_tflops(viml_ctx* ctx) {
  const int blocks = ctx->sm_count * 8, threads = 256, iters = 2048;
  if (ctx->scratch.reserve((size_t)blocks * threads * sizeof(double)) != cudaSuccess) return 0.0;
  double* out = ctx->scratch.take<double>((size_t)blocks * threads);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0, ctx->stream);
    {
      LaunchScope ls(ctx, K_MICRO);
      dmma_peak_kernel<<<blocks, threads, 0, ctx->stream>>>(out, 1.0000001, 0.9999999, iters);
    }
    cudaEventRecord(e1, ctx->stream);
    cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    const double flops = (double)blocks * (threads / 32) * iters * 8 * 512.0;  // m8n8k4 = 256 FMA
    const double r = flops / (ms * 1e-3) / 1e12;
    if (rep > 0 && r > best) best = r;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return best;
}
