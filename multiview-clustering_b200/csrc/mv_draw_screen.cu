// mv_draw_screen.cu — exact screening ahead of the tensor-core draw (DESIGN.md §4.1.1).
//
// For a row x at table t0, with every table slot live and every dish served by one table, k_draw_tc evaluates
//   lw_t  = LM_t  + sum_v (C_vt  - A_vt  |x_v|^2 + x_v.b_vt)                 (t != t0)
//   lw_t0 = LM1_t0 + sum_v (C1_vt0 - A1_vt0 |x_v|^2 + R_vt0 x_v.b_vt0)      (R = A1 / A as the kernel rounds it)
// and draws t0 for every uniform when lw_t0 - max_{t != t0} lw_t > 31 (the dominant-option shortcut of k_draw_tc).
// When k_draw_tc evaluates such a row it records g' = (lw_t0 - max_{t != t0} lw_t) - Q_row(s) in `margin`, where
// Q_row(s) = k0 + sum_v kA_v |x_v|^2 + kB_v |x_v| bounds the change of every log-weight between the parameters of the
// REFERENCE sweep and those of sweep s (each term counted twice: own table and best other) plus the error of the FP32 /
// 3-pass TF32 evaluation.  In a later sweep s' the row's gap is then at least g' - Q_row(s'); if that exceeds 31 its draw
// is t0 without reading x.  This kernel makes that test for every row of a tile of 128; a tile with a row that fails
// goes on the list of tiles k_draw_tc evaluates, the others get exactly what the draw would have written: choice = t0,
// no birth bit, no moved bit.
//
// The reference (a copy of the parameter block and the scaled means) is taken by k_draw_tc in a refresh sweep, in which
// every tile is evaluated.  A refresh happens when no reference is valid (new handle, set_state, a sweep that did not
// screen), every kScreenPeriod sweeps, and whenever a table's dish, its lone flag or which of its LM / LM1 / C1 are
// masked differ from the reference.  A sweep with a free table slot, a shared dish, blocked passes or debug exports does
// not screen (mode kScreenOff) and invalidates the reference.
#include "mv_ctx.h"

namespace mv {

namespace {

constexpr int kScrThreads = 512;
constexpr int kScrWarps = kScrThreads / 32;
constexpr int kScrTile = 128;                 // = kTileRows of k_draw_tc

__device__ __forceinline__ bool masked(float x) { return !(x > -1.0e29f); }
__device__ __forceinline__ double warp_max(double x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x = fmax(x, __shfl_xor_sync(0xffffffffu, x, o));
  return x;
}
__device__ __forceinline__ double warp_sum(double x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}
__device__ __forceinline__ float ratio(const TableParam& q) { return (q.A != 0.0f) ? __fdiv_rn(q.A1, q.A) : 0.0f; }   // as k_draw_tc stages it

}  // namespace

__global__ void __launch_bounds__(kScrThreads) k_draw_screen(const Ctx c) {
  pdl_wait();                                       // the parameter block of this sweep comes from k_finalize
  pdl_trigger();                                    // k_draw_tc reads nothing of ours before its own wait
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int V = c.V;
  ScreenRec* R = c.scr;
  const int n_tiles = (c.n_rows + kScrTile - 1) / kScrTile;
  __shared__ int s_flags;                           // bit 0: no screening this sweep, bit 1: refresh
  __shared__ double s_nb[kScrWarps][3], s_ndb[kScrWarps][3], s_sc[4][5];
  __shared__ float s_k[7];
  if (tid == 0) s_flags = 0;
  __syncthreads();

  // ---- the sweep's mode: the same inputs in every CTA, so the same verdict -----------------------------------------
  const GlobalParam g = *c.gparam;
  int off = (c.debug_export != 0 || c.blk_count != 1 || !masked(g.LMN0) || !masked(g.LMN1)) ? 1 : 0;
  int chg = (R->valid == 0u || g.sweep - R->ref_sweep >= (uint32_t)kScreenPeriod) ? 1 : 0;
  for (int i = tid; i < V * 64; i += kScrThreads) {
    const TableParam q = c.tparam[i], p = c.scr_tp[i];
    if (q.dish < 0 || !q.lone) off = 1;
    if (q.dish != p.dish || q.lone != p.lone || masked(q.C1) != masked(p.C1)) chg = 1;
  }
  if (tid < 64) {
    const TableMass m = c.tmass[tid], p = c.scr_tm[tid];
    if (masked(m.LM) != masked(p.LM) || masked(m.LM1) != masked(p.LM1)) chg = 1;
  }
  if (off) atomicOr(&s_flags, 1);
  if (chg) atomicOr(&s_flags, 2);
  __syncthreads();
  const int mode = (s_flags & 1) ? kScreenOff : ((s_flags & 2) ? kScreenRefresh : kScreenSkip);
  if (blockIdx.x == 0 && tid == 0) R->sweep = g.sweep;
  if (mode == kScreenOff) {
    if (blockIdx.x == 0 && tid == 0) { R->mode = mode; R->last_rows_screened = 0; R->last_tiles_evaluated = n_tiles; }
    return;
  }
  const bool skip = (mode == kScreenSkip);

  // ---- the coefficients of Q (FP64; every term an upper bound) ------------------------------------------------------
  // per (view, table), one warp each: |b|, and max(|b - b_ref|, |R b - R_ref b_ref|), over the 64 coordinates
  double wb[3] = {0, 0, 0}, wdb[3] = {0, 0, 0};
  const size_t half = (size_t)c.cap * c.Dsum;
  for (int i = warp; i < V * 64; i += kScrWarps) {
    const int v = i >> 6;
    const TableParam q = c.tparam[i], p = c.scr_tp[i];
    const double rq = ratio(q), rp = ratio(p);
    double sb = 0.0, sd = 0.0, sr = 0.0;
    const size_t base = (size_t)c.cap * c.doff[v] + (size_t)(i & 63) * 64;
#pragma unroll
    for (int d = lane; d < 64; d += 32) {
      const double b = (double)c.mean_hi[base + d] + (double)c.mean_lo[base + d];
      sb += b * b;
      if (skip) {
        const double bp = (double)c.scr_b[base + d] + (double)c.scr_b[half + base + d];
        sd += (b - bp) * (b - bp);
        sr += (rq * b - rp * bp) * (rq * b - rp * bp);
      }
    }
    sb = warp_sum(sb); sd = warp_sum(sd); sr = warp_sum(sr);
    wb[v] = fmax(wb[v], sqrt(sb));
    wdb[v] = fmax(wdb[v], fmax(sqrt(sd), sqrt(sr)));
  }
  if (lane == 0)
    for (int v = 0; v < 3; ++v) { s_nb[warp][v] = wb[v]; s_ndb[warp][v] = wdb[v]; }
  // warp v < V: max |dC|, |dC1| / max |dA|, |dA1| / max |C|, |C1| / max A, A1 / max R of view v;  warp 3: max |dLM|,
  // |dLM1| / - / max |LM|, |LM1|.  Masked C1 / LM1 (a table of one customer) are left out: they are masked in the
  // reference as well (a change refreshes), and a row at such a table never records a margin (its own weight is masked).
  double sc[5] = {0, 0, 0, 0, 1.0};
  if (warp < V) {
    for (int t = lane; t < 64; t += 32) {
      const TableParam q = c.tparam[warp * 64 + t], p = c.scr_tp[warp * 64 + t];
      const bool m1 = masked(q.C1);
      if (skip) {
        sc[0] = fmax(sc[0], fabs((double)q.C - (double)p.C));
        if (!m1) sc[0] = fmax(sc[0], fabs((double)q.C1 - (double)p.C1));
        sc[1] = fmax(sc[1], fmax(fabs((double)q.A - (double)p.A), fabs((double)q.A1 - (double)p.A1)));
      }
      sc[2] = fmax(sc[2], fabs((double)q.C));
      if (!m1) sc[2] = fmax(sc[2], fabs((double)q.C1));
      sc[3] = fmax(sc[3], fmax(fabs((double)q.A), fabs((double)q.A1)));
      sc[4] = fmax(sc[4], (double)ratio(q));
    }
  } else if (warp == 3) {
    for (int t = lane; t < 64; t += 32) {
      const TableMass m = c.tmass[t], p = c.scr_tm[t];
      if (skip) {
        sc[0] = fmax(sc[0], fabs((double)m.LM - (double)p.LM));
        if (!masked(m.LM1)) sc[0] = fmax(sc[0], fabs((double)m.LM1 - (double)p.LM1));
      }
      sc[2] = fmax(sc[2], fabs((double)m.LM));
      if (!masked(m.LM1)) sc[2] = fmax(sc[2], fabs((double)m.LM1));
    }
  }
#pragma unroll
  for (int k = 0; k < 5; ++k) sc[k] = warp_max(sc[k]);
  if (lane == 0 && warp < 4)
    for (int k = 0; k < 5; ++k) s_sc[warp][k] = sc[k];
  __syncthreads();
  if (tid == 0) {
    // Evaluation error, per evaluation (the record and the test each subtract their own): about 30 FP32 roundings of terms
    // no larger than the magnitudes (2^-14 is 2^4 above what they can add up to), and the 3-pass TF32 dot products, whose
    // error is ~2^-18 |x| |b| (2^-8 |x| |b| budgeted, times R >= 1 for the own table's R x.b).  The stored |x|^2 is an FMA
    // sum of 64 squares (relative error < 2^-17): |x| <= sqrt(|x|^2) (1 + 2^-12).
    double drift0 = s_sc[3][0], mag0 = s_sc[3][2];
    double kA[3] = {0, 0, 0}, kB[3] = {0, 0, 0};
    for (int v = 0; v < V; ++v) {
      drift0 += s_sc[v][0];
      mag0 += s_sc[v][2];
      double nb = 0.0, ndb = 0.0;
      for (int w = 0; w < kScrWarps; ++w) { nb = fmax(nb, s_nb[w][v]); ndb = fmax(ndb, s_ndb[w][v]); }
      kA[v] = 2.0 * s_sc[v][1] + 0x1p-14 * s_sc[v][3];
      kB[v] = (2.0 * ndb + (0x1p-8 + 0x1p-14) * s_sc[v][4] * nb) * (1.0 + 0x1p-12);
    }
    const double k0 = 2.0 * drift0 + 0x1p-14 * mag0;
    const double slack = 1.0 + 0x1p-30;             // the FP64 arithmetic above
    s_k[0] = __double2float_ru(k0 * slack);
    for (int v = 0; v < 3; ++v) { s_k[1 + v] = __double2float_ru(kA[v] * slack); s_k[4 + v] = __double2float_ru(kB[v] * slack); }
  }
  __syncthreads();
  if (blockIdx.x == 0 && tid < 7) R->k[tid] = s_k[tid];
  if (blockIdx.x == 0 && tid == 0) R->mode = mode;
  if (!skip) {
    if (blockIdx.x == 0 && tid == 0) { R->last_rows_screened = 0; R->last_tiles_evaluated = n_tiles; }
    return;
  }

  // ---- the rows: one warp per tile of 128 ------------------------------------------------------------------------------
  float kk[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) kk[i] = s_k[i];
  for (int tile = blockIdx.x * kScrWarps + warp; tile < n_tiles; tile += gridDim.x * kScrWarps) {
    bool pass = true;
    int t0[4];
    int nlive = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int row = tile * kScrTile + j * 32 + lane;
      t0[j] = 0;
      if (row < c.n_rows) {
        ++nlive;
        t0[j] = c.table_cur[row];
        float xx[3];
#pragma unroll
        for (int v = 0; v < 3; ++v) xx[v] = (v < V) ? c.xx[(size_t)v * c.xx_stride + row] : 0.0f;
        const float q = screen_row_bound(kk, xx, V);
        pass = pass && (__fsub_rd(c.margin[row], q) > 31.0f);
      }
    }
    if (__all_sync(0xffffffffu, pass)) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int row = tile * kScrTile + j * 32 + lane;
        if (row < c.n_rows) c.choice[row] = t0[j];
      }
      const int chunk = tile * (kScrTile / 32) + lane;
      if (lane < kScrTile / 32 && chunk < c.n_chunks) { c.birthmask[chunk] = 0u; c.movedmask[chunk] = 0u; }
      const unsigned rows = __reduce_add_sync(0xffffffffu, (unsigned)nlive);
      if (lane == 0) atomicAdd(&R->rows, rows);
    } else if (lane == 0) {
      c.scr_tiles[atomicAdd(&R->cnt, 1u)] = tile;
    }
  }
  // ---- the last CTA out publishes the list length and clears the scratch for the next launch --------------------------
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    if (atomicAdd(&R->done, 1u) == gridDim.x - 1) {
      __threadfence();
      const uint32_t n = atomicExch(&R->cnt, 0u);
      R->n_eval = (int32_t)n;
      R->last_tiles_evaluated = n;
      R->last_rows_screened = atomicExch(&R->rows, 0u);
      R->done = 0u;
      __threadfence();
    }
  }
}

cudaError_t launch_draw_screen(const Ctx& c, bool programmatic, cudaStream_t s) {
  if (c.n_rows <= 0 || !c.screen) return cudaSuccess;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int n_tiles = (c.n_rows + kScrTile - 1) / kScrTile;
  const int want = (n_tiles + kScrWarps - 1) / kScrWarps;
  const int grid = want < sms ? want : sms;
  return launch_chain(k_draw_screen, dim3(grid), dim3(kScrThreads), 0, s, programmatic, c);
}

}  // namespace mv
