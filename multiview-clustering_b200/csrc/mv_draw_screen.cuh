// mv_draw_screen.cuh — exact screening inside the tensor-core draw (DESIGN.md §4.1.1).  Included by mv_draw_tc.cu.
//
// For a row x at table t0, with every table slot live and every dish served by one table, k_draw_tc evaluates
//   lw_t  = LM_t  + sum_v (C_vt  - A_vt  |x_v|^2 + x_v.b_vt)                 (t != t0)
//   lw_t0 = LM1_t0 + sum_v (C1_vt0 - A1_vt0 |x_v|^2 + R_vt0 x_v.b_vt0)      (R = A1 / A as the kernel rounds it)
// and draws t0 for every uniform when lw_t0 - max_{t != t0} lw_t > 31 (the dominant-option shortcut of k_draw_tc).
// When k_draw_tc evaluates such a row it records g' = (lw_t0 - max_{t != t0} lw_t) - Q_row(s) in `margin`, where
// Q_row(s) = k0 + sum_v kA_v |x_v|^2 + kB_v |x_v| bounds the change of every log-weight between the parameters of the
// REFERENCE sweep and those of sweep s (each term counted twice: own table and best other) plus the error of the FP32 /
// 3-pass TF32 evaluation.  In a later sweep s' the row's gap is then at least g' - Q_row(s'); if that exceeds 31 its draw
// is t0 without reading x.  A tile of 128 rows in which every row passes is screened: it is left off the list of tiles the
// draw evaluates and written nothing, because what the draw would write there (choice = t0, no birth bit, no moved bit)
// is already in place (DESIGN.md §4.1.1: a finite margin is only ever recorded beside exactly these values).
//
// The reference (a copy of the parameter block and the scaled means) is taken in a refresh sweep, in which every tile is
// evaluated.  A refresh happens when no reference is valid (new handle, set_state, a sweep that did not screen), every
// kScreenPeriod sweeps, and whenever a table's dish, its lone flag or which of its LM / LM1 / C1 are masked differ from the
// reference.  A sweep with a free table slot, a shared dish, blocked passes or debug exports does not screen (mode
// kScreenOff) and invalidates the reference.
//
// Every CTA of k_draw_tc decides the mode and the coefficients for itself, from the same inputs, and tests its own tiles
// (blockIdx.x, + gridDim.x, ...: the tiles it would evaluate without screening).  An arrival counter finds the last CTA
// to have decided, and only that one writes what the decision reads (the reference, its sweep and the valid flag): a CTA
// that starts late still sees the inputs the others saw.  The other roles of the CTA are released (list_full) between
// decide() and publish(), so the arrival counter is not on their path.
#pragma once
#include "mv_ctx.h"

namespace mv {

namespace screen {

constexpr int kTile = 128;                    // = kTileRows of k_draw_tc
constexpr int kThreads = 512;                 // the epilogue warpgroups of k_draw_tc run the screening
constexpr int kWarps = kThreads / 32;

struct Scratch {                              // shared memory of the screening phase (k_draw_tc's exchange area)
  double w[kWarps][7];                        // per warp: |b|, max(|db|, |d(Rb)|), then the five scalar maxima below
  int flags;                                  // bit 0: no screening this sweep, bit 1: refresh
  int n_eval;                                 // tiles of this CTA on the list
  unsigned rows;                              // rows of this CTA screened
  int last;                                   // this CTA is the last to have decided
};

__device__ __forceinline__ bool masked(float x) { return !(x > -1.0e29f); }
__device__ __forceinline__ double warp_max(double x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x = fmax(x, __shfl_xor_sync(0xffffffffu, x, o));
  return x;
}
__device__ __forceinline__ float ratio(const TableParam& q) { return (q.A != 0.0f) ? __fdiv_rn(q.A1, q.A) : 0.0f; }   // as k_draw_tc stages it
__device__ __forceinline__ void sync() { asm volatile("bar.sync 9, 512;" ::: "memory"); }   // the epilogue warpgroups only

// The tile test.  Q_row (screen_row_bound) is nondecreasing in each |x_v|^2: every coefficient is >= 0 and every step is an
// upward-rounded FMA or square root, each nondecreasing in its operands.  __fsub_rd(m, q) is nondecreasing in m and
// nonincreasing in q.  So with m_min <= every row's margin and xx_max >= every row's norms,
//   __fsub_rd(m_min, Q(xx_max)) <= __fsub_rd(margin_row, Q(xx_row))   for every row of the tile,
// and a tile that passes this test passes the per-row test in every row.  A NaN norm enters xx_max as +inf (k_rownorms)
// and a NaN margin enters m_min as -inf (k_draw_tc), so that such a tile fails here as its row fails the per-row test.
__device__ __forceinline__ bool tile_passes(const float* k, const float* xx_max, float m_min, int V) {
  return __fsub_rd(m_min, screen_row_bound(k, xx_max, V)) > 31.0f;
}

// What the verdict reads, per epilogue thread et: (view, table) et < V * 64, table et - 256's masses for 256 <= et < 320,
// and the summaries of this warp's first batch of tiles (lane 4 i + j: chunk j and view j of tile i).  k_draw_tc loads it
// in the same round as the parameters it stages, right after the grid dependency.  margin_min must not be read earlier:
// the previous draw triggers this grid before it writes its margins.
struct Inputs {
  GlobalParam g;
  uint32_t valid, ref_sweep;
  TableParam q, p;                            // this sweep's and the reference's parameters of (view, table) et
  double s3[3];                               // k_finalize's sums of (view, table) et
  TableMass m, pm;                            // this sweep's and the reference's masses of table et - 256
  float mn, xm;                               // margin_min of chunk j, xx_tmax of view j of tile i of the first batch
};

constexpr int kBatch = 8;                     // tiles a warp tests together: lane 4 i + j reads chunk j and view j of tile i

__device__ __forceinline__ int batch_tile(int base, int lane) { return base + (lane >> 2) * kWarps * (int)gridDim.x; }

// Lane 4 i + j's summary loads for the batch of tiles base, + kWarps * gridDim.x, ... (tiles past the end: +inf / 0).
__device__ __forceinline__ void load_batch(const Ctx& c, int base, int lane, int n_tiles, float& mn, float& xm) {
  const int tile = batch_tile(base, lane), j = lane & 3;
  mn = INFINITY;
  xm = 0.0f;
  if (tile < n_tiles) {
    if (tile * (kTile / 32) + j < c.n_chunks) mn = c.margin_min[tile * (kTile / 32) + j];
    if (j < c.V) xm = c.xx_tmax[(size_t)j * n_tiles + tile];
  }
}

__device__ __forceinline__ void load(const Ctx& c, int et, Inputs& in) {
  const int lane = et & 31, n_tiles = (c.n_rows + kTile - 1) / kTile;
  in.g = *c.gparam;
  in.valid = c.scr->valid;
  in.ref_sweep = c.scr->ref_sweep;
  in.s3[0] = in.s3[1] = in.s3[2] = 0.0;
  if (et < c.V * 64) {
    in.q = c.tparam[et];
    in.p = c.scr_tp[et];
    const double* s3 = c.scr_sum + 3 * et;
    in.s3[0] = s3[0]; in.s3[1] = s3[1]; in.s3[2] = s3[2];
  } else if (et >= 256 && et < 256 + 64) {
    in.m = c.tmass[et - 256];
    in.pm = c.scr_tm[et - 256];
  }
  load_batch(c, blockIdx.x + (et >> 5) * gridDim.x, lane, n_tiles, in.mn, in.xm);
}

// Run by the 512 epilogue threads (et = 0..511) on what load() read.  Decides the sweep's mode, writes the bound
// coefficients to k_out[7] and, in a skip sweep, tests this CTA's tiles and lists the others at
// c.scr_work[blockIdx.x + j * gridDim.x], j < S->n_eval.  Returns the mode; the tile list is complete when it returns.
// A screened tile is written nothing: its rows already hold choice == table_cur and its birth and moved words are zero
// (DESIGN.md §4.1.1, the invariant of the margins).
__device__ int decide(const Ctx& c, int et, const Inputs& in, Scratch* S, float* k_out) {
  const int warp = et >> 5, lane = et & 31;
  const int V = c.V;
  ScreenRec* R = c.scr;
  const int n_tiles = (c.n_rows + kTile - 1) / kTile;
  if (et == 0) { S->flags = 0; S->n_eval = 0; S->rows = 0u; }
  sync();

  // ---- the sweep's mode: the same inputs in every CTA, so the same verdict ---------------------------------------
  // and, from the same loads, the maxima the coefficients are built from: threads v * 64 + t take (view v, table t),
  // threads 256 + t table t's masses.  Per (view, table) k_finalize has summed |b|^2, |b - b_ref|^2, |R b - R_ref b_ref|^2.
  // Masked C1 / LM1 (a table of one customer) are left out: they are masked in the reference as well (a change
  // refreshes), and a row at such a table never records a margin (its own weight is masked).
  const GlobalParam& g = in.g;
  int off = (c.debug_export != 0 || c.blk_count != 1 || !masked(g.LMN0) || !masked(g.LMN1)) ? 1 : 0;
  int chg = (in.valid == 0u || g.sweep - in.ref_sweep >= (uint32_t)kScreenPeriod) ? 1 : 0;
  double w[7] = {0, 0, 0, 0, 0, 0, 1.0};
  if (et < V * 64) {
    const TableParam& q = in.q;
    const TableParam& p = in.p;
    if (q.dish < 0 || !q.lone) off = 1;
    if (q.dish != p.dish || q.lone != p.lone || masked(q.C1) != masked(p.C1)) chg = 1;
    const bool m1 = masked(q.C1);
    w[0] = sqrt(in.s3[0]);
    w[1] = fmax(sqrt(in.s3[1]), sqrt(in.s3[2]));
    w[2] = fabs((double)q.C - (double)p.C);
    if (!m1) w[2] = fmax(w[2], fabs((double)q.C1 - (double)p.C1));
    w[3] = fmax(fabs((double)q.A - (double)p.A), fabs((double)q.A1 - (double)p.A1));
    w[4] = fabs((double)q.C);
    if (!m1) w[4] = fmax(w[4], fabs((double)q.C1));
    w[5] = fmax(fabs((double)q.A), fabs((double)q.A1));
    w[6] = fmax(1.0, (double)ratio(q));
  } else if (et >= 256 && et < 256 + 64) {
    const TableMass& m = in.m;
    const TableMass& p = in.pm;
    if (masked(m.LM) != masked(p.LM) || masked(m.LM1) != masked(p.LM1)) chg = 1;
    w[2] = fabs((double)m.LM - (double)p.LM);
    if (!masked(m.LM1)) w[2] = fmax(w[2], fabs((double)m.LM1 - (double)p.LM1));
    w[4] = fabs((double)m.LM);
    if (!masked(m.LM1)) w[4] = fmax(w[4], fabs((double)m.LM1));
  }
  if (off) atomicOr(&S->flags, 1);
  if (chg) atomicOr(&S->flags, 2);
#pragma unroll
  for (int i = 0; i < 7; ++i) w[i] = warp_max(w[i]);
  if (lane == 0)
    for (int i = 0; i < 7; ++i) S->w[warp][i] = w[i];
  sync();
  const int mode = (S->flags & 1) ? kScreenOff : ((S->flags & 2) ? kScreenRefresh : kScreenSkip);
  if (blockIdx.x == 0 && et == 0) R->sweep = g.sweep;
  if (mode == kScreenOff) {
    if (blockIdx.x == 0 && et == 0) { R->mode = mode; R->last_rows_screened = 0; R->last_tiles_evaluated = n_tiles; R->valid = 0u; }
    return mode;
  }
  const bool skip = (mode == kScreenSkip);

  // ---- the coefficients of Q (FP64; every term an upper bound) ------------------------------------------------------
  // Evaluation error, per evaluation (the record and the test each subtract their own): about 30 FP32 roundings of terms no
  // larger than the magnitudes (2^-14 is 2^4 above what they can add up to), and the 3-pass TF32 dot products, whose error
  // is ~2^-18 |x| |b| (2^-8 |x| |b| budgeted, times R >= 1 for the own table's R x.b).  The stored |x|^2 is an FMA sum of
  // 64 squares (relative error < 2^-17): |x| <= sqrt(|x|^2) (1 + 2^-12).  Drift terms count only against a reference.
  if (et < 7) {
    auto mx = [&](int w0, int i) { return fmax(S->w[w0][i], S->w[w0 + 1][i]); };   // the two warps of a view (8, 9: masses)
    double drift0 = skip ? mx(8, 2) : 0.0, mag0 = mx(8, 4);
    double kA[3] = {0, 0, 0}, kB[3] = {0, 0, 0};
    for (int v = 0; v < V; ++v) {
      drift0 += skip ? mx(2 * v, 2) : 0.0;
      mag0 += mx(2 * v, 4);
      const double nb = mx(2 * v, 0), ndb = skip ? mx(2 * v, 1) : 0.0;
      kA[v] = 2.0 * (skip ? mx(2 * v, 3) : 0.0) + 0x1p-14 * mx(2 * v, 5);
      kB[v] = (2.0 * ndb + (0x1p-8 + 0x1p-14) * mx(2 * v, 6) * nb) * (1.0 + 0x1p-12);
    }
    const double k0 = 2.0 * drift0 + 0x1p-14 * mag0;
    const double slack = 1.0 + 0x1p-30;             // the FP64 arithmetic above
    const double kd = (et == 0) ? k0 : ((et < 4) ? kA[et - 1] : kB[et - 4]);
    k_out[et] = __double2float_ru(kd * slack);
  }
  sync();
  if (blockIdx.x == 0 && et < 7) R->k[et] = k_out[et];
  if (blockIdx.x == 0 && et == 0) R->mode = mode;
  if (!skip) return mode;

  // ---- the tiles of this CTA: each warp tests kBatch tiles at a time from their summaries ------------------------------
  float kk[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) kk[i] = k_out[i];
  const int stride = kWarps * (int)gridDim.x;
  float mn = in.mn, xm = in.xm;
  unsigned rows = 0u;
  for (int base = blockIdx.x + warp * gridDim.x; base < n_tiles; base += kBatch * stride) {
    if (base != (int)blockIdx.x + warp * (int)gridDim.x) load_batch(c, base, lane, n_tiles, mn, xm);
    // lane 4 i: the least margin of tile i and its largest norms (a tile past the end passes with no rows)
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, 1));
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, 2));
    float xx[3];
#pragma unroll
    for (int v = 0; v < 3; ++v) xx[v] = __shfl_sync(0xffffffffu, xm, (lane & ~3) + v);
    const int tile = batch_tile(base, lane);
    const bool lead = (lane & 3) == 0 && tile < n_tiles;
    const bool pass = lead && tile_passes(kk, xx, mn, V);
    if (pass) rows += (unsigned)min(kTile, c.n_rows - tile * kTile);
    unsigned failed = __ballot_sync(0xffffffffu, lead && !pass);
    while (failed) {                                // today's per-row test: the verdict of the tile is exactly its rows'
      const int ft = __shfl_sync(0xffffffffu, tile, __ffs(failed) - 1);
      failed &= failed - 1u;
      bool ok = true;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int row = ft * kTile + j * 32 + lane;
        if (row < c.n_rows) {
          float xr[3];
#pragma unroll
          for (int v = 0; v < 3; ++v) xr[v] = (v < V) ? c.xx[(size_t)v * c.xx_stride + row] : 0.0f;
          ok = ok && (__fsub_rd(c.margin[row], screen_row_bound(kk, xr, V)) > 31.0f);
        }
      }
      if (__all_sync(0xffffffffu, ok)) {
        if (lane == 0) rows += (unsigned)min(kTile, c.n_rows - ft * kTile);
      } else if (lane == 0) {
        const int j = atomicAdd(&S->n_eval, 1);
        c.scr_work[blockIdx.x + j * gridDim.x] = ft;
        c.scr_tiles[atomicAdd(&R->cnt, 1u)] = ft;
      }
    }
  }
  rows = __reduce_add_sync(0xffffffffu, rows);
  if (lane == 0 && rows) atomicAdd(&S->rows, rows);
  sync();
  return mode;
}

// After decide(), once the other roles have the verdict and the list: the last CTA out publishes the counts and, in a
// refresh, writes the reference.
__device__ void publish(const Ctx& c, int et, int mode, uint32_t sweep, Scratch* S) {
  ScreenRec* R = c.scr;
  const int V = c.V;
  const int n_tiles = (c.n_rows + kTile - 1) / kTile;
  const bool skip = (mode == kScreenSkip);
  if (et == 0) {
    if (S->rows) atomicAdd(&R->rows, S->rows);
    __threadfence();
    S->last = (atomicAdd(&R->done, 1u) == gridDim.x - 1) ? 1 : 0;
    if (S->last) {
      __threadfence();
      R->done = 0u;
      if (skip) {
        const uint32_t n = atomicExch(&R->cnt, 0u);
        R->n_eval = (int32_t)n;
        R->last_tiles_evaluated = n;
        R->last_rows_screened = atomicExch(&R->rows, 0u);
      } else {
        R->last_rows_screened = 0;
        R->last_tiles_evaluated = n_tiles;
      }
    }
  }
  sync();
  if (S->last && !skip) {
    // A refresh makes this sweep's parameters the reference of the margins the draw records.  The reference is now this
    // sweep's own parameters, so the drift sums k_finalize left against the old one become zero (a draw repeated
    // without a new k_finalize in between screens against this reference).
    const int nb = c.cap * c.Dsum;
    for (int i = et; i < 2 * nb + V * 64 + 64; i += kThreads) {
      if (i < nb) c.scr_b[i] = c.mean_hi[i];
      else if (i < 2 * nb) c.scr_b[i] = c.mean_lo[i - nb];
      else if (i < 2 * nb + V * 64) {
        const int j = i - 2 * nb;
        c.scr_tp[j] = c.tparam[j];
        c.scr_sum[3 * j + 1] = 0.0;
        c.scr_sum[3 * j + 2] = 0.0;
      } else {
        c.scr_tm[i - 2 * nb - V * 64] = c.tmass[i - 2 * nb - V * 64];
      }
    }
    if (et == 0) { R->ref_sweep = sweep; R->valid = 1u; }
  }
}

}  // namespace screen

}  // namespace mv
