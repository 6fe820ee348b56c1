// mv_state_kernels.cu — everything of a sweep that is not the likelihood+draw kernel:
//
//   k_pack      ordered compaction of the rows that drew "new table" (first `nfree` in row order
//               become candidates; their features go into the exchange packet)
//   k_stats     segmented reduction of the rows into per-TABLE sufficient statistics
//               (fixed row->CTA->warp mapping, per-warp private accumulators: a fixed-order tree)
//   (k_reduce_x, mv_exchange.cu: fixed-order FP64 sums of the per-CTA partials, exchange, rank-ordered totals)
//   k_finalize  one CTA per level of the hierarchy (V views + the franchise): births (dish sampling) and
//               deaths, per-dish statistics, the Metropolis-Hastings hyperparameter step, and the
//               FP32 parameter block of the next sweep
//
// Reference code being replaced (paths under /root/reference/Multiview):
//   sufficient statistics      multiview_gibbs.cpp:64-73 (rebuild), multiview_utils.cpp:151-163,199-206
//   births                     create_empty_table / assign_dishes_new_table / sample_dish_for_new_table,
//                              multiview_utils.cpp:209-289
//   deaths                     remove_customer's empty-table branch, multiview_utils.cpp:168-191
//   hyper step                 update_hyperparameters and helpers, multiview_hyper.cpp:53-128,166-360
#include <stdlib.h>

#include "mv_ctx.h"

namespace mv {

constexpr double kEps = 1e-6;            // multiview_hyper.cpp:13
constexpr double kLog2e = 1.4426950408889634074;
constexpr double kPi = 3.14159265358979323846;

// k_finalize runs once per sweep with a cold instruction cache, and FP64 log/exp/lgamma expand to hundreds of
// instructions at every call site: one out-of-line copy of each keeps the kernel small enough to fetch quickly.
__device__ __noinline__ double fin_log(double x) { return log(x); }
__device__ __noinline__ double fin_exp(double x) { return exp(x); }
__device__ __noinline__ double fin_lgamma(double x) { return lgamma(x); }
__device__ __noinline__ double fin_log2(double x) { return log2(x); }

__device__ __forceinline__ int32_t* pkt_i32(const Ctx& c, int g, int off) {
  return reinterpret_cast<int32_t*>(c.packet + (size_t)g * c.pkt.bytes + off);
}
__device__ __forceinline__ double* pkt_f64(const Ctx& c, int g, int off) {
  return reinterpret_cast<double*>(c.packet + (size_t)g * c.pkt.bytes + off);
}
__device__ __forceinline__ float* pkt_f32(const Ctx& c, int g, int off) {
  return reinterpret_cast<float*>(c.packet + (size_t)g * c.pkt.bytes + off);
}

// =============================================================================================
// k_pack
// =============================================================================================
constexpr int kPackThreads = 1024;

__global__ void __launch_bounds__(kPackThreads, 1) k_pack(const Ctx c) {
  __shared__ int s_warp[32];
  __shared__ int s_total;
  pdl_trigger();
  pdl_wait();
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nfree = c.gparam->nfree;
  int32_t* cand_row = pkt_i32(c, c.rank, c.pkt.off_cand_row);
  int32_t* cand_t0 = pkt_i32(c, c.rank, c.pkt.off_cand_t0);
  if (nfree == 0) {
    // No free table slot at sweep start: the new-table option had no weight (capacity rule), so no row can have
    // drawn it and the birth mask is all zero — nothing to scan, nothing to compact.
    if (tid == 0) {
      int32_t* hdr = pkt_i32(c, c.rank, c.pkt.off_hdr);
      hdr[0] = 0; hdr[1] = 0; hdr[2] = c.rank; hdr[3] = 0;
      *reinterpret_cast<int64_t*>(hdr + 4) = c.row_offset;
      hdr[6] = 0; hdr[7] = 0;
    }
    return;
  }
  const int per = (c.n_chunks + kPackThreads - 1) / kPackThreads;
  const int lo = min(tid * per, c.n_chunks), hi = min(lo + per, c.n_chunks);
  int cnt = 0;
  for (int ch = lo; ch < hi; ++ch) cnt += __popc(c.birthmask[ch]);
  // block exclusive scan of cnt
  int incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int w = s_warp[lane];
    int wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += y;
    }
    s_warp[lane] = wi - w;            // exclusive prefix of the warp totals
    if (lane == 31) s_total = wi;
  }
  __syncthreads();
  int running = s_warp[wid] + incl - cnt;
  // chunk_prefix is only read for rows that drew a new table: with no birth anywhere it is not needed
  if (s_total > 0) for (int ch = lo; ch < hi; ++ch) {
    c.chunk_prefix[ch] = running;
    unsigned m = c.birthmask[ch];
    while (m) {
      const int b = __ffs(m) - 1;
      m &= m - 1;
      if (running < nfree) cand_row[running] = ch * 32 + b;
      ++running;
    }
  }
  __syncthreads();
  const int total = s_total;
  const int ncand = total < nfree ? total : nfree;
  if (tid == 0) {
    int32_t* hdr = pkt_i32(c, c.rank, c.pkt.off_hdr);
    hdr[0] = ncand; hdr[1] = total; hdr[2] = c.rank; hdr[3] = 0;
    *reinterpret_cast<int64_t*>(hdr + 4) = c.row_offset;
    hdr[6] = 0; hdr[7] = 0;
  }
  __threadfence_block();
  __syncthreads();
  float* cx = pkt_f32(c, c.rank, c.pkt.off_cand_x);
  for (int j = wid; j < ncand; j += kPackThreads / 32) {
    const int row = cand_row[j];
    if (lane == 0) cand_t0[j] = c.table_cur[row];
    for (int v = 0; v < c.V; ++v) {
      const int D = c.D[v];
      const float* src = c.x[v] + (size_t)row * D;
      float* dst = cx + (size_t)j * c.Dsum + c.doff[v];
      for (int dd = lane; dd < D; dd += 32) dst[dd] = src[dd];
    }
  }
}

cudaError_t launch_pack(const Ctx& c, cudaStream_t s) {
  return launch_chain(k_pack, dim3(1), dim3(kPackThreads), 0, s, c.pdl != 0, c);
}

// =============================================================================================
// k_stats
// =============================================================================================
// Segmented reduction of the rows into per-TABLE statistics: one CTA per SM walks a fixed range of 32-row
// chunks.  Its warps form R row groups x G column groups: a warp owns 32 of the concatenated feature
// columns (lane = column, so a row is one coalesced 128-byte load; the squared norms of the rows, computed
// once when a view is uploaded, are V more columns) and, for the rows of its row group, adds them into a
// private [cap][32] block of sums in shared memory —
// no two warps ever touch the same cell, rows are added in ascending order, the row groups are summed in
// ascending order: a fixed tree, bit-reproducible for a given launch shape.  Loads run a batch of rows
// ahead of their use.
struct StatsPlan { int Gp, R, passes, smem; };

static StatsPlan stats_plan(const Ctx& c) {
  const int Gtot = (c.Dsum + c.V + 31) / 32;         // feature columns, then one column of squared norms per view
  const int slot_bytes = c.cap * 32 * (int)sizeof(float);                // sums of one (row group, column group)
  const int slots = (200 * 1024) / slot_bytes;
  StatsPlan pl;
  int gmax = slots / 2 > 1 ? slots / 2 : 1;          // leave room for at least two row groups
  if (gmax > 16) gmax = 16;
  pl.Gp = Gtot < gmax ? Gtot : gmax;
  int R = slots / pl.Gp;
  if (R > 8) R = 8;
  if (R * pl.Gp > 24) R = 24 / pl.Gp;                  // at most 24 warps: 80 registers each
  if (R < 1) R = 1;
  pl.R = R;
  pl.passes = (Gtot + pl.Gp - 1) / pl.Gp;
  pl.smem = R * pl.Gp * slot_bytes + R * c.cap * (int)sizeof(int32_t);
  return pl;
}
int stats_smem_bytes(const Ctx& c) { return stats_plan(c).smem; }

constexpr int kStatBatch = 8;    // rows whose loads are in flight per warp while the previous batch is accumulated
constexpr int kStatAhead = 4;    // chunks (of 32 rows) the L2 prefetch runs ahead of the loads

__global__ void __launch_bounds__(768, 1) k_stats(const Ctx c, const int Gp, const int R, const int passes) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int cap = c.cap;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nthreads = blockDim.x;
  const int rg = wid / Gp, cg = wid - rg * Gp;
  float* s_sum = reinterpret_cast<float*>(smem_raw);                            // [R][Gp][cap][32]
  int32_t* s_cnt = reinterpret_cast<int32_t*>(s_sum + (size_t)R * Gp * cap * 32);  // [R][cap]
  float* acc = s_sum + ((size_t)rg * Gp + cg) * cap * 32;
  int32_t* cntw = s_cnt + rg * cap;

  // fixed mapping rows -> CTA -> row group, in whole 32-row chunks
  const int chunks_per_cta = (c.n_chunks + gridDim.x - 1) / gridDim.x;
  const int cta_lo = min((int)blockIdx.x * chunks_per_cta, c.n_chunks);
  const int cta_hi = min(cta_lo + chunks_per_cta, c.n_chunks);
  const int chunks_per_rg = (cta_hi - cta_lo + R - 1) / R;
  const int w_lo = min(cta_lo + rg * chunks_per_rg, cta_hi);
  const int w_hi = min(w_lo + chunks_per_rg, cta_hi);
  const int nfree = c.gparam->nfree;
  const int last_row = c.n_rows - 1;

  const size_t part_stride = (size_t)cap * c.Dsum + (size_t)c.V * cap;
  float* part = c.partial_f + (size_t)blockIdx.x * part_stride;
  float* part_s2 = part + (size_t)cap * c.Dsum;

  for (int pass = 0; pass < passes; ++pass) {
    // this lane's column of the concatenated views
    // (columns Dsum .. Dsum+V-1 are the precomputed squared norms of the rows, one array per view)
    const int col = (pass * Gp + cg) * 32 + lane;
    const bool has = col < c.Dsum + c.V;
    int v = 0;
    while (v + 1 < c.V && col >= c.doff[v + 1]) ++v;
    const bool is_norm = col >= c.Dsum;
    const int D = (is_norm || !has) ? 1 : c.D[v];
    const float* __restrict__ base = !has ? c.xx : (is_norm ? c.xx + (size_t)(col - c.Dsum) * c.xx_stride : c.x[v] + (col - c.doff[v]));
    for (int i = lane; i < cap * 32; i += 32) acc[i] = 0.0f;
    if (pass == 0 && cg == 0) for (int i = lane; i < cap; i += 32) cntw[i] = 0;
    __syncwarp();
    const bool owner = (pass == 0 && cg == 0);      // the warp that records the resolved assignment of its rows

    float nx[kStatBatch];
    auto issue = [&](int ch, int j0) {
#pragma unroll
      for (int u = 0; u < kStatBatch; ++u) {
        int r = ch * 32 + j0 + u;
        r = r < last_row ? r : last_row;
        nx[u] = __ldg(base + (size_t)r * D);
      }
    };
    // the assignment of a chunk's rows is fetched one chunk ahead of its use, like the features
    auto load_choice = [&](int ch) {
      const int row = ch * 32 + lane;
      return (ch < w_hi && row < c.n_rows) ? c.choice[row] : -3;
    };
    int tj_next = load_choice(w_lo);
    if (w_lo < w_hi) issue(w_lo, 0);
    for (int ch = w_lo; ch < w_hi; ++ch) {
      {   // one instruction pulls this warp's 128-byte segments of 32 rows, kStatAhead chunks on, into L2
        int pr = (ch + kStatAhead) * 32 + lane;
        pr = pr < last_row ? pr : last_row;
        asm volatile("prefetch.global.L2 [%0];" ::"l"(base + (size_t)pr * D));
      }
      const int row = ch * 32 + lane;
      int tj = tj_next;                              // -3: beyond the end
      tj_next = load_choice(ch + 1);
      if (row < c.n_rows) {
        if (tj == kNewTable) {                       // a birth: seated (candidate, -2) or overflow (stays put)
          const unsigned m = c.birthmask[ch];
          const int rank = c.chunk_prefix[ch] + __popc(m & ((1u << lane) - 1u));
          tj = (rank < nfree) ? -2 : c.table_cur[row];
          if (owner) c.choice[row] = tj;
        }
        if (owner && tj >= 0) c.table_cur[row] = tj;
      }
      if (owner) {
        // customers per table: the lanes of one table elect a leader, which adds their number — one
        // shared-memory update per distinct table of the chunk instead of one per row
        const unsigned peers = __match_any_sync(0xffffffffu, tj);
        if (tj >= 0 && lane == __ffs(peers) - 1) cntw[tj] += __popc(peers);
      }
      for (int j0 = 0; j0 < 32; j0 += kStatBatch) {
        float xs[kStatBatch];
        int ts[kStatBatch];
#pragma unroll
        for (int u = 0; u < kStatBatch; ++u) {
          xs[u] = has ? nx[u] : 0.0f;
          ts[u] = __shfl_sync(0xffffffffu, tj, j0 + u);
        }
        if (j0 + kStatBatch < 32) issue(ch, j0 + kStatBatch);
        else if (ch + 1 < w_hi) issue(ch + 1, 0);
#pragma unroll
        for (int u = 0; u < kStatBatch; ++u) {
          const int t = ts[u];
          if (t < 0) continue;                        // warp-uniform
          float* a = acc + t * 32 + lane;
          *a = __fadd_rn(*a, xs[u]);
        }
      }
    }
    __syncthreads();
    // fixed-order sums over the row groups -> this CTA's partials
    const int ncols_pass = Gp * 32;
    for (int i = tid; i < cap * ncols_pass; i += nthreads) {
      const int t = i / ncols_pass, cc = i - t * ncols_pass;
      const int gcol = pass * ncols_pass + cc;
      if (gcol < c.Dsum) {
        const int g = cc >> 5, l = cc & 31;
        float sum = 0.0f;
        for (int r = 0; r < R; ++r) sum = __fadd_rn(sum, s_sum[(((size_t)r * Gp + g) * cap + t) * 32 + l]);
        int vv = 0;
        while (vv + 1 < c.V && gcol >= c.doff[vv + 1]) ++vv;
        part[(size_t)cap * c.doff[vv] + (size_t)t * c.D[vv] + (gcol - c.doff[vv])] = sum;
      }
    }
    for (int i = tid; i < c.V * cap; i += nthreads) {       // sums of squared norms: the column Dsum + vv
      const int vv = i / cap, t = i - vv * cap;
      const int cc = c.Dsum + vv - pass * ncols_pass;
      if (cc >= 0 && cc < ncols_pass) {
        const int g = cc >> 5, l = cc & 31;
        float sum = 0.0f;
        for (int r = 0; r < R; ++r) sum = __fadd_rn(sum, s_sum[(((size_t)r * Gp + g) * cap + t) * 32 + l]);
        part_s2[i] = sum;
      }
    }
    if (pass == 0)
      for (int t = tid; t < cap; t += nthreads) {
        int n = 0;
        for (int r = 0; r < R; ++r) n += s_cnt[r * cap + t];
        c.partial_n[(size_t)blockIdx.x * cap + t] = n;
      }
    __syncthreads();
  }
}

cudaError_t launch_stats(const Ctx& c, bool delta, cudaStream_t s) {
  // the C3 shape has a register-accumulating, bulk-copy fed kernel (mv_stats_tile.cu); MVG_STATS_GENERIC=1
  // forces the general kernel below (used by the tests to check one against the other)
  const char* fg = getenv("MVG_STATS_GENERIC");
  const bool force_generic = fg && fg[0] == '1';
  if (stats_tile_supported(c) && (delta || !force_generic)) return launch_stats_tile(c, delta, s);
  if (delta) return cudaErrorInvalidValue;           // the caller asks stats_delta_supported first
  const StatsPlan pl = stats_plan(c);
  cudaError_t e = cudaFuncSetAttribute(k_stats, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem);
  if (e != cudaSuccess) return e;
  k_stats<<<c.stat_ctas, pl.R * pl.Gp * 32, pl.smem, s>>>(c, pl.Gp, pl.R, pl.passes);
  return cudaGetLastError();
}

// =============================================================================================
// k_finalize
// =============================================================================================
// Grid of V + 1 INDEPENDENT CTAs: CTA v < V owns view v (its dishes, tau_v, alpha_v, sigma_v, posterior means and
// parameter rows), CTA V owns the franchise level (customers per table, alpha_global, sigma_global, table masses, the
// sweep counter).  The integer bookkeeping every level needs (customers per table, the seating order of the births) is
// recomputed by every CTA from the same inputs, so that no CTA ever waits for another one's results: the levels of the
// hierarchy only meet in the parameter block of the next sweep.  The one hazard is the in-place update of what the
// others read at their start (n_t, the sweep counter): the franchise CTA publishes those last, after every CTA has
// announced that its reads are done (an arrival counter; all V + 1 CTAs are co-resident).
constexpr int kFinThreads = 1024;
constexpr int kMaxWorld = 16;
constexpr int kEppfSets = 4;             // (alpha, sigma) x (old, proposed): both Metropolis-Hastings steps of a level in one batch

// A set of the slots (tables, dishes) of one level, one bit per slot in W 64-bit words; members are visited in ascending
// order.
template <int W>
struct SlotSet {
  unsigned long long w[W];
  __device__ __forceinline__ void clear() {
#pragma unroll
    for (int i = 0; i < W; ++i) w[i] = 0ull;
  }
  __device__ __forceinline__ void set(int i) { w[i >> 6] |= 1ull << (i & 63); }
  __device__ __forceinline__ int lowest() const {   // -1 if empty
#pragma unroll
    for (int i = 0; i < W; ++i) if (w[i]) return 64 * i + __ffsll((long long)w[i]) - 1;
    return -1;
  }
  __device__ __forceinline__ int count() const {
    int n = 0;
#pragma unroll
    for (int i = 0; i < W; ++i) n += __popcll(w[i]);
    return n;
  }
  __device__ __forceinline__ int rank(int i) const {   // members below slot i
    int n = 0;
#pragma unroll
    for (int j = 0; j < W; ++j) {
      if (64 * j + 64 <= i) n += __popcll(w[j]);
      else if (64 * j < i) n += __popcll(w[j] & ((1ull << (i - 64 * j)) - 1ull));
    }
    return n;
  }
  __device__ __forceinline__ SlotSet without_lowest() const {
    SlotSet r = *this;
#pragma unroll
    for (int i = 0; i < W; ++i) if (r.w[i]) { r.w[i] &= r.w[i] - 1ull; break; }
    return r;
  }
  template <class F>
  __device__ __forceinline__ void for_each(F f) const {
#pragma unroll
    for (int i = 0; i < W; ++i)
      for (unsigned long long m = w[i]; m; m &= m - 1ull) f(64 * i + __ffsll((long long)m) - 1);
  }
};

// MAXCAP: the largest table capacity the instance serves (64: cap 32 / 64; 256: cap 128 / 256).
template <int MAXCAP>
struct FinShared {
  static constexpr int kMaxCap = MAXCAP;
  static constexpr int kWords = MAXCAP / 64;
  static constexpr int kBlocks = MAXCAP / 32;  // 32-cluster blocks of the batched EPPF
  int32_t n_new[kMaxCap];                 // customers per table after this sweep
  int32_t n_start[kMaxCap];               // ... at sweep start
  int32_t free_slots[kMaxCap];
  int32_t dish[kMaxCap];                  // working copy of dish_of[v]            (view CTAs)
  int32_t l_live[kMaxCap];                // tables per dish (live-updated by births, then recomputed)
  int32_t n_vk[kMaxCap];                  // customers per dish at sweep start, later the new ones
  int32_t cand_g[kMaxWorld * kMaxCap];    // candidates in global row order: shard, index in shard
  int32_t cand_j[kMaxWorld * kMaxCap];
  int32_t cand_final[kMaxWorld * kMaxCap];
  int32_t ncand_total, nseat, nfree, err;
  SlotSet<kWords> tmask[kMaxCap];         // bit t: table t serves dish k of this view (after births and deaths)
  SlotSet<kWords> live;                   // bit i: cluster i of this level has members (dishes: l_vk > 0; franchise: n_t > 0)
  long long total;                        // items of this level (tables of the view; customers for the franchise)
  double s2t[kMaxCap];                    // sums of squared norms per table (working copy of S2t[v])
  double s2k[kMaxCap];                    //   and per dish
  double s2k_start[kMaxCap];              // per dish at sweep START (count views: the token totals the births see)
  int32_t table_of_dish[kMaxCap];         // at sweep start: lowest table slot serving dish k, -1 = none
  double s1sq[kMaxCap];                   // |S1k|^2, later |m_t|^2
  double sse[kMaxCap];                    // max(0, S2k - |S1k|^2 / n_k)     (multiview_hyper.cpp:191-193)
  double termA[kEppfSets][kBlocks];       // scratch of the batched EPPF evaluations: per set, per 32-cluster block
  double termB[kEppfSets][kBlocks];
  double termC[kEppfSets][4];             // per set: lgamma(alpha + M), lgamma(alpha + 1), lgamma(1 - sigma)
  double eppf[kEppfSets];
  double s_alpha[kEppfSets], s_sigma[kEppfSets];
  double wbuf[kMaxCap + 1];
  double wexp[kMaxCap + 1];
  double result[4];
  double hyp[3];                          // view: alpha_v, sigma_v, tau_v; franchise: alpha_g, sigma_g
  double rn[3];                           // the sweep's standard normals of this level: [0] tau, [1] alpha, [2] sigma
  double lu[3];                           // log of its uniforms, same order
  double warm[2];                         // sink of the instruction-cache warm-up calls
};

template <int MAXCAP>
__host__ __device__ constexpr int fin_shared_bytes() { return (int)((sizeof(FinShared<MAXCAP>) + 15) & ~(size_t)15); }

// (The out-of-line helpers below take scalars and pointers, never `const Ctx&`: taking the address of the kernel
// parameter makes every thread copy the whole 1.5 KB struct into its local memory at kernel start.)
__device__ __noinline__ double dev_normal(uint64_t seed, uint32_t chain, uint32_t sweep, int idx) {
  const U4 r = stream_block(seed, chain, kDomHyperNormal, 0, sweep, (uint64_t)idx);
  const double u1 = uniform_f64_from(r.x, r.y), u2 = uniform_f64_from(r.z, r.w);
  return sqrt(-2.0 * fin_log(u1)) * cos(6.283185307179586476925286766559 * u2);
}
__device__ __noinline__ double dev_unif(uint64_t seed, uint32_t chain, uint32_t sweep, int idx) {
  const U4 r = stream_block(seed, chain, kDomHyperUnif, 0, sweep, (uint64_t)idx);
  return uniform_f64_from(r.x, r.y);
}

__device__ __forceinline__ double log_prior_alpha(double a) {       // multiview_hyper.cpp:344-351
  return (a <= 0.0) ? -INFINITY : (4.0 - 1.0) * fin_log(a) - 3.0 * a;
}
__device__ __forceinline__ double log_prior_sigma(double s) {       // :353-360
  return (s <= 0.0 || s >= 1.0) ? -INFINITY : (1.0 - 1.0) * fin_log(s) + (5.0 - 1.0) * fin_log(1.0 - s);
}
__device__ __forceinline__ double reflect_unit(double value) {      // :110-122
  double p = value;
  while (p <= kEps || p >= 1.0 - kEps) {
    if (p <= kEps) p = 2.0 * kEps - p;
    if (p >= 1.0 - kEps) p = 2.0 * (1.0 - kEps) - p;
  }
  return fmin(fmax(p, kEps), 1.0 - kEps);
}

__device__ __forceinline__ void group_sync(int bar_id, int gthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(gthreads) : "memory");
}

// log EPPF (multiview_hyper.cpp:53-83 franchise, :295-342 per view) of ONE level for kEppfSets parameter sets
// (S.s_alpha[q], S.s_sigma[q]).  `counts` are the cluster sizes of the level (tables per dish l_vk; customers per table
// n_t), S.live its live mask, S.total its item count.  The two inner loops are taken in closed form,
//   sum_{i=1}^{M-1} log(alpha+i) = lgamma(alpha+M) - lgamma(alpha+1),
//   sum_{m=1}^{c-1} log(m-sigma) = lgamma(c-sigma) - lgamma(1-sigma),
// the per-cluster terms are evaluated in parallel (one warp per (set, 32-cluster block), fixed shuffle tree) and one
// thread per set adds the blocks in ascending order (the order of oracle/mv_oracle.c:eppf_core).
// Called by ONE group of gthreads consecutive threads (gtid = index inside the group) synchronising on named barrier
// bar_id; the rest of the CTA is busy with the dish statistics and the posterior means meanwhile.
template <class FS>
__device__ __noinline__ void eppf_batch(const int cap, const int32_t* counts, FS& S, const int gtid, const int gthreads,
                                        const int bar_id) {
  const int lane = gtid & 31, wid = gtid >> 5;
  group_sync(bar_id, gthreads);
  const int wps = (cap + 31) / 32;                   // warps per set
  for (int base = 0; base < kEppfSets * wps; base += gthreads / 32) {
    const int unit = base + wid;                     // (set, 32-cluster block)
    double sa = 0.0, sb = 0.0;
    bool bad = false;
    if (unit < kEppfSets * wps) {
      const int set = unit / wps, i = (unit - set * wps) * 32 + lane;
      if (i < cap) {
        const double al = S.s_alpha[set], sg = S.s_sigma[set];
        const int cnt = counts[i];
        if (cnt > 0) {
          const int r = S.live.rank(i);
          const double term = al + (double)r * sg;
          if (term <= 0.0) bad = true; else sa = fin_log(term);
        }
        if (cnt > 1) sb = fin_lgamma((double)cnt - sg);   // minus lgamma(1 - sigma) per such cluster: added below
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      sa += __shfl_xor_sync(0xffffffffu, sa, o);
      sb += __shfl_xor_sync(0xffffffffu, sb, o);
    }
    bad = __any_sync(0xffffffffu, bad);
    if (unit < kEppfSets * wps && lane == 0) {
      const int set = unit / wps, blk = unit - set * wps;
      S.termA[set][blk] = bad ? -INFINITY : sa;
      S.termB[set][blk] = sb;
    }
  }
  // the three per-set lgamma values, one thread each (the last warps: the first ones carry the units above)
  for (int q = gtid - (gthreads - 128); q >= 0 && q < 3 * kEppfSets; q += gthreads) {
    const int set = q / 3, which = q - 3 * set;
    const double al = S.s_alpha[set], sg = S.s_sigma[set];
    double val = 0.0;
    if ((sg > kEps && sg < 1.0 - kEps) && al > -sg)
      val = (which == 0) ? fin_lgamma(al + (double)S.total) : ((which == 1) ? fin_lgamma(al + 1.0) : fin_lgamma(1.0 - sg));
    S.termC[set][which] = val;
  }
  group_sync(bar_id, gthreads);
  if (gtid < kEppfSets) {
    const int set = gtid;
    const double al = S.s_alpha[set], sg = S.s_sigma[set];
    const long long total = S.total;
    double logp;
    if (!(sg > kEps && sg < 1.0 - kEps) || al <= -sg) logp = -INFINITY;
    else if (total <= 0) logp = 0.0;
    else {
      int multi = 0;
      for (int i = 0; i < cap; ++i) multi += counts[i] > 1;
      double sa = 0.0, sb = 0.0;
      for (int w = 0; w < wps; ++w) { sa += S.termA[set][w]; sb += S.termB[set][w]; }
      logp = sa;
      if (total > 1) logp -= S.termC[set][0] - S.termC[set][1];
      logp += sb - (double)multi * S.termC[set][2];
    }
    S.eppf[set] = logp;
  }
  group_sync(bar_id, gthreads);
}

// The (alpha, sigma) Metropolis-Hastings pair of one level (multiview_hyper.cpp:239-291) on S.hyp[0..1], with the
// level's Philox numbers S.rn[1..2] / S.lu[1..2].  The sigma step needs the EPPF at the alpha the first step ends with:
// both candidates are evaluated up front — sets (a_old, s_old), (a_prop, s_old), (a_cur, s_prop), (a_prop, s_prop) in
// ONE batch — so the two dependent steps cost one round of lgamma latencies instead of two.  Each EPPF value is the
// same function of (alpha, sigma, counts) as in the sequential order, so the chain is unchanged.
template <class FS>
__device__ __forceinline__ void level_alpha_sigma(const int cap, const int32_t* counts, FS& S, const int gtid,
                                                  const int gthreads, const int bar_id, const bool enabled) {
  double a_cur = 0.0, a_old = 0.0, a_prop = 0.0, s_old = 0.0, s_prop = 0.0;
  if (gtid == 0 && enabled) {
    a_cur = S.hyp[0];
    a_old = a_cur;
    if (a_old <= 0.0) a_old = kEps;
    const double cand = fin_exp(fin_log(a_old > kEps ? a_old : kEps) + 0.0 + 0.1 * S.rn[1]);   // :100-108
    a_prop = cand > kEps ? cand : kEps;
    s_old = S.hyp[1];
    s_prop = reflect_unit(s_old + 0.0 + 0.05 * S.rn[2]);                                       // :124-128
    S.s_alpha[0] = a_old;  S.s_sigma[0] = s_old;
    S.s_alpha[1] = a_prop; S.s_sigma[1] = s_old;
    S.s_alpha[2] = a_cur;  S.s_sigma[2] = s_prop;
    S.s_alpha[3] = a_prop; S.s_sigma[3] = s_prop;
  }
  if (!enabled) return;                                                      // (group-uniform)
  eppf_batch(cap, counts, S, gtid, gthreads, bar_id);
  if (gtid == 0) {
    // alpha: log-normal random walk, :242-255 / :268-281
    const double lo = S.eppf[0] + log_prior_alpha(a_old), ln = S.eppf[1] + log_prior_alpha(a_prop);
    const double log_acc = (ln - lo) + (fin_log(a_prop) - fin_log(a_old));
    const bool acc_a = S.lu[1] < log_acc;
    if (acc_a) S.hyp[0] = a_prop;
    // sigma: reflected random walk at the alpha just fixed, :257-265 / :283-291
    // (not accepted: alpha stays a_cur; set 0 was evaluated at a_old, which differs from a_cur only for alpha <= 0,
    //  a state mvg_set_state rejects)
    const double e_old = acc_a ? S.eppf[1] : ((a_cur == a_old) ? S.eppf[0] : S.eppf[0]);
    const double e_new = acc_a ? S.eppf[3] : S.eppf[2];
    const double lpo = (s_old <= kEps || s_old >= 1.0 - kEps) ? -INFINITY : e_old + log_prior_sigma(s_old);
    const double lpn = (s_prop <= kEps || s_prop >= 1.0 - kEps) ? -INFINITY : e_new + log_prior_sigma(s_prop);
    if (S.lu[2] < lpn - lpo) S.hyp[1] = s_prop;
  }
}

// log predictive density of x (FP32, the coordinates of ONE view) under dish k of that view, optionally with
// x removed from the dish first (multiview_utils.cpp:307-338 in closed form, per coordinate).
__device__ __noinline__ double log_f_dish(const int D, const double* __restrict__ S1, const double n_vk, const float* x,
                                          bool loo, double tau) {
  const double n = n_vk - (loo ? 1.0 : 0.0);
  const double var = tau * (tau + n + 1.0) / (tau + n);
  double dist = 0.0;
  for (int dd = 0; dd < D; ++dd) {
    const double xv = (double)x[dd];
    const double s1 = S1[dd] - (loo ? xv : 0.0);
    const double diff = xv - s1 / (tau + n);
    dist += diff * diff;
  }
  return -0.5 * (double)D * fin_log(2.0 * kPi * var) - 0.5 * dist / var;
}

// Count view: log f of local ROW `row` under dish k from the sweep-start dish counts (cnt_d is indexed by TABLE
// slot: tk is any table serving dish k, or -1 for a dish without tables = empty), FP64
// (oracle/mv_oracle.c:counts_log_f_vk).
__device__ __noinline__ double log_f_dish_counts(const int32_t* __restrict__ rp, const int32_t* __restrict__ col,
                                                 const float* __restrict__ val, const int32_t* __restrict__ cnt_d,
                                                 const int cap, const double wbeta, const double beta, const double ctot_k,
                                                 const int tk, const int row, const bool loo) {
  double tot = 0.0;
  for (int j = rp[row]; j < rp[row + 1]; ++j) tot += (double)val[j];
  const double den = wbeta + ((tk >= 0) ? ctot_k : 0.0) - (loo ? tot : 0.0);
  double lf = 0.0;
  for (int j = rp[row]; j < rp[row + 1]; ++j) {
    const double x = (double)val[j];
    const double cd = (tk >= 0) ? (double)cnt_d[(size_t)col[j] * cap + tk] : 0.0;
    lf += x * fin_log((beta + cd - (loo ? x : 0.0)) / den);
  }
  return lf;
}

// The same under MVG_COUNT_DIRMULT (oracle/mv_oracle_dm.c:mvod_counts_log_f_vk): the collapsed Dirichlet-multinomial
// conditional, sum_w [lnΓ(beta + c + x_w) - lnΓ(beta + c)] - [lnΓ(W beta + C + n) - lnΓ(W beta + C)], by lgamma_diff
// (mv_device.cuh): at most ~2 kLgdLoop logs per nonzero and for the denominator, however long the row.
// tk = -1 (a dish without tables, or a new dish): c = C = 0.
__device__ __noinline__ double log_f_dish_counts_dm(const int32_t* __restrict__ rp, const int32_t* __restrict__ col,
                                                    const float* __restrict__ val, const int32_t* __restrict__ cnt_d,
                                                    const int cap, const double wbeta, const double beta, const double ctot_k,
                                                    const int tk, const int row, const bool loo) {
  int n = 0;
  double lf = 0.0;
  for (int j = rp[row]; j < rp[row + 1]; ++j) {
    const int x = (int)val[j];
    const int cd = (tk >= 0) ? cnt_d[(size_t)col[j] * cap + tk] - (loo ? x : 0) : 0;
    lf += lgamma_diff(beta + (double)cd, x);
    n += x;
  }
  const double den = wbeta + ((tk >= 0) ? ctot_k - (loo ? (double)n : 0.0) : 0.0);
  return lf - lgamma_diff(den, n);
}

// B1 of k_finalize for a count view: log f of the candidate's ROW under dish k (tk, ctot_k as above) or a new dish, by the
// handle's count model.  mode: bit 0 leave-one-out, bit 1 new dish, bit 2 Dirichlet-multinomial.  One out-of-line call with
// few arguments keeps the finalize kernel's register budget.
__device__ __noinline__ double birth_log_f_counts(const int32_t* __restrict__ rp, const int32_t* __restrict__ col,
                                                  const float* __restrict__ val, const int32_t* __restrict__ cnt_d,
                                                  const int cap, const int vocab, const double beta, const double ctot_k,
                                                  const int tk, const int row, const int mode) {
  const bool loo = (mode & 1) != 0, new_dish = (mode & 2) != 0, dm = (mode & 4) != 0;
  const double wbeta = (double)vocab * beta;
  if (dm) return log_f_dish_counts_dm(rp, col, val, cnt_d, cap, wbeta, beta, ctot_k, new_dish ? -1 : tk, row, loo && !new_dish);
  if (new_dish) {                    // plug-in: log f_new = -|x| log W
    double tot = 0.0;
    for (int j = rp[row]; j < rp[row + 1]; ++j) tot += (double)val[j];
    return -tot * fin_log((double)vocab);
  }
  return log_f_dish_counts(rp, col, val, cnt_d, cap, wbeta, beta, ctot_k, tk, row, loo);
}

// The Philox numbers of one level's hyper step, by the calling warp's lanes 0..5: rn/lu[which], which = 0 tau, 1 alpha,
// 2 sigma.  Stream positions are those the reference's sequential code would use: tau_v at v, (alpha_v, sigma_v) at
// V + 2v, the franchise pair at 3V.  `first`..`last`: the range of `which` this call draws.
template <class FS>
__device__ __forceinline__ void draw_level_randoms(FS& S, uint64_t seed, uint32_t chain, uint32_t sweep, int V, int v,
                                                   bool is_view, int first, int last, int lane) {
  const int which = first + (lane >> 1);
  if (which > last || lane >= 2 * (last - first + 1)) return;
  const int idx = (which == 0) ? v : ((is_view ? V + 2 * v : 3 * V) + which - 1);
  if (lane & 1) S.lu[which] = fin_log(dev_unif(seed, chain, sweep, idx));
  else S.rn[which] = dev_normal(seed, chain, sweep, idx);
}

template <int MAXCAP>
__global__ void __launch_bounds__(kFinThreads, 1) k_finalize(const Ctx c, const int32_t flags, const int32_t s1_in_smem,
                                                           const int32_t ref_in_smem) {
  extern __shared__ __align__(16) unsigned char fin_smem[];
  using FS = FinShared<MAXCAP>;
  using Set = SlotSet<FS::kWords>;
  FS& S = *reinterpret_cast<FS*>(fin_smem);
  // Programmatic dependent launch: the next sweep's draw kernel may be scheduled now (its CTAs set themselves up and
  // start streaming features on the idle SMs; they wait for this grid's completion before they touch its results).
  pdl_trigger();
  const int tid = threadIdx.x;
  const int cap = c.cap, V = c.V;
  const int role = blockIdx.x;                      // < V: that view; V: the franchise level
  const bool is_view = role < V;
  const int v = is_view ? role : 0;
  const int D = is_view ? c.D[v] : 0;
  const int doff = is_view ? c.doff[v] : 0;
  const bool is_count = is_view && c.kind[v] != 0;
  // A failed exchange (a peer's packet never arrived) freezes the chain: nothing is published, the sweep counter stays
  // (mvg_sweep / mvg_sync report it; csrc/mv_exchange.cu).
  // The per-table sums of this view, S1t [cap][D], live in shared memory behind FinShared when they fit (32 KB at C3):
  // the dish statistics and the posterior means are then built from on-chip data instead of global round trips.
  double* const S1t = s1_in_smem ? reinterpret_cast<double*>(fin_smem + fin_shared_bytes<MAXCAP>()) : (c.S1t + (size_t)cap * doff);
  // Draw screening's reference of this view (scaled means hi, lo [cap][D], then the parameter block [cap]), which the drift
  // sums of E1 read, follows in shared memory when it fits (32 KB at C3); otherwise E1 reads it from global memory.
  auto ref_smem = [&]() {
    return reinterpret_cast<float*>(fin_smem + fin_shared_bytes<MAXCAP>() + (s1_in_smem ? sizeof(double) * (size_t)cap * D : 0));
  };
  const uint32_t sweep = *reinterpret_cast<volatile uint32_t*>(c.sweep);
  double& alpha_l = S.hyp[0];                       // alpha_v / alpha_global
  double& sigma_l = S.hyp[1];                       // sigma_v / sigma_global
  double& tau_l = S.hyp[2];                         // tau_v (views only)

  const bool prof = (c.debug_export & 2) != 0 && c.dbg_prof != nullptr && tid == 0;
  long long* pout = c.dbg_prof + (200 + role) * 16;   // slots 200.. of the profile buffer: one row of stamps per CTA
  const long long t_begin = prof ? clock64() : 0;
  auto stamp = [&](int k) { if (prof) pout[k] = clock64() - t_begin; };
  if (tid == 0) { S.err = 0; S.ncand_total = 0; S.nseat = 0; S.nfree = 0; }
  if (tid == 32) {
    S.hyp[0] = is_view ? c.hyp[v] : c.hyp[3 * V];
    S.hyp[1] = is_view ? c.hyp[V + v] : c.hyp[3 * V + 1];
    S.hyp[2] = is_view ? c.hyp[2 * V + v] : 0.0;
  }
  // (The random numbers of the hyper step depend on nothing but (seed, sweep, index): they are drawn by otherwise idle
  //  warps right before the chains that use them — see draw_level_randoms — and never hold up a CTA-wide barrier.)

  // ---- A. this level's inputs: the sweep-start state (the previous finalize's, complete long ago: read while the
  //         statistics kernels of this sweep are still running — the launch is a programmatic dependent, mv_ctx.h) ... ----
  for (int t = tid; t < cap; t += kFinThreads) S.n_start[t] = c.n_t[t];
  if (is_view) {
    for (int t = tid; t < cap; t += kFinThreads) {
      S.dish[t] = c.dish_of[v * cap + t];
      S.l_live[t] = c.l_vk[v * cap + t];
      S.n_vk[t] = c.n_vk[v * cap + t];
    }
  }
  // ---- ... and, behind the grid dependency, the statistics summed over the shards (k_reduce_x) ----
  pdl_wait();
  // A failed exchange (a peer's packet never arrived) freezes the chain: nothing is published, the sweep counter stays
  // (mvg_sweep / mvg_sync report it; csrc/mv_exchange.cu).
  if (*reinterpret_cast<volatile int32_t*>(c.status + 1) != 0) return;
  if (tid == 0) kclock_begin(c.kclock + kClockFinalize);
  for (int t = tid; t < cap; t += kFinThreads) S.n_new[t] = c.sum_cnt[t];
  if (is_view) {
    if (s1_in_smem) {
      const double* src = c.sum_s1t + (size_t)cap * doff;
      const int n_s1 = cap * D;
      for (int i = tid; i < n_s1; i += kFinThreads) S1t[i] = src[i];
    }
    for (int t = tid; t < cap; t += kFinThreads) S.s2t[t] = c.sum_s2t[v * cap + t];
    if (ref_in_smem) {                              // after the wait: a refresh draw of this sweep wrote the reference
      const float* src = c.scr_b + (size_t)cap * doff;
      float* dst = ref_smem();
      const size_t half = (size_t)cap * c.Dsum;
      for (int i = tid; i < cap * D; i += kFinThreads) { dst[i] = src[i]; dst[cap * D + i] = src[half + i]; }
      TableParam* tp = reinterpret_cast<TableParam*>(dst + 2 * (size_t)cap * D);
      for (int t = tid; t < cap; t += kFinThreads) tp[t] = c.scr_tp[v * cap + t];
    }
  }
  __syncthreads();
  if (is_view && !s1_in_smem) {                     // large views: the sums stay in global memory (own block of S1t)
    const double* src = c.sum_s1t + (size_t)cap * doff;
    const int n_s1 = cap * D;
    for (int i = tid; i < n_s1; i += kFinThreads) S1t[i] = src[i];
  }
  if (is_count) {
    for (int k = tid; k < cap; k += kFinThreads) {
      S.s2k_start[k] = c.S2k[v * cap + k];
      int tk = -1;
      for (int t = cap - 1; t >= 0; --t) if (S.dish[t] == k && S.n_start[t] > 0) tk = t;
      S.table_of_dish[k] = tk;
    }
  }
  __syncthreads();
  // every read of what the franchise CTA updates in place is done: announce it
  if (tid == 0) { __threadfence(); atomicAdd(c.fin_arrive, 1u); }

  stamp(0);
  // ---- B. births: candidates in global row order, the first nfree are seated -----------------
  if (flags & kFinReseat) {
    if (tid == 0) {                       // usually no customer drew a new table: then the whole section is skipped
      int n = 0;
      for (int g = 0; g < c.world; ++g) n += pkt_i32(c, g, c.pkt.off_hdr)[0];
      S.ncand_total = n;
      if (n == 0 && c.debug_export && !is_view) *c.dbg_nseated = 0;
    }
    __syncthreads();
  }
  if ((flags & kFinReseat) && S.ncand_total > 0) {
    if (tid == 0) {
      int nf = 0;
      for (int t = 0; t < cap; ++t) if (S.n_start[t] <= 0) S.free_slots[nf++] = t;
      S.nfree = nf;
      int n = 0;
      for (int g = 0; g < c.world; ++g) {
        const int nc = pkt_i32(c, g, c.pkt.off_hdr)[0];
        for (int j = 0; j < nc && n < kMaxWorld * MAXCAP; ++j) { S.cand_g[n] = g; S.cand_j[n] = j; ++n; }
      }
      S.ncand_total = n;
      S.nseat = n < nf ? n : nf;
      if (c.debug_export && !is_view) *c.dbg_nseated = S.nseat;
    }
    __syncthreads();
    const int nseat = S.nseat, ncand = S.ncand_total;
    if (is_view) {
      // B1. log f of every seated candidate under every dish slot of this view (and a new dish), in parallel
      for (int idx = tid; idx < nseat * (cap + 1); idx += kFinThreads) {
        const int b = idx / (cap + 1), k = idx - b * (cap + 1);
        const float* x = pkt_f32(c, S.cand_g[b], c.pkt.off_cand_x) + (size_t)S.cand_j[b] * c.Dsum + doff;
        double val;
        if (is_count) {  // count view (one GPU per chain: the candidate's row is local)
          const int row = pkt_i32(c, S.cand_g[b], c.pkt.off_cand_row)[S.cand_j[b]];
          const int t0 = pkt_i32(c, S.cand_g[b], c.pkt.off_cand_t0)[S.cand_j[b]];
          const bool own = (k < cap) && (k == S.dish[t0]) && S.n_vk[k] > 0;
          val = birth_log_f_counts(c.rowptr[v], c.col[v], c.val[v], c.cnt_d[v], cap, c.vocab[v], c.beta_v[v],
                                   (k < cap) ? S.s2k_start[k] : 0.0, (k < cap) ? S.table_of_dish[k] : -1, row,
                                   (own ? 1 : 0) | (k == cap ? 2 : 0) | (c.count_model ? 4 : 0));
        } else if (k == cap) {   // new dish: N(x; 0, tau)   (multiview_utils.cpp:340-350)
          double q = 0.0;
          for (int dd = 0; dd < D; ++dd) q += (double)x[dd] * (double)x[dd];
          val = -0.5 * (double)D * fin_log(2.0 * kPi * tau_l) - 0.5 * q / tau_l;
        } else {
          const int t0 = pkt_i32(c, S.cand_g[b], c.pkt.off_cand_t0)[S.cand_j[b]];
          val = log_f_dish(D, c.S1k + (size_t)cap * doff + (size_t)k * D, (double)S.n_vk[k], x,
                           (k == S.dish[t0]) && S.n_vk[k] > 0, tau_l);
        }
        c.birth_lf[((size_t)b * V + v) * (cap + 1) + k] = val;
      }
      __syncthreads();
      // B2. seating in order; sample_dish_for_new_table (multiview_utils.cpp:224-276) for this view
      for (int b = 0; b < nseat; ++b) {
        const int g = S.cand_g[b], j = S.cand_j[b];
        const int t0 = pkt_i32(c, g, c.pkt.off_cand_t0)[j];
        const int64_t grow = *reinterpret_cast<const int64_t*>(pkt_i32(c, g, c.pkt.off_hdr) + 4) +
                             (int64_t)pkt_i32(c, g, c.pkt.off_cand_row)[j];
        const int tn = S.free_slots[b];
        const bool single = (S.n_start[t0] == 1);
        const int k0 = S.dish[t0];
        const double* lf = c.birth_lf + ((size_t)b * V + v) * (cap + 1);
        if (tid <= cap) {
          double lw = -INFINITY;
          if (tid < cap) {
            const int l = S.l_live[tid] - ((single && tid == k0) ? 1 : 0);
            const double w = (double)l - sigma_l;                            // :232-233
            if (l > 0 && w > 0.0) lw = fin_log(w) + lf[tid];
          } else {
            int K_act = 0;
            for (int k = 0; k < cap; ++k) K_act += (S.l_live[k] - ((single && k == k0) ? 1 : 0)) > 0;
            const double wn = alpha_l + sigma_l * (double)K_act;             // :241-243
            if (wn > 0.0) lw = fin_log(wn) + lf[cap];
          }
          S.wbuf[tid] = lw;
        }
        __syncthreads();
        if (tid == 0) {
          double M = -INFINITY;
          for (int k = 0; k <= cap; ++k) M = fmax(M, S.wbuf[k]);
          S.result[0] = M;
        }
        __syncthreads();
        if (tid <= cap) {
          const double M = S.result[0], lw = S.wbuf[tid];
          const double w = (M > -INFINITY && lw > -INFINITY) ? fin_exp(lw - M) : 0.0;
          S.wexp[tid] = w;
          if (c.debug_export) c.dbg_birth_w[((size_t)b * V + v) * (cap + 1) + tid] = w;
        }
        __syncthreads();
        if (tid == 0) {
          int pick = -1;
          if (S.result[0] > -INFINITY) {
            double total = 0.0;
            for (int k = 0; k <= cap; ++k) total += S.wexp[k];               // :247-248
            const U4 r = stream_block(c.seed, c.chain, kDomDish, (uint32_t)v, sweep, (uint64_t)grow);
            const double u = uniform_f64_from(r.x, r.y) * total;             // :261
            double cum = 0.0;
            for (int k = 0; k < cap; ++k) {
              if (!(S.wbuf[k] > -INFINITY)) continue;
              cum += S.wexp[k];
              if (u < cum) { pick = k; break; }
            }
          }
          if (pick < 0) {                                                     // new dish: lowest free slot
            for (int k = 0; k < cap; ++k) if (S.l_live[k] == 0) { pick = k; break; }
          }
          if (pick < 0) { S.err |= 1; pick = 0; }
          S.dish[tn] = pick;
          S.l_live[pick] += 1;                                                // :283
        }
        __syncthreads();
      }
    }
    // the seat every candidate ends at: a function of the candidate order and the free slots alone (every CTA's copy)
    for (int b = tid; b < ncand; b += kFinThreads)
      S.cand_final[b] = (b < nseat) ? S.free_slots[b] : pkt_i32(c, S.cand_g[b], c.pkt.off_cand_t0)[S.cand_j[b]];   // overflow: stay put
    __syncthreads();
    // B3. candidates join the statistics of their final table, in global row order
    if (tid == 0) for (int b = 0; b < ncand; ++b) S.n_new[S.cand_final[b]] += 1;
    // (This shard's own candidates also join its RUNNING statistics — the sums in its packet that the incremental mode
    //  carries from sweep to sweep; a full rebuild overwrites them.)
    if (!is_view) {
      if (tid == 32) {
        for (int b = 0; b < ncand; ++b)
          if (S.cand_g[b] == c.rank) {
            c.table_cur[pkt_i32(c, c.rank, c.pkt.off_cand_row)[S.cand_j[b]]] = S.cand_final[b];
            pkt_i32(c, c.rank, c.pkt.off_cnt)[S.cand_final[b]] += 1;
          }
      }
      if (tid == 64 && c.debug_export)
        for (int b = 0; b < nseat; ++b)
          c.dbg_birth_rows[b] = *reinterpret_cast<const int64_t*>(pkt_i32(c, S.cand_g[b], c.pkt.off_hdr) + 4) +
                                (int64_t)pkt_i32(c, S.cand_g[b], c.pkt.off_cand_row)[S.cand_j[b]];
    } else {
      if (tid == 64) {
        for (int b = 0; b < ncand; ++b) {
          const float* x = pkt_f32(c, S.cand_g[b], c.pkt.off_cand_x) + (size_t)S.cand_j[b] * c.Dsum + doff;
          double q = 0.0;
          for (int dd = 0; dd < D; ++dd) q += (double)x[dd] * (double)x[dd];
          if (is_count)      // count view: this slot carries token totals; the candidate's row is local (world = 1)
            q = (double)c.xx[(size_t)v * c.xx_stride + pkt_i32(c, S.cand_g[b], c.pkt.off_cand_row)[S.cand_j[b]]];
          S.s2t[S.cand_final[b]] += q;
          if (S.cand_g[b] == c.rank) pkt_f64(c, c.rank, c.pkt.off_s2t)[v * cap + S.cand_final[b]] += q;
        }
      }
      for (int dd = tid; dd < D; dd += kFinThreads) {
        double* loc = pkt_f64(c, c.rank, c.pkt.off_s1t) + (size_t)cap * doff;
        for (int b = 0; b < ncand; ++b) {
          const float xv = pkt_f32(c, S.cand_g[b], c.pkt.off_cand_x)[(size_t)S.cand_j[b] * c.Dsum + doff + dd];
          S1t[(size_t)S.cand_final[b] * D + dd] += (double)xv;
          if (S.cand_g[b] == c.rank) loc[(size_t)S.cand_final[b] * D + dd] += (double)xv;
        }
      }
    }
    __syncthreads();
  }

  stamp(1);
  constexpr int kGroupThreads = kFinThreads / 2;
  if (!is_view) {
    // =============================== the franchise level ===============================
    if (tid == kFinThreads - 32) {                               // every customer must have been counted exactly once
      long long tot = 0;
      for (int t = 0; t < cap; ++t) tot += S.n_new[t];
      if (tot != (long long)c.n_global) atomicOr(&S.err, 4);
    }
    if (tid == 0) {
      Set m;
      m.clear();
      for (int i = 0; i < cap; ++i) if (S.n_new[i] > 0) m.set(i);
      S.live = m;
      S.total = (long long)c.n_global;
    }
    if (flags & kFinTauInit) { if (tid == 0) { alpha_l = 1.0; sigma_l = 0.6; } }      // multiview_gibbs.cpp:97-98
    if ((flags & kFinHyper) && tid >= 32 && tid < 64) draw_level_randoms(S, c.seed, c.chain, sweep, V, v, false, 1, 2, tid - 32);
    __syncthreads();
    // (alpha_global, sigma_global), multiview_hyper.cpp:268-291, by the first half of the CTA
    if (tid < kGroupThreads)
      level_alpha_sigma(cap, S.n_new, S, tid, kGroupThreads, 1, (flags & kFinHyper) && (flags & kFinHyperGlobal));
    __syncthreads();
    stamp(2);
    // publish: only after every CTA has read the sweep-start values this overwrites
    if (tid == 0) {
      while (*reinterpret_cast<volatile uint32_t*>(c.fin_arrive) < (uint32_t)(V + 1)) { }
      __threadfence();
    }
    __syncthreads();
    for (int t = tid; t < cap; t += kFinThreads) {
      c.n_t[t] = S.n_new[t];
      const double mass = (double)S.n_new[t] - sigma_l, mass1 = mass - 1.0;
      TableMass tm;
      tm.LM = (S.n_new[t] > 0 && mass > 0.0) ? (float)fin_log2(mass) : kMasked;
      tm.LM1 = (S.n_new[t] > 1 && mass1 > 0.0) ? (float)fin_log2(mass1) : kMasked;
      tm.single = (S.n_new[t] == 1);
      tm.pad = 0;
      c.tmass[t] = tm;
    }
    if (tid == 15 * 32) {
      c.hyp[3 * V] = alpha_l;
      c.hyp[3 * V + 1] = sigma_l;
      int T_ne = 0;
      for (int t = 0; t < cap; ++t) T_ne += S.n_new[t] > 0;
      const int F = cap - T_ne;
      const double mn0 = alpha_l + sigma_l * (double)T_ne, mn1 = alpha_l + sigma_l * (double)(T_ne - 1);
      GlobalParam g;
      g.LMN0 = (F > 0 && mn0 > 0.0) ? (float)fin_log2(mn0) : kMasked;
      g.LMN1 = (F > 0 && mn1 > 0.0) ? (float)fin_log2(mn1) : kMasked;
      g.nfree = F;
      const uint32_t next = sweep + ((flags & kFinAdvance) ? 1u : 0u);
      g.sweep = next;
      *c.gparam = g;
      *c.sweep = next;
      *c.fin_arrive = 0u;                                        // ready for the next launch
      if (c.world > 1) *c.xseq += 1u;                            // one exchange precedes every finalize (mv_exchange.cu)
      if (S.err) atomicOr(c.status, S.err);
    }
    stamp(5);
    __syncthreads();
    if (tid == 0) kclock_end(c.kclock + kClockFinalize, gridDim.x);
    return;
  }

  // =============================== a view ===============================
  // ---- C. deaths and per-dish statistics -------------------------------------------------------
  for (int t = tid; t < cap; t += kFinThreads) {
    if (S.n_new[t] == 0) S.dish[t] = -1;                     // multiview_utils.cpp:168-191
    else if (S.dish[t] < 0 || S.dish[t] >= cap) { S.err |= 2; S.dish[t] = 0; }
  }
  // An empty table has exactly zero statistics: clear what incremental updates may have left of its sums (rounding
  // residue of the rows that came and went) in the totals and in this shard's running sums.
  for (int i = tid; i < cap * D; i += kFinThreads) {
    const int t = i / D;
    if (S.n_new[t] == 0) { S1t[i] = 0.0; pkt_f64(c, c.rank, c.pkt.off_s1t)[(size_t)cap * doff + i] = 0.0; }
  }
  for (int t = tid; t < cap; t += kFinThreads)
    if (S.n_new[t] == 0) { S.s2t[t] = 0.0; pkt_f64(c, c.rank, c.pkt.off_s2t)[v * cap + t] = 0.0; }
  __syncthreads();
  {
    // one warp per dish k: which tables serve it (ballots over the table slots), how many customers they hold
    const int lane = tid & 31, wid = tid >> 5;
    for (int k = wid; k < cap; k += kFinThreads / 32) {
      Set m;
      m.clear();
      int n = 0;
      double s2 = 0.0;
      for (int base = 0; base < cap; base += 32) {
        const int t = base + lane;
        const bool mine = (t < cap) && (S.dish[t] == k);
        m.w[base >> 6] |= (unsigned long long)__ballot_sync(0xffffffffu, mine) << (base & 63);
      }
      if (lane == 0) {
        m.for_each([&](int t) {                                      // ascending table order (usually one table)
          n += S.n_new[t];
          s2 += S.s2t[t];
        });
        const int l = m.count();
        S.l_live[k] = l;
        S.n_vk[k] = n;
        S.s2k[k] = s2;
        S.tmask[k] = m;
        const int i = v * cap + k;
        c.S2k[i] = s2;
        c.S2t[i] = S.s2t[k];                                  // (index reuse: slot k as a table)
        c.l_vk[i] = l;
        c.n_vk[i] = n;
        c.dish_of[i] = S.dish[k];
      }
    }
  }
  __syncthreads();
  stamp(7);
  // From here the CTA works as two halves that meet again before the parameter block:
  //   upper half (named barrier 1): the (alpha_v, sigma_v) Metropolis-Hastings pair — it only needs the COUNTS fixed
  //     above (tables per dish);
  //   lower half (named barrier 2): per-dish statistics -> tau_v step (needs their sums of squares) -> posterior means
  //     (need the new tau_v).
  // Two independent FP64 latency chains of similar length: side by side they cost the longer one.
  if (tid >= kGroupThreads) {
    const int gtid = tid - kGroupThreads;
    if (gtid == 0) {                            // live mask and item total of this level
      Set m;
      m.clear();
      long long tot = 0;
      for (int i = 0; i < cap; ++i) { if (S.l_live[i] > 0) m.set(i); tot += S.l_live[i]; }
      S.live = m;
      S.total = tot;
    }
    if ((flags & kFinHyper) && gtid >= 32 && gtid < 64) draw_level_randoms(S, c.seed, c.chain, sweep, V, v, true, 1, 2, gtid - 32);
    group_sync(1, kGroupThreads);
    if (!(flags & kFinTauInit))                 // (the reference's initial values are set by the lower half below)
      level_alpha_sigma(cap, S.l_live, S, gtid, kGroupThreads, 1, (flags & kFinHyper) && (flags & kFinHyperLocal));
    if ((c.debug_export & 2) != 0 && c.dbg_prof != nullptr && gtid == 0) pout[13] = clock64() - t_begin;   // upper half done
  } else {
    {
      // one warp per dish k: lanes stride over the coordinates; the tables serving the dish are added in
      // ascending order (warp-uniform loop), then |S1k|^2 by a fixed shuffle tree.  The last warp of this half draws the
      // tau step's Philox numbers meanwhile.
      const int lane = tid & 31, wid = tid >> 5;
      constexpr int kStatWarps = kGroupThreads / 32 - 1;
      if (wid == kStatWarps) {
        if (flags & kFinHyper) draw_level_randoms(S, c.seed, c.chain, sweep, V, v, true, 0, 0, lane);
      } else {
        for (int k = wid; k < cap; k += kStatWarps) {
          double* S1k_vk = c.S1k + (size_t)cap * doff + (size_t)k * D;
          const Set mask = S.tmask[k];
          const int t1 = mask.lowest();                              // usually the only table of the dish
          const Set more = mask.without_lowest();
          double q = 0.0;
          for (int dd = lane; dd < D; dd += 32) {
            double sum = (t1 >= 0) ? S1t[t1 * D + dd] : 0.0;
            more.for_each([&](int t) { sum += S1t[t * D + dd]; });
            S1k_vk[dd] = sum;
            q += sum * sum;
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
          if (lane == 0) S.s1sq[k] = q;
        }
      }
    }
    group_sync(2, kGroupThreads);
    // sums of squared errors, one thread per dish (the FP64 divisions side by side instead of one per warp step)
    if (tid < cap) {
      const int n_k = S.n_vk[tid];
      const double sse = (n_k > 0) ? S.s2k[tid] - S.s1sq[tid] / (double)n_k : 0.0;
      S.sse[tid] = sse < 0.0 ? 0.0 : sse;
    }
    group_sync(2, kGroupThreads);
    stamp(2);
    // ---- reference initialisation of the hyperparameters (multiview_gibbs.cpp:75-98) ------------
    if (flags & kFinTauInit) {
      if (tid == 0) {
        // all customers sit at table 0 / dish 0 during this call: pooled variance over coordinates
        const double n = (double)c.n_global;
        double var = 1.0;
        if (c.n_global > 1) var = (S.s2k[0] - S.s1sq[0] / n) / ((n - 1.0) * (double)D);
        if (!(var > 0.0)) var = 1.0;
        tau_l = is_count ? 1.0 : var * 0.25 * 0.01;          // a count view has no kernel variance
        alpha_l = 1.0;
        sigma_l = 0.5;
      }
      group_sync(2, kGroupThreads);
    }
    // ---- D1. tau_v (update_tau_v_MH, multiview_hyper.cpp:211-231): warp 0 ----
    if ((flags & kFinHyper) && (flags & kFinHyperTau) && !is_count && tid < 32) {   // no tau in a count view (its stream positions stay unused)
      const int lane = tid;
      double tau_old = tau_l;
      if (tau_old <= 0.0) tau_old = kEps;
      const double tau_prop = fin_exp(fin_log(tau_old) + 0.0 + 0.3 * S.rn[0]);   // :166-174
      // log_posterior_given_tau (:176-209) at both values: lanes stride over the dishes, shuffle-tree sum
      const double lg_o = fin_log(2.0 * kPi * tau_old), lg_p = fin_log(2.0 * kPi * tau_prop);
      const double Dd = (double)D;
      double lo = 0.0, ln = 0.0;
      for (int k = lane; k < cap; k += 32) {
        const int n_k = S.n_vk[k];
        if (n_k == 0) continue;
        lo += -0.5 * (double)n_k * Dd * lg_o - 0.5 * (S.sse[k] / tau_old);
        ln += -0.5 * (double)n_k * Dd * lg_p - 0.5 * (S.sse[k] / tau_prop);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        lo += __shfl_xor_sync(0xffffffffu, lo, o);
        ln += __shfl_xor_sync(0xffffffffu, ln, o);
      }
      if (lane == 0) {
        const double a_tau = 2.0, b_tau = 1.0;                                    // :133-134
        // a log(b) - lgamma(a) = 2 log 1 - lgamma 2 = 0 exactly
        const double log_old = lo + (-(a_tau + 1.0) * fin_log(tau_old) - b_tau / tau_old);
        const double log_new = ln + (-(a_tau + 1.0) * fin_log(tau_prop) - b_tau / tau_prop);
        const double log_acc = (log_new - log_old) + (fin_log(tau_prop) - fin_log(tau_old));
        if (S.lu[0] < log_acc) tau_l = tau_prop;
      }
    }
    group_sync(2, kGroupThreads);
    stamp(9);
    // ---- E1. posterior means of the next sweep (oracle/mv_oracle.c:mvo_make_params) ----------
    {
      // one warp per table: lanes stride over the coordinates of the posterior mean m = S1k / (tau + n),
      // S1k re-summed from the per-table sums (same order as above, so the same value), write it (and its TF32
      // split) and reduce |m|^2 by a fixed shuffle tree
      const int lane = tid & 31, wid = tid >> 5;
      for (int t = wid; t < cap; t += kGroupThreads / 32) {
        const int k = S.dish[t];
        const int off = cap * doff + t * D;
        const double rden = (k >= 0) ? 1.0 / (tau_l + (double)S.n_vk[k]) : 0.0;
        // The tensor-core engine reads the means pre-scaled by the table's slope, b = 2 A m, so that its dot products
        // are the data term 2 A x.m of log2 f directly (A as in the parameter block below: same expression, same value).
        float A_f = 0.f;
        if (k >= 0 && !is_count) {
          const double nk = (double)S.n_vk[k];
          A_f = (float)(kLog2e * ((tau_l + nk) / (2.0 * tau_l * (tau_l + nk + 1.0))));
        }
        Set mask;
        if (k >= 0) mask = S.tmask[k];
        else mask.clear();
        const int t1 = mask.lowest();
        const Set more = mask.without_lowest();
        // Draw screening (DESIGN.md §4.1.1) bounds the drift of the scaled means b = hi + lo since its reference sweep from
        // three sums per table, formed here in FP64 by the same lanes and shuffle tree as |m|^2: |b|^2, |b - b_ref|^2 and
        // |R b - R_ref b_ref|^2 (R = A1 / A as k_draw_tc rounds it; A1 as in the parameter block below).
        const bool scr = c.scr_sum != nullptr && c.mean_hi != nullptr;
        double rq = 0.0, rp = 0.0;
        if (scr) {
          float A1_f = 0.f;
          if (k >= 0 && !is_count && (double)S.n_vk[k] >= 2.0) {
            const double tau = tau_l, n = (double)S.n_vk[k];
            A1_f = (float)(kLog2e * ((tau + n) / (2.0 * tau * (tau + n - 1.0))));
          }
          const TableParam p = ref_in_smem ? reinterpret_cast<const TableParam*>(ref_smem() + 2 * (size_t)cap * D)[t]
                                           : c.scr_tp[v * cap + t];
          rq = (A_f != 0.0f) ? (double)__fdiv_rn(A1_f, A_f) : 0.0;
          rp = (p.A != 0.0f) ? (double)__fdiv_rn(p.A1, p.A) : 0.0;
        }
        double sb = 0.0, sd = 0.0, sr = 0.0;
        double mm = 0.0;
        for (int dd = lane; dd < D; dd += 32) {
          double s1 = (t1 >= 0) ? S1t[t1 * D + dd] : 0.0;
          more.for_each([&](int t) { s1 += S1t[t * D + dd]; });
          const float m = (float)(s1 * rden);
          c.mean[off + dd] = m;
          if (c.mean_hi) {
            const float bm = (float)(2.0 * (double)A_f * (double)m);    // one rounding of the exact product (the mirror repeats it)
            uint32_t hb, lb;                                            // TF32 split, both parts rounded to nearest
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(bm));
            const float hi = __uint_as_float(hb);
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lb) : "f"(__fadd_rn(bm, -hi)));
            c.mean_hi[off + dd] = hi;
            c.mean_lo[off + dd] = __uint_as_float(lb);
            if (scr) {
              const double b = (double)hi + (double)__uint_as_float(lb);
              const float* rb = ref_in_smem ? ref_smem() + t * D : c.scr_b + off;   // hi; lo one half further on
              const size_t rhalf = ref_in_smem ? (size_t)cap * D : (size_t)cap * c.Dsum;
              const double bp = (double)rb[dd] + (double)rb[rhalf + dd];
              const double db = b - bp, dr = __fma_rn(b, rq, -__dmul_rn(rp, bp));
              sb = __fma_rn(b, b, sb);
              sd = __fma_rn(db, db, sd);
              sr = __fma_rn(dr, dr, sr);
            }
          }
          mm += (double)m * (double)m;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          mm += __shfl_xor_sync(0xffffffffu, mm, o);
          if (scr) {
            sb += __shfl_xor_sync(0xffffffffu, sb, o);
            sd += __shfl_xor_sync(0xffffffffu, sd, o);
            sr += __shfl_xor_sync(0xffffffffu, sr, o);
          }
        }
        if (lane == 0) S.s1sq[t] = mm;               // (s1sq is free again: reused for |m_t|^2)
        if (scr && lane == 0) {
          double* o3 = c.scr_sum + 3 * ((size_t)v * cap + t);
          o3[0] = sb; o3[1] = sd; o3[2] = sr;
        }
      }
    }
    if (!s1_in_smem) {                               // the next launch re-reads sum_s1t; nothing to write back
    }
  }
  __syncthreads();
  stamp(4);
  if (tid == 32) { c.hyp[v] = alpha_l; c.hyp[V + v] = sigma_l; c.hyp[2 * V + v] = tau_l; }
  for (int t = tid; t < cap; t += kFinThreads) {          // the scalar part, one thread per table
    const int i = v * cap + t;
    const int k = S.dish[t];
    const double mm = S.s1sq[t];
    TableParam q;
    if (k < 0) {
      q.A = 0.f; q.C = kMasked; q.A1 = 0.f; q.C1 = kMasked; q.W = kMasked; q.W1 = kMasked; q.dish = -1; q.lone = 0;
    } else if (is_count) {
      // count view: the dot products are log2 f already (C + A (2 acc - 0) = acc); C1 carries W beta + the token
      // total of the dish for the leave-one-out term of the kernel
      q.A = 0.5f; q.C = 0.f; q.A1 = 0.f;
      q.C1 = (float)count_wbeta_total(c.vocab[v], c.beta_v[v], S.s2k[k]);
      const bool rep = (S.tmask[k].lowest() == t);
      const double w = (double)S.l_live[k] - sigma_l, w1 = w - 1.0;
      q.W = (rep && w > 0.0) ? (float)fin_log2(w) : kMasked;
      q.W1 = (rep && w1 > 0.0) ? (float)fin_log2(w1) : kMasked;
      q.dish = k;
      q.lone = (S.l_live[k] == 1);
    } else {
      const double tau = tau_l, n = (double)S.n_vk[k];
      const double a = (tau + n) / (2.0 * tau * (tau + n + 1.0));
      const double cc = -0.5 * fin_log(2.0 * kPi * tau * (tau + n + 1.0) / (tau + n));
      q.A = (float)(kLog2e * a);
      q.C = (float)(kLog2e * ((double)D * cc - a * mm));
      if (n >= 2.0) {
        const double a1 = (tau + n) / (2.0 * tau * (tau + n - 1.0));
        const double c1 = -0.5 * fin_log(2.0 * kPi * tau * (tau + n) / (tau + n - 1.0));
        q.A1 = (float)(kLog2e * a1);
        q.C1 = (float)(kLog2e * ((double)D * c1 - a1 * mm));
      } else {
        q.A1 = 0.f; q.C1 = kMasked;
      }
      const bool rep = (S.tmask[k].lowest() == t);      // lowest table of its dish
      const double w = (double)S.l_live[k] - sigma_l, w1 = w - 1.0;
      q.W = (rep && w > 0.0) ? (float)fin_log2(w) : kMasked;
      q.W1 = (rep && w1 > 0.0) ? (float)fin_log2(w1) : kMasked;
      q.dish = k;
      q.lone = (S.l_live[k] == 1);
    }
    c.tparam[i] = q;
    if constexpr (MAXCAP <= 64) c.tsame[i] = (k >= 0) ? S.tmask[k].w[0] : 0ull;   // read by the tensor-core engine (cap 64) only
  }
  if (tid == 12 * 32) {
    const double tau = tau_l;
    int K_act = 0;
    long long sum_l = 0;
    for (int k = 0; k < cap; ++k) if (S.l_live[k] > 0) { K_act++; sum_l += S.l_live[k]; }
    ViewParam p;
    p.AN = (float)(kLog2e / (2.0 * tau));
    p.CN = (float)(kLog2e * (-0.5 * (double)D * fin_log(2.0 * kPi * tau)));
    if (is_count) { p.AN = (float)fin_log2((double)c.vocab[v]); p.CN = 0.f; }      // log2 f_new = -|x| log2 W
    if (is_count && c.count_model) { p.AN = 1.f; p.CN = 0.f; }   // DIRMULT: the draw passes -log2 f_new itself (cnt_q)
    const double wn0 = alpha_l + (double)K_act * sigma_l, wn1 = alpha_l + (double)(K_act - 1) * sigma_l;
    p.WN0 = wn0 > 0.0 ? (float)fin_log2(wn0) : kMasked;
    p.WN1 = wn1 > 0.0 ? (float)fin_log2(wn1) : kMasked;
    const double d0 = alpha_l + (double)sum_l, d1 = alpha_l + (double)(sum_l - 1);
    p.LD0 = d0 > 0.0 ? (float)fin_log2(d0) : 0.f;
    p.LD1 = d1 > 0.0 ? (float)fin_log2(d1) : 0.f;
    p.pad0 = p.pad1 = 0.f;
    c.vparam[v] = p;
    if (S.err) atomicOr(c.status, S.err);
  }
  stamp(5);
  __syncthreads();
  if (tid == 0) kclock_end(c.kclock + kClockFinalize, gridDim.x);
}

template <int MAXCAP>
static cudaError_t launch_finalize_cap(const Ctx& c, int32_t flags, cudaStream_t s) {
  int dmax = 0;
  for (int v = 0; v < c.V; ++v) dmax = c.D[v] > dmax ? c.D[v] : dmax;
  const size_t s1_bytes = sizeof(double) * (size_t)c.cap * dmax;
  const size_t ref_bytes = (2 * sizeof(float) * dmax + sizeof(TableParam)) * (size_t)c.cap;
  const size_t smem_max = (size_t)227 * 1024;
  const int s1_in_smem = (fin_shared_bytes<MAXCAP>() + s1_bytes <= smem_max) ? 1 : 0;
  size_t smem = fin_shared_bytes<MAXCAP>() + (s1_in_smem ? s1_bytes : 0);
  const bool scr = c.scr_sum != nullptr && c.mean_hi != nullptr;   // the drift sums of draw screening are formed
  const int ref_in_smem = (scr && smem + ref_bytes <= smem_max) ? 1 : 0;
  if (ref_in_smem) smem += ref_bytes;
  cudaError_t e = cudaFuncSetAttribute(k_finalize<MAXCAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  return launch_chain(k_finalize<MAXCAP>, dim3(c.V + 1), dim3(kFinThreads), smem, s, c.pdl != 0, c, flags, (int32_t)s1_in_smem,
                      (int32_t)ref_in_smem);
}

// The cap-64 instance keeps the shared-memory footprint of the small capacities; 128 and 256 take the wide one.
cudaError_t launch_finalize(const Ctx& c, int32_t flags, cudaStream_t s) {
  if (c.cap > 256 || c.world > kMaxWorld || c.V > kMaxViews) return cudaErrorInvalidValue;
  return c.cap <= 64 ? launch_finalize_cap<64>(c, flags, s) : launch_finalize_cap<256>(c, flags, s);
}

// =============================================================================================
// initial assignments (multiview_gibbs.cpp:12-62) and small utilities
// =============================================================================================
// mode 0: every row to table 0 / dish 0 (used to obtain the pooled variance for tau_v)
// mode 1: the reference's random start: T = 4 tables, K = 2 dishes per view
__global__ void k_init_tables(const Ctx c, const int32_t mode) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < c.n_rows) {
    int t = 0;
    if (mode == 1) {
      const U4 r = stream_block(c.seed, c.chain, kDomInitTable, 0, 0, (uint64_t)(c.row_offset + i));
      t = (int)floor(uniform_f64_from(r.x, r.y) * 4.0);
      t = t < 0 ? 0 : (t > 3 ? 3 : t);
    }
    c.choice[i] = t;
  }
  if (i < c.n_chunks) c.birthmask[i] = 0u;
  if (i < c.V * c.cap) {
    const int v = i / c.cap, t = i - v * c.cap;
    int k = -1;
    if (mode == 0) k = (t == 0) ? 0 : -1;
    else if (t < 4) {
      const U4 r = stream_block(c.seed, c.chain, kDomInitDish, (uint32_t)v, 0, (uint64_t)t);
      k = (int)floor(uniform_f64_from(r.x, r.y) * 2.0);
      k = k < 0 ? 0 : (k > 1 ? 1 : k);
    }
    c.dish_of[i] = k;
    c.l_vk[i] = 0;
    c.n_vk[i] = 0;
  }
  if (i < c.cap) c.n_t[i] = 0;
  if (i == 0) {
    c.gparam->nfree = 0;
    int32_t* hdr = reinterpret_cast<int32_t*>(c.packet + (size_t)c.rank * c.pkt.bytes + c.pkt.off_hdr);
    hdr[0] = 0; hdr[1] = 0; hdr[2] = c.rank; hdr[3] = 0;
    *reinterpret_cast<int64_t*>(hdr + 4) = c.row_offset;
    hdr[6] = 0; hdr[7] = 0;
  }
}

cudaError_t launch_init_tables(const Ctx& c, int32_t mode, cudaStream_t s) {
  int n = c.n_rows;
  if (c.V * c.cap > n) n = c.V * c.cap;
  if (c.n_chunks > n) n = c.n_chunks;
  k_init_tables<<<(n + 255) / 256, 256, 0, s>>>(c, mode);
  return cudaGetLastError();
}

// Squared norms of the rows of one view, xx[i] = sum_d x[i][d]^2 as one ascending fmaf chain (the order
// the CUDA-core draw kernel and the CPU mirror use), and the largest of each tile of 128 rows (one block), a NaN taken
// as +inf, for the tile test of draw screening.  The data never change, so this runs once per upload.
__global__ void __launch_bounds__(128) k_rownorms(const float* __restrict__ x, float* __restrict__ xx, float* __restrict__ xx_tmax, int n, int D) {
  __shared__ float s_max[4];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  float q = 0.0f;
  if (i < n) {
    const float* r = x + (size_t)i * D;
    for (int d = 0; d < D; ++d) q = __fmaf_rn(r[d], r[d], q);
    xx[i] = q;
  }
  if (!xx_tmax) return;
  float m = (q == q) ? q : INFINITY;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) xx_tmax[blockIdx.x] = fmaxf(fmaxf(s_max[0], s_max[1]), fmaxf(s_max[2], s_max[3]));
}
cudaError_t launch_rownorms(const float* x, float* xx, float* xx_tmax, int n, int D, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  k_rownorms<<<(n + 127) / 128, 128, 0, s>>>(x, xx, xx_tmax, n, D);
  return cudaGetLastError();
}

__global__ void k_f64_to_f32(const double* __restrict__ src, float* __restrict__ dst, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = (float)src[i];
}
cudaError_t launch_f64_to_f32(const double* src, float* dst, int64_t n, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  k_f64_to_f32<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, dst, n);
  return cudaGetLastError();
}

}  // namespace mv
