// mv_ctx.h — the POD kernel context: every device pointer and size one chain shard needs.
// Passed by value to the kernels (well under the 4 KB parameter limit).
//
// HBM layout (DESIGN.md §3).  N = rows of this shard, V views, cap slots, D_v dims,
// Dsum = sum D_v, doff[v] = sum_{u<v} D_u:
//   x[v]            float  [N][D_v]        row-major features of view v            (y[v][i], multiview_state.h:22)
//   table_cur       int32  [N]             table slot of each row                  (table_of)
//   choice          int32  [N]             raw draw of the current sweep, -1 = new table
//   birthmask       uint32 [ceil(N/32)]    bit r of word c: row 32c+r drew a new table
//   chunk_prefix    int32  [ceil(N/32)]    births in rows before chunk c (this shard)
//   n_t             int32  [cap]           customers per table                     (n_t)
//   dish_of         int32  [V][cap]        dish of table t in view v, -1 = free    (dish_of)
//   n_vk, l_vk      int32  [V][cap]        customers / tables per dish             (ViewState::n_vk, l_vk)
//   S1t, S1k        double [cap*Dsum]      per view a [cap][D_v] block: sums of rows per TABLE / per DISH
//   S2t, S2k        double [V][cap]        sums of squared norms per table / dish  (ViewState::sum_y2)
//   hyp             double [3V+2]          alpha_v[V], sigma_v[V], tau_v[V], alpha_g, sigma_g
//   tparam..gparam  FP32 parameter block of the next sweep (mv_device.cuh)
//   mean            float  [cap*Dsum]      per view [cap][D_v] per-TABLE posterior means m
//   partial         float  [stat_ctas][cap*Dsum + V*cap] + int32 [stat_ctas][cap]   per-CTA statistics
//   packet          bytes  [world][pkt_bytes]   what the shards exchange once per sweep
#pragma once
#include <stdint.h>

#include "mv_device.cuh"

namespace mv {

struct PacketLayout {       // byte offsets inside one shard's packet
  int32_t off_hdr;          // int32[8]: ncand, nbirth_local, rank, 0, row_offset (int64 in words 4-5), 0, 0
  int32_t off_cnt;          // int32[cap]      rows per table among non-candidate rows
  int32_t off_cand_row;     // int32[cap]      local row index of each candidate birth
  int32_t off_cand_t0;      // int32[cap]      its current table
  int32_t off_s2t;          // double[V*cap]
  int32_t off_s1t;          // double[cap*Dsum]
  int32_t off_cand_x;       // float[cap][Dsum] features of the candidate rows, views concatenated
  int32_t bytes;            // total, multiple of 16
};

struct Ctx {
  int32_t n_rows, V, cap, Dsum;
  int64_t row_offset, n_global;
  uint64_t seed;
  uint32_t chain;
  int32_t rank, world;
  int32_t n_chunks;         // ceil(n_rows/32)
  int32_t stat_ctas;        // CTAs of the statistics kernel (fixes the summation tree)
  int32_t debug_export;
  int32_t blk_count, blk_index;   // blocked sweep: only rows with (global row) % blk_count == blk_index are redrawn by this pass
  int32_t D[kMaxViews];
  int32_t doff[kMaxViews];
  const float* x[kMaxViews];
  // sparse COUNT views (CSR; SURVEY.md A.3).  kind[v] = 1: view v has no dense columns (D[v] = 0); its rows are
  // val[rowptr[i] .. rowptr[i+1]) at columns col[..] of a vocabulary of vocab[v] words.
  int32_t kind[kMaxViews];
  int32_t vocab[kMaxViews];
  const int32_t* rowptr[kMaxViews];
  const int32_t* col[kMaxViews];
  const float* val[kMaxViews];
  const int32_t* row_order[kMaxViews];   // the rows by descending number of nonzeros (the order the likelihood kernel deals them out in)
  int32_t* cnt_t[kMaxViews];   // [vocab][cap] word counts per TABLE slot (kept current after every finalize: the rows that changed table leave one slot and join another)
  int32_t* cnt_d[kMaxViews];   // [vocab][cap] word counts of the DISH each table slot serves
  float* l2t[kMaxViews];       // [vocab][cap] log2 theta of that dish: log2((beta + cnt_d) / (W beta + total))
  float* cnt_acc[kMaxViews];   // [N][cap] log2 f of every row under every table slot's dish (stage A of the sweep)
  float* cnt_loo[kMaxViews];   // [N] the same under the row's own dish with the row removed
  double* beta_v;              // [V] symmetric Dirichlet pseudo-count of every count view (0 for a dense view); the one
                               // source of beta on the device, for both count models
  int32_t n_count_views;
  // MVG_COUNT_DIRMULT (count_model = 1, every count view of the handle; DESIGN.md §4.5): l2t holds log2(beta + cnt_d)
  // instead of log2 theta, and
  int32_t count_model;
  int32_t cnt_nmax[kMaxViews]; // the longest row in tokens (known at upload)
  float* cnt_den[kMaxViews];   // [n_max+1][cap] sum_{j<n} log2(W beta + C_k + j) of the dish each slot serves, length-major
  float* cnt_q[kMaxViews];     // [N] -log2 f_new of every row (a function of beta alone): what the new-dish term reads
  // Metropolis-Hastings step for beta_v (MVG_COUNT_DIRMULT with mvg_set_count_beta_prior; DESIGN.md §4.5): prior
  // Gamma(cb_shape, rate cb_rate), log-normal random walk of scale cb_step, one step per count view per hyper step
  int32_t cb_on;
  int32_t cb_ctas;             // CTAs per view of k_count_beta_step (fixed per handle: fixes the summation tree)
  double cb_shape, cb_rate, cb_step;
  double* cb_part;             // [V][cb_ctas] per-CTA partial sums of L(beta') - L(beta)
  uint32_t* cb_arrive;         // [V] arrival counters of k_count_beta_step (zero between launches)
  int32_t* cb_accept;          // [V] 1: the most recent step of view v moved beta_v[v] (the refresh kernels run), else 0
  double* cb_logA;             // [V] log acceptance ratio of the most recent step (mvg_get_count_beta_step)
  int32_t* table_prev;        // [N] count views: the table every row's words are currently counted at in cnt_t
  float* xx;                // [V][xx_stride] squared norms of the rows (count views: the rows' total counts), computed once per upload
  int64_t xx_stride;        // n_rows rounded up to a multiple of 4
  float* xx_tmax;           // [V][ceil(N/128)] largest xx of each tile of 128 rows (a NaN counts as +inf): draw screening

  int32_t* table_cur;
  int32_t* choice;
  uint32_t* birthmask;
  uint32_t* movedmask;      // [ceil(N/32)] bit r of word c: the draw of row 32c+r differs from its table (incl. new-table draws)
  int32_t* chunk_prefix;

  int32_t* n_t;
  int32_t* dish_of;
  int32_t* n_vk;
  int32_t* l_vk;
  double* S1t;
  double* S2t;
  double* S1k;
  double* S2k;
  double* hyp;
  uint32_t* sweep;          // [1] index of the next sweep
  int32_t* status;          // [4] device-side error flags: [0] invariants (cleared when reported), [1] STICKY exchange fault

  TableParam* tparam;       // [V][cap]
  ViewParam* vparam;        // [V]
  TableMass* tmass;         // [cap]
  GlobalParam* gparam;      // [1]
  unsigned long long* tsame; // [V][cap] bit t2 of entry (v, t): table slot t2 serves the same dish as slot t in view v
  float* mean;              // [cap*Dsum]
  float* mean_hi;           // tensor-core engine: TF32-representable part of mean
  float* mean_lo;           //   and the remainder

  float* partial_f;         // [stat_ctas][cap*Dsum + V*cap]
  int32_t* partial_n;       // [stat_ctas][cap]
  int32_t* cta_active;      // [stat_ctas] incremental statistics: did this CTA of the statistics kernel see a moved row
  unsigned char* packet;    // [world][pkt.bytes]; this shard writes slot `rank`
  PacketLayout pkt;

  // totals over all shards, in rank order (k_reduce_x): what k_finalize starts from
  int32_t* sum_cnt;         // [cap]
  double* sum_s1t;          // [cap*Dsum]
  double* sum_s2t;          // [V*cap]
  uint32_t* xseq;           // [1] exchanges completed (peer-memory transport; advanced by k_finalize)
  uint32_t* fin_arrive;     // [1] arrival counter of the k_finalize CTAs
  int32_t* host_fault;      // mapped host memory: a copy of the sticky fault status[1] the host can read without a sync
  struct KClockSlot* kclock; // [kClockSlots] in-kernel wall clocks (below)
  int32_t pdl;              // launch the kernels of the sweep tail as programmatic dependents of one another (below)

  double* birth_lf;         // [cap][V][cap+1] scratch: log f of each seated birth under each dish
  // debug exports
  float* dbg_acc;           // [N][V][cap]
  float* dbg_xx;            // [N][V]
  int32_t* dbg_choice;      // [N]
  float* dbg_lnew;          // [N] tensor-core engine: log2 weight of a new table as the kernel evaluated it
  float* dbg_loo;           // [N][V] count views: the leave-one-out log2 f of the row under its own dish
  int64_t* dbg_birth_rows;  // [cap]
  double* dbg_birth_w;      // [cap][V][cap+1]
  int32_t* dbg_nseated;     // [1]
  long long* dbg_prof;      // [CTAs][16] cycles spent waiting per role of the tcgen05 kernel (debug_export & 2)

  // draw screening (tensor-core engine, DESIGN.md §4.1.1): rows whose draw is provably their own table skip the draw
  int32_t screen;           // k_draw_tc screens its tiles in every draw of this handle
  struct ScreenRec* scr;    // [1] the verdict of the most recent draw, and the reference sweep
  TableParam* scr_tp;       // [V][cap] parameter block of the reference sweep
  TableMass* scr_tm;        // [cap]
  float* scr_b;             // [2][cap*Dsum] its mean_hi, mean_lo
  float* margin;            // [N] lower bound on (own-table log2 weight - best other) at the reference, see ScreenRec
  int32_t* scr_tiles;       // [ceil(N/128)] row tiles the draw evaluates (mode kScreenSkip)
  float* margin_min;        // [n_chunks] least margin of each 32 rows (a NaN counts as -inf), written with the margins
  double* scr_sum;          // [V][cap][3] per table, from k_finalize: |b|^2, |b - b_ref|^2, |R b - R_ref b_ref|^2 (b = hi + lo)
  int32_t* scr_work;        // [ceil(N/128)] each CTA's tiles to evaluate (mode kScreenSkip), at blockIdx.x + j * gridDim.x
};

// What the screening of the most recent draw decided, and the reference the margins are measured against.  Written by
// k_draw_tc: mode, sweep, k (CTA 0); n_eval, last_*, and in a refresh valid and ref_sweep (the last CTA to decide).
enum { kScreenOff = 0, kScreenRefresh = 1, kScreenSkip = 2 };
constexpr int kScreenPeriod = 64;      // sweeps between two full evaluations (new reference)
struct ScreenRec {
  int32_t mode;             // kScreenOff: every tile, nothing recorded; kScreenRefresh: every tile, new reference; kScreenSkip: the list
  int32_t n_eval;           // tiles in scr_tiles
  float k[1 + 2 * 3];       // row bound Q = k0 + sum_v kA_v |x_v|^2 + kB_v |x_v|: drift since the reference + evaluation error
  uint32_t valid;           // the reference parameters and the margins stand for the current seating
  uint32_t ref_sweep;
  uint32_t sweep;           // the sweep the most recent draw belongs to (mvg_get_draw_screen_record pairs it with its parameters)
  uint32_t cnt, done, rows; // scratch of one draw (tile counter, CTAs decided, rows screened), zero between launches
  int64_t last_rows_screened, last_tiles_evaluated;
};
#ifdef __CUDACC__
// The row's bound, rounded upward: k_draw_tc subtracts it when it records a margin and when it tests one.
__device__ __forceinline__ float screen_row_bound(const float* k, const float* xx, int V) {
  float q = k[0];
  for (int v = 0; v < V; ++v) {
    q = __fmaf_ru(k[1 + v], xx[v], q);
    q = __fmaf_ru(k[4 + v], __fsqrt_ru(xx[v]), q);
  }
  return q;
}
#endif

// Programmatic dependent launch along the sweep: draw -> pack -> statistics -> reduce -> finalize -> draw.  Every kernel of
// the chain lets its successor be scheduled at once (pdl_trigger) and orders itself behind its predecessor with pdl_wait
// before it touches anything: completion of the predecessor implies that the predecessor's own wait returned, so the order
// of the whole chain is kept while the launch latencies (~1-2 us per kernel, a quarter of the serial tail) overlap.
// Both are no-ops for an ordinary launch.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
template <class... KArgs, class... Args>
inline cudaError_t launch_chain(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool programmatic, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = programmatic ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, args...);
}
#endif

// In-kernel wall clocks: %globaltimer (ns) from the first CTA in to the last CTA out of every launch, summed per kernel.
// Events cannot be placed inside a replayed CUDA graph; this is how bench.py times the kernels of the very sweeps it
// reports (mvg_kernel_clock).  Zero-initialised: the start is kept complemented so that 0 means "none yet".
struct KClockSlot { unsigned long long nstart, end, done, total_ns, launches, last_start, last_end, prev_end; };   // last / previous launch: absolute ns
enum { kClockDraw = 0, kClockFinalize = 1, kClockSlots = 2 };
#ifdef __CUDACC__
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// one thread per CTA each
__device__ __forceinline__ void kclock_begin(KClockSlot* s) { atomicMax(&s->nstart, ~globaltimer_ns()); }
__device__ __forceinline__ void kclock_end(KClockSlot* s, unsigned n_ctas) {
  atomicMax(&s->end, globaltimer_ns());
  __threadfence();
  if (atomicAdd(&s->done, 1ull) == (unsigned long long)(n_ctas - 1)) {   // the last CTA out closes the launch
    __threadfence();
    const unsigned long long a = ~atomicAdd(&s->nstart, 0ull), b = atomicAdd(&s->end, 0ull);
    s->total_ns += (b > a) ? (b - a) : 0ull;
    s->launches += 1ull;
    s->prev_end = s->last_end; s->last_start = a; s->last_end = b;
    s->nstart = 0ull; s->end = 0ull; s->done = 0ull;
    __threadfence();
  }
}
#endif

// Peer-memory exchange (mv_exchange.cu): the receive buffer of every rank, as mapped into this process, and the
// layout of one (parity, source rank) slot: n_units 16-byte units (the statistics) then n_words 8-byte words (births).
struct XchgPeers { unsigned char* recv[16]; };
struct XchgLayout { int64_t n_units, n_words, word_off, slot_bytes; };
XchgLayout xchg_layout(const struct Ctx& c);

enum FinalizeFlags : int32_t {
  kFinReseat = 1,      // seat births / resolve candidates (after a draw)
  kFinHyper = 2,       // run the hyperparameter step: the parts selected by the three bits below
  kFinHyperTau = 16,   //   tau_v            (update_tau_v_MH)
  kFinHyperLocal = 32, //   alpha_v, sigma_v
  kFinHyperGlobal = 64,//   alpha_global, sigma_global
  kFinHyperCountBeta = 128, //  beta_v of the count views (k_count_beta_step after the tables; only with a prior set)
  kFinHyperAll = 2 | 16 | 32 | 64 | 128,
  kFinAdvance = 4,     // sweep += 1
  kFinTauInit = 8      // derive tau_v from pooled variance (reference init), alpha/sigma literals
};

// launchers (definitions in the .cu files)
cudaError_t launch_draw_simt(const Ctx& c, cudaStream_t s);
cudaError_t launch_draw_tc(const Ctx& c, const void* maps, bool fast_exp, bool programmatic, cudaStream_t s);
bool draw_tc_supported(const Ctx& c);
size_t draw_tc_maps_bytes();                                   // host blob holding the TMA tensor maps
cudaError_t draw_tc_make_maps(const Ctx& c, void* maps_out);  // (re)encode them for the current pointers
cudaError_t launch_pack(const Ctx& c, cudaStream_t s);
// delta: only the rows that moved this sweep are visited; the per-CTA partials then hold the CHANGE of the statistics
// (rows that arrived minus rows that left) and k_reduce_x adds it to the shard's running sums (mode flag there).
cudaError_t launch_stats(const Ctx& c, bool delta, cudaStream_t s);
bool stats_tile_supported(const Ctx& c);
bool stats_delta_supported(const Ctx& c);
cudaError_t launch_stats_tile(const Ctx& c, bool delta, cudaStream_t s);
cudaError_t launch_reduce_x(const Ctx& c, int mode, bool delta, const XchgPeers& peers, unsigned char* recv_local, cudaStream_t s);
cudaError_t launch_finalize(const Ctx& c, int32_t flags, cudaStream_t s);
cudaError_t launch_init_tables(const Ctx& c, int32_t mode, cudaStream_t s);
cudaError_t launch_rownorms(const float* x, float* xx, float* xx_tmax, int n, int D, cudaStream_t s);
cudaError_t launch_f64_to_f32(const double* src, float* dst, int64_t n, cudaStream_t s);
int stats_smem_bytes(const Ctx& c);
// count views (mv_counts.cu)
cudaError_t launch_rowtotals(const int32_t* rowptr, const float* val, float* out, int n, cudaStream_t s);
cudaError_t launch_counts_rebuild(const Ctx& c, bool delta, cudaStream_t s);   // per count view: word counts per table slot (from scratch, or only the rows that changed table), dish tables
cudaError_t launch_counts_loglik(const Ctx& c, cudaStream_t s);    // per count view: log2 f of every row under every table
cudaError_t launch_counts_newdish(const Ctx& c, cudaStream_t s);   // DIRMULT: cnt_q of every count view at beta_v
// the beta step of every count view (flags: the finalize flags of the same rebuild), then the refresh of what depends on
// beta in the views whose step accepted; refresh_only: no step, refresh the views whose cb_accept is set
cudaError_t launch_count_beta(const Ctx& c, int32_t flags, bool refresh_only, cudaStream_t s);
// the (float) W beta + C_k of a count view's dish: TableParam::C1 and the base of its denominator table
__host__ __device__ __forceinline__ double count_wbeta_total(int vocab, double beta, double total) { return (double)vocab * beta + total; }
// posterior summaries (mv_summary.cu)
cudaError_t launch_labels(const Ctx& c, int32_t* out, cudaStream_t s);
cudaError_t launch_cocluster(const Ctx& c, int view, uint32_t* counts, cudaStream_t s);
cudaError_t launch_contingency(const Ctx& c, int view, const int32_t* truth, int n_classes, int32_t* table, cudaStream_t s);
cudaError_t launch_loglik(const Ctx& c, double* out, cudaStream_t s);

}  // namespace mv
