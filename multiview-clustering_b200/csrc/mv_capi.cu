// mv_capi.cu — the C ABI of include/mvg.h: handle lifetime, HBM allocation, H2D/D2H, kernel
// sequencing of one sweep, NCCL attachment.  Host code only; every number the sampler produces
// comes from the kernels in mv_draw_*.cu and mv_state_kernels.cu.  There is no CPU fallback:
// if CUDA is unavailable mvg_create fails with MVG_ECUDA.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nvtx3/nvToolsExt.h>     // header-only NVTX 3: ranges per stage of a sweep (SURVEY.md §5); no-ops without a tool attached

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <algorithm>
#include <vector>

#include "../../include/mvg.h"
#include "mv_ctx.h"

namespace {

using namespace mv;

struct NvtxRange {                 // a stage of the sweep as it is enqueued (and, in a graph replay, one range per sweep)
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

// ---- minimal NCCL surface, resolved at run time so that one-GPU use needs no NCCL at all -------
struct UidByValue { char internal[128]; };   // ncclUniqueId is passed by value
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, UidByValue, int) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;
std::mutex g_nccl_mu;

bool load_nccl(std::string& err) {
  std::lock_guard<std::mutex> lk(g_nccl_mu);
  if (g_nccl.lib) return true;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  void* lib = nullptr;
  for (const char* n : names) {
    lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (lib) break;
  }
  if (!lib) { err = "NCCL not found (dlopen libnccl.so.2)"; return false; }
  g_nccl.GetUniqueId = reinterpret_cast<int (*)(void*)>(dlsym(lib, "ncclGetUniqueId"));
  g_nccl.CommInitRank = reinterpret_cast<int (*)(void**, int, UidByValue, int)>(dlsym(lib, "ncclCommInitRank"));
  g_nccl.AllGather = reinterpret_cast<int (*)(const void*, void*, size_t, int, void*, cudaStream_t)>(dlsym(lib, "ncclAllGather"));
  g_nccl.CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(lib, "ncclCommDestroy"));
  g_nccl.GetErrorString = reinterpret_cast<const char* (*)(int)>(dlsym(lib, "ncclGetErrorString"));
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllGather || !g_nccl.CommDestroy) {
    err = "NCCL symbols missing";
    return false;
  }
  g_nccl.lib = lib;
  return true;
}

thread_local std::string g_create_error;

}  // namespace

struct mvg_handle {
  mvg_config cfg{};
  Ctx c{};
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[8]{};
  std::string err;
  std::vector<void*> owned;          // device allocations to free
  void* view_owned[kMaxViews]{};     // uploaded views (owned); attached views are not
  bool layout_done = false;
  bool state_ready = false;
  int engine = MVG_ENGINE_SIMT;
  void* comm = nullptr;
  bool comm_owned = false;
  int64_t launches = 0;
  float last_ms = 0.f;
  int sms = 148;
  void* tc_maps = nullptr;           // host copy of the TMA tensor maps (tcgen05 engine)
  void* csr_owned[kMaxViews][4]{};   // uploaded CSR views: rowptr, col, val, rows by descending length
  uint32_t* cocl = nullptr;          // [n_rows][n_rows] co-clustering counts (mvg_coclustering_*)
  int32_t cocl_view = -2;
  int32_t cocl_samples = 0;
  // One sweep captured as a CUDA graph (world = 1): [0] without, [1] with the hyper step.  A replay costs the host
  // one launch instead of 5-8, which is what bounds several small chains sharing a GPU.
  cudaGraphExec_t sweep_graph[4]{};   // [hyper step on/off] + 2 * [incremental statistics]
  int64_t sweep_graph_launches[4]{};
  // statistics mode (mvg_set_stats_mode): 0 = full rebuild every sweep; 1 = incremental (moved rows only) with a full
  // rebuild every `rebuild_every` sweeps
  int stats_mode = 0;
  int rebuild_every = 64;
  int since_full = 0;                // incremental sweeps since the last full rebuild
  // The captured sweep is ordered tail-first: pack -> stats -> reduce -> finalize -> DRAW of the next sweep, the draw being
  // the programmatic successor of finalize (its set-up and first feature loads overlap the serial tail).  So between
  // replays the draw of the next sweep has already run: a pure function of the state, discarded (the flag cleared) by
  // anything that changes the state other than a sweep.
  bool draw_pending = false;
  bool counts_valid = false;         // count views: cnt_t / table_prev are consistent with table_cur (else the next rebuild starts from zero)
  bool pdl_draw = false;             // the next sweep's draw is launched as the programmatic dependent of k_finalize
  bool graphs_ok = true;
  int64_t sweeps_issued = 0;
  // peer-memory exchange (optional; ncclAllGather otherwise)
  unsigned char* xrecv = nullptr;    // this rank's receive buffer (cudaMalloc, exported through CUDA IPC)
  XchgPeers xpeers{};                // every rank's receive buffer as mapped here ([rank] = xrecv)
  bool xp2p = false;
  bool xattached = false;            // peer mappings exist (they live until mvg_destroy)
  double* loglik_dev = nullptr;      // [V + 1] scratch of mvg_run's per-kept-sweep log-likelihood
  int32_t* host_fault = nullptr;     // mapped pinned host word: the sticky exchange fault, readable without a sync
  bool screen_want = true;           // mvg_set_draw_screen (effective on the tensor-core engines)
  float count_beta = 0.5f;           // mvg_set_count_beta: every count view's beta_v until the first state call
  double* saved_beta = nullptr;      // mvg_set_count_beta_trace: [n_saved_max][V] host buffer mvg_run fills, or null
};

namespace {

int fail(mvg_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg; else g_create_error = msg;
  return code;
}
#define MVG_CUDA(h, expr)                                                                    \
  do {                                                                                       \
    cudaError_t e__ = (expr);                                                                \
    if (e__ != cudaSuccess)                                                                  \
      return fail(h, MVG_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));         \
  } while (0)

template <class T>
int dev_alloc(mvg_handle* h, T** p, size_t count) {
  void* q = nullptr;
  size_t bytes = sizeof(T) * (count ? count : 1);
  cudaError_t e = cudaMalloc(&q, bytes);
  if (e != cudaSuccess) return fail(h, MVG_ENOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
  e = cudaMemsetAsync(q, 0, bytes, h->stream);
  if (e != cudaSuccess) return fail(h, MVG_ECUDA, std::string("cudaMemset: ") + cudaGetErrorString(e));
  h->owned.push_back(q);
  *p = static_cast<T*>(q);
  return MVG_OK;
}

int align16(int x) { return (x + 15) & ~15; }

float* xx_tmax_of(const Ctx& c, int v) { return c.xx_tmax + (size_t)v * ((c.n_rows + 127) / 128); }

// Allocate everything that depends on the dims of all views; called once they are all known.
int ensure_layout(mvg_handle* h) {
  if (h->layout_done) return MVG_OK;
  Ctx& c = h->c;
  int dsum = 0;
  c.n_count_views = 0;
  for (int v = 0; v < c.V; ++v) {
    if (c.kind[v]) {
      if (!c.rowptr[v]) return fail(h, MVG_ESTATE, "view " + std::to_string(v) + " has no data yet");
      c.n_count_views += 1;
    } else if (!c.x[v] || c.D[v] <= 0) {
      return fail(h, MVG_ESTATE, "view " + std::to_string(v) + " has no data yet");
    }
    c.doff[v] = dsum;
    dsum += c.D[v];
  }
  c.Dsum = dsum;
  {
    static const bool no_pdl = [] { const char* e = getenv("MVG_NO_PDL"); return e && e[0] == '1'; }();   // (A/B switch for measurements)
    static const bool no_chain = [] { const char* e = getenv("MVG_NO_PDL_CHAIN"); return e && e[0] == '1'; }();   // (the same for the tail alone)
    h->pdl_draw = c.n_count_views == 0 && !no_pdl;          // (the count views put memsets between the kernels of the tail)
    c.pdl = (h->pdl_draw && !no_chain) ? 1 : 0;
  }
  if (c.n_count_views && c.world != 1)
    return fail(h, MVG_EUNSUPPORTED, "count (CSR) views are supported on one GPU per chain (world = 1) in this version");
  const size_t N = (size_t)c.n_rows, cap = (size_t)c.cap, V = (size_t)c.V;
  int rc;
#define A(ptr, count) if ((rc = dev_alloc(h, &(ptr), (count))) != MVG_OK) return rc
  A(c.table_cur, N + 4 /* bulk copies read whole 16-byte groups */); A(c.choice, N + 4); A(c.birthmask, (size_t)c.n_chunks); A(c.movedmask, (size_t)c.n_chunks + 2); A(c.chunk_prefix, (size_t)c.n_chunks);
  A(c.n_t, cap); A(c.dish_of, V * cap); A(c.n_vk, V * cap); A(c.l_vk, V * cap);
  A(c.S1t, cap * dsum); A(c.S2t, V * cap); A(c.S1k, cap * dsum); A(c.S2k, V * cap);
  A(c.hyp, 3 * V + 2); A(c.sweep, 1); A(c.status, 4); A(c.beta_v, V);
  A(c.sum_cnt, cap); A(c.sum_s1t, cap * dsum); A(c.sum_s2t, V * cap); A(c.xseq, 1); A(c.fin_arrive, 1); A(c.kclock, (size_t)kClockSlots);
  A(c.tparam, V * cap); A(c.vparam, V); A(c.tmass, cap); A(c.gparam, 1); A(c.tsame, V * cap);
  A(c.mean, cap * dsum); A(c.mean_hi, cap * dsum); A(c.mean_lo, cap * dsum);
  A(c.partial_f, (size_t)c.stat_ctas * (cap * dsum + V * cap)); A(c.partial_n, (size_t)c.stat_ctas * cap); A(c.cta_active, (size_t)c.stat_ctas);
  A(c.birth_lf, cap * V * (cap + 1));
  A(c.dbg_birth_rows, cap); A(c.dbg_birth_w, cap * V * (cap + 1)); A(c.dbg_nseated, 1);
  A(c.dbg_prof, (size_t)256 * 16);
  PacketLayout& p = c.pkt;
  int off = 0;
  p.off_hdr = off; off += 32;
  p.off_cnt = off; off += align16(4 * c.cap);
  p.off_cand_row = off; off += align16(4 * c.cap);
  p.off_cand_t0 = off; off += align16(4 * c.cap);
  p.off_s2t = off; off += align16(8 * c.V * c.cap);
  p.off_s1t = off; off += align16(8 * c.cap * dsum);
  p.off_cand_x = off; off += align16(4 * c.cap * dsum);
  p.bytes = off;
  A(c.packet, (size_t)c.world * p.bytes);
  if (c.debug_export & 1) { A(c.dbg_acc, N * V * cap); A(c.dbg_xx, N * V); A(c.dbg_choice, N); A(c.dbg_loo, N * V); A(c.dbg_lnew, N); }
  for (int v = 0; v < c.V; ++v)
    if (c.kind[v]) {
      const size_t cells = (size_t)c.vocab[v] * cap;
      A(c.cnt_t[v], cells); A(c.cnt_d[v], cells); A(c.l2t[v], cells);
      A(c.cnt_acc[v], N * cap); A(c.cnt_loo[v], N);
      if (!c.table_prev) { A(c.table_prev, N); }
    }
  if (c.n_count_views) {             // the beta step: a fixed grid per handle (one summation tree whatever the seating)
    size_t max_cells = 0;
    for (int v = 0; v < c.V; ++v)
      if (c.kind[v] && (size_t)c.vocab[v] * cap > max_cells) max_cells = (size_t)c.vocab[v] * cap;
    const size_t ctas = (max_cells + 1023) / 1024;   // about four cells per thread at the most
    c.cb_ctas = (int32_t)std::min<size_t>(std::max<size_t>(ctas, 1), 296);
    A(c.cb_part, V * (size_t)c.cb_ctas); A(c.cb_arrive, V); A(c.cb_accept, V); A(c.cb_logA, V);
  }
#undef A
  h->layout_done = true;
  // engine choice
  h->engine = MVG_ENGINE_SIMT;
  if (h->cfg.engine == MVG_ENGINE_TCGEN05 || h->cfg.engine == MVG_ENGINE_TCGEN05_FAST) {
    if (!draw_tc_supported(c)) return fail(h, MVG_EUNSUPPORTED, "tcgen05 engine needs cap = 64 and one to three dense views of dim 64");
    h->engine = h->cfg.engine;
  } else if (h->cfg.engine == MVG_ENGINE_AUTO && draw_tc_supported(c)) {
    h->engine = MVG_ENGINE_TCGEN05;
  }
  if (h->engine == MVG_ENGINE_TCGEN05 || h->engine == MVG_ENGINE_TCGEN05_FAST) {
    if (posix_memalign(&h->tc_maps, 128, draw_tc_maps_bytes()) != 0) return fail(h, MVG_ENOMEM, "tensor map allocation");
    cudaError_t e = draw_tc_make_maps(c, h->tc_maps);
    if (e != cudaSuccess) return fail(h, MVG_ECUDA, std::string("cuTensorMapEncodeTiled: ") + cudaGetErrorString(e));
    // draw screening (DESIGN.md §4.1.1): the verdict record, the reference parameters, a margin per row and its minimum
    // per 32 rows, the tile lists, k_finalize's drift sums
    if ((rc = dev_alloc(h, &c.scr, 1)) != MVG_OK || (rc = dev_alloc(h, &c.scr_tp, V * cap)) != MVG_OK ||
        (rc = dev_alloc(h, &c.scr_tm, cap)) != MVG_OK || (rc = dev_alloc(h, &c.scr_b, 2 * cap * dsum)) != MVG_OK ||
        (rc = dev_alloc(h, &c.margin, N)) != MVG_OK || (rc = dev_alloc(h, &c.margin_min, (N + 31) / 32)) != MVG_OK ||
        (rc = dev_alloc(h, &c.scr_tiles, (N + 127) / 128)) != MVG_OK || (rc = dev_alloc(h, &c.scr_work, (N + 127) / 128)) != MVG_OK ||
        (rc = dev_alloc(h, &c.scr_sum, 3 * V * cap)) != MVG_OK)
      return rc;
    c.screen = (h->screen_want && !c.debug_export) ? 1 : 0;   // debug handles export what the full path computed
  }
  return MVG_OK;
}

// The margins stand for the seating they were recorded at: anything that replaces it from outside drops the reference, and
// the next screened draw evaluates every row (a refresh).  Stream-ordered; a no-op without screening state.
int invalidate_screen(mvg_handle* h) {
  if (h->c.scr) MVG_CUDA(h, cudaMemsetAsync(&h->c.scr->valid, 0, sizeof(uint32_t), h->stream));
  return MVG_OK;
}

// This shard's statistics -> totals over all shards (csrc/mv_exchange.cu).  One launch with the peer-memory
// transport or on one GPU; reduce, ncclAllGather, rank-ordered sums with the NCCL transport.
int reduce_exchange(mvg_handle* h, cudaEvent_t* marks, bool delta) {
  const Ctx& c = h->c;
  if (c.world == 1 || h->xp2p) {
    MVG_CUDA(h, launch_reduce_x(c, c.world == 1 ? 0 : 1, delta, h->xpeers, h->xrecv, h->stream));
    h->launches += 1;
    if (marks) { MVG_CUDA(h, cudaEventRecord(marks[1], h->stream)); MVG_CUDA(h, cudaEventRecord(marks[2], h->stream)); }
    return MVG_OK;
  }
  if (!h->comm) return fail(h, MVG_ESTATE, "world > 1 but neither an NCCL communicator nor peer buffers are attached");
  MVG_CUDA(h, launch_reduce_x(c, 0, delta, h->xpeers, h->xrecv, h->stream));
  if (marks) MVG_CUDA(h, cudaEventRecord(marks[1], h->stream));
  unsigned char* base = c.packet;
  int r = g_nccl.AllGather(base + (size_t)c.rank * c.pkt.bytes, base, (size_t)c.pkt.bytes, /*ncclChar*/ 0, h->comm, h->stream);
  if (r != 0) return fail(h, MVG_ENCCL, std::string("ncclAllGather: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?"));
  MVG_CUDA(h, launch_reduce_x(c, 2, false, h->xpeers, h->xrecv, h->stream));
  if (marks) MVG_CUDA(h, cudaEventRecord(marks[2], h->stream));
  h->launches += 2;
  return MVG_OK;
}

// stats -> reduce + exchange -> finalize: shared by sweeps, set_state and init
int rebuild_pipeline(mvg_handle* h, int32_t flags, cudaEvent_t* marks /* 4 events or null */, bool delta = false) {
  { NvtxRange r(delta ? "mvg:statistics (moved rows)" : "mvg:statistics (rebuild)"); MVG_CUDA(h, launch_stats(h->c, delta, h->stream)); }
  if (marks) MVG_CUDA(h, cudaEventRecord(marks[0], h->stream));
  int rc;
  { NvtxRange r("mvg:reduce+exchange"); rc = reduce_exchange(h, marks, delta); }
  if (rc != MVG_OK) return rc;
  { NvtxRange r("mvg:births, hyper step, parameters"); MVG_CUDA(h, launch_finalize(h->c, flags, h->stream)); }
  if (h->c.n_count_views) {          // count views: word counts by the final seating, then the log2 theta tables
    MVG_CUDA(h, launch_counts_rebuild(h->c, /*delta=*/h->counts_valid, h->stream));
    h->counts_valid = true;            // cnt_t and table_prev now stand for the current seating
    h->launches += 2;
    if (h->c.cb_on && (flags & kFinHyper) && (flags & kFinHyperCountBeta)) {   // the beta step needs the dish counts
      NvtxRange r("mvg:count beta step");
      MVG_CUDA(h, launch_count_beta(h->c, flags, /*refresh_only=*/false, h->stream));
      h->launches += 3;
    }
  }
  if (marks) MVG_CUDA(h, cudaEventRecord(marks[3], h->stream));
  h->launches += 2;
  return MVG_OK;
}

// At the first state call (the views, the model and the setter's beta are frozen from then on): beta_v of every count view,
// then under MVG_COUNT_DIRMULT the denominator tables and the per-row new-dish terms.
int prepare_count_model(mvg_handle* h) {
  Ctx& c = h->c;
  if (h->state_ready || !c.n_count_views) return MVG_OK;
  std::vector<double> beta((size_t)c.V, 0.0);
  for (int v = 0; v < c.V; ++v) if (c.kind[v]) beta[(size_t)v] = (double)h->count_beta;
  MVG_CUDA(h, cudaMemcpyAsync(c.beta_v, beta.data(), sizeof(double) * beta.size(), cudaMemcpyHostToDevice, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));       // (a host temporary)
  if (!c.count_model) return MVG_OK;
  for (int v = 0; v < c.V; ++v) {
    if (!c.kind[v]) continue;
    if (c.cnt_nmax[v] >= (1 << 24))
      return fail(h, MVG_EINVAL, "the Dirichlet-multinomial count likelihood needs rows of fewer than 2^24 tokens");
    int rc;
    if (!c.cnt_den[v] && (rc = dev_alloc(h, &c.cnt_den[v], (size_t)(c.cnt_nmax[v] + 1) * c.cap)) != MVG_OK) return rc;
    if (!c.cnt_q[v] && (rc = dev_alloc(h, &c.cnt_q[v], (size_t)c.n_rows)) != MVG_OK) return rc;
  }
  MVG_CUDA(h, launch_counts_newdish(c, h->stream));
  h->launches += 1;
  return MVG_OK;
}

int launch_draw(mvg_handle* h, bool programmatic = false) {
  if (h->engine == MVG_ENGINE_TCGEN05 || h->engine == MVG_ENGINE_TCGEN05_FAST) {
    MVG_CUDA(h, launch_draw_tc(h->c, h->tc_maps, h->engine == MVG_ENGINE_TCGEN05_FAST, programmatic, h->stream));
  } else {
    MVG_CUDA(h, launch_draw_simt(h->c, h->stream));
  }
  h->launches += 1 + ((h->engine == MVG_ENGINE_SIMT && h->c.n_count_views) ? 1 : 0);
  return MVG_OK;
}

int check_status(mvg_handle* h) {
  int32_t st[4] = {0, 0, 0, 0};
  MVG_CUDA(h, cudaMemcpyAsync(st, h->c.status, sizeof(st), cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  if (st[1] != 0)
    return fail(h, MVG_ENCCL, "exchange fault (sticky): a peer's statistics did not arrive within the wait limit; this rank's chain is "
                              "frozen at its last completed sweep (mvg_get_state still reads it after mvg_clear_fault)");
  if (st[0] != 0) {
    MVG_CUDA(h, cudaMemsetAsync(h->c.status, 0, sizeof(int32_t), h->stream));
    return fail(h, MVG_EINVAL, "device-side invariant violated, flags=" + std::to_string(st[0]) +
                                   " (1: no free dish slot for a birth, 2: live table without a dish, 4: customers lost in the statistics rebuild, "
                                   "8: a peer's packet never arrived in the peer-memory exchange)");
  }
  return MVG_OK;
}

}  // namespace

extern "C" {

int mvg_abi_version(void) { return MVG_ABI_VERSION; }

const char* mvg_last_error(const mvg_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int mvg_create(const mvg_config* cfg, mvg_handle** out) {
  if (!cfg || !out) return fail(nullptr, MVG_EINVAL, "null argument");
  *out = nullptr;
  if (cfg->abi_version != MVG_ABI_VERSION) return fail(nullptr, MVG_EINVAL, "abi_version mismatch");
  if (cfg->n_rows <= 0 || cfg->n_rows > 0x7fffffffLL) return fail(nullptr, MVG_EINVAL, "n_rows out of range");
  if (cfg->n_views <= 0 || cfg->n_views > kMaxViews) return fail(nullptr, MVG_EINVAL, "n_views out of range");
  if (cfg->cap != 32 && cfg->cap != 64 && cfg->cap != 128 && cfg->cap != 256)
    return fail(nullptr, MVG_EUNSUPPORTED, "cap must be 32, 64, 128 or 256");
  if (cfg->world < 1 || cfg->world > 16 || cfg->rank < 0 || cfg->rank >= cfg->world)
    return fail(nullptr, MVG_EINVAL, "rank/world out of range");
  if (cfg->n_rows_global < cfg->n_rows || cfg->row_offset < 0 || cfg->row_offset + cfg->n_rows > cfg->n_rows_global)
    return fail(nullptr, MVG_EINVAL, "row_offset / n_rows_global inconsistent");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, MVG_ECUDA, std::string("no CUDA device: ") + cudaGetErrorString(e) +
                                        " (this library has no CPU path)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, MVG_EINVAL, "device ordinal out of range");
  mvg_handle* h = new (std::nothrow) mvg_handle();
  if (!h) return fail(nullptr, MVG_ENOMEM, "host allocation failed");
  h->cfg = *cfg;
  if ((e = cudaSetDevice(cfg->device)) != cudaSuccess ||
      (e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) {
    std::string m = std::string("cuda init: ") + cudaGetErrorString(e);
    delete h;
    return fail(nullptr, MVG_ECUDA, m);
  }
  for (auto& ev : h->ev) cudaEventCreate(&ev);
  cudaDeviceGetAttribute(&h->sms, cudaDevAttrMultiProcessorCount, cfg->device);
  Ctx& c = h->c;
  c.n_rows = (int32_t)cfg->n_rows;
  c.V = cfg->n_views;
  c.cap = cfg->cap;
  c.row_offset = cfg->row_offset;
  c.n_global = cfg->n_rows_global;
  c.seed = cfg->seed;
  c.chain = cfg->chain;
  c.rank = cfg->rank;
  c.world = cfg->world;
  c.n_chunks = (c.n_rows + 31) / 32;
  c.stat_ctas = c.n_chunks < h->sms ? c.n_chunks : h->sms;
  c.debug_export = cfg->debug_export;
  c.blk_count = 1;
  c.blk_index = 0;
  {
    void* q = nullptr;
    c.xx_stride = ((int64_t)c.n_rows + 3) & ~(int64_t)3;        // rows of xx start 16-byte aligned (bulk copies)
    // at least three rows: the tensor-core epilogue prefetches the norms of three views unconditionally
    const size_t xx_rows = c.V > 3 ? (size_t)c.V : 3;
    if (cudaMalloc(&q, sizeof(float) * (size_t)c.xx_stride * xx_rows) != cudaSuccess || cudaMemset(q, 0, sizeof(float) * (size_t)c.xx_stride * xx_rows) != cudaSuccess) {
      mvg_destroy(h);
      return fail(nullptr, MVG_ENOMEM, "cudaMalloc: squared norms");
    }
    h->owned.push_back(q);
    c.xx = static_cast<float*>(q);
    const size_t tiles = (size_t)(c.n_rows + 127) / 128 * xx_rows;
    if (cudaMalloc(&q, sizeof(float) * tiles) != cudaSuccess || cudaMemset(q, 0, sizeof(float) * tiles) != cudaSuccess) {
      mvg_destroy(h);
      return fail(nullptr, MVG_ENOMEM, "cudaMalloc: squared norms");
    }
    h->owned.push_back(q);
    c.xx_tmax = static_cast<float*>(q);
  }
  if (c.world > 1) {                               // the sticky exchange fault, mirrored where the host reads it without a sync
    void* hp = nullptr;
    void* dp = nullptr;
    if (cudaHostAlloc(&hp, 64, cudaHostAllocMapped) == cudaSuccess && cudaHostGetDevicePointer(&dp, hp, 0) == cudaSuccess) {
      std::memset(hp, 0, 64);
      h->host_fault = static_cast<int32_t*>(hp);
      c.host_fault = static_cast<int32_t*>(dp);
    } else {
      cudaGetLastError();
      if (hp) cudaFreeHost(hp);
    }
  }
  *out = h;
  return MVG_OK;
}

int mvg_destroy(mvg_handle* h) {
  if (!h) return MVG_OK;
  cudaSetDevice(h->cfg.device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->comm && h->comm_owned && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
  for (int g = 0; g < h->c.world && g < 16; ++g)
    if (g != h->c.rank && h->xpeers.recv[g]) cudaIpcCloseMemHandle(h->xpeers.recv[g]);
  if (h->xrecv) cudaFree(h->xrecv);
  if (h->host_fault) cudaFreeHost(h->host_fault);
  for (auto& g : h->sweep_graph) if (g) cudaGraphExecDestroy(g);
  for (void* p : h->owned) cudaFree(p);
  for (void* p : h->view_owned) if (p) cudaFree(p);
  for (auto& a : h->csr_owned) for (void* p : a) if (p) cudaFree(p);
  for (auto& ev : h->ev) if (ev) cudaEventDestroy(ev);
  if (h->stream) cudaStreamDestroy(h->stream);
  free(h->tc_maps);
  delete h;
  return MVG_OK;
}

static void invalidate_graphs(mvg_handle* h) {     // kernel arguments are baked into a captured sweep
  h->draw_pending = false;
  for (auto& g : h->sweep_graph) if (g) { cudaGraphExecDestroy(g); g = nullptr; }
}

static int set_view(mvg_handle* h, int32_t v, int32_t dim) {
  if (!h) return MVG_EINVAL;
  invalidate_graphs(h);
  if (v < 0 || v >= h->c.V) return fail(h, MVG_EINVAL, "view index out of range");
  if (dim <= 0) return fail(h, MVG_EINVAL, "dim must be positive");
  if (h->layout_done && h->c.D[v] != dim) return fail(h, MVG_ESTATE, "view dims are frozen after the first state call");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  return MVG_OK;
}

int mvg_upload_view_f32(mvg_handle* h, int32_t v, const float* x_host, int32_t dim) {
  int rc = set_view(h, v, dim);
  if (rc != MVG_OK) return rc;
  if (!x_host) return fail(h, MVG_EINVAL, "null data");
  const size_t bytes = sizeof(float) * (size_t)h->c.n_rows * dim;
  if (!h->view_owned[v] || h->c.D[v] != dim) {
    if (h->view_owned[v]) cudaFree(h->view_owned[v]);
    h->view_owned[v] = nullptr;
    MVG_CUDA(h, cudaMalloc(&h->view_owned[v], bytes));
  }
  MVG_CUDA(h, cudaMemcpyAsync(h->view_owned[v], x_host, bytes, cudaMemcpyHostToDevice, h->stream));
  h->c.x[v] = static_cast<const float*>(h->view_owned[v]);
  h->c.D[v] = dim;
  h->c.kind[v] = 0;
  MVG_CUDA(h, launch_rownorms(h->c.x[v], h->c.xx + (size_t)v * h->c.xx_stride, xx_tmax_of(h->c, v), h->c.n_rows, dim, h->stream));
  h->launches += 1;
  return MVG_OK;
}

int mvg_upload_view_f64(mvg_handle* h, int32_t v, const double* y_host, int32_t dim) {
  int rc = set_view(h, v, dim);
  if (rc != MVG_OK) return rc;
  if (!y_host) return fail(h, MVG_EINVAL, "null data");
  const size_t count = (size_t)h->c.n_rows * dim;
  if (!h->view_owned[v] || h->c.D[v] != dim) {
    if (h->view_owned[v]) cudaFree(h->view_owned[v]);
    h->view_owned[v] = nullptr;
    MVG_CUDA(h, cudaMalloc(&h->view_owned[v], sizeof(float) * count));
  }
  double* tmp = nullptr;
  MVG_CUDA(h, cudaMalloc(&tmp, sizeof(double) * count));
  cudaError_t e = cudaMemcpyAsync(tmp, y_host, sizeof(double) * count, cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) e = launch_f64_to_f32(tmp, static_cast<float*>(h->view_owned[v]), (int64_t)count, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(tmp);
  if (e != cudaSuccess) return fail(h, MVG_ECUDA, std::string("upload f64: ") + cudaGetErrorString(e));
  h->launches += 1;
  h->c.x[v] = static_cast<const float*>(h->view_owned[v]);
  h->c.D[v] = dim;
  MVG_CUDA(h, launch_rownorms(h->c.x[v], h->c.xx + (size_t)v * h->c.xx_stride, xx_tmax_of(h->c, v), h->c.n_rows, dim, h->stream));
  h->launches += 1;
  return MVG_OK;
}

int mvg_attach_view_device_f32(mvg_handle* h, int32_t v, const float* x_dev, int32_t dim) {
  int rc = set_view(h, v, dim);
  if (rc != MVG_OK) return rc;
  if (!x_dev || (reinterpret_cast<uintptr_t>(x_dev) & 15)) return fail(h, MVG_EINVAL, "device pointer null or not 16-byte aligned");
  if (h->view_owned[v]) { cudaFree(h->view_owned[v]); h->view_owned[v] = nullptr; }
  h->c.x[v] = x_dev;
  h->c.D[v] = dim;
  MVG_CUDA(h, launch_rownorms(x_dev, h->c.xx + (size_t)v * h->c.xx_stride, xx_tmax_of(h->c, v), h->c.n_rows, dim, h->stream));
  h->launches += 1;
  return MVG_OK;
}

int mvg_set_count_beta(mvg_handle* h, double beta) {
  if (!h) return MVG_EINVAL;
  if (!(beta > 0.0) || beta > 1.0e6) return fail(h, MVG_EINVAL, "count_beta must be positive");
  if (h->state_ready) return fail(h, MVG_ESTATE, "count_beta is frozen after the first state call");
  h->count_beta = (float)beta;
  return MVG_OK;
}

int mvg_set_count_beta_prior(mvg_handle* h, double shape, double rate, double step) {
  if (!h) return MVG_EINVAL;
  if (!(std::isfinite(shape) && shape > 0.0) || !(std::isfinite(rate) && rate > 0.0) || !(std::isfinite(step) && step > 0.0))
    return fail(h, MVG_EINVAL, "the count beta prior needs finite positive shape, rate and step");
  bool any_count = false;
  for (int v = 0; v < h->c.V; ++v) any_count = any_count || h->c.kind[v] != 0;
  if (h->c.count_model != MVG_COUNT_DIRMULT || !any_count)
    return fail(h, MVG_ESTATE, "the beta step needs a count view under MVG_COUNT_DIRMULT (the plug-in likelihood has no marginal)");
  if (h->state_ready) return fail(h, MVG_ESTATE, "the count beta prior is frozen after the first state call");
  h->c.cb_on = 1;
  h->c.cb_shape = shape;
  h->c.cb_rate = rate;
  h->c.cb_step = step;
  invalidate_graphs(h);
  return MVG_OK;
}

int mvg_get_count_beta(mvg_handle* h, double* beta) {
  if (!h || !beta) return MVG_EINVAL;
  const Ctx& c = h->c;
  if (!h->state_ready) {               // nothing on the device yet: what the first state call will set
    for (int v = 0; v < c.V; ++v) beta[v] = c.kind[v] ? (double)h->count_beta : 0.0;
    return MVG_OK;
  }
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  MVG_CUDA(h, cudaMemcpyAsync(beta, c.beta_v, sizeof(double) * (size_t)c.V, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  return MVG_OK;
}

int mvg_get_count_beta_step(mvg_handle* h, double* log_accept, int32_t* accepted) {
  if (!h) return MVG_EINVAL;
  const Ctx& c = h->c;
  if (!c.cb_on || !h->state_ready) return fail(h, MVG_ESTATE, "no count beta step has run (set a prior, then a state)");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  if (log_accept) MVG_CUDA(h, cudaMemcpyAsync(log_accept, c.cb_logA, sizeof(double) * (size_t)c.V, cudaMemcpyDeviceToHost, h->stream));
  if (accepted) MVG_CUDA(h, cudaMemcpyAsync(accepted, c.cb_accept, sizeof(int32_t) * (size_t)c.V, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  return MVG_OK;
}

int mvg_set_count_beta_trace(mvg_handle* h, double* saved_beta) {
  if (!h) return MVG_EINVAL;
  h->saved_beta = saved_beta;
  return MVG_OK;
}

int mvg_set_count_likelihood(mvg_handle* h, int32_t model) {
  if (!h) return MVG_EINVAL;
  if (model != MVG_COUNT_PLUGIN && model != MVG_COUNT_DIRMULT) return fail(h, MVG_EINVAL, "unknown count likelihood model");
  if (h->state_ready) return fail(h, MVG_ESTATE, "the count likelihood is frozen after the first state call");
  // (count values are checked to be non-negative integers at upload, whatever the model)
  h->c.count_model = model;
  return MVG_OK;
}

int mvg_upload_view_csr(mvg_handle* h, int32_t v, const int32_t* rowptr, const int32_t* col, const float* val,
                        int64_t nnz, int32_t vocab) {
  if (!h) return MVG_EINVAL;
  if (v < 0 || v >= h->c.V) return fail(h, MVG_EINVAL, "view index out of range");
  if (!rowptr || (nnz > 0 && (!col || !val))) return fail(h, MVG_EINVAL, "null data");
  if (vocab <= 0 || nnz < 0 || nnz > 0x7fffffffLL) return fail(h, MVG_EINVAL, "vocab / nnz out of range");
  if (h->layout_done) return fail(h, MVG_ESTATE, "views are frozen after the first state call");
  const int64_t n = h->c.n_rows;
  if (rowptr[0] != 0 || rowptr[n] != nnz) return fail(h, MVG_EINVAL, "rowptr[0] must be 0 and rowptr[n_rows] = nnz");
  for (int64_t i = 0; i < n; ++i)
    if (rowptr[i + 1] < rowptr[i]) return fail(h, MVG_EINVAL, "rowptr must be non-decreasing");
  for (int64_t j = 0; j < nnz; ++j) {
    if (col[j] < 0 || col[j] >= vocab) return fail(h, MVG_EINVAL, "column index outside [0, vocab)");
    if (!(val[j] >= 0.0f) || val[j] > 16777216.0f || val[j] != (float)(int32_t)val[j])
      return fail(h, MVG_EINVAL, "count views hold non-negative integer counts (< 2^24)");
  }
  int64_t n_max = 0;                 // the longest row in tokens: rows of the Dirichlet-multinomial denominator table
  for (int64_t i = 0; i < n; ++i) {
    int64_t tok = 0;
    for (int32_t j = rowptr[i]; j < rowptr[i + 1]; ++j) tok += (int64_t)val[j];
    n_max = tok > n_max ? tok : n_max;
  }
  if (n_max > 0x7fffffffLL) n_max = 0x7fffffffLL;   // (refused by the Dirichlet-multinomial model, prepare_count_model)
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  for (void*& p : h->csr_owned[v]) { if (p) cudaFree(p); p = nullptr; }
  if (h->view_owned[v]) { cudaFree(h->view_owned[v]); h->view_owned[v] = nullptr; }
  const size_t nz = (size_t)(nnz ? nnz : 1);
  MVG_CUDA(h, cudaMalloc(&h->csr_owned[v][0], sizeof(int32_t) * (size_t)(n + 1)));
  MVG_CUDA(h, cudaMalloc(&h->csr_owned[v][1], sizeof(int32_t) * nz));
  MVG_CUDA(h, cudaMalloc(&h->csr_owned[v][2], sizeof(float) * nz));
  MVG_CUDA(h, cudaMemcpyAsync(h->csr_owned[v][0], rowptr, sizeof(int32_t) * (size_t)(n + 1), cudaMemcpyHostToDevice, h->stream));
  if (nnz) {
    MVG_CUDA(h, cudaMemcpyAsync(h->csr_owned[v][1], col, sizeof(int32_t) * nz, cudaMemcpyHostToDevice, h->stream));
    MVG_CUDA(h, cudaMemcpyAsync(h->csr_owned[v][2], val, sizeof(float) * nz, cudaMemcpyHostToDevice, h->stream));
  }
  {
    // the rows by descending number of nonzeros (ties: ascending row), the order k_counts_loglik deals them out in
    std::vector<int32_t> order((size_t)n);
    for (int64_t i = 0; i < n; ++i) order[(size_t)i] = (int32_t)i;
    std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return rowptr[a + 1] - rowptr[a] > rowptr[b + 1] - rowptr[b]; });
    MVG_CUDA(h, cudaMalloc(&h->csr_owned[v][3], sizeof(int32_t) * (size_t)(n ? n : 1)));
    MVG_CUDA(h, cudaMemcpy(h->csr_owned[v][3], order.data(), sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice));
  }
  Ctx& c = h->c;
  c.kind[v] = 1;
  c.vocab[v] = vocab;
  c.cnt_nmax[v] = (int32_t)n_max;
  c.row_order[v] = static_cast<const int32_t*>(h->csr_owned[v][3]);
  c.D[v] = 0;
  c.x[v] = nullptr;
  c.rowptr[v] = static_cast<const int32_t*>(h->csr_owned[v][0]);
  c.col[v] = static_cast<const int32_t*>(h->csr_owned[v][1]);
  c.val[v] = static_cast<const float*>(h->csr_owned[v][2]);
  MVG_CUDA(h, launch_rowtotals(c.rowptr[v], c.val[v], c.xx + (size_t)v * c.xx_stride, c.n_rows, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));       // the caller's buffers may go away
  h->launches += 1;
  return MVG_OK;
}

int mvg_get_count_tables(mvg_handle* h, int32_t v, float* log2_theta, int32_t* dish_counts, int32_t* table_counts) {
  if (!h) return MVG_EINVAL;
  if (v < 0 || v >= h->c.V || !h->c.kind[v]) return fail(h, MVG_EINVAL, "not a count view");
  if (!h->state_ready) return fail(h, MVG_ESTATE, "no state yet");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  const size_t cells = (size_t)h->c.vocab[v] * h->c.cap;
  if (log2_theta) MVG_CUDA(h, cudaMemcpyAsync(log2_theta, h->c.l2t[v], sizeof(float) * cells, cudaMemcpyDeviceToHost, h->stream));
  if (dish_counts) MVG_CUDA(h, cudaMemcpyAsync(dish_counts, h->c.cnt_d[v], sizeof(int32_t) * cells, cudaMemcpyDeviceToHost, h->stream));
  if (table_counts) MVG_CUDA(h, cudaMemcpyAsync(table_counts, h->c.cnt_t[v], sizeof(int32_t) * cells, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  return MVG_OK;
}

int mvg_get_count_den(mvg_handle* h, int32_t v, float* den, int32_t* n_max) {
  if (!h) return MVG_EINVAL;
  if (v < 0 || v >= h->c.V || !h->c.kind[v]) return fail(h, MVG_EINVAL, "not a count view");
  if (n_max) *n_max = h->c.cnt_nmax[v];
  if (!den) return MVG_OK;
  if (!h->state_ready) return fail(h, MVG_ESTATE, "no state yet");
  if (!h->c.count_model) return fail(h, MVG_ESTATE, "the plug-in count likelihood has no denominator table");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  const size_t cells = (size_t)(h->c.cnt_nmax[v] + 1) * h->c.cap;
  MVG_CUDA(h, cudaMemcpyAsync(den, h->c.cnt_den[v], sizeof(float) * cells, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  return MVG_OK;
}

int mvg_get_debug_loo(mvg_handle* h, float* loo) {
  if (!h || !loo) return MVG_EINVAL;
  if (!h->c.dbg_loo) return fail(h, MVG_ESTATE, "debug_export was not enabled");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  MVG_CUDA(h, cudaMemcpyAsync(loo, h->c.dbg_loo, sizeof(float) * (size_t)h->c.n_rows * h->c.V, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  return MVG_OK;
}

int mvg_init_state_reference(mvg_handle* h) {
  if (!h) return MVG_EINVAL;
  h->draw_pending = false;
  h->counts_valid = false;           // the seating is replaced from outside: the word counts of count views start from zero
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  int rc = ensure_layout(h);
  if (rc == MVG_OK) rc = prepare_count_model(h);
  if (rc != MVG_OK) return rc;
  if (h->c.cap < 4) return fail(h, MVG_EINVAL, "reference initialisation needs cap >= 4");
  if ((rc = invalidate_screen(h)) != MVG_OK) return rc;
  const uint32_t zero = 0;
  MVG_CUDA(h, cudaMemcpyAsync(h->c.sweep, &zero, sizeof(zero), cudaMemcpyHostToDevice, h->stream));
  MVG_CUDA(h, launch_init_tables(h->c, 0, h->stream));
  if ((rc = rebuild_pipeline(h, kFinTauInit, nullptr)) != MVG_OK) return rc;
  MVG_CUDA(h, launch_init_tables(h->c, 1, h->stream));
  if ((rc = rebuild_pipeline(h, 0, nullptr)) != MVG_OK) return rc;
  h->launches += 2;
  h->state_ready = true;
  return check_status(h);
}

int mvg_set_state(mvg_handle* h, const mvg_state_host* s) {
  if (!h || !s) return MVG_EINVAL;
  h->draw_pending = false;
  h->counts_valid = false;           // the seating is replaced from outside: the word counts of count views start from zero
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  int rc = ensure_layout(h);
  if (rc == MVG_OK) rc = prepare_count_model(h);
  if (rc != MVG_OK) return rc;
  if ((rc = invalidate_screen(h)) != MVG_OK) return rc;
  const Ctx& c = h->c;
  if (!s->table_of || !s->dish_of || !s->alpha_v || !s->sigma_v || !s->tau_v || !s->alpha_sigma_global)
    return fail(h, MVG_EINVAL, "set_state needs table_of, dish_of, alpha_v, sigma_v, tau_v, alpha_sigma_global");
  for (int64_t i = 0; i < c.n_rows; ++i)
    if (s->table_of[i] < 0 || s->table_of[i] >= c.cap) return fail(h, MVG_EINVAL, "table_of entry outside [0,cap)");
  for (int i = 0; i < c.V * c.cap; ++i)
    if (s->dish_of[i] < -1 || s->dish_of[i] >= c.cap) return fail(h, MVG_EINVAL, "dish_of entry outside [-1,cap)");
  for (int v = 0; v < c.V; ++v)
    if (!(s->tau_v[v] > 0.0) || !(s->alpha_v[v] > 0.0) || !(s->sigma_v[v] > 0.0 && s->sigma_v[v] < 1.0))
      return fail(h, MVG_EINVAL, "hyperparameters out of range (tau>0, alpha>0, 0<sigma<1)");
  if (!(s->alpha_sigma_global[0] > 0.0) || !(s->alpha_sigma_global[1] > 0.0 && s->alpha_sigma_global[1] < 1.0))
    return fail(h, MVG_EINVAL, "global hyperparameters out of range");
  std::vector<double> hyp(3 * c.V + 2);
  for (int v = 0; v < c.V; ++v) {
    hyp[v] = s->alpha_v[v];
    hyp[c.V + v] = s->sigma_v[v];
    hyp[2 * c.V + v] = s->tau_v[v];
  }
  hyp[3 * c.V] = s->alpha_sigma_global[0];
  hyp[3 * c.V + 1] = s->alpha_sigma_global[1];
  const uint32_t sweep = s->sweep ? *s->sweep : 0u;
  MVG_CUDA(h, cudaMemcpyAsync(c.choice, s->table_of, sizeof(int32_t) * (size_t)c.n_rows, cudaMemcpyHostToDevice, h->stream));
  MVG_CUDA(h, cudaMemcpyAsync(c.dish_of, s->dish_of, sizeof(int32_t) * (size_t)c.V * c.cap, cudaMemcpyHostToDevice, h->stream));
  MVG_CUDA(h, cudaMemcpyAsync(c.hyp, hyp.data(), sizeof(double) * hyp.size(), cudaMemcpyHostToDevice, h->stream));
  MVG_CUDA(h, cudaMemcpyAsync(c.sweep, &sweep, sizeof(sweep), cudaMemcpyHostToDevice, h->stream));
  MVG_CUDA(h, cudaMemsetAsync(c.birthmask, 0, sizeof(uint32_t) * (size_t)c.n_chunks, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));   // hyp/sweep are stack/vector temporaries
  if ((rc = rebuild_pipeline(h, 0, nullptr)) != MVG_OK) return rc;
  h->state_ready = true;
  return check_status(h);
}

// ---- binary checkpoint of the chain state (SURVEY.md §8 f4) ------------------------------------------------------
// File: "MVGCKPT1", then int64 {n_rows, V, cap, seed, chain, row_offset, n_rows_global, sweep}, then table_of int32[n_rows],
// dish_of int32[V*cap], hyp double[3V+2].  Everything else (counts, sums, parameters) is a function of these and of the
// data, and is rebuilt on load exactly as mvg_set_state rebuilds it.
namespace {
const char kCkptMagic[8] = {'M', 'V', 'G', 'C', 'K', 'P', 'T', '1'};
}

int mvg_save_checkpoint(mvg_handle* h, const char* path) {
  if (!h || !path) return MVG_EINVAL;
  if (!h->state_ready) return fail(h, MVG_ESTATE, "no state yet");
  const Ctx& c = h->c;
  std::vector<int32_t> tab((size_t)c.n_rows), dish((size_t)c.V * c.cap);
  std::vector<double> av(c.V), sv(c.V), tv(c.V);
  double ag[2];
  uint32_t sweep = 0;
  mvg_state_host st{};
  st.table_of = tab.data(); st.dish_of = dish.data(); st.alpha_v = av.data(); st.sigma_v = sv.data(); st.tau_v = tv.data();
  st.alpha_sigma_global = ag; st.sweep = &sweep;
  int rc = mvg_get_state(h, &st);
  if (rc != MVG_OK) return rc;
  FILE* f = fopen(path, "wb");
  if (!f) return fail(h, MVG_EINVAL, std::string("cannot open ") + path + " for writing");
  const int64_t hdr[8] = {c.n_rows, c.V, c.cap, (int64_t)c.seed, (int64_t)c.chain, c.row_offset, c.n_global, (int64_t)sweep};
  std::vector<double> hyp;
  hyp.insert(hyp.end(), av.begin(), av.end()); hyp.insert(hyp.end(), sv.begin(), sv.end()); hyp.insert(hyp.end(), tv.begin(), tv.end());
  hyp.push_back(ag[0]); hyp.push_back(ag[1]);
  bool ok = fwrite(kCkptMagic, 1, 8, f) == 8 && fwrite(hdr, sizeof(int64_t), 8, f) == 8 &&
            fwrite(tab.data(), sizeof(int32_t), tab.size(), f) == tab.size() &&
            fwrite(dish.data(), sizeof(int32_t), dish.size(), f) == dish.size() &&
            fwrite(hyp.data(), sizeof(double), hyp.size(), f) == hyp.size();
  if (ok && c.n_count_views) {       // count views: beta_v [V] follows (a dense-only file ends with the hyperparameters)
    std::vector<double> beta((size_t)c.V);
    rc = mvg_get_count_beta(h, beta.data());
    ok = rc == MVG_OK && fwrite(beta.data(), sizeof(double), beta.size(), f) == beta.size();
    if (rc != MVG_OK) { fclose(f); return rc; }
  }
  ok = (fclose(f) == 0) && ok;
  return ok ? MVG_OK : fail(h, MVG_EINVAL, std::string("short write to ") + path);
}

int mvg_load_checkpoint(mvg_handle* h, const char* path) {
  if (!h || !path) return MVG_EINVAL;
  const Ctx& c = h->c;
  FILE* f = fopen(path, "rb");
  if (!f) return fail(h, MVG_EINVAL, std::string("cannot open ") + path);
  char magic[8];
  int64_t hdr[8];
  std::vector<int32_t> tab((size_t)c.n_rows), dish((size_t)c.V * c.cap);
  std::vector<double> hyp((size_t)3 * c.V + 2);
  bool ok = fread(magic, 1, 8, f) == 8 && memcmp(magic, kCkptMagic, 8) == 0 && fread(hdr, sizeof(int64_t), 8, f) == 8;
  if (ok && (hdr[0] != c.n_rows || hdr[1] != c.V || hdr[2] != c.cap || hdr[5] != c.row_offset || hdr[6] != c.n_global)) {
    fclose(f);
    return fail(h, MVG_EINVAL, "checkpoint was written for another shape (n_rows, views, cap, shard)");
  }
  ok = ok && fread(tab.data(), sizeof(int32_t), tab.size(), f) == tab.size() &&
       fread(dish.data(), sizeof(int32_t), dish.size(), f) == dish.size() && fread(hyp.data(), sizeof(double), hyp.size(), f) == hyp.size();
  // a file of a handle with count views may carry their beta_v; one written before it did keeps the handle's
  std::vector<double> beta((size_t)c.V);
  bool has_beta = false;
  if (ok) {
    for (int v = 0; v < c.V; ++v) has_beta = has_beta || c.kind[v] != 0;
    has_beta = has_beta && fread(beta.data(), sizeof(double), beta.size(), f) == beta.size();
  }
  fclose(f);
  if (!ok) return fail(h, MVG_EINVAL, std::string("not a checkpoint or truncated: ") + path);
  if (has_beta)
    for (int v = 0; v < c.V; ++v)
      if (c.kind[v] && !(std::isfinite(beta[v]) && beta[v] > 0.0)) return fail(h, MVG_EINVAL, "checkpoint holds a non-positive count beta");
  uint32_t sweep = (uint32_t)hdr[7];
  mvg_state_host st{};
  st.table_of = tab.data(); st.dish_of = dish.data(); st.alpha_v = hyp.data(); st.sigma_v = hyp.data() + c.V; st.tau_v = hyp.data() + 2 * c.V;
  st.alpha_sigma_global = hyp.data() + 3 * c.V; st.sweep = &sweep;
  int rc = mvg_set_state(h, &st);
  if (rc != MVG_OK || !has_beta) return rc;
  // beta_v, then everything that depends on it, by the refresh that follows an accepted beta step (every count view)
  std::vector<int32_t> all((size_t)c.V);
  for (int v = 0; v < c.V; ++v) all[(size_t)v] = c.kind[v] ? 1 : 0;
  MVG_CUDA(h, cudaMemcpyAsync(c.beta_v, beta.data(), sizeof(double) * beta.size(), cudaMemcpyHostToDevice, h->stream));
  MVG_CUDA(h, cudaMemcpyAsync(c.cb_accept, all.data(), sizeof(int32_t) * all.size(), cudaMemcpyHostToDevice, h->stream));
  MVG_CUDA(h, launch_count_beta(c, 0, /*refresh_only=*/true, h->stream));
  h->launches += 2;
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));       // (host temporaries)
  return MVG_OK;
}

int mvg_get_state(mvg_handle* h, const mvg_state_host* o) {
  if (!h || !o) return MVG_EINVAL;
  if (!h->state_ready) return fail(h, MVG_ESTATE, "no state yet: call mvg_set_state or mvg_init_state_reference");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  const Ctx& c = h->c;
  const size_t vc = (size_t)c.V * c.cap;
  std::vector<double> hyp(3 * c.V + 2);
#define D2H(dst, src, bytes) if (dst) MVG_CUDA(h, cudaMemcpyAsync((dst), (src), (bytes), cudaMemcpyDeviceToHost, h->stream))
  D2H(o->table_of, c.table_cur, sizeof(int32_t) * (size_t)c.n_rows);
  D2H(o->n_t, c.n_t, sizeof(int32_t) * (size_t)c.cap);
  D2H(o->dish_of, c.dish_of, sizeof(int32_t) * vc);
  D2H(o->n_vk, c.n_vk, sizeof(int32_t) * vc);
  D2H(o->l_vk, c.l_vk, sizeof(int32_t) * vc);
  D2H(o->sum_y, c.S1k, sizeof(double) * (size_t)c.cap * c.Dsum);
  D2H(o->sum_y2, c.S2k, sizeof(double) * vc);
  D2H(o->sweep, c.sweep, sizeof(uint32_t));
  D2H(hyp.data(), c.hyp, sizeof(double) * hyp.size());
#undef D2H
  int rc = check_status(h);   // synchronises
  if (rc != MVG_OK) return rc;
  for (int v = 0; v < c.V; ++v) {
    if (o->alpha_v) o->alpha_v[v] = hyp[v];
    if (o->sigma_v) o->sigma_v[v] = hyp[c.V + v];
    if (o->tau_v) o->tau_v[v] = hyp[2 * c.V + v];
  }
  if (o->alpha_sigma_global) { o->alpha_sigma_global[0] = hyp[3 * c.V]; o->alpha_sigma_global[1] = hyp[3 * c.V + 1]; }
  return MVG_OK;
}

namespace {
// Is the next sweep an incremental one?  (Advances the rebuild schedule.)
bool next_sweep_is_delta(mvg_handle* h) {
  if (h->stats_mode != 1 || h->c.blk_count > 1 || !stats_delta_supported(h->c)) { h->since_full = 0; return false; }
  if (h->since_full + 1 >= h->rebuild_every) { h->since_full = 0; return false; }
  h->since_full += 1;
  return true;
}

int one_sweep(mvg_handle* h, int32_t flags, bool delta) {
  // A blocked sweep (mvg_set_sweep_blocks) is B passes: pass b redraws the rows of block b against statistics that
  // already contain the moves of blocks 0..b-1; the hyper step and the sweep counter belong to the last pass.
  const int B = h->c.blk_count;
  for (int b = 0; b < B; ++b) {
    h->c.blk_index = b;
    int rc = MVG_OK;
    if (!(h->draw_pending && B == 1)) { NvtxRange r("mvg:likelihood+draw"); rc = launch_draw(h); }
    h->draw_pending = false;
    if (rc != MVG_OK) return rc;
    { NvtxRange r("mvg:pack births"); MVG_CUDA(h, launch_pack(h->c, h->stream)); }
    h->launches += 1;
    rc = rebuild_pipeline(h, (b == B - 1) ? flags : kFinReseat, nullptr, delta && B == 1);
    if (rc != MVG_OK) return rc;
  }
  h->c.blk_index = 0;
  return MVG_OK;
}

// The sweep as it is captured: everything after the draw, then the draw of the NEXT sweep as the programmatic successor of
// k_finalize.
int sweep_tail_then_draw(mvg_handle* h, int32_t flags, bool delta) {
  { NvtxRange r("mvg:pack births"); MVG_CUDA(h, launch_pack(h->c, h->stream)); }
  h->launches += 1;
  int rc = rebuild_pipeline(h, flags, nullptr, delta);
  if (rc != MVG_OK) return rc;
  NvtxRange r("mvg:likelihood+draw (next sweep)");
  return launch_draw(h, /*programmatic=*/h->pdl_draw);
}

// Capture one sweep into an executable graph (once per handle and hyper-step variant).  Returns false, leaving the
// stream usable, if anything about the capture fails: the caller then launches the kernels directly.
bool ensure_sweep_graph(mvg_handle* h, int which, int32_t flags, bool delta) {
  if (h->sweep_graph[which]) return true;
  // (debug handles read back what the LAST draw exported: no draw of the next sweep may have run behind their back)
  if (!h->graphs_ok || h->c.debug_export != 0 || h->c.blk_count > 1) return false;
  // NCCL transport: launched directly (a collective captured into the sweep graph did not complete on this stack);
  // the peer-memory transport is an ordinary kernel and is captured with the rest of the sweep
  if (h->c.world != 1 && !h->xp2p) return false;
  static const bool disabled = [] { const char* e = getenv("MVG_NO_GRAPHS"); return e && e[0] == '1'; }();
  if (disabled) { h->graphs_ok = false; return false; }
  const int64_t before = h->launches;
  if (cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); h->graphs_ok = false; return false; }
  const int rc = sweep_tail_then_draw(h, flags, delta);
  cudaGraph_t g = nullptr;
  const cudaError_t e = cudaStreamEndCapture(h->stream, &g);
  h->sweep_graph_launches[which] = h->launches - before;
  h->launches = before;                                  // nothing has run yet
  if (rc != MVG_OK || e != cudaSuccess || !g) { if (g) cudaGraphDestroy(g); cudaGetLastError(); h->graphs_ok = false; return false; }
  cudaGraphExec_t ex = nullptr;
  const cudaError_t e2 = cudaGraphInstantiate(&ex, g, 0);
  cudaGraphDestroy(g);
  if (e2 != cudaSuccess || !ex) { cudaGetLastError(); h->graphs_ok = false; return false; }
  h->sweep_graph[which] = ex;
  return true;
}
}  // namespace

int mvg_sweep(mvg_handle* h, int32_t n_sweeps, int32_t do_hyper) {
  if (!h) return MVG_EINVAL;
  if (!h->state_ready) return fail(h, MVG_ESTATE, "no state yet: call mvg_set_state or mvg_init_state_reference");
  if (n_sweeps < 0) return fail(h, MVG_EINVAL, "n_sweeps < 0");
  if (h->host_fault && *reinterpret_cast<volatile int32_t*>(h->host_fault) != 0)
    return fail(h, MVG_ENCCL, "exchange fault (sticky): a peer's statistics did not arrive; no further sweeps on this handle");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  const int32_t flags = kFinReseat | kFinAdvance | (do_hyper ? kFinHyperAll : 0);
  MVG_CUDA(h, cudaEventRecord(h->ev[0], h->stream));
  for (int it = 0; it < n_sweeps; ++it) {
    const bool delta = next_sweep_is_delta(h);
    const int which = (do_hyper ? 1 : 0) + (delta ? 2 : 0);
    const bool use_graph = (n_sweeps >= 2 || h->sweeps_issued >= 1) && ensure_sweep_graph(h, which, flags, delta);
    if (use_graph) {
      if (!h->draw_pending) {                        // the first sweep of a run: its draw is not in flight yet
        NvtxRange r("mvg:likelihood+draw");
        const int rc = launch_draw(h);
        if (rc != MVG_OK) return rc;
      }
      NvtxRange r("mvg:sweep (graph replay)");
      MVG_CUDA(h, cudaGraphLaunch(h->sweep_graph[which], h->stream));
      h->launches += h->sweep_graph_launches[which];
      h->draw_pending = true;
    } else {
      const int rc = one_sweep(h, flags, delta);
      if (rc != MVG_OK) return rc;
    }
  }
  h->sweeps_issued += n_sweeps;
  MVG_CUDA(h, cudaEventRecord(h->ev[1], h->stream));
  return MVG_OK;
}

int mvg_set_stats_mode(mvg_handle* h, int32_t mode, int32_t rebuild_every) {
  if (!h) return MVG_EINVAL;
  if (mode != MVG_STATS_REBUILD && mode != MVG_STATS_INCREMENTAL) return fail(h, MVG_EINVAL, "unknown statistics mode");
  if (mode == MVG_STATS_INCREMENTAL && rebuild_every < 1) return fail(h, MVG_EINVAL, "rebuild_every must be >= 1");
  h->stats_mode = mode;
  h->rebuild_every = (mode == MVG_STATS_INCREMENTAL) ? rebuild_every : 1;
  h->since_full = 0x3fffffff;        // the next sweep rebuilds
  return MVG_OK;
}

int mvg_set_sweep_blocks(mvg_handle* h, int32_t blocks) {
  if (!h) return MVG_EINVAL;
  if (blocks < 1 || blocks > (1 << 20)) return fail(h, MVG_EINVAL, "blocks must be in [1, 2^20]");
  h->c.blk_count = blocks;
  h->c.blk_index = 0;
  invalidate_graphs(h);
  return MVG_OK;
}

int mvg_set_draw_screen(mvg_handle* h, int32_t on) {
  if (!h) return MVG_EINVAL;
  h->screen_want = on != 0;
  invalidate_graphs(h);                              // the switch is part of the captured kernel arguments
  if (h->c.scr) {
    h->c.screen = (h->screen_want && !h->c.debug_export) ? 1 : 0;
    MVG_CUDA(h, cudaSetDevice(h->cfg.device));
    return invalidate_screen(h);                     // margins recorded before a stretch without screening are stale
  }
  return MVG_OK;
}

int mvg_get_draw_screen_stats(mvg_handle* h, int32_t* enabled, int64_t* rows_screened, int64_t* tiles_evaluated) {
  if (!h) return MVG_EINVAL;
  if (enabled) *enabled = h->c.screen;
  if (rows_screened) *rows_screened = 0;
  if (tiles_evaluated) *tiles_evaluated = 0;
  if (!h->c.scr || !h->c.screen) return MVG_OK;
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  ScreenRec r;
  MVG_CUDA(h, cudaMemcpyAsync(&r, h->c.scr, sizeof(r), cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  if (rows_screened) *rows_screened = r.last_rows_screened;
  if (tiles_evaluated) *tiles_evaluated = r.last_tiles_evaluated;
  return MVG_OK;
}

int mvg_get_draw_rows(mvg_handle* h, int32_t* choice, int32_t* table_cur, uint32_t* birthmask, uint32_t* movedmask) {
  if (!h) return MVG_EINVAL;
  const Ctx& c = h->c;
  if (!c.choice) return fail(h, MVG_ESTATE, "no state yet");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  const size_t n = (size_t)c.n_rows, w = (size_t)c.n_chunks;
  if (choice) MVG_CUDA(h, cudaMemcpyAsync(choice, c.choice, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, h->stream));
  if (table_cur) MVG_CUDA(h, cudaMemcpyAsync(table_cur, c.table_cur, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, h->stream));
  if (birthmask) MVG_CUDA(h, cudaMemcpyAsync(birthmask, c.birthmask, sizeof(uint32_t) * w, cudaMemcpyDeviceToHost, h->stream));
  if (movedmask) MVG_CUDA(h, cudaMemcpyAsync(movedmask, c.movedmask, sizeof(uint32_t) * w, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  return MVG_OK;
}

int mvg_get_draw_screen_record(mvg_handle* h, mvg_screen_host* o) {
  if (!h || !o) return MVG_EINVAL;
  const Ctx& c = h->c;
  if (!c.scr) return fail(h, MVG_ESTATE, "no draw screening state (tensor-core engines, after the first state call)");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  const size_t vc = (size_t)c.V * c.cap;
  ScreenRec r;
  std::vector<TableParam> tp(vc);
  std::vector<TableMass> tm(c.cap);
  MVG_CUDA(h, cudaMemcpyAsync(&r, c.scr, sizeof(r), cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaMemcpyAsync(tp.data(), c.scr_tp, sizeof(TableParam) * vc, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaMemcpyAsync(tm.data(), c.scr_tm, sizeof(TableMass) * c.cap, cudaMemcpyDeviceToHost, h->stream));
  if (o->tiles)
    MVG_CUDA(h, cudaMemcpyAsync(o->tiles, c.scr_tiles, sizeof(int32_t) * (size_t)((c.n_rows + 127) / 128), cudaMemcpyDeviceToHost, h->stream));
  if (o->margin) MVG_CUDA(h, cudaMemcpyAsync(o->margin, c.margin, sizeof(float) * (size_t)c.n_rows, cudaMemcpyDeviceToHost, h->stream));
  if (o->ref_b) MVG_CUDA(h, cudaMemcpyAsync(o->ref_b, c.scr_b, sizeof(float) * 2 * (size_t)c.cap * c.Dsum, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  o->mode = r.mode;
  o->sweep = r.sweep;
  o->valid = r.valid;
  o->ref_sweep = r.ref_sweep;
  for (int i = 0; i < 7; ++i) o->k[i] = r.k[i];
  o->n_eval = r.n_eval;
  const mvg_params_host& p = o->ref;
  for (size_t i = 0; i < vc; ++i) {
    if (p.dish) p.dish[i] = tp[i].dish;
    if (p.A) p.A[i] = tp[i].A;
    if (p.C) p.C[i] = tp[i].C;
    if (p.A1) p.A1[i] = tp[i].A1;
    if (p.C1) p.C1[i] = tp[i].C1;
    if (p.lone) p.lone[i] = tp[i].lone;
  }
  for (int t = 0; t < c.cap; ++t) {
    if (p.LM) p.LM[t] = tm[t].LM;
    if (p.LM1) p.LM1[t] = tm[t].LM1;
  }
  return MVG_OK;
}

int mvg_hyper_step_parts(mvg_handle* h, int32_t parts) {
  if (!h) return MVG_EINVAL;
  if (!h->state_ready) return fail(h, MVG_ESTATE, "no state yet");
  if (parts & ~(MVG_HYPER_TAU | MVG_HYPER_LOCAL | MVG_HYPER_GLOBAL | MVG_HYPER_COUNT_BETA)) return fail(h, MVG_EINVAL, "unknown hyper part");
  if ((parts & MVG_HYPER_COUNT_BETA) && !h->c.cb_on) return fail(h, MVG_ESTATE, "no count beta prior set (mvg_set_count_beta_prior)");
  h->draw_pending = false;                           // the parameters are about to change
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  // rebuild the statistics of the current assignment, then the selected Metropolis-Hastings updates
  // (no draw, no reseat).  The sweep counter that addresses the Philox stream does not advance.
  MVG_CUDA(h, cudaMemcpyAsync(h->c.choice, h->c.table_cur, sizeof(int32_t) * (size_t)h->c.n_rows,
                              cudaMemcpyDeviceToDevice, h->stream));
  int32_t flags = kFinHyper;
  if (parts & MVG_HYPER_TAU) flags |= kFinHyperTau;
  if (parts & MVG_HYPER_LOCAL) flags |= kFinHyperLocal;
  if (parts & MVG_HYPER_GLOBAL) flags |= kFinHyperGlobal;
  if (parts & MVG_HYPER_COUNT_BETA) flags |= kFinHyperCountBeta;
  return rebuild_pipeline(h, flags, nullptr);
}

int mvg_hyper_step(mvg_handle* h) {
  if (!h) return MVG_EINVAL;
  return mvg_hyper_step_parts(h, MVG_HYPER_TAU | MVG_HYPER_LOCAL | MVG_HYPER_GLOBAL | (h->c.cb_on ? MVG_HYPER_COUNT_BETA : 0));
}

int mvg_sync(mvg_handle* h) {
  if (!h) return MVG_EINVAL;
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  if (h->host_fault && *reinterpret_cast<volatile int32_t*>(h->host_fault) != 0)
    return fail(h, MVG_ENCCL, "exchange fault (sticky): a peer's statistics did not arrive within the wait limit");
  return MVG_OK;
}

int mvg_clear_fault(mvg_handle* h) {
  if (!h) return MVG_EINVAL;
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  MVG_CUDA(h, cudaMemsetAsync(h->c.status, 0, sizeof(int32_t) * 4, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  if (h->host_fault) *h->host_fault = 0;
  return MVG_OK;
}

int mvg_run(mvg_handle* h, int32_t M, int32_t burn_in, int32_t thin, int32_t n_saved_max,
            int32_t* saved_table_of, int32_t* saved_dish_of, double* saved_hypers, double* saved_loglik, int32_t* n_saved) {
  if (!h) return MVG_EINVAL;
  if (M < 0 || thin <= 0) return fail(h, MVG_EINVAL, "M >= 0 and thin >= 1 required");
  const Ctx& c = h->c;
  int saved = 0;
  for (int iter = 0; iter < M; ++iter) {
    int rc = mvg_sweep(h, 1, 1);
    if (rc != MVG_OK) return rc;
    if (iter >= burn_in && ((iter - burn_in) % thin == 0)) {      // multiview_gibbs.cpp:205
      if (saved >= n_saved_max) return fail(h, MVG_EINVAL, "trace buffers too small");
      if (saved_table_of)
        MVG_CUDA(h, cudaMemcpyAsync(saved_table_of + (size_t)saved * c.n_rows, c.table_cur,
                                    sizeof(int32_t) * (size_t)c.n_rows, cudaMemcpyDeviceToHost, h->stream));
      if (saved_dish_of)
        MVG_CUDA(h, cudaMemcpyAsync(saved_dish_of + (size_t)saved * c.V * c.cap, c.dish_of,
                                    sizeof(int32_t) * (size_t)c.V * c.cap, cudaMemcpyDeviceToHost, h->stream));
      if (saved_hypers)
        MVG_CUDA(h, cudaMemcpyAsync(saved_hypers + (size_t)saved * (3 * c.V + 2), c.hyp,
                                    sizeof(double) * (size_t)(3 * c.V + 2), cudaMemcpyDeviceToHost, h->stream));
      if (h->saved_beta && c.beta_v)
        MVG_CUDA(h, cudaMemcpyAsync(h->saved_beta + (size_t)saved * c.V, c.beta_v, sizeof(double) * (size_t)c.V,
                                    cudaMemcpyDeviceToHost, h->stream));
      if (saved_loglik) {           // saved_loglik of the reference's state (multiview_state.h:38): filled on every kept sweep
        if (!h->loglik_dev) {
          void* q = nullptr;
          MVG_CUDA(h, cudaMalloc(&q, sizeof(double) * (size_t)(kMaxViews + 1)));
          h->owned.push_back(q);
          h->loglik_dev = static_cast<double*>(q);
        }
        MVG_CUDA(h, launch_loglik(c, h->loglik_dev, h->stream));
        h->launches += 1;
        MVG_CUDA(h, cudaMemcpyAsync(saved_loglik + saved, h->loglik_dev + c.V, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
      }
      ++saved;
    }
  }
  if (n_saved) *n_saved = saved;
  return check_status(h);
}

int mvg_comm_attach(mvg_handle* h, void* nccl_comm) {
  if (!h || !nccl_comm) return MVG_EINVAL;
  std::string err;
  if (!load_nccl(err)) return fail(h, MVG_ENCCL, err);
  h->comm = nccl_comm;
  h->comm_owned = false;
  return MVG_OK;
}

void* mvg_comm_handle(mvg_handle* h) { return h ? h->comm : nullptr; }

int mvg_comm_unique_id(void* unique_id_128) {
  std::string err;
  if (!unique_id_128) return MVG_EINVAL;
  if (!load_nccl(err)) return fail(nullptr, MVG_ENCCL, err);
  int r = g_nccl.GetUniqueId(unique_id_128);
  return r == 0 ? MVG_OK : fail(nullptr, MVG_ENCCL, "ncclGetUniqueId failed");
}

int mvg_comm_init_rank(mvg_handle* h, const void* unique_id_128) {
  if (!h || !unique_id_128) return MVG_EINVAL;
  std::string err;
  if (!load_nccl(err)) return fail(h, MVG_ENCCL, err);
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  UidByValue uid;
  std::memcpy(uid.internal, unique_id_128, 128);
  void* comm = nullptr;
  int r = g_nccl.CommInitRank(&comm, h->c.world, uid, h->c.rank);
  if (r != 0) return fail(h, MVG_ENCCL, std::string("ncclCommInitRank: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?"));
  h->comm = comm;
  h->comm_owned = true;
  return MVG_OK;
}

int mvg_prepare(mvg_handle* h) {
  if (!h) return MVG_EINVAL;
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  return ensure_layout(h);
}

int mvg_comm_p2p_export(mvg_handle* h, void* ipc_handle_64) {
  if (!h || !ipc_handle_64) return MVG_EINVAL;
  if (h->c.world < 2) return fail(h, MVG_EINVAL, "peer exchange needs world > 1");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  int rc = ensure_layout(h);                       // the slot size depends on the views
  if (rc != MVG_OK) return rc;
  if (!h->xrecv) {
    const XchgLayout L = xchg_layout(h->c);
    const size_t bytes = (size_t)2 * h->c.world * (size_t)L.slot_bytes;
    void* q = nullptr;
    if (cudaMalloc(&q, bytes) != cudaSuccess) return fail(h, MVG_ENOMEM, "cudaMalloc: exchange buffer");
    MVG_CUDA(h, cudaMemset(q, 0, bytes));          // flag 0 never equals a sequence number (they start at 1)
    h->xrecv = static_cast<unsigned char*>(q);
  }
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
  cudaIpcMemHandle_t hd;
  MVG_CUDA(h, cudaIpcGetMemHandle(&hd, h->xrecv));
  std::memcpy(ipc_handle_64, &hd, 64);
  return MVG_OK;
}

int mvg_comm_p2p_attach(mvg_handle* h, const void* all_handles) {
  if (!h || !all_handles) return MVG_EINVAL;
  if (!h->xrecv) return fail(h, MVG_ESTATE, "call mvg_comm_p2p_export first");
  if (h->xattached)
    return fail(h, MVG_ESTATE, "peer buffers are already attached (the mappings and the exchange sequence live until mvg_destroy; "
                               "use mvg_comm_p2p_enable to switch the transport back on)");
  if (h->c.world > 16) return fail(h, MVG_EUNSUPPORTED, "peer exchange supports at most 16 ranks");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  for (int g = 0; g < h->c.world; ++g) {
    if (g == h->c.rank) { h->xpeers.recv[g] = h->xrecv; continue; }
    cudaIpcMemHandle_t hd;
    std::memcpy(&hd, static_cast<const unsigned char*>(all_handles) + (size_t)g * 64, 64);
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      for (int q = 0; q < g; ++q)
        if (q != h->c.rank && h->xpeers.recv[q]) { cudaIpcCloseMemHandle(h->xpeers.recv[q]); h->xpeers.recv[q] = nullptr; }
      return fail(h, MVG_ECUDA, std::string("cudaIpcOpenMemHandle (rank ") + std::to_string(g) + "): " + cudaGetErrorString(e));
    }
    h->xpeers.recv[g] = static_cast<unsigned char*>(p);
  }
  h->xattached = true;
  h->xp2p = true;
  invalidate_graphs(h);                            // a captured sweep has the transport baked in
  return MVG_OK;
}

int mvg_comm_p2p_disable(mvg_handle* h) {
  if (!h) return MVG_EINVAL;
  h->xp2p = false;                                 // back to the NCCL transport; mappings and sequence number stay
  invalidate_graphs(h);
  return MVG_OK;
}

int mvg_comm_p2p_enable(mvg_handle* h) {
  if (!h) return MVG_EINVAL;
  if (!h->xattached) return fail(h, MVG_ESTATE, "no peer buffers attached: call mvg_comm_p2p_export / mvg_comm_p2p_attach");
  h->xp2p = true;                                  // the sequence number only advances with finalize: every rank is at the same one
  invalidate_graphs(h);
  return MVG_OK;
}

int mvg_get_params(mvg_handle* h, const mvg_params_host* o) {
  if (!h || !o) return MVG_EINVAL;
  if (!h->state_ready) return fail(h, MVG_ESTATE, "no state yet");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  const Ctx& c = h->c;
  const size_t vc = (size_t)c.V * c.cap;
  std::vector<TableParam> tp(vc);
  std::vector<ViewParam> vp(c.V);
  std::vector<TableMass> tm(c.cap);
  GlobalParam g;
  MVG_CUDA(h, cudaMemcpyAsync(tp.data(), c.tparam, sizeof(TableParam) * vc, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaMemcpyAsync(vp.data(), c.vparam, sizeof(ViewParam) * c.V, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaMemcpyAsync(tm.data(), c.tmass, sizeof(TableMass) * c.cap, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaMemcpyAsync(&g, c.gparam, sizeof(g), cudaMemcpyDeviceToHost, h->stream));
  if (o->m) MVG_CUDA(h, cudaMemcpyAsync(o->m, c.mean, sizeof(float) * (size_t)c.cap * c.Dsum, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  for (size_t i = 0; i < vc; ++i) {
    if (o->dish) o->dish[i] = tp[i].dish;
    if (o->A) o->A[i] = tp[i].A;
    if (o->C) o->C[i] = tp[i].C;
    if (o->A1) o->A1[i] = tp[i].A1;
    if (o->C1) o->C1[i] = tp[i].C1;
    if (o->W) o->W[i] = tp[i].W;
    if (o->W1) o->W1[i] = tp[i].W1;
    if (o->lone) o->lone[i] = tp[i].lone;
  }
  for (int v = 0; v < c.V; ++v) {
    if (o->AN) o->AN[v] = vp[v].AN;
    if (o->CN) o->CN[v] = vp[v].CN;
    if (o->WN) { o->WN[2 * v] = vp[v].WN0; o->WN[2 * v + 1] = vp[v].WN1; }
    if (o->LD) { o->LD[2 * v] = vp[v].LD0; o->LD[2 * v + 1] = vp[v].LD1; }
  }
  for (int t = 0; t < c.cap; ++t) {
    if (o->LM) o->LM[t] = tm[t].LM;
    if (o->LM1) o->LM1[t] = tm[t].LM1;
    if (o->single) o->single[t] = tm[t].single;
  }
  if (o->LMN) { o->LMN[0] = g.LMN0; o->LMN[1] = g.LMN1; }
  return MVG_OK;
}

int mvg_get_debug_rows(mvg_handle* h, float* acc, float* xx, int32_t* choice) {
  if (!h) return MVG_EINVAL;
  const Ctx& c = h->c;
  if (!(c.debug_export & 1) || !c.dbg_acc) return fail(h, MVG_ESTATE, "handle was not created with debug_export");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  const size_t N = (size_t)c.n_rows;
  if (acc) MVG_CUDA(h, cudaMemcpyAsync(acc, c.dbg_acc, sizeof(float) * N * c.V * c.cap, cudaMemcpyDeviceToHost, h->stream));
  if (xx) MVG_CUDA(h, cudaMemcpyAsync(xx, c.dbg_xx, sizeof(float) * N * c.V, cudaMemcpyDeviceToHost, h->stream));
  if (choice) MVG_CUDA(h, cudaMemcpyAsync(choice, c.dbg_choice, sizeof(int32_t) * N, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  return MVG_OK;
}

int mvg_get_debug_lnew(mvg_handle* h, float* lnew) {
  if (!h || !lnew) return MVG_EINVAL;
  if (!(h->c.debug_export & 1) || !h->c.dbg_lnew) return fail(h, MVG_ESTATE, "handle was not created with debug_export");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  MVG_CUDA(h, cudaMemcpyAsync(lnew, h->c.dbg_lnew, sizeof(float) * (size_t)h->c.n_rows, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  return MVG_OK;
}

int mvg_get_debug_births(mvg_handle* h, int32_t* n_seated, int64_t* rows, double* w) {
  if (!h) return MVG_EINVAL;
  const Ctx& c = h->c;
  if (!c.debug_export) return fail(h, MVG_ESTATE, "handle was not created with debug_export");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  if (n_seated) MVG_CUDA(h, cudaMemcpyAsync(n_seated, c.dbg_nseated, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
  if (rows) MVG_CUDA(h, cudaMemcpyAsync(rows, c.dbg_birth_rows, sizeof(int64_t) * (size_t)c.cap, cudaMemcpyDeviceToHost, h->stream));
  if (w) MVG_CUDA(h, cudaMemcpyAsync(w, c.dbg_birth_w, sizeof(double) * (size_t)c.cap * c.V * (c.cap + 1), cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  return MVG_OK;
}

int mvg_get_debug_prof(mvg_handle* h, int64_t* out, int32_t n_ctas) {
  if (!h || !out || n_ctas < 0 || n_ctas > 256) return MVG_EINVAL;
  if (!h->c.dbg_prof) return fail(h, MVG_ESTATE, "no profile buffer");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  MVG_CUDA(h, cudaMemcpyAsync(out, h->c.dbg_prof, sizeof(int64_t) * 16 * (size_t)n_ctas, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  return MVG_OK;
}

int mvg_last_sweep_ms(mvg_handle* h, float* ms_total) {
  if (!h || !ms_total) return MVG_EINVAL;
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  MVG_CUDA(h, cudaEventSynchronize(h->ev[1]));
  MVG_CUDA(h, cudaEventElapsedTime(ms_total, h->ev[0], h->ev[1]));
  return MVG_OK;
}

int mvg_kernel_clock(mvg_handle* h, int32_t which, double* total_ms, int64_t* launches, int64_t last_ns[3], int32_t reset) {
  if (!h || which < 0 || which >= kClockSlots) return MVG_EINVAL;
  if (!h->c.kclock) return fail(h, MVG_ESTATE, "no state yet");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  KClockSlot k;
  MVG_CUDA(h, cudaMemcpyAsync(&k, h->c.kclock + which, sizeof(k), cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  if (total_ms) *total_ms = (double)k.total_ns * 1e-6;
  if (launches) *launches = (int64_t)k.launches;
  if (last_ns) { last_ns[0] = (int64_t)k.last_start; last_ns[1] = (int64_t)k.last_end; last_ns[2] = (int64_t)k.prev_end; }
  if (reset) {
    MVG_CUDA(h, cudaMemsetAsync(h->c.kclock + which, 0, sizeof(k), h->stream));
    MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  }
  return MVG_OK;
}

int64_t mvg_launch_count(const mvg_handle* h) { return h ? h->launches : 0; }

int mvg_profile_sweep(mvg_handle* h, int32_t do_hyper, float ms_out[6]) {
  if (!h || !ms_out) return MVG_EINVAL;
  if (!h->state_ready) return fail(h, MVG_ESTATE, "no state yet");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  const int32_t flags = kFinReseat | kFinAdvance | (do_hyper ? kFinHyperAll : 0);
  h->draw_pending = false;                           // (the draw is a pure function of the state: run again under the events)
  MVG_CUDA(h, cudaEventRecord(h->ev[2], h->stream));
  int rc = launch_draw(h);
  if (rc != MVG_OK) return rc;
  MVG_CUDA(h, cudaEventRecord(h->ev[3], h->stream));
  MVG_CUDA(h, launch_pack(h->c, h->stream));
  h->launches += 1;
  MVG_CUDA(h, cudaEventRecord(h->ev[4], h->stream));
  cudaEvent_t marks[4];
  for (auto& m : marks) MVG_CUDA(h, cudaEventCreate(&m));
  rc = rebuild_pipeline(h, flags, marks, next_sweep_is_delta(h));
  if (rc == MVG_OK) {
    MVG_CUDA(h, cudaStreamSynchronize(h->stream));
    cudaEventElapsedTime(&ms_out[0], h->ev[2], h->ev[3]);
    cudaEventElapsedTime(&ms_out[1], h->ev[3], h->ev[4]);
    cudaEventElapsedTime(&ms_out[2], h->ev[4], marks[0]);
    cudaEventElapsedTime(&ms_out[3], marks[0], marks[1]);
    cudaEventElapsedTime(&ms_out[5], marks[1], marks[2]);
    cudaEventElapsedTime(&ms_out[4], marks[2], marks[3]);
    if (getenv("MVG_FIN_TWICE")) {     // experiment: the same kernel again right away (flags 0: idempotent) = warm instruction cache
      cudaEventRecord(marks[0], h->stream);
      launch_finalize(h->c, 0, h->stream);
      cudaEventRecord(marks[1], h->stream);
      cudaStreamSynchronize(h->stream);
      float warm = 0.f;
      cudaEventElapsedTime(&warm, marks[0], marks[1]);
      fprintf(stderr, "finalize cold %.4f ms (all flags), warm rerun %.4f ms (flags 0)\n", ms_out[4], warm);
    }
  }
  for (auto& m : marks) cudaEventDestroy(m);
  return rc;
}

void* mvg_stream(mvg_handle* h) { return h ? static_cast<void*>(h->stream) : nullptr; }

// ---- posterior summaries (kernels in mv_summary.cu) ---------------------------------------------
int mvg_log_likelihood(mvg_handle* h, double* total, double* per_view) {
  if (!h || !total) return MVG_EINVAL;
  if (!h->state_ready) return fail(h, MVG_ESTATE, "no state yet");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  double* d = nullptr;
  MVG_CUDA(h, cudaMalloc(&d, sizeof(double) * (h->c.V + 1)));
  cudaError_t e = launch_loglik(h->c, d, h->stream);
  std::vector<double> out(h->c.V + 1);
  if (e == cudaSuccess) e = cudaMemcpyAsync(out.data(), d, sizeof(double) * out.size(), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(d);
  if (e != cudaSuccess) return fail(h, MVG_ECUDA, std::string("log_likelihood: ") + cudaGetErrorString(e));
  h->launches += 1;
  *total = out[h->c.V];
  if (per_view) for (int v = 0; v < h->c.V; ++v) per_view[v] = out[v];
  return MVG_OK;
}

int mvg_cluster_labels(mvg_handle* h, int32_t* labels) {
  if (!h || !labels) return MVG_EINVAL;
  if (!h->state_ready) return fail(h, MVG_ESTATE, "no state yet");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  const size_t count = (size_t)h->c.V * h->c.n_rows;
  int32_t* d = nullptr;
  MVG_CUDA(h, cudaMalloc(&d, sizeof(int32_t) * count));
  cudaError_t e = launch_labels(h->c, d, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(labels, d, sizeof(int32_t) * count, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(d);
  if (e != cudaSuccess) return fail(h, MVG_ECUDA, std::string("cluster_labels: ") + cudaGetErrorString(e));
  h->launches += 1;
  return MVG_OK;
}

int mvg_coclustering_begin(mvg_handle* h, int32_t view) {
  if (!h) return MVG_EINVAL;
  if (view < -1 || view >= h->c.V) return fail(h, MVG_EINVAL, "view must be -1 (tables) or a view index");
  if (h->c.world != 1) return fail(h, MVG_EUNSUPPORTED, "co-clustering counts need the whole chain on one GPU (world = 1)");
  if (h->c.n_rows > 46340) return fail(h, MVG_EUNSUPPORTED, "co-clustering matrix limited to n_rows <= 46340 (n^2 counters)");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  const size_t bytes = sizeof(uint32_t) * (size_t)h->c.n_rows * h->c.n_rows;
  if (!h->cocl) {
    void* q = nullptr;
    if (cudaMalloc(&q, bytes) != cudaSuccess) return fail(h, MVG_ENOMEM, "cudaMalloc: co-clustering matrix");
    h->owned.push_back(q);
    h->cocl = static_cast<uint32_t*>(q);
  }
  MVG_CUDA(h, cudaMemsetAsync(h->cocl, 0, bytes, h->stream));
  h->cocl_view = view;
  h->cocl_samples = 0;
  return MVG_OK;
}

int mvg_coclustering_accumulate(mvg_handle* h) {
  if (!h) return MVG_EINVAL;
  if (!h->cocl || h->cocl_view < -1) return fail(h, MVG_ESTATE, "call mvg_coclustering_begin first");
  if (!h->state_ready) return fail(h, MVG_ESTATE, "no state yet");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  MVG_CUDA(h, launch_cocluster(h->c, h->cocl_view, h->cocl, h->stream));
  h->launches += 1;
  h->cocl_samples += 1;
  return MVG_OK;
}

int mvg_coclustering_get(mvg_handle* h, uint32_t* counts, int32_t* n_samples) {
  if (!h) return MVG_EINVAL;
  if (!h->cocl) return fail(h, MVG_ESTATE, "call mvg_coclustering_begin first");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  if (counts)
    MVG_CUDA(h, cudaMemcpyAsync(counts, h->cocl, sizeof(uint32_t) * (size_t)h->c.n_rows * h->c.n_rows, cudaMemcpyDeviceToHost, h->stream));
  MVG_CUDA(h, cudaStreamSynchronize(h->stream));
  if (n_samples) *n_samples = h->cocl_samples;
  return MVG_OK;
}

int mvg_adjusted_rand_index(mvg_handle* h, int32_t view, const int32_t* truth, int32_t n_classes, double* ari,
                            int32_t* contingency) {
  if (!h || !truth || !ari) return MVG_EINVAL;
  if (view < -1 || view >= h->c.V) return fail(h, MVG_EINVAL, "view must be -1 (tables) or a view index");
  if (n_classes <= 0 || n_classes > 65536) return fail(h, MVG_EINVAL, "n_classes out of range");
  if (!h->state_ready) return fail(h, MVG_ESTATE, "no state yet");
  for (int64_t i = 0; i < h->c.n_rows; ++i)
    if (truth[i] < 0 || truth[i] >= n_classes) return fail(h, MVG_EINVAL, "truth label outside [0, n_classes)");
  MVG_CUDA(h, cudaSetDevice(h->cfg.device));
  const size_t cells = (size_t)h->c.cap * n_classes;
  int32_t *d_truth = nullptr, *d_tab = nullptr;
  MVG_CUDA(h, cudaMalloc(&d_truth, sizeof(int32_t) * (size_t)h->c.n_rows));
  cudaError_t e = cudaMalloc(&d_tab, sizeof(int32_t) * cells);
  std::vector<int32_t> tab(cells);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_truth, truth, sizeof(int32_t) * (size_t)h->c.n_rows, cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_tab, 0, sizeof(int32_t) * cells, h->stream);
  if (e == cudaSuccess) e = launch_contingency(h->c, view, d_truth, n_classes, d_tab, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(tab.data(), d_tab, sizeof(int32_t) * cells, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(d_truth);
  cudaFree(d_tab);
  if (e != cudaSuccess) return fail(h, MVG_ECUDA, std::string("adjusted_rand_index: ") + cudaGetErrorString(e));
  h->launches += 1;
  // closed form from the contingency table (Hubert & Arabie), as mcclust::arandi computes it
  auto c2 = [](double x) { return 0.5 * x * (x - 1.0); };
  double sum_ij = 0.0, sum_a = 0.0, sum_b = 0.0, n = 0.0;
  std::vector<double> col(n_classes, 0.0);
  for (int k = 0; k < h->c.cap; ++k) {
    double a = 0.0;
    for (int z = 0; z < n_classes; ++z) {
      const double x = (double)tab[(size_t)k * n_classes + z];
      sum_ij += c2(x); a += x; col[z] += x;
    }
    sum_a += c2(a); n += a;
  }
  for (int z = 0; z < n_classes; ++z) sum_b += c2(col[z]);
  const double expected = (n > 1.0) ? sum_a * sum_b / c2(n) : 0.0;
  const double maxidx = 0.5 * (sum_a + sum_b);
  *ari = (maxidx - expected != 0.0) ? (sum_ij - expected) / (maxidx - expected) : 1.0;
  if (contingency) memcpy(contingency, tab.data(), sizeof(int32_t) * cells);
  return MVG_OK;
}

void mvg_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  U4 c{ctr[0], ctr[1], ctr[2], ctr[3]};
  const U4 r = philox4x32_10(c, key[0], key[1]);
  out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
}
float mvg_philox_uniform_f32(uint64_t seed, uint32_t chain, uint32_t domain, uint32_t slot, uint32_t sweep, uint64_t index) {
  return uniform_f32_from(stream_block(seed, chain, domain, slot, sweep, index).x);
}
double mvg_philox_uniform_f64(uint64_t seed, uint32_t chain, uint32_t domain, uint32_t slot, uint32_t sweep, uint64_t index) {
  const U4 r = stream_block(seed, chain, domain, slot, sweep, index);
  return uniform_f64_from(r.x, r.y);
}
double mvg_philox_normal(uint64_t seed, uint32_t chain, uint32_t domain, uint32_t slot, uint32_t sweep, uint64_t index) {
  const U4 r = stream_block(seed, chain, domain, slot, sweep, index);
  const double u1 = uniform_f64_from(r.x, r.y), u2 = uniform_f64_from(r.z, r.w);
  return sqrt(-2.0 * log(u1)) * cos(6.283185307179586476925286766559 * u2);
}

}  // extern "C"
