/* include/mvg.h — the C ABI of the B200-native allocation sweep (libmvg_b200.so).
 *
 * This is the drop-in boundary: the host-side C++ that keeps the reference's headers
 * (multiview-clustering_b200/host/multiview_{gibbs,state,hyper,utils,rng}.h) and any foreign
 * binding (Rcpp, ctypes — see INTEGRATION.md) reach CUDA only through these entry points.
 * extern "C", plain pointers and sizes, int status codes, no C++/torch/Rcpp types.
 *
 * Reference interface each entry point replaces (paths under /root/reference/Multiview):
 *
 *   mvg_create / mvg_destroy        the process-global chain state, multiview_state.h:21-45 and
 *                                   multiview_state.cpp:4-27 (one handle = one chain on one GPU)
 *   mvg_upload_view_*               the copy-in of run_gibbs_cpp, multiview_gibbs.cpp:109-115
 *   mvg_init_state_reference        initialize_state_from_data, multiview_gibbs.cpp:12-103
 *   mvg_set_state / mvg_get_state   direct reads/writes of table_of, dish_of, views[v].* and the
 *                                   hyperparameters (multiview_state.h:7-33)
 *   mvg_sweep                       the loop body of gibbs_sampler, multiview_gibbs.cpp:157-202:
 *                                   remove / score / draw / insert for every customer
 *                                   (multiview_utils.cpp:71-289, :307-350) followed by
 *                                   update_hyperparameters (multiview_hyper.cpp:233-292)
 *   mvg_hyper_step                  update_hyperparameters alone, multiview_hyper.h:18
 *   mvg_run                         gibbs_sampler(M, burn_in, thin) + save_state,
 *                                   multiview_gibbs.cpp:134-212, multiview_utils.cpp:291-303
 *   mvg_philox_*                    uniform01 / rnorm_scalar, multiview_utils.cpp:305-306 and the
 *                                   unused multiview_rng.h:9-24 (host mirror of the device stream)
 *
 * Semantics that differ from the reference BY DESIGN (DESIGN.md §2):
 *   - the sweep is synchronous: every customer is scored against the sweep-start statistics with
 *     only its own contribution removed, instead of seeing the moves of customers 0..i-1;
 *   - table and dish slots have a fixed capacity `cap` (32, 64, 128 or 256; the reference's pool has no limit); a new
 *     table can only open in a slot that was free at sweep start, births are seated in global row order and the
 *     overflow stays put;
 *   - the random stream is Philox4x32-10 addressed by (seed, chain, sweep, row, slot) instead of
 *     R's call-ordered generator;
 *   - a customer for whom NO option has weight stays at its own table; the reference seats it at table 0 without drawing
 *     (multiview_gibbs.cpp:172-176) — a slot index has no meaning across recycled slots;
 *   - mvg_set_sweep_blocks moves the sweep back towards the reference's sequential order; mvg_seq_run (MVG_ENGINE_SEQ) IS
 *     the reference's sampler, rule for rule, for its own scalar-view configuration (see below).
 *
 * Threading: a handle is not re-entrant; calls on one handle must be serialised by the caller.
 * Every call returns MVG_OK (0) or a negative MVG_E*; mvg_last_error gives the message.
 */
#ifndef MVG_H
#define MVG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MVG_ABI_VERSION 2

enum {
  MVG_OK = 0,
  MVG_EINVAL = -1,      /* bad argument or state that violates an invariant */
  MVG_ECUDA = -2,       /* a CUDA runtime call failed (message has the CUDA error string) */
  MVG_ENOMEM = -3,
  MVG_ESTATE = -4,      /* call out of order (e.g. sweep before all views are uploaded) */
  MVG_ENCCL = -5,
  MVG_EUNSUPPORTED = -6 /* shape outside what the kernels were built for */
};

enum {
  MVG_ENGINE_AUTO = 0,
  MVG_ENGINE_SIMT = 1,          /* FP32 CUDA cores; every FP32 operation mirrored by the CPU checker */
  MVG_ENGINE_TCGEN05 = 2,       /* tensor-core dot products (3-pass TF32), mirrored epilogue */
  MVG_ENGINE_TCGEN05_FAST = 3   /* same, weights through MUFU ex2.approx (tolerance-level weights) */
};
enum { MVG_VIEW_DENSE = 0, MVG_VIEW_CSR = 1 };

#define MVG_NEW_TABLE (-1)
#define MVG_MAX_VIEWS 16

typedef struct mvg_handle mvg_handle;   /* opaque */

typedef struct mvg_config {
  int32_t abi_version;     /* MVG_ABI_VERSION */
  int32_t device;          /* CUDA device ordinal */
  int64_t n_rows;          /* rows (customers) held by THIS handle (its shard) */
  int64_t n_rows_global;   /* customers over all shards; == n_rows on one GPU */
  int64_t row_offset;      /* global index of this shard's row 0 (Philox addressing, birth order) */
  int32_t n_views;         /* d in the reference */
  int32_t cap;             /* capacity of table slots and of dish slots per view: 32, 64, 128 or 256 (other values:
                              MVG_EUNSUPPORTED).  128 and 256 run on the CUDA-core engine only: MVG_ENGINE_AUTO picks
                              it, an explicit MVG_ENGINE_TCGEN05 / _FAST is MVG_EUNSUPPORTED */
  uint64_t seed;           /* Philox key (echo of set.seed(1999), New_Simulation.R:12) */
  uint32_t chain;          /* chain id, folded into the Philox key */
  int32_t engine;          /* MVG_ENGINE_* : which likelihood+draw kernel */
  int32_t debug_export;    /* bit 0: keep the per-row dot products of the last sweep for mvg_get_debug_*; bit 1: role wait counters */
  int32_t rank;            /* shard index 0..world-1 (0 on one GPU) */
  int32_t world;           /* number of shards (1 on one GPU) */
  int32_t reserved[5];
} mvg_config;

/* Host-side view of the chain state.  All pointers are HOST buffers owned by the caller; a NULL
 * pointer skips that field.  Sizes: V = n_views, cap, D_v = dim of view v, Dsum = sum of D_v. */
typedef struct mvg_state_host {
  int32_t* table_of;   /* [n_rows]   table slot of each local row                       (table_of) */
  int32_t* n_t;        /* [cap]      customers per table slot, 0 = free                 (n_t) */
  int32_t* dish_of;    /* [V*cap]    dish slot of table t in view v, -1 = free table    (dish_of[v][t]) */
  int32_t* n_vk;       /* [V*cap]    customers per dish slot                            (ViewState::n_vk) */
  int32_t* l_vk;       /* [V*cap]    tables per dish slot                               (ViewState::l_vk) */
  double* sum_y;       /* [cap*Dsum] per view v a [cap][D_v] block, views concatenated  (ViewState::sum_y) */
  double* sum_y2;      /* [V*cap]    sum of squared norms per dish slot                 (ViewState::sum_y2) */
  double* alpha_v;     /* [V] */
  double* sigma_v;     /* [V] */
  double* tau_v;       /* [V] */
  double* alpha_sigma_global;  /* [2] = {alpha_global, sigma_global} */
  uint32_t* sweep;     /* [1] index of the next sweep */
} mvg_state_host;

/* ---- lifetime ------------------------------------------------------------------------ */
int mvg_abi_version(void);
int mvg_create(const mvg_config* cfg, mvg_handle** out);
int mvg_destroy(mvg_handle* h);
const char* mvg_last_error(const mvg_handle* h);   /* h may be NULL: error of the last failed create */

/* ---- data ------------------------------------------------------------------------------ */
/* Dense view v, row-major [n_rows][dim] in HOST memory (pageable or pinned); copied to the GPU.
 * Numerical range: features are held and summed in FP32 (per-CTA partial sums in a fixed tree, FP64 across CTAs), and the
 * likelihood uses 2 x.m - |x|^2 in FP32; the reference works in double throughout.  The tolerances of the parity suite
 * (sums <= 1e-5, log-likelihoods <= 1e-5 of the cancelling terms) hold for views whose |mean| / sd is of order 10 or
 * less per coordinate (the prior mean of a dish is 0, multiview_utils.cpp:307-338); data with |mean| / sd ~ 100 loses
 * digits in S2 - |S1|^2 / n (the tau_v step) and should be centred per coordinate before upload. */
int mvg_upload_view_f32(mvg_handle* h, int32_t v, const float* x_host, int32_t dim);
/* Same from doubles, the type of the reference's y[v] (multiview_state.h:22); rounded to FP32. */
int mvg_upload_view_f64(mvg_handle* h, int32_t v, const double* y_host, int32_t dim);
/* Use a DEVICE buffer in place (row-major [n_rows][dim], 16-byte aligned); the caller keeps ownership. */
int mvg_attach_view_device_f32(mvg_handle* h, int32_t v, const float* x_dev, int32_t dim);

/* Sparse COUNT view v in CSR form, HOST buffers: rowptr int32[n_rows+1], col int32[nnz] in [0, vocab), val
 * float[nnz] holding non-negative integer counts (the bag-of-words views of dataset/reuters; SURVEY.md §8b).
 * The reference has no count likelihood: the model is the plug-in multinomial of SURVEY.md A.3 /
 * oracle/mv_oracle.c:counts_log_f_vk, log f_vk(x) = sum_w x_w log((beta + c_kw) / (W beta + C_k)) with the row's own
 * counts removed for its own dish.  One GPU per chain (world = 1); the CUDA-core engine is used. */
int mvg_upload_view_csr(mvg_handle* h, int32_t v, const int32_t* rowptr, const int32_t* col, const float* val,
                        int64_t nnz, int32_t vocab);
/* Symmetric Dirichlet pseudo-count beta of the count views (default 0.5); before the first state call. */
int mvg_set_count_beta(mvg_handle* h, double beta);
/* The likelihood of every count view of the handle (DESIGN.md §4.5):
 *   MVG_COUNT_PLUGIN (default)  the plug-in multinomial above;
 *   MVG_COUNT_DIRMULT           the exact collapsed conditional of a Dirichlet-multinomial mixture,
 *       log f_vk(x) = sum_w [lnΓ(beta + c_kw + x_w) - lnΓ(beta + c_kw)] - [lnΓ(W beta + C_k + n) - lnΓ(W beta + C_k)],
 *       n = sum_w x_w (c_kw, C_k without the row for its own dish; c = C = 0 for a new dish), so that the sweep samples
 *       the posterior of that model.  Counts must be non-negative integers (mvg_upload_view_csr checks it) and rows
 *       shorter than 2^24 tokens.
 * Like mvg_set_count_beta: before the first state call (afterwards MVG_ESTATE); another value is MVG_EINVAL.  A handle
 * that never calls it runs the plug-in kernels unchanged. */
enum { MVG_COUNT_PLUGIN = 0, MVG_COUNT_DIRMULT = 1 };
int mvg_set_count_likelihood(mvg_handle* h, int32_t model);
/* Learn beta: under MVG_COUNT_DIRMULT, every count view v gets its own beta_v (starting at mvg_set_count_beta's value)
 * and one Metropolis-Hastings step per hyper step (mvg_sweep with do_hyper, mvg_run, mvg_hyper_step) at the seating the
 * sweep ends with: prior beta_v ~ Gamma(shape, rate), proposal log beta' = log beta + step z, acceptance
 *   log A = L(beta') - L(beta) + shape (log beta' - log beta) - rate (beta' - beta),
 * L(beta) = sum over live dishes k of sum_w [lnΓ(beta + c_kw) - lnΓ(beta)] - [lnΓ(W beta + C_k) - lnΓ(W beta)].
 * z and the uniform u are Philox numbers of domain 7, slot v, index 0 (normal) and 1 (uniform), at the sweep index of the
 * same hyper step's tau draws (mvg_philox_normal / mvg_philox_uniform_f64 regenerate them).  Before the first state call;
 * non-finite or non-positive arguments: MVG_EINVAL; no count view, the plug-in model or after the first state call:
 * MVG_ESTATE.  Without it beta stays where mvg_set_count_beta put it. */
int mvg_set_count_beta_prior(mvg_handle* h, double shape, double rate, double step);
/* beta [V]: beta_v of every count view, 0 for a dense view.  Synchronises. */
int mvg_get_count_beta(mvg_handle* h, double* beta);
/* The most recent beta step (read-only; any pointer may be NULL): log_accept [V] its log A per count view, accepted [V]
 * 1 where it moved beta_v.  MVG_ESTATE without a prior or before the first state call.  Synchronises. */
int mvg_get_count_beta_step(mvg_handle* h, double* log_accept, int32_t* accepted);
/* Host buffer [n_saved_max][V] that later mvg_run calls fill with beta_v (as mvg_get_count_beta) on every kept sweep,
 * beside saved_hypers; NULL turns it off. */
int mvg_set_count_beta_trace(mvg_handle* h, double* saved_beta);

/* ---- state ----------------------------------------------------------------------------- */
int mvg_init_state_reference(mvg_handle* h);
/* Needs table_of, dish_of, alpha_v, sigma_v, tau_v, alpha_sigma_global (sweep optional); the
 * sufficient statistics are rebuilt on the device. */
int mvg_set_state(mvg_handle* h, const mvg_state_host* s);
int mvg_get_state(mvg_handle* h, const mvg_state_host* out);
/* Binary checkpoint of the chain state in a file (SURVEY.md §8 f4; the reference keeps its chain in process globals and has
 * no resume: multiview_state.cpp:4-16, multiview_gibbs.cpp:117): assignments, dish_of, hyperparameters, sweep counter,
 * and for a handle with count views their beta_v [V] after the hyperparameters (a file without it loads and keeps the
 * handle's beta).
 * Loading into a handle of the same shape with the same views restarts the chain bit-identically (statistics are rebuilt in
 * a fixed order, draws are addressed by (seed, sweep, row)); with the views of a row shard, each rank saves / loads its own file. */
int mvg_save_checkpoint(mvg_handle* h, const char* path);
int mvg_load_checkpoint(mvg_handle* h, const char* path);

/* ---- the hot path ---------------------------------------------------------------------- */
/* n_sweeps synchronous allocation sweeps, each followed by the hyper step when do_hyper != 0.
 * Asynchronous on the handle's stream; any mvg_get_* / mvg_sync observes the result. */
int mvg_sweep(mvg_handle* h, int32_t n_sweeps, int32_t do_hyper);
/* How the sufficient statistics follow the assignments.
 *   MVG_STATS_REBUILD (default)  every sweep re-reads all rows: a segmented reduction in a fixed order
 *                                (multiview_gibbs.cpp:64-73 for all rows), bit-reproducible from the assignments alone.
 *   MVG_STATS_INCREMENTAL        what the reference does per customer (remove_customer / add_customer_to_*,
 *                                multiview_utils.cpp:151-163, 199-206), batched per sweep: only the rows whose table
 *                                changed are re-read, added to their new table and subtracted from their old one, in a
 *                                fixed order, into running FP64 sums; every `rebuild_every`-th sweep is a full rebuild,
 *                                which bounds the rounding drift (counts are integers and exact either way).  The
 *                                sweep then streams the features ONCE instead of twice.  Available where the tile
 *                                statistics kernel is (cap 64, up to three dense views of dim 64); elsewhere (cap 32,
 *                                128, 256, other view shapes) it falls back to rebuilding. */
enum { MVG_STATS_REBUILD = 0, MVG_STATS_INCREMENTAL = 1 };
int mvg_set_stats_mode(mvg_handle* h, int32_t mode, int32_t rebuild_every);
/* Blocked sweeps: one sweep becomes `blocks` passes; pass b redraws the customers with (global row) % blocks == b
 * against statistics that already hold the moves of passes 0..b-1 (statistics rebuild and birth/death bookkeeping after
 * every pass, the hyper step after the last).  blocks = 1 (default) is the synchronous sweep; blocks = N is the
 * reference's sequential order (multiview_gibbs.cpp:157-200) — the knob trades throughput for closeness to it.
 * The Philox addressing (sweep, row) is unchanged, so chains stay reproducible and shard-invariant. */
int mvg_set_sweep_blocks(mvg_handle* h, int32_t blocks);
/* Draw screening (tensor-core engines; on by default there, ignored by the CUDA-core engine and by debug handles).  Before every draw a
 * screening kernel tests, for every row, a stored lower bound on how far its own table leads every other table; a tile of
 * 128 rows that all lead by more than 2^31 in weight gets its draw (its own table) written without reading its features.
 * The bound is exact: a chain draws the same tables with screening on or off.  It applies to sweeps with every table slot
 * live and every dish served by one table; other sweeps evaluate every row.  Switching it changes no state. */
int mvg_set_draw_screen(mvg_handle* h, int32_t on);
/* What screening did in the most recent draw: enabled (0/1), rows whose draw was screened, row tiles (128 rows) the draw
 * evaluated.  Any pointer may be NULL.  Synchronises. */
int mvg_get_draw_screen_stats(mvg_handle* h, int32_t* enabled, int64_t* rows_screened, int64_t* tiles_evaluated);
int mvg_hyper_step(mvg_handle* h);
/* The same restricted to some of its Metropolis-Hastings updates: update_tau_v_MH alone
 * (multiview_hyper.cpp:211-231), the per-view alpha/sigma pairs (:242-265), the franchise pair (:268-291), the beta step
 * of the count views (mvg_set_count_beta_prior; without a prior MVG_ESTATE).  mvg_hyper_step includes the beta step when
 * a prior is set. */
enum { MVG_HYPER_TAU = 1, MVG_HYPER_LOCAL = 2, MVG_HYPER_GLOBAL = 4, MVG_HYPER_COUNT_BETA = 8 };
int mvg_hyper_step_parts(mvg_handle* h, int32_t parts);
int mvg_sync(mvg_handle* h);
/* gibbs_sampler(M, burn_in, thin): M sweeps; after sweep `iter` with iter >= burn_in and
 * (iter - burn_in) % thin == 0 the state is appended to the caller's trace buffers
 * (save rule of multiview_gibbs.cpp:205).  Buffers hold n_saved_max entries each:
 * table_of [S][n_rows], dish_of [S][V*cap], hypers [S][3V+2] = alpha_v, sigma_v, tau_v, alpha_g, sigma_g, loglik [S] =
 * mvg_log_likelihood of the kept state (the reference declares saved_loglik, multiview_state.h:38, and never fills it).
 * NULL buffers are skipped.  Returns the number of saved states in *n_saved. */
int mvg_run(mvg_handle* h, int32_t M, int32_t burn_in, int32_t thin, int32_t n_saved_max,
            int32_t* saved_table_of, int32_t* saved_dish_of, double* saved_hypers, double* saved_loglik, int32_t* n_saved);

/* ---- multi-GPU (row-sharded) -------------------------------------------------------------- */
/* Attach an initialised NCCL communicator (ncclComm_t passed as void*) whose rank/size match the
 * config.  Without one, world must be 1.  The library issues one all-gather per sweep on it. */
int mvg_comm_attach(mvg_handle* h, void* nccl_comm);
/* The communicator this handle uses (ncclComm_t as void*, NULL if none): several handles of one process (chains,
 * or a second run over the same ranks) can share it through mvg_comm_attach; its owner must outlive the borrowers. */
void* mvg_comm_handle(mvg_handle* h);
/* Convenience for callers without their own NCCL: unique_id is the 128-byte ncclUniqueId made by
 * mvg_comm_unique_id on rank 0 and distributed by the caller (e.g. over torch.distributed/gloo). */
int mvg_comm_unique_id(void* unique_id_128);
int mvg_comm_init_rank(mvg_handle* h, const void* unique_id_128);

/* Peer-memory transport for the same exchange (optional, one node): instead of reduce + ncclAllGather + sum, ONE kernel
 * (csrc/mv_exchange.cu) stores every reduced value straight into its peers' receive buffers over NVLink as 8-byte
 * {payload, sequence number} words and adds the peers' words in rank order as they arrive; the results are bit-identical
 * to the NCCL transport.  With it the whole sweep is one CUDA graph also for world > 1.
 * Setup, after the views are known: every rank calls mvg_comm_p2p_export (a 64-byte cudaIpcMemHandle_t comes back), the
 * caller all-gathers the handles in rank order and gives the world x 64 bytes to mvg_comm_p2p_attach on every rank (once
 * per handle: the mappings and the exchange sequence number live until mvg_destroy; a second attach is MVG_ESTATE).
 * mvg_comm_p2p_disable / mvg_comm_p2p_enable switch between this transport and NCCL; every rank must switch at the same
 * point of the chain.
 * Failure: a peer whose words do not arrive within 2 s (%globaltimer) raises a STICKY fault on this handle: the device
 * publishes nothing further (the chain stays frozen at this rank's last completed sweep), mvg_sweep refuses to queue
 * more work and mvg_sync / mvg_get_state / mvg_run return MVG_ENCCL.  mvg_clear_fault re-arms the handle once the
 * caller has brought the ranks back to a common state (e.g. mvg_set_state on every rank). */
int mvg_prepare(mvg_handle* h);                       /* fix the layout now (all views uploaded/attached) */
int mvg_comm_p2p_export(mvg_handle* h, void* ipc_handle_64);
int mvg_comm_p2p_attach(mvg_handle* h, const void* all_handles);
int mvg_comm_p2p_disable(mvg_handle* h);              /* back to the NCCL transport (e.g. a peer failed to attach) */
int mvg_comm_p2p_enable(mvg_handle* h);               /* peer-memory transport again (mappings are kept) */
int mvg_clear_fault(mvg_handle* h);

/* ---- inspection (tests, profiling) ----------------------------------------------------- */
/* The FP32 parameter block of the NEXT sweep, as the likelihood kernel will read it; pointers
 * are host buffers, NULL skips.  Layouts are those of oracle/mv_oracle.h:mvo_params_f32. */
typedef struct mvg_params_host {
  int32_t* dish; float* A; float* C; float* A1; float* C1; float* W; float* W1; int32_t* lone;
  float* AN; float* CN; float* WN; float* LD; float* LM; float* LM1; int32_t* single; float* LMN;
  float* m;     /* [cap*Dsum]: per view a [cap][D_v] block of per-table means, views concatenated */
} mvg_params_host;
int mvg_get_params(mvg_handle* h, const mvg_params_host* out);
/* Draw screening (tensor-core engines, DESIGN.md §4.1.1): what the most recent draw's screening decided and what it left
 * behind, read without changing it.  mode is that of the most recent screened draw (0 off, 1 refresh, 2 skip) and sweep the
 * sweep it belongs to: after a replayed sweep that is the next sweep's draw, already issued (mvg_get_state's sweep); after a
 * sweep launched directly, the sweep before.  valid / ref_sweep: whether a reference stands and the sweep it was taken at.
 * k: the coefficients of the row bound that draw used (k0, kA[3], kB[3]; not written by a draw in off mode).  n_eval and
 * tiles: the tile list of a skip draw (first n_eval entries meaningful).  margin: the per-row margins as they stand.  ref:
 * the reference parameter block (dish, A, C, A1, C1, lone, LM, LM1 filled; the other pointers are ignored) and ref_b its
 * [2][cap*Dsum] mean_hi, mean_lo.  Host buffers; NULL skips.  Synchronises; MVG_ESTATE on a handle without screening
 * state (CUDA-core engine, or before the first state call).  For tests: nothing here is needed to run a chain. */
typedef struct mvg_screen_host {
  int32_t mode;
  uint32_t sweep;
  uint32_t valid, ref_sweep;
  float k[7];
  int32_t n_eval;
  int32_t* tiles;      /* [ceil(n_rows/128)] */
  float* margin;       /* [n_rows] */
  mvg_params_host ref;
  float* ref_b;        /* [2][cap*Dsum] */
} mvg_screen_host;
int mvg_get_draw_screen_record(mvg_handle* h, mvg_screen_host* out);
/* Read-only: the draw's per-row buffers as the most recent sweep left them: choice [n_rows] (the draw, a seated birth -2),
 * table_cur [n_rows] (the seating), birthmask and movedmask [ceil(n_rows/32)] (bit r of word w: row 32 w + r drew a new
 * table / a table other than its own).  Any pointer may be NULL. */
int mvg_get_draw_rows(mvg_handle* h, int32_t* choice, int32_t* table_cur, uint32_t* birthmask, uint32_t* movedmask);
/* With debug_export: per-row stage-A outputs of the LAST sweep: acc [n_rows][V][cap] dot products
 * x.m and xx [n_rows][V] squared norms, plus the raw draw (before births are seated) [n_rows].  A count view: acc is
 * log2 f under each table's dish and xx what the new-dish term read, the token total (plug-in) or -log2 f_new
 * (MVG_COUNT_DIRMULT). */
int mvg_get_debug_rows(mvg_handle* h, float* acc, float* xx, int32_t* choice);
/* Tensor-core engines, with debug_export: acc above holds the dot products with the PRE-SCALED means b = 2 A m (the data
 * term of log2 f), and lnew [n_rows] the log2 weight of a new table as the kernel evaluated it (MUFU log-sum-exp: a float
 * statistic inside the stated tolerance; the CPU mirror checks it and draws from it). */
int mvg_get_debug_lnew(mvg_handle* h, float* lnew);
/* Count view v: the tables of the NEXT sweep, host [vocab][cap] each (NULL skips): log2 theta of the dish each
 * table slot serves, that dish's word counts, and the word counts per table slot.  Under MVG_COUNT_DIRMULT the first
 * output holds log2(beta + c) of the dish's count c instead of log2 theta. */
int mvg_get_count_tables(mvg_handle* h, int32_t v, float* log2_theta, int32_t* dish_counts, int32_t* table_counts);
/* MVG_COUNT_DIRMULT, count view v: *n_max = its longest row in tokens (any model; den may be NULL), and den (host
 * [n_max+1][cap], length-major) the denominator table of the NEXT sweep, den[n][t] = sum_{j<n} log2(W beta + C_k + j)
 * of the dish k table slot t serves (0 for a free slot), formed in FP64 and rounded once.  den under the plug-in model:
 * MVG_ESTATE. */
int mvg_get_count_den(mvg_handle* h, int32_t v, float* den, int32_t* n_max);
/* With debug_export, count views: loo [n_rows][V] leave-one-out log2 f of every row under its own dish (LAST sweep). */
int mvg_get_debug_loo(mvg_handle* h, float* loo);
/* Births of the LAST sweep: rows (global index) seated at new tables in order, and the
 * V*(cap+1) max-normalised dish weights each saw.  rows holds cap entries, w cap*V*(cap+1). */
int mvg_get_debug_births(mvg_handle* h, int32_t* n_seated, int64_t* rows, double* w);
/* With debug_export & 2 (tcgen05 engines): cycles each role of the draw kernel spent waiting on its
 * barriers during the LAST sweep, 16 counters per CTA (layout: csrc/mv_draw_tc.cu). */
int mvg_get_debug_prof(mvg_handle* h, int64_t* out, int32_t n_ctas);
/* Device time of the last mvg_sweep call's kernels, by CUDA events on the handle's stream (ms). */
int mvg_last_sweep_ms(mvg_handle* h, float* ms_total);
/* Number of kernel launches the library issued since the handle was created. */
int64_t mvg_launch_count(const mvg_handle* h);
/* In-kernel wall clocks of the tensor-core draw kernel (which = 0) and of the finalize kernel (which = 1): every launch adds
 * the time from its first CTA in (the draw: from the moment its grid dependency resolved) to its last CTA out, read from
 * %globaltimer.  total_ms / launches accumulate since the last reset; they also cover launches replayed from a CUDA graph,
 * where events cannot be placed (bench.py times the kernels of the very sweeps it reports this way).  last_ns (may be NULL):
 * absolute %globaltimer values {start, end} of the most recent launch and {end} of the one before.  Synchronises. */
int mvg_kernel_clock(mvg_handle* h, int32_t which, double* total_ms, int64_t* launches, int64_t last_ns[3], int32_t reset);
/* Per-kernel device time of the most recent sweep measured with CUDA events (ms):
 * [0] likelihood+draw, [1] pack, [2] stats, [3] reduce, [4] finalize, [5] collective. */
int mvg_profile_sweep(mvg_handle* h, int32_t do_hyper, float ms_out[6]);
/* The CUDA stream (cudaStream_t as void*) all work of this handle is issued on. */
void* mvg_stream(mvg_handle* h);

/* ---- posterior summaries (SURVEY.md §8 f2; what New_Simulation.R does with the trace) ------ */
/* Joint log marginal likelihood of the data given the current partition: the sum over live dishes of the
 * reference's log p(y_S) (multiview_utils.cpp:316-320, per coordinate).  This is what the reference's
 * declared-but-never-defined compute_log_likelihood() (multiview_gibbs.h:13) / saved_loglik
 * (multiview_state.h:38) would hold.  per_view: [V] or NULL.  A count view under MVG_COUNT_DIRMULT contributes the
 * collapsed marginal of the partition up to the multinomial coefficients (which do not depend on it):
 *   sum over live dishes k of  sum_w [lnΓ(beta + c_kw) - lnΓ(beta)] - lnΓ(W beta + C_k) + lnΓ(W beta). */
int mvg_log_likelihood(mvg_handle* h, double* total, double* per_view);
/* Cluster of every customer in every view, dish_of[v][table_of[i]]: get_final_clusters of
 * New_Simulation.R:135-149.  labels: host [V][n_rows]. */
int mvg_cluster_labels(mvg_handle* h, int32_t* labels);
/* Co-clustering (posterior similarity) counts kept on the device: begin zeroes an [n_rows][n_rows] uint32
 * matrix for `view` (-1: tables), accumulate adds [label_i == label_j] for the current state, get copies
 * the counts and the number of accumulated states out.  One GPU holds the whole chain (world = 1). */
int mvg_coclustering_begin(mvg_handle* h, int32_t view);
int mvg_coclustering_accumulate(mvg_handle* h);
int mvg_coclustering_get(mvg_handle* h, uint32_t* counts, int32_t* n_samples);
/* Adjusted Rand index of the current clustering of `view` (-1: tables) against host labels
 * truth[n_rows] in [0, n_classes): mcclust::arandi of New_Simulation.R:189.  contingency (optional, host
 * [cap][n_classes]) receives the Predicted x Truth table of :192-196.  With world > 1 both are this shard's. */
int mvg_adjusted_rand_index(mvg_handle* h, int32_t view, const int32_t* truth, int32_t n_classes, double* ari,
                            int32_t* contingency);

/* ---- MVG_ENGINE_SEQ: the reference-exact sequential sampler (csrc/mv_seq_core.h, csrc/mv_seq.cu) ------------------
 * run_gibbs_cpp(data_views, M, burn_in, thin) of multiview_gibbs.cpp:105-131 for scalar views, every rule of the reference
 * kept (customers re-seated one after the other, unbounded table / dish slots, swap-with-last deletion, dish slots never
 * recycled, FP64, the reference's operation order) on the call-ordered Philox stream the compiled reference is driven with
 * in oracle/refshim: given the same data and seed the chain visits the same integer states as the unmodified reference.
 * One device thread per chain: the anchor for the reference's own configuration (N ~ 500), not a throughput path.
 * y: host [d][n] doubles.  t_cap / k_cap: capacities of the table and dish-slot arrays (dish slots are never recycled by the
 * reference: k_cap ~ 2 + sweeps is safe).  Outputs (host, NULL skips): saved_table_of [S][n] (0-based, dense),
 * saved_T [S], saved_dish_of [S][d][t_cap] (first saved_T[s] entries of every row valid), saved_hypers [S][3d+2]
 * (alpha_v, sigma_v, tau_v, alpha_global, sigma_global), *n_saved, *stream_calls (uniforms + normals consumed). */
int mvg_seq_run(int32_t device, int32_t n, int32_t d, const double* y, int32_t M, int32_t burn_in, int32_t thin,
                uint64_t seed, int32_t t_cap, int32_t k_cap, int32_t n_saved_max, int32_t* saved_table_of,
                int32_t* saved_T, int32_t* saved_dish_of, double* saved_hypers, int32_t* n_saved,
                uint64_t* stream_calls);
const char* mvg_seq_last_error(void);

/* ---- Philox host mirror (multiview_rng.h surface) ---------------------------------------- */
void mvg_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
float mvg_philox_uniform_f32(uint64_t seed, uint32_t chain, uint32_t domain, uint32_t slot,
                             uint32_t sweep, uint64_t index);
double mvg_philox_uniform_f64(uint64_t seed, uint32_t chain, uint32_t domain, uint32_t slot,
                              uint32_t sweep, uint64_t index);
double mvg_philox_normal(uint64_t seed, uint32_t chain, uint32_t domain, uint32_t slot,
                         uint32_t sweep, uint64_t index);

#ifdef __cplusplus
}
#endif
#endif /* MVG_H */
