// multiview_state.h — host-side chain state of the B200 sampler.
//
// Same declarations as the reference's header (/root/reference/Multiview/multiview_state.h:7-45):
// struct ViewState with its nine members and the process-global chain state, so that code written
// against the reference (the Rcpp glue, New_Simulation.R through it, inspection code) keeps compiling.
// Here these globals are a MIRROR: the chain lives in HBM behind the C ABI (include/mvg.h) and is copied
// into them by mvhost::pull_state() — after initialisation, on every saved sweep and at the end of
// gibbs_sampler().  Labels are compacted on the way out: live table slots become 0..T-1 and live dish
// slots of view v become 0..K-1 in slot order, the dense labelling the reference maintains.
#ifndef MULTIVIEW_STATE_H
#define MULTIVIEW_STATE_H

#include <vector>

struct ViewState {
  int K = 0;                                        // live dishes of this view
  std::vector<int> n_vk;                            // customers per dish
  std::vector<int> l_vk;                            // tables per dish
  std::vector<double> sum_y;                        // K x D sums (D = 1: one value per dish)
  std::vector<double> sum_y2;                       // sum of squared norms per dish
  std::vector<std::vector<int>> customers_at_dish;  // membership lists, ascending customer index

  double alpha_v = 1.0;                             // local concentration
  double sigma_v = 0.5;                             // local discount
  double tau_v = 1.0;                               // kernel variance
};

extern int n, d;                                    // customers, views
extern std::vector<std::vector<double>> y;          // y[v][i*D_v + j]: view v of customer i (D_v = 1 in the reference)

extern double alpha_global;                         // franchise concentration
extern double sigma_global;                         // franchise discount

extern int T;                                       // live tables
extern std::vector<int> table_of;                   // table of each customer, 0-based
extern std::vector<int> n_t;                        // customers per table
extern std::vector<std::vector<int>> customers_at_table;
extern std::vector<std::vector<int>> dish_of;       // dish_of[v][t]

extern std::vector<ViewState> views;

// saved trace (returned to R by run_gibbs_cpp)
extern std::vector<std::vector<int>> saved_table_of;
extern std::vector<std::vector<std::vector<int>>> saved_dish_of;
extern std::vector<double> saved_loglik;
extern std::vector<std::vector<double>> saved_alpha_v;
extern std::vector<std::vector<double>> saved_sigma_v;
extern std::vector<std::vector<double>> saved_tau_v;
extern std::vector<double> saved_alpha_global;
extern std::vector<double> saved_sigma_global;

// ---- additions (not in the reference): the device chain behind the mirror -------------------------
struct mvg_handle;
namespace mvhost {
extern int table_capacity;          // table / dish slots per view on the device (32, 64, 128 or 256; default 64)
extern unsigned long long seed;     // Philox key (set.seed(1999) of New_Simulation.R:12 by default)
extern int engine;                  // MVG_ENGINE_* (0 = automatic)
extern std::vector<int> view_dim;   // D_v; empty = all 1 (the reference's scalar views)
struct CsrView { std::vector<int> rowptr, col; std::vector<float> val; int vocab = 0; };
extern std::vector<CsrView> csr_views;   // csr_views[v].vocab > 0: view v is a sparse COUNT view (a dgCMatrix in data_views), y[v] is empty
extern bool sequential;             // true: run_gibbs_cpp uses MVG_ENGINE_SEQ, the reference-exact sequential sampler (scalar views)
mvg_handle* chain();                // the live device chain or nullptr
void open_chain();                  // create the handle from n, d, y, view_dim and upload the views
void close_chain();
void pull_state();                  // device -> the globals above (compacted labels)
[[noreturn]] void fail(const char* where);   // raises the last device error (Rcpp::stop in the R build)
}  // namespace mvhost

#endif  // MULTIVIEW_STATE_H
