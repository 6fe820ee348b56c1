/* oracle/mv_oracle_dm.c — TEST INFRASTRUCTURE (CPU oracle), not product code.
 *
 * The Dirichlet-multinomial count likelihood (MVG_COUNT_DIRMULT of include/mvg.h), restated next to the plug-in one of
 * mv_oracle.c.  Every function takes the same mvo_state; a count view is scored by the exact collapsed conditional
 *   log f_vk(x) = sum_w [lgamma(beta + c_kw + x_w) - lgamma(beta + c_kw)] - [lgamma(W beta + C_k + n) - lgamma(W beta + C_k)]
 * (n = |x|, the row removed first for its own dish, c = C = 0 for a new dish) by libm lgamma in FP64 — independent of
 * the device's lgamma_diff — and dense views exactly as mv_oracle.c scores them.  The draw, the reseat (births) and the
 * marginal likelihood use it.  mvod_stageA_counts_f32 is the FP32 mirror of the device's k_counts_loglik_dm.
 * Built by oracle/pydirmult.py (gcc -ffp-contract=off, linked with mv_oracle.c); mv_oracle.c itself is not changed.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "mv_oracle.h"
#include "mv_philox_ref.h"

#ifdef _OPENMP
#include <omp.h>
#endif

static int is_counts(const mvo_state* s, int v) { return s->csr != NULL && s->csr[v].rowptr != NULL; }

double mvod_counts_log_f_vk(const mvo_state* s, int v, int k, int i, int loo) {
  const mvo_csr* cs = &s->csr[v];
  const double beta = s->count_beta;
  double tot = 0.0, lf = 0.0;
  for (int j = cs->rowptr[i]; j < cs->rowptr[i + 1]; ++j) {
    const double x = (double)cs->val[j];
    const double c = (double)cs->cd[(size_t)k * cs->vocab + cs->col[j]] - (loo ? x : 0.0);
    lf += lgamma(beta + c + x) - lgamma(beta + c);
    tot += x;
  }
  const double C = (double)cs->vocab * beta + (double)cs->ctot[k] - (loo ? tot : 0.0);
  return lf - (lgamma(C + tot) - lgamma(C));
}

double mvod_counts_log_f_new(const mvo_state* s, int v, int i) {
  const mvo_csr* cs = &s->csr[v];
  const double beta = s->count_beta, wbeta = (double)cs->vocab * beta;
  double tot = 0.0, lf = 0.0;
  for (int j = cs->rowptr[i]; j < cs->rowptr[i + 1]; ++j) {
    const double x = (double)cs->val[j];
    lf += lgamma(beta + x) - lgamma(beta);
    tot += x;
  }
  return lf - (lgamma(wbeta + tot) - lgamma(wbeta));
}

/* The collapsed marginal of the current partition up to the multinomial coefficients:
 * sum over live dishes k of sum_w [lgamma(beta + c_kw) - lgamma(beta)] - lgamma(W beta + C_k) + lgamma(W beta). */
double mvod_log_marginal_counts(const mvo_state* s, int v) {
  const mvo_csr* cs = &s->csr[v];
  const double beta = s->count_beta, wbeta = (double)cs->vocab * beta;
  double lm = 0.0;
  for (int k = 0; k < s->cap; ++k) {
    if (s->n_vk[(size_t)v * s->cap + k] <= 0) continue;
    for (int w = 0; w < cs->vocab; ++w) {
      const int64_t c = cs->cd[(size_t)k * cs->vocab + w];
      if (c > 0) lm += lgamma(beta + (double)c) - lgamma(beta);
    }
    lm -= lgamma(wbeta + (double)cs->ctot[k]) - lgamma(wbeta);
  }
  return lm;
}

static double row_log_f_vk(const mvo_state* s, int v, int k, int i, int loo) {
  if (is_counts(s, v)) return mvod_counts_log_f_vk(s, v, k, i, loo);
  return mvo_log_f_vk(s, v, k, s->x[v] + (size_t)i * s->D[v], loo);
}
static double row_log_f_new(const mvo_state* s, int v, int i) {
  if (is_counts(s, v)) return mvod_counts_log_f_new(s, v, i);
  return mvo_log_f_new(s, v, s->x[v] + (size_t)i * s->D[v]);
}

static double lse2(double a, double b) {
  if (a == -INFINITY) return b;
  if (b == -INFINITY) return a;
  double m = a > b ? a : b;
  return m + log(exp(a - m) + exp(b - m));
}

/* mv_oracle.c:log_marginal_new_table with this file's likelihood */
static double log_marginal_new_table(const mvo_state* s, int v, int i, int t0, double* lf, double lf_new) {
  const int cap = s->cap;
  const int32_t* l_vk = s->l_vk + (size_t)v * cap;
  const int k0 = s->dish_of[(size_t)v * cap + t0];
  const int single = (s->n_t[t0] == 1);
  const double alpha = s->alpha_v[v], sigma = s->sigma_v[v];
  double total_tables = 0.0;
  int K_active = 0;
  double acc = -INFINITY;
  for (int k = 0; k < cap; ++k) {
    int l = l_vk[k] - ((single && k == k0) ? 1 : 0);
    lf[k] = -INFINITY;
    if (l <= 0) continue;
    total_tables += (double)l;
    K_active++;
    lf[k] = row_log_f_vk(s, v, k, i, k == k0);
    double w = (double)l - sigma;
    if (w > 0.0) acc = lse2(acc, log(w) + lf[k]);
  }
  double denominator = alpha + total_tables;
  if (denominator <= 0.0) return lf_new;
  double w_new = alpha + (double)K_active * sigma;
  if (w_new > 0.0) acc = lse2(acc, log(w_new) + lf_new);
  return acc - log(denominator);
}

/* mv_oracle.c:mvo_row_logweights with this file's likelihood */
int mvod_row_logweights(const mvo_state* s, int i, double* lw, double* Lvt) {
  const int cap = s->cap, V = s->V;
  const int t0 = s->table_of[i];
  const int single = (s->n_t[t0] == 1);
  double* lf = (double*)malloc(sizeof(double) * (size_t)cap);
  int T_nonempty = 0, F = 0;
  for (int t = 0; t < cap; ++t) {
    if (s->n_t[t] > 0) T_nonempty++; else F++;
    lw[t] = 0.0;
  }
  double log_new = 0.0;
  for (int v = 0; v < V; ++v) {
    double lf_new = row_log_f_new(s, v, i);
    log_new += log_marginal_new_table(s, v, i, t0, lf, lf_new);
    for (int t = 0; t < cap; ++t) {
      int k = s->dish_of[(size_t)v * cap + t];
      double val = (k >= 0) ? lf[k] : -INFINITY;
      lw[t] += val;
      if (Lvt) Lvt[(size_t)v * (cap + 1) + t] = val;
    }
    if (Lvt) Lvt[(size_t)v * (cap + 1) + cap] = lf_new;
  }
  for (int t = 0; t < cap; ++t) {
    int nt = s->n_t[t] - (t == t0 ? 1 : 0);
    double mass = (double)nt - s->sigma_g;
    if (nt <= 0 || mass <= 0.0) lw[t] = -INFINITY;
    else lw[t] += log(mass);
  }
  double mass_new = s->alpha_g + s->sigma_g * (double)(T_nonempty - single);
  if (mass_new <= 0.0 || F == 0) lw[cap] = -INFINITY;
  else lw[cap] = log(mass_new) + log_new;
  free(lf);
  return 0;
}

int mvod_draw_rows(const mvo_state* s, int32_t* choice, int threads) {
  const int cap = s->cap;
  if (threads <= 0) threads = 1;
#ifdef _OPENMP
#pragma omp parallel num_threads(threads)
#endif
  {
    double* lw = (double*)malloc(sizeof(double) * (size_t)(cap + 1));
#ifdef _OPENMP
#pragma omp for schedule(static)
#endif
    for (int i = 0; i < s->n; ++i) {
      mvod_row_logweights(s, i, lw, NULL);
      double u = (double)mvo_uniform_f32(s->seed, s->chain, MVO_DOM_TABLE, 0, s->sweep, (uint64_t)(s->row_offset + i));
      choice[i] = mvo_draw_from_logweights(s, i, lw, u);
    }
    free(lw);
  }
  return 0;
}

/* mv_oracle.c:sample_dish_birth with this file's likelihood */
static int sample_dish_birth(const mvo_state* s, int v, int b, const int32_t* l_live, double* w_out) {
  const int cap = s->cap;
  const int t0 = s->table_of[b];
  const int k0 = s->dish_of[(size_t)v * cap + t0];
  const int single = (s->n_t[t0] == 1);
  const double alpha = s->alpha_v[v], sigma = s->sigma_v[v];
  double* lwt = (double*)malloc(sizeof(double) * (size_t)(cap + 1));
  int K_active = 0;
  double M = -INFINITY;
  for (int k = 0; k < cap; ++k) {
    int l = l_live[k] - ((single && k == k0) ? 1 : 0);
    lwt[k] = -INFINITY;
    if (l <= 0) continue;
    K_active++;
    double w = (double)l - sigma;
    if (w <= 0.0) continue;
    lwt[k] = log(w) + row_log_f_vk(s, v, k, b, (k == k0) && s->n_vk[(size_t)v * cap + k] > 0);
    if (lwt[k] > M) M = lwt[k];
  }
  double w_new = alpha + sigma * (double)K_active;
  lwt[cap] = (w_new > 0.0) ? log(w_new) + row_log_f_new(s, v, b) : -INFINITY;
  if (lwt[cap] > M) M = lwt[cap];
  int pick = -1;
  if (M > -INFINITY) {
    double total = 0.0;
    for (int k = 0; k <= cap; ++k) {
      double w = (lwt[k] == -INFINITY) ? 0.0 : exp(lwt[k] - M);
      if (w_out) w_out[k] = w;
      total += w;
    }
    double u = mvo_uniform53(s->seed, s->chain, MVO_DOM_DISH, (uint32_t)v, s->sweep, (uint64_t)(s->row_offset + b)) * total;
    double cum = 0.0;
    for (int k = 0; k < cap; ++k) {
      if (lwt[k] == -INFINITY) continue;
      cum += exp(lwt[k] - M);
      if (u < cum) { pick = k; break; }
    }
  } else if (w_out) {
    for (int k = 0; k <= cap; ++k) w_out[k] = 0.0;
  }
  free(lwt);
  if (pick >= 0) return pick;
  for (int k = 0; k < cap; ++k) if (l_live[k] == 0) return k;
  return -1;
}

/* mv_oracle.c:mvo_reseat with this file's likelihood */
int mvod_reseat(mvo_state* s, const int32_t* choice, int32_t* n_seated, int32_t* birth_rows, double* birth_w) {
  const int cap = s->cap, V = s->V;
  int32_t* free_slots = (int32_t*)malloc(sizeof(int32_t) * (size_t)cap);
  int32_t* l_live = (int32_t*)malloc(sizeof(int32_t) * (size_t)V * cap);
  int32_t* new_table = (int32_t*)malloc(sizeof(int32_t) * (size_t)s->n);
  int32_t* new_dish = (int32_t*)malloc(sizeof(int32_t) * (size_t)V * cap);
  int F = 0, seated = 0;
  for (int t = 0; t < cap; ++t) if (s->n_t[t] == 0) free_slots[F++] = t;
  memcpy(l_live, s->l_vk, sizeof(int32_t) * (size_t)V * cap);
  memcpy(new_dish, s->dish_of, sizeof(int32_t) * (size_t)V * cap);
  for (int i = 0; i < s->n; ++i) {
    if (choice[i] != MVO_NEW) { new_table[i] = choice[i]; continue; }
    if (seated >= F) { new_table[i] = s->table_of[i]; continue; }
    int tn = free_slots[seated];
    new_table[i] = tn;
    for (int v = 0; v < V; ++v) {
      double* w_out = birth_w ? birth_w + ((size_t)seated * V + v) * (cap + 1) : NULL;
      int k = sample_dish_birth(s, v, i, l_live + (size_t)v * cap, w_out);
      if (k < 0) { free(free_slots); free(l_live); free(new_table); free(new_dish); return 3; }
      new_dish[(size_t)v * cap + tn] = k;
      l_live[(size_t)v * cap + k]++;
    }
    if (birth_rows) birth_rows[seated] = i;
    seated++;
  }
  if (n_seated) *n_seated = seated;
  memcpy(s->table_of, new_table, sizeof(int32_t) * (size_t)s->n);
  memcpy(s->dish_of, new_dish, sizeof(int32_t) * (size_t)V * cap);
  free(free_slots); free(l_live); free(new_table); free(new_dish);
  return mvo_rebuild_stats(s);
}

/* FP32 mirror of k_counts_loglik_dm (multiview-clustering_b200/csrc/mv_counts.cu), from the device's tables: l2c
 * [vocab][cap] log2(beta + c), cdt [vocab][cap] dish word counts, den [n_max+1][cap] sum_{j<n} log2(W beta + C_k + j);
 * n = the row's token total (ascending FP32 sum).  Per table t:
 *   a = 0;  per nonzero j ascending with x_j > 0: s = l2c[w_j][t]; s += log2m((beta + c) + i), i = 1 .. x_j - 1;  a += s;
 *   acc[t] = a - den[n][t].
 * Own dish t0, leave-one-out: per nonzero term_j = sum_{i < x_j} log2m((beta + (c - x_j)) + i) (i ascending), summed in
 * nonzero order; minus ld = the 32-lane sum of log2m((wbeta_plus_ctot - n) + j), lane l taking j = l, l + 32, ...
 * ascending, combined by an xor butterfly over offsets 16, 8, 4, 2, 1 (lane 0's value).  Must be compiled with
 * -ffp-contract=off. */
void mvod_stageA_counts_f32(const int32_t* col, const float* val, int nnz, const float* l2c, const int32_t* cdt,
                            const float* den, int cap, int t0, float beta, float wbeta_plus_ctot, float* acc, float* acc_loo) {
  float tot = 0.0f;
  for (int j = 0; j < nnz; ++j) tot = tot + val[j];
  const int n = (int)tot;
  for (int t = 0; t < cap; ++t) {
    float a = 0.0f;
    for (int j = 0; j < nnz; ++j) {
      const int x = (int)val[j];
      if (x == 0) continue;                                  /* a stored zero count adds nothing */
      float sv = l2c[(size_t)col[j] * cap + t];
      const float bc = beta + (float)cdt[(size_t)col[j] * cap + t];
      for (int i = 1; i < x; ++i) sv = sv + mvo_log2m(bc + (float)i);
      a = a + sv;
    }
    acc[t] = a + (-den[(size_t)n * cap + t]);
  }
  const float lbase = wbeta_plus_ctot + (-tot);
  float lane[32];
  for (int l = 0; l < 32; ++l) {
    float p = 0.0f;
    for (int j = l; j < n; j += 32) p = p + mvo_log2m(lbase + (float)j);
    lane[l] = p;
  }
  for (int o = 16; o > 0; o >>= 1) {
    float nxt[32];
    for (int l = 0; l < 32; ++l) nxt[l] = lane[l] + lane[l ^ o];
    memcpy(lane, nxt, sizeof(lane));
  }
  float a = 0.0f;
  for (int j = 0; j < nnz; ++j) {
    const int x = (int)val[j];
    const float b0 = beta + (float)(cdt[(size_t)col[j] * cap + t0] - x);
    float term = 0.0f;
    for (int i = 0; i < x; ++i) term = term + mvo_log2m(b0 + (float)i);
    a = a + term;
  }
  *acc_loo = a + (-lane[0]);
}
