// mv_counts.cu — sufficient statistics and per-sweep tables of the sparse COUNT views (CSR).
//
// The reference has no count likelihood (SURVEY.md §0, A.3): this is new capability, parity pinned only to the
// FP64 restatement in oracle/mv_oracle.c (counts_log_f_vk).  Model: the rows of a dish are draws of one
// multinomial whose probabilities are the plug-in estimate theta_kw = (beta + c_kw) / (W beta + C_k) from the
// dish's word counts; log f_vk(x) = sum_w x_w log theta_kw, the row's own counts removed for its own dish.
//
//   k_rowtotals       |x| of every row, once per upload (kept in the squared-norm slot of the view)
//   k_counts_scatter  word counts per TABLE slot: cnt_t[w][t] += x_w over the rows seated at t — from scratch after a
//                     state upload, otherwise only for the rows that changed table since the last call.  Integer
//                     atomics: the sums are exact and independent of the order (north_star: integer counts
//                     bit-exact)
//   k_counts_tables   per (word, table slot): the counts of the DISH the slot serves (sum over the slots of that
//                     dish, ascending) and log2 theta, the table the likelihood kernel reads feature-major
//
// MVG_COUNT_DIRMULT (opt-in, DESIGN.md §4.5) replaces the plug-in by the exact collapsed conditional of a
// Dirichlet-multinomial mixture, log f_vk(x) = sum_w [lnΓ(beta + c_kw + x_w) - lnΓ(beta + c_kw)]
// - [lnΓ(W beta + C_k + n) - lnΓ(W beta + C_k)], n = |x| (oracle/mv_oracle_dm.c:mvod_counts_log_f_vk): the same
// scatter and tables with log2(beta + c) cells plus a per-slot denominator table, and k_counts_loglik_dm for stage A.
#include "mv_ctx.h"

namespace mv {

constexpr double kLog2eD = 1.4426950408889634074;

__global__ void k_rowtotals(const int32_t* __restrict__ rowptr, const float* __restrict__ val, float* __restrict__ out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float tot = 0.0f;
  for (int j = rowptr[i]; j < rowptr[i + 1]; ++j) tot = __fadd_rn(tot, val[j]);   // ascending: the mirror's order
  out[i] = tot;
}

// blockIdx.y-th count view of the chain
__device__ __forceinline__ int nth_count_view(const Ctx& c, int nth) {
  int v = 0;
  for (; v < c.V; ++v)
    if (c.kind[v] && nth-- == 0) break;
  return v;
}

// delta: cnt_t is current for the seating table_prev; only the rows that changed table since are visited — their words
// leave the old slot and join the new one (the reference's remove_customer / add_customer bookkeeping,
// multiview_utils.cpp:151-163, 199-206, batched).  Integer atomics either way: exact, order-independent.
__global__ void k_counts_scatter(const Ctx c, const int delta) {
  const int v = nth_count_view(c, blockIdx.y);
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const int32_t* __restrict__ rp = c.rowptr[v];
  const int32_t* __restrict__ col = c.col[v];
  const float* __restrict__ val = c.val[v];
  int32_t* cnt = c.cnt_t[v];
  for (int i = warp; i < c.n_rows; i += nwarps) {
    const int t = c.table_cur[i];
    const int p = delta ? c.table_prev[i] : -1;
    if (delta && p == t) continue;
    for (int j = rp[i] + lane; j < rp[i + 1]; j += 32) {
      const int32_t x = (int32_t)val[j];
      atomicAdd(&cnt[(size_t)col[j] * c.cap + t], x);
      if (p >= 0) atomicAdd(&cnt[(size_t)col[j] * c.cap + p], -x);
    }
  }
}

// MAXCAP: 64 (one mask word per slot) or 256; cap is a power of two <= MAXCAP.
// DM (MVG_COUNT_DIRMULT): the cell is log2(beta + cd) instead of log2 theta, and the denominator table follows the cells.
// gate != null: the refresh after a beta step (launch_count_beta): only the views whose step accepted (gate[v] != 0) run,
// with the new beta_v; the same cells and denominators, and TableParam::C1 of the view's live tables.
template <int MAXCAP, bool DM>
__global__ void k_counts_tables(const Ctx c, const int log2cap, const int32_t* __restrict__ gate) {
  constexpr int kWords = MAXCAP / 64;
  const int v = nth_count_view(c, blockIdx.y);
  if (gate && gate[v] == 0) return;
  const double beta = c.beta_v[v];
  __shared__ int32_t s_dish[MAXCAP];
  __shared__ double s_den[MAXCAP];
  __shared__ float s_l2zero[MAXCAP];                         // log2 theta of a word the dish has never seen: most cells of the table
  __shared__ unsigned long long s_mask[MAXCAP][kWords];      // the table slots serving the same dish as slot t
  const int cap = c.cap;
  if (threadIdx.x < cap) {
    const int k = c.dish_of[v * cap + threadIdx.x];
    s_dish[threadIdx.x] = k;
    // S2k of a count view holds the token total of the dish (an exact integer)
    s_den[threadIdx.x] = (k >= 0) ? count_wbeta_total(c.vocab[v], beta, c.S2k[v * cap + k]) : 1.0;
    if constexpr (DM) s_l2zero[threadIdx.x] = (float)log2(beta);
    else s_l2zero[threadIdx.x] = (float)log2((beta + 0.0) / s_den[threadIdx.x]);   // the cell expression at cd = 0
    // (k_finalize wrote C1 by the same expression at the beta it saw)
    if (gate && blockIdx.x == 0 && k >= 0) c.tparam[v * cap + threadIdx.x].C1 = (float)s_den[threadIdx.x];
  }
  __syncthreads();
  if (threadIdx.x < cap) {
    const int k = s_dish[threadIdx.x];
#pragma unroll
    for (int wi = 0; wi < kWords; ++wi) {
      unsigned long long m = 0ull;
      if (k >= 0) for (int j = 0; j < 64 && 64 * wi + j < cap; ++j) if (s_dish[64 * wi + j] == k) m |= 1ull << j;
      s_mask[threadIdx.x][wi] = m;
    }
    s_mask[threadIdx.x][threadIdx.x >> 6] &= ~(1ull << (threadIdx.x & 63));   // the slot itself is read first
  }
  __syncthreads();
  // (every view's scatter has read table_prev by now — this kernel follows it in the stream: the seating the counts now
  //  stand for is the current one)
  if (!gate && blockIdx.y == 0)
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < c.n_rows; i += gridDim.x * blockDim.x) c.table_prev[i] = c.table_cur[i];
  const size_t total = (size_t)c.vocab[v] * cap;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const int t = (int)(e & (size_t)(cap - 1));             // cap is a power of two (mvg_create): no 64-bit division per cell
    const size_t w = e >> log2cap;
    int32_t cd = 0;
    float l2 = 0.0f;
    if (s_dish[t] >= 0) {
      const int32_t* row = c.cnt_t[v] + w * cap;
      cd = row[t];                                              // usually the dish's only table
#pragma unroll
      for (int wi = 0; wi < kWords; ++wi)
        for (unsigned long long m = s_mask[t][wi]; m; m &= m - 1ull) cd += row[64 * wi + __ffsll((long long)m) - 1];
      if constexpr (DM) l2 = (cd == 0) ? s_l2zero[t] : (float)log2(beta + (double)cd);
      else l2 = (cd == 0) ? s_l2zero[t] : (float)log2((beta + (double)cd) / s_den[t]);
    }
    c.cnt_d[v][e] = cd;
    c.l2t[v][e] = l2;
  }
  if constexpr (DM) {
    // den[n][t] = sum_{j<n} log2(W beta + C_k + j) for every row length n <= n_max, in FP64 (lgamma_diff), rounded once
    const size_t dcells = (size_t)(c.cnt_nmax[v] + 1) * cap;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < dcells; e += (size_t)gridDim.x * blockDim.x) {
      const int t = (int)(e & (size_t)(cap - 1));
      const int n = (int)(e >> log2cap);
      c.cnt_den[v][e] = (s_dish[t] >= 0) ? (float)(kLog2eD * lgamma_diff(s_den[t], n)) : 0.0f;
    }
  }
}

// MVG_COUNT_DIRMULT, at the first state call and again whenever beta_v moves (the rows never change):
// q[i] = -log2 f_new(x_i) = -(sum_w lnΓ(beta + x_w) - lnΓ(beta)  -  [lnΓ(W beta + n) - lnΓ(W beta)]) / ln 2, FP64, ascending
// over the row's nonzeros, rounded once.  The draw's new-dish term reads it where the plug-in reads the token total.
// gate as in k_counts_tables.
__global__ void k_counts_newdish(const Ctx c, const int32_t* __restrict__ gate) {
  const int v = nth_count_view(c, blockIdx.y);
  if (gate && gate[v] == 0) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c.n_rows) return;
  const double beta = c.beta_v[v];
  double lf = 0.0;
  int n = 0;
  for (int j = c.rowptr[v][i]; j < c.rowptr[v][i + 1]; ++j) {
    const int x = (int)c.val[v][j];
    lf += lgamma_diff(beta, x);
    n += x;
  }
  lf -= lgamma_diff((double)c.vocab[v] * beta, n);
  c.cnt_q[v][i] = (float)(-kLog2eD * lf);
}

// Stage A of a count view: log2 f of every row under every table slot's dish, acc[i][t] = sum_j x_j l2t[col_j][t], and
// the leave-one-out value under the row's own dish.  One WARP per row (a thread per row would make the longest row
// everybody's wait): lane l owns tables l*PER .. l*PER+PER-1, the row's nonzeros are read 32 at a time and broadcast,
// eight table rows are in flight at once; per table the chain is ascending over the nonzeros, the order
// oracle/mv_oracle.c:mvo_stageA_counts_f32 restates.  Document lengths are heavy-tailed (Reuters bodies: 1 .. several
// hundred distinct words) and there are only two or three rows per warp, so the rows are dealt out by descending
// length (row_order, built at upload): every warp gets one long, one middling and one short row instead of whatever
// its index happens to hold.  The table is feature-major: one nonzero reads CAP consecutive
// floats (the SpMM "CSR row x dense feature-major table" of SURVEY.md A.3).
template <int CAP>
__global__ void __launch_bounds__(512) k_counts_loglik(const Ctx c) {
  const int v = nth_count_view(c, blockIdx.y);
  constexpr int PER = CAP / 32;
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const int32_t* __restrict__ rp = c.rowptr[v];
  const int32_t* __restrict__ colv = c.col[v];
  const float* __restrict__ valv = c.val[v];
  const float* __restrict__ l2t = c.l2t[v];
  const int32_t* __restrict__ cdt = c.cnt_d[v];
  const TableParam* __restrict__ tp = c.tparam + v * CAP;
  const int32_t* __restrict__ order = c.row_order[v];
  const float beta = (float)c.beta_v[v];
  constexpr int kFlight = 8;                         // table rows in flight per warp
  for (int ri = warp; ri < c.n_rows; ri += nwarps) {
    const int row = order ? __ldg(order + ri) : ri;
    const int j0 = rp[row], j1 = rp[row + 1];
    const int t0 = c.table_cur[row];
    // leave-one-out under the own dish: counts and total with this row removed (TableParam::C1 of a count view
    // carries W beta + the dish's token total)
    const float lden = log2m(__fadd_rn(tp[t0].C1, -c.xx[(size_t)v * c.xx_stride + row]));
    float a[PER];
#pragma unroll
    for (int q = 0; q < PER; ++q) a[q] = 0.0f;
    float aloo = 0.0f;
    for (int jb = j0; jb < j1; jb += 32) {
      const int j = jb + lane;
      const bool has = j < j1;
      const float xv_l = has ? __ldg(valv + j) : 0.0f;
      const int col_l = has ? __ldg(colv + j) : 0;
      float term_l = 0.0f;
      if (has) {
        const float cown = (float)__ldg(cdt + (size_t)col_l * CAP + t0);
        term_l = __fadd_rn(log2m(__fadd_rn(__fadd_rn(beta, cown), -xv_l)), -lden);
      }
      const int cnt = min(32, j1 - jb);
      for (int u0 = 0; u0 < cnt; u0 += kFlight) {
        float lv[kFlight][PER], xs[kFlight];
#pragma unroll
        for (int u = 0; u < kFlight; ++u) {
          const int src = min(u0 + u, cnt - 1);
          const int cl = __shfl_sync(0xffffffffu, col_l, src);
          xs[u] = __shfl_sync(0xffffffffu, xv_l, src);
          const float* p = l2t + (size_t)cl * CAP + lane * PER;
          if constexpr (PER >= 4) {
#pragma unroll
            for (int q = 0; q < PER; q += 4) {
              const float4 t4 = __ldg(reinterpret_cast<const float4*>(p) + q / 4);
              lv[u][q] = t4.x; lv[u][q + 1] = t4.y; lv[u][q + 2] = t4.z; lv[u][q + 3] = t4.w;
            }
          } else if constexpr (PER == 2) {
            const float2 t2 = __ldg(reinterpret_cast<const float2*>(p)); lv[u][0] = t2.x; lv[u][PER - 1] = t2.y;
          } else {
            lv[u][0] = __ldg(p);
          }
        }
#pragma unroll
        for (int u = 0; u < kFlight; ++u) {
          if (u0 + u < cnt) {                                  // warp-uniform
#pragma unroll
            for (int q = 0; q < PER; ++q) a[q] = __fmaf_rn(xs[u], lv[u][q], a[q]);
            aloo = __fmaf_rn(xs[u], __shfl_sync(0xffffffffu, term_l, u0 + u), aloo);
          }
        }
      }
    }
    float* dst = c.cnt_acc[v] + (size_t)row * CAP + lane * PER;
#pragma unroll
    for (int q = 0; q < PER; ++q) dst[q] = a[q];
    if (lane == 0) c.cnt_loo[v][row] = aloo;
  }
}

// Stage A of a count view under MVG_COUNT_DIRMULT: the same warp per row, row_order dealing and broadcast of the
// nonzeros as k_counts_loglik.  Per table t (l2c = log2(beta + c) of the dish's count c of word w, from k_counts_tables):
//   s_j = l2c[w_j][t], then for x_j > 1: s_j += log2m(beta + c + i), i = 1 .. x_j - 1;   a += s_j   (ascending j, x_j > 0)
//   a -= den[n][t]                                                                          (n = |x|, the row's tokens)
// The row's own dish, leave-one-out (counts c - x, total C_k - n, so the denominator is not the table's):
//   term_j = sum_{i < x_j} log2m(beta + (c - x_j) + i);   loo += term_j   (ascending j)
//   loo -= ld,  ld = sum_{j<n} log2m(W beta + C_k - n + j): lane l sums j = l, l+32, ... ascending, then an xor butterfly
//   (offsets 16, 8, 4, 2, 1; IEEE addition commutes, so every lane holds the same value).
// Every operation is one oracle/mv_oracle_dm.c:mvod_stageA_counts_f32 repeats bit for bit.
template <int CAP>
__global__ void __launch_bounds__(512) k_counts_loglik_dm(const Ctx c) {
  const int v = nth_count_view(c, blockIdx.y);
  constexpr int PER = CAP / 32;
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const int32_t* __restrict__ rp = c.rowptr[v];
  const int32_t* __restrict__ colv = c.col[v];
  const float* __restrict__ valv = c.val[v];
  const float* __restrict__ l2c = c.l2t[v];
  const int32_t* __restrict__ cdt = c.cnt_d[v];
  const float* __restrict__ den = c.cnt_den[v];
  const TableParam* __restrict__ tp = c.tparam + v * CAP;
  const int32_t* __restrict__ order = c.row_order[v];
  const float beta = (float)c.beta_v[v];
  constexpr int kFlight = 8;
  for (int ri = warp; ri < c.n_rows; ri += nwarps) {
    const int row = order ? __ldg(order + ri) : ri;
    const int j0 = rp[row], j1 = rp[row + 1];
    const int t0 = c.table_cur[row];
    const float nf = c.xx[(size_t)v * c.xx_stride + row];
    const int n = (int)nf;
    const float lbase = __fadd_rn(tp[t0].C1, -nf);          // TableParam::C1 of a count view: W beta + C_k
    float ld = 0.0f;
    for (int j = lane; j < n; j += 32) ld = __fadd_rn(ld, log2m(__fadd_rn(lbase, (float)j)));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ld = __fadd_rn(ld, __shfl_xor_sync(0xffffffffu, ld, o));
    float a[PER];
#pragma unroll
    for (int q = 0; q < PER; ++q) a[q] = 0.0f;
    float aloo = 0.0f;
    for (int jb = j0; jb < j1; jb += 32) {
      const int j = jb + lane;
      const bool has = j < j1;
      const float xv_l = has ? __ldg(valv + j) : 0.0f;
      const int col_l = has ? __ldg(colv + j) : 0;
      float term_l = 0.0f;
      if (has) {
        const int xi = (int)xv_l;
        const float b0 = __fadd_rn(beta, (float)(__ldg(cdt + (size_t)col_l * CAP + t0) - xi));
        for (int i = 0; i < xi; ++i) term_l = __fadd_rn(term_l, log2m(__fadd_rn(b0, (float)i)));
      }
      const int cnt = min(32, j1 - jb);
      for (int u0 = 0; u0 < cnt; u0 += kFlight) {
        float lv[kFlight][PER], xs[kFlight];
        int cls[kFlight];
#pragma unroll
        for (int u = 0; u < kFlight; ++u) {
          const int src = min(u0 + u, cnt - 1);
          cls[u] = __shfl_sync(0xffffffffu, col_l, src);
          xs[u] = __shfl_sync(0xffffffffu, xv_l, src);
          const float* p = l2c + (size_t)cls[u] * CAP + lane * PER;
          if constexpr (PER >= 4) {
#pragma unroll
            for (int q = 0; q < PER; q += 4) {
              const float4 t4 = __ldg(reinterpret_cast<const float4*>(p) + q / 4);
              lv[u][q] = t4.x; lv[u][q + 1] = t4.y; lv[u][q + 2] = t4.z; lv[u][q + 3] = t4.w;
            }
          } else if constexpr (PER == 2) {
            const float2 t2 = __ldg(reinterpret_cast<const float2*>(p)); lv[u][0] = t2.x; lv[u][PER - 1] = t2.y;
          } else {
            lv[u][0] = __ldg(p);
          }
        }
#pragma unroll
        for (int u = 0; u < kFlight; ++u) {
          if (u0 + u < cnt) {                                  // warp-uniform
            if (xs[u] > 1.0f) {                                // a repeated word (warp-uniform): the rising factorial
              const int xi = (int)xs[u];
              const int32_t* cp = cdt + (size_t)cls[u] * CAP + lane * PER;
#pragma unroll
              for (int q = 0; q < PER; ++q) {
                const float bc = __fadd_rn(beta, (float)__ldg(cp + q));
                float sq = lv[u][q];
                for (int i = 1; i < xi; ++i) sq = __fadd_rn(sq, log2m(__fadd_rn(bc, (float)i)));
                a[q] = __fadd_rn(a[q], sq);
              }
            } else if (xs[u] > 0.0f) {                         // (a stored zero count adds nothing)
#pragma unroll
              for (int q = 0; q < PER; ++q) a[q] = __fadd_rn(a[q], lv[u][q]);
            }
            aloo = __fadd_rn(aloo, __shfl_sync(0xffffffffu, term_l, u0 + u));
          }
        }
      }
    }
    const float* dn = den + (size_t)n * CAP + lane * PER;
    float* dst = c.cnt_acc[v] + (size_t)row * CAP + lane * PER;
#pragma unroll
    for (int q = 0; q < PER; ++q) dst[q] = __fadd_rn(a[q], -__ldg(dn + q));
    if (lane == 0) c.cnt_loo[v][row] = __fadd_rn(aloo, -ld);
  }
}

cudaError_t launch_counts_loglik(const Ctx& c, cudaStream_t s) {
  if (!c.n_count_views) return cudaSuccess;
  int blocks = (c.n_rows + 15) / 16;               // 16 warps per block
  if (blocks > 148 * 4) blocks = 148 * 4;
  const dim3 grid(blocks, c.n_count_views);         // all count views in one launch
  if (c.count_model) {
    switch (c.cap) {
      case 32: k_counts_loglik_dm<32><<<grid, 512, 0, s>>>(c); break;
      case 64: k_counts_loglik_dm<64><<<grid, 512, 0, s>>>(c); break;
      case 128: k_counts_loglik_dm<128><<<grid, 512, 0, s>>>(c); break;
      case 256: k_counts_loglik_dm<256><<<grid, 512, 0, s>>>(c); break;
      default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
  }
  switch (c.cap) {
    case 32: k_counts_loglik<32><<<grid, 512, 0, s>>>(c); break;
    case 64: k_counts_loglik<64><<<grid, 512, 0, s>>>(c); break;
    case 128: k_counts_loglik<128><<<grid, 512, 0, s>>>(c); break;
    case 256: k_counts_loglik<256><<<grid, 512, 0, s>>>(c); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

cudaError_t launch_counts_newdish(const Ctx& c, cudaStream_t s) {
  if (!c.n_count_views || !c.count_model || c.n_rows <= 0) return cudaSuccess;
  k_counts_newdish<<<dim3((c.n_rows + 255) / 256, c.n_count_views), 256, 0, s>>>(c, nullptr);
  return cudaGetLastError();
}

cudaError_t launch_rowtotals(const int32_t* rowptr, const float* val, float* out, int n, cudaStream_t s) {
  k_rowtotals<<<(n + 255) / 256, 256, 0, s>>>(rowptr, val, out, n);
  return cudaGetLastError();
}

static cudaError_t launch_counts_tables(const Ctx& c, size_t max_cells, const int32_t* gate, cudaStream_t s) {
  int tb = (int)((max_cells + 255) / 256);
  if (tb > 148 * 8) tb = 148 * 8;
  const int log2cap = __builtin_ctz((unsigned)c.cap);
  if (c.count_model) {
    if (c.cap <= 64) k_counts_tables<64, true><<<dim3(tb, c.n_count_views), 256, 0, s>>>(c, log2cap, gate);
    else k_counts_tables<256, true><<<dim3(tb, c.n_count_views), 256, 0, s>>>(c, log2cap, gate);
  } else if (c.cap <= 64) {
    k_counts_tables<64, false><<<dim3(tb, c.n_count_views), 256, 0, s>>>(c, log2cap, gate);
  } else {
    k_counts_tables<256, false><<<dim3(tb, c.n_count_views), 256, 0, s>>>(c, log2cap, gate);   // one thread per slot: 256 threads
  }
  return cudaGetLastError();
}

cudaError_t launch_counts_rebuild(const Ctx& c, bool delta, cudaStream_t s) {
  if (!c.n_count_views) return cudaSuccess;
  size_t max_cells = 0;
  for (int v = 0; v < c.V; ++v) {
    if (!c.kind[v]) continue;
    const size_t cells = (size_t)c.vocab[v] * c.cap;
    max_cells = cells > max_cells ? cells : max_cells;
    if (!delta) {
      cudaError_t e = cudaMemsetAsync(c.cnt_t[v], 0, sizeof(int32_t) * cells, s);
      if (e != cudaSuccess) return e;
    }
  }
  int blocks = (c.n_rows + 7) / 8;                 // 8 warps per block, one row per warp per step
  if (blocks > 148 * 4) blocks = 148 * 4;
  k_counts_scatter<<<dim3(blocks, c.n_count_views), 256, 0, s>>>(c, delta ? 1 : 0);
  return launch_counts_tables(c, max_cells, nullptr, s);
}

// ---- the beta step (MVG_COUNT_DIRMULT with a prior; DESIGN.md §4.5) -----------------------------------------------------
// For count view v at the seating k_counts_tables just counted, with L(beta) = sum over live dishes k of
//   sum_{w : c_kw > 0} lnΓ(beta + c_kw) - lnΓ(beta)  -  [lnΓ(W beta + C_k) - lnΓ(W beta)]
// (the beta-dependent part of the collapsed marginal; k_loglik's cell expression, lowest table slot of each dish):
//   z = Philox normal (kDomCountBeta, slot v, index 0),  log beta' = log beta + step z,
//   log A = L(beta') - L(beta) + shape (log beta' - log beta) - rate (beta' - beta),
//   u = Philox uniform (index 1): beta_v[v] = beta' when log u < log A.
// The (word, live dish) cells and the dish denominators are spread over cb_ctas CTAs per view; every thread sums
// lnΓ-differences at beta' minus those at beta of its cells in grid-stride order, the CTA by a fixed tree, and the last
// CTA to arrive adds the CTA partials in ascending order and decides.  The grid is fixed per handle, so the sum (and the
// decision) depends on neither timing nor graph replay.
constexpr int kBetaThreads = 256;
__global__ void __launch_bounds__(kBetaThreads) k_count_beta_step(const Ctx c, const int32_t advance) {
  const int v = nth_count_view(c, blockIdx.y);
  const int cap = c.cap;
  __shared__ int32_t s_rep[256];                  // lowest table slot of every live dish, -1 = none
  __shared__ int32_t s_lt[256], s_lk[256];        // the live dishes, ascending: representative slot, dish
  __shared__ int32_t s_nlive;
  __shared__ double s_red[kBetaThreads];
  __shared__ bool s_last;
  if (threadIdx.x < cap) {
    const int k = threadIdx.x;
    int rep = -1;
    if (c.n_vk[v * cap + k] > 0)
      for (int t = cap - 1; t >= 0; --t) if (c.dish_of[v * cap + t] == k) rep = t;
    s_rep[k] = rep;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int n = 0;
    for (int k = 0; k < cap; ++k)
      if (s_rep[k] >= 0) { s_lt[n] = s_rep[k]; s_lk[n] = k; ++n; }
    s_nlive = n;
  }
  __syncthreads();
  const uint32_t sweep = *c.sweep - (advance ? 1u : 0u);   // k_finalize of this rebuild has advanced it already
  const double beta = c.beta_v[v];
  const U4 rz = stream_block(c.seed, c.chain, kDomCountBeta, (uint32_t)v, sweep, 0);
  const double z = sqrt(-2.0 * log(uniform_f64_from(rz.x, rz.y))) * cos(6.283185307179586476925286766559 * uniform_f64_from(rz.z, rz.w));
  const double lb = log(beta), lbp = lb + c.cb_step * z, betap = exp(lbp);
  const double wb = (double)c.vocab[v] * beta, wbp = (double)c.vocab[v] * betap;
  const int nl = s_nlive;
  const int32_t* __restrict__ cd = c.cnt_d[v];
  const size_t cells = (size_t)c.vocab[v] * nl;
  double d = 0.0;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < cells + nl; e += (size_t)gridDim.x * blockDim.x) {
    if (e < cells) {
      const size_t w = e / nl;
      const int x = cd[w * cap + s_lt[e - w * nl]];
      if (x > 0) d += lgamma_diff(betap, x) - lgamma_diff(beta, x);   // a zero cell contributes exactly 0
    } else {
      const int tot = (int)c.S2k[v * cap + s_lk[e - cells]];        // the dish's token total (an exact integer)
      d -= lgamma_diff(wbp, tot) - lgamma_diff(wb, tot);
    }
  }
  s_red[threadIdx.x] = d;
  __syncthreads();
#pragma unroll
  for (int o = kBetaThreads / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) s_red[threadIdx.x] += s_red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    c.cb_part[(size_t)v * gridDim.x + blockIdx.x] = s_red[0];
    __threadfence();
    s_last = atomicAdd(&c.cb_arrive[v], 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last || threadIdx.x != 0) return;
  __threadfence();
  const volatile double* part = c.cb_part + (size_t)v * gridDim.x;
  double dl = 0.0;
  for (unsigned b = 0; b < gridDim.x; ++b) dl += part[b];
  const double log_a = dl + c.cb_shape * (lbp - lb) - c.cb_rate * (betap - beta);
  const U4 ru = stream_block(c.seed, c.chain, kDomCountBeta, (uint32_t)v, sweep, 1);
  const bool acc = log(uniform_f64_from(ru.x, ru.y)) < log_a;
  if (acc) c.beta_v[v] = betap;
  c.cb_accept[v] = acc ? 1 : 0;
  c.cb_logA[v] = log_a;
  c.cb_arrive[v] = 0u;                                              // ready for the next launch
}

cudaError_t launch_count_beta(const Ctx& c, int32_t flags, bool refresh_only, cudaStream_t s) {
  if (!c.n_count_views) return cudaSuccess;
  if (!refresh_only) {
    if (!c.cb_on || !(flags & kFinHyper) || !(flags & kFinHyperCountBeta)) return cudaSuccess;
    k_count_beta_step<<<dim3(c.cb_ctas, c.n_count_views), kBetaThreads, 0, s>>>(c, (flags & kFinAdvance) ? 1 : 0);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  // the refresh: every CTA of a view whose step rejected returns at once
  size_t max_cells = 0;
  for (int v = 0; v < c.V; ++v)
    if (c.kind[v] && (size_t)c.vocab[v] * c.cap > max_cells) max_cells = (size_t)c.vocab[v] * c.cap;
  cudaError_t e = launch_counts_tables(c, max_cells, c.cb_accept, s);
  if (e != cudaSuccess) return e;
  if (c.count_model) k_counts_newdish<<<dim3((c.n_rows + 255) / 256, c.n_count_views), 256, 0, s>>>(c, c.cb_accept);
  return cudaGetLastError();
}

}  // namespace mv
