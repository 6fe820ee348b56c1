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
#include "mv_ctx.h"

namespace mv {

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
template <int MAXCAP>
__global__ void k_counts_tables(const Ctx c, const int log2cap) {
  constexpr int kWords = MAXCAP / 64;
  const int v = nth_count_view(c, blockIdx.y);
  __shared__ int32_t s_dish[MAXCAP];
  __shared__ double s_den[MAXCAP];
  __shared__ float s_l2zero[MAXCAP];                         // log2 theta of a word the dish has never seen: most cells of the table
  __shared__ unsigned long long s_mask[MAXCAP][kWords];      // the table slots serving the same dish as slot t
  const int cap = c.cap;
  if (threadIdx.x < cap) {
    const int k = c.dish_of[v * cap + threadIdx.x];
    s_dish[threadIdx.x] = k;
    // S2k of a count view holds the token total of the dish (an exact integer)
    s_den[threadIdx.x] = (k >= 0) ? (double)c.vocab[v] * (double)c.count_beta + c.S2k[v * cap + k] : 1.0;
    s_l2zero[threadIdx.x] = (float)log2(((double)c.count_beta + 0.0) / s_den[threadIdx.x]);   // the cell expression at cd = 0
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
  if (blockIdx.y == 0)
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
      l2 = (cd == 0) ? s_l2zero[t] : (float)log2(((double)c.count_beta + (double)cd) / s_den[t]);
    }
    c.cnt_d[v][e] = cd;
    c.l2t[v][e] = l2;
  }
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
        term_l = __fadd_rn(log2m(__fadd_rn(__fadd_rn(c.count_beta, cown), -xv_l)), -lden);
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

cudaError_t launch_counts_loglik(const Ctx& c, cudaStream_t s) {
  if (!c.n_count_views) return cudaSuccess;
  int blocks = (c.n_rows + 15) / 16;               // 16 warps per block
  if (blocks > 148 * 4) blocks = 148 * 4;
  const dim3 grid(blocks, c.n_count_views);         // all count views in one launch
  switch (c.cap) {
    case 32: k_counts_loglik<32><<<grid, 512, 0, s>>>(c); break;
    case 64: k_counts_loglik<64><<<grid, 512, 0, s>>>(c); break;
    case 128: k_counts_loglik<128><<<grid, 512, 0, s>>>(c); break;
    case 256: k_counts_loglik<256><<<grid, 512, 0, s>>>(c); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

cudaError_t launch_rowtotals(const int32_t* rowptr, const float* val, float* out, int n, cudaStream_t s) {
  k_rowtotals<<<(n + 255) / 256, 256, 0, s>>>(rowptr, val, out, n);
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
  int tb = (int)((max_cells + 255) / 256);
  if (tb > 148 * 8) tb = 148 * 8;
  const int log2cap = __builtin_ctz((unsigned)c.cap);
  if (c.cap <= 64) k_counts_tables<64><<<dim3(tb, c.n_count_views), 256, 0, s>>>(c, log2cap);
  else k_counts_tables<256><<<dim3(tb, c.n_count_views), 256, 0, s>>>(c, log2cap);   // one thread per slot: 256 threads
  return cudaGetLastError();
}

}  // namespace mv
