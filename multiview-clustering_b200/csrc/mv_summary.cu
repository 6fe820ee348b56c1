// mv_summary.cu — posterior summaries of a chain, computed where the state lives:
//
//   k_labels        the cluster of every customer in every view, dish_of[v][table_of[i]]
//                   (get_final_clusters of /root/reference/Multiview/New_Simulation.R:135-149)
//   k_cocluster     co-clustering counts: C[i][j] += [label_i == label_j] over the kept sweeps (the pairwise
//                   posterior similarity matrix north_star's third correctness bullet compares across chains)
//   k_contingency   the Predicted x Truth table of New_Simulation.R:192-196, from which the adjusted Rand
//                   index (mcclust::arandi, :189) follows in closed form
//   k_loglik        joint log marginal likelihood of the data given the partition: the sum over live dishes of
//                   the reference's log p(y_S) (multiview_utils.cpp:316-320, per coordinate) — what the
//                   declared-but-never-defined compute_log_likelihood() (multiview_gibbs.h:13) would return; for a
//                   count view under MVG_COUNT_DIRMULT the collapsed Dirichlet-multinomial marginal
#include "mv_ctx.h"

namespace mv {

__global__ void k_labels(const Ctx c, int32_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c.n_rows) return;
  const int t = c.table_cur[i];
  for (int v = 0; v < c.V; ++v) out[(size_t)v * c.n_rows + i] = c.dish_of[v * c.cap + t];
}

// view < 0: tables; else dishes of that view.  One thread per 4 consecutive j of a row i.
__global__ void __launch_bounds__(256) k_cocluster(const Ctx c, const int view, uint32_t* __restrict__ counts) {
  __shared__ int32_t s_dish[256];                 // cap <= 256 = blockDim.x (mvg_create)
  if (threadIdx.x < c.cap) s_dish[threadIdx.x] = (view < 0) ? (int32_t)threadIdx.x : c.dish_of[view * c.cap + threadIdx.x];
  __syncthreads();
  const int n = c.n_rows;
  const int i = blockIdx.y;
  const int li = s_dish[c.table_cur[i]];
  uint32_t* row = counts + (size_t)i * n;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x)
    if (s_dish[c.table_cur[j]] == li) row[j] += 1u;
}

__global__ void k_contingency(const Ctx c, const int view, const int32_t* __restrict__ truth, const int n_classes,
                              int32_t* __restrict__ table /* [cap][n_classes] */) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c.n_rows) return;
  const int t = c.table_cur[i];
  const int k = (view < 0) ? t : c.dish_of[view * c.cap + t];
  const int z = truth[i];
  if (k >= 0 && z >= 0 && z < n_classes) atomicAdd(&table[k * n_classes + z], 1);
}

// A count view under MVG_COUNT_DIRMULT: the collapsed marginal of the partition up to the multinomial coefficients (which
// do not depend on it), sum over live dishes k of sum_w lnΓ(beta + c_kw) - lnΓ(beta)  -  [lnΓ(W beta + C_k) - lnΓ(W beta)],
// the word counts read from the lowest table slot serving each dish (cnt_d, current after every rebuild).  Thread tid takes
// the words w = tid mod blockDim.x over all live dishes, then its dish denominators; the block sums in ascending order.
// (scalars and pointers, not `const Ctx&`: the address of the kernel parameter would copy the struct per thread)
__device__ double loglik_dirmult_term(const int32_t* __restrict__ cd, const double* __restrict__ ctot, int vocab, int cap,
                                      double beta, const int32_t* s_rep) {
  double term = 0.0;
  for (int w = threadIdx.x; w < vocab; w += blockDim.x)
    for (int k = 0; k < cap; ++k) {
      const int tk = s_rep[k];
      if (tk < 0) continue;
      const int x = cd[(size_t)w * cap + tk];
      if (x > 0) term += lgamma_diff(beta, x);
    }
  for (int k = threadIdx.x; k < cap; k += blockDim.x)
    if (s_rep[k] >= 0) term -= lgamma_diff((double)vocab * beta, (int)ctot[k]);
  return term;
}

__global__ void __launch_bounds__(256) k_loglik(const Ctx c, double* __restrict__ out /* [V+1]: per view, then the total */) {
  __shared__ double s_term[256];
  __shared__ int32_t s_rep[256];                  // DIRMULT: lowest table slot of every live dish, -1 = none
  const double kPi = 3.14159265358979323846;
  double total = 0.0;
  for (int v = 0; v < c.V; ++v) {
    const double tau = c.hyp[2 * c.V + v];
    const int D = c.D[v];
    double term = 0.0;
    if (c.kind[v] && c.count_model) {
      if (threadIdx.x < c.cap) {
        const int k = threadIdx.x;
        int rep = -1;
        if (c.n_vk[v * c.cap + k] > 0)
          for (int t = c.cap - 1; t >= 0; --t) if (c.dish_of[v * c.cap + t] == k) rep = t;
        s_rep[k] = rep;
      }
      __syncthreads();
      term = loglik_dirmult_term(c.cnt_d[v], c.S2k + v * c.cap, c.vocab[v], c.cap, c.beta_v[v], s_rep);
    } else {
      for (int k = threadIdx.x; k < c.cap; k += blockDim.x) {
        const int n = c.n_vk[v * c.cap + k];
        if (n <= 0) continue;
        const double* S1 = c.S1k + (size_t)c.cap * c.doff[v] + (size_t)k * D;
        double q = 0.0;
        for (int dd = 0; dd < D; ++dd) q += S1[dd] * S1[dd];
        const double nn = (double)n;
        term += -0.5 * nn * (double)D * log(2.0 * kPi * tau) - 0.5 * (double)D * log(tau * (tau + nn)) -
                0.5 * c.S2k[v * c.cap + k] / tau + 0.5 * q / (tau * (tau + nn));
      }
    }
    s_term[threadIdx.x] = term;
    __syncthreads();
    if (threadIdx.x == 0) {
      double sum = 0.0;
      for (int i = 0; i < blockDim.x; ++i) sum += s_term[i];   // ascending: a fixed order
      out[v] = sum;
      total += sum;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) out[c.V] = total;
}

cudaError_t launch_labels(const Ctx& c, int32_t* out, cudaStream_t s) {
  k_labels<<<(c.n_rows + 255) / 256, 256, 0, s>>>(c, out);
  return cudaGetLastError();
}
cudaError_t launch_cocluster(const Ctx& c, int view, uint32_t* counts, cudaStream_t s) {
  int gx = (c.n_rows + 255) / 256;
  if (gx > 64) gx = 64;
  k_cocluster<<<dim3(gx, c.n_rows), 256, 0, s>>>(c, view, counts);
  return cudaGetLastError();
}
cudaError_t launch_contingency(const Ctx& c, int view, const int32_t* truth, int n_classes, int32_t* table, cudaStream_t s) {
  k_contingency<<<(c.n_rows + 255) / 256, 256, 0, s>>>(c, view, truth, n_classes, table);
  return cudaGetLastError();
}
cudaError_t launch_loglik(const Ctx& c, double* out, cudaStream_t s) {
  k_loglik<<<1, 256, 0, s>>>(c, out);
  return cudaGetLastError();
}

}  // namespace mv
