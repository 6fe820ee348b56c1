// mv_draw_simt.cu — likelihood + draw on FP32 CUDA cores (engine MVG_ENGINE_SIMT).
//
// One thread owns one customer.  For every view it forms the dot products x.m_t against the
// per-table posterior means (staged in shared memory, broadcast reads) as ONE ascending fmaf chain
// per table — the order oracle/mv_oracle.c:mvo_stageA_f32 restates — and hands them to
// RowEpilogue (mv_device.cuh).  Any dim, any number of views; used for the reference's scalar
// views (D = 1, New_Simulation.R) and wherever the tcgen05 engine's shape constraints do not hold.
//
// Replaces, per customer: remove_customer + compute_table_probs_with_cache + the inverse-CDF draw
// (/root/reference/Multiview/multiview_utils.cpp:71-192, multiview_gibbs.cpp:157-199).
#include "mv_ctx.h"

namespace mv {

constexpr int kSimtThreads = 128;
constexpr int kSimtDChunk = 128;   // columns of m staged per pass

// Bytes of the first shared-memory region: the staged means of a dense view.
template <int CAP>
__host__ __device__ inline size_t simt_first_region_bytes(const Ctx& c) {
  const int dch_max = (c.Dsum < kSimtDChunk) ? (c.Dsum > 0 ? c.Dsum : 1) : kSimtDChunk;   // upper bound on any view's chunk
  return (sizeof(float) * (size_t)CAP * (size_t)dch_max + 15) & ~(size_t)15;
}

template <int CAP, bool VEC4>
__global__ void __launch_bounds__(kSimtThreads, 2) k_draw_simt(const Ctx c) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_m = reinterpret_cast<float*>(smem_raw);                       // [CAP][dch]
  PairHot* s_hot = reinterpret_cast<PairHot*>(smem_raw + simt_first_region_bytes<CAP>(c));                 // [CAP/2]
  TableCold* s_cold = reinterpret_cast<TableCold*>(s_hot + CAP / 2);                                        // [CAP]
  __shared__ TableMass s_tm[CAP];
  __shared__ __align__(16) float s_lm[CAP];
  __shared__ GlobalParam s_g;
  __shared__ ViewParam s_vp;

  const int tid = threadIdx.x;
  for (int t = tid; t < CAP; t += kSimtThreads) { s_tm[t] = c.tmass[t]; s_lm[t] = c.tmass[t].LM; }
  if (tid == 0) s_g = *c.gparam;
  __syncthreads();
  const uint32_t sweep = s_g.sweep;

  const int n_tiles = (c.n_rows + kSimtThreads - 1) / kSimtThreads;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int row = tile * kSimtThreads + tid;
    const bool live = row < c.n_rows;
    const int rowc = live ? row : (c.n_rows - 1);
    RowEpilogue<CAP> epi;
    epi.begin(s_tm, s_lm, s_g, c.table_cur[rowc]);

    for (int v = 0; v < c.V; ++v) {
      if (c.kind[v]) {
        // ---- sparse count view: acc[t] = sum_j x_j log2 theta[col_j][t], one ascending fmaf chain per table over
        //      the row's nonzeros (the order of oracle/mv_oracle.c:mvo_stageA_counts_f32); the table is
        //      feature-major, so one nonzero reads CAP consecutive floats ----
        __syncthreads();   // previous users of s_hot / s_cold are done
        stage_view_params(c.tparam + v * CAP, CAP, s_hot, s_cold, tid, kSimtThreads);
        if (tid == 0) s_vp = c.vparam[v];
        __syncthreads();
        // k_counts_loglik (mv_counts.cu, one warp per row) left the CAP log2 f values of every customer and its
        // leave-one-out value in global memory (L2-resident at Reuters size); here: the common per-customer epilogue.
        // The new-dish term is -AN rowtot + CN: the token total under the plug-in, -log2 f_new under DIRMULT (AN = 1, CN = 0)
        const float rowtot = c.count_model ? __ldg(c.cnt_q[v] + rowc) : c.xx[(size_t)v * c.xx_stride + rowc];
        float acc[CAP];
        {
          const float4* __restrict__ src = reinterpret_cast<const float4*>(c.cnt_acc[v] + (size_t)rowc * CAP);
#pragma unroll
          for (int q = 0; q < CAP / 4; ++q) {
            const float4 a4 = __ldg(src + q);
            acc[4 * q] = a4.x; acc[4 * q + 1] = a4.y; acc[4 * q + 2] = a4.z; acc[4 * q + 3] = a4.w;
          }
        }
        const float acc_loo = __ldg(c.cnt_loo[v] + rowc);
        if ((c.debug_export & 1) && live) {
          float* da = c.dbg_acc + ((size_t)row * c.V + v) * CAP;
#pragma unroll
          for (int t = 0; t < CAP; ++t) da[t] = acc[t];
          c.dbg_xx[(size_t)row * c.V + v] = rowtot;
          c.dbg_loo[(size_t)row * c.V + v] = acc_loo;
        }
        epi.view_counts(s_hot, s_cold, s_vp, acc, acc_loo, rowtot);
        continue;
      }
      const int D = c.D[v];
      const float* __restrict__ xrow = c.x[v] + (size_t)rowc * D;
      const float* __restrict__ mean_v = c.mean + (size_t)c.cap * c.doff[v];
      float acc[CAP];
#pragma unroll
      for (int t = 0; t < CAP; ++t) acc[t] = 0.0f;
      float xx = 0.0f;

      for (int d0 = 0; d0 < D; d0 += kSimtDChunk) {
        const int dch = (D - d0 < kSimtDChunk) ? (D - d0) : kSimtDChunk;
        __syncthreads();   // previous users of s_m / s_hot / s_cold are done
        for (int idx = tid; idx < CAP * dch; idx += kSimtThreads) {
          const int t = idx / dch, dd = idx - t * dch;
          s_m[t * dch + dd] = mean_v[(size_t)t * D + d0 + dd];
        }
        if (d0 == 0) {
          stage_view_params(c.tparam + v * CAP, CAP, s_hot, s_cold, tid, kSimtThreads);
          if (tid == 0) s_vp = c.vparam[v];
        }
        __syncthreads();
        if (VEC4) {
          for (int dd = 0; dd < dch; dd += 4) {
            const float4 xv = __ldg(reinterpret_cast<const float4*>(xrow + d0 + dd));
            xx = __fmaf_rn(xv.x, xv.x, xx);
            xx = __fmaf_rn(xv.y, xv.y, xx);
            xx = __fmaf_rn(xv.z, xv.z, xx);
            xx = __fmaf_rn(xv.w, xv.w, xx);
#pragma unroll
            for (int t = 0; t < CAP; ++t) {
              const float4 mv4 = *reinterpret_cast<const float4*>(s_m + t * dch + dd);
              float a = acc[t];
              a = __fmaf_rn(xv.x, mv4.x, a);
              a = __fmaf_rn(xv.y, mv4.y, a);
              a = __fmaf_rn(xv.z, mv4.z, a);
              a = __fmaf_rn(xv.w, mv4.w, a);
              acc[t] = a;
            }
          }
        } else {
          for (int dd = 0; dd < dch; ++dd) {
            const float xs = __ldg(xrow + d0 + dd);
            xx = __fmaf_rn(xs, xs, xx);
#pragma unroll
            for (int t = 0; t < CAP; ++t) acc[t] = __fmaf_rn(xs, s_m[t * dch + dd], acc[t]);
          }
        }
      }
      if ((c.debug_export & 1) && live) {
        float* da = c.dbg_acc + ((size_t)row * c.V + v) * CAP;
#pragma unroll
        for (int t = 0; t < CAP; ++t) da[t] = acc[t];
        c.dbg_xx[(size_t)row * c.V + v] = xx;
      }
      epi.view(s_hot, s_cold, s_vp, acc, xx);
    }

    const U4 rnd = stream_block(c.seed, c.chain, kDomTable, 0, sweep, (uint64_t)(c.row_offset + rowc));
    int choice = epi.finish(uniform_f32_from(rnd.x));
    if (c.blk_count > 1 && (int)((c.row_offset + rowc) % c.blk_count) != c.blk_index) choice = epi.ha.t0;   // not this pass's block
    if (live) {
      c.choice[row] = choice;
      if (c.debug_export & 1) c.dbg_choice[row] = choice;
    }
    const unsigned births = __ballot_sync(0xffffffffu, live && choice == kNewTable);
    const unsigned moved = __ballot_sync(0xffffffffu, live && choice != epi.ha.t0);
    if ((tid & 31) == 0 && (row >> 5) < c.n_chunks) { c.birthmask[row >> 5] = births; c.movedmask[row >> 5] = moved; }
  }
}

// CAP = 128 / 256: the same draw with the running log-weights in shared memory (WideRowEpilogue, 1 KB per customer at
// 256) and the dot products formed kSimtTableGroup tables at a time — each one the same ascending fmaf chain over d as
// above, over the means of the group staged in kSimtDChunk-column pieces — and handed to the epilogue in ascending
// 16-table chunks.  Registers hold one group's dot products instead of all CAP, so nothing spills.
constexpr int kSimtTableGroup = 32;

template <int CAP>
__host__ __device__ inline size_t simt_wide_smem_bytes() {
  return sizeof(float) * kSimtTableGroup * kSimtDChunk                                // s_m  [group][dch]
         + sizeof(PairHot) * (CAP / 2) + sizeof(TableCold) * CAP                       // s_hot, s_cold
         + sizeof(float2) * (CAP / 2) * kSimtThreads;                                  // s_lw [CAP/2][threads]
}

template <int CAP, bool VEC4>
__global__ void __launch_bounds__(kSimtThreads, 1) k_draw_simt_wide(const Ctx c) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_m = reinterpret_cast<float*>(smem_raw);
  PairHot* s_hot = reinterpret_cast<PairHot*>(s_m + kSimtTableGroup * kSimtDChunk);
  TableCold* s_cold = reinterpret_cast<TableCold*>(s_hot + CAP / 2);
  float2* s_lw = reinterpret_cast<float2*>(s_cold + CAP);
  __shared__ TableMass s_tm[CAP];
  __shared__ __align__(16) float s_lm[CAP];
  __shared__ GlobalParam s_g;
  __shared__ ViewParam s_vp;

  const int tid = threadIdx.x;
  for (int t = tid; t < CAP; t += kSimtThreads) { s_tm[t] = c.tmass[t]; s_lm[t] = c.tmass[t].LM; }
  if (tid == 0) s_g = *c.gparam;
  __syncthreads();
  const uint32_t sweep = s_g.sweep;

  const int n_tiles = (c.n_rows + kSimtThreads - 1) / kSimtThreads;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int row = tile * kSimtThreads + tid;
    const bool live = row < c.n_rows;
    const int rowc = live ? row : (c.n_rows - 1);
    WideRowEpilogue<CAP, kSimtThreads> epi;
    epi.begin(s_lw + tid, s_tm, s_lm, s_g, c.table_cur[rowc]);

    for (int v = 0; v < c.V; ++v) {
      __syncthreads();   // previous users of s_hot / s_cold / s_m are done
      stage_view_params(c.tparam + v * CAP, CAP, s_hot, s_cold, tid, kSimtThreads);
      if (tid == 0) s_vp = c.vparam[v];
      __syncthreads();
      float* const da = c.dbg_acc + ((size_t)row * c.V + v) * CAP;
      const bool dbg = (c.debug_export & 1) && live;
      if (c.kind[v]) {
        // count view: the CAP log2 f values and the leave-one-out value that k_counts_loglik left in global memory
        const float rowtot = c.count_model ? __ldg(c.cnt_q[v] + rowc) : c.xx[(size_t)v * c.xx_stride + rowc];
        const float acc_loo = __ldg(c.cnt_loo[v] + rowc);
        epi.view_begin(s_hot, s_cold, 0.0f);
        epi.A1r = 0.0f; epi.C1r = acc_loo;
        const float4* __restrict__ src = reinterpret_cast<const float4*>(c.cnt_acc[v] + (size_t)rowc * CAP);
        for (int base = 0; base < CAP; base += kEpiChunk) {
          float acc[kEpiChunk];
#pragma unroll
          for (int q = 0; q < kEpiChunk / 4; ++q) {
            const float4 a4 = __ldg(src + base / 4 + q);
            acc[4 * q] = a4.x; acc[4 * q + 1] = a4.y; acc[4 * q + 2] = a4.z; acc[4 * q + 3] = a4.w;
          }
          if (dbg)
#pragma unroll
            for (int j = 0; j < kEpiChunk; ++j) da[base + j] = acc[j];
          epi.chunk(s_hot, s_cold, base, acc);
        }
        if (dbg) { c.dbg_xx[(size_t)row * c.V + v] = rowtot; c.dbg_loo[(size_t)row * c.V + v] = acc_loo; }
        epi.view_end(s_vp, rowtot);
        continue;
      }
      const int D = c.D[v];
      const float* __restrict__ xrow = c.x[v] + (size_t)rowc * D;
      const float* __restrict__ mean_v = c.mean + (size_t)c.cap * c.doff[v];
      float xx = 0.0f;
      for (int dd = 0; dd < D; ++dd) { const float xs = __ldg(xrow + dd); xx = __fmaf_rn(xs, xs, xx); }
      epi.view_begin(s_hot, s_cold, xx);
      for (int tg = 0; tg < CAP; tg += kSimtTableGroup) {
        float acc[kSimtTableGroup];
#pragma unroll
        for (int t = 0; t < kSimtTableGroup; ++t) acc[t] = 0.0f;
        for (int d0 = 0; d0 < D; d0 += kSimtDChunk) {
          const int dch = (D - d0 < kSimtDChunk) ? (D - d0) : kSimtDChunk;
          __syncthreads();   // previous users of s_m are done
          for (int idx = tid; idx < kSimtTableGroup * dch; idx += kSimtThreads) {
            const int t = idx / dch, dd = idx - t * dch;
            s_m[t * dch + dd] = mean_v[(size_t)(tg + t) * D + d0 + dd];
          }
          __syncthreads();
          if (VEC4) {
            for (int dd = 0; dd < dch; dd += 4) {
              const float4 xv = __ldg(reinterpret_cast<const float4*>(xrow + d0 + dd));
#pragma unroll
              for (int t = 0; t < kSimtTableGroup; ++t) {
                const float4 mv4 = *reinterpret_cast<const float4*>(s_m + t * dch + dd);
                float a = acc[t];
                a = __fmaf_rn(xv.x, mv4.x, a);
                a = __fmaf_rn(xv.y, mv4.y, a);
                a = __fmaf_rn(xv.z, mv4.z, a);
                a = __fmaf_rn(xv.w, mv4.w, a);
                acc[t] = a;
              }
            }
          } else {
            for (int dd = 0; dd < dch; ++dd) {
              const float xs = __ldg(xrow + d0 + dd);
#pragma unroll
              for (int t = 0; t < kSimtTableGroup; ++t) acc[t] = __fmaf_rn(xs, s_m[t * dch + dd], acc[t]);
            }
          }
        }
        if (dbg)
#pragma unroll
          for (int t = 0; t < kSimtTableGroup; ++t) da[tg + t] = acc[t];
#pragma unroll
        for (int b = 0; b < kSimtTableGroup; b += kEpiChunk) {
          float ch[kEpiChunk];
#pragma unroll
          for (int j = 0; j < kEpiChunk; ++j) ch[j] = acc[b + j];
          epi.chunk(s_hot, s_cold, tg + b, ch);
        }
      }
      if (dbg) c.dbg_xx[(size_t)row * c.V + v] = xx;
      epi.view_end(s_vp, xx);
    }

    const U4 rnd = stream_block(c.seed, c.chain, kDomTable, 0, sweep, (uint64_t)(c.row_offset + rowc));
    int choice = epi.finish(uniform_f32_from(rnd.x));
    if (c.blk_count > 1 && (int)((c.row_offset + rowc) % c.blk_count) != c.blk_index) choice = epi.t0;   // not this pass's block
    if (live) {
      c.choice[row] = choice;
      if (c.debug_export & 1) c.dbg_choice[row] = choice;
    }
    const unsigned births = __ballot_sync(0xffffffffu, live && choice == kNewTable);
    const unsigned moved = __ballot_sync(0xffffffffu, live && choice != epi.t0);
    if ((tid & 31) == 0 && (row >> 5) < c.n_chunks) { c.birthmask[row >> 5] = births; c.movedmask[row >> 5] = moved; }
  }
}

template <int CAP>
static cudaError_t launch_simt_wide(const Ctx& c, cudaStream_t s) {
  bool vec4 = true;
  for (int v = 0; v < c.V; ++v)
    if (!c.kind[v] && ((c.D[v] & 3) != 0 || (reinterpret_cast<uintptr_t>(c.x[v]) & 15) != 0)) vec4 = false;
  const size_t smem = simt_wide_smem_bytes<CAP>();
  const int n_tiles = (c.n_rows + kSimtThreads - 1) / kSimtThreads;
  const auto kern = vec4 ? k_draw_simt_wide<CAP, true> : k_draw_simt_wide<CAP, false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  int dev = 0, sms = 148, per_sm = 1;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kSimtThreads, smem);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) return cudaErrorInvalidConfiguration;
  const int grid = n_tiles < per_sm * sms ? n_tiles : per_sm * sms;   // one resident wave strides over the tiles
  kern<<<grid, kSimtThreads, smem, s>>>(c);
  return cudaGetLastError();
}

template <int CAP>
static cudaError_t launch_simt_cap(const Ctx& c, cudaStream_t s) {
  bool vec4 = true;
  for (int v = 0; v < c.V; ++v)
    if (!c.kind[v] && ((c.D[v] & 3) != 0 || (reinterpret_cast<uintptr_t>(c.x[v]) & 15) != 0)) vec4 = false;
  const size_t smem = simt_first_region_bytes<CAP>(c) + sizeof(TableParam) * CAP;
  const int n_tiles = (c.n_rows + kSimtThreads - 1) / kSimtThreads;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int grid = n_tiles < 2 * sms ? n_tiles : 2 * sms;
  cudaError_t e;
  if (vec4) {
    e = cudaFuncSetAttribute(k_draw_simt<CAP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k_draw_simt<CAP, true><<<grid, kSimtThreads, smem, s>>>(c);
  } else {
    e = cudaFuncSetAttribute(k_draw_simt<CAP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k_draw_simt<CAP, false><<<grid, kSimtThreads, smem, s>>>(c);
  }
  return cudaGetLastError();
}

cudaError_t launch_draw_simt(const Ctx& c, cudaStream_t s) {
  if (c.n_rows <= 0) return cudaSuccess;
  if (c.n_count_views) {                       // stage A of the count views: its own high-occupancy kernel
    cudaError_t e = launch_counts_loglik(c, s);
    if (e != cudaSuccess) return e;
  }
  switch (c.cap) {
    case 32: return launch_simt_cap<32>(c, s);
    case 64: return launch_simt_cap<64>(c, s);
    case 128: return launch_simt_wide<128>(c, s);
    case 256: return launch_simt_wide<256>(c, s);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace mv
