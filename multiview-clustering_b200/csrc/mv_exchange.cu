// mv_exchange.cu — k_reduce_x: this shard's sufficient statistics (fixed-order FP64 sums of the per-CTA partials of
// the statistics kernel) and, in the same launch, their exchange with the other shards and the rank-ordered totals
// k_finalize starts from.
//
// north_star asks for "an NCCL allreduce of the per-cluster sufficient statistics over NVLink" once per sweep.  The
// totals must not depend on a ring's summation order (every rank replays the same chain from them), so what travels
// is each rank's FP64 values and every rank adds them in rank order.  Two transports produce bit-identical results:
//
//   p2p (default on one node)   ONE kernel, no separate collective.  Every rank owns a receive buffer its peers have
//       mapped (CUDA IPC over NVLink / NVSwitch).  The thread that has just reduced element i stores it straight into
//       every peer's buffer as two 8-byte words {payload, sequence number} (the flag travels INSIDE the data, as in
//       NCCL's LL protocol: an 8-byte store arrives whole, so a word whose flag equals the current sequence number is
//       valid and no fence, counter or second round trip is needed), then polls its own buffer for the peers' words of
//       the same element and adds them in rank order.  Two parities: a rank can be at most one exchange ahead of a
//       peer that still reads the previous one (it cannot finish exchange s+1 without that peer's words of s+1).
//       The sequence number lives in device memory and is advanced by k_finalize, so the whole sweep is one CUDA graph.
//   nccl    reduce (mode 0) -> ncclAllGather of the packets -> rank-ordered sums (mode 2): the library baseline.
//
// A peer that never arrives must not hang the GPU: polls are bounded by %globaltimer (kWaitLimitNs); on expiry the
// kernel raises the STICKY fault status[1] (mirrored to mapped host memory), k_finalize then publishes nothing — the
// chain stays frozen at the last completed sweep on this rank — and mvg_sweep / mvg_sync refuse to continue.
//
// Replaces the incremental sum_y / sum_y2 / n_vk maintenance of /root/reference/Multiview/multiview_utils.cpp:151-163,
// 199-206 (as seen from all shards) together with csrc/mv_stats_tile.cu / k_stats.
#include "mv_ctx.h"

namespace mv {

namespace {

constexpr int kRedSlices = 8;
constexpr unsigned long long kWaitLimitNs = 2000000000ull;     // 2 s: documented in include/mvg.h

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// One 16-byte unit = two LL words {lo32, seq}, {hi32, seq} of a 64-bit payload.
__device__ __forceinline__ void ll_store_unit(void* dst, unsigned long long payload, uint32_t seq) {
  const uint32_t lo = (uint32_t)payload, hi = (uint32_t)(payload >> 32);
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(lo), "r"(seq), "r"(hi), "r"(seq) : "memory");
}
__device__ __forceinline__ void ll_store_word(void* dst, uint32_t payload, uint32_t seq) {
  asm volatile("st.volatile.global.v2.u32 [%0], {%1, %2};" ::"l"(dst), "r"(payload), "r"(seq) : "memory");
}
struct Waiter {          // bounded polling: the clock is read every 256 polls
  unsigned long long t0 = 0;
  uint32_t polls = 0;
  bool expired = false;
  __device__ __forceinline__ bool keep_waiting() {
    if ((++polls & 255u) != 0u) return true;
    const unsigned long long now = globaltimer_ns();
    if (t0 == 0) { t0 = now; return true; }
    if (now - t0 > kWaitLimitNs) { expired = true; return false; }
    return true;
  }
};
__device__ __forceinline__ bool ll_load_word(const void* src, uint32_t seq, uint32_t* payload, Waiter& w) {
  uint32_t a, fa;
  for (;;) {
    asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(a), "=r"(fa) : "l"(src) : "memory");
    if (fa == seq) break;
    if (!w.keep_waiting()) return false;
  }
  *payload = a;
  return true;
}

__device__ __forceinline__ void raise_fault(const Ctx& c) {
  atomicExch(c.status + 1, 8);
  if (c.host_fault) *reinterpret_cast<volatile int32_t*>(c.host_fault) = 8;
}

}  // namespace

XchgLayout xchg_layout(const Ctx& c) {
  XchgLayout L;
  L.n_units = (int64_t)c.cap * c.Dsum + (int64_t)c.V * c.cap + c.cap;
  L.n_words = 8 + 2 * (int64_t)c.cap + (int64_t)c.cap * c.Dsum;
  L.word_off = L.n_units * 16;
  L.slot_bytes = (L.word_off + L.n_words * 8 + 255) & ~(int64_t)255;
  return L;
}

// mode 0: reduce the partials into this rank's packet (and, with world = 1, into the totals)
// mode 1: reduce, push to the peers, pull, rank-ordered totals      (peer-memory transport)
// mode 2: rank-ordered totals from the all-gathered packets          (NCCL transport, second launch)
// Blocks [0, n_sum_blocks): 32 consecutive elements x 8 slices (slice j adds the partials of CTAs j, j+8, ... in
// ascending order, then the 8 slice sums are added in ascending order: a fixed tree), walking the elements with a
// grid stride.  Blocks [n_sum_blocks, n_sum_blocks + world) in mode 1: the birth candidates of / for rank g.
// delta: the partials hold the CHANGE of this shard's statistics (mv_stats_tile.cu, DELTA): it is added to the shard's
// running FP64 sums, which live in its packet, instead of replacing them.
__global__ void __launch_bounds__(256, 3) k_reduce_x(const Ctx c, const int mode, const int delta, const int n_sum_blocks, const XchgPeers peers,
                                                  unsigned char* __restrict__ recv_local, const XchgLayout L) {
  __shared__ double s_part[kRedSlices][32];
  __shared__ int s_cnt[kRedSlices][32];
  __shared__ int s_ncand;
  __shared__ unsigned char s_active[1024];       // delta: which CTAs of the statistics kernel wrote partials
  pdl_trigger();
  pdl_wait();
  const int n_s1 = c.cap * c.Dsum, n_s2 = c.V * c.cap;
  const int n_el = n_s1 + n_s2 + c.cap;
  const uint32_t seq = (mode == 1) ? *reinterpret_cast<volatile uint32_t*>(c.xseq) + 1u : 0u;
  const size_t slot0 = (size_t)(seq & 1u) * c.world * (size_t)L.slot_bytes;        // this exchange's parity
  if (mode == 1 && *reinterpret_cast<volatile int32_t*>(c.status + 1) != 0) return;   // frozen after a fault
  Waiter wt;

  if ((int)blockIdx.x >= n_sum_blocks) {
    // ---------------- birth candidates: push mine to rank g, pull rank g's ----------------
    const int g = (int)blockIdx.x - n_sum_blocks;
    if (g == c.rank) return;
    const int tid = threadIdx.x;
    const int32_t* my_hdr = reinterpret_cast<const int32_t*>(c.packet + (size_t)c.rank * c.pkt.bytes + c.pkt.off_hdr);
    const int my_n = my_hdr[0];
    {
      unsigned char* dst = peers.recv[g] + slot0 + (size_t)c.rank * L.slot_bytes + L.word_off;
      const uint32_t* h32 = reinterpret_cast<const uint32_t*>(my_hdr);
      const uint32_t* row = reinterpret_cast<const uint32_t*>(c.packet + (size_t)c.rank * c.pkt.bytes + c.pkt.off_cand_row);
      const uint32_t* t0 = reinterpret_cast<const uint32_t*>(c.packet + (size_t)c.rank * c.pkt.bytes + c.pkt.off_cand_t0);
      const uint32_t* cx = reinterpret_cast<const uint32_t*>(c.packet + (size_t)c.rank * c.pkt.bytes + c.pkt.off_cand_x);
      // candidates first, the header (which tells the receiver how many to expect) with them: every word carries its own flag
      for (int i = tid; i < my_n; i += blockDim.x) {
        ll_store_word(dst + (size_t)(8 + i) * 8, row[i], seq);
        ll_store_word(dst + (size_t)(8 + c.cap + i) * 8, t0[i], seq);
      }
      for (int i = tid; i < my_n * c.Dsum; i += blockDim.x) ll_store_word(dst + (size_t)(8 + 2 * c.cap + i) * 8, cx[i], seq);
      if (tid < 8) ll_store_word(dst + (size_t)tid * 8, h32[tid], seq);
    }
    {
      const unsigned char* src = recv_local + slot0 + (size_t)g * L.slot_bytes + L.word_off;
      unsigned char* pk = c.packet + (size_t)g * c.pkt.bytes;
      if (tid < 8) {
        uint32_t w = 0;
        if (!ll_load_word(src + (size_t)tid * 8, seq, &w, wt)) raise_fault(c);
        reinterpret_cast<uint32_t*>(pk + c.pkt.off_hdr)[tid] = w;
        if (tid == 0) s_ncand = wt.expired ? 0 : (int)w;
      }
      __syncthreads();
      const int n = min(max(s_ncand, 0), c.cap);
      for (int i = tid; i < n; i += blockDim.x) {
        uint32_t a = 0, b = 0;
        if (!ll_load_word(src + (size_t)(8 + i) * 8, seq, &a, wt) || !ll_load_word(src + (size_t)(8 + c.cap + i) * 8, seq, &b, wt)) raise_fault(c);
        reinterpret_cast<uint32_t*>(pk + c.pkt.off_cand_row)[i] = a;
        reinterpret_cast<uint32_t*>(pk + c.pkt.off_cand_t0)[i] = b;
      }
      for (int i = tid; i < n * c.Dsum; i += blockDim.x) {
        uint32_t a = 0;
        if (!ll_load_word(src + (size_t)(8 + 2 * c.cap + i) * 8, seq, &a, wt)) raise_fault(c);
        reinterpret_cast<uint32_t*>(pk + c.pkt.off_cand_x)[i] = a;
      }
    }
    return;
  }

  // ---------------- statistics ----------------
  const bool use_flags = delta && mode != 2 && c.stat_ctas <= 1024;
  if (use_flags) {
    for (int b = threadIdx.x; b < c.stat_ctas; b += blockDim.x) s_active[b] = (unsigned char)(c.cta_active[b] != 0);
    __syncthreads();
  }
  const size_t part_stride = (size_t)n_s1 + n_s2;
  const int e = threadIdx.x & 31, slice = threadIdx.x >> 5;
  double* pk_s1 = reinterpret_cast<double*>(c.packet + (size_t)c.rank * c.pkt.bytes + c.pkt.off_s1t);
  double* pk_s2 = reinterpret_cast<double*>(c.packet + (size_t)c.rank * c.pkt.bytes + c.pkt.off_s2t);
  int32_t* pk_cnt = reinterpret_cast<int32_t*>(c.packet + (size_t)c.rank * c.pkt.bytes + c.pkt.off_cnt);
  for (int blk = blockIdx.x; blk * 32 < n_el; blk += n_sum_blocks) {
    const int i = blk * 32 + e;
    double sum = 0.0;
    int n = 0;
    if (mode != 2) {
      if (i < n_s1 + n_s2) {
        for (int b = slice; b < c.stat_ctas; b += kRedSlices)
          if (!use_flags || s_active[b]) sum += (double)c.partial_f[(size_t)b * part_stride + i];
      } else if (i < n_el) {
        const int t = i - n_s1 - n_s2;
        for (int b = slice; b < c.stat_ctas; b += kRedSlices)
          if (!use_flags || s_active[b]) n += c.partial_n[(size_t)b * c.cap + t];
      }
      s_part[slice][e] = sum;
      s_cnt[slice][e] = n;
      __syncthreads();
    }
    if (slice == 0 && i < n_el) {
      const bool is_cnt = i >= n_s1 + n_s2;
      if (mode != 2) {
        sum = 0.0; n = 0;
#pragma unroll
        for (int j = 0; j < kRedSlices; ++j) { sum += s_part[j][e]; n += s_cnt[j][e]; }
        if (delta) {
          if (i < n_s1) sum += pk_s1[i];
          else if (!is_cnt) sum += pk_s2[i - n_s1];
          else n += pk_cnt[i - n_s1 - n_s2];
        }
        if (i < n_s1) pk_s1[i] = sum;
        else if (!is_cnt) pk_s2[i - n_s1] = sum;
        else pk_cnt[i - n_s1 - n_s2] = n;
      }
      double tot = sum;
      int ntot = n;
      if (mode == 1) {
        const unsigned long long mine = is_cnt ? (unsigned long long)(uint32_t)n : (unsigned long long)__double_as_longlong(sum);
        for (int g = 0; g < c.world; ++g)
          if (g != c.rank) ll_store_unit(peers.recv[g] + slot0 + (size_t)c.rank * L.slot_bytes + (size_t)i * 16, mine, seq);
        // all peers are polled together (their loads are independent: one round trip per pass, not one per peer); the
        // values are then added in rank order
        unsigned long long val[16];
        uint32_t pending = ((c.world >= 32) ? 0xffffffffu : ((1u << c.world) - 1u)) & ~(1u << c.rank);
        val[c.rank & 15] = mine;
        while (pending) {
#pragma unroll
          for (int g = 0; g < 16; ++g) {
            if (!((pending >> g) & 1u)) continue;
            uint32_t a, fa, b, fb;
            const void* src = recv_local + slot0 + (size_t)g * L.slot_bytes + (size_t)i * 16;
            asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(fa), "=r"(b), "=r"(fb) : "l"(src) : "memory");
            if (fa == seq && fb == seq) { val[g] = (unsigned long long)a | ((unsigned long long)b << 32); pending &= ~(1u << g); }
          }
          if (pending && !wt.keep_waiting()) {
            raise_fault(c);
#pragma unroll
            for (int g = 0; g < 16; ++g) if ((pending >> g) & 1u) val[g] = 0ull;
            pending = 0u;
          }
        }
        tot = 0.0; ntot = 0;
#pragma unroll
        for (int g = 0; g < 16; ++g) {                          // rank order, starting from rank 0's value
          if (g >= c.world) break;
          if (is_cnt) ntot += (int)(uint32_t)val[g];
          else tot = (g == 0) ? __longlong_as_double((long long)val[g]) : tot + __longlong_as_double((long long)val[g]);
        }
      } else if (mode == 2) {
        tot = 0.0; ntot = 0;
        for (int g = 0; g < c.world; ++g) {
          const unsigned char* pg = c.packet + (size_t)g * c.pkt.bytes;
          if (is_cnt) ntot += reinterpret_cast<const int32_t*>(pg + c.pkt.off_cnt)[i - n_s1 - n_s2];
          else {
            const double val = (i < n_s1) ? reinterpret_cast<const double*>(pg + c.pkt.off_s1t)[i]
                                          : reinterpret_cast<const double*>(pg + c.pkt.off_s2t)[i - n_s1];
            tot = (g == 0) ? val : tot + val;
          }
        }
      }
      if (mode != 0 || c.world == 1) {
        if (i < n_s1) c.sum_s1t[i] = tot;
        else if (!is_cnt) c.sum_s2t[i - n_s1] = tot;
        else c.sum_cnt[i - n_s1 - n_s2] = ntot;
      }
    }
    if (mode != 2) __syncthreads();                             // s_part is reused by the next element block
  }
}

cudaError_t launch_reduce_x(const Ctx& c, int mode, bool delta, const XchgPeers& peers, unsigned char* recv_local, cudaStream_t s) {
  const XchgLayout L = xchg_layout(c);
  const int n_el = (int)L.n_units;
  // every block of one launch, the `extra` ones included, is resident at once (3 per SM by the launch bounds): peers wait
  // for each other's pushes
  const int extra = (mode == 1) ? c.world : 0;
  int nb = (n_el + 31) / 32;
  if (nb > 148 * 3 - extra) nb = 148 * 3 - extra;
  return launch_chain(k_reduce_x, dim3(nb + extra), dim3(256), 0, s, c.pdl != 0, c, mode, delta ? 1 : 0, nb, peers, recv_local, L);
}

}  // namespace mv
