// mv_draw_tc.cu — likelihood + draw on the 5th-generation tensor cores (engines MVG_ENGINE_TCGEN05*).
//
// Shape: cap = 64 table slots, every view dense with dim 64, one to three views (BASELINE config C3 has three).
// One persistent CTA per SM walks row tiles of 128 customers.  For every (tile, view):
//
//   TMA producer (1 thread)    cp.async.bulk.tensor: the tile's [128 x 64] FP32 features arrive in
//                              shared memory as two K-halves of [128 x 32] in the 128B-swizzled
//                              K-major layout UMMA reads directly (4-deep ring plus an L2 prefetch of the tile-views behind it).
//   converters (2 x 128 thr.)  one warpgroup per K-half; thread r owns customer r: the remainder
//                              x_lo = x - trunc_tf32(x) (exact in FP32; two instructions per element), written
//                              with tcgen05.st into TMEM lane r (the remainder tile never touches shared
//                              memory).  |x|^2 is not recomputed here: it was stored when the view was uploaded.
//   MMA issuer (1 thread)      tcgen05.mma kind::tf32, M=128 N=64 K=8, three passes accumulated in
//                              one TMEM tile:  x.m_hi + x.m_lo (A = the raw tile in shared memory; the
//                              hardware reads the top 19 bits of each FP32 word, so it serves as
//                              x_hi) and x_lo.m_hi (A = the remainder tile in TMEM).  The split
//                              restores ~2^-19 relative accuracy (north_star: FP32 tolerance).
//   epilogue (4 x 128 threads) two PAIRS of warpgroups take alternate row tiles; inside a pair each
//                              warpgroup owns one half of the 64 tables.  tcgen05.ld: thread r of either
//                              warpgroup reads TMEM lane r = customer r, 16 dot products at a time.
//                              The B operand is the means PRE-SCALED by the table's slope (b = 2 A m, written by
//                              k_finalize), so a dot product is the data term of log2 f and the per-(customer, view,
//                              table) work is ONE packed add:
//                                  lw[t] = base[t] + sum_v A_vt (-|x_v|^2) + sum_v x_v.b_vt
//                              (base = log2 table mass + sum_v C_vt, staged per sweep).  The customer's own dish is
//                              scored with the customer removed (multiview_utils.cpp:138-192): that is a per-customer
//                              SCALAR correction delta_v = loo_v - plain_v from the dot product at its own table,
//                              added to the tables that serve the dish (usually its own table only).  With a free
//                              table slot the per-view marginal of a new table is a log-sum-exp over the dishes
//                              (MUFU ex2/lg2: a float statistic inside the stated tolerance, exported for the mirror);
//                              the categorical weights and the inverse-CDF scan stay bit-reproducible.  The two
//                              threads of a customer trade a few scalars through shared memory (three named-barrier
//                              rendezvous per tile) to merge marginals, totals and the inverse-CDF counts.
//
// TMEM (512 columns): [0,384) six accumulator tiles, [384,512) two remainder tiles.
// The [N x 64] log-likelihood matrices never exist in memory: HBM traffic is the features once
// (N*V*256 B) plus 8 B per customer (table in, choice out).
//
// Replaces, per customer: remove_customer + compute_table_probs_with_cache + the draw of
// /root/reference/Multiview/multiview_utils.cpp:71-192, :307-350 and multiview_gibbs.cpp:157-199.
#include <cuda.h>

#include "mv_ctx.h"
#include "mv_draw_screen.cuh"

namespace mv {

namespace {

constexpr int kTileRows = 128;
constexpr int kHalfCols = 32;                       // floats per 128-byte swizzled row
constexpr int kHalfBytes = kTileRows * 128;         // 16 KB: one K-half of an A tile
constexpr int kBHalfBytes = 64 * 128;               // 8 KB: one K-half of a B matrix (64 tables)
constexpr int kRawStages = 4;                       // K-halves of raw features in flight (64 KB) + L2 prefetch two tile-views ahead
constexpr int kLoStages = 2;                        // TMEM remainder tiles (64 columns each)
constexpr int kDStages = 6;                         // TMEM accumulator tiles (64 columns each): three per epilogue pair
constexpr int kTmemCols = 512;
constexpr int kLoCol0 = kDStages * 64;              // first TMEM column of the remainder tiles
constexpr int kMaxTcViews = 3;
constexpr int kThreads = 896;                       // WG0: control, WG1+WG2: converters (one per K-half), WG3..WG6: epilogue
constexpr int kMmaWarps = 2;                        // MMA-issuing warps of WG0; tile-view i belongs to warp 1 + i % 2
constexpr int kExFields = 16;                       // scalars two epilogue threads of one customer trade per tile
constexpr int kEpiGroups = 2;
constexpr int kTcViewParamBytes = 9 * 64 * 4;           // TcViewParams: nine per-table arrays

struct __align__(64) TcMaps {
  CUtensorMap x[kMaxTcViews];
  CUtensorMap mean_hi;
  CUtensorMap mean_lo;
};

// ---- shared memory carve-up (dynamic, 1024-byte aligned for SWIZZLE_128B) --------------------
struct SmemLayout {
  static constexpr int b_off = 0;                                            // [V][hi,lo][2 halves][8 KB]
  static constexpr int raw_off = b_off + kMaxTcViews * 4 * kBHalfBytes;      // 96 KB
  static constexpr int tp_off = raw_off + kRawStages * kHalfBytes;           // +112 KB
  static constexpr int tm_off = tp_off + kMaxTcViews * kTcViewParamBytes;          // per view: TcViewParams
  static constexpr int vp_off = tm_off + 64 * (int)sizeof(TableMass);
  static constexpr int lm_off = vp_off + kMaxTcViews * (int)sizeof(ViewParam);              // float[64]: base = LM + sum_v C_v of every table
  static constexpr int dlm_off = lm_off + 64 * (int)sizeof(float);                          // float[64]: LM1 - LM
  static constexpr int same_off = dlm_off + 64 * (int)sizeof(float);                        // u64[V][64]: same-dish table masks
  static constexpr int ex_off = same_off + kMaxTcViews * 64 * 8;
  static constexpr int bar_off = ex_off + 4 * kExFields * kTileRows * (int)sizeof(float);   // ex: [pair][half][field][row]
  static constexpr int n_bars = 2 * kRawStages + 2 * kLoStages + 2 * kDStages + 2;
  static constexpr int misc_off = bar_off + n_bars * 8;
  static constexpr int total = misc_off + 64;
};
static_assert(SmemLayout::total <= 227 * 1024, "shared memory budget");
static_assert(sizeof(screen::Scratch) <= 4 * kExFields * kTileRows * sizeof(float), "screening scratch in the exchange area");

// ---- PTX helpers ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"   // %2: suspend-time hint (ns): a waiting warp
      "@p bra DONE;\n\t"                                                 //     sleeps in hardware instead of polling
      "bra WAIT_LOOP;\n\t"                                               //     away the epilogue's issue slots
      "DONE:\n\t"
      "}\n" ::"r"(bar), "r"(parity), "r"(2000u)
      : "memory");
}
// mbar_wait that also adds the cycles spent waiting to *acc when profiling is on (debug_export & 2).
__device__ __forceinline__ void mbar_wait_t(uint32_t bar, uint32_t parity, bool prof, long long& acc) {
  if (prof) {
    const long long t0 = clock64();
    mbar_wait(bar, parity);
    acc += clock64() - t0;
  } else {
    mbar_wait(bar, parity);
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// Same with an L2 cache policy: the feature stream (768 MB per sweep at C3) is marked evict-first so that it
// does not push the resident working set (parameters, packets, the other kernels' code) out of the 126 MB L2.
__device__ __forceinline__ void tma_load_2d_hint(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1,
                                                 uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// cute::UMMA::InstrDescriptor for kind::tf32: D = F32 (1 at [4,6)), A = B = TF32 (2 at [7,10) and
// [10,13)), both K-major, N >> 3 at [17,23), M >> 4 at [24,29).
constexpr uint32_t kIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((64u >> 3) << 17) | ((128u >> 4) << 24);

// The shared-memory operand descriptor is 64 bits; everything that varies per MMA (the start address,
// bits [0,14), in 16-byte units) lives in the low word, so the issuer only ever adds to `lo`.
template <bool ACC>
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 da, {%1, %3};\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %4, p;\n\t"
      "}\n" ::"r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(kIdesc), "n"(ACC ? 1 : 0)
      : "memory");
}
// Same with the A operand in tensor memory: lane = row, one 32-bit column per K element.
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t desc_hi) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 db;\n\t"
      "setp.ne.b32 p, 1, 0;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], db, %4, p;\n\t"
      "}\n" ::"r"(d_tmem), "r"(a_tmem), "r"(b_lo), "r"(desc_hi), "r"(kIdesc)
      : "memory");
}
__device__ __forceinline__ void tmem_st_16(uint32_t taddr, const uint32_t (&u)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]),
        "r"(u[8]), "r"(u[9]), "r"(u[10]), "r"(u[11]), "r"(u[12]), "r"(u[13]), "r"(u[14]), "r"(u[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// K-major, SWIZZLE_128B operand descriptor (cute::UMMA::SmemDescriptor): start address >> 4 in bits
// [0,14), leading byte offset [16,30) (unused for swizzled K-major: 1), stride byte offset [32,46) =
// 1024 B between 8-row groups, version 1 at [46,48), layout type SWIZZLE_128B = 2 at [61,64).
__device__ __forceinline__ uint32_t desc_lo(uint32_t smem_addr) { return ((smem_addr >> 4) & 0x3FFFu) | (1u << 16); }
constexpr uint32_t kDescHi = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);

// One lane of a converged warp (cute::elect_one_sync): lets ptxas keep single-lane tcgen05 issue
// free of the lane-serialising loop it otherwise wraps around uniform-datapath instructions.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n" : "=r"(pred));
  return pred != 0;
}

// Programmatic dependent launch: when this kernel is launched as the programmatic successor of k_finalize (the sweep graph,
// csrc/mv_capi.cu), its CTAs start while k_finalize is still running; everything k_finalize (or an earlier kernel of the
// sweep) writes may only be touched after this wait.  A no-op for an ordinary launch.
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <int REGS> __device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS)); }
template <int REGS> __device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS)); }

struct Ring {   // stage index + mbarrier phase parity of one pipeline role
  int stage = 0;
  uint32_t phase = 0;
  int n;
  __device__ explicit Ring(int n_) : n(n_) {}
  __device__ __forceinline__ void next() { if (++stage == n) { stage = 0; phase ^= 1u; } }
};

}  // namespace

// 16 consecutive accumulator columns of this thread's TMEM lane (issue only; pair with tmem_ld_wait).
__device__ __forceinline__ void tmem_ld_16(uint32_t taddr, uint32_t (&u)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
        "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- per-sweep parameters of one view as the epilogue reads them (built at kernel start from TableParam) ----------
struct __align__(16) TcViewParams {
  float A[64], C[64], W[64];          // per table, read four tables at a time
  float A1[64], C1[64], R[64], W1[64];// the customer's own table: leave-one-out slope / offset, R = A1 / A, W with l_vk - 1
  int32_t lone[64];
  float CW[64];                       // C + W: the constant of a dish's term of the new-table marginal (masked like W)
};
static_assert(sizeof(TcViewParams) == kTcViewParamBytes, "parameter staging area");

// -trunc_tf32(x): mantissa cut to 10 bits; the negation folds into the consuming add
__device__ __forceinline__ float neg_trunc_tf32(float x) { return -__uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }
__device__ __forceinline__ float ex2f(float d) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d)); return r; }
__device__ __forceinline__ float lg2f(float d) { float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d)); return r; }

// u[i & 15] for a per-thread index: a binary tree of 15 selects (registers cannot be indexed).
__device__ __forceinline__ float pick16(const uint32_t (&u)[16], int i) {
  const bool b0 = i & 1, b1 = i & 2, b2 = i & 4, b3 = i & 8;
  uint32_t a[8], b[4];
#pragma unroll
  for (int k = 0; k < 8; ++k) a[k] = b0 ? u[2 * k + 1] : u[2 * k];
#pragma unroll
  for (int k = 0; k < 4; ++k) b[k] = b1 ? a[2 * k + 1] : a[2 * k];
  const uint32_t c0 = b2 ? b[1] : b[0], c1 = b2 ? b[3] : b[2];
  return __uint_as_float(b3 ? c1 : c0);
}

// lw2[BASE/2 ..] += the 16 dot products of one chunk (tables tbase + BASE ..), optionally exported first.
template <int BASE>
__device__ __forceinline__ void add_chunk(float2 (&lw2)[16], const uint32_t (&u)[16], const Ctx& c, int row, int v, int tbase, bool live) {
  if (live) {
    float* da = c.dbg_acc + ((size_t)row * c.V + v) * 64 + tbase + BASE;
#pragma unroll
    for (int t = 0; t < 16; ++t) da[t] = __uint_as_float(u[t]);
  }
#pragma unroll
  for (int p = 0; p < 8; ++p)
    lw2[BASE / 2 + p] = fadd2(lw2[BASE / 2 + p], make_float2(__uint_as_float(u[2 * p]), __uint_as_float(u[2 * p + 1])));
}

// Streaming log-sum-exp over the dishes of one chunk for the new-table marginal (a free slot exists):
// term_t = (x.b_t + (A_t (-|x|^2) + C_t)) + W_t, W masked except at the lowest table of each dish.  MUFU exponentials:
// the marginal is a float statistic (tolerance), not part of the bit-reproducible draw.
// MASKED: the term of table `skip` (relative to tbase; the lowest table of the customer's own dish) is left out here and
// now.  The cheap alternative — sum everything and subtract that one term afterwards — cancels catastrophically when the
// own dish dominates the sum AND its leave-one-out term is much smaller than its plain term, i.e. for small dishes (a
// newborn table: the dish is the customer itself); the caller picks MASKED per warp for exactly those.
template <int BASE, bool MASKED>
__device__ __forceinline__ void lse_chunk(const TcViewParams& P, int tbase, const uint32_t (&u)[16], float nxx, int skip, float& mx, float& s) {
  float2 term[8];
  float c0 = kMasked, c1 = kMasked;
  const float2 nxx2 = splat2(nxx);
  const float4* A4 = reinterpret_cast<const float4*>(P.A + tbase + BASE);
  const float4* CW4 = reinterpret_cast<const float4*>(P.CW + tbase + BASE);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 a = A4[q], cw = CW4[q];
    term[2 * q] = fadd2(make_float2(__uint_as_float(u[4 * q]), __uint_as_float(u[4 * q + 1])), ffma2(make_float2(a.x, a.y), nxx2, make_float2(cw.x, cw.y)));
    term[2 * q + 1] = fadd2(make_float2(__uint_as_float(u[4 * q + 2]), __uint_as_float(u[4 * q + 3])), ffma2(make_float2(a.z, a.w), nxx2, make_float2(cw.z, cw.w)));
    if (MASKED) {
      if (skip == BASE + 4 * q) term[2 * q].x = kMasked;
      if (skip == BASE + 4 * q + 1) term[2 * q].y = kMasked;
      if (skip == BASE + 4 * q + 2) term[2 * q + 1].x = kMasked;
      if (skip == BASE + 4 * q + 3) term[2 * q + 1].y = kMasked;
    }
    c0 = fmaxf(c0, fmaxf(term[2 * q].x, term[2 * q + 1].x));
    c1 = fmaxf(c1, fmaxf(term[2 * q].y, term[2 * q + 1].y));
  }
  const float mn = fmaxf(mx, fmaxf(c0, c1));
  s *= ex2f(mx - mn);
  mx = mn;
  const float2 nmn2 = splat2(-mn);
  float2 acc2;
#pragma unroll
  for (int p = 0; p < 8; ++p) {
    const float2 d = fadd2(term[p], nmn2);
    const float2 e = make_float2(ex2f(d.x), ex2f(d.y));
    acc2 = (p == 0) ? e : fadd2(acc2, e);
  }
  s += acc2.x + acc2.y;
}

template <bool B> struct BoolC { static constexpr bool value = B; };

// FAST: categorical weights through MUFU as well (tolerance-level draws).  DEBUG: the handle exports per-row intermediates
// (debug_export bit 0) and / or per-role wait counters (bit 1); a separate instantiation keeps that code and its registers
// out of the production kernel.
template <bool FAST, bool DEBUG>
__global__ void __launch_bounds__(kThreads, 1) k_draw_tc(const Ctx c, const __grid_constant__ TcMaps maps) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int V = c.V;

  unsigned char* s_tp = smem + SmemLayout::tp_off;   // per view 2 KB: PairHot[32] (hot, pair-interleaved) then TableCold[64]
  TableMass* s_tm = reinterpret_cast<TableMass*>(smem + SmemLayout::tm_off);
  ViewParam* s_vp = reinterpret_cast<ViewParam*>(smem + SmemLayout::vp_off);
  float* s_lm = reinterpret_cast<float*>(smem + SmemLayout::lm_off);
  uint32_t* s_misc = reinterpret_cast<uint32_t*>(smem + SmemLayout::misc_off);   // [0] TMEM base, [1] sweep, [2..3] GlobalParam floats,
                                                                                 // [4] all_lone, [5] screening mode, [6..12] its bound coefficients,
                                                                                 // [13] tiles of this CTA on the screening list

  // barrier addresses
  const uint32_t bar0 = sbase + SmemLayout::bar_off;
  auto raw_full = [&](int s) { return bar0 + 8u * s; };
  auto raw_empty = [&](int s) { return bar0 + 8u * (kRawStages + s); };
  auto lo_full = [&](int s) { return bar0 + 8u * (2 * kRawStages + s); };
  auto lo_empty = [&](int s) { return bar0 + 8u * (2 * kRawStages + kLoStages + s); };
  auto d_full = [&](int s) { return bar0 + 8u * (2 * kRawStages + 2 * kLoStages + s); };
  auto d_empty = [&](int s) { return bar0 + 8u * (2 * kRawStages + 2 * kLoStages + kDStages + s); };
  const uint32_t b_full = bar0 + 8u * (2 * kRawStages + 2 * kLoStages + 2 * kDStages);
  const uint32_t list_full = b_full + 8u;            // the screening verdict and this CTA's tile list are in place

  // ---- one-time setup --------------------------------------------------------------------------
  // Nothing here depends on the previous kernels of the sweep: with a programmatic launch it runs — like the first
  // feature loads and their conversion below — while k_finalize is still computing the parameters.
  TcViewParams* s_p = reinterpret_cast<TcViewParams*>(s_tp);
  float* s_dlm = reinterpret_cast<float*>(smem + SmemLayout::dlm_off);
  unsigned long long* s_same = reinterpret_cast<unsigned long long*>(smem + SmemLayout::same_off);
  if (tid == 0) {
    s_misc[4] = 1u;                                    // all_lone, and-ed down by the threads that stage the parameters
    for (int s = 0; s < kRawStages; ++s) { mbar_init(raw_full(s), 1); mbar_init(raw_empty(s), 5); }     // the four warps of one converter warpgroup + the MMA commit
    for (int s = 0; s < kLoStages; ++s) { mbar_init(lo_full(s), 8); mbar_init(lo_empty(s), 1); }        // the eight converter warps
    for (int s = 0; s < kDStages; ++s) { mbar_init(d_full(s), 1); mbar_init(d_empty(s), 8); }     // the eight warps of a pair
    // (arrivals are per WARP — one lane after __syncwarp — not per thread: a waiter sleeping on the barrier is woken by every
    //  arrival, and 256 wake-ups per phase cost the epilogue's schedulers issue slots)
    mbar_init(b_full, 1);
    mbar_init(list_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) {   // TMEM allocation: one warp, address published through shared memory
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_misc[0])), "n"(kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s_misc[0];

  const int n_tiles = (c.n_rows + kTileRows - 1) / kTileRows;
  // The tiles this launch evaluates: all of them, or those of its own tiles that the screening of the epilogue warpgroups
  // (DESIGN.md §4.1.1) could not settle, listed at scr_work[blockIdx.x + j * gridDim.x], j < s_misc[13].  Every role walks
  // the same sequence k = blockIdx.x, + gridDim.x, ... below the returned bound.
  auto work_list = [&](const int*& list) -> int {
    list = nullptr;
    if (!c.screen) return n_tiles;
    mbar_wait(list_full, 0);
    if (s_misc[5] != (uint32_t)kScreenSkip) return n_tiles;
    list = c.scr_work;
    return (int)blockIdx.x + (int)s_misc[13] * (int)gridDim.x;
  };
  const bool prof = DEBUG && (c.debug_export & 2) != 0 && c.dbg_prof != nullptr;
  const bool dbg_rows = DEBUG && (c.debug_export & 1) != 0;
  long long* prof_out = prof ? c.dbg_prof + (size_t)blockIdx.x * 16 : nullptr;
  long long w0 = 0, w1 = 0, w2 = 0;
  const long long t_start = prof ? clock64() : 0;

  if (warp < 4) {
    // =========================== WG0: control ==================================================
    reg_dec<24>();
    if (warp == 0 && lane == 0) {
      // ---- TMA producer ----
      // The features do not depend on the sweep's parameters: the first ring of tile halves is requested right away; the
      // B operand (this sweep's scaled means, written by k_finalize) only after the grid dependency has resolved.
      Ring r(kRawStages);
      const uint64_t stream_policy = l2_evict_first_policy();
      int issued = 0;
      bool b_loaded = false;
      auto load_b = [&]() {
        grid_dependency_wait();
        mbar_expect_tx(b_full, (uint32_t)(V * 4 * kBHalfBytes));
        for (int v = 0; v < V; ++v)
          for (int part = 0; part < 2; ++part)         // 0: b_hi, 1: b_lo
            for (int h = 0; h < 2; ++h)
              tma_load_2d(sbase + SmemLayout::b_off + ((v * 2 + part) * 2 + h) * kBHalfBytes,
                          part ? &maps.mean_lo : &maps.mean_hi, b_full, h * kHalfCols, v * 64);
        b_loaded = true;
      };
      const int* list;
      const int n_work = work_list(list);
      for (int k = blockIdx.x; k < n_work; k += gridDim.x) {
        const int tile = list ? list[k] : k;
        const int kn = k + gridDim.x;
        const int tn = (kn < n_work) ? (list ? list[kn] : kn) : -1;
        for (int v = 0; v < V; ++v)
#pragma unroll 1
          for (int h = 0; h < 2; ++h) {
            if (issued == kRawStages && !b_loaded) load_b();   // the ring is full: nothing more to do without the MMAs
            mbar_wait_t(raw_empty(r.stage), r.phase ^ 1u, prof, w0);
            mbar_expect_tx(raw_full(r.stage), kHalfBytes);
            tma_load_2d_hint(sbase + SmemLayout::raw_off + r.stage * kHalfBytes, &maps.x[v], raw_full(r.stage),
                             h * kHalfCols, tile * kTileRows, stream_policy);
            {                                           // pull the same half of the CTA's next tile into L2 meanwhile
              if (tn >= 0)
                asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.L2::cache_hint [%0, {%1, %2}], %3;"
                             ::"l"(reinterpret_cast<uint64_t>(&maps.x[v])), "r"(h * kHalfCols), "r"(tn * kTileRows),
                               "l"(stream_policy) : "memory");
            }
            r.next();
            ++issued;
          }
      }
      if (!b_loaded && n_work > (int)blockIdx.x) load_b();   // a CTA whose screened list is empty needs no B operand
      if (prof) { prof_out[0] = w0; prof_out[1] = clock64() - t_start; }
    } else if (warp >= 1 && warp <= kMmaWarps) {
      // ---- MMA issuers: warps 1 and 2 take alternate tile-views.  One tcgen05.mma of this shape keeps the
      //      tensor pipe busy for 32 cycles but costs its issuing warp ~100 cycles of uniform-datapath
      //      bookkeeping, so a single issuer cannot feed the pipe.  An mbarrier phase is one parity bit: a
      //      waiter that is a whole use ahead would sail through, so every barrier must be waited on in
      //      use order by ONE thread of control.  The stage counts are chosen for that: tile-view i goes to
      //      warp i % 2, and raw stages (4 = 2 per tile-view), remainder stages (2) and accumulator stages
      //      (6) all give consecutive uses of a stage the same parity of i.  The whole warp walks the loop
      //      (descriptor arithmetic stays warp-uniform); one elected lane issues. ----
      const int me = warp - 1;
      const uint32_t a_me = desc_lo(sbase + SmemLayout::raw_off + me * 2 * kHalfBytes);   // this warp's two raw stages
      const uint32_t b_lo0 = desc_lo(sbase + SmemLayout::b_off);
      const uint32_t lo_tmem = tmem_base + (uint32_t)(kLoCol0 + me * 64);                 // this warp's remainder stage
      const int* list;
      const int n_work = work_list(list);
      const int n_tv = (n_work > (int)blockIdx.x) ? ((n_work - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x) * V : 0;
      if (n_tv > 0) {                                // the producer loads the B operand exactly when this CTA has work
        mbar_wait(b_full, 0);
        tc_fence_after();
      }
      int v = me % V, ds = me;                       // view and accumulator stage of tile-view i
      const int vstep = kMmaWarps % V;
      uint32_t use = 0;                              // how many tile-views this warp has issued
      uint32_t dph = 0;                              // accumulator-stage phase: flips every third tile-view of this warp
      int dcnt = 0;
      for (int i = me; i < n_tv; i += kMmaWarps) {
        const uint32_t ph = use & 1u;                // raw and remainder stages: one use per tile-view of this warp
        mbar_wait_t(d_empty(ds), dph ^ 1u, prof, w0);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(ds * 64);
        const uint32_t b_v = b_lo0 + (uint32_t)(v * 4 * (kBHalfBytes >> 4));   // [hi|lo][h] blocks of this view
        // passes 1+2 on the raw halves: x_hi . m_hi  and  x_hi . m_lo   (4 x K=8 per 128-byte row, +32 B each)
        mbar_wait_t(raw_full(2 * me), ph, prof, w1);
        tc_fence_after();
        if (elect_one()) {
          umma_tf32<false>(d_tmem, a_me, b_v, kDescHi);
#pragma unroll
          for (int k = 1; k < 4; ++k) umma_tf32<true>(d_tmem, a_me + 2 * k, b_v + 2 * k, kDescHi);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_tf32<true>(d_tmem, a_me + 2 * k, b_v + 2 * (kBHalfBytes >> 4) + 2 * k, kDescHi);
          umma_commit(raw_empty(2 * me));             // this raw half is free once these MMAs retire
        }
        __syncwarp();
        mbar_wait_t(raw_full(2 * me + 1), ph, prof, w1);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a = a_me + (uint32_t)(kHalfBytes >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_tf32<true>(d_tmem, a + 2 * k, b_v + (kBHalfBytes >> 4) + 2 * k, kDescHi);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_tf32<true>(d_tmem, a + 2 * k, b_v + 3 * (kBHalfBytes >> 4) + 2 * k, kDescHi);
          umma_commit(raw_empty(2 * me + 1));
        }
        __syncwarp();
        // pass 3 from tensor memory: x_lo . m_hi
        mbar_wait_t(lo_full(me), ph, prof, w2);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_tf32_ts(d_tmem, lo_tmem + (uint32_t)(k * 8), b_v + 2 * k, kDescHi);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_tf32_ts(d_tmem, lo_tmem + (uint32_t)(32 + k * 8), b_v + (kBHalfBytes >> 4) + 2 * k, kDescHi);
          umma_commit(lo_empty(me));
          umma_commit(d_full(ds));
        }
        __syncwarp();
        ++use;
        v += vstep; if (v >= V) v -= V;              // view of tile-view i + 2 (vstep = 2 mod V, no division on the issue path)
        ds += kMmaWarps; if (ds >= kDStages) ds -= kDStages;
        if (++dcnt == kDStages / kMmaWarps) { dcnt = 0; dph ^= 1u; }
      }
      if (prof && lane == 0 && me == 0) { prof_out[2] = w0; prof_out[3] = w1; prof_out[4] = w2; prof_out[5] = clock64() - t_start; }
    }
  } else if (warp < 12) {
    // =========================== WG1, WG2: converters, one K-half each ===========================
    reg_dec<48>();
    const int h = (warp >> 2) - 1;                     // K-half of this warpgroup
    const int r = tid & 127;                           // row of the tile = 128-byte line of the half = TMEM lane
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t line = (uint32_t)r * 128u;
    int i = 0;                                         // tile-view counter of this CTA
    const int* list;
    const int n_work = work_list(list);
    for (int k = blockIdx.x; k < n_work; k += gridDim.x)
      for (int v = 0; v < V; ++v, ++i) {
        const int rs = (2 * i + h) % kRawStages;
        const uint32_t rph = (uint32_t)((2 * i + h) / kRawStages) & 1u;
        const int ls = i % kLoStages;
        const uint32_t lph = (uint32_t)(i / kLoStages) & 1u;
        mbar_wait_t(raw_full(rs), rph, prof, w0);
        mbar_wait_t(lo_empty(ls), lph ^ 1u, prof, w1);
        tc_fence_after();
        const unsigned char* src = smem + SmemLayout::raw_off + rs * kHalfBytes + line;
        const uint32_t lo_addr = tmem_base + lane_base + (uint32_t)(kLoCol0 + ls * 64 + h * 32);
#pragma unroll
        for (int half16 = 0; half16 < 2; ++half16) {
          uint32_t lo[16];
#pragma unroll
          for (int cc = 0; cc < 4; ++cc) {             // logical 16-byte chunk cidx sits at physical chunk cidx ^ (r & 7)
            const int cidx = half16 * 4 + cc;
            const float4 x4 = *reinterpret_cast<const float4*>(src + ((cidx ^ (r & 7)) << 4));
            // the tensor core reads trunc_tf32(x); the remainder x - trunc_tf32(x) is exact in FP32 and the
            // hardware again keeps its top 19 bits: x_hi + x_lo carries >= 21 significant bits of x
            const float2 l01 = fadd2(make_float2(x4.x, x4.y), make_float2(neg_trunc_tf32(x4.x), neg_trunc_tf32(x4.y)));
            const float2 l23 = fadd2(make_float2(x4.z, x4.w), make_float2(neg_trunc_tf32(x4.z), neg_trunc_tf32(x4.w)));
            lo[cc * 4 + 0] = __float_as_uint(l01.x);
            lo[cc * 4 + 1] = __float_as_uint(l01.y);
            lo[cc * 4 + 2] = __float_as_uint(l23.x);
            lo[cc * 4 + 3] = __float_as_uint(l23.y);
          }
          tmem_st_16(lo_addr + (uint32_t)(half16 * 16), lo);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(raw_empty(rs));     // this warp no longer reads the raw half
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(lo_full(ls));
      }
    if (prof && r == 0) { prof_out[6 + 3 * h] = w0; prof_out[7 + 3 * h] = w1; prof_out[8 + 3 * h] = clock64() - t_start; }
  } else {
    // =========================== WG3..WG6: epilogue (thread r <-> TMEM lane r <-> customer r) ====
    // pool: 896 threads x 72 registers = 128 x (24 + 2*48 + 4*96)
    reg_inc<96>();
    // ---- this sweep's parameters: staged by the 512 epilogue threads once the grid dependency has resolved ----
    grid_dependency_wait();
    {
      const int et = tid - 3 * 128;                     // 0 .. 511
      if (et == 0) {
        kclock_begin(c.kclock + kClockDraw);            // the launch's clock runs from the moment its inputs exist
        // The kernels of the sweep's tail may queue up behind this grid from here on (mv_ctx.h) — not earlier: what they
        // read ahead of their own wait (k_finalize: the sweep-start state) must come from a COMPLETED previous finalize.
        pdl_trigger();
      }
      // One round of loads for the staging and the screening verdict (screen::load): threads et < V * 64 take (view, table)
      // et, threads 256 + t table t's masses.
      screen::Inputs in;
      unsigned long long same = 0ull;
      float cv[kMaxTcViews] = {0.0f, 0.0f, 0.0f};
      if (c.screen) {
        screen::load(c, et, in);
      } else {
        in.g = *c.gparam;
        if (et < V * 64) in.q = c.tparam[et];
        else if (et >= 256 && et < 256 + 64) in.m = c.tmass[et - 256];
      }
      if (et < V * 64) same = c.tsame[et];
      else if (et >= 256 && et < 256 + 64)
        for (int v = 0; v < V; ++v) cv[v] = c.tparam[v * 64 + et - 256].C;
      const ViewParam vp = (et < V) ? c.vparam[et] : ViewParam{};
      int lone_ok = 1;                                  // every live table's dishes are served by that table alone?
      if (et < V * 64) {
        const int v = et >> 6, t = et & 63;
        const TableParam& q = in.q;
        TcViewParams& P = s_p[v];
        P.A[t] = q.A; P.C[t] = q.C; P.W[t] = q.W; P.CW[t] = __fadd_rn(q.C, q.W);
        P.A1[t] = q.A1; P.C1[t] = q.C1; P.W1[t] = q.W1;
        P.R[t] = (q.A != 0.0f) ? __fdiv_rn(q.A1, q.A) : 0.0f;
        // bit 0: the dish is served by this table alone; bit 1: the dish is SMALL (<= ~500 customers: R = 1 + 2 / (tau + n - 1),
        // or n < 2), where removing the customer changes its likelihood by orders of magnitude (see lse_chunk)
        P.lone[t] = (q.lone ? 1 : 0) | ((q.dish >= 0 && (P.R[t] > 1.004f || P.R[t] == 0.0f)) ? 2 : 0);
        if (q.dish >= 0 && !q.lone) lone_ok = 0;
        s_same[et] = same;
      } else if (et >= 256 && et < 256 + 64) {
        const int t = et - 256;
        const TableMass& m = in.m;
        s_tm[t] = m;
        float b = m.LM;
        for (int v = 0; v < V; ++v) b = __fadd_rn(b, cv[v]);
        s_lm[t] = b;                                    // base: log2 table mass + the views' offsets, in view order
        s_dlm[t] = __fadd_rn(m.LM1, -m.LM);             // what changes for the customer's own table (n_t - 1)
      }
      if (et < V) s_vp[et] = vp;
      if (et == 64) {
        s_misc[1] = in.g.sweep;
        s_misc[2] = __float_as_uint(in.g.LMN0);
        s_misc[3] = __float_as_uint(in.g.LMN1);
      }
      if (c.screen) {
        // The screening verdict of this sweep, its bound coefficients and, in a skip sweep, this CTA's list.  The other
        // roles wait for the verdict and the list only; the bookkeeping of the last CTA comes after their release.
        screen::Scratch* S = reinterpret_cast<screen::Scratch*>(smem + SmemLayout::ex_off);
        const int mode = screen::decide(c, et, in, S, reinterpret_cast<float*>(s_misc + 6));
        if (et == 0) {
          s_misc[5] = (uint32_t)mode;
          s_misc[13] = (uint32_t)S->n_eval;
          mbar_arrive(list_full);
        }
        if (mode != kScreenOff) screen::publish(c, et, mode, in.g.sweep, S);
      } else if (et == 0) {
        s_misc[5] = (uint32_t)kScreenOff;
      }
      if (!lone_ok) atomicAnd(&s_misc[4], 0u);
      asm volatile("bar.sync 9, 512;" ::: "memory");    // the epilogue warpgroups only: the other roles never read these
    }
    const uint32_t sweep = s_misc[1];
    GlobalParam gp;
    gp.LMN0 = __uint_as_float(s_misc[2]);
    gp.LMN1 = __uint_as_float(s_misc[3]);
    const bool all_lone_rt = s_misc[4] != 0u;
    const bool record_rt = s_misc[5] != (uint32_t)kScreenOff;   // then with_new is off and all_lone on (screening's precondition)
    const int* list;
    const int n_work = work_list(list);
    // Two CTA-uniform properties of the sweep select one of four copies of the loop, so that the registers and the code of
    // the rarer cases stay out of the common one:
    //   with_new   a table slot is free: the new-table option has weight and the per-view marginals are evaluated;
    //   all_lone   every live table's dishes are served by that table alone: the leave-one-out correction touches the
    //              customer's own table only.
    auto epilogue = [&](auto WN, auto AL) {
    constexpr bool with_new = decltype(WN)::value;
    constexpr bool all_lone = decltype(AL)::value;
    const int wg = (warp >> 2) - 3;
    const int pair = wg >> 1;                          // this pair takes tiles j = pair, pair+2, ...
    const int hf = wg & 1;                             // tables [32 hf, 32 hf + 32)
    const int tb = 32 * hf;
    const int r = tid & 127;
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    float* ex_own = reinterpret_cast<float*>(smem + SmemLayout::ex_off) + ((pair * 2 + hf) * kExFields) * kTileRows + r;
    float* ex_oth = reinterpret_cast<float*>(smem + SmemLayout::ex_off) + ((pair * 2 + (hf ^ 1)) * kExFields) * kTileRows + r;
    // exchange fields: 0-5 (mx, s) of the views' dish sums, 6-8 the own-dish term per view, 9 half maximum, 10 half total,
    // 11 uniform / upper count, 12-14 the leave-one-out corrections (only when tables share dishes)
    // the two threads of a customer sit in the same warp slot of the pair's two warpgroups: only those two warps meet
    auto rendezvous = [&]() { asm volatile("bar.sync %0, 64;" ::"r"(1 + pair * 4 + (warp & 3)) : "memory"); };
    const float4* base4 = reinterpret_cast<const float4*>(s_lm + tb);
    // margins (DESIGN.md §4.1.1): only the variant without a new-table option and with lone dishes records them
    constexpr bool can_record = !with_new && all_lone;
    const bool record = can_record && record_rt;
    int j = pair;
    const int k0 = blockIdx.x + pair * gridDim.x;
    const int tile0 = (k0 < n_work) ? (list ? list[k0] : k0) : n_tiles;
    int t0_next = (tile0 < n_tiles) ? c.table_cur[min(tile0 * kTileRows + r, c.n_rows - 1)] : 0;
    // |x|^2 of the customer in every view: computed once when the view was uploaded (c.xx), fetched a tile ahead
    float xx_next[kMaxTcViews];
#pragma unroll
    for (int v = 0; v < kMaxTcViews; ++v)
      xx_next[v] = (tile0 < n_tiles) ? c.xx[(size_t)v * c.xx_stride + min(tile0 * kTileRows + r, c.n_rows - 1)] : 0.0f;   // (xx has >= 3 rows)
    long long ph[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, tlast = prof ? clock64() : 0;      // DEBUG: cycles per phase of the tile loop
    auto phase = [&](int k) { if (prof) { const long long now = clock64(); ph[k] += now - tlast; tlast = now; } };
    int tile_next = tile0;
    for (int k = k0; k < n_work; k += kEpiGroups * gridDim.x, j += kEpiGroups) {
      const int tile = tile_next;
      const int row = tile * kTileRows + r;
      const bool live = row < c.n_rows;
      const int rowc = live ? row : (c.n_rows - 1);
      const int t0 = t0_next;
      const int single = s_tm[t0].single;
      const int rel = t0 - tb;                        // the customer's own table inside this half?
      const bool mine = (unsigned)rel < 32u;
      float xxv[kMaxTcViews];
#pragma unroll
      for (int v = 0; v < kMaxTcViews; ++v) xxv[v] = xx_next[v];
      {                                               // the next tile's tables and norms travel while this one is computed
        const int kn = k + kEpiGroups * gridDim.x;
        const int tn = (kn < n_work) ? (list ? list[kn] : kn) : n_tiles;
        tile_next = tn;
        if (tn < n_tiles) {
          const int rn = min(tn * kTileRows + r, c.n_rows - 1);
          t0_next = c.table_cur[rn];
#pragma unroll
          for (int v = 0; v < kMaxTcViews; ++v) xx_next[v] = c.xx[(size_t)v * c.xx_stride + rn];
        }
      }
      // lw = base + sum_v A_v (-|x_v|^2): everything that does not need the dot products, before they arrive
      float2 lw2[16];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 q = base4[i];
        lw2[2 * i] = make_float2(q.x, q.y);
        lw2[2 * i + 1] = make_float2(q.z, q.w);
      }
#pragma unroll
      for (int v = 0; v < kMaxTcViews; ++v) {
        if (v < V) {
          const float2 nxx2 = splat2(-xxv[v]);
          const float4* A4 = reinterpret_cast<const float4*>(s_p[v].A + tb);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 a = A4[i];
            lw2[2 * i] = ffma2(make_float2(a.x, a.y), nxx2, lw2[2 * i]);
            lw2[2 * i + 1] = ffma2(make_float2(a.z, a.w), nxx2, lw2[2 * i + 1]);
          }
        }
      }
      float dsum = 0.0f;                              // ((0 + delta_0) + delta_1) + delta_2
      phase(0);
      for (int v = 0; v < V; ++v) {
        const int idx = j * V + v;
        const int stage = idx % kDStages;             // V = 3: stages 0-2 serve this CTA's even tiles, 3-5 the odd ones
        mbar_wait_t(d_full(stage), (uint32_t)(idx / kDStages) & 1u, prof, w0);
        tc_fence_after();
        const uint32_t taddr = tmem_base + lane_base + (uint32_t)(stage * 64 + tb);
        const float xx = (v == 0) ? xxv[0] : ((v == 1) ? xxv[1] : xxv[2]);
        const float nxx = -xx;
        const TcViewParams& P = s_p[v];
        if (dbg_rows && live && hf == 0) c.dbg_xx[(size_t)row * V + v] = xx;
        // 16 dot products at a time through ONE register buffer (two live buffers do not fit beside the 32 running log-weights)
        uint32_t u[16];
        tmem_ld_16(taddr, u);
        float mx = kMasked, s = 0.0f;
        const int rep = all_lone ? t0 : (__ffsll((long long)s_same[v * 64 + t0]) - 1);   // lowest table of the own dish
        const int rrel = rep - tb;
        // own dish small and its term in this half: leave it out exactly (warp-uniform choice of the variant)
        const bool masked = with_new && __any_sync(0xffffffffu, (unsigned)rrel < 32u && (P.lone[t0] & 2));
        tmem_ld_wait();
        add_chunk<0>(lw2, u, c, row, v, tb, live && dbg_rows);
        if (with_new) {
          if (masked) lse_chunk<0, true>(P, tb, u, nxx, rrel, mx, s);
          else lse_chunk<0, false>(P, tb, u, nxx, rrel, mx, s);
        }
        const float pa = pick16(u, rel);
        float pra = 0.0f;
        if (with_new && !all_lone && !masked) pra = pick16(u, rrel);
        tmem_ld_16(taddr + 16, u);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(d_empty(stage));   // this warp's columns are in registers
        add_chunk<16>(lw2, u, c, row, v, tb, live && dbg_rows);
        if (with_new) {
          if (masked) lse_chunk<16, true>(P, tb, u, nxx, rrel, mx, s);
          else lse_chunk<16, false>(P, tb, u, nxx, rrel, mx, s);
        }
        const float pb = pick16(u, rel);
        // the customer's own table in this view: plain and leave-one-out value of log2 f from its dot product
        const float own_acc = (rel & 16) ? pb : pa;
        const float plain = __fadd_rn(own_acc, __fmaf_rn(P.A[t0], nxx, P.C[t0]));
        const float loo = __fmaf_rn(P.R[t0], own_acc, __fmaf_rn(P.A1[t0], nxx, P.C1[t0]));
        const float dlt = __fadd_rn(loo, -plain);
        dsum = __fadd_rn(dsum, dlt);
        if (!all_lone) ex_own[(12 + v) * kTileRows] = mine ? dlt : 0.0f;
        if (with_new) {
          // the own dish enters the marginal with the customer removed: take its plain term out of this half's sum
          // (it sits at the dish's lowest table) and publish the leave-one-out term for the merge
          if (!masked && (unsigned)rrel < 32u) {
            float acc_rep = own_acc;
            if (!all_lone) acc_rep = (rrel & 16) ? pick16(u, rrel) : pra;
            const float trp = __fadd_rn(acc_rep, __fmaf_rn(P.A[rep], nxx, P.CW[rep]));   // the term exactly as lse_chunk formed it
            s = fmaxf(s - ex2f(trp - mx), 0.0f);
          }
          ex_own[(2 * v) * kTileRows] = mx;
          ex_own[(2 * v + 1) * kTileRows] = s;
          ex_own[(6 + v) * kTileRows] = mine ? __fadd_rn(loo, single ? P.W1[rep] : P.W[rep]) : kMasked;
        }
      }
      phase(1);
      // ---- the leave-one-out corrections: to the own table alone, or to every table serving an own dish ----
      if (all_lone) {
        // registers cannot be indexed: one predicated packed add per PAIR of tables, the partner element gets + 0.0f
        // (exact for every value a log-weight can take)
        const float corr = __fadd_rn(dsum, s_dlm[t0]);
        const int rp = mine ? (rel >> 1) : -1;
        const float2 c2 = (rel & 1) ? make_float2(0.0f, corr) : make_float2(corr, 0.0f);
#pragma unroll
        for (int p2 = 0; p2 < 16; ++p2) if (p2 == rp) lw2[p2] = fadd2(lw2[p2], c2);
      } else {
        rendezvous();                                 // #0: the corrections, known to the thread that holds the own table
        float dl[kMaxTcViews];
        uint32_t mk[kMaxTcViews];
#pragma unroll
        for (int v = 0; v < kMaxTcViews; ++v) {
          dl[v] = (v < V) ? (mine ? ex_own[(12 + v) * kTileRows] : ex_oth[(12 + v) * kTileRows]) : 0.0f;
          mk[v] = (v < V) ? (uint32_t)(s_same[v * 64 + t0] >> tb) : 0u;
        }
        const float dlm = s_dlm[t0];
        float* lw = reinterpret_cast<float*>(lw2);
#pragma unroll
        for (int q = 0; q < 32; ++q) {
          float cq = 0.0f;
#pragma unroll
          for (int v = 0; v < kMaxTcViews; ++v) if ((mk[v] >> q) & 1u) cq = __fadd_rn(cq, dl[v]);
          if (q == rel) cq = __fadd_rn(cq, dlm);
          lw[q] = __fadd_rn(lw[q], cq);
        }
      }
      float uf = 0.0f;
      if (hf == 0) {
        const U4 rnd = stream_block(c.seed, c.chain, kDomTable, 0, sweep, (uint64_t)(c.row_offset + rowc));
        uf = uniform_f32_from(rnd.x);
        ex_own[11 * kTileRows] = uf;
      }
      float hmax;
      {
        float M0 = kMasked, M1 = kMasked;
#pragma unroll
        for (int i = 0; i < 16; ++i) { M0 = fmaxf(M0, lw2[i].x); M1 = fmaxf(M1, lw2[i].y); }
        hmax = fmaxf(M0, M1);
      }
      ex_own[9 * kTileRows] = hmax;
      if (can_record) {                               // this half's best table other than the customer's own
        if (record) {
          float X0 = kMasked, X1 = kMasked;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            X0 = fmaxf(X0, (2 * i == rel) ? kMasked : lw2[i].x);
            X1 = fmaxf(X1, (2 * i + 1 == rel) ? kMasked : lw2[i].y);
          }
          ex_own[0] = fmaxf(X0, X1);                  // field 0 belongs to the new-table marginal, absent here
        }
      }
      // which tables of this half lie within 2^-31 of its best one (see the shortcut below)
      uint32_t nmask = 0u;
      {
        const float thr = __fadd_rn(hmax, -31.0f);
        const float* lw = reinterpret_cast<const float*>(lw2);
#pragma unroll
        for (int q = 0; q < 32; ++q) if (lw[q] > thr) nmask |= 1u << q;
      }
      ex_own[15 * kTileRows] = __uint_as_float(nmask);
      phase(2);
      rendezvous();                                   // #1: dish sums, own-dish terms, half maxima, the uniform
      phase(3);
      float second = kMasked;                         // best table other than the own one (read before the partner's next write)
      if (can_record && record && hf == 0) second = fmaxf(ex_own[0], ex_oth[0]);
      float lnew = single ? gp.LMN1 : gp.LMN0;
      for (int v = 0; with_new && v < V; ++v) {
        const float mo = ex_oth[(2 * v) * kTileRows], so = ex_oth[(2 * v + 1) * kTileRows];
        const float mi = ex_own[(2 * v) * kTileRows], si = ex_own[(2 * v + 1) * kTileRows];
        const float mA = hf ? mo : mi, sA = hf ? so : si, mB = hf ? mi : mo, sB = hf ? si : so;   // half A first in both threads
        const float ot = fmaxf(ex_own[(6 + v) * kTileRows], ex_oth[(6 + v) * kTileRows]);
        const float xx = (v == 0) ? xxv[0] : ((v == 1) ? xxv[1] : xxv[2]);
        const ViewParam vp = s_vp[v];
        const float termnew = __fmaf_rn(-vp.AN, xx, vp.CN) + ((single && (s_p[v].lone[t0] & 1)) ? vp.WN1 : vp.WN0);
        const float m2 = fmaxf(fmaxf(mA, mB), fmaxf(ot, termnew));
        const float ssum = ((sA * ex2f(mA - m2) + sB * ex2f(mB - m2)) + ex2f(ot - m2)) + ex2f(termnew - m2);
        lnew += (m2 + lg2f(ssum)) - (single ? vp.LD1 : vp.LD0);
      }
      if (hf == 1) uf = ex_oth[11 * kTileRows];
      const float hoth = ex_oth[9 * kTileRows];
      const float M = hf ? fmaxf(fmaxf(lnew, hoth), hmax) : fmaxf(fmaxf(lnew, hmax), hoth);
      int choice = t0;                                // nothing has weight: stay (cf. multiview_gibbs.cpp:172-176)
      const bool any_weight = (M > -1.0e29f);         // identical in both threads of the customer
      // Shortcut.  If ONE option dominates — every other TABLE is more than 31 below it in log2 and the new-table option more
      // than 27 — the draw below is that option for every uniform the stream can produce: the other weights sum to less than
      // 64 * 2^-31 + 2^-27 < 2^-24, so in FP32 every partial sum that contains the winner's weight (exactly 1) rounds to 1,
      // the grand total is exactly 1 and the target exactly u >= 2^-24; every cumulative sum before the winner is < 2^-24 <= u
      // and from the winner on it is 1 > u (u <= 1 - 2^-24).  So the inverse-CDF scan — and the CPU mirror, which always
      // runs it — returns the winner, and the exponentials, totals and the scan can be skipped.  (With a free table slot the
      // new-table option of a well-fitting customer sits ~2^-30 below its table: the asymmetric thresholds keep such rows
      // on the shortcut.)  Both threads of a customer decide from the same exchanged values (half maxima, near masks, lnew),
      // and a warp skips only when all its customers can, so the rendezvous counts of the two warps stay equal.
      const uint32_t nm_oth = __float_as_uint(ex_oth[15 * kTileRows]);
      const float near_thr = __fadd_rn(M, -31.0f);
      const int near_own = (hmax == M) ? __popc(nmask) : ((hmax > near_thr) ? 2 : 0);
      const int near_oth = (hoth == M) ? __popc(nm_oth) : ((hoth > near_thr) ? 2 : 0);
      const int near_new = (lnew == M) ? 1 : ((lnew > __fadd_rn(M, -27.0f)) ? 2 : 0);
      const bool sure = any_weight && (near_own + near_oth + near_new) == 1;
      const bool all_sure = __all_sync(0xffffffffu, sure);
      if (all_sure) {
        if (hf == 0) choice = (hmax == M) ? (__ffs(nmask) - 1) : ((hoth == M) ? (32 + __ffs(nm_oth) - 1) : kNewTable);
        rendezvous();                                 // the partner has read this tile's exchange fields before the next tile's are written
      } else {
      float Hown = 0.0f;
      if (any_weight) {                               // lw2 <- 2^(lw2 - M); this half's total (partial sums over t mod 4, fixed tree)
        const float2 nM2 = splat2(-M);
        float2 qa = splat2(0.0f), qb = splat2(0.0f);
#pragma unroll
        for (int i = 0; i < 16; i += 2) {
          lw2[i] = exp2w2<FAST>(fadd2(lw2[i], nM2));         qa = fadd2(qa, lw2[i]);
          lw2[i + 1] = exp2w2<FAST>(fadd2(lw2[i + 1], nM2)); qb = fadd2(qb, lw2[i + 1]);
        }
        Hown = __fadd_rn(__fadd_rn(qa.x, qa.y), __fadd_rn(qb.x, qb.y));
      }
      ex_own[10 * kTileRows] = Hown;
      phase(4);
      rendezvous();                                   // #2: half totals
      phase(5);
      const float Hoth = ex_oth[10 * kTileRows];
      const float HA = hf ? Hoth : Hown, HB = hf ? Hown : Hoth;
      const float total = __fadd_rn(__fadd_rn(HA, HB), exp2w<FAST>(__fadd_rn(lnew, -M)));
      const float target = __fmul_rn(uf, total);
      int cnt = 0, last = -1;
      if (any_weight) {                               // tables of this half whose cumulative weight is <= target
        float cum = hf ? HA : 0.0f;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          cum = __fadd_rn(cum, lw2[i].x);
          cnt += (target < cum) ? 0 : 1;
          cum = __fadd_rn(cum, lw2[i].y);
          cnt += (target < cum) ? 0 : 1;
        }
      }
      if (hf == 1) {
        int enc = cnt;
        if (cnt == 32) {                              // only needed when the draw ran past every table
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            if (lw2[i].x > 1.0e-30f) last = 2 * i;
            if (lw2[i].y > 1.0e-30f) last = 2 * i + 1;
          }
          enc |= (last + 1) << 8;
        }
        ex_own[11 * kTileRows] = __int_as_float(enc);
      }
      phase(6);
      rendezvous();                                   // #3: the upper half's count
      phase(7);
      if (hf == 0 && any_weight) {
        {
          const int enc = __float_as_int(ex_oth[11 * kTileRows]);
          const int total_cnt = cnt + (enc & 0xFF);
          choice = (total_cnt < 64) ? total_cnt : kNewTable;
          if (total_cnt >= 64 && !(lnew > -1.0e29f)) {   // rounding fall-through with no new-table mass: last live table
            const int lb = (enc >> 8) - 1;
            int la = -1;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              if (lw2[i].x > 1.0e-30f) la = 2 * i;
              if (lw2[i].y > 1.0e-30f) la = 2 * i + 1;
            }
            choice = (lb >= 0) ? (32 + lb) : ((la >= 0) ? la : t0);
          }
        }
      }
      }   // (full path)
      if (hf == 0) {
        if (c.blk_count > 1 && (int)((c.row_offset + rowc) % c.blk_count) != c.blk_index) choice = t0;   // not this pass's block
        if (can_record && record) {
          // The row's margin: its own table's lead over the best other, less this sweep's bound (drift since the reference,
          // evaluation error), rounded down.  Only where the draw is provably the own table (the shortcut's condition).
          float m = kMasked;
          if (sure && choice == t0) {
            const float* kq = reinterpret_cast<const float*>(s_misc + 6);
            m = __fsub_rd(__fsub_rd(M, second), screen_row_bound(kq, xxv, V));
          }
          if (live) c.margin[row] = m;
          // and the least margin of these 32 rows, for the tile test of later sweeps (a NaN margin counts as -inf)
          float mn = live ? ((m == m) ? m : -INFINITY) : INFINITY;
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
          if (lane == 0 && (row >> 5) < c.n_chunks) c.margin_min[row >> 5] = mn;
        }
        if (live) {
          c.choice[row] = choice;
          if (dbg_rows) { c.dbg_choice[row] = choice; c.dbg_lnew[row] = lnew; }
        }
        const unsigned births = __ballot_sync(0xffffffffu, live && choice == kNewTable);
        const unsigned moved = __ballot_sync(0xffffffffu, live && choice != t0);
        if (lane == 0 && (row >> 5) < c.n_chunks) { c.birthmask[row >> 5] = births; c.movedmask[row >> 5] = moved; }
      }
    }
    phase(8);
    if (prof && r == 0 && hf == 0) { prof_out[12 + 2 * pair] = w0 + w1; prof_out[13 + 2 * pair] = clock64() - t_start; }
    if (prof && r == 0 && blockIdx.x == 0 && pair == 0) {
      // phases: 0 prologue (base, A|x|^2), 1 views (incl. the accumulator waits, reported separately), 2 corrections + max,
      // 3 rendezvous 1, 4 marginals + weights, 5 rendezvous 2, 6 scan, 7 rendezvous 3, 8 write-out
      long long* po = c.dbg_prof + (230 + hf) * 16;
      for (int k = 0; k < 9; ++k) po[k] = ph[k];
      po[9] = w0;
    }
    };
    const bool with_new_rt = (gp.LMN0 > -1.0e29f) || (gp.LMN1 > -1.0e29f);
    if (with_new_rt) { if (all_lone_rt) epilogue(BoolC<true>(), BoolC<true>()); else epilogue(BoolC<true>(), BoolC<false>()); }
    else { if (all_lone_rt) epilogue(BoolC<false>(), BoolC<true>()); else epilogue(BoolC<false>(), BoolC<false>()); }
  }

  // ---- teardown ------------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols));
  }
  if (tid == 3 * 128) kclock_end(c.kclock + kClockDraw, gridDim.x);
}

// =================================================================================================
// host side
// =================================================================================================
bool draw_tc_supported(const Ctx& c) {
  if (c.cap != 64 || c.V < 1 || c.V > kMaxTcViews) return false;   // shared memory and TMEM are laid out for up to three views
  for (int v = 0; v < c.V; ++v)
    if (c.D[v] != 64 || (reinterpret_cast<uintptr_t>(c.x[v]) & 15) != 0) return false;
  return true;
}

size_t draw_tc_maps_bytes() { return sizeof(TcMaps); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static cudaError_t encode_2d(EncodeTiledFn fn, CUtensorMap* map, const void* base, uint64_t rows, uint32_t box_rows) {
  cuuint64_t dims[2] = {64, rows};
  cuuint64_t strides[1] = {64 * sizeof(float)};
  cuuint32_t box[2] = {kHalfCols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}

cudaError_t draw_tc_make_maps(const Ctx& c, void* maps_out) {
  void* fnp = nullptr;
  cudaDriverEntryPointQueryResult q;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fnp, cudaEnableDefault, &q);
  if (e != cudaSuccess) return e;
  if (!fnp || q != cudaDriverEntryPointSuccess) return cudaErrorNotSupported;
  EncodeTiledFn fn = reinterpret_cast<EncodeTiledFn>(fnp);
  TcMaps* m = static_cast<TcMaps*>(maps_out);
  for (int v = 0; v < c.V; ++v)
    if ((e = encode_2d(fn, &m->x[v], c.x[v], (uint64_t)c.n_rows, kTileRows)) != cudaSuccess) return e;
  for (int v = c.V; v < kMaxTcViews; ++v) m->x[v] = m->x[0];
  if ((e = encode_2d(fn, &m->mean_hi, c.mean_hi, (uint64_t)c.V * 64, 64)) != cudaSuccess) return e;
  if ((e = encode_2d(fn, &m->mean_lo, c.mean_lo, (uint64_t)c.V * 64, 64)) != cudaSuccess) return e;
  return cudaSuccess;
}

cudaError_t launch_draw_tc(const Ctx& c, const void* maps, bool fast, bool programmatic, cudaStream_t s) {
  if (c.n_rows <= 0) return cudaSuccess;
  if (!draw_tc_supported(c) || !maps) return cudaErrorInvalidValue;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int n_tiles = (c.n_rows + kTileRows - 1) / kTileRows;
  const int grid = n_tiles < sms ? n_tiles : sms;
  const bool dbg = c.debug_export != 0;
  auto kern = fast ? (dbg ? k_draw_tc<true, true> : k_draw_tc<true, false>) : (dbg ? k_draw_tc<false, true> : k_draw_tc<false, false>);
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SmemLayout::total);
  if (e != cudaSuccess) return e;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = SmemLayout::total;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // may start while its predecessor in the stream still runs;
  attr[0].val.programmaticStreamSerializationAllowed = 1;             // the kernel orders itself with griddepcontrol.wait
  cfg.attrs = attr;
  cfg.numAttrs = programmatic ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, c, *static_cast<const TcMaps*>(maps));
}

}  // namespace mv
