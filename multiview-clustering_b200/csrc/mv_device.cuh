// mv_device.cuh — shared device-side definitions of the allocation sweep:
//   * the per-sweep FP32 parameter block (table-major) the likelihood+draw kernels read,
//   * the bit-reproducible exp2 / log2 used by the draw,
//   * RowEpilogue<CAP>: leave-one-out table weights, log-sum-exp marginal of a new table and the
//     inverse-CDF draw for ONE customer held by ONE thread.
//
// Reference arithmetic being replaced (paths under /root/reference/Multiview):
//   compute_f_vk / compute_f_vk_new               multiview_utils.cpp:307-350
//   compute_marginal_likelihood_new_table          multiview_utils.cpp:40-69
//   compute_table_probs_with_cache                 multiview_utils.cpp:71-136
//   normalise + inverse-CDF draw                   multiview_gibbs.cpp:169-199
//   remove_customer (as a leave-one-out view)      multiview_utils.cpp:138-192
//
// Every FP32 operation of the epilogue is an explicit round-to-nearest intrinsic in a fixed
// order, so that oracle/mv_oracle.c:mvo_stageB_f32 (an independent plain-C restatement) produces
// the same integer draw bit for bit from the same dot products.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "mv_philox.h"

namespace mv {

constexpr int kMaxViews = 16;
constexpr float kMasked = -1.0e30f;   // log2-domain sentinel of a zero-weight option
constexpr int kNewTable = -1;

// ---- per-sweep parameter block (built by the finalize kernel, DESIGN.md §3) ----------------
struct __align__(16) TableParam {   // one per (view, table slot); 32 bytes, hot half first
  float A, C;        // log2 f = C + A*e,  e = 2 x.m - |x|^2      (dish statistics as they are)
  float W;           // log2 (l_vk - sigma_v)+ carried by the lowest table of each dish, else masked
  int32_t dish;      // dish slot of this table in this view, -1 = free table slot
  float A1, C1;      // A, C with the customer itself removed from the dish (n-1, S1-x)
  float W1;          // W with l_vk-1
  int32_t lone;      // 1 if that dish is served by exactly one table
};
struct __align__(16) ViewParam {    // one per view; 32 bytes
  float AN, CN;      // log2 f_new = CN - AN |x|^2
  float WN0, WN1;    // log2 (alpha_v + K_act sigma_v)+ ; WN1 with K_act-1
  float LD0, LD1;    // log2 (alpha_v + sum_k l_vk) ; LD1 with the sum reduced by one
  float pad0, pad1;
};
struct __align__(16) TableMass {    // one per table slot; 16 bytes
  float LM, LM1;     // log2 (n_t - sigma_g)+ ; LM1 with n_t-1
  int32_t single;    // n_t == 1
  int32_t pad;
};
struct __align__(16) GlobalParam {
  float LMN0, LMN1;  // log2 (alpha_g + sigma_g T_nonempty)+ ; LMN1 with T_nonempty-1; masked if no free slot
  int32_t nfree;     // free table slots at sweep start
  uint32_t sweep;    // index of the sweep these parameters are for
};

// ---- bit-reproducible transcendental pieces ---------------------------------------------
// 2^d for d <= 0 (clamped at -125): n = rint(d) via the 1.5*2^23 trick, 2^f by a degree-5
// polynomial on [-1/2,1/2] (rel. err 1.9e-7), exponent added in the integer domain.
__device__ __forceinline__ float exp2m(float d) {
  d = fmaxf(d, -125.0f);
  const float r = __fadd_rn(d, 12582912.0f);
  const float n = __fadd_rn(r, -12582912.0f);
  const float f = __fadd_rn(d, -n);
  float p = 0x1.5bba14p-10f;
  p = __fmaf_rn(p, f, 0x1.3cea88p-7f);
  p = __fmaf_rn(p, f, 0x1.c6b752p-5f);
  p = __fmaf_rn(p, f, 0x1.ebf9bcp-3f);
  p = __fmaf_rn(p, f, 0x1.62e42ap-1f);
  p = __fmaf_rn(p, f, 1.0f);
  return __uint_as_float(__float_as_uint(p) + (__float_as_uint(r) << 23));
}

// log2(s) for a normal s > 0: atanh series in t = (m-1)/(m+1), m in [sqrt(1/2), sqrt(2)).  The
// quotient is a fixed sequence of fused multiply-adds (linear seed on [1.707, 2.414], three Newton
// steps, one residual correction): no division subroutine, and the CPU mirror repeats it exactly.
__device__ __forceinline__ float log2m(float s) {
  const uint32_t b = __float_as_uint(s);
  int32_t e = (int32_t)(b >> 23) - 127;
  float m = __uint_as_float((b & 0x007FFFFFu) | 0x3F800000u);
  if (m > 1.41421354f) { m = __fmul_rn(m, 0.5f); e += 1; }
  const float num = __fadd_rn(m, -1.0f), den = __fadd_rn(m, 1.0f);
  float y = __fmaf_rn(-0.24264069f, den, 0.99258476f);
  y = __fmaf_rn(y, __fmaf_rn(-den, y, 1.0f), y);
  y = __fmaf_rn(y, __fmaf_rn(-den, y, 1.0f), y);
  y = __fmaf_rn(y, __fmaf_rn(-den, y, 1.0f), y);
  float t = __fmul_rn(num, y);
  t = __fmaf_rn(__fmaf_rn(-t, den, num), y, t);
  const float t2 = __fmul_rn(t, t);
  float q = 0x1.c71c72p-4f;
  q = __fmaf_rn(q, t2, 0x1.24924ap-3f);
  q = __fmaf_rn(q, t2, 0x1.99999ap-3f);
  q = __fmaf_rn(q, t2, 0x1.555556p-2f);
  q = __fmaf_rn(q, t2, 1.0f);
  const float r = __fmul_rn(__fmul_rn(t, q), 0x1.715476p+1f);
  return __fadd_rn((float)e, r);
}

// ---- Dirichlet-multinomial count views (MVG_COUNT_DIRMULT): lnΓ(a + x) - lnΓ(a), FP64 --------------
// a > 0, x >= 0 an integer.  Up to kLgdLoop the sum of log(a + j), j < x; above it a is first shifted to >= kLgdLoop by at
// most kLgdLoop such terms, then the Stirling difference
//   lnΓ(b) - lnΓ(a) = (a - 1/2) log1p(x / a) + x (log b - 1) + R(b) - R(a),   b = a + x,
//   R(z) = 1/(12 z) - 1/(360 z^3) + 1/(1260 z^5) - 1/(1680 z^7)   (truncation < 1.3e-14 at z >= 16),
// whose two main terms are both positive: no cancellation between large lnΓ values, and at most ~2 kLgdLoop logs per
// call whatever x is (a long row's births and denominators do not become per-token loops).
constexpr int kLgdLoop = 16;
__device__ __forceinline__ double stirling_tail(double z) {
  const double r = 1.0 / z, r2 = r * r;
  return r * (1.0 / 12.0 - r2 * (1.0 / 360.0 - r2 * (1.0 / 1260.0 - r2 * (1.0 / 1680.0))));
}
static __device__ __noinline__ double lgamma_diff(double a, int x) {
  double s = 0.0;
  if (x <= kLgdLoop) {
    for (int j = 0; j < x; ++j) s += log(a + (double)j);
    return s;
  }
  while (a < (double)kLgdLoop) { s += log(a); a += 1.0; x -= 1; }
  const double xd = (double)x, b = a + xd;
  return s + (a - 0.5) * log1p(xd / a) + xd * (log(b) - 1.0) + (stirling_tail(b) - stirling_tail(a));
}

// ---- packed FP32 (sm_100 FFMA2 / FADD2): two IEEE-rounded operations per instruction ------------
// Each half is rounded exactly like the scalar fmaf / add, so packing changes the instruction count,
// not a single bit of the result (the CPU mirror stays scalar).
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d)
      : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)),
        "l"(*reinterpret_cast<unsigned long long*>(&c)));
  return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
  unsigned long long d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d)
      : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)));
  return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 splat2(float x) { return make_float2(x, x); }

// 2^d for the weights, two at a time.  EXACT: the polynomial of exp2m (the CPU mirror reproduces it
// bit for bit).  FAST: MUFU.EX2 (ex2.approx.ftz, <= 2 ulp) — the weights are then tolerance-level and
// only the scan that turns them into a table index is mirrored exactly (DESIGN.md §5).
template <bool FAST>
__device__ __forceinline__ float exp2w(float d) {
  if (FAST) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d));
    return r;
  } else {
    return exp2m(d);
  }
}
template <bool FAST>
__device__ __forceinline__ float2 exp2w2(float2 d) {
  if (FAST) {
    return make_float2(exp2w<true>(d.x), exp2w<true>(d.y));
  } else {
    d.x = fmaxf(d.x, -125.0f);
    d.y = fmaxf(d.y, -125.0f);
    const float2 r = fadd2(d, splat2(12582912.0f));
    const float2 n = fadd2(r, splat2(-12582912.0f));
    const float2 f = ffma2(n, splat2(-1.0f), d);                 // d - n, one rounding of the exact difference
    float2 p = splat2(0x1.5bba14p-10f);
    p = ffma2(p, f, splat2(0x1.3cea88p-7f));
    p = ffma2(p, f, splat2(0x1.c6b752p-5f));
    p = ffma2(p, f, splat2(0x1.ebf9bcp-3f));
    p = ffma2(p, f, splat2(0x1.62e42ap-1f));
    p = ffma2(p, f, splat2(1.0f));
    return make_float2(__uint_as_float(__float_as_uint(p.x) + (__float_as_uint(r.x) << 23)),
                       __uint_as_float(__float_as_uint(p.y) + (__float_as_uint(r.y) << 23)));
  }
}

// ---- shared-memory staging of the parameter block for the epilogue ----------------------------------
// Hot part, per PAIR of tables (2t, 2t+1) so that packed arithmetic reads its operands as 64-bit halves
// of two 128-bit loads; cold part per table, read once per customer and view at its own table.
struct __align__(16) PairHot {
  float A0, A1, C0, C1;
  float W0, W1;
  int32_t dish0, dish1;
};
struct __align__(16) TableCold {
  float A1, C1, W1;
  int32_t lone;
};
// Cooperative copy of one view's TableParam[cap] from global memory into the two shared arrays.
__device__ __forceinline__ void stage_view_params(const TableParam* __restrict__ g, int cap, PairHot* hot,
                                                  TableCold* cold, int tid, int nthreads) {
  for (int t = tid; t < cap; t += nthreads) {
    const TableParam q = g[t];
    PairHot& h = hot[t >> 1];
    if (t & 1) { h.A1 = q.A; h.C1 = q.C; h.W1 = q.W; h.dish1 = q.dish; }
    else { h.A0 = q.A; h.C0 = q.C; h.W0 = q.W; h.dish0 = q.dish; }
    TableCold cq;
    cq.A1 = q.A1; cq.C1 = q.C1; cq.W1 = q.W1; cq.lone = q.lone;
    cold[t] = cq;
  }
}

// ---- one customer's epilogue ---------------------------------------------------------------
// The cap table slots of a customer are handled as two HALVES of cap/2 tables.  In the tensor-core
// kernel two threads (one per half) share a customer and trade a few scalars through shared memory;
// in the CUDA-core kernel one thread runs both halves back to back.  Either way the arithmetic is the
// sequence below, restated by oracle/mv_oracle.c:mvo_stageB_f32:
//   begin        lw[t] = log2 mass of table t (customer removed)
//   per view     view_begin, view_chunk x (cap/2)/16: L[t] = log2 f under table t's dish (leave-one-out
//                for the customer's own dish), lw[t] += L[t], streaming log-sum-exp (running max mx,
//                sum s) over this half's dishes;  merge_view: the two halves' (mx, s) and the new-dish
//                term -> log2 marginal of a new table, added to lnew
//   draw         M = max over both halves and lnew; weights(M) -> half totals HA, HB;
//                total = (HA + HB) + 2^(lnew - M); target = u * total; scan: half A counts its
//                cumulative weights <= target starting from 0, half B starting from HA;
//                choice = count (cap = new table)
constexpr int kEpiChunk = 16;

template <int HALF, bool FAST = false>
struct HalfEpilogue {
  static_assert(HALF % kEpiChunk == 0, "half of the table capacity must be a multiple of the epilogue chunk");
  float2 lw2[HALF / 2];  // running log2 weight of tables tbase + (2i, 2i+1); after weights(): the weights
  int t0;                // current table of the customer (absolute slot)
  int single;            // the customer sits alone at t0
  int any_single;        // some customer of this warp does (warp-uniform slow path)
  // per-view state
  float mx, s, nxx, A1r, C1r;
  int k0, lone0;
  uint32_t samemask;     // USE_MASK engines: bit j = table tbase + j serves the customer's own dish (set by the caller)

  // tm: all cap table masses, lm: the same LM values as a plain float array (vector loads); this
  // object covers tables [tbase, tbase + HALF).
  __device__ __forceinline__ void begin(const TableMass* __restrict__ tm, const float* __restrict__ lm, int t0_, int tbase) {
    t0 = t0_;
    const TableMass own = tm[t0_];
    single = own.single;
    any_single = __any_sync(0xffffffffu, single);
    const int rel = t0_ - tbase;
    const float4* lm4 = reinterpret_cast<const float4*>(lm + tbase);
#pragma unroll
    for (int i = 0; i < HALF / 4; ++i) {              // the customer's own table (if in this half) counts n_t - 1
      const float4 q = lm4[i];
      lw2[2 * i] = make_float2((rel == 4 * i) ? own.LM1 : q.x, (rel == 4 * i + 1) ? own.LM1 : q.y);
      lw2[2 * i + 1] = make_float2((rel == 4 * i + 2) ? own.LM1 : q.z, (rel == 4 * i + 3) ? own.LM1 : q.w);
    }
  }

  // hot/cold: the FULL per-view arrays (the customer's own table may lie in the other half).
  __device__ __forceinline__ void view_begin(const PairHot* __restrict__ hot, const TableCold* __restrict__ cold, float xx) {
    const TableCold own = cold[t0];
    k0 = reinterpret_cast<const int32_t*>(&hot[t0 >> 1].dish0)[t0 & 1];
    lone0 = own.lone; A1r = own.A1; C1r = own.C1;
    nxx = -xx;
    mx = kMasked;
    s = 0.0f;
  }

  // hoth/coldh: the arrays offset to this half's first table.  acc[j] = x . m_{tbase + BASE + j} (consumed).
  // WITH_NEW = false: no table slot is free, so a new table has no weight (capacity rule) and the
  // per-view marginal over the dishes — the whole log-sum-exp — is not needed; only lw is updated.
  // USE_MASK: the same-dish test comes from `samemask` (one bit per table, precomputed per (view, own table) by the
  // finalize kernel) instead of a compare against the loaded dish of every table: same values, fewer instructions.
  template <int BASE, bool SINGLE, bool WITH_NEW, bool USE_MASK>
  __device__ __forceinline__ void chunk_impl(const PairHot* __restrict__ hoth, const TableCold* __restrict__ coldh,
                                             float (&acc)[kEpiChunk]) {
    float2 term[kEpiChunk / 2];
    float c0 = kMasked, c1 = kMasked;
    const float2 two = splat2(2.0f), nxx2 = splat2(nxx);
#pragma unroll
    for (int p = 0; p < kEpiChunk / 2; ++p) {
      const float4 qa = reinterpret_cast<const float4*>(&hoth[BASE / 2 + p])[0];   // A0 A1 C0 C1
      float4 qb = make_float4(0.f, 0.f, 0.f, 0.f);
      if (WITH_NEW || !USE_MASK) qb = reinterpret_cast<const float4*>(&hoth[BASE / 2 + p])[1];   // W0 W1 dish0 dish1
      const float2 e = ffma2(two, make_float2(acc[2 * p], acc[2 * p + 1]), nxx2);
      const float2 Lg = ffma2(make_float2(qa.x, qa.y), e, make_float2(qa.z, qa.w));
      const bool same0 = USE_MASK ? ((samemask >> (BASE + 2 * p)) & 1u) != 0u : (__float_as_int(qb.z) == k0);
      const bool same1 = USE_MASK ? ((samemask >> (BASE + 2 * p + 1)) & 1u) != 0u : (__float_as_int(qb.w) == k0);
      float2 L = Lg;                                   // leave-one-out only where the dish is the customer's own
      if (same0) L.x = __fmaf_rn(A1r, e.x, C1r);
      if (same1) L.y = __fmaf_rn(A1r, e.y, C1r);
      lw2[BASE / 2 + p] = fadd2(lw2[BASE / 2 + p], L);
      if (!WITH_NEW) continue;
      float2 w = make_float2(qb.x, qb.y);
      if (SINGLE) {
        if (same0 && single) w.x = coldh[BASE + 2 * p].W1;
        if (same1 && single) w.y = coldh[BASE + 2 * p + 1].W1;
      }
      term[p] = fadd2(L, w);
      c0 = fmaxf(c0, term[p].x);
      c1 = fmaxf(c1, term[p].y);
      if ((p & 3) == 3) asm volatile("" ::: "memory");   // keep at most 8 parameter loads in flight (registers)
    }
    if (!WITH_NEW) return;
    const float mn = fmaxf(mx, fmaxf(c0, c1));
    s = __fmul_rn(s, exp2w<FAST>(__fadd_rn(mx, -mn)));
    mx = mn;
    const float2 nmn2 = splat2(-mn);
    float2 pa = splat2(0.0f), pb = splat2(0.0f);        // partial sums over j mod 4 = (0,1) and (2,3)
#pragma unroll
    for (int p = 0; p < kEpiChunk / 2; p += 2) {
      pa = fadd2(pa, exp2w2<FAST>(fadd2(term[p], nmn2)));
      pb = fadd2(pb, exp2w2<FAST>(fadd2(term[p + 1], nmn2)));
    }
    s = __fadd_rn(s, __fadd_rn(__fadd_rn(pa.x, pa.y), __fadd_rn(pb.x, pb.y)));
  }

  template <int BASE, bool WITH_NEW = true, bool USE_MASK = false>
  __device__ __forceinline__ void view_chunk(const PairHot* __restrict__ hoth, const TableCold* __restrict__ coldh,
                                             float (&acc)[kEpiChunk]) {
    if (!WITH_NEW) chunk_impl<BASE, false, false, USE_MASK>(hoth, coldh, acc);
    else if (any_single) chunk_impl<BASE, true, true, USE_MASK>(hoth, coldh, acc);
    else chunk_impl<BASE, false, true, USE_MASK>(hoth, coldh, acc);
  }

  // All chunks of this half from an array of HALF dot products (CUDA-core engine).
  template <int BASE>
  __device__ __forceinline__ void view_chunks_from(const PairHot* __restrict__ hoth, const TableCold* __restrict__ coldh,
                                                   const float* acc) {
    if constexpr (BASE < HALF) {
      float ch[kEpiChunk];
#pragma unroll
      for (int j = 0; j < kEpiChunk; ++j) ch[j] = acc[BASE + j];
      view_chunk<BASE>(hoth, coldh, ch);
      view_chunks_from<BASE + kEpiChunk>(hoth, coldh, acc);
    }
  }

  __device__ __forceinline__ float halfmax() const {
    float M0 = kMasked, M1 = kMasked;
#pragma unroll
    for (int i = 0; i < HALF / 2; ++i) { M0 = fmaxf(M0, lw2[i].x); M1 = fmaxf(M1, lw2[i].y); }
    return fmaxf(M0, M1);
  }

  // lw2 <- 2^(lw2 - M); returns this half's total (partial sums over t mod 4, then a fixed tree).
  __device__ __forceinline__ float weights(float M) {
    const float2 nM2 = splat2(-M);
    float2 qa = splat2(0.0f), qb = splat2(0.0f);
#pragma unroll
    for (int i = 0; i < HALF / 2; i += 2) {
      lw2[i] = exp2w2<FAST>(fadd2(lw2[i], nM2));         qa = fadd2(qa, lw2[i]);
      lw2[i + 1] = exp2w2<FAST>(fadd2(lw2[i + 1], nM2)); qb = fadd2(qb, lw2[i + 1]);
    }
    return __fadd_rn(__fadd_rn(qa.x, qa.y), __fadd_rn(qb.x, qb.y));
  }

  // Number of this half's tables whose cumulative weight (starting from cum0) is <= target.
  __device__ __forceinline__ int scan(float target, float cum0) const {
    float cum = cum0;
    int cnt = 0;
#pragma unroll
    for (int i = 0; i < HALF / 2; ++i) {
      cum = __fadd_rn(cum, lw2[i].x);
      cnt += (target < cum) ? 0 : 1;
      cum = __fadd_rn(cum, lw2[i].y);
      cnt += (target < cum) ? 0 : 1;
    }
    return cnt;
  }

  // Highest table of this half (relative index) that still has weight, or -1.
  __device__ __forceinline__ int last_live() const {
    int last = -1;
#pragma unroll
    for (int i = 0; i < HALF / 2; ++i) {
      if (lw2[i].x > 1.0e-30f) last = 2 * i;
      if (lw2[i].y > 1.0e-30f) last = 2 * i + 1;
    }
    return last;
  }
};

// log2 marginal of a new table in one view from the two halves' streaming sums (half A first).
template <bool FAST>
__device__ __forceinline__ float merge_view(float mxA, float sA, float mxB, float sB, const ViewParam& vp, float xx,
                                            int single, int lone0) {
  float mn = fmaxf(mxA, mxB);
  float s = __fadd_rn(__fmul_rn(sA, exp2w<FAST>(__fadd_rn(mxA, -mn))), __fmul_rn(sB, exp2w<FAST>(__fadd_rn(mxB, -mn))));
  const float Lnew = __fmaf_rn(-vp.AN, xx, vp.CN);
  const float termnew = __fadd_rn(Lnew, (single && lone0) ? vp.WN1 : vp.WN0);
  const float m2 = fmaxf(mn, termnew);
  s = __fmul_rn(s, exp2w<FAST>(__fadd_rn(mn, -m2)));
  s = __fadd_rn(s, exp2w<FAST>(__fadd_rn(termnew, -m2)));
  return __fadd_rn(__fadd_rn(m2, log2m(s)), -(single ? vp.LD1 : vp.LD0));
}

// The whole draw of one customer by ONE thread (CUDA-core engine): both halves back to back.
template <int CAP, bool FAST = false>
struct RowEpilogue {
  static constexpr int HALF = CAP / 2;
  HalfEpilogue<HALF, FAST> ha, hb;
  float lnew;

  __device__ __forceinline__ void begin(const TableMass* __restrict__ tm, const float* __restrict__ lm,
                                        const GlobalParam& g, int t0) {
    ha.begin(tm, lm, t0, 0);
    hb.begin(tm, lm, t0, HALF);
    lnew = ha.single ? g.LMN1 : g.LMN0;
  }
  __device__ __forceinline__ void view(const PairHot* __restrict__ hot, const TableCold* __restrict__ cold,
                                       const ViewParam& vp, const float (&acc)[CAP], float xx) {
    ha.view_begin(hot, cold, xx);
    ha.template view_chunks_from<0>(hot, cold, acc);
    hb.view_begin(hot, cold, xx);
    hb.template view_chunks_from<0>(hot + HALF / 2, cold + HALF, acc + HALF);
    lnew = __fadd_rn(lnew, merge_view<FAST>(ha.mx, ha.s, hb.mx, hb.s, vp, xx, ha.single, ha.lone0));
  }
  // A COUNT view (mv_counts.cu): acc[t] is already log2 f under table t's dish (the parameter block carries
  // A = 1/2, C = 0, so that C + A (2 acc - 0) = acc exactly), acc_loo the leave-one-out value under the customer's
  // own dish, rowtot = |x| enters only the new-dish term log2 f_new = -|x| log2 W (AN = log2 W, CN = 0).
  __device__ __forceinline__ void view_counts(const PairHot* __restrict__ hot, const TableCold* __restrict__ cold,
                                              const ViewParam& vp, const float (&acc)[CAP], float acc_loo, float rowtot) {
    ha.view_begin(hot, cold, 0.0f);
    ha.A1r = 0.0f; ha.C1r = acc_loo;
    ha.template view_chunks_from<0>(hot, cold, acc);
    hb.view_begin(hot, cold, 0.0f);
    hb.A1r = 0.0f; hb.C1r = acc_loo;
    hb.template view_chunks_from<0>(hot + HALF / 2, cold + HALF, acc + HALF);
    lnew = __fadd_rn(lnew, merge_view<FAST>(ha.mx, ha.s, hb.mx, hb.s, vp, rowtot, ha.single, ha.lone0));
  }
  // uf in (0,1). Returns the table slot or kNewTable.
  __device__ __forceinline__ int finish(float uf) {
    const float M = fmaxf(fmaxf(lnew, ha.halfmax()), hb.halfmax());
    if (!(M > -1.0e29f)) return ha.t0;   // nothing has weight: stay (cf. multiview_gibbs.cpp:172-176)
    const float HA = ha.weights(M), HB = hb.weights(M);
    const float total = __fadd_rn(__fadd_rn(HA, HB), exp2w<FAST>(__fadd_rn(lnew, -M)));
    const float target = __fmul_rn(uf, total);
    const int cnt = ha.scan(target, 0.0f) + hb.scan(target, HA);
    int choice = (cnt < CAP) ? cnt : kNewTable;
    if (cnt >= CAP && !(lnew > -1.0e29f)) {   // rounding fall-through with no new-table mass: last live table
      const int lb = hb.last_live(), la = ha.last_live();
      choice = (lb >= 0) ? (HALF + lb) : ((la >= 0) ? la : ha.t0);
    }
    return choice;
  }
};

// The same draw for CAP = 128 / 256 (CUDA-core engine).  There, CAP running log-weights per thread do not fit in registers,
// so they live in shared memory — float2 pairs (2i, 2i+1) at lw[i * NT], one column per thread of an NT-thread block — and
// the caller hands over the dot products 16 tables at a time, in ascending table order, instead of all CAP at once.  The
// arithmetic is RowEpilogue's operation for operation (oracle/mv_oracle.c:mvo_stageB_f32_mixed restates it for any cap):
// per view each half streams its log-sum-exp over ascending chunks, the halves merge half A first, and the draw takes
// the per-half totals (partial sums over t mod 4, fixed tree) and scans half B from HA.
template <int CAP, int NT>
struct WideRowEpilogue {
  static constexpr int HALF = CAP / 2;
  static_assert(HALF % kEpiChunk == 0, "half of the table capacity must be a multiple of the epilogue chunk");
  float2* lw;            // this thread's column of the block's [CAP/2][NT] array
  int t0, single;
  float lnew;
  // per view
  float mx, s, mxA, sA, nxx, A1r, C1r;
  int k0, lone0;

  __device__ __forceinline__ float2& at(int i) const { return lw[i * NT]; }

  __device__ __forceinline__ void begin(float2* lw_col, const TableMass* __restrict__ tm, const float* __restrict__ lm,
                                        const GlobalParam& g, int t0_) {
    lw = lw_col;
    t0 = t0_;
    const TableMass own = tm[t0_];
    single = own.single;
    lnew = single ? g.LMN1 : g.LMN0;
    for (int i = 0; i < CAP / 2; ++i)             // the customer's own table counts n_t - 1
      at(i) = make_float2((2 * i == t0_) ? own.LM1 : lm[2 * i], (2 * i + 1 == t0_) ? own.LM1 : lm[2 * i + 1]);
  }

  // A dense view: A1r / C1r from the own table; a count view overrides them after this call (see RowEpilogue::view_counts).
  __device__ __forceinline__ void view_begin(const PairHot* __restrict__ hot, const TableCold* __restrict__ cold, float xx) {
    const TableCold own = cold[t0];
    k0 = reinterpret_cast<const int32_t*>(&hot[t0 >> 1].dish0)[t0 & 1];
    lone0 = own.lone; A1r = own.A1; C1r = own.C1;
    nxx = -xx;
    mx = kMasked;
    s = 0.0f;
  }

  // Tables base .. base+15 (base a multiple of 16, called in ascending order): acc[j] = x . m_{base + j}.
  __device__ __forceinline__ void chunk(const PairHot* __restrict__ hot, const TableCold* __restrict__ cold, int base,
                                        const float (&acc)[kEpiChunk]) {
    if (base == HALF) { mxA = mx; sA = s; mx = kMasked; s = 0.0f; }   // half A is complete
    float2 term[kEpiChunk / 2];
    float c0 = kMasked, c1 = kMasked;
    const float2 two = splat2(2.0f), nxx2 = splat2(nxx);
#pragma unroll
    for (int p = 0; p < kEpiChunk / 2; ++p) {
      const int i = base / 2 + p;
      const float4 qa = reinterpret_cast<const float4*>(&hot[i])[0];   // A0 A1 C0 C1
      const float4 qb = reinterpret_cast<const float4*>(&hot[i])[1];   // W0 W1 dish0 dish1
      const float2 e = ffma2(two, make_float2(acc[2 * p], acc[2 * p + 1]), nxx2);
      float2 L = ffma2(make_float2(qa.x, qa.y), e, make_float2(qa.z, qa.w));
      const bool same0 = __float_as_int(qb.z) == k0, same1 = __float_as_int(qb.w) == k0;
      if (same0) L.x = __fmaf_rn(A1r, e.x, C1r);     // leave-one-out only where the dish is the customer's own
      if (same1) L.y = __fmaf_rn(A1r, e.y, C1r);
      at(i) = fadd2(at(i), L);
      float2 w = make_float2(qb.x, qb.y);
      if (same0 && single) w.x = cold[2 * i].W1;
      if (same1 && single) w.y = cold[2 * i + 1].W1;
      term[p] = fadd2(L, w);
      c0 = fmaxf(c0, term[p].x);
      c1 = fmaxf(c1, term[p].y);
    }
    const float mn = fmaxf(mx, fmaxf(c0, c1));
    s = __fmul_rn(s, exp2m(__fadd_rn(mx, -mn)));
    mx = mn;
    const float2 nmn2 = splat2(-mn);
    float2 pa = splat2(0.0f), pb = splat2(0.0f);        // partial sums over j mod 4 = (0,1) and (2,3)
#pragma unroll
    for (int p = 0; p < kEpiChunk / 2; p += 2) {
      pa = fadd2(pa, exp2w2<false>(fadd2(term[p], nmn2)));
      pb = fadd2(pb, exp2w2<false>(fadd2(term[p + 1], nmn2)));
    }
    s = __fadd_rn(s, __fadd_rn(__fadd_rn(pa.x, pa.y), __fadd_rn(pb.x, pb.y)));
  }

  // After the last chunk of a view; xx = |x|^2 (dense) or the row's token total (count view).
  __device__ __forceinline__ void view_end(const ViewParam& vp, float xx) {
    lnew = __fadd_rn(lnew, merge_view<false>(mxA, sA, mx, s, vp, xx, single, lone0));
  }

  // lw <- 2^(lw - M) over half h; returns the half's total (partial sums over t mod 4, then a fixed tree).
  __device__ __forceinline__ float weights(int h, float M) {
    const float2 nM2 = splat2(-M);
    float2 qa = splat2(0.0f), qb = splat2(0.0f);
    for (int i = h * HALF / 2; i < (h + 1) * HALF / 2; i += 2) {
      const float2 wa = exp2w2<false>(fadd2(at(i), nM2)), wb = exp2w2<false>(fadd2(at(i + 1), nM2));
      at(i) = wa;     qa = fadd2(qa, wa);
      at(i + 1) = wb; qb = fadd2(qb, wb);
    }
    return __fadd_rn(__fadd_rn(qa.x, qa.y), __fadd_rn(qb.x, qb.y));
  }

  __device__ __forceinline__ int finish(float uf) {
    float M0 = lnew, M1 = kMasked;
    for (int i = 0; i < CAP / 2; ++i) { const float2 q = at(i); M0 = fmaxf(M0, q.x); M1 = fmaxf(M1, q.y); }
    const float M = fmaxf(M0, M1);
    if (!(M > -1.0e29f)) return t0;     // nothing has weight: stay (cf. multiview_gibbs.cpp:172-176)
    const float HA = weights(0, M), HB = weights(1, M);
    const float total = __fadd_rn(__fadd_rn(HA, HB), exp2m(__fadd_rn(lnew, -M)));
    const float target = __fmul_rn(uf, total);
    int cnt = 0;
    for (int h = 0; h < 2; ++h) {
      float cum = h ? HA : 0.0f;
      for (int i = h * HALF / 2; i < (h + 1) * HALF / 2; ++i) {
        const float2 q = at(i);
        cum = __fadd_rn(cum, q.x);
        cnt += (target < cum) ? 0 : 1;
        cum = __fadd_rn(cum, q.y);
        cnt += (target < cum) ? 0 : 1;
      }
    }
    if (cnt < CAP) return cnt;
    if (lnew > -1.0e29f) return kNewTable;
    int last = t0;                      // rounding fall-through with no new-table mass: last live table
    for (int i = 0; i < CAP / 2; ++i) {
      const float2 q = at(i);
      if (q.x > 1.0e-30f) last = 2 * i;
      if (q.y > 1.0e-30f) last = 2 * i + 1;
    }
    return last;
  }
};

}  // namespace mv
