// mv_philox.h — Philox4x32-10 counter-based stream, one source for host and device.
//
// Replaces the reference's RNG surface: uniform01()/rnorm_scalar() over R::runif/R::rnorm
// (/root/reference/Multiview/multiview_utils.cpp:305-306, :261; multiview_gibbs.cpp:26,56) and the
// unused std::mt19937 header multiview_rng.h:9-24.  A draw is addressed, not sequenced:
//
//   key     = ( lo32(seed), hi32(seed) + chain )
//   counter = ( lo32(index), hi32(index), sweep, domain << 24 | slot )
//
// so any GPU thread and the host mirror obtain the same number for (sweep, row, slot) without
// sharing state, and results do not depend on how rows are sharded over GPUs.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define MV_HD __host__ __device__ __forceinline__
#else
#define MV_HD inline
#endif

namespace mv {

enum PhiloxDomain : uint32_t {
  kDomTable = 0,        // table draw of a row                      (multiview_gibbs.cpp:181)
  kDomDish = 1,         // dish draw for a new table, slot = view   (multiview_utils.cpp:261)
  kDomHyperNormal = 2,  // hyper-step proposal normals              (multiview_hyper.cpp:104,126,170)
  kDomHyperUnif = 3,    // hyper-step acceptance uniforms           (multiview_hyper.cpp:228,253,260,279,286)
  kDomInitTable = 4,    // random initial table                     (multiview_gibbs.cpp:26)
  kDomInitDish = 5,     // random initial dish, slot = view         (multiview_gibbs.cpp:56)
  kDomCallSeq = 6,      // call-ordered host stream (multiview_rng.h mirror)
  kDomCountBeta = 7     // beta step of count view `slot`: index 0 the proposal normal, 1 the acceptance uniform
                        // (sweep = the sweep index of the hyper step's tau draws)
};

struct U4 { uint32_t x, y, z, w; };

MV_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

MV_HD U4 philox4x32_10(U4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = mulhi32(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = mulhi32(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    U4 n;
    n.x = hi1 ^ c.y ^ k0;
    n.y = lo1;
    n.z = hi0 ^ c.w ^ k1;
    n.w = lo0;
    c = n;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}

MV_HD U4 stream_block(uint64_t seed, uint32_t chain, uint32_t domain, uint32_t slot, uint32_t sweep,
                      uint64_t index) {
  U4 c;
  c.x = (uint32_t)index;
  c.y = (uint32_t)(index >> 32);
  c.z = sweep;
  c.w = (domain << 24) | (slot & 0xFFFFFFu);
  return philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32) + chain);
}

// (k + 1/2) 2^-23 with k the top 23 bits: every step is exact in FP32, result in (0,1).
MV_HD float uniform_f32_from(uint32_t x0) {
  return ((float)(x0 >> 9) + 0.5f) * 1.1920928955078125e-07f;
}
// (k + 1/2) 2^-53 with k = 53 bits from two words; in (0,1).
MV_HD double uniform_f64_from(uint32_t a, uint32_t b) {
  const uint64_t k = ((uint64_t)(a >> 5) << 26) | (uint64_t)(b >> 6);
  return ((double)k + 0.5) * 1.1102230246251565e-16;
}

}  // namespace mv
