/* philox.h -- Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy
 * as 1, 2, 3", SC'11), the counter-based generator of the closed-loop
 * rollouts (DESIGN.md section 7).  Plain C so that host code, device code and
 * the CPU oracle of the tests compile the same definition; curand's Philox is
 * device-only.  Known answers (Random123 kat_vectors):
 *   counter 0, key 0             -> 6627e8d5 e169c58d bc57ac4c 9b00dbd8
 *   counter ~0, key ~0           -> 408f276d 41c83b0e a20bc7c6 6d5451fd
 *   counter 243f6a88 85a308d3 13198a2e 03707344, key a4093822 299f31d0
 *                                -> d16cfe09 94fdcceb 5001e420 24126ea1 */
#ifndef PP2D_PHILOX_H_
#define PP2D_PHILOX_H_
#include <stdint.h>

#ifdef __CUDACC__
#define PP2D_HD __host__ __device__ __forceinline__
#else
#define PP2D_HD static inline
#endif

/* c[0..3] <- Philox4x32-10(c, (k0, k1)) */
PP2D_HD void pp2d_philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; ++r) {
    if (r > 0) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    const uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
    const uint32_t c1 = c[1], c3 = c[3];
    c[0] = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    c[1] = (uint32_t)p1;
    c[2] = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c[3] = (uint32_t)p0;
  }
}

/* The uniform of a word: its top 24 bits times 2^-24, exact, in [0, 1). */
PP2D_HD float pp2d_uniform24(uint32_t w) { return (float)(w >> 8) * 0x1p-24f; }

/* The five uniforms of step t of episode e: r[0] picks the motion slot, r[1..4]
 * flip the sensors up, left, right, down.  Blocks (t, e_lo, e_hi, 0) and
 * (t, e_lo, e_hi, 1); the last three words of the second block are unused. */
PP2D_HD void pp2d_step_uniforms(uint64_t seed, uint64_t e, uint32_t t, float r[5]) {
  uint32_t a[4] = {t, (uint32_t)e, (uint32_t)(e >> 32), 0u};
  uint32_t b[4] = {t, (uint32_t)e, (uint32_t)(e >> 32), 1u};
  pp2d_philox4x32_10(a, (uint32_t)seed, (uint32_t)(seed >> 32));
  pp2d_philox4x32_10(b, (uint32_t)seed, (uint32_t)(seed >> 32));
  r[0] = pp2d_uniform24(a[0]);
  r[1] = pp2d_uniform24(a[1]);
  r[2] = pp2d_uniform24(a[2]);
  r[3] = pp2d_uniform24(a[3]);
  r[4] = pp2d_uniform24(b[0]);
}

#undef PP2D_HD
#endif /* PP2D_PHILOX_H_ */
