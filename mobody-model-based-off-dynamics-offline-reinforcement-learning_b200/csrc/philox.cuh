// Philox4x32-10 (Salmon et al., SC'11) for the production-mode draws.
// Replaces torch.normal (mobody_dynamics.py:220), np.random.choice (mobody_module.py:356)
// and np.random.randint (algo/utils.py:128) with counter-based draws keyed on the
// *global* row id so results do not depend on how rows are sharded over GPUs.
// Checked bit-for-bit against oracle/philox.py.  Only the low 32 bits of a seed key the generator ((uint32_t)seed):
// seeds that differ by a multiple of 2^32 give the same draws (pinned by tests/test_gpu_philox_draws.py).
#pragma once
#include <stdint.h>

#define MB_STREAM_NOISE 0x6E6F6973u
#define MB_STREAM_ELITE 0x656C6974u
#define MB_STREAM_INDEX 0x696E6478u

struct Philox4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                          uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c1 = (uint32_t)p1; c3 = (uint32_t)p0; c0 = n0; c2 = n2;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return Philox4{c0, c1, c2, c3};
}

__host__ __device__ __forceinline__ float philox_u01(uint32_t x) {
  return ((float)(x >> 9) + 0.5f) * 1.1920928955078125e-07f;   // (0,1), exact in fp32
}

// four N(0,1) from one block (Box-Muller on (x,y) and (z,w))
__device__ __forceinline__ void philox_normal4(const Philox4& b, float out[4]) {
  const float two_pi = 6.283185307179586f;
  float r0 = sqrtf(-2.0f * logf(philox_u01(b.x))), t0 = two_pi * philox_u01(b.y);
  float r1 = sqrtf(-2.0f * logf(philox_u01(b.z))), t1 = two_pi * philox_u01(b.w);
  float s, c;
  sincosf(t0, &s, &c); out[0] = r0 * c; out[1] = r0 * s;
  sincosf(t1, &s, &c); out[2] = r1 * c; out[3] = r1 * s;
}

// one N(0,1): word w (0..3) of the block, philox_normal4()[w] up to the error of the SFU sine / cosine.
// The radius takes the precise logf: lg2.approx.f32 has an ABSOLUTE error of about 2^-22 (PTX ISA), the size of ln u
// itself at the top word (x >> 9 = 2^23 - 1, u = 1 - 2^-24, ln u = -6e-8), where __logf gave r = 0 or NaN instead of
// 3.45e-4.  With logf (1 ulp) and a correctly rounded sqrtf, r is within 2^-23 r; sin/cos.approx.f32 are within 2^-20.5
// absolute on t in (0, 2 pi) (PTX ISA); the product adds 2^-24 |n|.  So for every word
//   |n - r cos t| <= 2^-20.5 r + 2^-22 |n|,   r = sqrt(-2 ln u) <= 5.77,
// and the tests hold the sample to 2e-6 (1 + |n| + r) of the numpy oracle's, which covers the oracle's own few ulps.
__device__ __forceinline__ float philox_normal1(const Philox4& b, int w) {
  const float two_pi = 6.283185307179586f;
  const uint32_t xa = (w & 2) ? b.z : b.x, xb = (w & 2) ? b.w : b.y;
  const float r = sqrtf(-2.0f * logf(philox_u01(xa))), t = two_pi * philox_u01(xb);
  return (w & 1) ? r * __sinf(t) : r * __cosf(t);
}

__device__ __forceinline__ Philox4 philox_noise_block(unsigned long long seed, unsigned int step,
                                                     unsigned long long row, unsigned int block) {
  return philox4x32_10((uint32_t)row, (uint32_t)(row >> 32), step, block, (uint32_t)seed, MB_STREAM_NOISE);
}
__device__ __forceinline__ int philox_elite_slot(unsigned long long seed, unsigned int step,
                                                 unsigned long long row, int n_elites) {
  Philox4 b = philox4x32_10((uint32_t)row, (uint32_t)(row >> 32), step, 0u, (uint32_t)seed, MB_STREAM_ELITE);
  return (int)(((uint64_t)b.x * (uint64_t)n_elites) >> 32);
}
