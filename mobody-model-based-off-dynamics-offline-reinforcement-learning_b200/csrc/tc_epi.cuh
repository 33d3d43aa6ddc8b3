// Epilogue helpers shared by the tensor-core rollout kernels (step_tc.cu: one CTA per 128-row tile;
// step_pair.cu: CTA pair, two interleaved tiles): activation math on accumulator columns, bf16 hi/lo
// operand stores in the UMMA K-major layout, TMEM loads, the epilogue-only named barrier.
#pragma once
#include "tc_prims.cuh"

namespace tce {

template <int W> __device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, %0;" ::"n"(32 * W) : "memory"); }   // epilogue warps only

template <int NS>
__device__ __forceinline__ void store8(unsigned char* base, uint32_t plane_stride, uint32_t off, const float (&v)[8]) {
  if (NS == 2) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) tc::split2(v[2 * i], v[2 * i + 1], h[i], l[i]);
    *reinterpret_cast<uint4*>(base + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(base + plane_stride + off) = make_uint4(l[0], l[1], l[2], l[3]);
  } else {
    *reinterpret_cast<uint4*>(base + off) = make_uint4(tc::pack_bf16(v[0], v[1]), tc::pack_bf16(v[2], v[3]),
                                                       tc::pack_bf16(v[4], v[5]), tc::pack_bf16(v[6], v[7]));
  }
}

// argument is the PRE-SCALED pre-activation (see tc_swish_scales); result carries the mode's output scale
template <int NS> __device__ __forceinline__ float swish_ns(float t) { return NS == 1 ? tc::swish_pre_tanh(t) : tc::swish_pre_ex2_rcp(t); }

// v[i] = act(x[i] + b[i]) for 8 accumulator columns.  Swish layers arrive pre-scaled (tc_swish_scales); the SFU ops
// are volatile so they stay batched: 8 independent MUFUs in flight per warp, then the dependent ones.
template <int NS>
__device__ __forceinline__ void act8(const uint32_t* x, const float* b, float (&v)[8], bool relu) {
  float t[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) t[i] = __uint_as_float(x[i]) + b[i];
  if (relu) {
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = fmaxf(t[i], 0.f);
  } else if (NS == 1) {
    float th[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) asm volatile("tanh.approx.f32 %0, %1;" : "=f"(th[i]) : "f"(t[i]));
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = fmaf(t[i], th[i], t[i]);
  } else {
    float e[8];
    // One reciprocal serves a pair: 1/a_0 = a_1 * (1 / (a_0 a_1)), 1/a_1 = a_0 * (1 / (a_0 a_1)), a = 1 + 2^t >= 1 (measured
    // against one reciprocal per element and one per quad: the pair is fastest).  The exponent argument is clamped so the
    // product stays finite (2^60 per factor): beyond the clamp swish(x) is below 3e-8 in magnitude either way (x < -20.8), far
    // inside the fp32-parity bound.
    constexpr float kClamp = 60.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=f"(e[i]) : "f"(fminf(t[i], kClamp)));
#pragma unroll
    for (int i = 0; i < 8; ++i) e[i] += 1.0f;
    float r[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) asm volatile("rcp.approx.ftz.f32 %0, %1;" : "=f"(r[i]) : "f"(e[2 * i] * e[2 * i + 1]));
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] = (t[2 * i] * e[2 * i + 1]) * r[i];
      v[2 * i + 1] = (t[2 * i + 1] * e[2 * i]) * r[i];
    }
  }
}

// ---------------- fp16 single-pass mode: packed-half epilogue ----------------
// The accumulator of a swish layer holds t = x / 2 (pre-scaled weights, tc_swish_scales(ns = 1)); two columns are packed
// into one f16x2 word, tanh.approx.f16x2 is ONE SFU op for both, and t + t tanh(t) = swish(x) is one packed FMA whose
// result is already the next layer's operand word: 2.5 instructions and half an SFU op per element (fp32 path: ~5.6 / 1).
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));   // saturates at +-65504 instead of producing inf
  return d;
}
__device__ __forceinline__ void unpack_f16x2(uint32_t w, float& lo, float& hi) {
  asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %2;\n\tcvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, h;\n\t}" : "=f"(lo), "=f"(hi) : "r"(w));
}
// out[4] = packed f16x2 of act(x[i] + b[i]), i = 0..7
__device__ __forceinline__ void act8_f16(const uint32_t* x, const float* b, uint32_t (&out)[4], bool relu) {
  uint32_t t[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float t0 = __uint_as_float(x[2 * i]) + b[2 * i], t1 = __uint_as_float(x[2 * i + 1]) + b[2 * i + 1];
    if (relu) { t0 = fmaxf(t0, 0.f); t1 = fmaxf(t1, 0.f); }
    t[i] = pack_f16x2(t0, t1);
  }
  if (relu) {
#pragma unroll
    for (int i = 0; i < 4; ++i) out[i] = t[i];
  } else {
    uint32_t th[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) asm volatile("tanh.approx.f16x2 %0, %1;" : "=r"(th[i]) : "r"(t[i]));
#pragma unroll
    for (int i = 0; i < 4; ++i) asm("fma.rn.f16x2 %0, %1, %2, %1;" : "=r"(out[i]) : "r"(t[i]), "r"(th[i]));
  }
}
__device__ __forceinline__ void store8_f16(unsigned char* base, uint32_t off, const float (&v)[8]) {
  *reinterpret_cast<uint4*>(base + off) = make_uint4(pack_f16x2(v[0], v[1]), pack_f16x2(v[2], v[3]), pack_f16x2(v[4], v[5]), pack_f16x2(v[6], v[7]));
}

template <int CW> __device__ __forceinline__ void tmem_ldw(uint32_t taddr, uint32_t (&x)[CW]);
template <> __device__ __forceinline__ void tmem_ldw<8>(uint32_t taddr, uint32_t (&x)[8]) { tc::tmem_ld8(taddr, x); }

}  // namespace tce
