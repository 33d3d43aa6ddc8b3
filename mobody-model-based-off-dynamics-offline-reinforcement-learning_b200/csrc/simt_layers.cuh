// fp32 CUDA-core layer routines shared by the fp32 rollout step (step_simt.cu) and the train step
// (train.cu): a CTA of 256 threads owns a tile of 64 rows whose activations live in shared memory;
// weights are read from the live nn.Parameter storage and staged 16 rows at a time with cp.async.
#pragma once
#include "common.cuh"

namespace simt {

constexpr int TM = 64;     // rows per CTA
constexpr int NT = 256;    // threads per CTA
constexpr int KC = 16;     // weight rows staged per chunk
constexpr int H = MB_H;

enum { ACT_NONE = 0, ACT_SWISH = 1, ACT_RELU = 2, ACT_TANH = 3, ACT_MASK = 4 };

__device__ __forceinline__ float apply_act(float v, int act, float scale) {
  if (act == ACT_SWISH) return mb_swish(v);
  if (act == ACT_RELU) return fmaxf(v, 0.0f);
  if (act == ACT_TANH) return tanhf(v) * scale;
  return v;
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, int src_bytes) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// Stage W rows [k0, k0+KC) x 256 columns into Wst[KC][256]; rows >= K are zero-filled.
template <bool WT>
__device__ __forceinline__ void stage_w(float* Wst, const float* __restrict__ Wg, int K, int k0) {
  const int tid = threadIdx.x;
  if (!WT) {   // Wg is [K][256] row-major: 16-byte async copies
#pragma unroll
    for (int i = 0; i < (KC * H / 4) / NT; ++i) {
      int f = tid + NT * i;
      int row = f >> 6, c4 = f & 63;
      bool ok = (k0 + row) < K;
      const float* src = ok ? (Wg + (size_t)(k0 + row) * H + c4 * 4) : Wg;
      cp_async16(Wst + row * H + c4 * 4, src, ok ? 16 : 0);
    }
  } else {     // Wg is nn.Linear [256][K]: thread n copies the K-run of output n (4-byte async copies, rows may be unaligned)
    const float* src = Wg + (size_t)tid * K + k0;
#pragma unroll
    for (int kk = 0; kk < KC; ++kk) {
      const bool ok = (k0 + kk) < K;
      unsigned d = (unsigned)__cvta_generic_to_shared(Wst + kk * H + tid);
      asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(d), "l"(ok ? src + kk : Wg), "r"(ok ? 4 : 0));
    }
  }
  cp_async_commit();
}

// Y[TM][256] = act(X[TM][K] * W + b).  X columns in [K, roundup16(K)) must be zero; ldx % 4 == 0.
// act == ACT_MASK: Y = (X W) where Y's previous content is > 0, else 0 (relu backward, in place on Ys); bias unused.
// RPT = rows per thread; the CTA's row tile is 8 * RPT rows (64 by default, 16 for small batches).
// NSTG = depth of the weight-chunk ring in Wst (NSTG * KC * 256 floats); NSTG - 1 chunks are prefetched ahead.
template <bool WT, int RPT = 8, int NSTG = 2>
__device__ void big_layer(const float* __restrict__ Xs, int ldx, int K, const float* __restrict__ Wg,
                          const float* __restrict__ bias, float* __restrict__ Ys, float* Wst, int act) {
  const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
  float acc[RPT][8];
#pragma unroll
  for (int i = 0; i < RPT; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
  const int nchunks = (K + KC - 1) / KC;
#pragma unroll
  for (int p = 0; p < NSTG - 1; ++p) {                       // prologue: one commit group per chunk, possibly empty
    if (p < nchunks) stage_w<WT>(Wst + p * (KC * H), Wg, K, p * KC); else cp_async_commit();
  }
  for (int c = 0; c < nchunks; ++c) {
    float* cur = Wst + (c % NSTG) * (KC * H);
    if (c + NSTG - 1 < nchunks) stage_w<WT>(Wst + ((c + NSTG - 1) % NSTG) * (KC * H), Wg, K, (c + NSTG - 1) * KC);
    else cp_async_commit();
    cp_async_wait<NSTG - 1>();                               // chunk c has landed (groups retire in order)
    __syncthreads();
    const float* xrow = Xs + (size_t)(ty * RPT) * ldx + c * KC;
#pragma unroll
    for (int kk = 0; kk < KC; kk += 4) {
      float4 xv[RPT];
#pragma unroll
      for (int i = 0; i < RPT; ++i) xv[i] = *reinterpret_cast<const float4*>(xrow + (size_t)i * ldx + kk);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float4 w0 = *reinterpret_cast<const float4*>(cur + (kk + q) * H + tx * 4);
        float4 w1 = *reinterpret_cast<const float4*>(cur + (kk + q) * H + 128 + tx * 4);
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
          float x = q == 0 ? xv[i].x : q == 1 ? xv[i].y : q == 2 ? xv[i].z : xv[i].w;
          acc[i][0] = fmaf(x, w0.x, acc[i][0]); acc[i][1] = fmaf(x, w0.y, acc[i][1]);
          acc[i][2] = fmaf(x, w0.z, acc[i][2]); acc[i][3] = fmaf(x, w0.w, acc[i][3]);
          acc[i][4] = fmaf(x, w1.x, acc[i][4]); acc[i][5] = fmaf(x, w1.y, acc[i][5]);
          acc[i][6] = fmaf(x, w1.z, acc[i][6]); acc[i][7] = fmaf(x, w1.w, acc[i][7]);
        }
      }
    }
    __syncthreads();
  }
  if (act == ACT_MASK) {
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
      float4* p0 = reinterpret_cast<float4*>(Ys + (size_t)(ty * RPT + i) * H + tx * 4);
      float4* p1 = reinterpret_cast<float4*>(Ys + (size_t)(ty * RPT + i) * H + 128 + tx * 4);
      const float4 m0 = *p0, m1 = *p1;
      *p0 = make_float4(m0.x > 0.f ? acc[i][0] : 0.f, m0.y > 0.f ? acc[i][1] : 0.f, m0.z > 0.f ? acc[i][2] : 0.f, m0.w > 0.f ? acc[i][3] : 0.f);
      *p1 = make_float4(m1.x > 0.f ? acc[i][4] : 0.f, m1.y > 0.f ? acc[i][5] : 0.f, m1.z > 0.f ? acc[i][6] : 0.f, m1.w > 0.f ? acc[i][7] : 0.f);
    }
    __syncthreads();
    return;
  }
  float4 b0 = *reinterpret_cast<const float4*>(bias + tx * 4);
  float4 b1 = *reinterpret_cast<const float4*>(bias + 128 + tx * 4);
#pragma unroll
  for (int i = 0; i < RPT; ++i) {
    float4 o0, o1;
    o0.x = apply_act(acc[i][0] + b0.x, act, 1.f); o0.y = apply_act(acc[i][1] + b0.y, act, 1.f);
    o0.z = apply_act(acc[i][2] + b0.z, act, 1.f); o0.w = apply_act(acc[i][3] + b0.w, act, 1.f);
    o1.x = apply_act(acc[i][4] + b1.x, act, 1.f); o1.y = apply_act(acc[i][5] + b1.y, act, 1.f);
    o1.z = apply_act(acc[i][6] + b1.z, act, 1.f); o1.w = apply_act(acc[i][7] + b1.w, act, 1.f);
    *reinterpret_cast<float4*>(Ys + (size_t)(ty * RPT + i) * H + tx * 4) = o0;
    *reinterpret_cast<float4*>(Ys + (size_t)(ty * RPT + i) * H + 128 + tx * 4) = o1;
  }
  __syncthreads();
}

// ---------------- warp-level tensor-core version of big_layer (train step) ----------------
// Same contract as big_layer (Xs/Ys fp32 tiles in shared memory, live fp32 weights in global memory), but the
// contraction runs on mma.sync m16n8k8 TF32 with both operands split on the fly into hi + lo ("3xTF32":
// lo*hi + hi*lo + hi*hi, 22 significand bits per operand, fp32 accumulate) — fp32-class accuracy (~3e-7 relative),
// which the train step needs: Q values of a fresh critic are small differences of O(1) terms and feed exp(3 q/mean|q|).
// Why warp-level MMA here and tcgen05 in the rollout: the train step at batch 128 is 320 rows in 16-row tiles, a
// latency-bound chain of ~13 dependent 256x256 layers per kernel; a 16-row tile is exactly one m16 fragment and every
// weight is used once per CTA, so weights go straight from L2 into B fragments (nn.Linear's [out][in] layout IS the
// "col" operand layout) with no shared-memory staging, and a layer takes a few us instead of ~23 us on the FMA pipe.
// Warp w owns output columns [32w, 32w+32) (4 n-tiles) of every 16-row m-tile.
__device__ __forceinline__ void mma_tf32_1688(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// hi = top 19 bits (exactly a TF32 value), lo = v - hi (exact in fp32).  The MMA reads only the top 19 bits of an
// operand, so lo gets half an ulp of TF32 added to its magnitude first: round-to-nearest instead of truncation
// (unbiased; the truncation of hi is fully compensated by lo).
__device__ __forceinline__ void split_tf32(float v, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(v) & 0xFFFFE000u;
  lo = __float_as_uint(v - __uint_as_float(hi)) + 0x1000u;
}

// [rows][256] activation tiles in shared memory are stored SWIZZLED: the 16-byte group index of a column is XORed with a
// 3-bit function of the row, so that (a) the two rows a quarter-warp reads in one 128-bit A-fragment load and (b) the
// eight rows a warp writes in one C-fragment store fall into different banks (row pitch 1 KB = same banks otherwise:
// 2-way conflicts on every A load, 8-way on every epilogue store).  XOR within a 128-byte segment: an involution that
// keeps float2 / float4 groups intact.  Every accessor of such a tile goes through swz().
__device__ __forceinline__ int swz(int r, int c) { return c ^ ((((r & 1) << 2) | ((r >> 1) & 3)) << 2); }

// Operand slots are permuted so that every global / shared load is a 128-bit vector (the contraction does not care
// which actual k sits in which k-slot as long as A and B agree, and the epilogue knows which column an n-slot is):
//   k16 block, thread (g, t): actual k = kb + 4t + i, i = 0..3; MMA #0 takes i = 0 (slot t) and 1 (slot t+4), MMA #1
//   takes i = 2, 3.  A: one LDS.128 per row.  B, nn.Linear [out][in] (WT): one LDG.128 per n-tile along k.
//   B, [k][256] row-major (!WT): n-slot g of tile nt is column n0 + 4g + nt, one LDG.128 along n per actual k.
// SWX: Xs is a swizzled [rows][256] tile (ldx = H); otherwise a plain staging buffer.  Ys is always a swizzled tile.
template <bool WT, int RPT = 8, bool SWX = false>
__device__ void big_layer_mma(const float* __restrict__ Xs, int ldx, int K, const float* __restrict__ Wg,
                              const float* __restrict__ bias, float* __restrict__ Ys, int act) {
  constexpr int MT = RPT / 2;                                  // 16-row m-tiles of the 8*RPT-row tile
  static_assert(RPT % 2 == 0, "row tile must be a multiple of 16 rows");
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int n0 = warp * 32;
  float acc[MT][4][4];
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int n = 0; n < 4; ++n)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[m][n][j] = 0.f;
  const int kblocks = (K + 15) >> 4;                           // Xs columns up to roundup16(K) are readable (zero or finite)
  const bool vec = WT ? ((K & 3) == 0) : true;                 // rows of an odd-K nn.Linear weight are not 16-byte aligned
  // raw fp32 B values of one k16 block: raw[nt][i] = B[actual k = kb + 4t + i][n-slot g of tile nt]
  auto load_b = [&](int blk, float (&raw)[4][4]) {
    const int k0 = blk * 16 + 4 * t;
    if (WT) {
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const float* w = Wg + (size_t)(n0 + nt * 8 + g) * K + k0;
        if (vec && k0 + 3 < K) {
          const float4 v = __ldg(reinterpret_cast<const float4*>(w));
          raw[nt][0] = v.x; raw[nt][1] = v.y; raw[nt][2] = v.z; raw[nt][3] = v.w;
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i) raw[nt][i] = (k0 + i < K) ? __ldg(w + i) : 0.f;
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k0 + i < K) v = __ldg(reinterpret_cast<const float4*>(Wg + (size_t)(k0 + i) * H + n0 + 4 * g));
        raw[0][i] = v.x; raw[1][i] = v.y; raw[2][i] = v.z; raw[3][i] = v.w;
      }
    }
  };
  constexpr int PF = (RPT <= 2) ? 4 : 2;              // k16 blocks of weights in flight (deeper did not pay at 64 rows)
  float rb[PF][4][4];
#pragma unroll
  for (int p = 0; p < PF; ++p) if (p < kblocks) load_b(p, rb[p]);
  auto consume = [&](int blk, float (&raw)[4][4]) {
    uint32_t bh[4][4], bl[4][4];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) split_tf32(raw[nt][i], bh[nt][i], bl[nt][i]);
    if (blk + PF < kblocks) load_b(blk + PF, raw);             // refill this slot: PF blocks of weights stay in flight
    const int k0 = blk * 16 + 4 * t;
#pragma unroll
    for (int m = 0; m < MT; ++m) {
      const int r0 = m * 16 + g, r1 = r0 + 8;
      const float4 x0 = *reinterpret_cast<const float4*>(Xs + (size_t)r0 * ldx + (SWX ? swz(r0, k0) : k0));
      const float4 x1 = *reinterpret_cast<const float4*>(Xs + (size_t)r1 * ldx + (SWX ? swz(r1, k0) : k0));
      const float xr0[4] = {x0.x, x0.y, x0.z, x0.w}, xr1[4] = {x1.x, x1.y, x1.z, x1.w};
#pragma unroll
      for (int h2 = 0; h2 < 2; ++h2) {                          // the two k8 MMAs of the block: i = 2 h2, 2 h2 + 1
        uint32_t ah[4], al[4];
        split_tf32(xr0[2 * h2], ah[0], al[0]); split_tf32(xr1[2 * h2], ah[1], al[1]);
        split_tf32(xr0[2 * h2 + 1], ah[2], al[2]); split_tf32(xr1[2 * h2 + 1], ah[3], al[3]);
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          mma_tf32_1688(acc[m][nt], al, bh[nt][2 * h2], bh[nt][2 * h2 + 1]);
          mma_tf32_1688(acc[m][nt], ah, bl[nt][2 * h2], bl[nt][2 * h2 + 1]);
          mma_tf32_1688(acc[m][nt], ah, bh[nt][2 * h2], bh[nt][2 * h2 + 1]);
        }
      }
    }
  };
  for (int blk = 0; blk < kblocks; blk += PF) {
#pragma unroll
    for (int p = 0; p < PF; ++p)
      if (blk + p < kblocks) consume(blk + p, rb[p]);          // static slot index: rb stays in registers
  }
  __syncthreads();
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int j = 0; j < 4; ++j) {                             // C fragment: row g + 8 (j >> 1), n-slot 2t + (j & 1)
        const int slot = 2 * t + (j & 1);
        const int c = WT ? (n0 + nt * 8 + slot) : (n0 + 4 * slot + nt);
        const int row = m * 16 + g + 8 * (j >> 1);
        float* p = Ys + (size_t)row * H + swz(row, c);
        const float a = acc[m][nt][j];
        if (act == ACT_MASK) *p = (*p > 0.f) ? a : 0.f;
        else *p = apply_act(a + __ldg(bias + c), act, 1.f);
      }
  __syncthreads();
}

// Narrow layers (N <= 32 or so): one thread per (row, column).  W is [K][ldw] (or [N][K] if WT).
template <bool WT, int RPT = 8, bool SWZ = false>
__device__ void small_layer(const float* __restrict__ Xs, int ldx, int K, const float* __restrict__ Wg, int ldw,
                            const float* __restrict__ bias, int N, float* __restrict__ Ys, int ldy, int act,
                            float scale) {
  for (int idx = threadIdx.x; idx < 8 * RPT * N; idx += NT) {
    int r = idx / N, n = idx - r * N;
    const float* x = Xs + (size_t)r * ldx;
    auto xi = [&](int k) { return SWZ ? swz(r, k) : k; };     // k is a multiple of 4 in the unrolled loops: the group stays intact
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int k = 0;
    if (!WT) {
      const float* w = Wg + n;
      for (; k + 4 <= K; k += 4) {
        a0 = fmaf(x[xi(k)], __ldg(w + (size_t)k * ldw), a0);
        a1 = fmaf(x[xi(k) + 1], __ldg(w + (size_t)(k + 1) * ldw), a1);
        a2 = fmaf(x[xi(k) + 2], __ldg(w + (size_t)(k + 2) * ldw), a2);
        a3 = fmaf(x[xi(k) + 3], __ldg(w + (size_t)(k + 3) * ldw), a3);
      }
      for (; k < K; ++k) a0 = fmaf(x[xi(k)], __ldg(w + (size_t)k * ldw), a0);
    } else {
      const float* w = Wg + (size_t)n * ldw;
      for (; k + 4 <= K; k += 4) {
        a0 = fmaf(x[xi(k)], __ldg(w + k), a0); a1 = fmaf(x[xi(k) + 1], __ldg(w + k + 1), a1);
        a2 = fmaf(x[xi(k) + 2], __ldg(w + k + 2), a2); a3 = fmaf(x[xi(k) + 3], __ldg(w + k + 3), a3);
      }
      for (; k < K; ++k) a0 = fmaf(x[xi(k)], __ldg(w + k), a0);
    }
    float v = ((a0 + a1) + (a2 + a3)) + (bias ? __ldg(bias + n) : 0.0f);
    Ys[(size_t)r * ldy + n] = apply_act(v, act, scale);
  }
  __syncthreads();
}

__host__ __device__ inline int rup16(int x) { return (x + 15) & ~15; }

}  // namespace simt
