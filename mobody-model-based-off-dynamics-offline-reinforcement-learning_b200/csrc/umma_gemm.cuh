// fp32-class GEMM tiles on the 5th-gen tensor cores: C[128 x N] (+)= A[128 x K] * B[K x N] with tcgen05.mma.kind::tf32,
// both operands split into TF32 hi + lo planes and three MMAs per K step (lo*hi + hi*lo + hi*hi: "3xTF32", ~2^-21 per
// product -- the precision the Q-weighted BC update needs, see DESIGN.md 4.5), fp32 accumulation in TMEM.
//
// The train step at large batch is a handful of such GEMMs per layer (forward, backward-data, weight gradient) whose
// operands are fp32 tensors PyTorch owns: activations [rows][256], nn.Linear weights [out][in], batch rows.  They cannot be
// fed to the tensor core as they are (fp32 -> TF32 hi/lo needs ALU work), so a CTA's 8 warps stream K chunks of 32
// global -> registers (next chunk in flight) -> split -> shared memory in the UMMA K-major no-swizzle layout, and one thread
// issues the chunk's 12 MMAs asynchronously (tcgen05.commit -> mbarrier frees the stage): the tensor pipe works on chunk c
// while the CUDA cores split chunk c + 1.  Epilogues read the accumulator with tcgen05.ld and fuse bias / ReLU / ReLU mask /
// the one-output Q head.
//
// Operand sources (element (row, k) of a K-major operand plane; row = m for A, n for B):
//   SRC_KCONTIG : src[row * ld + k]      (activations, nn.Linear weight used "forward")
//   SRC_RCONTIG : src[k * ld + row]      (weight used "backward", and both operands of a weight gradient)
//   SRC_PACKED  : (B only) a weight matrix split ONCE per update into its hi / lo planes, already in the stage layout
//                 [chunk][plane][kgroup][n][4 k]: one cp.async.bulk per chunk replaces two thirds of the per-chunk ALU work
#pragma once
#include "common.cuh"
#include "tc_prims.cuh"
#include <stdio.h>

namespace ug {

constexpr int BM = 128;          // rows of C per CTA (UMMA M)
constexpr int KC = 16;           // K per pipeline stage = 2 UMMA K steps of 8 (two stages of a 128 x 256 tile = 96 KB: two CTAs per SM)
constexpr int NT = 256;          // threads per CTA

enum { SRC_KCONTIG = 0, SRC_RCONTIG = 1,
       SRC_PACKED = 2 };   // B only: pre-split TF32 hi/lo image in stage layout (pack_b_kernel), streamed by TMA bulk copies
// Epilogue kinds.  EPI_STORE and EPI_HEAD share one compiled epilogue (a job without w3 has no head), the others are their own
// instantiations: the epilogue body is unrolled per 32 x 32 block, so every variant compiled into it is paid in issue slots.
enum { EPI_STORE = 0,   // C = act(acc + bias)                       -> C[m][n]
       EPI_MASK = 1,    // C = mask[m][n] > 0 ? acc : 0              -> C[m][n]          (ReLU backward)
       EPI_HEAD = 2,    // h = relu(acc + bias); out1[m] = h . w3 + b3; optional C = h     (Q network tail)
       EPI_PART = 3,    // C[split][m][n] = acc, db[split][m] = row sums of the A operand (weight gradient partials)
       EPI_SWISH = 4,   // x = acc + bias -> pre[m][n] (kept for the backward pass); C = x * sigmoid(x)   (ensemble layers, dynfit.cu)
       EPI_DSWISH = 5 };// C = acc * swish'(mask[m][n]), mask = the layer's stored pre-activation         (Swish backward)
__host__ __device__ constexpr int epi_class(int epi) { return epi == EPI_HEAD ? EPI_STORE : epi; }

struct Job {
  const float* A; int lda; const float* A2; int lda2; int ksplit;     // A2: columns k >= ksplit of a KCONTIG A come from A2[m][k - ksplit]
  const float* B; int ldb;
  int M, N, K;                                                          // N <= 256; operands are zero-padded to Np = roundup16(N), KC
  int a_src, b_src, epi, relu;
  const float* bias; const float* mask; int ldmask;
  const float* w3; const float* b3;
  float* C; int ldc; float* out1; float* db;
  float* pre;                                                           // EPI_SWISH: pre-activation copy, same pitch as C (may be null)
};
struct Args { Job job[8]; int njobs, nsplit; };

__host__ __device__ inline int rup16(int x) { return (x + 15) & ~15; }
__host__ __device__ inline size_t stage_bytes(int np) { return (size_t)2 * (BM + np) * (KC / 4) * 16; }   // hi + lo planes of A and B

__device__ __forceinline__ float swish_f(float x) { return x / (1.f + expf(-x)); }
__device__ __forceinline__ float dswish_f(float x) { const float s = 1.f / (1.f + expf(-x)); return s * (1.f + x * (1.f - s)); }
__device__ __forceinline__ void split_tf32(float v, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(v) & 0xFFFFE000u;                               // exactly a TF32 value
  lo = __float_as_uint(v - __uint_as_float(hi)) + 0x1000u;             // the MMA truncates: pre-round the residual
}
__device__ __forceinline__ void put_unit(unsigned char* hi_plane, uint32_t plane_bytes, uint32_t off, const float (&v)[4]) {
  uint4 h, l;
  split_tf32(v[0], h.x, l.x); split_tf32(v[1], h.y, l.y); split_tf32(v[2], h.z, l.z); split_tf32(v[3], h.w, l.w);
  *reinterpret_cast<uint4*>(hi_plane + off) = h;
  *reinterpret_cast<uint4*>(hi_plane + plane_bytes + off) = l;
}
// kind::tf32 instruction descriptor: fp32 accumulate, TF32 A/B (format 2), both K-major, dense
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

// One operand (R rows x KC k) of one chunk: U = R / 32 units of (row, kgroup) per thread.  Mapping: a warp-iteration covers
// 8 rows x 4 kgroups (KCONTIG: each quarter-warp writes 128 contiguous bytes of shared memory, each row reads 64 contiguous
// bytes) or 32 rows x 1 kgroup (RCONTIG: 128-byte coalesced reads per k, 128-byte contiguous writes per quarter-warp).
template <int R>
struct Operand {
  static constexpr int KG = KC / 4;                 // 16-byte k groups per chunk (4)
  static constexpr int U = R * KG / NT;             // units of (row, kgroup) per thread
  float v[U][4];

  // KCONTIG: warp-iteration b covers rows 8b .. 8b+7 x all 4 kgroups (lane & 7 = row, lane >> 3 = kgroup)
  // RCONTIG: warp-iteration b covers 32 rows x 1 kgroup: kgroup = warp & 3, rows 32 (2u + (warp >> 2)) + lane
  __device__ __forceinline__ void where(int mode, int u, int& row, int& kg) const {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (mode == SRC_KCONTIG) { row = (warp * U + u) * 8 + (lane & 7); kg = lane >> 3; }
    else { row = (2 * u + (warp >> 2)) * 32 + lane; kg = warp & 3; }
  }
  __device__ __forceinline__ void load(const float* __restrict__ src, int ld, int mode, int row0, int rows, int k0, int kend,
                                       const float* __restrict__ src2, int ld2, int ksplit, float* rowsum) {
    if (mode == SRC_KCONTIG) {
      const bool vec = ((ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0) && src2 == nullptr;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        int row, kg; where(mode, u, row, kg);
        const int k = k0 + kg * 4;
        const bool rok = row < rows;
        const float* p = src + (size_t)(row0 + row) * ld + k;
        if (vec && rok && k + 4 <= kend) {
          const float4 q = __ldg(reinterpret_cast<const float4*>(p));
          v[u][0] = q.x; v[u][1] = q.y; v[u][2] = q.z; v[u][3] = q.w;
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float x = 0.f;
            if (rok && k + i < kend) x = (src2 && k + i >= ksplit) ? __ldg(src2 + (size_t)(row0 + row) * ld2 + (k + i - ksplit)) : __ldg(p + i);
            v[u][i] = x;
          }
        }
      }
    } else {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        int row, kg; where(mode, u, row, kg);
        const int k = k0 + kg * 4;
        const bool rok = row < rows;
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float x = (rok && k + i < kend) ? __ldg(src + (size_t)(k + i) * ld + row0 + row) : 0.f;
          v[u][i] = x; s += x;
        }
        if (rowsum) rowsum[u] += s;
      }
    }
  }
  __device__ __forceinline__ void store(unsigned char* hi_plane, int mode) const {
    constexpr uint32_t plane = (uint32_t)R * KG * 16;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      int row, kg; where(mode, u, row, kg);
      put_unit(hi_plane, plane, (uint32_t)kg * (R * 16) + (uint32_t)row * 16, v[u]);
    }
  }
};

// NP = padded N of the tile (B rows staged): 256 for the hidden layers, 64 for the narrow ones.
// A_SRC / B_SRC are compile-time (every job of a launch shares them): the kernel is a straight line of unrolled code that
// each CTA walks once, so its size is instruction-fetch time -- dead operand paths are not compiled in.
template <int NP, int A_SRC, int B_SRC, int EPI>
__global__ void __launch_bounds__(NT, 2) gemm_kernel(const __grid_constant__ Args args) {
  mb_pdl_begin();
#ifdef UG_TRACE
  long long t_[6]; t_[0] = clock64();
#endif
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ uint64_t bar_free[2], bar_done, bar_fullb[2];
  __shared__ uint32_t tmem_slot;
  __shared__ float red[8 * BM];
  __shared__ __align__(16) float bias_s[256], w3_s[256];     // epilogue vectors, fetched while the main loop runs
  const Job& jb = args.job[blockIdx.y];
  const int m0 = blockIdx.x * BM;
  if (m0 >= jb.M) return;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rows = min(BM, jb.M - m0);
  constexpr uint32_t A_PLANE = BM * (KC / 4) * 16, B_PLANE = NP * (KC / 4) * 16, STAGE = 2 * (A_PLANE + B_PLANE);
  constexpr uint32_t TCOLS = NP <= 32 ? 32 : NP <= 64 ? 64 : NP <= 128 ? 128 : 256;
  // K range of this CTA: whole K, or one of nsplit ranges of whole chunks (weight gradients)
  int kbeg = 0, kend = jb.K;
  if (args.nsplit > 1) {
    const long long chunks = (jb.K + KC - 1) / KC;
    kbeg = (int)(chunks * blockIdx.z / args.nsplit) * KC;
    kend = min(jb.K, (int)(chunks * (blockIdx.z + 1) / args.nsplit) * KC);
  }
  const int nchunks = kend > kbeg ? (kend - kbeg + KC - 1) / KC : 0;

  if (tid == 0) {
    tc::mbar_init(&bar_free[0], 1); tc::mbar_init(&bar_free[1], 1); tc::mbar_init(&bar_done, 1);
    tc::mbar_init(&bar_fullb[0], 1); tc::mbar_init(&bar_fullb[1], 1); tc::mbar_fence_init();
  }
  if (EPI == EPI_STORE || EPI == EPI_SWISH) {
    bias_s[tid] = (jb.bias && tid < jb.N) ? __ldg(jb.bias + tid) : 0.f;
    w3_s[tid] = (EPI == EPI_STORE && jb.w3 && tid < jb.N) ? __ldg(jb.w3 + tid) : 0.f;
  }
  if (warp == 0) tc::tmem_alloc(&tmem_slot, TCOLS);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = tmem_slot;

#ifdef UG_TRACE
  t_[1] = clock64();
#endif
  Operand<BM> oa0, oa1; Operand<NP> ob0, ob1;                           // chunk c lives in register set c & 1
  float rowsum[Operand<BM>::U];
#pragma unroll
  for (int u = 0; u < Operand<BM>::U; ++u) rowsum[u] = 0.f;
  float* rs = (A_SRC == SRC_RCONTIG && EPI == EPI_PART && jb.db) ? rowsum : nullptr;
  const int nrows_b = jb.N;                                             // valid rows of the B operand (n < N)
  const uint32_t idesc = make_idesc_tf32(BM, NP);
  // Software pipeline, global loads TWO chunks ahead: step c stores chunk c (fetched during step c - 2) into stage c & 1,
  // fetches chunk c + 2 into the registers it just freed and issues the MMAs of chunk c -- a DRAM / L2 round trip is
  // covered by two steps instead of one.  The packed B image of chunk c + 1 is requested AFTER the step's barrier, by a thread
  // that is not the MMA issuer: its wait for the MMAs of chunk c - 1 (which free that stage) no longer holds back the
  // barrier, so chunk c's MMAs are queued while chunk c - 1's still run.
  // (Measured and not kept, round 2: a ninth warp as dedicated MMA issuer with per-stage "full" mbarriers instead of the
  // barrier, with two stages of K = 16 or four of K = 8 -- 2 145 / 2 120 updates/s at batch 4096 against 2 244 for this loop.
  // A clock64 trace of the phases shows where a tile's ~45 k cycles go: the tensor pipe needs 12.6 k (96 MMAs of 128 x 256 x 8 at
  // 131 cycles), the operand path ~400 - 700 per K = 16 chunk in store + load issue + proxy fence, the chain "MMAs done -> free
  // barrier -> bulk copy -> full barrier" ~830 cycles whatever the copy size, and the epilogue 8 - 16 k.)
  auto fetch = [&](Operand<BM>& a, Operand<NP>& b, int c) {
    const int k0 = kbeg + c * KC;
    a.load(jb.A, jb.lda, A_SRC, m0, rows, k0, kend, jb.A2, jb.lda2, jb.ksplit, rs);
    if (B_SRC != SRC_PACKED) b.load(jb.B, jb.ldb, B_SRC, 0, nrows_b, k0, kend, nullptr, 0, 0, nullptr);
  };
  auto tma_b = [&](int c) {                                             // chunk c of the packed weight image -> stage c & 1
    const int nb = c & 1;
    if (c >= 2) tc::mbar_wait(&bar_free[nb], (uint32_t)(((c >> 1) - 1) & 1));
    tc::mbar_arrive_expect_tx(&bar_fullb[nb], 2 * B_PLANE);
    tc::bulk_g2s(smem + (size_t)nb * STAGE + 2 * A_PLANE, reinterpret_cast<const unsigned char*>(jb.B) + (size_t)(kbeg / KC + c) * (2 * B_PLANE),
                 2 * B_PLANE, &bar_fullb[nb]);
  };
  auto step = [&](Operand<BM>& a, Operand<NP>& b, int c) {
    const int buf = c & 1;
    unsigned char* st = smem + (size_t)buf * STAGE;
    if (c >= 2) tc::mbar_wait(&bar_free[buf], (uint32_t)(((c >> 1) - 1) & 1));      // the MMAs that read this stage are done
    a.store(st, A_SRC);
    if (B_SRC != SRC_PACKED) b.store(st + 2 * A_PLANE, B_SRC);
    if (c + 2 < nchunks) fetch(a, b, c + 2);
    tc::fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {
      if (B_SRC == SRC_PACKED) tc::mbar_wait(&bar_fullb[buf], (uint32_t)((c >> 1) & 1));
      tc::tc_fence_after();
      const uint32_t a0 = tc::smem_u32(st), b0 = a0 + 2 * A_PLANE;
#pragma unroll
      for (int s = 0; s < KC / 8; ++s) {
        const uint32_t ao = a0 + (uint32_t)s * 2u * (BM * 16), bo = b0 + (uint32_t)s * 2u * (NP * 16);
        const uint64_t ah = tc::make_smem_desc(ao, BM * 16, 128), al = tc::make_smem_desc(ao + A_PLANE, BM * 16, 128);
        const uint64_t bh = tc::make_smem_desc(bo, NP * 16, 128), bl = tc::make_smem_desc(bo + B_PLANE, NP * 16, 128);
        umma_tf32(tmem, al, bh, idesc, (c > 0 || s > 0) ? 1u : 0u);
        umma_tf32(tmem, ah, bl, idesc, 1u);
        umma_tf32(tmem, ah, bh, idesc, 1u);
      }
      tc::umma_commit(&bar_free[buf]);
      if (c + 1 == nchunks) tc::umma_commit(&bar_done);
    } else if (B_SRC == SRC_PACKED && tid == 32 && c + 1 < nchunks) tma_b(c + 1);
  };
  if (nchunks > 0) { fetch(oa0, ob0, 0); if (B_SRC == SRC_PACKED && tid == 32) tma_b(0); }
  if (nchunks > 1) fetch(oa1, ob1, 1);
#pragma unroll 1
  for (int c = 0; c < nchunks; c += 2) {
    step(oa0, ob0, c);
    if (c + 1 < nchunks) step(oa1, ob1, c + 1);
  }
#ifdef UG_TRACE
  t_[2] = clock64();
#endif
  if (nchunks > 0) tc::mbar_wait(&bar_done, 0);
  tc::tc_fence_after();
#ifdef UG_TRACE
  t_[3] = clock64();
#endif

  // ---------------- epilogue ----------------
  // Warp w owns TMEM lane quadrant q = w & 3 (32 rows) and every second 32-column block (w >> 2).  tcgen05.ld hands each
  // lane one ROW; global memory wants lanes along COLUMNS, so every 32 x 32 block is transposed through shared memory (the
  // operand stages are free now; pitch 36 floats: 128-bit stores and loads, conflict-free both ways) and all global
  // traffic -- ReLU mask in, C out -- is 128 contiguous bytes per row.
  const int q = warp & 3, half = warp >> 2;
  float* tb = reinterpret_cast<float*>(smem) + warp * (32 * 36);
  const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16);
  const int cl = (lane & 7) * 4, rl = lane >> 3;                        // coalesced phase: lane -> (row rl + 4 it, columns cl .. cl + 3)
  const int ldc = EPI == EPI_PART ? jb.N : jb.ldc;
  float* cbase = jb.C ? jb.C + (EPI == EPI_PART ? (size_t)blockIdx.z * jb.M * jb.N : 0) + (size_t)(m0 + q * 32 + rl) * ldc : nullptr;
  // fast path: whole 4-column groups, 16-byte aligned rows (every 256-wide tensor of the update)
  constexpr bool MASKED = EPI == EPI_MASK || EPI == EPI_DSWISH;
  const bool fast = (jb.N & 3) == 0 && (!jb.C || ((ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(jb.C) & 15) == 0)) &&
                    (!MASKED || ((jb.ldmask & 3) == 0 && (reinterpret_cast<uintptr_t>(jb.mask) & 15) == 0)) &&
                    (EPI != EPI_SWISH || !jb.pre || (reinterpret_cast<uintptr_t>(jb.pre) & 15) == 0);
  float* pbase = (EPI == EPI_SWISH && jb.pre) ? jb.pre + (size_t)(m0 + q * 32 + rl) * ldc : nullptr;
  float head[8];
#pragma unroll
  for (int it = 0; it < 8; ++it) head[it] = 0.f;
  for (int cb = half; cb * 32 < NP; cb += 2) {
    const int n0 = cb * 32, n = n0 + cl;
    if (n0 >= jb.N) break;
    const bool colok = n + 4 <= jb.N;
    float4 mkv[8];                                                      // ReLU-mask block: all 8 loads in flight before anything waits
    if (MASKED && fast) {
      const float* mrow = jb.mask + (size_t)(m0 + q * 32 + rl) * jb.ldmask + n;
#pragma unroll
      for (int it = 0; it < 8; ++it)
        mkv[it] = !(q * 32 + it * 4 + rl < rows && colok) ? make_float4(0.f, 0.f, 0.f, 0.f)
                  : EPI == EPI_DSWISH ? *reinterpret_cast<const float4*>(mrow + (size_t)it * 4 * jb.ldmask)     // may alias C (in place): coherent load
                                      : __ldg(reinterpret_cast<const float4*>(mrow + (size_t)it * 4 * jb.ldmask));
    }
    uint32_t x[32];
    if (nchunks > 0) { tc::tmem_ld32(taddr + (uint32_t)n0, x); tc::tmem_ld_wait(); }
    else {
#pragma unroll
      for (int jj = 0; jj < 32; ++jj) x[jj] = 0u;
    }
#pragma unroll
    for (int jj = 0; jj < 32; jj += 4)
      *reinterpret_cast<uint4*>(tb + lane * 36 + jj) = make_uint4(x[jj], x[jj + 1], x[jj + 2], x[jj + 3]);
    __syncwarp();
    if (fast) {
      float4 bq = make_float4(0.f, 0.f, 0.f, 0.f), wq = bq;
      if (EPI == EPI_STORE || EPI == EPI_SWISH) { bq = *reinterpret_cast<const float4*>(bias_s + n); wq = *reinterpret_cast<const float4*>(w3_s + n); }
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        const int rr = it * 4 + rl;
        float4 v = *reinterpret_cast<const float4*>(tb + rr * 36 + cl);
        if (EPI == EPI_MASK) {
          v.x = mkv[it].x > 0.f ? v.x : 0.f; v.y = mkv[it].y > 0.f ? v.y : 0.f; v.z = mkv[it].z > 0.f ? v.z : 0.f; v.w = mkv[it].w > 0.f ? v.w : 0.f;
        } else if (EPI == EPI_DSWISH) {
          v.x *= dswish_f(mkv[it].x); v.y *= dswish_f(mkv[it].y); v.z *= dswish_f(mkv[it].z); v.w *= dswish_f(mkv[it].w);
        } else if (EPI == EPI_SWISH) {
          v.x += bq.x; v.y += bq.y; v.z += bq.z; v.w += bq.w;
          if (pbase && colok && q * 32 + rr < rows) *reinterpret_cast<float4*>(pbase + (size_t)it * 4 * ldc + n) = v;
          v.x = swish_f(v.x); v.y = swish_f(v.y); v.z = swish_f(v.z); v.w = swish_f(v.w);
        } else if (EPI != EPI_PART) {
          v.x += bq.x; v.y += bq.y; v.z += bq.z; v.w += bq.w;
          if (jb.relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
          if (EPI == EPI_STORE) head[it] = fmaf(v.x, wq.x, fmaf(v.y, wq.y, fmaf(v.z, wq.z, fmaf(v.w, wq.w, head[it]))));
        }
        if (cbase && colok && q * 32 + rr < rows) *reinterpret_cast<float4*>(cbase + (size_t)it * 4 * ldc + n) = v;
      }
    } else {   // ragged / unaligned outputs (narrow heads, the 35-column first-layer gradients): compact scalar loop
#pragma unroll 1
      for (int e = lane; e < 32 * 32; e += 32) {
        const int rr = e >> 5, c = e & 31, nn = n0 + c, r = q * 32 + rr;
        if (nn >= jb.N || r >= rows) continue;
        float t = tb[rr * 36 + c];
        if (EPI == EPI_MASK) t = __ldg(jb.mask + (size_t)(m0 + r) * jb.ldmask + nn) > 0.f ? t : 0.f;
        else if (EPI == EPI_DSWISH) t *= dswish_f(jb.mask[(size_t)(m0 + r) * jb.ldmask + nn]);
        else if (EPI == EPI_SWISH) {
          t += bias_s[nn];
          if (jb.pre) jb.pre[(size_t)(m0 + r) * ldc + nn] = t;
          t = swish_f(t);
        } else if (EPI != EPI_PART) {
          t += bias_s[nn];
          if (jb.relu) t = fmaxf(t, 0.f);
        }
        if (jb.C) jb.C[(EPI == EPI_PART ? (size_t)blockIdx.z * jb.M * jb.N : 0) + (size_t)(m0 + r) * ldc + nn] = t;
      }
    }
    __syncwarp();
  }
  if (EPI == EPI_STORE && jb.w3) {   // a row's dot product: 8 lanes (column groups) of this warp, then the two column halves through shared memory
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      float h = head[it];
      h += __shfl_xor_sync(0xffffffffu, h, 1); h += __shfl_xor_sync(0xffffffffu, h, 2); h += __shfl_xor_sync(0xffffffffu, h, 4);
      if ((lane & 7) == 0) red[half * BM + q * 32 + it * 4 + rl] = h;
    }
    __syncthreads();
    if (tid < rows) jb.out1[m0 + tid] = red[tid] + red[BM + tid] + __ldg(jb.b3);
  }
  if (A_SRC == SRC_RCONTIG && EPI == EPI_PART && jb.db) {         // bias gradient: row sums of A (= column sums of D), fixed order
#pragma unroll
    for (int u = 0; u < Operand<BM>::U; ++u) red[(warp & 3) * BM + (2 * u + (warp >> 2)) * 32 + lane] = rowsum[u];   // [kgroup][row]
    __syncthreads();
    if (tid < rows) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < 4; ++w) s += red[w * BM + tid];
      jb.db[(size_t)blockIdx.z * jb.M + m0 + tid] = s;
    }
  }
#ifdef UG_TRACE
  t_[4] = clock64();
#endif
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem, TCOLS);
#ifdef UG_TRACE
  t_[5] = clock64();
  if (tid == 0 && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0)
    printf("UG_TRACE NP=%d K=%d chunks=%d epi=%d: setup %lld loop %lld drain %lld epilogue %lld dealloc %lld\n", NP, jb.K, nchunks, jb.epi, t_[1]-t_[0], t_[2]-t_[1], t_[3]-t_[2], t_[4]-t_[3], t_[5]-t_[4]);
#endif
}

// ---- packed B images: a weight matrix split once per update into TF32 hi / lo planes, in the stage layout of gemm_kernel<NP> ----
// image[chunk][plane][kgroup 0..3][n 0..NP)[4 k]; logical B[n][k] = src[n * ld + k] (mode SRC_KCONTIG) or src[k * ld + n] (SRC_RCONTIG)
struct PackJob { const float* src; int ld, mode, N, K, NP; uint32_t* dst; };
struct PackArgs { PackJob job[16]; int njobs; };
__host__ __device__ inline size_t packed_floats(int K, int NP) { return (size_t)((K + KC - 1) / KC) * 2 * (KC / 4) * NP * 4; }
}  // namespace ug
