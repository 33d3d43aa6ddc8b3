// Large-batch MOBODY.train step on tcgen05 (3xTF32 GEMM tiles, umma_gemm.cuh).  See the orchestration below.
#include "umma_gemm.cuh"
#include "../../include/mobody_b200.h"

template <int NP, int AS, int BS, int EPI> static const char* launch_gemm(const ug::Args& a, int max_m, cudaStream_t st) {
  const size_t bytes = 2 * ug::stage_bytes(NP);
  static bool attr_set = false;            // per instantiation
  if (!attr_set) {
    if (cudaFuncSetAttribute(ug::gemm_kernel<NP, AS, BS, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
      return "cudaFuncSetAttribute(gemm_kernel) failed";
    attr_set = true;
  }
  const dim3 grid((max_m + ug::BM - 1) / ug::BM, a.njobs, a.nsplit);
  if (mb_launch(ug::gemm_kernel<NP, AS, BS, EPI>, grid, dim3(ug::NT), bytes, st, a) != cudaSuccess) return "gemm_kernel launch failed";
  return nullptr;
}
template <int AS, int BS, int EPI> static const char* launch_np(const ug::Args& a, int max_m, bool narrow, cudaStream_t st) {
  return narrow ? launch_gemm<64, AS, BS, EPI>(a, max_m, st) : launch_gemm<256, AS, BS, EPI>(a, max_m, st);
}
// one launch: every job of `a` must use the same operand sources and epilogue class, and fit the chosen tile width
const char* mb_gemm_launch(const ug::Args& a, cudaStream_t st) {
  int max_m = 0, max_n = 0;
  for (int j = 0; j < a.njobs; ++j) {
    const ug::Job& jb = a.job[j];
    if (jb.M < 1 || jb.N < 1 || jb.N > 256 || jb.K < 0) return "gemm: bad M / N / K";
    if (jb.a_src != a.job[0].a_src || jb.b_src != a.job[0].b_src || ug::epi_class(jb.epi) != ug::epi_class(a.job[0].epi))
      return "gemm: the jobs of one launch must share their operand sources and epilogue class";
    if (jb.epi == ug::EPI_HEAD && !jb.w3) return "gemm: head job without w3";
    if (jb.M > max_m) max_m = jb.M;
    if (jb.N > max_n) max_n = jb.N;
  }
  const int as = a.job[0].a_src, bs = a.job[0].b_src, ec = ug::epi_class(a.job[0].epi);
  const bool narrow = max_n <= 64;
  using namespace ug;
  if (as == SRC_KCONTIG && bs == SRC_PACKED) {           // forward / backward-data layers on packed weight images
    if (ec == EPI_STORE) return launch_np<0, 2, EPI_STORE>(a, max_m, narrow, st);
    if (ec == EPI_MASK) return launch_np<0, 2, EPI_MASK>(a, max_m, narrow, st);
  } else if (as == SRC_KCONTIG && bs == SRC_KCONTIG) {   // forward layers
    if (ec == EPI_STORE) return launch_np<0, 0, EPI_STORE>(a, max_m, narrow, st);
    if (ec == EPI_DSWISH) return launch_np<0, 0, EPI_DSWISH>(a, max_m, narrow, st);   // ensemble layers backward: W[e][in][out] is K-contiguous in `out`
  } else if (as == SRC_KCONTIG && bs == SRC_RCONTIG) {   // backward-data
    if (ec == EPI_STORE) return launch_np<0, 1, EPI_STORE>(a, max_m, narrow, st);
    if (ec == EPI_SWISH) return launch_np<0, 1, EPI_SWISH>(a, max_m, narrow, st);     // ensemble layers forward
  } else if (as == SRC_RCONTIG && bs == SRC_RCONTIG) {   // weight gradients (and the test hook)
    if (ec == EPI_PART) return launch_np<1, 1, EPI_PART>(a, max_m, narrow, st);
    if (ec == EPI_STORE) return launch_np<1, 1, EPI_STORE>(a, max_m, narrow, st);
  } else if (ec == EPI_STORE) return launch_np<1, 0, EPI_STORE>(a, max_m, narrow, st);
  return "gemm: this operand-source / epilogue combination is not instantiated";
}

// Test hook (C ABI: mobody_selftest_gemm): C[M][N] = A * B through the tile kernel, any operand source combination.
const char* mb_gemm_selftest_launch(const float* A, const float* B, int M, int N, int K, int a_src, int b_src, int lda, int ldb,
                                    float* C, cudaStream_t st) {
  ug::Args a{}; a.njobs = 1; a.nsplit = 1;
  ug::Job& j = a.job[0];
  j.A = A; j.lda = lda; j.B = B; j.ldb = ldb; j.M = M; j.N = N; j.K = K; j.a_src = a_src; j.b_src = b_src;
  j.epi = ug::EPI_STORE; j.C = C; j.ldc = N;
  return mb_gemm_launch(a, st);
}

namespace ug {
__global__ void __launch_bounds__(256) pack_b_kernel(const __grid_constant__ PackArgs args) {
  mb_pdl_begin();
  const PackJob& jb = args.job[blockIdx.y];
  const int nchunks = (jb.K + KC - 1) / KC;
  const long long units = (long long)nchunks * (KC / 4) * jb.NP;       // one unit = (chunk, kgroup, n): 4 k values -> hi uint4 + lo uint4
  for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u < units; u += (long long)gridDim.x * blockDim.x) {
    int n, kg, c;
    if (jb.mode == SRC_KCONTIG) { kg = (int)(u % (KC / 4)); const long long t = u / (KC / 4); n = (int)(t % jb.NP); c = (int)(t / jb.NP); }   // lanes along k: coalesced reads
    else { n = (int)(u % jb.NP); const long long t = u / jb.NP; kg = (int)(t % (KC / 4)); c = (int)(t / (KC / 4)); }                            // lanes along n
    float v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int k = c * KC + kg * 4 + i;
      v[i] = (n < jb.N && k < jb.K) ? (jb.mode == SRC_KCONTIG ? __ldg(jb.src + (size_t)n * jb.ld + k) : __ldg(jb.src + (size_t)k * jb.ld + n)) : 0.f;
    }
    uint4 h, l;
    split_tf32(v[0], h.x, l.x); split_tf32(v[1], h.y, l.y); split_tf32(v[2], h.z, l.z); split_tf32(v[3], h.w, l.w);
    const size_t plane = (size_t)(KC / 4) * jb.NP * 4, base = (size_t)c * 2 * plane + ((size_t)kg * jb.NP + n) * 4;
    *reinterpret_cast<uint4*>(jb.dst + base) = h;
    *reinterpret_cast<uint4*>(jb.dst + base + plane) = l;
  }
}

}  // namespace ug

const char* mb_pack_b_launch(const ug::PackArgs& a, cudaStream_t st) {
  if (a.njobs < 1 || a.njobs > 16) return "pack_b: bad job count";
  if (mb_launch(ug::pack_b_kernel, dim3(32, a.njobs), dim3(256), 0, st, a) != cudaSuccess) return "pack_b_kernel launch failed";
  return nullptr;
}
