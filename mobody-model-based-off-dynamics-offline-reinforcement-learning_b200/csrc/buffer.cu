// Replay-buffer and rollout plumbing kernels: HBM-bound byte movers.
//
// Device-resident replacement for ReplayBuffer (reference algo/utils.py:13-193) and for the
// host-side masking/concat in MOBODY.rollout (algo/offline_offline/mobody.py:624-653).
// A transition is one packed row of RW = roundup4(2S+A+2) floats:
//     [ state(S) | action(A) | next_state(S) | reward | not_done | 0-pad ]
// so that sample() is a 128-bit-vectorised row gather and add_batch() a row scatter.
#include "common.cuh"
#include "philox.cuh"
#include "term.cuh"
#include "../../include/mobody_b200.h"

namespace buf {

constexpr int NT = 256;

// out[i,:] = rows[idx[i],:]   (ReplayBuffer.sample, utils.py:127-148, with idx given)
__global__ void gather_rows_kernel(const float4* __restrict__ rows, const int64_t* __restrict__ idx,
                                   long long n, int rw4, float4* __restrict__ out) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = n * rw4;
  for (; t < total; t += (long long)gridDim.x * blockDim.x) {
    long long i = t / rw4; int c = (int)(t - i * rw4);
    out[t] = __ldg(rows + (size_t)idx[i] * rw4 + c);
  }
}

// idx[i] = mulhi(philox(i, draw), size)   (np.random.randint(0,size,n), utils.py:128)
__global__ void philox_indices_kernel(int64_t* __restrict__ idx, long long n, unsigned long long seed,
                                      unsigned int draw, unsigned int size) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i < n; i += (long long)gridDim.x * blockDim.x) {
    Philox4 b = philox4x32_10((uint32_t)i, (uint32_t)((unsigned long long)i >> 32), draw, 0u, (uint32_t)seed, MB_STREAM_INDEX);
    idx[i] = (int64_t)(((uint64_t)b.x * (uint64_t)size) >> 32);
  }
}

// Fused Philox index draw + row gather for up to 4 buffers in one launch (blockIdx.y = job): the three buffer samples of
// one MOBODY.train step (mobody.py:399-400, 524).  Indices are exactly those of philox_indices_kernel.
struct SampleJobs { const float4* rows[4]; float4* out[4]; long long n[4]; unsigned int size[4], draw[4]; unsigned long long seed[4]; };
__global__ void sample_rows_kernel(SampleJobs j, int rw4) {
  const int b = blockIdx.y;
  const long long total = j.n[b] * rw4;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long i = t / rw4; const int c = (int)(t - i * rw4);
    Philox4 p = philox4x32_10((uint32_t)i, (uint32_t)((unsigned long long)i >> 32), j.draw[b], 0u, (uint32_t)j.seed[b], MB_STREAM_INDEX);
    const size_t src = (size_t)(((uint64_t)p.x * (uint64_t)j.size[b]) >> 32);
    j.out[b][t] = __ldg(j.rows[b] + src * rw4 + c);
  }
}

// Pack separate [n,S],[n,A],[n,S],[n,1],[n,1] arrays into rows; done_is_terminal: store 1 - d (utils.py:73).
__global__ void pack_rows_kernel(const float* __restrict__ s, const float* __restrict__ a, const float* __restrict__ ns,
                                 const float* __restrict__ r, const float* __restrict__ d, long long n, int S, int A,
                                 int rw, int done_is_terminal, float* __restrict__ out) {
  const int rw4 = rw >> 2;                                  // one thread per 16-byte group of an output row (128-bit stores)
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = n * rw4;
  for (; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long i = t / rw4; const int c0 = (int)(t - i * rw4) * 4;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = c0 + j;
      float x = 0.f;
      if (c < S) x = __ldg(s + i * S + c);
      else if (c < S + A) x = __ldg(a + i * A + (c - S));
      else if (c < 2 * S + A) x = __ldg(ns + i * S + (c - S - A));
      else if (c == 2 * S + A) x = __ldg(r + i);
      else if (c == 2 * S + A + 1) x = done_is_terminal ? 1.0f - __ldg(d + i) : __ldg(d + i);
      v[j] = x;
    }
    reinterpret_cast<float4*>(out)[t] = make_float4(v[0], v[1], v[2], v[3]);
  }
}

// Same, for 16-byte aligned sources: a tile of TR rows is a CONTIGUOUS range of each source array, so the tile is fetched with
// 128-bit loads straight down each array (all of a thread's loads in flight before the first use), assembled as the row
// image in shared memory and written out as one contiguous run of 128-bit stores.  (The per-16-byte-group kernel above reads
// with 4-byte loads from five places per store: 0.49 of the HBM peak at 2 M rows; this one is bound by bytes in flight.)
constexpr int PACK_TR = 64;
template <int NV>     // NV = 128-bit loads per thread per source array (compile-time so they are all issued before use)
__device__ __forceinline__ void pack_src(const float* __restrict__ src, int len, int w, int col0, int rw, float* img, bool flip) {
  const int nv = len >> 2;
  float4 v[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int i = threadIdx.x + k * blockDim.x;
    v[k] = i < nv ? __ldg(reinterpret_cast<const float4*>(src) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int i = threadIdx.x + k * blockDim.x;
    if (i < nv) {
      const float x[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
      int row = (4 * i) / w, col = (4 * i) - row * w;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        img[row * rw + col0 + col] = flip ? 1.0f - x[j] : x[j];
        if (++col == w) { col = 0; ++row; }
      }
    }
  }
  for (int e = (nv << 2) + threadIdx.x; e < len; e += blockDim.x) {      // (only a ragged last tile has a tail)
    const float x = __ldg(src + e);
    img[(e / w) * rw + col0 + e % w] = flip ? 1.0f - x : x;
  }
}
template <int NVS, int NVA>
__global__ void __launch_bounds__(256) pack_rows_tile_kernel(const float* __restrict__ s, const float* __restrict__ a, const float* __restrict__ ns,
                                                             const float* __restrict__ r, const float* __restrict__ d, long long n, int S, int A,
                                                             int rw, int done_is_terminal, float* __restrict__ out) {
  extern __shared__ __align__(16) float img[];                          // [PACK_TR][rw]
  const long long tiles = (n + PACK_TR - 1) / PACK_TR;
  for (int e = threadIdx.x; e < PACK_TR * rw; e += blockDim.x) img[e] = 0.f;     // the pad columns stay zero
  for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
    const long long r0 = t * PACK_TR;
    const int rows = (int)min((long long)PACK_TR, n - r0);
    __syncthreads();                                                    // the previous tile's stores have read the image
    pack_src<NVS>(s + r0 * S, rows * S, S, 0, rw, img, false);
    pack_src<NVA>(a + r0 * A, rows * A, A, S, rw, img, false);
    pack_src<NVS>(ns + r0 * S, rows * S, S, S + A, rw, img, false);
    pack_src<1>(r + r0, rows, 1, 2 * S + A, rw, img, false);
    pack_src<1>(d + r0, rows, 1, 2 * S + A + 1, rw, img, done_is_terminal != 0);
    __syncthreads();
    float4* dst = reinterpret_cast<float4*>(out + r0 * rw);
    const float4* src = reinterpret_cast<const float4*>(img);
    for (int i = threadIdx.x; i < rows * (rw >> 2); i += blockDim.x) dst[i] = src[i];
  }
}

// Ring insert with the reference's single wrap (utils.py:43-92): src row i -> dst row (ptr + i) % cap.
// n_dev (nullable) holds the live row count on device (rollout output) so no host sync is needed.
__global__ void ring_insert_kernel(const float4* __restrict__ src, long long n_cap, const int* __restrict__ n_dev,
                                   int rw4, long long ptr, long long cap, float4* __restrict__ dst) {
  long long n = n_dev ? min((long long)*n_dev, n_cap) : n_cap;
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = n * rw4;
  for (; t < total; t += (long long)gridDim.x * blockDim.x) {
    long long i = t / rw4; int c = (int)(t - i * rw4);
    long long j = ptr + i; if (j >= cap) j -= cap;
    dst[(size_t)j * rw4 + c] = src[t];
  }
}

// add_batch straight from a rollout slab: packed row [obs | act | next_obs | reward | terminal | penalty] (W = 2S+A+3 floats)
// -> buffer row [obs | act | next_obs | reward | 1 - terminal | 0-pad] (rw floats) at ring position (ptr + i) % cap.
__global__ void ring_insert_transitions_kernel(const float* __restrict__ packed, long long n_cap, const int* __restrict__ n_dev,
                                               int S, int A, int rw4, long long ptr, long long cap, float4* __restrict__ dst) {
  const long long n = n_dev ? min((long long)*n_dev, n_cap) : n_cap;
  const int W = 2 * S + A + 3, nd = 2 * S + A + 1;
  const long long total = n * rw4;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long i = t / rw4; const int c0 = (int)(t - i * rw4) * 4;
    const float* src = packed + i * W;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { const int c = c0 + j; v[j] = c < nd ? src[c] : (c == nd ? 1.0f - src[nd] : 0.f); }
    long long r = ptr + i; if (r >= cap) r -= cap;
    dst[(size_t)r * rw4 + (c0 >> 2)] = make_float4(v[0], v[1], v[2], v[3]);
  }
}

// terminal[i] = term_fn(next_obs[i,:])   (terminal_funs.py via mobody_dynamics.py:237)
__global__ void termination_kernel(const float* __restrict__ x, long long n, int S, int kind, unsigned char* __restrict__ out) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (unsigned char)mb_terminal(kind, x + i * S, S);
}

// ---------------- stable stream compaction: keep[i] != 0 rows, original order ----------------
// pass 1: per-block (1024 rows) counts; pass 2: exclusive scan of block counts (one CTA) + total;
// pass 3: each block recomputes local ranks and emits pos[rank] = i.  n may live on device.
constexpr int CB = 1024;

__device__ __forceinline__ int block_exclusive_scan_1024(int flag, int* warp_sums, int& block_total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  unsigned bal = __ballot_sync(0xffffffffu, flag);
  int local = __popc(bal & ((1u << lane) - 1u));
  if (lane == 0) warp_sums[w] = __popc(bal);
  __syncthreads();
  if (w == 0) {
    int v = warp_sums[lane], x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    warp_sums[lane] = x - v;
    if (lane == 31) warp_sums[32] = x;
  }
  __syncthreads();
  block_total = warp_sums[32];
  return warp_sums[w] + local;
}

// keep predicate kinds
enum { KEEP_U8_ZERO = 0,   // keep where flags_u8[i] == 0   (non-terminal rows, mobody.py:635)
       KEEP_F32_LE = 1,    // keep where vals[i] <= thr     (rollout filter, mobody.py:649)
       KEEP_F32_LT = 2,    // keep where vals[i] <  thr     (dataset-(s,a) filter, mobody.py:468)
       KEEP_U8_VALID = 3 };// keep where flags_u8[i] != 0xFF (rows a rollout step actually wrote)

__device__ __forceinline__ int keep_pred(int kind, const unsigned char* f, const float* v, float thr, long long i) {
  if (kind == KEEP_U8_ZERO) return f[i] == 0;
  if (kind == KEEP_U8_VALID) return f[i] != 0xFF;
  if (kind == KEEP_F32_LE) return v[i] <= thr;
  return v[i] < thr;
}

__global__ void __launch_bounds__(CB) compact_count_kernel(int kind, const unsigned char* __restrict__ f, const float* __restrict__ v,
                                                          float thr, long long n_cap, const int* __restrict__ n_dev,
                                                          int* __restrict__ block_counts) {
  __shared__ int ws[33];
  long long n = n_dev ? min((long long)*n_dev, n_cap) : n_cap;
  long long i = (long long)blockIdx.x * CB + threadIdx.x;
  int flag = (i < n) ? keep_pred(kind, f, v, thr, i) : 0;
  int tot; block_exclusive_scan_1024(flag, ws, tot);
  if (threadIdx.x == 0) block_counts[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(1024) compact_scan_kernel(int* __restrict__ block_counts, int nblocks, int* __restrict__ total_out) {
  __shared__ int ws[33];
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < nblocks; base += 1024) {
    int i = base + threadIdx.x;
    int v = (i < nblocks) ? block_counts[i] : 0;
    // inclusive scan of v over the CTA
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) ws[w] = x;
    __syncthreads();
    if (w == 0) {
      int s = ws[lane], t = s;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, t, o); if (lane >= o) t += y; }
      ws[lane] = t - s;
      if (lane == 31) ws[32] = t;
    }
    __syncthreads();
    int excl = carry + ws[w] + x - v;
    if (i < nblocks) block_counts[i] = excl;
    __syncthreads();
    if (threadIdx.x == 0) carry += ws[32];
    __syncthreads();
  }
  if (threadIdx.x == 0) *total_out = carry;
}

__global__ void __launch_bounds__(CB) compact_emit_kernel(int kind, const unsigned char* __restrict__ f, const float* __restrict__ v,
                                                         float thr, long long n_cap, const int* __restrict__ n_dev,
                                                         const int* __restrict__ block_offsets, int* __restrict__ pos) {
  __shared__ int ws[33];
  long long n = n_dev ? min((long long)*n_dev, n_cap) : n_cap;
  long long i = (long long)blockIdx.x * CB + threadIdx.x;
  int flag = (i < n) ? keep_pred(kind, f, v, thr, i) : 0;
  int tot; int rank = block_exclusive_scan_1024(flag, ws, tot);
  if (flag) pos[block_offsets[blockIdx.x] + rank] = (int)i;
}

// dst[j, 0:w] = src[pos[j], 0:w] for j < *m_dev  (row gather by int32 positions; generic width)
__global__ void gather_pos_kernel(const float* __restrict__ src, int w, int src_ld, const int* __restrict__ pos,
                                  const int* __restrict__ m_dev, long long m_cap, float* __restrict__ dst, int dst_ld) {
  long long m = m_dev ? min((long long)*m_dev, m_cap) : m_cap;
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = m * w;
  for (; t < total; t += (long long)gridDim.x * blockDim.x) {
    long long j = t / w; int c = (int)(t - j * w);
    dst[j * dst_ld + c] = src[(size_t)pos[j] * src_ld + c];
  }
}
__global__ void gather_pos_i64_kernel(const long long* __restrict__ src, const int* __restrict__ pos,
                                      const int* __restrict__ m_dev, long long m_cap, long long* __restrict__ dst) {
  long long m = m_dev ? min((long long)*m_dev, m_cap) : m_cap;
  long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (; j < m; j += (long long)gridDim.x * blockDim.x) dst[j] = src[pos[j]];
}

// ---------------- whole-rollout plumbing (MOBODY.rollout, mobody.py:596-657) ----------------
// init: row ids of step 0, "never produced" markers for the rows of steps >= 1 (penalty +inf fails every `<=`
// filter, terminal 0xFF marks a slot no step wrote), live-row counts.
__global__ void rollout_init_kernel(long long* __restrict__ row_ids, unsigned long long row0, int B, int T,
                                    float* __restrict__ pens, unsigned char* __restrict__ terms, int* __restrict__ counts) {
  const long long total = (long long)T * B;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    if (i < B) row_ids[i] = (long long)(row0 + (unsigned long long)i);
    else { pens[i] = __int_as_float(0x7f800000); terms[i] = 0xFF; }
  }
  if (blockIdx.x == 0 && threadIdx.x <= T + 1) counts[threadIdx.x] = threadIdx.x == 0 ? B : 0;
}

// next step's inputs: obs[j,:] = next_obs[pos[j],:], row_ids[j] = row_ids_prev[pos[j]] for j < *m_dev (mobody.py:635-639)
__global__ void rollout_advance_kernel(const float* __restrict__ nexts, const long long* __restrict__ ids_prev, int S,
                                       const int* __restrict__ pos, const int* __restrict__ m_dev, long long m_cap,
                                       float* __restrict__ obs_next, long long* __restrict__ ids_next) {
  const long long m = min((long long)*m_dev, m_cap);
  const long long total = m * (S + 1);
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long j = t / (S + 1); const int c = (int)(t - j * (S + 1));
    const size_t p = (size_t)pos[j];
    if (c < S) obs_next[j * S + c] = nexts[p * S + c];
    else ids_next[j] = ids_prev[p];
  }
}

// packed[j,:] = [obs | act | next_obs | reward | terminal | penalty] of slot pos[j], j < *m_dev  (mobody.py:641-653)
__global__ void rollout_pack_kernel(const float* __restrict__ obss, const float* __restrict__ acts, const float* __restrict__ nexts,
                                    const float* __restrict__ rews, const unsigned char* __restrict__ terms,
                                    const float* __restrict__ pens, int S, int A, const int* __restrict__ pos,
                                    const int* __restrict__ m_dev, long long m_cap, float* __restrict__ packed) {
  const int W = 2 * S + A + 3;
  const long long m = min((long long)*m_dev, m_cap);
  const long long total = m * W;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long j = t / W; const int c = (int)(t - j * W);
    const size_t p = (size_t)pos[j];
    float v;
    if (c < S) v = obss[p * S + c];
    else if (c < S + A) v = acts[p * A + (c - S)];
    else if (c < 2 * S + A) v = nexts[p * S + (c - S - A)];
    else if (c == 2 * S + A) v = rews[p];
    else if (c == 2 * S + A + 1) v = (float)terms[p];
    else v = pens[p];
    packed[t] = v;
  }
}

// stats[0] = sum of rewards over every produced slot (terminal != 0xFF), stats[1] = number of produced slots.
// Fixed-order reduction: per-block partials, the last block to finish adds them in block order (deterministic).
constexpr int SB = 256;
__global__ void __launch_bounds__(SB) rollout_stats_kernel(const float* __restrict__ rews, const unsigned char* __restrict__ terms,
                                                          long long n, double* __restrict__ partial, unsigned int* __restrict__ ticket,
                                                          double* __restrict__ stats) {
  __shared__ double sh[2][SB];
  __shared__ bool last;
  double s = 0.0, c = 0.0;
  const long long per = (n + gridDim.x - 1) / gridDim.x;
  const long long lo = (long long)blockIdx.x * per, hi = min(n, lo + per);
  for (long long i = lo + threadIdx.x; i < hi; i += SB) if (terms[i] != 0xFF) { s += (double)rews[i]; c += 1.0; }
  sh[0][threadIdx.x] = s; sh[1][threadIdx.x] = c;
  __syncthreads();
  for (int o = SB / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) { sh[0][threadIdx.x] += sh[0][threadIdx.x + o]; sh[1][threadIdx.x] += sh[1][threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    partial[2 * blockIdx.x] = sh[0][0]; partial[2 * blockIdx.x + 1] = sh[1][0];
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (last && threadIdx.x == 0) {
    __threadfence();
    double ts = 0.0, tc = 0.0;
    for (unsigned b = 0; b < gridDim.x; ++b) { ts += partial[2 * b]; tc += partial[2 * b + 1]; }
    stats[0] = ts; stats[1] = tc;
    *ticket = 0u;                      // re-armed for the next call on this stream
  }
}

// ---------------- policy evaluation in the model (mobody_model_eval) ----------------
// init: zeroed per-start outputs, row ids of step 0, live rows entering step 0
__global__ void model_eval_init_kernel(long long* __restrict__ row_ids, unsigned long long row0, int B, double* __restrict__ ret,
                                       double* __restrict__ ret_disc, int* __restrict__ length, int* __restrict__ counts) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B; i += gridDim.x * blockDim.x) {
    row_ids[i] = (long long)(row0 + (unsigned long long)i);
    ret[i] = 0.0; ret_disc[i] = 0.0; length[i] = 0;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) counts[0] = B;
}

// live row i < *n_dev of step t: its start row gets the step's reward.  Explicitly rounded product and sum (no FMA
// contraction): the host reproduces the same float64 sequence bit for bit.
__global__ void model_eval_accumulate_kernel(const float* __restrict__ reward, const long long* __restrict__ row_ids,
                                             unsigned long long row0, const int* __restrict__ n_dev, int t, double disc,
                                             double* __restrict__ ret, double* __restrict__ ret_disc, int* __restrict__ length) {
  const int n = *n_dev;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const long long id = (long long)((unsigned long long)row_ids[i] - row0);
    const double r = (double)reward[i];
    ret[id] = __dadd_rn(ret[id], r);
    ret_disc[id] = __dadd_rn(ret_disc[id], __dmul_rn(disc, r));
    length[id] = t + 1;
  }
}

// `par` reward penalty (mobody.py:428-434): reward[i] -= coef * mean_j (next_state[i,j] - pred[i,j])^2 on the first n batch
// rows, in place; mean_out = batch mean of the penalty.  One CTA (n is a batch size): thread t owns rows t, t+1024, ...;
// the per-thread sums are combined in a fixed tree, so the logged mean is deterministic.
__global__ void __launch_bounds__(1024) par_penalty_kernel(float* __restrict__ rows, int n, int S, int A, int rw,
                                                          const float* __restrict__ pred, float coef, float* __restrict__ mean_out) {
  __shared__ float sh[1024];
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += 1024) {
    float* x = rows + (size_t)i * rw;
    const float* ns = x + S + A;
    const float* p = pred + (size_t)i * S;
    float s = 0.f;
    for (int j = 0; j < S; ++j) { const float d = ns[j] - p[j]; s = fmaf(d, d, s); }
    const float pen = s / (float)S;
    x[2 * S + A] -= coef * pen;
    acc += pen;
  }
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0 && mean_out) *mean_out = sh[0] / (float)n;
}

}  // namespace buf

static inline int grid_for(long long work, int nt, int max_blocks = 148 * 16) {
  long long g = (work + nt - 1) / nt;
  if (g < 1) g = 1;
  if (g > max_blocks) g = max_blocks;
  return (int)g;
}

// ---- host launchers ----
void mb_gather_rows_launch(const float* rows, const int64_t* idx, long long n, int rw, float* out, cudaStream_t st) {
  if (n <= 0) return;
  buf::gather_rows_kernel<<<grid_for(n * (rw / 4), buf::NT), buf::NT, 0, st>>>(
      reinterpret_cast<const float4*>(rows), idx, n, rw / 4, reinterpret_cast<float4*>(out));
}
void mb_philox_indices_launch(int64_t* idx, long long n, unsigned long long seed, unsigned int draw, unsigned int size, cudaStream_t st) {
  if (n <= 0) return;
  buf::philox_indices_kernel<<<grid_for(n, buf::NT), buf::NT, 0, st>>>(idx, n, seed, draw, size);
}
void mb_pack_rows_launch(const float* s, const float* a, const float* ns, const float* r, const float* d, long long n,
                         int S, int A, int rw, int done_is_terminal, float* out, cudaStream_t st) {
  if (n <= 0) return;
  const bool aligned = ((reinterpret_cast<uintptr_t>(s) | reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(ns) |
                         reinterpret_cast<uintptr_t>(r) | reinterpret_cast<uintptr_t>(d) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  const size_t smem = (size_t)buf::PACK_TR * rw * sizeof(float);
  constexpr int threads = 128, per_sm = 16;   // measured: 128 x 16 CTAs per SM 0.91 of the HBM peak, 256 x 8: 0.73
  const int nvs = (buf::PACK_TR / 4 * S + threads - 1) / threads, nva = (buf::PACK_TR / 4 * A + threads - 1) / threads;   // 128-bit loads per thread per array
  if (aligned && n >= 4096 && smem <= 48 * 1024 && nvs <= 8 && nva <= 4) {
    const long long tiles = (n + buf::PACK_TR - 1) / buf::PACK_TR;
    const unsigned grid = (unsigned)(tiles < 148LL * per_sm ? tiles : 148LL * per_sm);
#define MB_PACK(NS_, NA_) buf::pack_rows_tile_kernel<NS_, NA_><<<grid, threads, smem, st>>>(s, a, ns, r, d, n, S, A, rw, done_is_terminal, out)
    if (nvs <= 1 && nva <= 1) MB_PACK(1, 1);
    else if (nvs <= 2 && nva <= 1) MB_PACK(2, 1);
    else if (nvs <= 4 && nva <= 2) MB_PACK(4, 2);
    else MB_PACK(8, 4);
#undef MB_PACK
    return;
  }
  buf::pack_rows_kernel<<<grid_for(n * (rw / 4), buf::NT), buf::NT, 0, st>>>(s, a, ns, r, d, n, S, A, rw, done_is_terminal, out);
}
void mb_ring_insert_launch(const float* src, long long n_cap, const int* n_dev, int rw, long long ptr, long long cap,
                           float* dst, cudaStream_t st) {
  if (n_cap <= 0) return;
  buf::ring_insert_kernel<<<grid_for(n_cap * (rw / 4), buf::NT), buf::NT, 0, st>>>(
      reinterpret_cast<const float4*>(src), n_cap, n_dev, rw / 4, ptr, cap, reinterpret_cast<float4*>(dst));
}
void mb_termination_launch(const float* x, long long n, int S, int kind, unsigned char* out, cudaStream_t st) {
  if (n <= 0) return;
  buf::termination_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, n, S, kind, out);
}
// scratch: int[ceil(n_cap/1024) + 1]
void mb_compact_launch(int kind, const unsigned char* flags, const float* vals, float thr, long long n_cap, const int* n_dev,
                       int* scratch, int* pos, int* count_out, cudaStream_t st) {
  if (n_cap <= 0) { cudaMemsetAsync(count_out, 0, sizeof(int), st); return; }
  int nb = (int)((n_cap + buf::CB - 1) / buf::CB);
  buf::compact_count_kernel<<<nb, buf::CB, 0, st>>>(kind, flags, vals, thr, n_cap, n_dev, scratch);
  buf::compact_scan_kernel<<<1, 1024, 0, st>>>(scratch, nb, count_out);
  buf::compact_emit_kernel<<<nb, buf::CB, 0, st>>>(kind, flags, vals, thr, n_cap, n_dev, scratch, pos);
}
void mb_gather_pos_launch(const float* src, int w, int src_ld, const int* pos, const int* m_dev, long long m_cap,
                          float* dst, int dst_ld, cudaStream_t st) {
  if (m_cap <= 0) return;
  buf::gather_pos_kernel<<<grid_for(m_cap * w, buf::NT), buf::NT, 0, st>>>(src, w, src_ld, pos, m_dev, m_cap, dst, dst_ld);
}
void mb_gather_pos_i64_launch(const long long* src, const int* pos, const int* m_dev, long long m_cap, long long* dst, cudaStream_t st) {
  if (m_cap <= 0) return;
  buf::gather_pos_i64_kernel<<<grid_for(m_cap, buf::NT), buf::NT, 0, st>>>(src, pos, m_dev, m_cap, dst);
}

void mb_ring_insert_transitions_launch(const float* packed, long long n_cap, const int* n_dev, int S, int A, int rw, long long ptr, long long cap,
                                        float* dst, cudaStream_t st) {
  if (n_cap <= 0) return;
  buf::ring_insert_transitions_kernel<<<grid_for(n_cap * (rw / 4), buf::NT), buf::NT, 0, st>>>(packed, n_cap, n_dev, S, A, rw / 4, ptr, cap,
                                                                                             reinterpret_cast<float4*>(dst));
}
void mb_par_penalty_launch(float* rows, int n, int S, int A, int rw, const float* pred, float coef, float* mean_out, cudaStream_t st) {
  buf::par_penalty_kernel<<<1, 1024, 0, st>>>(rows, n, S, A, rw, pred, coef, mean_out);
}

// ---- whole-rollout plumbing ----
void mb_rollout_init_launch(long long* row_ids, unsigned long long row0, int B, int T, float* pens, unsigned char* terms,
                            int* counts, cudaStream_t st) {
  buf::rollout_init_kernel<<<grid_for((long long)T * B, buf::NT), buf::NT, 0, st>>>(row_ids, row0, B, T, pens, terms, counts);
}
void mb_rollout_advance_launch(const float* nexts, const long long* ids_prev, int S, const int* pos, const int* m_dev,
                               long long m_cap, float* obs_next, long long* ids_next, cudaStream_t st) {
  if (m_cap <= 0) return;
  buf::rollout_advance_kernel<<<grid_for(m_cap * (S + 1), buf::NT), buf::NT, 0, st>>>(nexts, ids_prev, S, pos, m_dev, m_cap, obs_next, ids_next);
}
void mb_rollout_pack_launch(const float* obss, const float* acts, const float* nexts, const float* rews, const unsigned char* terms,
                            const float* pens, int S, int A, const int* pos, const int* m_dev, long long m_cap, float* packed,
                            cudaStream_t st) {
  if (m_cap <= 0) return;
  buf::rollout_pack_kernel<<<grid_for(m_cap * (2 * S + A + 3), buf::NT), buf::NT, 0, st>>>(obss, acts, nexts, rews, terms, pens, S, A,
                                                                                          pos, m_dev, m_cap, packed);
}
// scratch: double[2 * MB_STATS_BLOCKS] partials followed by one unsigned ticket (zero-initialised once by the caller)
void mb_rollout_stats_launch(const float* rews, const unsigned char* terms, long long n, double* partial, unsigned int* ticket,
                             double* stats, cudaStream_t st) {
  int nb = (int)((n + 4095) / 4096); if (nb < 1) nb = 1; if (nb > MB_STATS_BLOCKS) nb = MB_STATS_BLOCKS;
  buf::rollout_stats_kernel<<<nb, buf::SB, 0, st>>>(rews, terms, n, partial, ticket, stats);
}

void mb_model_eval_init_launch(long long* row_ids, unsigned long long row0, int B, double* ret, double* ret_disc, int* length,
                               int* counts, cudaStream_t st) {
  buf::model_eval_init_kernel<<<grid_for(B, buf::NT), buf::NT, 0, st>>>(row_ids, row0, B, ret, ret_disc, length, counts);
}
void mb_model_eval_accumulate_launch(const float* reward, const long long* row_ids, unsigned long long row0, const int* n_dev,
                                     long long n_cap, int t, double disc, double* ret, double* ret_disc, int* length, cudaStream_t st) {
  buf::model_eval_accumulate_kernel<<<grid_for(n_cap, buf::NT), buf::NT, 0, st>>>(reward, row_ids, row0, n_dev, t, disc, ret,
                                                                                 ret_disc, length);
}

void mb_sample_rows_launch(const mobody_sample_job* jobs, int njobs, int rw, cudaStream_t st) {
  buf::SampleJobs j{};
  long long maxn = 0;
  for (int b = 0; b < njobs; ++b) {
    j.rows[b] = reinterpret_cast<const float4*>(jobs[b].rows); j.out[b] = reinterpret_cast<float4*>(jobs[b].out);
    j.n[b] = jobs[b].n; j.size[b] = jobs[b].size; j.draw[b] = jobs[b].draw; j.seed[b] = jobs[b].seed;
    if (jobs[b].n > maxn) maxn = jobs[b].n;
  }
  if (maxn <= 0) return;
  buf::sample_rows_kernel<<<dim3(grid_for(maxn * (rw / 4), buf::NT), njobs), buf::NT, 0, st>>>(j, rw / 4);
}
