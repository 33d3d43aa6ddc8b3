// Steady-state MOBODY.train step as fused fp32 forward/backward MLP kernels.
//
// Replaces, on packed batch rows [N, RW] = [state | action | next_state | reward | not_done | pad]
// (rows ordered src, tar, fake; the first n_true rows are the "true" src+tar rows):
//   update_q_functions + q backward          algo/offline_offline/mobody.py:189-208, 546-548
//   update_target (Polyak, every step)        :183-187, 552
//   update_policy + bc_loss + pi backward     :314-345, 246-276, 571-573
//   torch.optim.Adam (lr, betas .9/.999, eps 1e-8) :127-131
// Math: SURVEY.md Appendix A.3.  All networks are MLPNetwork (Linear-ReLU-Linear-ReLU-Linear, :35-48).
// The reference's other update branches select phases and loss terms of the same chain (mobody_train_step_ex):
//   advantage=1: the value step first (update_v_function, :210-242: expectile loss on min Q'(s, a) - V(s), Adam on
//                ValueFunc), TD target r + nd gamma V(s') with the updated V, BC weights exp(3 (min Q(s_t, a_t) - V(s_t)))
//   scale_Q=0:   p_w = 1 (update_policy_1, :278-310)         q_weighted=0: BC weights 1 (:262-263)
//
// A CTA owns a tile of 64 rows; hidden activations stay in shared memory for the whole
// forward + backward-data chain of that tile (simt_layers.cuh).  Only what the weight-gradient
// GEMMs need (H1, H2, dH1, dH2 per network) goes to HBM.  Weight gradients are row-reductions done
// by a tiled GEMM over the whole batch (deterministic, no atomics), optionally split over row
// ranges whose partials are summed inside the fused Adam(+Polyak) kernel.
#include "simt_layers.cuh"
#include "philox.cuh"
#include "umma_gemm.cuh"
#include "../../include/mobody_b200.h"
#include <math.h>

namespace trn {
using namespace simt;

// The chains of one update are independent per network until they meet (TD target, min over the twin critics), so
// each phase runs the networks side by side: blockIdx.y selects the role, blockIdx.x the row tile.
struct CriticArgs {
  const float* X; int N, S, A, rw;
  MlpPtrs pi, q[2], qt[2];
  float gamma, max_action;
  float* a2;           // pi(s'), [N][A]                                  (phase 1 role 0 -> phase 2)
  float* qk[2];        // Q_k(s, a), [N]                                  (phase 1 roles 1, 2 -> phase 3)
  float* qtk[2];       // Q'_k(s', pi(s')), [N]                           (phase 2 -> phase 3)
  float* Hq[2][2];     // [net][layer] relu activations of Q_k(s,a), [N][256]
  float* Dq[2][2];     // [net][layer] dLoss/d(pre-activation), [N][256]
  float* d3[2];        // [net] dLoss/dq_k, [N]
  float* part;         // [n_tiles][4]: sum (q1-y)^2, sum (q2-y)^2, sum q1, sum q2
  float* Hp[2];        // relu activations of pi(s), [N][256]      (phase 1 role 3: the actor's forward does not depend on
  float* api;          // pi(s), [N][A]                             the critic update, so it rides along with it)
  // advantage=1 only (vn == nullptr otherwise): the UPDATED value function replaces pi(s') and the target critics --
  // phase 1 role 0 = V(s') (the TD target), role 4 = V(s_t) on the n_true true rows (the actor's advantage weights)
  MlpPtrs v; float* vn; float* vh; int n_true;
};

struct ActorArgs {
  const float* X; int N, n_true, S, A, rw;
  MlpPtrs pi, q[2];
  float max_action;
  float* Hp[2];        // relu activations of pi(s), [N][256]
  float* api;          // pi(s), [N][A]
  float* qv[2];        // Q_k(s, pi(s)), [N]
  float* gak[2];       // d Q_k / d action, [N][A]
  float* qh[2];        // Q_k(s_t, a_t), [n_true]
  // the last CTA to finish reduces the batch scalars the backward needs (fixed order; see actor_finish)
  const float* part; int ntiles_c;   // critic tile partials [ntiles_c][4]
  float weight;
  float* out;          // scalars [16]
  int* counter;        // zeroed by the critic's Adam launch of the same update
  // update branches: scale_q = 0 -> p_w = 1; branch = 1 (any non-default flag) -> q_hat on all n_qh = N rows and out[14];
  // part_v (advantage=1): the value step's tile partials [ntiles_c][4] -> out[11..13]
  int scale_q, branch, n_qh; const float* part_v;
};

template <int TMv>
__device__ __forceinline__ void store_tile(const float* __restrict__ Xs, float* __restrict__ g, int row0, int rows) {
  // swizzled [TM][256] smem tile -> global [N][256] (plain), 128-bit stores
  for (int i = threadIdx.x; i < rows * (H / 4); i += NT) {
    int r = i / (H / 4), c = i - r * (H / 4);
    reinterpret_cast<float4*>(g + (size_t)(row0 + r) * H)[c] = *reinterpret_cast<const float4*>(Xs + r * H + swz(r, 4 * c));
  }
}
template <int TMv>
__device__ __forceinline__ void load_tile(float* __restrict__ Xs, const float* __restrict__ g, int row0, int rows) {
  for (int i = threadIdx.x; i < TMv * (H / 4); i += NT) {
    int r = i / (H / 4), c = i - r * (H / 4);
    *reinterpret_cast<float4*>(Xs + r * H + swz(r, 4 * c)) = r < rows ? reinterpret_cast<const float4*>(g + (size_t)(row0 + r) * H)[c]
                                                                      : make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// out[r] = X1[r,:] . w + b   (last Linear of a Q network, one output)
template <int TMv>
__device__ __forceinline__ void q_head(const float* __restrict__ X1, const float* __restrict__ w, const float* __restrict__ b,
                                       float* __restrict__ out) {
  constexpr int TPR = NT / TMv;                               // threads per row (4 for 64 rows, 16 for 16 rows)
  const int r = threadIdx.x / TPR, q = threadIdx.x % TPR;
  const float* x = X1 + r * H;
  float s = 0.f;
  for (int k = q; k < H; k += TPR) s = fmaf(x[swz(r, k)], __ldg(w + k), s);
#pragma unroll
  for (int o = 1; o < TPR; o <<= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (q == 0) out[r] = s + __ldg(b);
  __syncthreads();
}

// relu backward of the last Linear (one output): X1[r][n] = X1[r][n] > 0 ? g[r] * w[n] : 0   (in place)
template <int TMv>
__device__ __forceinline__ void head_backward(float* __restrict__ X1, const float* __restrict__ w, const float* __restrict__ g) {
  for (int i = threadIdx.x; i < TMv * H; i += NT) {
    int r = i >> 8, n = swz(r, i & 255);                        // i is a physical position; n its logical column
    X1[i] = X1[i] > 0.f ? g[r] * __ldg(w + n) : 0.f;
  }
  __syncthreads();
}

// ---- critic phase 1: role 0 = pi(s') (:190), roles 1, 2 = Q_k(s, a) forward with stored activations (:196),
//      role 3 = pi(s) with stored activations for the actor update that follows (:315; same policy parameters) ----
template <int RPT>
__global__ void __launch_bounds__(NT, RPT == 4 ? 2 : 1) critic_fwd_kernel(CriticArgs a) {
  mb_pdl_begin();
  constexpr int TM = 8 * RPT;
  extern __shared__ __align__(16) float sm[];
  const int S = a.S, A = a.A, ldi = rup16(S + A);
  float* X0 = sm; float* X1 = X0 + TM * H; float* in_s = X1 + TM * H; float* qa = in_s + TM * ldi;
  const int tid = threadIdx.x, row0 = blockIdx.x * TM, rows = min(TM, a.N - row0), role = blockIdx.y;
  if (role == 4 && row0 >= a.n_true) return;
  for (int i = tid; i < TM * ldi; i += NT) {
    const int r = i / ldi, j = i - r * ldi;
    const float* x = a.X + (size_t)(row0 + r) * a.rw;
    in_s[i] = role == 0 ? ((r < rows && j < S) ? x[S + A + j] : 0.f)                  // [s', 0]
            : (role == 3 || role == 4) ? ((r < rows && j < S) ? x[j] : 0.f)            // [s, 0]
                                       : ((r < rows && j < S + A) ? x[j] : 0.f);       // [s, a, 0]
  }
  __syncthreads();
  if (a.vn && (role == 0 || role == 4)) {                     // V(s') / V(s_t) through the updated value function
    big_layer_mma<true, RPT>(in_s, ldi, S, a.v.w[0], a.v.b[0], X0, ACT_RELU);
    big_layer_mma<true, RPT, true>(X0, H, H, a.v.w[1], a.v.b[1], X1, ACT_RELU);
    q_head<TM>(X1, a.v.w[2], a.v.b[2], qa);
    if (tid < rows && (role == 0 || row0 + tid < a.n_true)) (role == 0 ? a.vn : a.vh)[row0 + tid] = qa[tid];
  } else if (role == 3) {
    big_layer_mma<true, RPT>(in_s, ldi, S, a.pi.w[0], a.pi.b[0], X0, ACT_RELU);
    store_tile<TM>(X0, a.Hp[0], row0, rows);
    big_layer_mma<true, RPT, true>(X0, H, H, a.pi.w[1], a.pi.b[1], X1, ACT_RELU);
    store_tile<TM>(X1, a.Hp[1], row0, rows);
    small_layer<true, RPT, true>(X1, H, H, a.pi.w[2], H, a.pi.b[2], A, in_s, ldi, ACT_TANH, a.max_action);
    for (int i = tid; i < rows * A; i += NT) { const int r = i / A, j = i - r * A; a.api[(size_t)(row0 + r) * A + j] = in_s[r * ldi + j]; }
  } else if (role == 0) {
    big_layer_mma<true, RPT>(in_s, ldi, S, a.pi.w[0], a.pi.b[0], X0, ACT_RELU);
    big_layer_mma<true, RPT, true>(X0, H, H, a.pi.w[1], a.pi.b[1], X1, ACT_RELU);
    small_layer<true, RPT, true>(X1, H, H, a.pi.w[2], H, a.pi.b[2], A, in_s, ldi, ACT_TANH, a.max_action);
    for (int i = tid; i < rows * A; i += NT) { const int r = i / A, j = i - r * A; a.a2[(size_t)(row0 + r) * A + j] = in_s[r * ldi + j]; }
  } else {
    const int k = role - 1;
    big_layer_mma<true, RPT>(in_s, ldi, S + A, a.q[k].w[0], a.q[k].b[0], X0, ACT_RELU);
    store_tile<TM>(X0, a.Hq[k][0], row0, rows);
    big_layer_mma<true, RPT, true>(X0, H, H, a.q[k].w[1], a.q[k].b[1], X1, ACT_RELU);
    store_tile<TM>(X1, a.Hq[k][1], row0, rows);
    q_head<TM>(X1, a.q[k].w[2], a.q[k].b[2], qa);
    if (tid < rows) a.qk[k][row0 + tid] = qa[tid];
  }
}

// ---- critic phase 2: role k = Q'_k(s', pi(s')) (no grad, :191-193) ----
template <int RPT>
__global__ void __launch_bounds__(NT, RPT == 4 ? 2 : 1) critic_tgt_kernel(CriticArgs a) {
  mb_pdl_begin();
  constexpr int TM = 8 * RPT;
  extern __shared__ __align__(16) float sm[];
  const int S = a.S, A = a.A, ldi = rup16(S + A);
  float* X0 = sm; float* X1 = X0 + TM * H; float* in_s = X1 + TM * H; float* qa = in_s + TM * ldi;
  const int tid = threadIdx.x, row0 = blockIdx.x * TM, rows = min(TM, a.N - row0), k = blockIdx.y;
  for (int i = tid; i < TM * ldi; i += NT) {
    const int r = i / ldi, j = i - r * ldi;
    float v = 0.f;
    if (r < rows) {
      if (j < S) v = a.X[(size_t)(row0 + r) * a.rw + S + A + j];
      else if (j < S + A) v = a.a2[(size_t)(row0 + r) * A + (j - S)];
    }
    in_s[i] = v;
  }
  __syncthreads();
  big_layer_mma<true, RPT>(in_s, ldi, S + A, a.qt[k].w[0], a.qt[k].b[0], X0, ACT_RELU);
  big_layer_mma<true, RPT, true>(X0, H, H, a.qt[k].w[1], a.qt[k].b[1], X1, ACT_RELU);
  q_head<TM>(X1, a.qt[k].w[2], a.qt[k].b[2], qa);
  if (tid < rows) a.qtk[k][row0 + tid] = qa[tid];
}

// ---- critic phase 3: role k = TD target, mse gradient of Q_k and backward to the pre-activations (:194-207) ----
template <int RPT>
__global__ void __launch_bounds__(NT, RPT == 4 ? 2 : 1) critic_bwd_kernel(CriticArgs a) {
  mb_pdl_begin();
  constexpr int TM = 8 * RPT;
  extern __shared__ __align__(16) float sm[];
  const int S = a.S, A = a.A;
  float* X0 = sm; float* X1 = X0 + TM * H; float* g3 = X1 + TM * H; float* redbuf = g3 + TM;   // redbuf[4]
  const int tid = threadIdx.x, row0 = blockIdx.x * TM, rows = min(TM, a.N - row0), k = blockIdx.y;
  load_tile<TM>(X0, a.Hq[k][0], row0, rows);
  load_tile<TM>(X1, a.Hq[k][1], row0, rows);
  float l0 = 0.f, l1 = 0.f;
  if (tid < TM) {
    float d = 0.f, q = 0.f;
    if (tid < rows) {
      const float* x = a.X + (size_t)(row0 + tid) * a.rw;
      const float boot = a.vn ? a.vn[row0 + tid] : fminf(a.qtk[0][row0 + tid], a.qtk[1][row0 + tid]);
      const float y = x[2 * S + A] + x[2 * S + A + 1] * a.gamma * boot;
      q = a.qk[k][row0 + tid];
      d = q - y;
      a.d3[k][row0 + tid] = 2.0f * d / (float)a.N;
    }
    g3[tid] = 2.0f * d / (float)a.N;                          // d mean((q-y)^2) / dq
    l0 = d * d; l1 = q;
  }
  __syncthreads();
  head_backward<TM>(X1, a.q[k].w[2], g3);                     // dH2 (masked)
  store_tile<TM>(X1, a.Dq[k][1], row0, rows);
  big_layer_mma<false, RPT, true>(X1, H, H, a.q[k].w[1], nullptr, X0, ACT_MASK);   // dH1 = (dH2 W2) * 1[H1>0], in place on H1
  store_tile<TM>(X0, a.Dq[k][0], row0, rows);
  // tile partial sums in a fixed order (deterministic): threads 0..TM-1 hold one row each
  if (tid < 4) redbuf[tid] = 0.f;
  __syncthreads();
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    float v = tid < TM ? (c == 0 ? l0 : l1) : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (tid < TM && (tid & 31) == 0) redbuf[(tid >> 5) * 2 + c] = v;
  }
  __syncthreads();
  if (tid < 2) a.part[blockIdx.x * 4 + 2 * tid + k] = redbuf[tid] + redbuf[2 + tid];     // [0..1] = sq err of Q1, Q2; [2..3] = sum q
}

// Batch scalars of the actor loss that the backward needs, reduced by the LAST CTA of actor_q_kernel to finish (every CTA
// bumps a counter after its results are globally visible; no float atomics, so the sums have a fixed order):
//   out[0] = q loss   out[1] = mean q1   (critic tile partials)      out[4] = mean q(s, pi(s))   out[5] = mean|q(s, pi(s))|
//   out[9] = p_w = weight / mean|q|   out[10] = mean|q_hat|          (out[2, 3, 6..8] come from policy_bwd_kernel)
__device__ float block_sum(float v, float* sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  float t = 0.f;
  if (w == 0) {
    t = lane < (int)(blockDim.x >> 5) ? sh[lane] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) sh[32] = t;
  }
  __syncthreads();
  return sh[32];
}
__device__ float block_minmax(float v, float* sh, bool is_max) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { float u = __shfl_xor_sync(0xffffffffu, v, o); v = is_max ? fmaxf(v, u) : fminf(v, u); }
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  if (w == 0) {
    float t = lane < (int)(blockDim.x >> 5) ? sh[lane] : sh[0];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { float u = __shfl_xor_sync(0xffffffffu, t, o); t = is_max ? fmaxf(t, u) : fminf(t, u); }
    if (lane == 0) sh[32] = t;
  }
  __syncthreads();
  return sh[32];
}
__device__ void actor_reduce(const ActorArgs& a, float* sh) {
  float s_abs = 0.f, s_q = 0.f, s_h = 0.f;
  for (int i = threadIdx.x; i < a.N; i += blockDim.x) { const float q = fminf(__ldcg(a.qv[0] + i), __ldcg(a.qv[1] + i)); s_abs += fabsf(q); s_q += q; }
  for (int i = threadIdx.x; i < a.n_true; i += blockDim.x) s_h += fabsf(fminf(__ldcg(a.qh[0] + i), __ldcg(a.qh[1] + i)));
  const float mean_abs = block_sum(s_abs, sh) / (float)a.N;                 // mobody.py:318
  const float mean_q = block_sum(s_q, sh) / (float)a.N;
  const float mean_h = block_sum(s_h, sh) / (float)a.n_true;                // :252
  float l = 0.f, q1s = 0.f;
  for (int t = threadIdx.x; t < a.ntiles_c; t += blockDim.x) { l += a.part[t * 4] + a.part[t * 4 + 1]; q1s += a.part[t * 4 + 2]; }
  l = block_sum(l, sh); q1s = block_sum(q1s, sh);
  if (threadIdx.x == 0) {
    a.out[0] = l / (float)a.N; a.out[1] = q1s / (float)a.N;                 // mse(q1,y) + mse(q2,y) (:207)
    a.out[4] = mean_q; a.out[5] = mean_abs; a.out[9] = a.scale_q ? a.weight / mean_abs : 1.0f; a.out[10] = mean_h;
  }
  if (a.branch) {                                                           // train/q_behavior: mean min Q(s, a), all rows
    float s_b = 0.f;
    for (int i = threadIdx.x; i < a.N; i += blockDim.x) s_b += fminf(__ldcg(a.qh[0] + i), __ldcg(a.qh[1] + i));
    s_b = block_sum(s_b, sh);
    if (threadIdx.x == 0) a.out[14] = s_b / (float)a.N;
  }
  if (a.part_v) {                                                           // value step: v_loss, mean adv, mean V(s)
    float lv = 0.f, sa = 0.f, sv = 0.f;
    for (int t = threadIdx.x; t < a.ntiles_c; t += blockDim.x) { lv += a.part_v[t * 4]; sa += a.part_v[t * 4 + 1]; sv += a.part_v[t * 4 + 2]; }
    lv = block_sum(lv, sh); sa = block_sum(sa, sh); sv = block_sum(sv, sh);
    if (threadIdx.x == 0) { a.out[11] = lv / (float)a.N; a.out[12] = sa / (float)a.N; a.out[13] = sv / (float)a.N; }
  }
}
__device__ void actor_finish(const ActorArgs& a, float* sh) {
  __shared__ int last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(a.counter, 1) == (int)(gridDim.x * gridDim.y) - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  actor_reduce(a, sh);
}

// ---- actor: roles 0, 1 = Q_k(s, pi(s)) and d Q_k / d action with Q frozen (:316-317, 555-556);
//      roles 2, 3 = q_hat_k = Q_k(s_t, a_t) on the true rows (no grad, :249-251).  pi(s) was computed next to the critic. ----
template <int RPT>
__global__ void __launch_bounds__(NT, RPT == 4 ? 2 : 1) actor_q_kernel(ActorArgs a) {
  mb_pdl_begin();
  constexpr int TM = 8 * RPT;
  extern __shared__ __align__(16) float sm[];
  const int S = a.S, A = a.A, ldi = rup16(S + A);
  float* X0 = sm; float* X1 = X0 + TM * H; float* sap_s = X1 + TM * H;
  float* qa = sap_s + TM * ldi; float* ones = qa + TM; float* gk = ones + TM;      // gk [TM][A]
  const int tid = threadIdx.x, row0 = blockIdx.x * TM, rows = min(TM, a.N - row0), k = blockIdx.y & 1;
  const bool qhat = blockIdx.y >= 2;
  if (qhat && row0 >= a.n_qh) { actor_finish(a, sm); return; }
  for (int i = tid; i < TM * ldi; i += NT) {
    const int r = i / ldi, j = i - r * ldi;
    float v = 0.f;
    if (r < rows) {
      if (j < S || (qhat && j < S + A)) v = a.X[(size_t)(row0 + r) * a.rw + j];          // [s, a_t] for q_hat
      else if (j < S + A) v = a.api[(size_t)(row0 + r) * A + (j - S)];                    // [s, pi(s)]
    }
    sap_s[i] = v;
  }
  if (tid < TM) ones[tid] = 1.0f;
  __syncthreads();
  if (qhat) {
    big_layer_mma<true, RPT>(sap_s, ldi, S + A, a.q[k].w[0], a.q[k].b[0], X0, ACT_RELU);
    big_layer_mma<true, RPT, true>(X0, H, H, a.q[k].w[1], a.q[k].b[1], X1, ACT_RELU);
    q_head<TM>(X1, a.q[k].w[2], a.q[k].b[2], qa);
    if (tid < rows && row0 + tid < a.n_qh) a.qh[k][row0 + tid] = qa[tid];
    actor_finish(a, sm);
    return;
  }
  big_layer_mma<true, RPT>(sap_s, ldi, S + A, a.q[k].w[0], a.q[k].b[0], X0, ACT_RELU);
  big_layer_mma<true, RPT, true>(X0, H, H, a.q[k].w[1], a.q[k].b[1], X1, ACT_RELU);
  q_head<TM>(X1, a.q[k].w[2], a.q[k].b[2], qa);
  head_backward<TM>(X1, a.q[k].w[2], ones);
  big_layer_mma<false, RPT, true>(X1, H, H, a.q[k].w[1], nullptr, X0, ACT_MASK);
  // d q / d a_j = sum_n dH1[n] * W1[n][S+j]
  small_layer<false, RPT, true>(X0, H, H, a.q[k].w[0] + S, S + A, nullptr, A, gk, A, ACT_NONE, 1.f);
  for (int i = tid; i < rows * A; i += NT) a.gak[k][(size_t)row0 * A + i] = gk[i];
  if (tid < rows) a.qv[k][row0 + tid] = qa[tid];
  actor_finish(a, sm);
}

// Policy backward.  Prologue = d loss / d (pre-tanh policy output) of the tile's rows (mobody.py:321-330: the
// -p_w mean(min Q) term through dQ/da of the smaller twin, plus the Q-weighted BC term on the true rows), written to
// d3p for the weight gradient of the last layer; then dH2 = (d3p W3) * 1[H2>0], dH1 = (dH2 W2) * 1[H1>0].
// Logging scalars (exp-advantage weight statistics, BC loss, policy loss) are tile partials reduced by the last CTA:
//   out[2] = policy loss   out[3] = bc loss   out[6..8] = mean / min / max of the exp-advantage weights
struct PolicyBwdArgs {
  int N, n_true, S, A, rw; MlpPtrs pi; const float* Hp[2]; float* Dp[2];
  const float* gak[2]; const float* qv[2]; const float* qh[2]; const float* api; const float* X;
  float bc_coef, max_action;
  float* d3p;          // [N][A]
  float* part;         // [ntiles][4]: sum w, min w, max w, sum w * |pi(s) - a|^2
  float* out;          // scalars [16]; [9] = p_w and [10] = mean|q_hat| were written by actor_q_kernel
  int* counter;
  const float* vh;     // advantage=1: V(s_t) of the updated value function, [n_true]; nullptr: q_hat / mean|q_hat|
  int q_weighted;      // 0: plain BC (weights 1)
};
// exp-advantage weight of true row r (:252-263)
__device__ __forceinline__ float bc_weight(const PolicyBwdArgs& a, int r, float mean_h) {
  if (!a.q_weighted) return 1.0f;
  const float qb = fminf(a.qh[0][r], a.qh[1][r]);
  return fminf(expf(3.0f * (a.vh ? qb - a.vh[r] : qb / mean_h)), 100.0f);
}
template <int RPT>
__global__ void __launch_bounds__(NT, RPT == 4 ? 2 : 1) policy_bwd_kernel(PolicyBwdArgs a) {
  mb_pdl_begin();
  constexpr int TM = 8 * RPT;
  extern __shared__ __align__(16) float sm[];
  float* X0 = sm; float* X1 = X0 + TM * H; float* Wst = X1 + TM * H;
  const int lda = rup16(a.A);
  float* d3 = Wst;                                       // [TM][lda]
  float* wrow = d3 + TM * lda;                           // [TM] exp-advantage weight of a true row
  float* red = wrow + TM;                                // [40]
  const int tid = threadIdx.x, row0 = blockIdx.x * TM, rows = min(TM, a.N - row0);
  const float pw = a.out[9], mean_h = a.out[10];
  float w_s = 0.f, w_mn = 3.4e38f, w_mx = -3.4e38f, w_e = 0.f;
  if (tid < TM) {
    const int r = row0 + tid;
    float w = 0.f;
    if (tid < rows && r < a.n_true) {
      w = bc_weight(a, r, mean_h);                                                         // :252-263
      const float* x = a.X + (size_t)r * a.rw + a.S;
      float e = 0.f;
      for (int j = 0; j < a.A; ++j) { const float d = a.api[(size_t)r * a.A + j] - x[j]; e += d * d; }
      w_s = w; w_mn = w; w_mx = w; w_e = w * e;
    }
    wrow[tid] = w;
  }
  __syncthreads();
  for (int i = tid; i < TM * lda; i += NT) {
    const int rl = i / lda, j = i - rl * lda, r = row0 + rl;
    float g3 = 0.f;
    if (rl < rows && j < a.A) {
      const size_t e = (size_t)r * a.A + j;
      const float ap = a.api[e];
      const float ga = a.qv[0][r] <= a.qv[1][r] ? a.gak[0][e] : a.gak[1][e];   // torch.min(q1, q2): gradient follows the smaller one
      float g = -pw / (float)a.N * ga;                                          // d [pw * mean(-q)] / d a
      if (r < a.n_true) g += a.bc_coef * wrow[rl] * 2.0f * (ap - a.X[(size_t)r * a.rw + a.S + j]) / (float)((size_t)a.n_true * a.A);
      const float t = ap / a.max_action;                                        // tanh(u)
      g3 = g * a.max_action * (1.0f - t * t);
      a.d3p[e] = g3;
    }
    d3[i] = g3;
  }
  load_tile<TM>(X1, a.Hp[1], row0, rows);
  load_tile<TM>(X0, a.Hp[0], row0, rows);
  // tile partials of the logging scalars (rows of a tile sit in the first TM threads: warps 0 .. TM/32 - 1, or half a warp)
  w_s = block_sum(w_s, red); w_e = block_sum(w_e, red);
  w_mn = block_minmax(w_mn, red, false); w_mx = block_minmax(w_mx, red, true);
  if (tid == 0) { float* p = a.part + (size_t)blockIdx.x * 4; p[0] = w_s; p[1] = w_mn; p[2] = w_mx; p[3] = w_e; }
  __syncthreads();
  big_layer_mma<false, RPT>(d3, lda, a.A, a.pi.w[2], nullptr, X1, ACT_MASK);    // W3 is [A][256]: dH2[r][i] = sum_j d3[r][j] W3[j][i]
  store_tile<TM>(X1, a.Dp[1], row0, rows);
  big_layer_mma<false, RPT, true>(X1, H, H, a.pi.w[1], nullptr, X0, ACT_MASK);
  store_tile<TM>(X0, a.Dp[0], row0, rows);
  // last CTA: logging scalars in tile order
  __shared__ int last;
  __threadfence();
  __syncthreads();
  if (tid == 0) last = atomicAdd(a.counter, 1) == (int)gridDim.x - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  float s_w = 0.f, s_e = 0.f, mn = 3.4e38f, mx = -3.4e38f;
  for (int t = tid; t < (int)gridDim.x; t += NT) {
    const float* p = a.part + (size_t)t * 4;
    s_w += __ldcg(p); mn = fminf(mn, __ldcg(p + 1)); mx = fmaxf(mx, __ldcg(p + 2)); s_e += __ldcg(p + 3);
  }
  s_w = block_sum(s_w, red); s_e = block_sum(s_e, red);
  mn = block_minmax(mn, red, false); mx = block_minmax(mx, red, true);
  if (tid == 0) {
    const float bc = s_e / (float)((size_t)a.n_true * a.A);                   // mean over rows AND action dims (:271)
    a.out[2] = pw * (-a.out[4]) + a.bc_coef * bc;                             // :321, 330
    a.out[3] = bc; a.out[6] = s_w / (float)a.n_true; a.out[7] = mn; a.out[8] = mx;
  }
}

// ---------------- weight gradients: dW[o][i] = sum_r D[r][o] X[r][i], db[o] = sum_r D[r][o] ----------------
// One launch covers every Linear of a phase (job = layer of a network), row range split `nsplit` ways; the partial sums
// of the splits are added in a fixed order by adam_kernel, so the result does not depend on the schedule.
// Layers with O a multiple of 128 (the 256-wide ones: > 99 % of the work) run on warp-level 3xTF32 tensor-core MMA
// (wgrad_mma_tile); the one- / A-output heads run on the FMA pipe (wgrad_narrow_tile).
struct WgradJob { const float* D; int ldD; const float* X; int ldX; float* dW; float* db; int O, I; };
struct WgradArgs { WgradJob job[6]; int njobs, N, nsplit; };
constexpr int WM_O = 128, WM_I = 64, WM_R = 32, WM_PD = WM_O + 8, WM_PX = WM_I + 8;   // pitches = 8 mod 32 words: conflict-free fragments
constexpr size_t WGRAD_SMEM = (size_t)2 * 2 * WM_R * (WM_PD + WM_PX) * sizeof(uint32_t);   // two stages of {hi, lo} x {D, X} planes (106 496 B)
__host__ __device__ inline bool wgrad_use_mma(int O) { return O % WM_O == 0; }
__host__ __device__ inline int wgrad_tiles(int O, int I) {
  return wgrad_use_mma(O) ? (O / WM_O) * ((I + WM_I - 1) / WM_I) : ((O + 7) / 8) * ((I + 255) / 256);
}

// Heads with few outputs (the Q head: O = 1, the policy head: O = A, the classifier head: O = 2): a tile is 8 outputs x
// 256 input columns; the eight warps take the rows of the split round-robin (a lane owns 2 x 4 columns: coalesced 128-bit
// loads of X, broadcast loads of D) and their partial sums are added through shared memory in warp order.
constexpr int WN_O = 8, WN_I = 256;
static_assert(WGRAD_SMEM >= (size_t)(8 * WN_O * WN_I + 8 * WN_O) * sizeof(float), "narrow-head reduction buffer");
__device__ __forceinline__ void wgrad_narrow_tile(const WgradJob& jb, int tile, int split, int rbeg, int rend, float* red) {
  const int tiles_i = (jb.I + WN_I - 1) / WN_I;
  const int o0 = (tile / tiles_i) * WN_O, i0 = (tile % tiles_i) * WN_I;
  const int no = min(WN_O, jb.O - o0);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int c0 = i0 + 4 * lane, c1 = c0 + 128;
  const bool v0 = c0 < jb.I, v1 = c1 < jb.I;                  // I and ldX are multiples of 4 (checked at launch)
  float acc[WN_O][8], bs[WN_O];
#pragma unroll
  for (int u = 0; u < WN_O; ++u) {
    bs[u] = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[u][j] = 0.f;
  }
#pragma unroll 2
  for (int r = rbeg + warp; r < rend; r += 8) {
    const float* x = jb.X + (size_t)r * jb.ldX;
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 xa = v0 ? __ldg(reinterpret_cast<const float4*>(x + c0)) : z, xb = v1 ? __ldg(reinterpret_cast<const float4*>(x + c1)) : z;
    const float* d = jb.D + (size_t)r * jb.ldD + o0;
#pragma unroll
    for (int u = 0; u < WN_O; ++u) {
      const float dv = u < no ? __ldg(d + u) : 0.f;
      bs[u] += dv;
      acc[u][0] = fmaf(dv, xa.x, acc[u][0]); acc[u][1] = fmaf(dv, xa.y, acc[u][1]); acc[u][2] = fmaf(dv, xa.z, acc[u][2]); acc[u][3] = fmaf(dv, xa.w, acc[u][3]);
      acc[u][4] = fmaf(dv, xb.x, acc[u][4]); acc[u][5] = fmaf(dv, xb.y, acc[u][5]); acc[u][6] = fmaf(dv, xb.z, acc[u][6]); acc[u][7] = fmaf(dv, xb.w, acc[u][7]);
    }
  }
  float* redb = red + 8 * WN_O * WN_I;
#pragma unroll
  for (int u = 0; u < WN_O; ++u) {
    float* p = red + (size_t)(warp * WN_O + u) * WN_I + 4 * lane;
    *reinterpret_cast<float4*>(p) = make_float4(acc[u][0], acc[u][1], acc[u][2], acc[u][3]);
    *reinterpret_cast<float4*>(p + 128) = make_float4(acc[u][4], acc[u][5], acc[u][6], acc[u][7]);
    if (lane == 0) redb[warp * WN_O + u] = bs[u];
  }
  __syncthreads();
  const size_t poff = (size_t)split * jb.O * jb.I;
  for (int u = 0; u < no; ++u) {
    float sum = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) sum += red[(size_t)(w * WN_O + u) * WN_I + tid];
    if (i0 + tid < jb.I) jb.dW[poff + (size_t)(o0 + u) * jb.I + i0 + tid] = sum;
  }
  if (i0 == 0 && tid < no) {
    float sum = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) sum += redb[w * WN_O + tid];
    jb.db[(size_t)split * jb.O + o0 + tid] = sum;
  }
}

// 128 (o) x 64 (i) tile of one row split on mma.sync.m16n8k8 TF32 with both operands split hi + lo ("3xTF32":
// lo*hi + hi*lo + hi*hi, fp32-class accuracy).  D and X are [row][.] in memory, i.e. k-major for both operands: a chunk of
// 32 rows is loaded with 128-bit loads (next chunk in flight in registers while this one is multiplied), split ONCE
// while it is staged, and the fragments are read with 64- / 128-bit shared loads through permuted operand slots:
//   m-slot g, g+8 of a 16-row m-tile = output rows 2g, 2g+1 (one 64-bit load = one register pair of the A fragment).
// 8 warps = 4 (o) x 2 (i), warp tile 32 x 32 = 2 m-tiles x 4 n-tiles, 24 MMAs per 8 rows.
__device__ __forceinline__ void wgrad_mma_tile(const WgradJob& jb, int tile, int split, int rbeg, int rend, uint32_t* sm) {
  constexpr uint32_t STAGE_WORDS = 2 * WM_R * (WM_PD + WM_PX);     // one stage = {Dh, Dl, Xh, Xl}; two stages alternate
  const int tiles_i = (jb.I + WM_I - 1) / WM_I;
  const int o0 = (tile / tiles_i) * WM_O, i0 = (tile % tiles_i) * WM_I;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int wo = (warp >> 1) * 32, wi = (warp & 1) * 32;
  const int dc4 = tid & 31, dr = tid >> 5;          // D staging: columns 4 dc4 .. +3, rows dr + 8 j (j < 4)
  const int xc4 = tid & 15, xr = tid >> 4;          // X staging: columns 4 xc4 .. +3, rows xr + 16 j (j < 2)
  const bool xcol_ok = i0 + 4 * xc4 < ((jb.I + 3) & ~3);     // a row of X is readable up to roundup4(I) (<= ldX)
  float4 pd[4], px[2];
  auto fetch = [&](int r0) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = r0 + dr + 8 * j;
      pd[j] = r < rend ? __ldg(reinterpret_cast<const float4*>(jb.D + (size_t)r * jb.ldD + o0 + 4 * dc4)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int r = r0 + xr + 16 * j;
      px[j] = (r < rend && xcol_ok) ? __ldg(reinterpret_cast<const float4*>(jb.X + (size_t)r * jb.ldX + i0 + 4 * xc4)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto stage = [&](const float4& v, uint32_t* hp, uint32_t* lp) {
    uint4 h, l;
    simt::split_tf32(v.x, h.x, l.x); simt::split_tf32(v.y, h.y, l.y); simt::split_tf32(v.z, h.z, l.z); simt::split_tf32(v.w, h.w, l.w);
    *reinterpret_cast<uint4*>(hp) = h; *reinterpret_cast<uint4*>(lp) = l;
  };
  float acc[2][4][4], bsum[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int m = 0; m < 2; ++m)
#pragma unroll
    for (int n = 0; n < 4; ++n)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[m][n][j] = 0.f;
  auto stage_chunk = [&](uint32_t* base) {          // split the fetched chunk into the hi / lo planes of one stage
    uint32_t (*Dh)[WM_PD] = reinterpret_cast<uint32_t (*)[WM_PD]>(base);
    uint32_t (*Dl)[WM_PD] = Dh + WM_R;
    uint32_t (*Xh)[WM_PX] = reinterpret_cast<uint32_t (*)[WM_PX]>(base + 2 * WM_R * WM_PD);
    uint32_t (*Xl)[WM_PX] = Xh + WM_R;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      stage(pd[j], &Dh[dr + 8 * j][4 * dc4], &Dl[dr + 8 * j][4 * dc4]);
      bsum[0] += pd[j].x; bsum[1] += pd[j].y; bsum[2] += pd[j].z; bsum[3] += pd[j].w;
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) stage(px[j], &Xh[xr + 16 * j][4 * xc4], &Xl[xr + 16 * j][4 * xc4]);
  };
  // chunk c is multiplied out of stage c & 1 while chunk c + 1 is split into the other stage and chunk c + 2 is in
  // flight in registers: one barrier per chunk
  if (rbeg < rend) {
    fetch(rbeg);
    stage_chunk(sm);
    if (rbeg + WM_R < rend) fetch(rbeg + WM_R);
  }
  __syncthreads();
  int cur = 0;
  for (int r0 = rbeg; r0 < rend; r0 += WM_R, cur ^= 1) {
    const uint32_t* base = sm + cur * STAGE_WORDS;
    const uint32_t (*Dh)[WM_PD] = reinterpret_cast<const uint32_t (*)[WM_PD]>(base);
    const uint32_t (*Dl)[WM_PD] = Dh + WM_R;
    const uint32_t (*Xh)[WM_PX] = reinterpret_cast<const uint32_t (*)[WM_PX]>(base + 2 * WM_R * WM_PD);
    const uint32_t (*Xl)[WM_PX] = Xh + WM_R;
#pragma unroll
    for (int ks = 0; ks < WM_R / 8; ++ks) {
      const int k = ks * 8 + t;
      uint32_t bh[4][2], bl[4][2];                 // scalar loads: (b0, b1) of a tile land in adjacent registers, no moves
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        bh[nt][0] = Xh[k][wi + nt * 8 + g]; bh[nt][1] = Xh[k + 4][wi + nt * 8 + g];
        bl[nt][0] = Xl[k][wi + nt * 8 + g]; bl[nt][1] = Xl[k + 4][wi + nt * 8 + g];
      }
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        const int oc = wo + m * 16 + 2 * g;
        const uint2 h0 = *reinterpret_cast<const uint2*>(&Dh[k][oc]), h1 = *reinterpret_cast<const uint2*>(&Dh[k + 4][oc]);
        const uint2 l0 = *reinterpret_cast<const uint2*>(&Dl[k][oc]), l1 = *reinterpret_cast<const uint2*>(&Dl[k + 4][oc]);
        const uint32_t ah[4] = {h0.x, h0.y, h1.x, h1.y}, al[4] = {l0.x, l0.y, l1.x, l1.y};
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          simt::mma_tf32_1688(acc[m][nt], al, bh[nt][0], bh[nt][1]);
          simt::mma_tf32_1688(acc[m][nt], ah, bl[nt][0], bl[nt][1]);
          simt::mma_tf32_1688(acc[m][nt], ah, bh[nt][0], bh[nt][1]);
        }
      }
    }
    if (r0 + WM_R < rend) {
      stage_chunk(sm + (cur ^ 1) * STAGE_WORDS);    // last read as the multiplicand of chunk c - 1, before the previous barrier
      if (r0 + 2 * WM_R < rend) fetch(r0 + 2 * WM_R);
    }
    __syncthreads();
  }
  // C fragment: j = 0, 1 -> row 2g, columns 2t, 2t+1 of n-tile nt;  j = 2, 3 -> row 2g+1
  const size_t poff = (size_t)split * jb.O * jb.I;
#pragma unroll
  for (int m = 0; m < 2; ++m)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int o = o0 + wo + m * 16 + 2 * g + (j >> 1), i = i0 + wi + nt * 8 + 2 * t + (j & 1);
        if (i < jb.I) jb.dW[poff + (size_t)o * jb.I + i] = acc[m][nt][j];
      }
  if (i0 == 0) {                                     // bias gradient: column sums of D, eight row classes added in order
    float* red = reinterpret_cast<float*>(sm);
#pragma unroll
    for (int c = 0; c < 4; ++c) red[dr * WM_O + 4 * dc4 + c] = bsum[c];
    __syncthreads();
    if (tid < WM_O) {
      float b = 0.f;
#pragma unroll
      for (int q = 0; q < 8; ++q) b += red[q * WM_O + tid];
      jb.db[(size_t)split * jb.O + o0 + tid] = b;
    }
  }
}

__global__ void __launch_bounds__(256, 2) wgrad_kernel(WgradArgs a) {
  mb_pdl_begin();
  extern __shared__ __align__(16) uint32_t wg_sm[];
  const WgradJob jb = a.job[blockIdx.z];
  if ((int)blockIdx.x >= wgrad_tiles(jb.O, jb.I)) return;
  const int split = blockIdx.y;
  const long long chunks = (a.N + WM_R - 1) / WM_R;               // splits are whole 32-row chunks, spread evenly
  const int rbeg = (int)(chunks * split / a.nsplit) * WM_R, rend = min(a.N, (int)(chunks * (split + 1) / a.nsplit) * WM_R);
  if (wgrad_use_mma(jb.O)) wgrad_mma_tile(jb, blockIdx.x, split, rbeg, rend, wg_sm);
  else wgrad_narrow_tile(jb, blockIdx.x, split, rbeg, rend, reinterpret_cast<float*>(wg_sm));
}

// ---------------- fused Adam (+ Polyak target update) over a table of tensors ----------------
struct AdamJob { float* p; const float* g; float* m; float* v; float* tgt; int n; };
struct AdamArgs { AdamJob job[12]; int njobs, nsplit; float lr_over_bc1, inv_sqrt_bc2, b1, b2, eps, tau; int* zero2; };   // zero2: the actor phase's two "last CTA" counters
__global__ void adam_kernel(AdamArgs a) {
  mb_pdl_begin();
  if (a.zero2 && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < 2) a.zero2[threadIdx.x] = 0;
  const AdamJob jb = a.job[blockIdx.y];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < jb.n; i += gridDim.x * blockDim.x) {
    float g = 0.f;                                                          // fixed order over the row splits;
    int s = 0;                                                              // loads batched four at a time (L2 latency)
    for (; s + 4 <= a.nsplit; s += 4) {
      const float g0 = jb.g[(size_t)s * jb.n + i], g1 = jb.g[(size_t)(s + 1) * jb.n + i];
      const float g2 = jb.g[(size_t)(s + 2) * jb.n + i], g3 = jb.g[(size_t)(s + 3) * jb.n + i];
      g += g0; g += g1; g += g2; g += g3;
    }
    for (; s < a.nsplit; ++s) g += jb.g[(size_t)s * jb.n + i];
    const float m = a.b1 * jb.m[i] + (1.0f - a.b1) * g;
    const float v = a.b2 * jb.v[i] + (1.0f - a.b2) * g * g;
    jb.m[i] = m; jb.v[i] = v;
    const float denom = sqrtf(v) * a.inv_sqrt_bc2 + a.eps;
    const float p = jb.p[i] - a.lr_over_bc1 * (m / denom);
    jb.p[i] = p;
    if (jb.tgt) jb.tgt[i] = a.tau * p + (1.0f - a.tau) * jb.tgt[i];          // :183-187, uses the updated Q
  }
}

// ---------------- DARA domain classifier (mobody.py:11-33, 146-181, 364-378) ----------------
// Two MLPNetworks in -> 256 -> 256 -> 2: sas_classifier on [s, a, s'] and sa_classifier on [s, a], trained on
// noise-perturbed inputs with cross_entropy applied to the SOFTMAXED outputs (the reference's double softmax).
#define MB_STREAM_CLSN 0x636C736Eu
struct ClsArgs {
  const float* X; int N, S, A, rw;
  const int* label;
  const float* noise[2];     // [N][2S+A], [N][S+A] injected N(0,1) or nullptr -> Philox(seed, draw)
  float std; unsigned long long seed; unsigned int draw;
  MlpPtrs net[2];            // 0 = sas_classifier, 1 = sa_classifier
  float* Xn[2];              // noisy inputs [N][ld_k] (weight-gradient operand of layer 1)
  float* Hc[2][2];           // relu activations [N][256]
  float* Dc[2][2];           // dLoss/d(pre-activation) [N][256]
  float* d3[2];              // dLoss/d(logit) [N][2]
  float* part;               // [n_tiles][2] cross-entropy sums (sas, sa)
};

__device__ __forceinline__ void softmax2(float z0, float z1, float& p0, float& p1) {
  const float m = fmaxf(z0, z1), e0 = expf(z0 - m), e1 = expf(z1 - m), inv = 1.0f / (e0 + e1);
  p0 = e0 * inv; p1 = e1 * inv;
}

template <int RPT>
__global__ void __launch_bounds__(NT, RPT == 4 ? 2 : 1) classifier_kernel(ClsArgs a) {
  mb_pdl_begin();
  constexpr int TM = 8 * RPT;
  extern __shared__ __align__(16) float sm[];
  const int S = a.S, A = a.A;
  float* X0 = sm; float* X1 = X0 + TM * H;
  float* in_s = X1 + TM * H;                       // [TM][ld], ld <= rup16(2S+A)
  float* z_s = in_s + TM * rup16(2 * S + A);       // [TM][2] logits
  float* g_s = z_s + 2 * TM;                       // [TM][2] dLoss/dlogit
  float* redbuf = g_s + 2 * TM;                    // [8]
  const int tid = threadIdx.x, row0 = blockIdx.x * TM, rows = min(TM, a.N - row0);
  float lsum[2] = {0.f, 0.f};
  for (int k = 0; k < 2; ++k) {
    const int K = k == 0 ? 2 * S + A : S + A, ld = rup16(K);
    for (int i = tid; i < TM * ld; i += NT) {
      const int r = i / ld, j = i - r * ld;
      float v = 0.f;
      if (r < rows && j < K) {
        const size_t gr = (size_t)row0 + r;
        v = a.X[gr * a.rw + j];                                              // [s | a | s'] are the first 2S+A columns of a row
        if (a.std != 0.f) {
          float nz;
          if (a.noise[k]) nz = a.noise[k][gr * K + j];
          else nz = philox_normal1(philox4x32_10((uint32_t)gr, ((uint32_t)k << 16) | (uint32_t)(j >> 2), a.draw, 0u,
                                                 (uint32_t)a.seed, MB_STREAM_CLSN), j & 3);
          v += nz * a.std;                                                     // sas += randn_like(sas) * std (:24-25, 30-31)
        }
        a.Xn[k][gr * ld + j] = v;
      } else if (r < rows) a.Xn[k][((size_t)row0 + r) * ld + j] = 0.f;
      in_s[i] = v;
    }
    __syncthreads();
    big_layer_mma<true, RPT>(in_s, ld, K, a.net[k].w[0], a.net[k].b[0], X0, ACT_RELU);
    store_tile<TM>(X0, a.Hc[k][0], row0, rows);
    big_layer_mma<true, RPT, true>(X0, H, H, a.net[k].w[1], a.net[k].b[1], X1, ACT_RELU);
    store_tile<TM>(X1, a.Hc[k][1], row0, rows);
    small_layer<true, RPT, true>(X1, H, H, a.net[k].w[2], H, a.net[k].b[2], 2, z_s, 2, ACT_NONE, 1.f);
    if (tid < TM) {
      float g0 = 0.f, g1 = 0.f;
      if (tid < rows) {
        float p0, p1, q0, q1;
        softmax2(z_s[2 * tid], z_s[2 * tid + 1], p0, p1);                      // Softmax inside Classifier.forward (:26, 32)
        softmax2(p0, p1, q0, q1);                                              // F.cross_entropy softmaxes again (:170-171)
        const int y = a.label[row0 + tid];
        lsum[k] = -logf(y ? q1 : q0);
        const float invn = 1.0f / (float)a.N;
        const float dp0 = (q0 - (y == 0 ? 1.f : 0.f)) * invn, dp1 = (q1 - (y == 1 ? 1.f : 0.f)) * invn;   // dL/dp
        const float dot = dp0 * p0 + dp1 * p1;
        g0 = p0 * (dp0 - dot); g1 = p1 * (dp1 - dot);                          // through the inner softmax
        a.d3[k][(size_t)(row0 + tid) * 2] = g0; a.d3[k][(size_t)(row0 + tid) * 2 + 1] = g1;
      }
      g_s[2 * tid] = g0; g_s[2 * tid + 1] = g1;
    }
    __syncthreads();
    {   // relu backward of the 2-output head: dH2[r][n] = H2 > 0 ? g0 W3[0][n] + g1 W3[1][n] : 0
      const float* w3 = a.net[k].w[2];
      for (int i = tid; i < TM * H; i += NT) {
        const int r = i >> 8, n = swz(r, i & 255);
        X1[i] = X1[i] > 0.f ? g_s[2 * r] * __ldg(w3 + n) + g_s[2 * r + 1] * __ldg(w3 + H + n) : 0.f;
      }
      __syncthreads();
    }
    store_tile<TM>(X1, a.Dc[k][1], row0, rows);
    big_layer_mma<false, RPT, true>(X1, H, H, a.net[k].w[1], nullptr, X0, ACT_MASK);
    store_tile<TM>(X0, a.Dc[k][0], row0, rows);
    __syncthreads();
  }
  if (tid < 8) redbuf[tid] = 0.f;
  __syncthreads();
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    float v = tid < TM ? lsum[c] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (tid < TM && (tid & 31) == 0) redbuf[(tid >> 5) * 2 + c] = v;
  }
  __syncthreads();
  if (tid < 2) a.part[blockIdx.x * 2 + tid] = redbuf[tid] + redbuf[2 + tid] + redbuf[4 + tid] + redbuf[6 + tid];
}

__global__ void cls_scalar_kernel(const float* __restrict__ part, int ntiles, int N, float* __restrict__ out) {
  mb_pdl_begin();
  if (threadIdx.x < 2) {
    float s = 0.f;
    for (int t = 0; t < ntiles; ++t) s += part[t * 2 + threadIdx.x];
    out[1 - threadIdx.x] = s / (float)N;                                      // out[0] = loss_sa, out[1] = loss_sas
  }
}

// reward relabel (mobody.py:364-378): rows[i].reward += coef * clamp(log-ratio of the twice-softmaxed outputs, -10, 10)
struct RelabelArgs { float* X; long long n; int S, A, rw; MlpPtrs net[2]; float coef; float* pen_out; };
__global__ void __launch_bounds__(NT, 1) dara_relabel_kernel(RelabelArgs a) {
  mb_pdl_begin();
  constexpr int RPT = 8, TM = 64;
  extern __shared__ __align__(16) float sm[];
  const int S = a.S, A = a.A;
  float* X0 = sm; float* X1 = X0 + TM * H;
  float* in_s = X1 + TM * H;
  float* z_s = in_s + TM * rup16(2 * S + A);       // [2][TM][2]
  const int tid = threadIdx.x;
  for (long long row0 = (long long)blockIdx.x * TM; row0 < a.n; row0 += (long long)gridDim.x * TM) {
    const int rows = (int)min((long long)TM, a.n - row0);
    for (int k = 0; k < 2; ++k) {
      const int K = k == 0 ? 2 * S + A : S + A, ld = rup16(K);
      for (int i = tid; i < TM * ld; i += NT) {
        const int r = i / ld, j = i - r * ld;
        in_s[i] = (r < rows && j < K) ? a.X[(size_t)(row0 + r) * a.rw + j] : 0.f;
      }
      __syncthreads();
      big_layer_mma<true, RPT>(in_s, ld, K, a.net[k].w[0], a.net[k].b[0], X0, ACT_RELU);
      big_layer_mma<true, RPT, true>(X0, H, H, a.net[k].w[1], a.net[k].b[1], X1, ACT_RELU);
      small_layer<true, RPT, true>(X1, H, H, a.net[k].w[2], H, a.net[k].b[2], 2, z_s + k * 2 * TM, 2, ACT_NONE, 1.f);
    }
    if (tid < rows) {
      float lp[2][2];
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        float p0, p1, q0, q1;
        softmax2(z_s[k * 2 * TM + 2 * tid], z_s[k * 2 * TM + 2 * tid + 1], p0, p1);
        softmax2(p0, p1, q0, q1);
        lp[k][0] = logf(q0 + 1e-10f); lp[k][1] = logf(q1 + 1e-10f);
      }
      float pen = lp[0][1] - lp[1][1] - lp[0][0] + lp[1][0];                   // sas_lp[1] - sa_lp[1] - sas_lp[0] + sa_lp[0]
      pen = fminf(fmaxf(pen, -10.f), 10.f);
      a.X[(size_t)(row0 + tid) * a.rw + 2 * S + A] += a.coef * pen;
      if (a.pen_out) a.pen_out[row0 + tid] = pen;
    }
    __syncthreads();
  }
}

// ================= large-batch path: the update as a sequence of tcgen05 GEMM tiles (umma_gemm.cuh) =================
// Element-wise glue between the GEMMs (everything else of the math lives in GEMM epilogues).

// TD target, MSE gradient and the logging partials (mobody.py:189-207): one thread per row, 256-row blocks
struct TdArgs { const float* X; int N, S, A, rw; float gamma; const float* qk[2]; const float* qtk[2]; float* d3[2]; float* part;
                const float* vn; };   // vn: V(s') (advantage=1) replaces min Q'(s', pi(s'))
__global__ void __launch_bounds__(256) td_kernel(const TdArgs a) {
  mb_pdl_begin();
  __shared__ float sh[40];
  const int r = blockIdx.x * 256 + threadIdx.x;
  float e0 = 0.f, e1 = 0.f, s0 = 0.f, s1 = 0.f;
  if (r < a.N) {
    const float* x = a.X + (size_t)r * a.rw;
    const float boot = a.vn ? a.vn[r] : fminf(a.qtk[0][r], a.qtk[1][r]);
    const float y = x[2 * a.S + a.A] + x[2 * a.S + a.A + 1] * a.gamma * boot;
    const float q0 = a.qk[0][r], q1 = a.qk[1][r], d0 = q0 - y, d1 = q1 - y;
    a.d3[0][r] = 2.0f * d0 / (float)a.N; a.d3[1][r] = 2.0f * d1 / (float)a.N;
    e0 = d0 * d0; e1 = d1 * d1; s0 = q0; s1 = q1;
  }
  e0 = block_sum(e0, sh); e1 = block_sum(e1, sh); s0 = block_sum(s0, sh); s1 = block_sum(s1, sh);
  if (threadIdx.x == 0) { float* p = a.part + (size_t)blockIdx.x * 4; p[0] = e0; p[1] = e1; p[2] = s0; p[3] = s1; }
}

// ReLU backward of a one-output head: dH2[k][r][n] = H2[k][r][n] > 0 ? g_k[r] * w3_k[n] : 0   (g == nullptr: g = 1, dQ/dH2)
struct HeadBwdArgs { const float* H2[2]; const float* g[2]; const float* w3[2]; float* D[2]; int N; };
__global__ void __launch_bounds__(256) head_bwd_kernel(const HeadBwdArgs a) {
  mb_pdl_begin();
  const int k = blockIdx.y;
  const float4* h = reinterpret_cast<const float4*>(a.H2[k]);
  const float4* w = reinterpret_cast<const float4*>(a.w3[k]);
  float4* d = reinterpret_cast<float4*>(a.D[k]);
  const long long total = (long long)a.N * (H / 4);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i >> 6), c = (int)(i & 63);
    const float g = a.g[k] ? a.g[k][r] : 1.0f;
    const float4 hv = h[i], wv = __ldg(w + c);
    d[i] = make_float4(hv.x > 0.f ? g * wv.x : 0.f, hv.y > 0.f ? g * wv.y : 0.f, hv.z > 0.f ? g * wv.z : 0.f, hv.w > 0.f ? g * wv.w : 0.f);
  }
}

// Narrow tails with 256 inputs and A <= 32 outputs per row (policy head: tanh(h W3^T + b) * max_action; dQ/da = dH1 W1[:, S:]):
// one warp per row, the A x 256 weight slice in shared memory, lanes along the 256 inputs (two 128-bit loads each).
struct RowDotJob { const float* X; const float* W; int ldw, wt; const float* b; float* out; int M; };    // wt = 0: W[j][k] (ld = ldw); 1: W[k][j]
struct RowDotArgs { RowDotJob job[4]; int njobs, A; float scale; int tanh_act; };
__global__ void __launch_bounds__(256) rowdot_kernel(const RowDotArgs a) {
  mb_pdl_begin();
  extern __shared__ __align__(16) float wsm[];                      // [A][256]
  const RowDotJob& jb = a.job[blockIdx.y];
  for (int i = threadIdx.x; i < a.A * H; i += 256) {
    const int j = i >> 8, k = i & 255;
    wsm[i] = jb.wt ? __ldg(jb.W + (size_t)k * jb.ldw + j) : __ldg(jb.W + (size_t)j * jb.ldw + k);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int step = gridDim.x * 8;
  int m = blockIdx.x * 8 + warp;
  float4 x0 = make_float4(0.f, 0.f, 0.f, 0.f), x1 = x0;
  if (m < jb.M) { x0 = __ldg(reinterpret_cast<const float4*>(jb.X + (size_t)m * H) + lane); x1 = __ldg(reinterpret_cast<const float4*>(jb.X + (size_t)m * H) + 32 + lane); }
  for (; m < jb.M; m += step) {
    float4 n0 = x0, n1 = x1;                                         // next row in flight while this one is reduced
    if (m + step < jb.M) {
      n0 = __ldg(reinterpret_cast<const float4*>(jb.X + (size_t)(m + step) * H) + lane);
      n1 = __ldg(reinterpret_cast<const float4*>(jb.X + (size_t)(m + step) * H) + 32 + lane);
    }
    float mine = 0.f;
    for (int j = 0; j < a.A; ++j) {
      const float4 w0 = *(reinterpret_cast<const float4*>(wsm + j * H) + lane), w1 = *(reinterpret_cast<const float4*>(wsm + j * H) + 32 + lane);
      float s = x0.x * w0.x + x0.y * w0.y + x0.z * w0.z + x0.w * w0.w + x1.x * w1.x + x1.y * w1.y + x1.z * w1.z + x1.w * w1.w;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == j) mine = s;
    }
    if (lane < a.A) {
      float t = mine + (jb.b ? __ldg(jb.b + lane) : 0.f);
      if (a.tanh_act) t = tanhf(t) * a.scale;
      jb.out[(size_t)m * a.A + lane] = t;
    }
    x0 = n0; x1 = n1;
  }
}

__global__ void __launch_bounds__(1024) actor_scalar_kernel(const ActorArgs a) {
  mb_pdl_begin();
  __shared__ float sh[40];
  actor_reduce(a, sh);
}

// d loss / d (pre-tanh policy output) per row (mobody.py:321-330) + the logging scalars; 128 rows per block, last block reduces
__global__ void __launch_bounds__(128) policy_grad_kernel(const PolicyBwdArgs a) {
  mb_pdl_begin();
  __shared__ float red[40];
  __shared__ int last;
  const int tid = threadIdx.x, r = blockIdx.x * 128 + tid;
  const float pw = a.out[9], mean_h = a.out[10];
  float w = 0.f, w_s = 0.f, w_mn = 3.4e38f, w_mx = -3.4e38f, w_e = 0.f;
  if (r < a.N) {
    if (r < a.n_true) {
      w = bc_weight(a, r, mean_h);                                                               // :252-263
      const float* x = a.X + (size_t)r * a.rw + a.S;
      float e = 0.f;
      for (int j = 0; j < a.A; ++j) { const float d = a.api[(size_t)r * a.A + j] - x[j]; e += d * d; }
      w_s = w; w_mn = w; w_mx = w; w_e = w * e;
    }
    const bool first = a.qv[0][r] <= a.qv[1][r];                                                // torch.min(q1, q2): gradient follows the smaller one
    for (int j = 0; j < a.A; ++j) {
      const size_t e = (size_t)r * a.A + j;
      const float ap = a.api[e];
      float g = -pw / (float)a.N * (first ? a.gak[0][e] : a.gak[1][e]);
      if (r < a.n_true) g += a.bc_coef * w * 2.0f * (ap - a.X[(size_t)r * a.rw + a.S + j]) / (float)((size_t)a.n_true * a.A);
      const float t = ap / a.max_action;
      a.d3p[e] = g * a.max_action * (1.0f - t * t);
    }
  }
  w_s = block_sum(w_s, red); w_e = block_sum(w_e, red);
  w_mn = block_minmax(w_mn, red, false); w_mx = block_minmax(w_mx, red, true);
  if (tid == 0) { float* p = a.part + (size_t)blockIdx.x * 4; p[0] = w_s; p[1] = w_mn; p[2] = w_mx; p[3] = w_e; }
  __threadfence();
  __syncthreads();
  if (tid == 0) last = atomicAdd(a.counter, 1) == (int)gridDim.x - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  float s_w = 0.f, s_e = 0.f, mn = 3.4e38f, mx = -3.4e38f;
  for (int t = tid; t < (int)gridDim.x; t += 128) {
    const float* p = a.part + (size_t)t * 4;
    s_w += __ldcg(p); mn = fminf(mn, __ldcg(p + 1)); mx = fmaxf(mx, __ldcg(p + 2)); s_e += __ldcg(p + 3);
  }
  s_w = block_sum(s_w, red); s_e = block_sum(s_e, red);
  mn = block_minmax(mn, red, false); mx = block_minmax(mx, red, true);
  if (tid == 0) {
    const float bc = s_e / (float)((size_t)a.n_true * a.A);
    a.out[2] = pw * (-a.out[4]) + a.bc_coef * bc;
    a.out[3] = bc; a.out[6] = s_w / (float)a.n_true; a.out[7] = mn; a.out[8] = mx;
  }
}

// ================= value step (advantage=1, mobody.py:210-242), first in the update =================
// adv = min(Q'1(s, a), Q'2(s, a)) - V(s) with the target critics before this update's Polyak step, all N rows;
// v_loss = mean(|0.7 - 1[adv < 0]| adv^2) (asymmetric_l2_loss, :85-86).  d v_loss / d V(s) of a row; loss / adv / V partials.
__device__ __forceinline__ float expectile_grad(float qt0, float qt1, float v, int N, float& loss, float& adv) {
  adv = fminf(qt0, qt1) - v;
  const float wt = fabsf(0.7f - (adv < 0.f ? 1.0f : 0.0f));
  loss = wt * adv * adv;
  return -2.0f * wt * adv / (float)N;
}
struct ValueArgs {
  const float* X; int N, S, A, rw;
  MlpPtrs v, qt[2];
  float* qts[2];       // Q'_k(s, a), [N]
  float* vs;           // V(s), [N]
  float* Hv[2];        // relu activations of V(s), [N][256]
  float* Dv[2];        // dLoss/d(pre-activation), [N][256]
  float* d3;           // dLoss/dV(s), [N]
  float* part;         // [n_tiles][4]: sum loss, sum adv, sum V(s), 0
};

// roles 0, 1 = Q'_k(s, a) (no grad), role 2 = V(s) with stored activations
template <int RPT>
__global__ void __launch_bounds__(NT, RPT == 4 ? 2 : 1) value_fwd_kernel(ValueArgs a) {
  mb_pdl_begin();
  constexpr int TM = 8 * RPT;
  extern __shared__ __align__(16) float sm[];
  const int S = a.S, A = a.A, ldi = rup16(S + A);
  float* X0 = sm; float* X1 = X0 + TM * H; float* in_s = X1 + TM * H; float* qa = in_s + TM * ldi;
  const int tid = threadIdx.x, row0 = blockIdx.x * TM, rows = min(TM, a.N - row0), role = blockIdx.y;
  const int K = role == 2 ? S : S + A;
  for (int i = tid; i < TM * ldi; i += NT) {
    const int r = i / ldi, j = i - r * ldi;
    in_s[i] = (r < rows && j < K) ? a.X[(size_t)(row0 + r) * a.rw + j] : 0.f;       // [s, 0] or [s, a, 0]
  }
  __syncthreads();
  if (role == 2) {
    big_layer_mma<true, RPT>(in_s, ldi, S, a.v.w[0], a.v.b[0], X0, ACT_RELU);
    store_tile<TM>(X0, a.Hv[0], row0, rows);
    big_layer_mma<true, RPT, true>(X0, H, H, a.v.w[1], a.v.b[1], X1, ACT_RELU);
    store_tile<TM>(X1, a.Hv[1], row0, rows);
    q_head<TM>(X1, a.v.w[2], a.v.b[2], qa);
    if (tid < rows) a.vs[row0 + tid] = qa[tid];
  } else {
    big_layer_mma<true, RPT>(in_s, ldi, S + A, a.qt[role].w[0], a.qt[role].b[0], X0, ACT_RELU);
    big_layer_mma<true, RPT, true>(X0, H, H, a.qt[role].w[1], a.qt[role].b[1], X1, ACT_RELU);
    q_head<TM>(X1, a.qt[role].w[2], a.qt[role].b[2], qa);
    if (tid < rows) a.qts[role][row0 + tid] = qa[tid];
  }
}

// expectile gradient and V's backward to the pre-activations
template <int RPT>
__global__ void __launch_bounds__(NT, RPT == 4 ? 2 : 1) value_bwd_kernel(ValueArgs a) {
  mb_pdl_begin();
  constexpr int TM = 8 * RPT;
  extern __shared__ __align__(16) float sm[];
  __shared__ float red[40];
  float* X0 = sm; float* X1 = X0 + TM * H; float* g3 = X1 + TM * H;
  const int tid = threadIdx.x, row0 = blockIdx.x * TM, rows = min(TM, a.N - row0);
  load_tile<TM>(X0, a.Hv[0], row0, rows);
  load_tile<TM>(X1, a.Hv[1], row0, rows);
  float l = 0.f, ad = 0.f, vv = 0.f;
  if (tid < TM) {
    float g = 0.f;
    if (tid < rows) {
      const int r = row0 + tid;
      vv = a.vs[r];
      g = expectile_grad(a.qts[0][r], a.qts[1][r], vv, a.N, l, ad);
      a.d3[r] = g;
    }
    g3[tid] = g;
  }
  __syncthreads();
  head_backward<TM>(X1, a.v.w[2], g3);
  store_tile<TM>(X1, a.Dv[1], row0, rows);
  big_layer_mma<false, RPT, true>(X1, H, H, a.v.w[1], nullptr, X0, ACT_MASK);
  store_tile<TM>(X0, a.Dv[0], row0, rows);
  l = block_sum(l, red); ad = block_sum(ad, red); vv = block_sum(vv, red);
  if (tid == 0) { float* p = a.part + (size_t)blockIdx.x * 4; p[0] = l; p[1] = ad; p[2] = vv; p[3] = 0.f; }
}

// large-batch path: the same row math between the GEMMs, 256-row blocks (one partial per block)
__global__ void __launch_bounds__(256) value_loss_kernel(const ValueArgs a) {
  mb_pdl_begin();
  __shared__ float sh[40];
  const int r = blockIdx.x * 256 + threadIdx.x;
  float l = 0.f, ad = 0.f, vv = 0.f;
  if (r < a.N) {
    vv = a.vs[r];
    a.d3[r] = expectile_grad(a.qts[0][r], a.qts[1][r], vv, a.N, l, ad);
  }
  l = block_sum(l, sh); ad = block_sum(ad, sh); vv = block_sum(vv, sh);
  if (threadIdx.x == 0) { float* p = a.part + (size_t)blockIdx.x * 4; p[0] = l; p[1] = ad; p[2] = vv; p[3] = 0.f; }
}

}  // namespace trn

// ---------------- host launchers ----------------
// Row tile of the mma.sync kernels: 16 rows per CTA so that a 320-row batch still spreads over 20 SMs.  The train step runs
// them only below MOBODY_TC_TRAIN_MIN_ROWS, where 16-row tiles are always used.  The classifier takes 32 rows per CTA once the
// 16-row tiles would exceed one CTA per SM (>= 2 368 rows; measured cross-over between 1 280 and 2 560 rows), two CTAs per SM
// (128 registers, 70 KB shared memory each): 16 warps per SM hide the L2 / HMMA latencies that one 64-row CTA per SM (8 warps)
// exposes -- train step at batch 4096: 1 025 -> 1 304 updates/s.
constexpr int TRAIN_TM = 16;
static int pick_tm(int N) { return N >= 148 * 16 ? 32 : 16; }
template <typename K> static const char* set_smem(K kern, size_t bytes) {
  if (bytes > 227 * 1024) return "train step: shared memory budget exceeded for this (S, A)";
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess) return "cudaFuncSetAttribute failed";
  return nullptr;
}

const char* mb_train_critic_launch(const trn::CriticArgs& a, cudaStream_t st) {
  constexpr int tm = TRAIN_TM;
  const int ntiles = (a.N + tm - 1) / tm;
  const size_t bytes = (2 * (size_t)tm * simt::H + (size_t)tm * simt::rup16(a.S + a.A) + 2 * tm + 8) * sizeof(float);
  auto k1 = trn::critic_fwd_kernel<tm / 8>;
  auto k2 = trn::critic_tgt_kernel<tm / 8>;
  auto k3 = trn::critic_bwd_kernel<tm / 8>;
  if (const char* e = set_smem(k1, bytes)) return e;
  if (const char* e = set_smem(k2, bytes)) return e;
  if (const char* e = set_smem(k3, bytes)) return e;
  mb_launch(k1, dim3(ntiles, a.vn ? 5 : 4), dim3(simt::NT), bytes, st, a);
  if (!a.vn) mb_launch(k2, dim3(ntiles, 2), dim3(simt::NT), bytes, st, a);     // advantage=1: the TD target is V(s')
  mb_launch(k3, dim3(ntiles, 2), dim3(simt::NT), bytes, st, a);
  return nullptr;
}
const char* mb_train_value_launch(const trn::ValueArgs& a, cudaStream_t st) {
  constexpr int tm = TRAIN_TM;
  const int ntiles = (a.N + tm - 1) / tm;
  const size_t bytes = (2 * (size_t)tm * simt::H + (size_t)tm * simt::rup16(a.S + a.A) + 2 * tm + 8) * sizeof(float);
  auto k1 = trn::value_fwd_kernel<tm / 8>;
  auto k2 = trn::value_bwd_kernel<tm / 8>;
  if (const char* e = set_smem(k1, bytes)) return e;
  if (const char* e = set_smem(k2, bytes)) return e;
  mb_launch(k1, dim3(ntiles, 3), dim3(simt::NT), bytes, st, a);
  mb_launch(k2, dim3(ntiles), dim3(simt::NT), bytes, st, a);
  return nullptr;
}
const char* mb_train_actor_launch(const trn::ActorArgs& a, cudaStream_t st) {
  constexpr int tm = TRAIN_TM;
  const int ntiles = (a.N + tm - 1) / tm;
  const size_t bytes = (2 * (size_t)tm * simt::H + (size_t)tm * simt::rup16(a.S + a.A) + 2 * tm + (size_t)tm * a.A + 8) * sizeof(float);
  auto k2 = trn::actor_q_kernel<tm / 8>;
  if (const char* e = set_smem(k2, bytes)) return e;
  mb_launch(k2, dim3(ntiles, 4), dim3(simt::NT), bytes, st, a);
  return nullptr;
}
const char* mb_train_policy_bwd_launch(const trn::PolicyBwdArgs& a, cudaStream_t st) {
  constexpr int tm = TRAIN_TM;
  size_t bytes = (2 * (size_t)tm * simt::H + (size_t)tm * simt::rup16(a.A) + tm + 40) * sizeof(float);
  auto kern = trn::policy_bwd_kernel<tm / 8>;
  if (const char* e = set_smem(kern, bytes)) return e;
  mb_launch(kern, dim3((a.N + tm - 1) / tm), dim3(simt::NT), bytes, st, a);
  return nullptr;
}
const char* mb_train_wgrad_launch(const trn::WgradArgs& a, cudaStream_t st) {
  int maxt = 1;
  for (int j = 0; j < a.njobs; ++j) {
    const trn::WgradJob& jb = a.job[j];
    if (trn::wgrad_use_mma(jb.O) && ((jb.ldD | jb.ldX) & 3)) return "weight gradient: operand rows must be 16-byte aligned";
    if (!trn::wgrad_use_mma(jb.O) && (jb.O > 32 || ((jb.I | jb.ldX) & 3))) return "weight gradient: unsupported head shape";
    const int t = trn::wgrad_tiles(jb.O, jb.I);
    if (t > maxt) maxt = t;
  }
  if (const char* e = set_smem(trn::wgrad_kernel, trn::WGRAD_SMEM)) return e;
  mb_launch(trn::wgrad_kernel, dim3(maxt, a.nsplit, a.njobs), dim3(256), trn::WGRAD_SMEM, st, a);
  return nullptr;
}
const char* mb_train_adam_launch(const trn::AdamArgs& a, cudaStream_t st) {
  int maxn = 1;
  for (int j = 0; j < a.njobs; ++j) if (a.job[j].n > maxn) maxn = a.job[j].n;
  int gx = (maxn + 255) / 256; if (gx > 256) gx = 256;
  mb_launch(trn::adam_kernel, dim3(gx, a.njobs), dim3(256), 0, st, a);
  return nullptr;
}

// ---------------- whole train step (C ABI: mobody_train_step) ----------------
struct TrainWs {   // float offsets into the workspace
  size_t Hq[2][2], Dq[2][2], d3[2], part, Hp[2], Dp[2], api, a2, qk[2], qtk[2], qv[2], qh[2], gak[2], d3p, scal, part2, cnt, gq[2][6], gp[6], T[2], img[17], total;
  // advantage=1, past `total` (mobody_train_ex_workspace_bytes): V(s), V(s'), V(s_t), dLoss/dV, value partials, V's
  // weight-gradient partials and weight images.  V's activations use Hp / Dp, which the value step finishes with before
  // the critic phase writes pi(s) there.
  size_t vs, vn, vh, d3v, partv, gv[6], img_v[3], total_ex;
  int ntiles;
};
static TrainWs train_ws(int N, int S, int A, int nsplit) {
  TrainWs w{}; size_t o = 0;
  auto take = [&](size_t n) { size_t r = o; o += (n + 3) & ~(size_t)3; return r; };
  const size_t act = (size_t)N * 256;
  w.ntiles = (N + TRAIN_TM - 1) / TRAIN_TM;          // upper bound: the tcgen05 path's 256-row blocks need fewer
  for (int k = 0; k < 2; ++k) for (int l = 0; l < 2; ++l) { w.Hq[k][l] = take(act); w.Dq[k][l] = take(act); }
  for (int k = 0; k < 2; ++k) w.d3[k] = take(N);
  w.part = take((size_t)w.ntiles * 4);
  for (int l = 0; l < 2; ++l) { w.Hp[l] = take(act); w.Dp[l] = take(act); }
  w.api = take((size_t)N * A); w.a2 = take((size_t)N * A); w.d3p = take((size_t)N * A);
  for (int k = 0; k < 2; ++k) { w.qk[k] = take(N); w.qtk[k] = take(N); w.qv[k] = take(N); w.qh[k] = take(N); w.gak[k] = take((size_t)N * A); }
  w.scal = take(16); w.part2 = take((size_t)w.ntiles * 4); w.cnt = take(4);
  const size_t qn[6] = {(size_t)256 * (S + A), 256, 256 * 256, 256, 256, 1};       // w1 b1 w2 b2 w3 b3
  const size_t pn[6] = {(size_t)256 * S, 256, 256 * 256, 256, (size_t)A * 256, (size_t)A};
  for (int k = 0; k < 2; ++k) for (int t = 0; t < 6; ++t) w.gq[k][t] = take(qn[t] * nsplit);
  for (int t = 0; t < 6; ++t) w.gp[t] = take(pn[t] * nsplit);
  for (int l = 0; l < 2; ++l) w.T[l] = take(act);      // transient hidden activations of the tensor-core path (pi(s'), Q', q_hat)
  {   // packed TF32 hi/lo weight images of the tensor-core path (umma_gemm.cuh: SRC_PACKED); slots: see mb_train_step_tc_launch
    const int ik[17] = {S, 256, 256, S + A, S + A, 256, 256, S + A, S + A, 256, 256, 256, 256, A, 256, 256, 256};
    const int inp[17] = {256, 256, 64, 256, 256, 256, 256, 256, 256, 256, 256, 256, 256, 256, 256, 64, 64};
    for (int i = 0; i < 17; ++i) w.img[i] = take(ug::packed_floats(ik[i], inp[i]));
  }
  w.total = o;
  w.vs = take(N); w.vn = take(N); w.vh = take(N); w.d3v = take(N); w.partv = take((size_t)w.ntiles * 4);
  const size_t vn6[6] = {(size_t)256 * S, 256, 256 * 256, 256, 256, 1};
  for (int t = 0; t < 6; ++t) w.gv[t] = take(vn6[t] * nsplit);
  w.img_v[0] = take(ug::packed_floats(S, 256)); w.img_v[1] = take(ug::packed_floats(256, 256)); w.img_v[2] = take(ug::packed_floats(256, 256));
  w.total_ex = o;
  return w;
}
long long mb_train_workspace_bytes(int N, int S, int A, int nsplit) { return (long long)train_ws(N, S, A, nsplit).total * 4; }
long long mb_train_ex_workspace_bytes(int N, int S, int A, int nsplit) { return (long long)train_ws(N, S, A, nsplit).total_ex * 4; }

static MlpPtrs as_ptrs(const mobody_mlp_state& s) { MlpPtrs p; for (int i = 0; i < 3; ++i) { p.w[i] = s.w[i]; p.b[i] = s.b[i]; } return p; }

// Adam on ValueFunc (lr = critic_lr, :132) from the row-split partials of its weight gradients
static const char* value_adam(const mobody_train_ex_desc& x, const TrainWs& w, float* ws, cudaStream_t st) {
  const int S = x.base.S;
  trn::AdamArgs av{}; av.nsplit = x.base.nsplit; av.b1 = 0.9f; av.b2 = 0.999f; av.eps = 1e-8f; av.tau = 0.f; av.njobs = 6;
  const double bc1 = 1.0 - pow(0.9, (double)x.t_v), bc2 = 1.0 - pow(0.999, (double)x.t_v);
  av.lr_over_bc1 = (float)(x.base.critic_lr / bc1); av.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
  const int vn6[6] = {256 * S, 256, 256 * 256, 256, 256, 1};
  for (int t = 0; t < 6; ++t) {
    const int li = t >> 1; const bool isw = (t & 1) == 0;
    av.job[t] = {isw ? x.value.w[li] : x.value.b[li], ws + w.gv[t], isw ? x.value_m.w[li] : x.value_m.b[li],
                 isw ? x.value_v.w[li] : x.value_v.b[li], nullptr, vn6[t]};
  }
  return mb_train_adam_launch(av, st);
}
static trn::ValueArgs value_args(const mobody_train_ex_desc& x, const TrainWs& w, float* ws) {
  const mobody_train_desc& d = x.base;
  trn::ValueArgs v{};
  v.X = d.rows; v.N = d.N; v.S = d.S; v.A = d.A; v.rw = d.row_width;
  v.v = as_ptrs(x.value); v.qt[0] = as_ptrs(d.q1_target); v.qt[1] = as_ptrs(d.q2_target);
  v.qts[0] = ws + w.qtk[0]; v.qts[1] = ws + w.qtk[1]; v.vs = ws + w.vs;     // (qtk is free: the TD target is V(s'))
  for (int l = 0; l < 2; ++l) { v.Hv[l] = ws + w.Hp[l]; v.Dv[l] = ws + w.Dp[l]; }
  v.d3 = ws + w.d3v; v.part = ws + w.partv;
  return v;
}
// scalars_out: slots [0..10] always, [11..13] with the value step, [14] (q_behavior) with any non-default flag
static void copy_scalars(const mobody_train_ex_desc& x, const float* scal, cudaStream_t st) {
  float* out = x.base.scalars_out;
  if (!out) return;
  cudaMemcpyAsync(out, scal, (x.advantage ? 15 : 11) * sizeof(float), cudaMemcpyDeviceToDevice, st);
  if (!x.advantage && (!x.scale_q || !x.q_weighted)) cudaMemcpyAsync(out + 14, scal + 14, sizeof(float), cudaMemcpyDeviceToDevice, st);
}

// ---------------- large-batch update on tcgen05 (rows >= MOBODY_TC_TRAIN_MIN_ROWS: the GEMMs are throughput bound) ----------------
const char* mb_gemm_launch(const ug::Args& a, cudaStream_t st);     // train_tc.cu

static ug::Job gemm_job(const float* A, int lda, int a_src, const float* B, int ldb, int b_src, int M, int N, int K) {
  ug::Job j{}; j.A = A; j.lda = lda; j.a_src = a_src; j.B = B; j.ldb = ldb; j.b_src = b_src; j.M = M; j.N = N; j.K = K;
  j.epi = ug::EPI_STORE;
  return j;
}
// forward layer: C = act(A W^T + b); nn.Linear weight [out][in] is the K-contiguous B operand
static ug::Job fwd_job(const float* A, int lda, int M, int K, const float* W, const float* b, int Nout, float* C, bool relu = true) {
  ug::Job j = gemm_job(A, lda, ug::SRC_KCONTIG, W, K, ug::SRC_KCONTIG, M, Nout, K);
  j.bias = b; j.relu = relu ? 1 : 0; j.C = C; j.ldc = Nout;
  return j;
}
// backward-data through a Linear + ReLU: C = (D W) * 1[mask > 0]; the weight is read "k = out, n = in"
static ug::Job bwd_job(const float* D, int ldd, int M, int Kout, const float* W, int ldw, int Nin, const float* mask, float* C) {
  ug::Job j = gemm_job(D, ldd, ug::SRC_KCONTIG, W, ldw, ug::SRC_RCONTIG, M, Nin, Kout);
  j.epi = mask ? ug::EPI_MASK : ug::EPI_STORE; j.mask = mask; j.ldmask = Nin; j.C = C; j.ldc = Nin;
  return j;
}
// weight gradient: dW[o][i] = sum_r D[r][o] X[r][i] (+ db[o] = sum_r D[r][o]); both operands are row-contiguous in k = r
static ug::Job wgrad_job(const float* D, int ldd, int O, const float* X, int ldx, int I, int rows, float* dW, float* db) {
  ug::Job j = gemm_job(D, ldd, ug::SRC_RCONTIG, X, ldx, ug::SRC_RCONTIG, O, I, rows);
  j.epi = ug::EPI_PART; j.C = dW; j.db = db;
  return j;
}
const char* mb_pack_b_launch(const ug::PackArgs& a, cudaStream_t st);     // train_tc.cu
static ug::PackJob pack_job(const float* src, int ld, int mode, int N, int K, int NP, float* dst) {
  return ug::PackJob{src, ld, mode, N, K, NP, reinterpret_cast<uint32_t*>(dst)};
}
static const char* run_gemm_list(cudaStream_t st, int nsplit, const ug::Job* list, int n) {
  ug::Args a{}; a.nsplit = nsplit; a.njobs = n;
  for (int i = 0; i < n; ++i) a.job[i] = list[i];
  return mb_gemm_launch(a, st);
}
template <typename... J> static const char* run_gemms(cudaStream_t st, int nsplit, J... jobs) {
  const ug::Job list[] = {jobs...};
  return run_gemm_list(st, nsplit, list, (int)sizeof...(jobs));
}

// Launches of the large-batch update that do not depend on each other run on a side stream (fork by event, join by event):
// the layer-2 / head weight gradients beside the backward-data GEMM that produces layer 1's error signal, the single-CTA
// actor scalar reduction beside the dQ/da chain.  Same kernels, same partial-sum layout: bit-identical to the single-stream
// chain (MOBODY_TRAIN_SIDE=0), tested.
struct TrainSide { cudaStream_t s = nullptr; cudaEvent_t fork[4] = {}, join[3] = {}; bool ok = false, tried = false; };
static TrainSide& train_side() {
  static TrainSide per_dev[64];
  int dev = 0; cudaGetDevice(&dev);
  TrainSide& ss = per_dev[dev & 63];
  if (!ss.tried) {
    ss.tried = true;
    const char* e = getenv("MOBODY_TRAIN_SIDE");
    if (!(e && e[0] == '0') && cudaStreamCreateWithFlags(&ss.s, cudaStreamNonBlocking) == cudaSuccess) {
      ss.ok = true;
      for (int i = 0; i < 4 && ss.ok; ++i) ss.ok = cudaEventCreateWithFlags(&ss.fork[i], cudaEventDisableTiming) == cudaSuccess;
      for (int i = 0; i < 3 && ss.ok; ++i) ss.ok = cudaEventCreateWithFlags(&ss.join[i], cudaEventDisableTiming) == cudaSuccess;
    }
  }
  return ss;
}

static const char* mb_train_step_tc_launch(const mobody_train_ex_desc& x, const TrainWs& w, cudaStream_t st) {
  const mobody_train_desc& d = x.base;
  const bool adv = x.advantage, branch = adv || !x.scale_q || !x.q_weighted;
  TrainSide& side = train_side();
  // fork(i): the side stream continues after everything enqueued on `st` so far; join(i): `st` waits for the side stream
  auto fork = [&](int i) -> cudaStream_t {
    if (!side.ok) return st;
    if (cudaEventRecord(side.fork[i], st) != cudaSuccess || cudaStreamWaitEvent(side.s, side.fork[i], 0) != cudaSuccess) return st;
    return side.s;
  };
  auto join = [&](int i) {
    if (side.ok) { cudaEventRecord(side.join[i], side.s); cudaStreamWaitEvent(st, side.join[i], 0); }
  };
  const int N = d.N, nt = d.n_true, S = d.S, A = d.A, rw = d.row_width, ns = d.nsplit, SA = S + A;
  float* ws = (float*)d.workspace;
  const float* X = d.rows;
  const MlpPtrs pi = as_ptrs(d.policy), q[2] = {as_ptrs(d.q1), as_ptrs(d.q2)}, qt[2] = {as_ptrs(d.q1_target), as_ptrs(d.q2_target)};
  float* Hq[2][2]; float* Dq[2][2]; float* T[2] = {ws + w.T[0], ws + w.T[1]};
  for (int k = 0; k < 2; ++k) for (int l = 0; l < 2; ++l) { Hq[k][l] = ws + w.Hq[k][l]; Dq[k][l] = ws + w.Dq[k][l]; }
  float* Hp[2] = {ws + w.Hp[0], ws + w.Hp[1]}; float* Dp[2] = {ws + w.Dp[0], ws + w.Dp[1]};
  float* api = ws + w.api; float* a2 = ws + w.a2; float* d3p = ws + w.d3p;
  float* qk[2] = {ws + w.qk[0], ws + w.qk[1]}; float* qtk[2] = {ws + w.qtk[0], ws + w.qtk[1]};
  float* qv[2] = {ws + w.qv[0], ws + w.qv[1]}; float* qh[2] = {ws + w.qh[0], ws + w.qh[1]};
  float* gak[2] = {ws + w.gak[0], ws + w.gak[1]}; float* d3[2] = {ws + w.d3[0], ws + w.d3[1]};
  const char* e;
  // ---- weight images: every weight matrix the GEMMs use as a B operand, split into TF32 hi / lo planes ONCE (one launch) ----
  // slots: 0-2 pi W1 W2 W3 (forward) | 3,4 Q_k W1 | 5,6 Q_k W2 | 7,8 Q'_k W1 | 9,10 Q'_k W2 | 11,12 Q_k W2 (backward) |
  //        13 pi W3 (backward) | 14 pi W2 (backward) | 15,16 action columns of Q_k W1 (backward)
  float* img[17];
  for (int i = 0; i < 17; ++i) img[i] = ws + w.img[i];
  auto P = [&](ug::Job j, int slot) { j.B = img[slot]; j.b_src = ug::SRC_PACKED; return j; };   // B operand: weight image `slot`
  auto pack_q = [&](ug::PackArgs& pa, bool with_slices) {
    for (int k = 0; k < 2; ++k) {
      pa.job[pa.njobs++] = pack_job(q[k].w[0], SA, ug::SRC_KCONTIG, 256, SA, 256, img[3 + k]);
      pa.job[pa.njobs++] = pack_job(q[k].w[1], 256, ug::SRC_KCONTIG, 256, 256, 256, img[5 + k]);
      pa.job[pa.njobs++] = pack_job(q[k].w[1], 256, ug::SRC_RCONTIG, 256, 256, 256, img[11 + k]);
      if (with_slices) pa.job[pa.njobs++] = pack_job(q[k].w[0] + S, SA, ug::SRC_RCONTIG, A, 256, 64, img[15 + k]);
    }
  };
  {
    ug::PackArgs pa{};
    pa.job[pa.njobs++] = pack_job(pi.w[0], S, ug::SRC_KCONTIG, 256, S, 256, img[0]);
    pa.job[pa.njobs++] = pack_job(pi.w[1], 256, ug::SRC_KCONTIG, 256, 256, 256, img[1]);
    pa.job[pa.njobs++] = pack_job(pi.w[2], 256, ug::SRC_KCONTIG, A, 256, 64, img[2]);
    pa.job[pa.njobs++] = pack_job(pi.w[2], 256, ug::SRC_RCONTIG, 256, A, 256, img[13]);
    pa.job[pa.njobs++] = pack_job(pi.w[1], 256, ug::SRC_RCONTIG, 256, 256, 256, img[14]);
    for (int k = 0; k < 2; ++k) {
      pa.job[pa.njobs++] = pack_job(qt[k].w[0], SA, ug::SRC_KCONTIG, 256, SA, 256, img[7 + k]);
      pa.job[pa.njobs++] = pack_job(qt[k].w[1], 256, ug::SRC_KCONTIG, 256, 256, 256, img[9 + k]);
    }
    pack_q(pa, false);
    if ((e = mb_pack_b_launch(pa, st))) return e;
  }
  // ---- advantage=1: value step.  Q'_k(s, a) and V(s) (V's activations in Hp / Dp), expectile gradient, V's backward,
  //      weight gradients, Adam, and V's images again for V(s') / V(s_t) below.  Images: V W1, W2 forward, W2 backward ----
  const MlpPtrs vf = as_ptrs(x.value);
  float* img_v[3] = {ws + w.img_v[0], ws + w.img_v[1], ws + w.img_v[2]};
  auto PV = [&](ug::Job j, int slot) { j.B = img_v[slot]; j.b_src = ug::SRC_PACKED; return j; };
  auto pack_v = [&](int n) {
    ug::PackArgs pa{};
    pa.job[pa.njobs++] = pack_job(vf.w[0], S, ug::SRC_KCONTIG, 256, S, 256, img_v[0]);
    pa.job[pa.njobs++] = pack_job(vf.w[1], 256, ug::SRC_KCONTIG, 256, 256, 256, img_v[1]);
    if (n == 3) pa.job[pa.njobs++] = pack_job(vf.w[1], 256, ug::SRC_RCONTIG, 256, 256, 256, img_v[2]);
    return mb_pack_b_launch(pa, st);
  };
  if (adv) {
    const trn::ValueArgs v = value_args(x, w, ws);
    if ((e = pack_v(3))) return e;
    if ((e = run_gemms(st, 1, P(fwd_job(X, rw, N, SA, qt[0].w[0], qt[0].b[0], 256, T[0]), 7), P(fwd_job(X, rw, N, SA, qt[1].w[0], qt[1].b[0], 256, T[1]), 8),
                       PV(fwd_job(X, rw, N, S, vf.w[0], vf.b[0], 256, v.Hv[0]), 0)))) return e;
    ug::Job h[3] = {fwd_job(T[0], 256, N, 256, qt[0].w[1], qt[0].b[1], 256, nullptr), fwd_job(T[1], 256, N, 256, qt[1].w[1], qt[1].b[1], 256, nullptr),
                    fwd_job(v.Hv[0], 256, N, 256, vf.w[1], vf.b[1], 256, v.Hv[1])};
    const MlpPtrs* hn[3] = {&qt[0], &qt[1], &vf};
    float* ho[3] = {v.qts[0], v.qts[1], v.vs};
    for (int i = 0; i < 3; ++i) { h[i].epi = ug::EPI_HEAD; h[i].w3 = hn[i]->w[2]; h[i].b3 = hn[i]->b[2]; h[i].out1 = ho[i]; }
    if ((e = run_gemms(st, 1, P(h[0], 9), P(h[1], 10), PV(h[2], 1)))) return e;
    mb_launch(trn::value_loss_kernel, dim3((N + 255) / 256), dim3(256), 0, st, v);
    trn::HeadBwdArgs hb{{v.Hv[1], nullptr}, {v.d3, nullptr}, {vf.w[2], nullptr}, {v.Dv[1], nullptr}, N};
    mb_launch(trn::head_bwd_kernel, dim3(296, 1), dim3(256), 0, st, hb);
    if ((e = run_gemms(st, 1, PV(bwd_job(v.Dv[1], 256, N, 256, vf.w[1], 256, 256, v.Hv[0], v.Dv[0]), 2)))) return e;
    if ((e = run_gemms(st, ns, wgrad_job(v.Dv[0], 256, 256, X, rw, S, N, ws + w.gv[0], ws + w.gv[1]),
                       wgrad_job(v.Dv[1], 256, 256, v.Hv[0], 256, 256, N, ws + w.gv[2], ws + w.gv[3]),
                       wgrad_job(v.d3, 1, 1, v.Hv[1], 256, 256, N, ws + w.gv[4], ws + w.gv[5])))) return e;
    if ((e = value_adam(x, w, ws, st))) return e;
    if ((e = pack_v(2))) return e;
  }
  // ---- critic forward.  layer 1 of pi(s') (advantage=1: V(s') and V(s_t) instead), Q1(s,a), Q2(s,a), pi(s) side by side;
  //      then layer 2 (+ Q / V heads); then the policy tails ----
  float* vn = ws + w.vn; float* vh = ws + w.vh;
  {
    ug::Job l1[5] = {adv ? PV(fwd_job(X + SA, rw, N, S, vf.w[0], vf.b[0], 256, T[0]), 0) : P(fwd_job(X + SA, rw, N, S, pi.w[0], pi.b[0], 256, T[0]), 0),
                     P(fwd_job(X, rw, N, SA, q[0].w[0], q[0].b[0], 256, Hq[0][0]), 3), P(fwd_job(X, rw, N, SA, q[1].w[0], q[1].b[0], 256, Hq[1][0]), 4),
                     P(fwd_job(X, rw, N, S, pi.w[0], pi.b[0], 256, Hp[0]), 0), PV(fwd_job(X, rw, nt, S, vf.w[0], vf.b[0], 256, T[1]), 0)};
    if ((e = run_gemm_list(st, 1, l1, adv ? 5 : 4))) return e;
  }
  {
    ug::Job j1 = fwd_job(Hq[0][0], 256, N, 256, q[0].w[1], q[0].b[1], 256, Hq[0][1]), j2 = fwd_job(Hq[1][0], 256, N, 256, q[1].w[1], q[1].b[1], 256, Hq[1][1]);
    j1.epi = j2.epi = ug::EPI_HEAD; j1.w3 = q[0].w[2]; j1.b3 = q[0].b[2]; j1.out1 = qk[0]; j2.w3 = q[1].w[2]; j2.b3 = q[1].b[2]; j2.out1 = qk[1];
    ug::Job l2[5] = {P(fwd_job(T[0], 256, N, 256, pi.w[1], pi.b[1], 256, T[1]), 1), P(j1, 5), P(j2, 6),
                     P(fwd_job(Hp[0], 256, N, 256, pi.w[1], pi.b[1], 256, Hp[1]), 1), {}};
    if (adv) {   // V(s') -> vn, V(s_t) -> vh: heads only, no activations stored
      ug::Job hv[2] = {fwd_job(T[0], 256, N, 256, vf.w[1], vf.b[1], 256, nullptr), fwd_job(T[1], 256, nt, 256, vf.w[1], vf.b[1], 256, nullptr)};
      for (int i = 0; i < 2; ++i) { hv[i].epi = ug::EPI_HEAD; hv[i].w3 = vf.w[2]; hv[i].b3 = vf.b[2]; hv[i].out1 = i ? vh : vn; }
      l2[0] = PV(hv[0], 1); l2[4] = PV(hv[1], 1);
    }
    if ((e = run_gemm_list(st, 1, l2, adv ? 5 : 4))) return e;
  }
  {
    trn::RowDotArgs rd{}; rd.njobs = 2; rd.A = A; rd.scale = d.max_action; rd.tanh_act = 1;
    rd.job[0] = {T[1], pi.w[2], 256, 0, pi.b[2], a2, N}; rd.job[1] = {Hp[1], pi.w[2], 256, 0, pi.b[2], api, N};
    if (adv) { rd.job[0] = rd.job[1]; rd.njobs = 1; }                  // no pi(s'): only pi(s)
    mb_launch(trn::rowdot_kernel, dim3(296, rd.njobs), dim3(256), (size_t)A * 256 * sizeof(float), st, rd);
  }
  // ---- target critics on (s', pi(s')): the input is [s' | a2], read from two sources ----
  if (!adv) {
    ug::Job j1 = fwd_job(X + SA, rw, N, SA, qt[0].w[0], qt[0].b[0], 256, T[0]), j2 = fwd_job(X + SA, rw, N, SA, qt[1].w[0], qt[1].b[0], 256, T[1]);
    j1.A2 = j2.A2 = a2; j1.lda2 = j2.lda2 = A; j1.ksplit = j2.ksplit = S;
    if ((e = run_gemms(st, 1, P(j1, 7), P(j2, 8)))) return e;
    // layer 2 + head in place is not possible (C would overwrite A of another tile's... no: tiles own their rows) -> no C store at all
    ug::Job h1 = fwd_job(T[0], 256, N, 256, qt[0].w[1], qt[0].b[1], 256, nullptr), h2 = fwd_job(T[1], 256, N, 256, qt[1].w[1], qt[1].b[1], 256, nullptr);
    h1.epi = h2.epi = ug::EPI_HEAD; h1.w3 = qt[0].w[2]; h1.b3 = qt[0].b[2]; h1.out1 = qtk[0]; h2.w3 = qt[1].w[2]; h2.b3 = qt[1].b[2]; h2.out1 = qtk[1];
    if ((e = run_gemms(st, 1, P(h1, 9), P(h2, 10)))) return e;
  }
  // ---- TD target + MSE gradient, head backward, backward-data ----
  {
    trn::TdArgs t{X, N, S, A, rw, d.gamma, {qk[0], qk[1]}, {qtk[0], qtk[1]}, {d3[0], d3[1]}, ws + w.part, adv ? vn : nullptr};
    mb_launch(trn::td_kernel, dim3((N + 255) / 256), dim3(256), 0, st, t);
    trn::HeadBwdArgs hb{{Hq[0][1], Hq[1][1]}, {d3[0], d3[1]}, {q[0].w[2], q[1].w[2]}, {Dq[0][1], Dq[1][1]}, N};
    mb_launch(trn::head_bwd_kernel, dim3(296, 2), dim3(256), 0, st, hb);
    // layer-2 and head weight gradients need only head_bwd's output: beside the backward-data GEMM
    cudaStream_t s2 = fork(0);
    if ((e = run_gemms(s2, ns, wgrad_job(Dq[0][1], 256, 256, Hq[0][0], 256, 256, N, ws + w.gq[0][2], ws + w.gq[0][3]),
                       wgrad_job(Dq[1][1], 256, 256, Hq[1][0], 256, 256, N, ws + w.gq[1][2], ws + w.gq[1][3]),
                       wgrad_job(d3[0], 1, 1, Hq[0][1], 256, 256, N, ws + w.gq[0][4], ws + w.gq[0][5]),     // the one-output heads: one
                       wgrad_job(d3[1], 1, 1, Hq[1][1], 256, 256, N, ws + w.gq[1][4], ws + w.gq[1][5])))) return e;   // (mostly empty) tile each
    if ((e = run_gemms(st, 1, P(bwd_job(Dq[0][1], 256, N, 256, q[0].w[1], 256, 256, Hq[0][0], Dq[0][0]), 11),
                       P(bwd_job(Dq[1][1], 256, N, 256, q[1].w[1], 256, 256, Hq[1][0], Dq[1][0]), 12)))) return e;
  }
  // ---- critic weight gradients (row-split partials) + Adam + Polyak ----
  const mobody_mlp_state* qs[2] = {&d.q1, &d.q2};
  const mobody_mlp_state* qts[2] = {&d.q1_target, &d.q2_target};
  const mobody_mlp_state* qm[2] = {&d.q1_m, &d.q2_m};
  const mobody_mlp_state* qvv[2] = {&d.q1_v, &d.q2_v};
  if ((e = run_gemms(st, ns, wgrad_job(Dq[0][0], 256, 256, X, rw, SA, N, ws + w.gq[0][0], ws + w.gq[0][1]),
                     wgrad_job(Dq[1][0], 256, 256, X, rw, SA, N, ws + w.gq[1][0], ws + w.gq[1][1])))) return e;
  join(0);
  trn::AdamArgs ad{}; ad.nsplit = ns; ad.b1 = 0.9f; ad.b2 = 0.999f; ad.eps = 1e-8f; ad.tau = d.tau; ad.njobs = 12;
  ad.zero2 = reinterpret_cast<int*>(ws + w.cnt);
  {
    const double bc1 = 1.0 - pow(0.9, (double)d.t_q), bc2 = 1.0 - pow(0.999, (double)d.t_q);
    ad.lr_over_bc1 = (float)(d.critic_lr / bc1); ad.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
    const int qn[6] = {256 * SA, 256, 256 * 256, 256, 256, 1};
    for (int k = 0; k < 2; ++k)
      for (int t = 0; t < 6; ++t) {
        const int li = t >> 1; const bool isw = (t & 1) == 0;
        ad.job[6 * k + t] = {isw ? qs[k]->w[li] : qs[k]->b[li], ws + w.gq[k][t], isw ? qm[k]->w[li] : qm[k]->b[li],
                             isw ? qvv[k]->w[li] : qvv[k]->b[li], isw ? qts[k]->w[li] : qts[k]->b[li], qn[t]};
      }
  }
  if ((e = mb_train_adam_launch(ad, st))) return e;
  {   // the critics just changed: their images again (+ the action columns of W1 for dQ/da)
    ug::PackArgs pa{};
    pack_q(pa, true);
    if ((e = mb_pack_b_launch(pa, st))) return e;
  }
  // ---- actor: Q_k(s, pi(s)) with the UPDATED, frozen critics (activations kept for the backward), q_hat_k on the true rows
  //      (any non-default flag: on all rows, for q_behavior) ----
  const int nq = branch ? N : nt;
  {
    ug::Job j1 = fwd_job(X, rw, N, SA, q[0].w[0], q[0].b[0], 256, Hq[0][0]), j2 = fwd_job(X, rw, N, SA, q[1].w[0], q[1].b[0], 256, Hq[1][0]);
    j1.A2 = j2.A2 = api; j1.lda2 = j2.lda2 = A; j1.ksplit = j2.ksplit = S;
    if ((e = run_gemms(st, 1, P(j1, 3), P(j2, 4), P(fwd_job(X, rw, nq, SA, q[0].w[0], q[0].b[0], 256, T[0]), 3),
                       P(fwd_job(X, rw, nq, SA, q[1].w[0], q[1].b[0], 256, T[1]), 4)))) return e;
    ug::Job h[4] = {fwd_job(Hq[0][0], 256, N, 256, q[0].w[1], q[0].b[1], 256, Hq[0][1]), fwd_job(Hq[1][0], 256, N, 256, q[1].w[1], q[1].b[1], 256, Hq[1][1]),
                    fwd_job(T[0], 256, nq, 256, q[0].w[1], q[0].b[1], 256, nullptr), fwd_job(T[1], 256, nq, 256, q[1].w[1], q[1].b[1], 256, nullptr)};
    for (int i = 0; i < 4; ++i) { h[i].epi = ug::EPI_HEAD; h[i].w3 = q[i & 1].w[2]; h[i].b3 = q[i & 1].b[2]; h[i].out1 = i < 2 ? qv[i] : qh[i - 2]; }
    if ((e = run_gemms(st, 1, P(h[0], 5), P(h[1], 6), P(h[2], 5), P(h[3], 6)))) return e;
  }
  trn::ActorArgs ac{};
  ac.X = X; ac.N = N; ac.n_true = nt; ac.S = S; ac.A = A; ac.rw = rw; ac.max_action = d.max_action;
  for (int k = 0; k < 2; ++k) { ac.qv[k] = qv[k]; ac.qh[k] = qh[k]; ac.gak[k] = gak[k]; }
  ac.part = ws + w.part; ac.ntiles_c = (N + 255) / 256; ac.weight = d.weight; ac.out = ws + w.scal;
  ac.counter = reinterpret_cast<int*>(ws + w.cnt);
  ac.scale_q = x.scale_q; ac.branch = branch; ac.n_qh = nq; ac.part_v = adv ? ws + w.partv : nullptr;
  mb_launch(trn::actor_scalar_kernel, dim3(1), dim3(1024), 0, fork(1), ac);      // single CTA: beside the dQ/da chain below
  {   // dQ_k / d action: head backward with unit gradient, backward-data through layers 2 and 1 (action columns of W1 only)
    trn::HeadBwdArgs hb{{Hq[0][1], Hq[1][1]}, {nullptr, nullptr}, {q[0].w[2], q[1].w[2]}, {Dq[0][1], Dq[1][1]}, N};
    mb_launch(trn::head_bwd_kernel, dim3(296, 2), dim3(256), 0, st, hb);
    if ((e = run_gemms(st, 1, P(bwd_job(Dq[0][1], 256, N, 256, q[0].w[1], 256, 256, Hq[0][0], Dq[0][0]), 11),
                       P(bwd_job(Dq[1][1], 256, N, 256, q[1].w[1], 256, 256, Hq[1][0], Dq[1][0]), 12)))) return e;
    trn::RowDotArgs rd{}; rd.njobs = 2; rd.A = A; rd.scale = 1.f; rd.tanh_act = 0;
    for (int k = 0; k < 2; ++k) rd.job[k] = {Dq[k][0], q[k].w[0] + S, SA, 0, nullptr, gak[k], N};     // W1 is [256 out][S+A in]: gak[m][j] = sum_n dH1[m][n] W1[n][S+j]
    for (int k = 0; k < 2; ++k) rd.job[k].wt = 1;
    mb_launch(trn::rowdot_kernel, dim3(296, 2), dim3(256), (size_t)A * 256 * sizeof(float), st, rd);
  }
  trn::PolicyBwdArgs pb{}; pb.N = N; pb.n_true = nt; pb.S = S; pb.A = A; pb.rw = rw; pb.pi = pi;
  for (int k = 0; k < 2; ++k) { pb.gak[k] = gak[k]; pb.qv[k] = qv[k]; pb.qh[k] = qh[k]; }
  pb.api = api; pb.X = X; pb.bc_coef = d.bc_coef; pb.max_action = d.max_action;
  pb.d3p = d3p; pb.part = ws + w.part2; pb.out = ws + w.scal; pb.counter = reinterpret_cast<int*>(ws + w.cnt) + 1;
  pb.vh = adv ? vh : nullptr; pb.q_weighted = x.q_weighted;
  join(1);
  mb_launch(trn::policy_grad_kernel, dim3((N + 127) / 128), dim3(128), 0, st, pb);
  // ---- policy backward-data: dH2 = (d3 W3) * 1[H2 > 0], dH1 = (dH2 W2) * 1[H1 > 0]; weight gradients; Adam ----
  {
    cudaStream_t s2 = fork(2);                                           // head weight gradient beside the first backward-data GEMM
    if ((e = run_gemms(s2, ns, wgrad_job(d3p, A, A, Hp[1], 256, 256, N, ws + w.gp[4], ws + w.gp[5])))) return e;
    if ((e = run_gemms(st, 1, P(bwd_job(d3p, A, N, A, pi.w[2], 256, 256, Hp[1], Dp[1]), 13)))) return e;
    s2 = fork(3);                                                        // layer 2's beside the second
    if ((e = run_gemms(s2, ns, wgrad_job(Dp[1], 256, 256, Hp[0], 256, 256, N, ws + w.gp[2], ws + w.gp[3])))) return e;
    if ((e = run_gemms(st, 1, P(bwd_job(Dp[1], 256, N, 256, pi.w[1], 256, 256, Hp[0], Dp[0]), 14)))) return e;
    if ((e = run_gemms(st, ns, wgrad_job(Dp[0], 256, 256, X, rw, S, N, ws + w.gp[0], ws + w.gp[1])))) return e;
    join(2);
  }
  trn::AdamArgs ap{}; ap.nsplit = ns; ap.b1 = 0.9f; ap.b2 = 0.999f; ap.eps = 1e-8f; ap.tau = 0.f; ap.njobs = 6;
  {
    const double bc1 = 1.0 - pow(0.9, (double)d.t_pi), bc2 = 1.0 - pow(0.999, (double)d.t_pi);
    ap.lr_over_bc1 = (float)(d.actor_lr / bc1); ap.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
    const int pn[6] = {256 * S, 256, 256 * 256, 256, A * 256, A};
    for (int t = 0; t < 6; ++t) {
      const int li = t >> 1; const bool isw = (t & 1) == 0;
      ap.job[t] = {isw ? d.policy.w[li] : d.policy.b[li], ws + w.gp[t], isw ? d.policy_m.w[li] : d.policy_m.b[li],
                   isw ? d.policy_v.w[li] : d.policy_v.b[li], nullptr, pn[t]};
    }
  }
  if ((e = mb_train_adam_launch(ap, st))) return e;
  copy_scalars(x, ws + w.scal, st);
  return nullptr;
}

const char* mb_train_step_launch(const mobody_train_ex_desc& x, cudaStream_t st) {
  const mobody_train_desc& d = x.base;
  const int N = d.N, S = d.S, A = d.A, ns = d.nsplit;
  if (N < 1 || d.n_true < 1 || d.n_true > N || S < 1 || S > 128 || A < 1 || A > 32 || ns < 1 || ns > 64) return "train step: bad N/n_true/S/A/nsplit";
  const TrainWs w = train_ws(N, S, A, ns);
  if (!d.workspace || d.workspace_bytes < (long long)(x.advantage ? w.total_ex : w.total) * 4) return "train step: workspace too small";
  // large batches: every contraction as tcgen05 GEMM tiles.  Cross-over measured on the tuned tiles (S17/A6, updates/s tcgen05
  // vs mma.sync): 640 rows 4 540 vs 6 435, 1 280 rows 4 350 vs 4 220, 1 920 rows 3 920 vs 3 340, 2 560 rows 4 180 vs 3 600
  if (N >= MOBODY_TC_TRAIN_MIN_ROWS) return mb_train_step_tc_launch(x, w, st);
  float* ws = (float*)d.workspace;
  const bool branch = x.advantage || !x.scale_q || !x.q_weighted;
  // ---- advantage=1: value step (forward, expectile gradient, backward, weight gradients, Adam) ----
  if (x.advantage) {
    const trn::ValueArgs v = value_args(x, w, ws);
    if (const char* e = mb_train_value_launch(v, st)) return e;
    trn::WgradArgs g{}; g.N = N; g.nsplit = ns; g.njobs = 3;
    g.job[0] = {v.Dv[0], 256, d.rows, d.row_width, ws + w.gv[0], ws + w.gv[1], 256, S};
    g.job[1] = {v.Dv[1], 256, v.Hv[0], 256, ws + w.gv[2], ws + w.gv[3], 256, 256};
    g.job[2] = {v.d3, 1, v.Hv[1], 256, ws + w.gv[4], ws + w.gv[5], 1, 256};
    if (const char* e = mb_train_wgrad_launch(g, st)) return e;
    if (const char* e = value_adam(x, w, ws, st)) return e;
  }
  const mobody_mlp_state* qs[2] = {&d.q1, &d.q2};
  const mobody_mlp_state* qts[2] = {&d.q1_target, &d.q2_target};
  const mobody_mlp_state* qm[2] = {&d.q1_m, &d.q2_m};
  const mobody_mlp_state* qv[2] = {&d.q1_v, &d.q2_v};
  // ---- critic: TD target, forward, backward-data ----
  trn::CriticArgs c{};
  c.X = d.rows; c.N = N; c.S = S; c.A = A; c.rw = d.row_width; c.pi = as_ptrs(d.policy);
  for (int k = 0; k < 2; ++k) {
    c.q[k] = as_ptrs(*qs[k]); c.qt[k] = as_ptrs(*qts[k]);
    for (int l = 0; l < 2; ++l) { c.Hq[k][l] = ws + w.Hq[k][l]; c.Dq[k][l] = ws + w.Dq[k][l]; }
    c.d3[k] = ws + w.d3[k];
  }
  c.gamma = d.gamma; c.max_action = d.max_action; c.part = ws + w.part; c.a2 = ws + w.a2;
  c.Hp[0] = ws + w.Hp[0]; c.Hp[1] = ws + w.Hp[1]; c.api = ws + w.api;
  for (int k = 0; k < 2; ++k) { c.qk[k] = ws + w.qk[k]; c.qtk[k] = ws + w.qtk[k]; }
  if (x.advantage) { c.v = as_ptrs(x.value); c.vn = ws + w.vn; c.vh = ws + w.vh; c.n_true = d.n_true; }
  if (const char* e = mb_train_critic_launch(c, st)) return e;
  // ---- critic weight gradients + Adam + Polyak ----
  trn::WgradArgs g{}; g.N = N; g.nsplit = ns; g.njobs = 6;
  for (int k = 0; k < 2; ++k) {
    g.job[3 * k + 0] = {c.Dq[k][0], 256, d.rows, d.row_width, ws + w.gq[k][0], ws + w.gq[k][1], 256, S + A};
    g.job[3 * k + 1] = {c.Dq[k][1], 256, c.Hq[k][0], 256, ws + w.gq[k][2], ws + w.gq[k][3], 256, 256};
    g.job[3 * k + 2] = {c.d3[k], 1, c.Hq[k][1], 256, ws + w.gq[k][4], ws + w.gq[k][5], 1, 256};
  }
  if (const char* e = mb_train_wgrad_launch(g, st)) return e;
  trn::AdamArgs ad{}; ad.nsplit = ns; ad.b1 = 0.9f; ad.b2 = 0.999f; ad.eps = 1e-8f; ad.tau = d.tau; ad.njobs = 12;
  ad.zero2 = reinterpret_cast<int*>(ws + w.cnt);
  {
    const double bc1 = 1.0 - pow(0.9, (double)d.t_q), bc2 = 1.0 - pow(0.999, (double)d.t_q);
    ad.lr_over_bc1 = (float)(d.critic_lr / bc1); ad.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
    const int qn[6] = {256 * (S + A), 256, 256 * 256, 256, 256, 1};
    for (int k = 0; k < 2; ++k)
      for (int t = 0; t < 6; ++t) {
        const int li = t >> 1; const bool isw = (t & 1) == 0;
        ad.job[6 * k + t] = {isw ? qs[k]->w[li] : qs[k]->b[li], ws + w.gq[k][t], isw ? qm[k]->w[li] : qm[k]->b[li],
                             isw ? qv[k]->w[li] : qv[k]->b[li], isw ? qts[k]->w[li] : qts[k]->b[li], qn[t]};
      }
  }
  if (const char* e = mb_train_adam_launch(ad, st)) return e;
  // ---- actor: forward through the UPDATED, frozen Q; loss scalars; backward ----
  trn::ActorArgs ac{};
  ac.X = d.rows; ac.N = N; ac.n_true = d.n_true; ac.S = S; ac.A = A; ac.rw = d.row_width; ac.pi = as_ptrs(d.policy);
  ac.q[0] = as_ptrs(d.q1); ac.q[1] = as_ptrs(d.q2); ac.max_action = d.max_action;
  ac.Hp[0] = ws + w.Hp[0]; ac.Hp[1] = ws + w.Hp[1]; ac.api = ws + w.api;
  for (int k = 0; k < 2; ++k) { ac.qv[k] = ws + w.qv[k]; ac.qh[k] = ws + w.qh[k]; ac.gak[k] = ws + w.gak[k]; }
  ac.part = ws + w.part; ac.ntiles_c = (N + TRAIN_TM - 1) / TRAIN_TM; ac.weight = d.weight; ac.out = ws + w.scal;
  ac.counter = reinterpret_cast<int*>(ws + w.cnt);
  ac.scale_q = x.scale_q; ac.branch = branch; ac.n_qh = branch ? N : d.n_true; ac.part_v = x.advantage ? ws + w.partv : nullptr;
  if (const char* e = mb_train_actor_launch(ac, st)) return e;
  trn::PolicyBwdArgs pb{}; pb.N = N; pb.n_true = d.n_true; pb.S = S; pb.A = A; pb.rw = d.row_width; pb.pi = ac.pi;
  pb.Hp[0] = ac.Hp[0]; pb.Hp[1] = ac.Hp[1]; pb.Dp[0] = ws + w.Dp[0]; pb.Dp[1] = ws + w.Dp[1];
  for (int k = 0; k < 2; ++k) { pb.gak[k] = ac.gak[k]; pb.qv[k] = ac.qv[k]; pb.qh[k] = ac.qh[k]; }
  pb.api = ac.api; pb.X = d.rows; pb.bc_coef = d.bc_coef; pb.max_action = d.max_action;
  pb.d3p = ws + w.d3p; pb.part = ws + w.part2; pb.out = ws + w.scal; pb.counter = reinterpret_cast<int*>(ws + w.cnt) + 1;
  pb.vh = x.advantage ? ws + w.vh : nullptr; pb.q_weighted = x.q_weighted;
  if (const char* e = mb_train_policy_bwd_launch(pb, st)) return e;
  trn::WgradArgs gp{}; gp.N = N; gp.nsplit = ns; gp.njobs = 3;
  gp.job[0] = {pb.Dp[0], 256, d.rows, d.row_width, ws + w.gp[0], ws + w.gp[1], 256, S};
  gp.job[1] = {pb.Dp[1], 256, ac.Hp[0], 256, ws + w.gp[2], ws + w.gp[3], 256, 256};
  gp.job[2] = {pb.d3p, A, ac.Hp[1], 256, ws + w.gp[4], ws + w.gp[5], A, 256};
  if (const char* e = mb_train_wgrad_launch(gp, st)) return e;
  trn::AdamArgs ap{}; ap.nsplit = ns; ap.b1 = 0.9f; ap.b2 = 0.999f; ap.eps = 1e-8f; ap.tau = 0.f; ap.njobs = 6;
  {
    const double bc1 = 1.0 - pow(0.9, (double)d.t_pi), bc2 = 1.0 - pow(0.999, (double)d.t_pi);
    ap.lr_over_bc1 = (float)(d.actor_lr / bc1); ap.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
    const int pn[6] = {256 * S, 256, 256 * 256, 256, A * 256, A};
    for (int t = 0; t < 6; ++t) {
      const int li = t >> 1; const bool isw = (t & 1) == 0;
      ap.job[t] = {isw ? d.policy.w[li] : d.policy.b[li], ws + w.gp[t], isw ? d.policy_m.w[li] : d.policy_m.b[li],
                   isw ? d.policy_v.w[li] : d.policy_v.b[li], nullptr, pn[t]};
    }
  }
  if (const char* e = mb_train_adam_launch(ap, st)) return e;
  copy_scalars(x, ws + w.scal, st);
  return nullptr;
}

// ---------------- DARA classifier step / relabel (C ABI: mobody_classifier_step, mobody_dara_relabel) ----------------
struct ClsWs { size_t Xn[2], Hc[2][2], Dc[2][2], d3[2], part, scal, g[2][6], total; int ntiles; };
static ClsWs cls_ws(int N, int S, int A, int nsplit) {
  ClsWs w{}; size_t o = 0;
  auto take = [&](size_t n) { size_t r = o; o += (n + 3) & ~(size_t)3; return r; };
  const int K[2] = {2 * S + A, S + A};
  w.ntiles = (N + 15) / 16;
  for (int k = 0; k < 2; ++k) {
    w.Xn[k] = take((size_t)N * simt::rup16(K[k]));
    for (int l = 0; l < 2; ++l) { w.Hc[k][l] = take((size_t)N * 256); w.Dc[k][l] = take((size_t)N * 256); }
    w.d3[k] = take((size_t)N * 2);
  }
  w.part = take((size_t)w.ntiles * 2); w.scal = take(16);
  for (int k = 0; k < 2; ++k) {
    const size_t n6[6] = {(size_t)256 * K[k], 256, 256 * 256, 256, 2 * 256, 2};
    for (int t = 0; t < 6; ++t) w.g[k][t] = take(n6[t] * nsplit);
  }
  w.total = o;
  return w;
}
long long mb_classifier_workspace_bytes(int N, int S, int A, int nsplit) { return (long long)cls_ws(N, S, A, nsplit).total * 4; }

const char* mb_classifier_step_launch(const mobody_classifier_desc& d, cudaStream_t st) {
  const int N = d.N, S = d.S, A = d.A, ns = d.nsplit;
  if (N < 1 || S < 1 || S > 128 || A < 1 || A > 32 || ns < 1 || ns > 64) return "classifier step: bad N/S/A/nsplit";
  const ClsWs w = cls_ws(N, S, A, ns);
  if (!d.workspace || d.workspace_bytes < (long long)w.total * 4) return "classifier step: workspace too small";
  float* ws = (float*)d.workspace;
  const mobody_mlp_state* nets[2] = {&d.sas, &d.sa};
  const mobody_mlp_state* ms[2] = {&d.sas_m, &d.sa_m};
  const mobody_mlp_state* vs[2] = {&d.sas_v, &d.sa_v};
  trn::ClsArgs c{};
  c.X = d.rows; c.N = N; c.S = S; c.A = A; c.rw = d.row_width; c.label = d.label;
  c.noise[0] = d.noise_sas; c.noise[1] = d.noise_sa; c.std = d.noise_std; c.seed = d.seed; c.draw = d.draw;
  for (int k = 0; k < 2; ++k) {
    c.net[k] = as_ptrs(*nets[k]); c.Xn[k] = ws + w.Xn[k]; c.d3[k] = ws + w.d3[k];
    for (int l = 0; l < 2; ++l) { c.Hc[k][l] = ws + w.Hc[k][l]; c.Dc[k][l] = ws + w.Dc[k][l]; }
  }
  c.part = ws + w.part;
  const int tm = pick_tm(N);
  const size_t bytes = (2 * (size_t)tm * simt::H + (size_t)tm * simt::rup16(2 * S + A) + 4 * tm + 8) * sizeof(float);
  auto kern = tm == 32 ? trn::classifier_kernel<4> : trn::classifier_kernel<2>;
  if (const char* e = set_smem(kern, bytes)) return e;
  const int ntiles = (N + tm - 1) / tm;
  mb_launch(kern, dim3(ntiles), dim3(simt::NT), bytes, st, c);
  mb_launch(trn::cls_scalar_kernel, dim3(1), dim3(32), 0, st, (const float*)c.part, ntiles, N, ws + w.scal);
  const int K[2] = {2 * S + A, S + A};
  trn::WgradArgs g{}; g.N = N; g.nsplit = ns; g.njobs = 6;
  for (int k = 0; k < 2; ++k) {
    g.job[3 * k + 0] = {c.Dc[k][0], 256, c.Xn[k], simt::rup16(K[k]), ws + w.g[k][0], ws + w.g[k][1], 256, K[k]};
    g.job[3 * k + 1] = {c.Dc[k][1], 256, c.Hc[k][0], 256, ws + w.g[k][2], ws + w.g[k][3], 256, 256};
    g.job[3 * k + 2] = {c.d3[k], 2, c.Hc[k][1], 256, ws + w.g[k][4], ws + w.g[k][5], 2, 256};
  }
  if (const char* e = mb_train_wgrad_launch(g, st)) return e;
  trn::AdamArgs ad{}; ad.nsplit = ns; ad.b1 = 0.9f; ad.b2 = 0.999f; ad.eps = 1e-8f; ad.tau = 0.f; ad.njobs = 12;
  const double bc1 = 1.0 - pow(0.9, (double)d.t), bc2 = 1.0 - pow(0.999, (double)d.t);
  ad.lr_over_bc1 = (float)(d.lr / bc1); ad.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
  for (int k = 0; k < 2; ++k) {
    const int n6[6] = {256 * K[k], 256, 256 * 256, 256, 2 * 256, 2};
    for (int t = 0; t < 6; ++t) {
      const int li = t >> 1; const bool isw = (t & 1) == 0;
      ad.job[6 * k + t] = {isw ? nets[k]->w[li] : nets[k]->b[li], ws + w.g[k][t], isw ? ms[k]->w[li] : ms[k]->b[li],
                           isw ? vs[k]->w[li] : vs[k]->b[li], nullptr, n6[t]};
    }
  }
  if (const char* e = mb_train_adam_launch(ad, st)) return e;
  if (d.scalars_out) cudaMemcpyAsync(d.scalars_out, ws + w.scal, 2 * sizeof(float), cudaMemcpyDeviceToDevice, st);
  return nullptr;
}

const char* mb_dara_relabel_launch(float* rows, long long n, int S, int A, int rw, const MlpPtrs& sas, const MlpPtrs& sa,
                                   float coef, float* pen_out, cudaStream_t st) {
  if (n <= 0) return nullptr;
  if (S < 1 || S > 128 || A < 1 || A > 32) return "dara relabel: bad S/A";
  trn::RelabelArgs a{rows, n, S, A, rw, {sas, sa}, coef, pen_out};
  const size_t bytes = (2 * (size_t)64 * simt::H + (size_t)64 * simt::rup16(2 * S + A) + 4 * 64) * sizeof(float);
  if (const char* e = set_smem(trn::dara_relabel_kernel, bytes)) return e;
  long long tiles = (n + 63) / 64;
  int grid = (int)(tiles < 148 * 4 ? tiles : 148 * 4);
  mb_launch(trn::dara_relabel_kernel, dim3(grid), dim3(simt::NT), bytes, st, a);
  return nullptr;
}
