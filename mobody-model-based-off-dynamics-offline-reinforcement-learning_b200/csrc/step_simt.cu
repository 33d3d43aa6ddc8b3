// Fused one-step model rollout, fp32 CUDA-core path ("fp32" precision mode).
//
// One CTA owns a tile of 64 start states and runs, without leaving the SM:
//   [policy MLP]  ->  7 x (state encoder -> action encoder -> latent add -> transition decoder)
//   -> ensemble mean/std, noise, elite pick, next_obs, termination, pairwise-diff penalty
//   -> 7 x reward head -> mean reward - coef * penalty.
// Replaces MOBODYEnsembleDynamics.step (reference algo/dynamics/mobody_dynamics.py:193-265),
// MOBODYModule.forward_trg/forward_src/encode_reward (algo/dynamics/mobody_module.py:217-330)
// and Policy.forward (algo/offline_offline/mobody.py:60-72).  Math: SURVEY.md Appendix A.1.
//
// Activations stay in shared memory ([64][256] fp32 ping-pong); weights are read straight from the
// live nn.Parameter storage ([E,in,out] fp32) and staged in 16-row chunks with cp.async.
// This is the bit-faithful fp32 path; the tcgen05 path (step_tc.cu) is the fast one.
#include "common.cuh"
#include "philox.cuh"
#include "term.cuh"
#include "simt_layers.cuh"

namespace simt {

struct Smem {   // carve-up of dynamic shared memory (floats)
  float *X0, *X1, *Wst, *obs, *act, *nobs, *sas, *sa, *g, *zs, *z, *racc, *pen;
  int ld_obs, ld_sas, ld_sa;
};

__host__ __device__ inline size_t smem_floats(int S, int A, int TM) {
  size_t n = 2 * (size_t)TM * H + 2 * KC * H;
  n += (size_t)TM * rup16(S);                 // obs (padded, zero tail)
  n += (size_t)TM * A;                        // act
  n += (size_t)TM * S;                        // next_obs
  n += (size_t)TM * rup16(2 * S + A);         // sas
  n += (size_t)TM * rup16(MB_LATENT + A);     // [zs, act]
  n += (size_t)TM * MB_ZAH;                   // g
  n += (size_t)TM * MB_LATENT * 2;            // zs, z
  n += (size_t)TM * 2;                        // reward accumulator, penalty
  return n;
}

__device__ inline Smem carve(float* base, int S, int A, int TM) {
  Smem m; float* p = base;
  m.X0 = p; p += TM * H; m.X1 = p; p += TM * H; m.Wst = p; p += 2 * KC * H;
  m.ld_obs = rup16(S); m.obs = p; p += TM * m.ld_obs;
  m.ld_sas = rup16(2 * S + A); m.sas = p; p += TM * m.ld_sas;
  m.ld_sa = rup16(MB_LATENT + A); m.sa = p; p += TM * m.ld_sa;
  m.g = p; p += TM * MB_ZAH; m.zs = p; p += TM * MB_LATENT; m.z = p; p += TM * MB_LATENT;
  m.act = p; p += TM * A; m.nobs = p; p += TM * S; m.racc = p; p += TM; m.pen = p; p += TM;
  return m;
}

// RPT rows per thread: the row tile is 8 * RPT rows (64 by default; 32 for wide observations, S > 64, whose
// [obs | act | next_obs] operands would not fit next to two 64-row activation tiles).
template <int RPT>
__global__ void __launch_bounds__(NT, 1)
step_kernel(StepArgs a, DynPtrs dp, MlpPtrs pol, int has_policy) {
  constexpr int TM = 8 * RPT, TPR = NT / TM;        // rows per CTA, threads per row in the per-row phases
  extern __shared__ __align__(16) float smem_f[];
  const int S = a.S, A = a.A, B = a.B;
  const int live = a.n_rows_dev ? min(*a.n_rows_dev, B) : B;
  const int row0 = blockIdx.x * TM;
  if (row0 >= live) return;                   // whole CTA exits together
  Smem m = carve(smem_f, S, A, TM);
  const int tid = threadIdx.x;
  const int rows = min(TM, live - row0);

  // ---- load obs tile (zero padded), action tile ----
  for (int i = tid; i < TM * m.ld_obs; i += NT) {
    int r = i / m.ld_obs, j = i - r * m.ld_obs;
    m.obs[i] = (r < rows && j < S) ? a.obs[(size_t)(row0 + r) * a.obs_ld + j] : 0.0f;
  }
  if (!has_policy)
    for (int i = tid; i < TM * A; i += NT) {
      int r = i / A, j = i - r * A;
      m.act[i] = (r < rows) ? a.act[(size_t)(row0 + r) * a.act_ld + j] : 0.0f;
    }
  __syncthreads();
  if (has_policy) {   // Policy.forward: relu MLP, tanh * max_action  (mobody.py:35-72)
    big_layer<true, RPT>(m.obs, m.ld_obs, S, pol.w[0], pol.b[0], m.X0, m.Wst, ACT_RELU);
    big_layer<true, RPT>(m.X0, H, H, pol.w[1], pol.b[1], m.X1, m.Wst, ACT_RELU);
    small_layer<true, RPT>(m.X1, H, H, pol.w[2], H, pol.b[2], A, m.act, A, ACT_TANH, a.max_action);
  }
  if (a.act_out)
    for (int i = tid; i < rows * A; i += NT) a.act_out[(size_t)row0 * A + i] = m.act[i];

  // [zs | act | 0-pad] operand of the action encoder: the act part is member independent
  for (int i = tid; i < TM * m.ld_sa; i += NT) {
    int r = i / m.ld_sa, j = i - r * m.ld_sa;
    m.sa[i] = (j >= MB_LATENT && j < MB_LATENT + A) ? m.act[r * A + (j - MB_LATENT)] : 0.0f;
  }
  __syncthreads();

  const int za1 = a.use_trg ? L_ZATRG1 : L_ZASRC1, za2 = a.use_trg ? L_ZATRG2 : L_ZASRC2;
  // ---- 7 members: forward_trg / forward_src (mobody_module.py:315-330) ----
  for (int e = 0; e < MB_E; ++e) {
    big_layer<false, RPT>(m.obs, m.ld_obs, S, dp.w[L_ZS1] + (size_t)e * S * H, dp.b[L_ZS1] + e * H, m.X0, m.Wst, ACT_SWISH);
    big_layer<false, RPT>(m.X0, H, H, dp.w[L_ZS2] + (size_t)e * H * H, dp.b[L_ZS2] + e * H, m.X1, m.Wst, ACT_SWISH);
    // zs3: only the mu half (first 16 of 32 columns) is used at inference (:223-225, 237-243)
    small_layer<false, RPT>(m.X1, H, H, dp.w[L_ZS3] + (size_t)e * H * 2 * MB_LATENT, 2 * MB_LATENT,
                       dp.b[L_ZS3] + e * 2 * MB_LATENT, MB_LATENT, m.zs, MB_LATENT, ACT_NONE, 1.f);
    for (int i = tid; i < TM * MB_LATENT; i += NT) m.sa[(i >> 4) * m.ld_sa + (i & 15)] = m.zs[i];
    __syncthreads();
    small_layer<false, RPT>(m.sa, m.ld_sa, MB_LATENT + A, dp.w[za1] + (size_t)e * (MB_LATENT + A) * MB_ZAH, MB_ZAH,
                       dp.b[za1] + e * MB_ZAH, MB_ZAH, m.g, MB_ZAH, ACT_SWISH, 1.f);
    small_layer<false, RPT>(m.g, MB_ZAH, MB_ZAH, dp.w[za2] + (size_t)e * MB_ZAH * 2 * MB_LATENT, 2 * MB_LATENT,
                       dp.b[za2] + e * 2 * MB_LATENT, MB_LATENT, m.z, MB_LATENT, ACT_NONE, 1.f);
    for (int i = tid; i < TM * MB_LATENT; i += NT) m.z[i] = m.zs[i] + m.z[i];      // z_ns = zs + za
    __syncthreads();
    big_layer<false, RPT>(m.z, MB_LATENT, MB_LATENT, dp.w[L_T1] + (size_t)e * MB_LATENT * H, dp.b[L_T1] + e * H, m.X0, m.Wst, ACT_SWISH);
    big_layer<false, RPT>(m.X0, H, H, dp.w[L_T2] + (size_t)e * H * H, dp.b[L_T2] + e * H, m.X1, m.Wst, ACT_SWISH);
    // transition3 -> mean[e] ; staged through nobs then written to global (info['samples'])
    small_layer<false, RPT>(m.X1, H, H, dp.w[L_T3] + (size_t)e * H * S, S, dp.b[L_T3] + e * S, S, m.nobs, S, ACT_NONE, 1.f);
    for (int i = tid; i < rows * S; i += NT) a.mean[((size_t)e * B + row0) * S + i] = m.nobs[i];
    __syncthreads();
  }

  // ---- ensemble statistics, noise, pick, penalty (mobody_dynamics.py:218-259) ----
  {
    const int r = tid / TPR, q = tid % TPR;  // TPR threads per row; thread q owns dim blocks q, q+TPR, ...
    float d2[MB_E];
#pragma unroll
    for (int e = 0; e < MB_E; ++e) d2[e] = 0.f;
    int member = 0;
    if (r < rows) {
      const unsigned long long grow = a.row_ids ? (unsigned long long)a.row_ids[row0 + r]
                                                : a.row0 + (unsigned long long)(row0 + r);
      if (a.idx) member = (int)a.idx[row0 + r];
      else member = (int)a.elites[philox_elite_slot(a.seed, a.step, grow, a.n_elites)];
      for (int blk = q; blk * 4 < S; blk += TPR) {
        float nrm[4] = {0.f, 0.f, 0.f, 0.f};
        if (!a.eps) philox_normal4(philox_noise_block(a.seed, a.step, grow, (unsigned)blk), nrm);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          int j = blk * 4 + t;
          if (j >= S) break;
          float mv[MB_E], sum = 0.f;
#pragma unroll
          for (int e = 0; e < MB_E; ++e) { mv[e] = a.mean[((size_t)e * B + row0 + r) * S + j]; sum += mv[e]; }
          float mbar = sum / (float)MB_E, ss = 0.f, mk = 0.f;
#pragma unroll
          for (int e = 0; e < MB_E; ++e) {
            float d = mv[e] - mbar; ss = fmaf(d, d, ss);
            if (j < S - 1) d2[e] = fmaf(d, d, d2[e]);      // quirk: last state dim excluded (:246)
            if (e == member) mk = mv[e];
          }
          float sd = sqrtf(ss / (float)(MB_E - 1));         // unbiased, shared by all members (:218)
          float ep = a.eps ? a.eps[((size_t)member * B + row0 + r) * S + j] : nrm[t];
          m.nobs[r * S + j] = mk + ep * sd;                 // sample of the picked member (:220-226)
        }
      }
    }
    float pmax = 0.f;
#pragma unroll
    for (int e = 0; e < MB_E; ++e) {
      float v = d2[e];
#pragma unroll
      for (int o = 1; o < TPR; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      pmax = fmaxf(pmax, sqrtf(v));
    }
    if (q == 0) { m.pen[r] = pmax; m.racc[r] = 0.f; }
  }
  __syncthreads();
  for (int i = tid; i < rows * S; i += NT) a.next_obs[(size_t)row0 * S + i] = m.nobs[i];
  if (tid < rows) a.terminal[row0 + tid] = (unsigned char)mb_terminal(a.term_kind, m.nobs + tid * S, S);
  // sas = [obs, act, next_obs, 0-pad]  (mobody_module.py:296)
  for (int i = tid; i < TM * m.ld_sas; i += NT) {
    int r = i / m.ld_sas, j = i - r * m.ld_sas;
    float v = 0.f;
    if (r < rows) {
      if (j < S) v = m.obs[r * m.ld_obs + j];
      else if (j < S + A) v = m.act[r * A + (j - S)];
      else if (j < 2 * S + A) v = m.nobs[r * S + (j - S - A)];
    }
    m.sas[i] = v;
  }
  __syncthreads();

  // ---- reward head, all 7 members (mobody_module.py:295-302; mean over members :236) ----
  for (int e = 0; e < MB_E; ++e) {
    big_layer<false, RPT>(m.sas, m.ld_sas, 2 * S + A, dp.w[L_R1] + (size_t)e * (2 * S + A) * H, dp.b[L_R1] + e * H, m.X0, m.Wst, ACT_SWISH);
    big_layer<false, RPT>(m.X0, H, H, dp.w[L_R2] + (size_t)e * H * H, dp.b[L_R2] + e * H, m.X1, m.Wst, ACT_SWISH);
    // reward_model3 column 0 (mu); column 1 (logvar) is discarded by step() (:235)
    {
      const int r = tid / TPR, q = tid % TPR;
      const float* w = dp.w[L_R3] + (size_t)e * H * 2;
      const float* x = m.X1 + r * H;
      float s = 0.f;
      for (int k = q; k < H; k += TPR) s = fmaf(x[k], __ldg(w + 2 * k), s);
#pragma unroll
      for (int o = 1; o < TPR; o <<= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (q == 0) m.racc[r] += s + __ldg(dp.b[L_R3] + e * 2);
    }
    __syncthreads();
  }
  if (tid < rows) {
    float raw = m.racc[tid] / (float)MB_E, pen = m.pen[tid];
    if (a.raw_reward) a.raw_reward[row0 + tid] = raw;
    a.penalty[row0 + tid] = pen;
    a.reward[row0 + tid] = (a.coef != 0.f && a.use_penalty) ? raw - a.coef * pen : raw;   // :261-263
  }
}

// Policy forward only: select_action (mobody.py:138-144).
__global__ void __launch_bounds__(NT, 1)
policy_kernel(const float* __restrict__ obs, int B, int S, int A, MlpPtrs pol, float max_action, float* __restrict__ act_out) {
  constexpr int RPT = 8;
  extern __shared__ __align__(16) float smem_f[];
  float* X0 = smem_f; float* X1 = X0 + TM * H; float* Wst = X1 + TM * H;
  const int ld = rup16(S);
  float* o = Wst + 2 * KC * H; float* act = o + TM * ld;
  const int tid = threadIdx.x, row0 = blockIdx.x * TM, rows = min(TM, B - row0);
  for (int i = tid; i < TM * ld; i += NT) {
    int r = i / ld, j = i - r * ld;
    o[i] = (r < rows && j < S) ? obs[(size_t)(row0 + r) * S + j] : 0.0f;
  }
  __syncthreads();
  big_layer<true, RPT>(o, ld, S, pol.w[0], pol.b[0], X0, Wst, ACT_RELU);
  big_layer<true, RPT>(X0, H, H, pol.w[1], pol.b[1], X1, Wst, ACT_RELU);
  small_layer<true, RPT>(X1, H, H, pol.w[2], H, pol.b[2], A, act, A, ACT_TANH, max_action);
  for (int i = tid; i < rows * A; i += NT) act_out[(size_t)row0 * A + i] = act[i];
}

}  // namespace simt

// ---- host launchers (called from api.cu) ----
const char* mb_simt_step_launch(const StepArgs& a, const DynPtrs& dp, const MlpPtrs* pol, cudaStream_t st) {
  if (a.B <= 0) return nullptr;
  if (a.S < 2 || a.S > 128 || a.A < 1 || a.A > 32) return "fp32 step kernel supports 2 <= S <= 128, 1 <= A <= 32";
  // 64-row tiles, or 32-row tiles where 64 rows of operands exceed the shared-memory budget (observations wider than
  // about 40 columns: the [s, a, s'] plane of the reward model grows with 2S+A)
  const int tm = simt::smem_floats(a.S, a.A, 64) * sizeof(float) <= 227 * 1024 ? 64 : 32;
  size_t bytes = simt::smem_floats(a.S, a.A, tm) * sizeof(float);
  if (bytes > 227 * 1024) return "fp32 step kernel: shared memory budget exceeded for this (S, A)";
  auto kern = tm == 64 ? simt::step_kernel<8> : simt::step_kernel<4>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
    return "cudaFuncSetAttribute(step_kernel) failed";
  MlpPtrs none{};
  int grid = (a.B + tm - 1) / tm;
  kern<<<grid, simt::NT, bytes, st>>>(a, dp, pol ? *pol : none, pol ? 1 : 0);
  return nullptr;
}

const char* mb_simt_policy_launch(const float* obs, int B, int S, int A, const MlpPtrs& pol, float max_action,
                                  float* act_out, cudaStream_t st) {
  if (B <= 0) return nullptr;
  if (S < 1 || S > 128 || A < 1 || A > 64) return "policy kernel supports S <= 128, A <= 64";
  size_t bytes = (2 * (size_t)simt::TM * simt::H + 2 * simt::KC * simt::H + (size_t)simt::TM * simt::rup16(S) +
                  (size_t)simt::TM * A) * sizeof(float);
  static size_t configured = 0;
  if (bytes > configured) {
    if (cudaFuncSetAttribute(simt::policy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
      return "cudaFuncSetAttribute(policy_kernel) failed";
    configured = bytes;
  }
  int grid = (B + simt::TM - 1) / simt::TM;
  simt::policy_kernel<<<grid, simt::NT, bytes, st>>>(obs, B, S, A, pol, max_action, act_out);
  return nullptr;
}
