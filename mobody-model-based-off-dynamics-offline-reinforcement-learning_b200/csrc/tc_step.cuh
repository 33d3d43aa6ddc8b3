// Code shared by the three tensor-core rollout step kernels (step_tc.cu: one 128-row tile per CTA; step_duo.cu: two
// 128-row tiles per CTA; step_wide.cu: one 64-row tile per CTA).  The kernels differ in their MMA issue, GEMM epilogues,
// shared-memory carve-up and stage sizing; what is here is the same in all of them:
//  * host: the per-tile layer schedule (TcSched) and the launch with the weight image persisting in L2;
//  * device: the producer's bias staging, and everything after transition3's means -- member pick, ensemble statistics,
//    noise, penalty, termination, the [s | a | s'] operand of the reward head and the final reward write.  One copy of
//    the reference semantics (noise counter, elite pick, the penalty's "last dim excluded" quirk) for every mode.
#pragma once
#include "common.cuh"
#include "philox.cuh"
#include "term.cuh"
#include "tc_prims.cuh"
#include "tc_layout.h"
#include "tc_epi.cuh"
#include <utility>

namespace tst {
using namespace tce;

constexpr int NB = 4;                    // bias ring slots (one layer's bias each)
constexpr int BSLOT = 528;               // floats per slot: 256 bias + reward_model3 vector (272) behind reward_model2's bias

// ---------------- host ----------------

// Layer schedule of one step: [policy 3 layers] + 7 x 8 dynamics layers + 7 x 2 reward layers.  `cw` is the number of
// accumulator columns per operand chunk the kernel's epilogue announces (32, 64, or 256 = a whole layer); a layer's a_wait
// counts the chunks of its A operand that it waits for.  The policy blob's bias base is returned in *pol_bias_base.
static inline TcSched tc_step_sched(const StepArgs& a, int ns, bool has_policy, int cw, uint32_t* pol_bias_base) {
  const int S = a.S, A = a.A;
  const int wide = 256 / cw, sas = (tc_rup16(2 * S + A) + cw - 1) / cw;   // chunks of a 256-wide / the [s | a | s'] operand
  const TcDynLayout DL = tc_dyn_layout(S, A, ns);
  TcSched sc{}; int n = 0;
  auto add = [&](size_t w_off, uint32_t b_off, const TcGeom& g, int region, int a_wait, int kind, int blob) {
    TcLayer& L = sc.L[n++];
    L.w_off = (uint32_t)w_off; L.b_off = b_off; L.ksteps = (uint16_t)(g.Kp / 16); L.n = (uint16_t)g.Np;
    L.a_region = (uint8_t)region; L.a_wait = (uint8_t)a_wait; L.kind = (uint8_t)kind; L.blob = (uint8_t)blob;
  };
  if (has_policy) {
    const TcMlpLayout PL = tc_mlp_layout(S, A, ns);
    add(PL.w_off[0], PL.b_off[0], PL.g[0], REG_OBS, 1, EPI_RELU256, 1);
    add(PL.w_off[1], PL.b_off[1], PL.g[1], REG_MAIN, wide, EPI_RELU256, 1);
    add(PL.w_off[2], PL.b_off[2], PL.g[2], REG_MAIN, wide, EPI_ACTION, 1);
    *pol_bias_base = (uint32_t)PL.bias_base;
  }
  sc.first_dyn = n;
  const int za1 = a.use_trg ? PK_ZATRG1 : PK_ZASRC1, za2 = a.use_trg ? PK_ZATRG2 : PK_ZASRC2;
  for (int e = 0; e < MB_E; ++e) {
    const size_t wb = (size_t)e * DL.member_w_bytes; const uint32_t bb = (uint32_t)e * DL.member_b_floats;
    auto lay = [&](int pk, int region, int a_wait, int kind) { add(wb + DL.w_off[pk], bb + DL.b_off[pk], tc_dyn_geom(pk, S, A), region, a_wait, kind, 0); };
    lay(PK_ZS1, REG_OBS, (e == 0 && !has_policy) ? 1 : 0, EPI_SWISH256);   // obs is announced once, by the prologue
    lay(PK_ZS2, REG_MAIN, wide, EPI_SWISH256);
    lay(PK_ZS3, REG_MAIN, wide, EPI_ZS);
    lay(za1, REG_SA, 1, EPI_G);
    lay(za2, REG_MAIN, 1, EPI_Z);
    lay(PK_T1, REG_MAIN, 1, EPI_SWISH256);
    lay(PK_T2, REG_MAIN, wide, EPI_SWISH256);
    lay(PK_T3, REG_MAIN, wide, EPI_MEAN);
  }
  for (int e = 0; e < MB_E; ++e) {   // [s | a | s'] is announced once, by the statistics phase
    const size_t wb = (size_t)e * DL.member_w_bytes; const uint32_t bb = (uint32_t)e * DL.member_b_floats;
    add(wb + DL.w_off[PK_R1], bb + DL.b_off[PK_R1], tc_dyn_geom(PK_R1, S, A), REG_SAS, e == 0 ? sas : 0, EPI_SWISH256, 0);
    add(wb + DL.w_off[PK_R2], bb + DL.b_off[PK_R2], tc_dyn_geom(PK_R2, S, A), REG_MAIN, wide, EPI_REWARD, 0);
  }
  sc.n_layers = n;
  return sc;
}

// Whether `scratch_bytes` of operand planes hold tc_stats's scratch for a tile of tm rows: next states, member picks and at
// least one member's squared deviations (a member batch of 0 would never finish).
static inline bool tc_stats_scratch_fits(size_t scratch_bytes, int tm, int S) { return scratch_bytes / 4 >= (size_t)2 * (tm * S + tm); }

// Launch with the dynamics weight image [window, window + window_bytes) marked persisting in L2: every tile streams the
// whole image (6.5 MB at obs 17 / act 6, 9.2 MB at obs 111 / act 8) from L2, and the rows flowing through L2 -- the
// kernel's own I/O and, on a multi-GPU box, the peers' incoming transitions -- must not evict it.
template <typename... KArgs, typename... Args>
static cudaError_t tc_launch_persisting(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                        const void* window, size_t window_bytes, Args&&... args) {
  static thread_local int limit_dev = -1;
  int dev = 0; cudaGetDevice(&dev);
  if (limit_dev != dev) { cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)32 << 20); limit_dev = dev; }
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeAccessPolicyWindow;
  at[0].val.accessPolicyWindow.base_ptr = const_cast<void*>(window);
  at[0].val.accessPolicyWindow.num_bytes = window_bytes;
  at[0].val.accessPolicyWindow.hitRatio = 1.0f;
  at[0].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
  at[0].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  cudaLaunchConfig_t lc = {};
  lc.gridDim = grid; lc.blockDim = block; lc.dynamicSmemBytes = smem; lc.stream = st;
  lc.attrs = at; lc.numAttrs = 1;
  return cudaLaunchKernelEx(&lc, kern, std::forward<Args>(args)...);
}

// ---------------- device: producer warp ----------------

// Layer li's bias (and reward_model3's vector right behind reward_model2's bias) -> bias ring slot li % NB
__device__ __forceinline__ void tc_stage_bias(int li, const TcLayer& L, const unsigned char* dynb, const unsigned char* polb,
                                              uint32_t dyn_bias_base, uint32_t pol_bias_base, float* bias_s,
                                              uint64_t* b_full, uint64_t* b_empty) {
  const int slot = li & (NB - 1);
  const float* bsrc = reinterpret_cast<const float*>(L.blob ? polb + pol_bias_base : dynb + dyn_bias_base) + L.b_off;
  const uint32_t bb = (L.kind == EPI_REWARD ? (uint32_t)BSLOT : (uint32_t)L.n) * 4u;
  tc::mbar_wait(&b_empty[slot], (uint32_t)(((li / NB) & 1) ^ 1));
  tc::mbar_arrive_expect_tx(&b_full[slot], bb);
  tc::bulk_g2s(bias_s + slot * BSLOT, bsrc, bb, &b_full[slot]);
}

// ---------------- device: epilogue warps, after the last dynamics GEMM of a tile ----------------
// A tile of TM rows (global rows row0 ..), EPI_WARPS epilogue warps (threads 0 .. 32 * EPI_WARPS - 1), SLOTS threads per
// row: thread `slot` of row r.  Every dynamics MMA of the tile has completed, so the kernel hands over operand planes as
// fp32 scratch: [TM * S] next states (nobs_s) | [TM] member picks | [TM] pad | member batches of squared deviations.

// Member pick, ensemble statistics, noise and next state.  The picked member of every row (injected idx, or the Philox
// pick among the elites) goes to member_s.  After the epilogue barrier (every mean column of the tile has been written,
// member_s is visible) the loop runs element-wise over the tile's contiguous [TM x S] block of every member (coalesced
// loads; there is no L1 to speak of next to ~227 KB of shared memory), all epilogue threads in flight, and writes next_obs
// and nobs_s.  Per-row sums of squared deviations go through the scratch in member batches and are added in a fixed order
// (deterministic).  Returns this thread's share of row r's penalty max (0 for the others).
// Row is int or size_t, whichever the kernel keeps its row indices in.  stamp(k) is a debug trace hook, called at point 0
// (before the pick) and 1 (after its barrier) of the phase; tc_penalty_terminal calls stamp(3).
template <int TM, int EPI_WARPS, int SLOTS, typename Row, typename Stamp>
__device__ __forceinline__ float tc_stats(const StepArgs& a, int S, int B, Row row0, int live, int r, int slot, bool valid,
                                          float* nobs_s, uint32_t scratch_bytes, Stamp stamp) {
  constexpr int NEPI = 32 * EPI_WARPS;
  const int n_el = TM * S;
  int* member_s = reinterpret_cast<int*>(nobs_s + n_el);            // [TM]      picked member per row
  float* dsq_s = reinterpret_cast<float*>(member_s + TM) + TM;      // [batch][TM*S] squared deviations
  const int scratch_floats = (int)(scratch_bytes / 4) - n_el - 2 * TM;
  const int mbatch = min(MB_E, scratch_floats / n_el);
  const int etid = threadIdx.x;                                     // epilogue threads are 0 .. NEPI-1
  stamp(0);
  if (etid < TM) {
    int mem = 0;
    if (row0 + etid < (Row)live) {
      const size_t gr = (size_t)row0 + etid;
      const unsigned long long gid = a.row_ids ? (unsigned long long)a.row_ids[gr] : a.row0 + gr;
      mem = a.idx ? (int)a.idx[gr] : (int)a.elites[philox_elite_slot(a.seed, a.step, gid, a.n_elites)];
    }
    member_s[etid] = mem;
  }
  epi_bar<EPI_WARPS>();
  stamp(1);
  float row_pmax = 0.f;
  for (int e0 = 0; e0 < MB_E; e0 += mbatch) {
#pragma unroll 1   // one code path for every element: a row's result must not depend on its position in the tile
    for (int i = etid; i < n_el; i += NEPI) {
      const int rr = i / S, j = i - rr * S;
      const size_t gr = (size_t)row0 + rr;
      if (row0 + rr < (Row)live) {
        float mv[MB_E], sum = 0.f;
#pragma unroll
        for (int e = 0; e < MB_E; ++e) { mv[e] = a.mean[((size_t)e * B + row0) * S + i]; sum += mv[e]; }
        const float mbar = sum / (float)MB_E;
        const int member = member_s[rr];
        float ss = 0.f, mk = 0.f;
#pragma unroll
        for (int e = 0; e < MB_E; ++e) {
          const float d = mv[e] - mbar, dd = __fmul_rn(d, d);    // explicit roundings (no contraction choices)
          ss = __fadd_rn(ss, dd);
          if (e >= e0 && e < e0 + mbatch) dsq_s[(e - e0) * n_el + i] = (j < S - 1) ? dd : 0.f;   // quirk: last dim excluded (:246)
          if (e == member) mk = mv[e];
        }
        if (e0 == 0) {
          const float sd = sqrtf(ss / (float)(MB_E - 1));
          float ep;
          if (a.eps) ep = a.eps[((size_t)member * B + gr) * S + j];
          else {
            const unsigned long long gid = a.row_ids ? (unsigned long long)a.row_ids[gr] : a.row0 + gr;
            ep = philox_normal1(philox_noise_block(a.seed, a.step, gid, (unsigned)(j >> 2)), j & 3);
          }
          const float nv = __fmaf_rn(ep, sd, mk);
          a.next_obs[(size_t)row0 * S + i] = nv;
          nobs_s[i] = nv;
        }
      }
    }
    epi_bar<EPI_WARPS>();
    // (row, member) sums in a fixed order; slot s takes members s, s + SLOTS, ... of its row r
    if (valid) {
      for (int e = slot; e < mbatch && e0 + e < MB_E; e += SLOTS) {
        const float* p = dsq_s + e * n_el + r * S;
        float v0 = 0.f, v1 = 0.f;
        int j = 0;
        for (; j + 2 <= S - 1; j += 2) { v0 += p[j]; v1 += p[j + 1]; }
        if (j < S - 1) v0 += p[j];
        row_pmax = fmaxf(row_pmax, sqrtf(v0 + v1));
      }
    }
    if (e0 + mbatch < MB_E) epi_bar<EPI_WARPS>();   // dsq_s is rewritten by the next batch
  }
  return row_pmax;
}

// Row r's penalty (max over the SLOTS shares, through red[SLOTS][TM]) and its terminal flag.  Returns the penalty in slot
// 0 of a valid row, 0 elsewhere.
template <int TM, int EPI_WARPS, int SLOTS, typename Stamp>
__device__ __forceinline__ float tc_penalty_terminal(const StepArgs& a, int S, float row_pmax, float* red, int r, int slot,
                                                     bool valid, size_t grow, const float* nobs_s, Stamp stamp) {
  red[slot * TM + r] = row_pmax;
  if (slot == 0 && valid) a.terminal[grow] = (unsigned char)mb_terminal(a.term_kind, nobs_s + r * S, S);
  epi_bar<EPI_WARPS>();
  stamp(3);
  float pm = 0.f;
  if (slot == 0 && valid) {
#pragma unroll
    for (int s2 = 0; s2 < SLOTS; ++s2) pm = fmaxf(pm, red[s2 * TM + r]);
  }
  return pm;
}

// sas = [obs, act, next_obs, 0-pad] operand of the reward head (mobody_module.py:296), K groups slot, slot + SLOTS, ... of
// row r; put(kg, v) stores the 8 values of K group kg in the kernel's operand format.  Ends with the async-proxy fence.
template <int SLOTS, typename Put8>
__device__ __forceinline__ void tc_sas_operand(const StepArgs& a, int S, int A, bool has_policy, int sas_kp, int r, int slot,
                                               bool valid, size_t grow, const float* nobs_s, Put8 put) {
  const float* actp = has_policy ? a.act_out : a.act;
  const int act_ld = has_policy ? A : a.act_ld;
  for (int kg = slot; kg < sas_kp / 8; kg += SLOTS) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int k = kg * 8 + i;
      float t = 0.f;
      if (valid) {
        if (k < S) t = __ldg(a.obs + grow * a.obs_ld + k);
        else if (k < S + A) t = actp[grow * act_ld + (k - S)];
        else if (k < 2 * S + A) t = nobs_s[r * S + (k - S - A)];
      }
      v[i] = t;
    }
    put(kg, v);
  }
  tc::fence_proxy_async_smem();
}

// raw_reward (mean of the members' reward heads), penalty and reward of one row (mobody_dynamics.py:236, :261-263)
__device__ __forceinline__ void tc_write_reward(const StepArgs& a, size_t grow, float racc, float pen) {
  const float raw = racc / (float)MB_E;
  if (a.raw_reward) a.raw_reward[grow] = raw;
  a.penalty[grow] = pen;
  a.reward[grow] = (a.coef != 0.f && a.use_penalty) ? raw - a.coef * pen : raw;
}

}  // namespace tst
