// Fused one-step model rollout on the tensor cores for wide observations (65 <= S <= 128, 1 <= A <= 32), sm_100a.
//
// Sibling of step_tc.cu with the same arithmetic (bf16 hi+lo split of both operands, 3 MMAs per K step, inside the 1e-4
// bound; swish layers pre-scaled by the packer) and the same packed weight images (mobody_dyn_pack / mobody_mlp_pack with
// two planes).  What changes is the row tile: one CTA owns 64 rows (UMMA M = 64), so every operand plane is half the size
// of step_tc.cu's and the planes of S <= 128, A <= 32 (the [s | a | s'] plane of the reward model reaches K = 288) fit in
// shared memory next to a weight ring of at least 4 stages (DESIGN.md 4.1c).
//
//  * producer warp: per layer, its bias (ring of NB slots) and one K step of both weight planes per stage (1-D TMA bulk
//    copies, mbarrier complete_tx);
//  * MMA warp: one elected thread issues tcgen05.mma 64 x N x 16 into TMEM (two 256-column accumulators, ping-pong);
//  * 16 epilogue warps (4 groups x 4 TMEM lane quadrants).  An M = 64 accumulator puts row i in TMEM lane
//    32 * (i / 16) + i % 16, so quadrant q holds rows 16q .. 16q+15 in its first 16 lanes.  tcgen05.ld 16x32bx2 gives
//    thread `lane` row 16q + lane % 16 and, per 64-column chunk, the 8 columns group * 16 + (lane / 16) * 8: one K group
//    of the next layer's operand per thread and chunk.  The 8 threads of a row (4 groups x 2 halves) are its `slot`s.
//    Chunks are announced in order (one mbarrier per 64 columns) and the next layer's MMAs trail the epilogue by a chunk.
#include "common.cuh"
#include "philox.cuh"
#include "term.cuh"
#include "tc_prims.cuh"
#include "tc_layout.h"
#include "tc_epi.cuh"

namespace tcw {
using namespace tce;

constexpr int TM = 64;                   // rows per CTA (UMMA M)
constexpr int NS = 2;                    // bf16 hi + lo planes
constexpr int NG = 4;                    // epilogue groups of 4 warps (one warp per TMEM lane quadrant)
constexpr int SLOTS = 2 * NG;            // epilogue threads per row
constexpr int CHUNK = 64;                // accumulator columns per announced chunk
constexpr uint32_t KG = TM * 16;         // bytes of one 8-wide K group of one plane (64 rows x 8 x bf16)
constexpr uint32_t MAIN_PLANE = 32 * KG; // 64 rows x 256 k x bf16
constexpr int MAX_NST = 12;
constexpr int NB = 4;                    // bias ring slots (one layer's bias each)
constexpr int BSLOT = 528;               // floats per slot: 256 bias + reward_model3 vector (272) behind reward_model2's bias
constexpr int NCHUNK = 5;                // announced chunks: 4 of a 256-wide layer, 5 of the widest [s | a | s'] plane (K 288)

struct Cfg {
  int nst;
  uint32_t stage_bytes, small_plane, sa_off, obs_kp, sa_kp, sas_kp;
  uint32_t dyn_bias_base, pol_bias_base;
  int has_policy;
};

struct Bars {
  uint64_t w_full[MAX_NST], w_empty[MAX_NST], a_ready[NCHUNK], d_full[2], d_empty[2], b_full[NB], b_empty[NB];
  uint32_t tmem_slot, pad;
};

__global__ void __launch_bounds__(32 * (4 * NG + 2), 1)
step_wide_kernel(const StepArgs a, const unsigned char* __restrict__ dynb, const unsigned char* __restrict__ polb,
                 const __grid_constant__ TcSched sched, const Cfg cfg) {
  constexpr int EPI_WARPS = 4 * NG, PROD_WARP = EPI_WARPS, MMA_WARP = EPI_WARPS + 1;
  extern __shared__ __align__(128) unsigned char smem[];
  const int S = a.S, A = a.A, B = a.B;
  const int live = a.n_rows_dev ? min(*a.n_rows_dev, B) : B;
  const int row0 = blockIdx.x * TM;
  if (row0 >= live) return;

  unsigned char* A_main = smem;
  unsigned char* A_small = A_main + NS * MAIN_PLANE;
  unsigned char* wst = A_small + NS * cfg.small_plane;
  float* red = reinterpret_cast<float*>(wst + (size_t)cfg.nst * cfg.stage_bytes);      // [2][SLOTS][64]
  float* bias_s = red + 2 * SLOTS * TM;                                                // [NB][BSLOT]
  Bars* bars = reinterpret_cast<Bars*>(bias_s + NB * BSLOT);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    for (int i = 0; i < cfg.nst; ++i) { tc::mbar_init(&bars->w_full[i], 1); tc::mbar_init(&bars->w_empty[i], 1); }
    for (int i = 0; i < NCHUNK; ++i) tc::mbar_init(&bars->a_ready[i], EPI_WARPS);   // every epilogue warp announces every chunk
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&bars->d_full[i], 1); tc::mbar_init(&bars->d_empty[i], EPI_WARPS); }
    for (int i = 0; i < NB; ++i) { tc::mbar_init(&bars->b_full[i], 1); tc::mbar_init(&bars->b_empty[i], EPI_WARPS); }
    tc::mbar_fence_init();
  }
  if (warp == PROD_WARP) tc::tmem_alloc(&bars->tmem_slot, 512);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = bars->tmem_slot;

  if (warp == PROD_WARP) {
    // ================= weight producer: L2 -> SMEM ring, one K step (both planes) per stage =================
    if (tc::elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int li = 0; li < sched.n_layers; ++li) {
        const TcLayer L = sched.L[li];
        const unsigned char* src = (L.blob ? polb : dynb) + L.w_off;
        const uint32_t bytes = (uint32_t)NS * L.n * 32u;
        {   // this layer's bias (and reward_model3's vector right behind reward_model2's bias) -> bias ring slot li % NB
          const int slot = li & (NB - 1);
          const float* bsrc = reinterpret_cast<const float*>(L.blob ? polb + cfg.pol_bias_base : dynb + cfg.dyn_bias_base) + L.b_off;
          const uint32_t bb = (L.kind == EPI_REWARD ? (uint32_t)BSLOT : (uint32_t)L.n) * 4u;
          tc::mbar_wait(&bars->b_empty[slot], (uint32_t)(((li / NB) & 1) ^ 1));
          tc::mbar_arrive_expect_tx(&bars->b_full[slot], bb);
          tc::bulk_g2s(bias_s + slot * BSLOT, bsrc, bb, &bars->b_full[slot]);
        }
        for (int s = 0; s < L.ksteps; ++s) {
          tc::mbar_wait(&bars->w_empty[stage], phase ^ 1u);
          tc::mbar_arrive_expect_tx(&bars->w_full[stage], bytes);
          tc::bulk_g2s(wst + (size_t)stage * cfg.stage_bytes, src + (size_t)s * bytes, bytes, &bars->w_full[stage]);
          if (++stage == cfg.nst) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == MMA_WARP) {
    // ================= MMA issuer =================
    if (tc::elect_one()) {
      int stage = 0; uint32_t wphase = 0, aph = 0;
      const uint32_t small0 = tc::smem_u32(A_small), main0 = tc::smem_u32(A_main), wst0 = tc::smem_u32(wst);
      for (int li = 0; li < sched.n_layers; ++li) {
        const TcLayer L = sched.L[li];
        const int buf = li & 1;
        const uint32_t dcol = tmem + (uint32_t)buf * 256u;
        if (li >= 2) tc::mbar_wait(&bars->d_empty[buf], (uint32_t)(((li >> 1) - 1) & 1));
        tc::tc_fence_after();
        uint32_t abase, aplane;
        if (L.a_region == REG_MAIN) { abase = main0; aplane = MAIN_PLANE; }
        else { aplane = cfg.small_plane; abase = small0 + (L.a_region == REG_SA ? cfg.sa_off : 0u); }
        const uint32_t idesc = tc::make_idesc_bf16(TM, L.n);
        const uint32_t bplane = (uint32_t)L.n * 32u, blbo = (uint32_t)L.n * 16u;
        for (int s = 0; s < L.ksteps; ++s) {
          if ((s & 3) == 0 && (s >> 2) < L.a_wait) {     // a chunk is 64 columns = 4 K steps
            const int c = s >> 2;
            tc::mbar_wait(&bars->a_ready[c], (aph >> c) & 1u); aph ^= (1u << c);
            tc::tc_fence_after();
          }
          tc::mbar_wait(&bars->w_full[stage], wphase);
          tc::tc_fence_after();
          const uint32_t ao = abase + (uint32_t)s * 2u * KG, bo = wst0 + (uint32_t)stage * cfg.stage_bytes;
          const uint64_t ah = tc::make_smem_desc(ao, KG, 128), bh = tc::make_smem_desc(bo, blbo, 128);
          const uint64_t al = tc::make_smem_desc(ao + aplane, KG, 128), bl = tc::make_smem_desc(bo + bplane, blbo, 128);
          tc::umma_bf16(dcol, ah, bh, idesc, s > 0 ? 1u : 0u);
          tc::umma_bf16(dcol, al, bh, idesc, 1u);
          tc::umma_bf16(dcol, ah, bl, idesc, 1u);
          tc::umma_commit(&bars->w_empty[stage]);
          if (++stage == cfg.nst) { stage = 0; wphase ^= 1u; }
        }
        tc::umma_commit(&bars->d_full[buf]);
      }
    }
  } else {
    // ================= epilogue warps =================
    const int q = warp & 3, group = warp >> 2, half = lane >> 4;
    const int r = q * 16 + (lane & 15);                       // row of the tile
    const int slot = group * 2 + half;                        // 0 .. SLOTS-1: this thread's share of row r
    const bool valid = (row0 + r) < live;
    const size_t grow = (size_t)row0 + r;                     // row in this launch's arrays
    const int col0 = group * 16 + half * 8;                   // this thread's first column inside a 64-column chunk
    const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(group * 16);
    const uint32_t sp = cfg.small_plane;
    const uint32_t roff = (uint32_t)r * 16u;
    int li = 0;
    float zs[8];
    float racc = 0.f, pen = 0.f;

    auto wait_d = [&](int l) { tc::mbar_wait(&bars->d_full[l & 1], (uint32_t)((l >> 1) & 1)); tc::tc_fence_after(); };
    auto release_d = [&](int l) {
      tc::tc_fence_before(); __syncwarp();
      if (lane == 0) tc::mbar_arrive(&bars->d_empty[l & 1]);
    };
    auto signal_a = [&](int c) {
      tc::fence_proxy_async_smem(); __syncwarp();
      if (lane == 0) tc::mbar_arrive(&bars->a_ready[c]);
    };
    auto bias_of = [&](int l) -> const float* {
      tc::mbar_wait(&bars->b_full[l & (NB - 1)], (uint32_t)((l / NB) & 1));
      return bias_s + (l & (NB - 1)) * BSLOT;
    };
    auto bias_done = [&](int l) { __syncwarp(); if (lane == 0) tc::mbar_arrive(&bars->b_empty[l & (NB - 1)]); };
    auto ld8 = [&](const float* b, float (&bv)[8]) {
      const float4 t0 = *reinterpret_cast<const float4*>(b), t1 = *(reinterpret_cast<const float4*>(b) + 1);
      bv[0] = t0.x; bv[1] = t0.y; bv[2] = t0.z; bv[3] = t0.w; bv[4] = t1.x; bv[5] = t1.y; bv[6] = t1.z; bv[7] = t1.w;
    };
    // the accumulator columns [c * 64 + col0, +8) of layer l, this thread's row
    auto ld_acc = [&](int l, int c, uint32_t (&x)[8]) { tc::tmem_ld16x2_8(lane_addr + (uint32_t)(l & 1) * 256u + (uint32_t)(c * CHUNK), x); };

    // 256-wide hidden layer: act(x + b) -> A_main planes; chunks complete in order, TMEM loads one chunk ahead
    auto epi_act256 = [&](int l, bool relu) {
      const float* bias = bias_of(l) + col0;
      wait_d(l);
      uint32_t xa[8], xb[8];
      auto chunk = [&](int c, const uint32_t (&x)[8]) {
        float bv[8], v[8];
        ld8(bias + c * CHUNK, bv);
        act8<NS>(x, bv, v, relu);
        store8<NS>(A_main, MAIN_PLANE, (uint32_t)((c * CHUNK + col0) / 8) * KG + roff, v);
        signal_a(c);
      };
      ld_acc(l, 0, xa);
#pragma unroll 1
      for (int c = 0; c < 4; c += 2) {
        tc::tmem_ld_wait();
        ld_acc(l, c + 1, xb);
        chunk(c, xa);
        tc::tmem_ld_wait();
        if (c + 2 < 4) ld_acc(l, c + 2, xa);
        chunk(c + 1, xb);
      }
      release_d(l);
      bias_done(l);
    };

    // ---------------- prologue: obs (and given actions) -> bf16 operand planes ----------------
    {
      const float* orow = a.obs + grow * a.obs_ld;
      for (int kg = slot; kg < (int)cfg.obs_kp / 8; kg += SLOTS) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { int j = kg * 8 + i; v[i] = (valid && j < S) ? __ldg(orow + j) : 0.f; }
        store8<NS>(A_small, sp, (uint32_t)kg * KG + roff, v);
      }
      if (!cfg.has_policy && 2 + slot < (int)cfg.sa_kp / 8) {   // [zs | a]: K groups 2 .. sa_kp/8 - 1 hold a, zero-padded
        const float* arow = a.act + grow * a.act_ld;
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { int j = slot * 8 + i; v[i] = (valid && j < A) ? __ldg(arow + j) : 0.f; }
        store8<NS>(A_small, sp, cfg.sa_off + (uint32_t)(2 + slot) * KG + roff, v);
      }
      signal_a(0);
    }

    // ---------------- policy: relu MLP, tanh * max_action (mobody.py:35-72) ----------------
    if (cfg.has_policy) {
      epi_act256(li++, true);
      epi_act256(li++, true);
      {
        const int l = li++;
        const float* bias = bias_of(l);
        wait_d(l);
        // columns col0 .. col0+7 < sa_kp - 16 (N = rup16(A) <= 32); sa_kp / 8 is even, so whole warps take part in the load
        if (2 + 2 * group < (int)cfg.sa_kp / 8) {
          uint32_t x[8];
          ld_acc(l, 0, x);
          tc::tmem_ld_wait();
          float v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int j = col0 + i;
            v[i] = (j < A) ? tanhf(__uint_as_float(x[i]) + bias[j]) * a.max_action : 0.f;
            if (valid && j < A && a.act_out) a.act_out[grow * A + j] = v[i];
          }
          store8<NS>(A_small, sp, cfg.sa_off + (uint32_t)(2 + slot) * KG + roff, v);
        }
        release_d(l);
        bias_done(l);
      }
    }

    // ---------------- 7 members: forward_trg / forward_src (mobody_module.py:315-330) ----------------
#pragma unroll 1
    for (int e = 0; e < MB_E; ++e) {
      epi_act256(li++, false);                                  // zs1
      epi_act256(li++, false);                                  // zs2
      {                                                         // zs3 mu half -> [zs | act] operand
        const int l = li++;
        const float* bias = bias_of(l);
        wait_d(l);
        if (col0 < 16) {
          uint32_t x[8];
          ld_acc(l, 0, x);
          tc::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j) zs[j] = __uint_as_float(x[j]) + bias[col0 + j];
          store8<NS>(A_small, sp, cfg.sa_off + (uint32_t)slot * KG + roff, zs);
        }
        signal_a(0);
        release_d(l);
        bias_done(l);
      }
      {                                                         // za1: swish -> 32-wide operand (aliases A_main)
        const int l = li++;
        const float* bias = bias_of(l);
        wait_d(l);
        if (col0 < 32) {
          uint32_t x[8];
          ld_acc(l, 0, x);
          tc::tmem_ld_wait();
          float v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = swish_ns<NS>(__uint_as_float(x[i]) + bias[col0 + i]);
          store8<NS>(A_main, MAIN_PLANE, (uint32_t)slot * KG + roff, v);
        }
        signal_a(0);
        release_d(l);
        bias_done(l);
      }
      {                                                         // za2 mu half: z = zs + za -> 16-wide operand
        const int l = li++;
        const float* bias = bias_of(l);
        wait_d(l);
        if (col0 < 16) {
          uint32_t x[8];
          ld_acc(l, 0, x);
          tc::tmem_ld_wait();
          float v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = zs[i] + (__uint_as_float(x[i]) + bias[col0 + i]);
          store8<NS>(A_main, MAIN_PLANE, (uint32_t)slot * KG + roff, v);
        }
        signal_a(0);
        release_d(l);
        bias_done(l);
      }
      epi_act256(li++, false);                                  // transition1
      epi_act256(li++, false);                                  // transition2
      {                                                         // transition3 -> mean[e] (info['samples'])
        const int l = li++;
        const float* bias = bias_of(l);
        wait_d(l);
        for (int c = 0; c * CHUNK < S; ++c) {                   // the loads are warp-collective: every thread takes part
          uint32_t x[8];
          ld_acc(l, c, x);
          tc::tmem_ld_wait();
          if (valid) {
            float* mrow = a.mean + ((size_t)e * B + grow) * S;
#pragma unroll
            for (int j = 0; j < 8; ++j) { const int col = c * CHUNK + col0 + j; if (col < S) mrow[col] = __uint_as_float(x[j]) + bias[col]; }
          }
        }
        release_d(l);
        bias_done(l);
      }
    }

    // ---------------- ensemble statistics, noise, pick, penalty, termination ----------------
    // As in step_tc.cu: element-wise over the tile's contiguous [64 x S] block of every member, all epilogue threads in
    // flight; per-row sums of squared deviations go through shared memory in member batches, added in a fixed order.
    // Every dynamics MMA has completed, so both operand regions (A_main and the small planes behind it, contiguous) serve
    // as fp32 scratch: at S = 128 that holds 3 members' squared deviations per batch.
    constexpr int NEPI = 32 * EPI_WARPS;
    const int n_el = TM * S;
    float* nobs_s = reinterpret_cast<float*>(A_main);                 // [64*S]    next_obs of the tile
    int* member_s = reinterpret_cast<int*>(nobs_s + n_el);            // [64]      picked member per row
    float* dsq_s = reinterpret_cast<float*>(member_s + TM) + TM;      // [batch][64*S] squared deviations
    const int scratch_floats = (int)((NS * MAIN_PLANE + NS * cfg.small_plane) / 4) - n_el - 2 * TM;
    const int mbatch = min(MB_E, scratch_floats / n_el);
    const int etid = tid;                                             // epilogue threads are 0 .. NEPI-1
    if (etid < TM) {
      int mem = 0;
      if (row0 + etid < live) {
        const size_t gr = (size_t)row0 + etid;
        const unsigned long long gid = a.row_ids ? (unsigned long long)a.row_ids[gr] : a.row0 + gr;
        mem = a.idx ? (int)a.idx[gr] : (int)a.elites[philox_elite_slot(a.seed, a.step, gid, a.n_elites)];
      }
      member_s[etid] = mem;
    }
    epi_bar<EPI_WARPS>();   // every mean column of this tile has been written; member_s is visible
    float row_pmax = 0.f;
    for (int e0 = 0; e0 < MB_E; e0 += mbatch) {
#pragma unroll 1   // one code path for every element: a row's result must not depend on its position in the tile
      for (int i = etid; i < n_el; i += NEPI) {
        const int rr = i / S, j = i - rr * S;
        const size_t gr = (size_t)row0 + rr;
        if (row0 + rr < live) {
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
      // (row, member) sums in a fixed order; slot s takes members s, s+SLOTS, ... of its row r
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
    red[slot * TM + r] = row_pmax;
    if (slot == 0 && valid) a.terminal[grow] = (unsigned char)mb_terminal(a.term_kind, nobs_s + r * S, S);
    epi_bar<EPI_WARPS>();
    if (slot == 0 && valid) {
      float pm = 0.f;
#pragma unroll
      for (int s2 = 0; s2 < SLOTS; ++s2) pm = fmaxf(pm, red[s2 * TM + r]);
      pen = pm;
    }
    {   // sas = [obs, act, next_obs, 0-pad] operand of the reward head (mobody_module.py:296); over the obs / sa planes
      const float* actp = cfg.has_policy ? a.act_out : a.act;
      const int act_ld = cfg.has_policy ? A : a.act_ld;
      for (int kg = slot; kg < (int)cfg.sas_kp / 8; kg += SLOTS) {
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
        store8<NS>(A_small, sp, (uint32_t)kg * KG + roff, v);
      }
      tc::fence_proxy_async_smem();
    }
    epi_bar<EPI_WARPS>();   // every sas plane is written (and nobs_s / red are no longer read) before any chunk is announced
    for (int c = 0; c * CHUNK < (int)cfg.sas_kp; ++c) { __syncwarp(); if (lane == 0) tc::mbar_arrive(&bars->a_ready[c]); }

    // ---------------- reward head, all 7 members (mobody_module.py:295-302; mean over members :236) ----------------
#pragma unroll 1
    for (int e = 0; e < MB_E; ++e) {
      epi_act256(li++, false);                                  // reward_model1
      {                                                         // reward_model2 -> swish -> dot reward_model3[:,0]
        const int l = li++;
        const float* bslot = bias_of(l);
        const float* w3 = bslot + 256;                              // reward_model3[:,0] (256) and its bias at [256]
        float part = 0.f;
        wait_d(l);
        uint32_t x[8], xn[8];
        ld_acc(l, 0, x);
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          tc::tmem_ld_wait();
          if (c + 1 < 4) ld_acc(l, c + 1, xn);
          float bv[8], wv[8];
          ld8(bslot + c * CHUNK + col0, bv);
          ld8(w3 + c * CHUNK + col0, wv);
#pragma unroll
          for (int i = 0; i < 8; ++i) part = fmaf(swish_ns<NS>(__uint_as_float(x[i]) + bv[i]), wv[i], part);
          if (c + 1 < 4) {
            tc::tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 8; ++i) x[i] = xn[i];
          }
        }
        const float b3 = w3[256];
        release_d(l);
        bias_done(l);
        red[((e & 1) * SLOTS + slot) * TM + r] = part;
        epi_bar<EPI_WARPS>();
        if (slot == 0) {
          float sum = 0.f;
#pragma unroll
          for (int s2 = 0; s2 < SLOTS; ++s2) sum += red[((e & 1) * SLOTS + s2) * TM + r];
          racc += sum + b3;
        }
      }
    }
    if (slot == 0 && valid) {
      const float raw = racc / (float)MB_E;
      if (a.raw_reward) a.raw_reward[grow] = raw;
      a.penalty[grow] = pen;
      a.reward[grow] = (a.coef != 0.f && a.use_penalty) ? raw - a.coef * pen : raw;     // :261-263
    }
  }

  tc::tc_fence_before();
  __syncthreads();
  if (warp == PROD_WARP) tc::tmem_dealloc(tmem, 512);
}

}  // namespace tcw

const char* mb_tc_wide_step_launch(const StepArgs& a, const unsigned char* dynb, const unsigned char* polb, cudaStream_t st) {
  if (a.B <= 0) return nullptr;
  const int S = a.S, A = a.A;
  if (S < 65 || S > 128 || A < 1 || A > 32) return "wide tensor-core step kernel supports 65 <= S <= 128, 1 <= A <= 32";
  if (!dynb) return "tensor-core step needs dyn_pack (mobody_dyn_pack)";
  const bool has_policy = polb != nullptr;
  if (has_policy && !a.act_out) return "tensor-core step with a fused policy needs act_out";
  constexpr int ns = tcw::NS;
  const TcDynLayout DL = tc_dyn_layout(S, A, ns);
  TcSched sc{}; int n = 0;
  auto add = [&](size_t w_off, uint32_t b_off, const TcGeom& g, int region, int a_wait, int kind, int blob) {
    TcLayer& L = sc.L[n++];
    L.w_off = (uint32_t)w_off; L.b_off = b_off; L.ksteps = (uint16_t)(g.Kp / 16); L.n = (uint16_t)g.Np;
    L.a_region = (uint8_t)region; L.a_wait = (uint8_t)a_wait; L.kind = (uint8_t)kind; L.blob = (uint8_t)blob;
  };
  // a_wait counts 64-column chunks here (4 per 256-wide layer)
  tcw::Cfg cfg{};
  if (has_policy) {
    const TcMlpLayout PL = tc_mlp_layout(S, A, ns);
    add(PL.w_off[0], PL.b_off[0], PL.g[0], REG_OBS, 1, EPI_RELU256, 1);
    add(PL.w_off[1], PL.b_off[1], PL.g[1], REG_MAIN, 4, EPI_RELU256, 1);
    add(PL.w_off[2], PL.b_off[2], PL.g[2], REG_MAIN, 4, EPI_ACTION, 1);
    cfg.pol_bias_base = (uint32_t)PL.bias_base;
  }
  sc.first_dyn = n;
  const int za1 = a.use_trg ? PK_ZATRG1 : PK_ZASRC1, za2 = a.use_trg ? PK_ZATRG2 : PK_ZASRC2;
  const int sas_kp = tc_rup16(2 * S + A);
  for (int e = 0; e < MB_E; ++e) {
    const size_t wb = (size_t)e * DL.member_w_bytes; const uint32_t bb = (uint32_t)e * DL.member_b_floats;
    auto lay = [&](int pk, int region, int a_wait, int kind) { add(wb + DL.w_off[pk], bb + DL.b_off[pk], tc_dyn_geom(pk, S, A), region, a_wait, kind, 0); };
    lay(PK_ZS1, REG_OBS, (e == 0 && !has_policy) ? 1 : 0, EPI_SWISH256);
    lay(PK_ZS2, REG_MAIN, 4, EPI_SWISH256);
    lay(PK_ZS3, REG_MAIN, 4, EPI_ZS);
    lay(za1, REG_SA, 1, EPI_G);
    lay(za2, REG_MAIN, 1, EPI_Z);
    lay(PK_T1, REG_MAIN, 1, EPI_SWISH256);
    lay(PK_T2, REG_MAIN, 4, EPI_SWISH256);
    lay(PK_T3, REG_MAIN, 4, EPI_MEAN);
  }
  for (int e = 0; e < MB_E; ++e) {
    const size_t wb = (size_t)e * DL.member_w_bytes; const uint32_t bb = (uint32_t)e * DL.member_b_floats;
    add(wb + DL.w_off[PK_R1], bb + DL.b_off[PK_R1], tc_dyn_geom(PK_R1, S, A), REG_SAS, e == 0 ? (sas_kp + tcw::CHUNK - 1) / tcw::CHUNK : 0, EPI_SWISH256, 0);
    add(wb + DL.w_off[PK_R2], bb + DL.b_off[PK_R2], tc_dyn_geom(PK_R2, S, A), REG_MAIN, 4, EPI_REWARD, 0);
  }
  sc.n_layers = n;
  cfg.obs_kp = (uint32_t)tc_rup16(S); cfg.sa_kp = (uint32_t)tc_rup16(MB_LATENT + A); cfg.sas_kp = (uint32_t)sas_kp;
  cfg.sa_off = (cfg.obs_kp / 8) * tcw::KG;
  const uint32_t small = cfg.sa_off + (cfg.sa_kp / 8) * tcw::KG, sasb = (cfg.sas_kp / 8) * tcw::KG;
  cfg.small_plane = small > sasb ? small : sasb;
  cfg.stage_bytes = (uint32_t)ns * 256u * 32u;
  cfg.dyn_bias_base = (uint32_t)DL.bias_base;
  cfg.has_policy = has_policy ? 1 : 0;
  const size_t fixed = (size_t)ns * tcw::MAIN_PLANE + (size_t)ns * cfg.small_plane + (2 * tcw::SLOTS * tcw::TM + tcw::NB * tcw::BSLOT) * sizeof(float) +
                       sizeof(tcw::Bars) + 128;
  const size_t budget = 227 * 1024;
  if (fixed + 4 * cfg.stage_bytes > budget) return "wide tensor-core step kernel: shared memory budget exceeded for this (S, A)";
  int nst = (int)((budget - fixed) / cfg.stage_bytes);
  if (nst > tcw::MAX_NST) nst = tcw::MAX_NST;
  cfg.nst = nst;
  const size_t bytes = fixed + (size_t)nst * cfg.stage_bytes;
  if (cudaFuncSetAttribute(tcw::step_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
    return "cudaFuncSetAttribute(step_wide_kernel) failed";
  // every tile streams the whole weight image from L2 (9.2 MB at obs 111 / act 8): keep it persisting, as step_tc.cu does
  static thread_local int limit_dev = -1;
  int dev = 0; cudaGetDevice(&dev);
  if (limit_dev != dev) { cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)32 << 20); limit_dev = dev; }
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeAccessPolicyWindow;
  at[0].val.accessPolicyWindow.base_ptr = const_cast<unsigned char*>(dynb);
  at[0].val.accessPolicyWindow.num_bytes = DL.total_bytes;
  at[0].val.accessPolicyWindow.hitRatio = 1.0f;
  at[0].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
  at[0].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  cudaLaunchConfig_t lc = {};
  lc.gridDim = dim3((a.B + tcw::TM - 1) / tcw::TM); lc.blockDim = dim3(32 * (4 * tcw::NG + 2)); lc.dynamicSmemBytes = bytes; lc.stream = st;
  lc.attrs = at; lc.numAttrs = 1;
  const unsigned char* polp = polb ? polb : dynb;
  if (cudaLaunchKernelEx(&lc, tcw::step_wide_kernel, a, dynb, polp, sc, cfg) != cudaSuccess) return "step_wide_kernel launch failed";
  return nullptr;
}
