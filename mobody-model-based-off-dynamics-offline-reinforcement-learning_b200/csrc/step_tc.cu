// Fused one-step model rollout on the 5th-gen tensor cores (tcgen05 + TMEM), sm_100a.
//
// Same math as step_simt.cu / SURVEY.md Appendix A.1 (reference
// algo/dynamics/mobody_dynamics.py:193-265, algo/dynamics/mobody_module.py:217-330,
// algo/offline_offline/mobody.py:60-72), restructured for Blackwell:
//
//  * one CTA owns 128 start states (UMMA M = 128) and walks the whole per-row chain
//      [policy 3 GEMMs] + 7 x 8 dynamics GEMMs + ensemble statistics + 7 x 2 reward GEMMs
//    without the activations ever leaving the SM;
//  * layer weights are pre-packed (mobody_dyn_pack) as bf16 planes in the exact UMMA K-major
//    shared-memory image and streamed L2 -> SMEM by a producer warp with 1-D TMA bulk copies
//    (cp.async.bulk + mbarrier complete_tx) through an NST-deep ring;
//  * one elected thread issues tcgen05.mma (128 x N x 16 per instruction), accumulators live in
//    TMEM (two 256-column buffers, ping-pong across layers);
//  * 16 epilogue warps (4 groups x 4 TMEM lane quadrants) read TMEM (tcgen05.ld, one chunk ahead), apply
//    bias + swish/relu, split to bf16 planes with integer ops and write the next layer's A operand in
//    place in SMEM.  All groups work on the same 32-column chunk (8 columns per warp), so chunks are
//    announced in order (one mbarrier per chunk) and the next layer's MMAs trail the epilogue by one chunk:
//    tensor pipe and epilogue overlap inside a single row tile.
//  Siblings: step_duo.cu (two tiles in flight per CTA; the single-pass fp16 mode runs there) and step_wide.cu (64-row
//  tiles).  The three share tc_step.cuh: the layer schedule, the launch, the bias staging and everything after the last
//  dynamics GEMM (ensemble statistics, noise, pick, penalty, termination, the reward head's operand, the final write).
//  The CTA-pair experiment of round 1 (cta_group::2; correct, 3x slower) lives in scripts/experimental/ and is not part of
//  the library; DESIGN.md 4.1.
//
// Precision: NS = 2 -> bf16 hi+lo split of both operands, 3 MMAs per K step (hi*hi + lo*hi + hi*lo), ~2^-16 per
// product: inside the 1e-4 bound (the default mode).  NS = 1 -> single bf16 pass (bound 2e-2; used when the two-tile
// kernel does not fit).  Biases come from a shared-memory ring staged by the producer warp; swish
// layers are packed pre-scaled (tc_layout.h: tc_swish_scales) so the epilogue needs no multiply before the SFU op.
#include "tc_step.cuh"
#include <cuda_fp16.h>

namespace tcs {
using namespace tst;

constexpr int TM = 128;
constexpr int NG = 4;                    // epilogue groups of 4 warps (one warp per TMEM lane quadrant)
constexpr uint32_t MAIN_PLANE = 65536;   // 128 rows x 256 k x bf16
constexpr int MAX_NST = 12;

struct Cfg {
  int nst;
  uint32_t stage_bytes, small_plane, sa_off, obs_kp, sas_kp;
  uint32_t dyn_bias_base, pol_bias_base;
  int has_policy;
  long long* trace;     // debug: per-layer clock64 timestamps of CTA 0 ([layer][8]); nullptr in production
};

struct Bars {
  uint64_t w_full[MAX_NST], w_empty[MAX_NST], a_ready[8], d_full[2], d_empty[2], b_full[NB], b_empty[NB];
  uint32_t tmem_slot, pad;
};

// NG groups of 4 epilogue warps (one warp per TMEM lane quadrant).  Every 32-column accumulator chunk is
// processed by ALL groups at once (group g takes columns [g*CW, (g+1)*CW) of the chunk, CW = 32/NG), so
// chunks complete in order and the next layer's MMAs trail the epilogue by one chunk.
template <int NS>
__global__ void __launch_bounds__(32 * (4 * NG + 2), 1)
step_tc_kernel(const StepArgs a, const unsigned char* __restrict__ dynb, const unsigned char* __restrict__ polb,
               const __grid_constant__ TcSched sched, const Cfg cfg) {
  constexpr int EPI_WARPS = 4 * NG, PROD_WARP = EPI_WARPS, MMA_WARP = EPI_WARPS + 1;
  constexpr int CW = 32 / NG, KGW = CW / 8;
  extern __shared__ __align__(128) unsigned char smem[];
  const int S = a.S, A = a.A, B = a.B;
  const int live = a.n_rows_dev ? min(*a.n_rows_dev, B) : B;
  const int row0 = blockIdx.x * TM;
  if (row0 >= live) return;

  unsigned char* A_main = smem;
  unsigned char* A_small = A_main + NS * MAIN_PLANE;
  unsigned char* wst = A_small + NS * cfg.small_plane;
  float* red = reinterpret_cast<float*>(wst + (size_t)cfg.nst * cfg.stage_bytes);      // [2][4][128]
  float* bias_s = red + 2 * 4 * 128;                                                   // [NB][BSLOT]
  Bars* bars = reinterpret_cast<Bars*>(bias_s + NB * BSLOT);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    for (int i = 0; i < cfg.nst; ++i) { tc::mbar_init(&bars->w_full[i], 1); tc::mbar_init(&bars->w_empty[i], 1); }
    for (int i = 0; i < 8; ++i) tc::mbar_init(&bars->a_ready[i], EPI_WARPS);   // every epilogue warp announces every chunk
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
    // ================= weight producer: L2 -> SMEM ring, one K step (all planes) per stage =================
    if (tc::elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int li = 0; li < sched.n_layers; ++li) {
        const TcLayer L = sched.L[li];
        const unsigned char* src = (L.blob ? polb : dynb) + L.w_off;
        const uint32_t bytes = (uint32_t)NS * L.n * 32u;
        tc_stage_bias(li, L, dynb, polb, cfg.dyn_bias_base, cfg.pol_bias_base, bias_s, bars->b_full, bars->b_empty);
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
      uint32_t aph = 0; int stage = 0; uint32_t wphase = 0;
      const uint32_t small0 = tc::smem_u32(A_small), main0 = tc::smem_u32(A_main), wst0 = tc::smem_u32(wst);
      for (int li = 0; li < sched.n_layers; ++li) {
        const TcLayer L = sched.L[li];
        const int buf = li & 1;
        const uint32_t dcol = tmem + (uint32_t)buf * 256u;
        if (li >= 2) tc::mbar_wait(&bars->d_empty[buf], (uint32_t)(((li >> 1) - 1) & 1));
        tc::tc_fence_after();
        if (cfg.trace && blockIdx.x == 0) cfg.trace[li * 8 + 0] = clock64();
        uint32_t abase, aplane;
        if (L.a_region == REG_MAIN) { abase = main0; aplane = MAIN_PLANE; }
        else { aplane = cfg.small_plane; abase = small0 + (L.a_region == REG_SA ? cfg.sa_off : 0u); }
        const uint32_t idesc = tc::make_idesc_bf16(128, L.n);
        const uint32_t bplane = (uint32_t)L.n * 32u, blbo = (uint32_t)L.n * 16u;
        for (int s = 0; s < L.ksteps; ++s) {
          if ((s & 1) == 0 && (s >> 1) < L.a_wait) {
            const int c = s >> 1;
            tc::mbar_wait(&bars->a_ready[c], (aph >> c) & 1u); aph ^= (1u << c);
            tc::tc_fence_after();
          }
          tc::mbar_wait(&bars->w_full[stage], wphase);
          tc::tc_fence_after();
          const uint32_t ao = abase + (uint32_t)s * 4096u, bo = wst0 + (uint32_t)stage * cfg.stage_bytes;
          const uint64_t ah = tc::make_smem_desc(ao, 2048, 128), bh = tc::make_smem_desc(bo, blbo, 128);
          if (cfg.trace && blockIdx.x == 0 && s == 0) cfg.trace[li * 8 + 1] = clock64();
          tc::umma_bf16(dcol, ah, bh, idesc, s > 0 ? 1u : 0u);
          if (NS == 2) {
            const uint64_t al = tc::make_smem_desc(ao + aplane, 2048, 128), bl = tc::make_smem_desc(bo + bplane, blbo, 128);
            tc::umma_bf16(dcol, al, bh, idesc, 1u);
            tc::umma_bf16(dcol, ah, bl, idesc, 1u);
          }
          tc::umma_commit(&bars->w_empty[stage]);
          if (++stage == cfg.nst) { stage = 0; wphase ^= 1u; }
        }
        tc::umma_commit(&bars->d_full[buf]);
        if (cfg.trace && blockIdx.x == 0) cfg.trace[li * 8 + 2] = clock64();
      }
    }
  } else {
    // ================= epilogue warps =================
    const int q = warp & 3, group = warp >> 2;
    const int r = q * 32 + lane;
    const bool valid = (row0 + r) < live;
    const size_t grow = (size_t)row0 + r;                     // row in this launch's arrays
    const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(group * CW);
    const uint32_t sp = cfg.small_plane;
    const int col0 = group * CW;                              // this warp's first column inside a 32-column chunk
    int li = 0;
    float zs[CW];
    float racc = 0.f, pen = 0.f;

    const bool tracer = cfg.trace && blockIdx.x == 0 && lane == 0 && q == 0 && group < 2;
    auto wait_d = [&](int l) {
      tc::mbar_wait(&bars->d_full[l & 1], (uint32_t)((l >> 1) & 1)); tc::tc_fence_after();
      if (tracer) cfg.trace[l * 8 + 3 + 2 * group] = clock64();
    };
    auto release_d = [&](int l) {
      if (tracer) cfg.trace[l * 8 + 4 + 2 * group] = clock64();
      tc::tc_fence_before(); __syncwarp();
      if (lane == 0) tc::mbar_arrive(&bars->d_empty[l & 1]);
    };
    auto signal_a = [&](int c) {
      tc::fence_proxy_async_smem(); __syncwarp();
      if (lane == 0) tc::mbar_arrive(&bars->a_ready[c]);
    };
    // biases are staged per layer by the producer warp (bias ring); every epilogue warp acquires and releases every layer
    auto bias_of = [&](int l) -> const float* {
      tc::mbar_wait(&bars->b_full[l & (NB - 1)], (uint32_t)((l / NB) & 1));
      return bias_s + (l & (NB - 1)) * BSLOT;
    };
    auto bias_done = [&](int l) { __syncwarp(); if (lane == 0) tc::mbar_arrive(&bars->b_empty[l & (NB - 1)]); };
    auto ldbias = [&](const float* b, float (&bv)[CW]) {
#pragma unroll
      for (int i = 0; i < CW / 4; ++i) {
        const float4 t = *(reinterpret_cast<const float4*>(b) + i);
        bv[4 * i] = t.x; bv[4 * i + 1] = t.y; bv[4 * i + 2] = t.z; bv[4 * i + 3] = t.w;
      }
    };

    // 256-wide hidden layer: act(x + b) -> A_main planes; chunks complete in order, TMEM loads one chunk ahead.
    // Two register sets alternate (no copies); the SFU ops of a chunk are issued back to back (act8) so their
    // latency overlaps inside one warp instead of relying on the other three warps of the scheduler.
    auto epi_act256 = [&](int l, bool relu) {
      const float* bias = bias_of(l) + col0;
      const uint32_t t0 = lane_addr + (uint32_t)(l & 1) * 256u;
      wait_d(l);
      uint32_t xa[CW], xb[CW];
      auto chunk = [&](int c, const uint32_t (&x)[CW]) {
        float bv[CW];
        ldbias(bias + c * 32, bv);
#pragma unroll
        for (int kg = 0; kg < KGW; ++kg) {
          float v[8];
          act8<NS>(&x[kg * 8], &bv[kg * 8], v, relu);
          store8<NS>(A_main, MAIN_PLANE, (uint32_t)(c * 4 + group * KGW + kg) * 2048u + (uint32_t)r * 16u, v);
        }
        signal_a(c);
      };
      tmem_ldw<CW>(t0, xa);
#pragma unroll 1
      for (int c = 0; c < 8; c += 2) {
        tc::tmem_ld_wait();
        tmem_ldw<CW>(t0 + (uint32_t)(c + 1) * 32u, xb);
        chunk(c, xa);
        tc::tmem_ld_wait();
        if (c + 2 < 8) tmem_ldw<CW>(t0 + (uint32_t)(c + 2) * 32u, xa);
        chunk(c + 1, xb);
      }
      release_d(l);
      bias_done(l);
    };

    // ---------------- prologue: obs (and given actions) -> bf16 operand planes ----------------
    {
      const float* orow = a.obs + grow * a.obs_ld;
      for (int kg = group; kg < (int)cfg.obs_kp / 8; kg += NG) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { int j = kg * 8 + i; v[i] = (valid && j < S) ? __ldg(orow + j) : 0.f; }
        store8<NS>(A_small, sp, (uint32_t)kg * 2048u + (uint32_t)r * 16u, v);
      }
      if (!cfg.has_policy && group < 2) {
        const float* arow = a.act + grow * a.act_ld;
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { int j = group * 8 + i; v[i] = (valid && j < A) ? __ldg(arow + j) : 0.f; }
        store8<NS>(A_small, sp, cfg.sa_off + (uint32_t)(2 + group) * 2048u + (uint32_t)r * 16u, v);
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
        if (col0 < 16) {
          uint32_t x[CW];
          tmem_ldw<CW>(lane_addr + (uint32_t)(l & 1) * 256u, x);
          tc::tmem_ld_wait();
#pragma unroll
          for (int kg = 0; kg < KGW; ++kg) {
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int j = col0 + kg * 8 + i;
              v[i] = (j < A) ? tanhf(__uint_as_float(x[kg * 8 + i]) + bias[j]) * a.max_action : 0.f;
              if (valid && j < A && a.act_out) a.act_out[grow * A + j] = v[i];
            }
            store8<NS>(A_small, sp, cfg.sa_off + (uint32_t)(2 + group * KGW + kg) * 2048u + (uint32_t)r * 16u, v);
          }
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
          uint32_t x[CW];
          tmem_ldw<CW>(lane_addr + (uint32_t)(l & 1) * 256u, x);
          tc::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < CW; ++j) zs[j] = __uint_as_float(x[j]) + bias[col0 + j];
#pragma unroll
          for (int kg = 0; kg < KGW; ++kg) {
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = zs[kg * 8 + i];
            store8<NS>(A_small, sp, cfg.sa_off + (uint32_t)(group * KGW + kg) * 2048u + (uint32_t)r * 16u, v);
          }
        }
        signal_a(0);
        release_d(l);
        bias_done(l);
      }
      {                                                         // za1: swish -> 32-wide operand (aliases A_main)
        const int l = li++;
        const float* bias = bias_of(l);
        wait_d(l);
        {
          uint32_t x[CW];
          tmem_ldw<CW>(lane_addr + (uint32_t)(l & 1) * 256u, x);
          tc::tmem_ld_wait();
#pragma unroll
          for (int kg = 0; kg < KGW; ++kg) {
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = swish_ns<NS>(__uint_as_float(x[kg * 8 + i]) + bias[col0 + kg * 8 + i]);
            store8<NS>(A_main, MAIN_PLANE, (uint32_t)(group * KGW + kg) * 2048u + (uint32_t)r * 16u, v);
          }
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
          uint32_t x[CW];
          tmem_ldw<CW>(lane_addr + (uint32_t)(l & 1) * 256u, x);
          tc::tmem_ld_wait();
#pragma unroll
          for (int kg = 0; kg < KGW; ++kg) {
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = zs[kg * 8 + i] + (__uint_as_float(x[kg * 8 + i]) + bias[col0 + kg * 8 + i]);
            store8<NS>(A_main, MAIN_PLANE, (uint32_t)(group * KGW + kg) * 2048u + (uint32_t)r * 16u, v);
          }
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
        const int np = sched.L[l].n;
        wait_d(l);
        for (int c = 0; c * 32 + col0 < np; ++c) {
          uint32_t x[CW];
          tmem_ldw<CW>(lane_addr + (uint32_t)(l & 1) * 256u + (uint32_t)c * 32u, x);
          tc::tmem_ld_wait();
          if (valid) {
            float* mrow = a.mean + ((size_t)e * B + grow) * S;
#pragma unroll
            for (int j = 0; j < CW; ++j) { const int col = c * 32 + col0 + j; if (col < S) mrow[col] = __uint_as_float(x[j]) + bias[col]; }
          }
        }
        release_d(l);
        bias_done(l);
      }
    }

    // ---------------- ensemble statistics, noise, pick, penalty, termination (tc_step.cuh) ----------------
    // All epilogue warps take part: the NG threads of a row split its member sums (slot = group).  A_main is free here
    // (every dynamics MMA has completed) and serves as fp32 scratch.
    float* nobs_s = reinterpret_cast<float*>(A_main);
    auto stamp = [&](int k) { if (tracer && group == 0) cfg.trace[79 * 8 + k] = clock64(); };   // trace stamps of the phase
    const float row_pmax = tc_stats<TM, EPI_WARPS, NG>(a, S, B, row0, live, r, group, valid, nobs_s, NS * MAIN_PLANE,
                                                       stamp);
    stamp(2);
    pen = tc_penalty_terminal<TM, EPI_WARPS, NG>(a, S, row_pmax, red, r, group, valid, grow, nobs_s, stamp);
    stamp(4);
    // [s | a | s'] aliases the obs / sa planes
    tc_sas_operand<NG>(a, S, A, cfg.has_policy, (int)cfg.sas_kp, r, group, valid, grow, nobs_s,
                       [&](int kg, const float (&v)[8]) { store8<NS>(A_small, sp, (uint32_t)kg * 2048u + (uint32_t)r * 16u, v); });
    stamp(5);
    epi_bar<EPI_WARPS>();   // every sas plane is written (and nobs_s is no longer needed) before any chunk is announced
    stamp(6);
    for (int c = 0; c * 32 < (int)cfg.sas_kp; ++c) { __syncwarp(); if (lane == 0) tc::mbar_arrive(&bars->a_ready[c]); }

    // ---------------- reward head, all 7 members (mobody_module.py:295-302; mean over members :236) ----------------
#pragma unroll 1
    for (int e = 0; e < MB_E; ++e) {
      epi_act256(li++, false);                                  // reward_model1
      {                                                         // reward_model2 -> swish -> dot reward_model3[:,0]
        const int l = li++;
        const float* bslot = bias_of(l);
        const float* bias = bslot + col0;
        const float* w3 = bslot + 256;                              // reward_model3[:,0] (256) and its bias at [256]
        const uint32_t t0 = lane_addr + (uint32_t)(l & 1) * 256u;
        float part = 0.f;
        wait_d(l);
        uint32_t x[CW], xn[CW];
        tmem_ldw<CW>(t0, x);
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {
          tc::tmem_ld_wait();
          if (c + 1 < 8) tmem_ldw<CW>(t0 + (uint32_t)(c + 1) * 32u, xn);
          float bv[CW], wv[CW];
          ldbias(bias + c * 32, bv);
          ldbias(w3 + col0 + c * 32, wv);
#pragma unroll
          for (int i = 0; i < CW; ++i) part = fmaf(swish_ns<NS>(__uint_as_float(x[i]) + bv[i]), wv[i], part);
          if (c + 1 < 8) {
            tc::tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < CW; ++i) x[i] = xn[i];
          }
        }
        const float b3 = w3[256];
        release_d(l);
        bias_done(l);
        red[((e & 1) * NG + group) * 128 + r] = part;
        epi_bar<EPI_WARPS>();
        if (group == 0) {
          float sum = 0.f;
#pragma unroll
          for (int g2 = 0; g2 < NG; ++g2) sum += red[((e & 1) * NG + g2) * 128 + r];
          racc += sum + b3;
        }
      }
    }
    if (group == 0 && valid) tc_write_reward(a, grow, racc, pen);
  }

  tc::tc_fence_before();
  __syncthreads();
  if (warp == PROD_WARP) tc::tmem_dealloc(tmem, 512);
}

// ---------------- weight packing: fp32 [K][N] (any strides) -> bf16 planes in UMMA B layout ----------------
// image of one layer: [kstep s][plane p][kgroup g][n < Np][8 k]   (one CTA stages a whole K step with one bulk copy)
__device__ __forceinline__ void pack_weight(const float* __restrict__ W, long long stride_k, long long stride_n, const TcGeom& g,
                                            int ns, int fp16, float scale, __nv_bfloat16* __restrict__ out) {
  const long long total = (long long)(g.Kp / 16) * ns * 2 * g.Np * 8;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(t & 7); long long u = t >> 3;
    const int n = (int)(u % g.Np); u /= g.Np;
    const int kg = (int)(u & 1); u >>= 1;
    const int p = (int)(u % ns), s = (int)(u / ns);
    const int k = s * 16 + kg * 8 + j;
    const float v = (k < g.K && n < g.N) ? W[k * stride_k + n * stride_n] * scale : 0.f;
    if (fp16) { reinterpret_cast<__half*>(out)[t] = __float2half_rn(v); continue; }     // single fp16 plane (ns == 1)
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    out[t] = (p == 0) ? h : __float2bfloat16_rn(v - __bfloat162float(h));
  }
}
__device__ __forceinline__ void pack_bias(const float* __restrict__ b, long long stride, int N, int Np, float scale, float* __restrict__ out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < Np; i += gridDim.x * blockDim.x) out[i] = (i < N) ? b[i * stride] * scale : 0.f;
}

// ---------------- change detection for the packed images ----------------
// state (device u64[4], zeroed once by the caller): [0] checksum of the parameters the image was packed from, [1] checksum
// of the live parameters (accumulated by params_checksum_kernel, consumed and re-zeroed by the pack kernel), [2] image
// valid flag, [3] ticket.  The checksum is position dependent (a value moved to another slot changes it) and is a sum of
// 64-bit integers, so the atomics make it order independent: any write to the live fp32 parameters -- optimiser step,
// load_state_dict, `.data.copy_()` (mobody_module.py:407-408), a raw pointer write -- is seen without asking the host.
struct ChecksumArgs { const float* p[26]; unsigned int n[26]; int count; };
__global__ void __launch_bounds__(256) params_checksum_kernel(const ChecksumArgs a, unsigned long long* __restrict__ state) {
  const int t = blockIdx.y;
  const unsigned int n = a.n[t];
  const unsigned int per = 256u * 8u;                               // elements per block per sweep: 8 independent loads per thread
  if (blockIdx.x * per >= n) return;
  const uint32_t* x = reinterpret_cast<const uint32_t*>(a.p[t]);
  const uint32_t salt = 0x9E3779B9u * (uint32_t)(t + 1);
  unsigned long long h = 0;
  for (unsigned int base = blockIdx.x * per; base < n; base += gridDim.x * per) {
    uint32_t v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { const unsigned int i = base + k * 256u + threadIdx.x; v[k] = i < n ? x[i] : 0u; }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const unsigned int i = base + k * 256u + threadIdx.x;
      if (i < n) h += (unsigned long long)(v[k] ^ salt) * (2ull * i + 1ull) + (unsigned long long)(t + 1);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
  __shared__ unsigned long long sh[8];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = h;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long s = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += sh[w];
    if (s) atomicAdd(state + 1, s);
  }
}
// true -> this block must (re)pack.  Every block reads the two checksums first; the last block to finish commits.
__device__ __forceinline__ bool pack_needed(const unsigned long long* state) {
  if (!state) return true;
  return !(state[2] != 0ull && state[0] == state[1]);
}
__device__ __forceinline__ void pack_commit(unsigned long long* state, unsigned long long cur) {
  if (!state) return;
  __shared__ bool last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(state + 3, 1ull) == (unsigned long long)gridDim.x * gridDim.y - 1ull;
  __syncthreads();
  if (last && threadIdx.x == 0) { state[0] = cur; state[1] = 0ull; state[2] = 1ull; state[3] = 0ull; }
}

// mobody_dyn_pack as ONE launch: blockIdx.y = member * 13 + job; jobs 0..11 = the MMA layers (weights + bias), job 12 =
// reward_model3's column 0 and bias (the epilogue dot of the reward head)
__device__ void pack_dyn_job(const DynPtrs& dp, int S, int A, int ns, int fp16, unsigned char* __restrict__ blob) {
  const int e = blockIdx.y / (PK_COUNT + 1), i = blockIdx.y % (PK_COUNT + 1);
  const TcDynLayout L = tc_dyn_layout(S, A, ns);
  float* bias = reinterpret_cast<float*>(blob + L.bias_base) + (size_t)e * L.member_b_floats;
  double so, si;
  tc_swish_scales(ns, &so, &si);
  if (i == PK_COUNT) {                                   // consumes reward_model2's swish: carries the input scale
    float* o = bias + L.b_off[PK_COUNT];
    pack_bias(dp.w[L_R3] + (size_t)e * MB_H * 2, 2, MB_H, MB_H, (float)si, o);
    pack_bias(dp.b[L_R3] + (size_t)e * 2, 1, 1, 16, 1.0f, o + MB_H);
    return;
  }
  const int src[PK_COUNT] = {L_ZS1, L_ZS2, L_ZS3, L_ZASRC1, L_ZASRC2, L_ZATRG1, L_ZATRG2, L_T1, L_T2, L_T3, L_R1, L_R2};
  const float wscale = (float)((tc_out_is_swish(i) ? so : 1.0) * (tc_in_is_swish(i) ? si : 1.0));
  const float bscale = (float)(tc_out_is_swish(i) ? so : 1.0);
  const TcGeom g = tc_dyn_geom(i, S, A);
  const int nfull = (i == PK_ZS3 || i == PK_ZASRC2 || i == PK_ZATRG2) ? 32 : g.N;     // mu half of 32 columns
  pack_weight(dp.w[src[i]] + (size_t)e * g.K * nfull, nfull, 1, g, ns, fp16, wscale,
              reinterpret_cast<__nv_bfloat16*>(blob + (size_t)e * L.member_w_bytes + L.w_off[i]));
  pack_bias(dp.b[src[i]] + (size_t)e * nfull, 1, g.N, g.Np, bscale, bias + L.b_off[i]);
}
__global__ void pack_dyn_kernel(const DynPtrs dp, int S, int A, int ns, int fp16, unsigned char* __restrict__ blob,
                                unsigned long long* __restrict__ state) {
  const unsigned long long cur = state ? state[1] : 0ull;
  if (pack_needed(state)) pack_dyn_job(dp, S, A, ns, fp16, blob);
  pack_commit(state, cur);
}

// mobody_mlp_pack as one launch: blockIdx.y = layer.  nn.Linear weight is [out][in]: stride_k = 1, stride_n = K
__global__ void pack_mlp_kernel(const MlpPtrs mp, int din, int dout, int ns, int fp16, unsigned char* __restrict__ blob,
                                unsigned long long* __restrict__ state) {
  const unsigned long long cur = state ? state[1] : 0ull;
  if (pack_needed(state)) {
    const TcMlpLayout L = tc_mlp_layout(din, dout, ns);
    const int i = blockIdx.y;
    pack_weight(mp.w[i], 1, L.g[i].K, L.g[i], ns, fp16, 1.0f, reinterpret_cast<__nv_bfloat16*>(blob + L.w_off[i]));
    pack_bias(mp.b[i], 1, L.g[i].N, L.g[i].Np, 1.0f, reinterpret_cast<float*>(blob + L.bias_base) + L.b_off[i]);
  }
  pack_commit(state, cur);
}

}  // namespace tcs

const char* mb_tc_dyn_pack(const DynPtrs& dp, int S, int A, int ns, int fp16, unsigned char* blob, unsigned long long* state, cudaStream_t st) {
  if (fp16 && ns != 1) return "dyn_pack: fp16 is a single-plane format";
  if (ns != 1 && ns != 2) return "dyn_pack: nsplit must be 1 or 2";
  if (state) {
    tcs::ChecksumArgs c{}; c.count = 2 * L_COUNT;
    for (int l = 0; l < L_COUNT; ++l) {
      int in, out; tc_dyn_full_dims(l, S, A, &in, &out);
      c.p[2 * l] = dp.w[l]; c.n[2 * l] = (unsigned)(MB_E * in * out);
      c.p[2 * l + 1] = dp.b[l]; c.n[2 * l + 1] = (unsigned)(MB_E * out);
    }
    tcs::params_checksum_kernel<<<dim3(64, c.count), 256, 0, st>>>(c, state);
  }
  tcs::pack_dyn_kernel<<<dim3(8, MB_E * (PK_COUNT + 1)), 256, 0, st>>>(dp, S, A, ns, fp16, blob, state);
  return nullptr;
}

const char* mb_tc_mlp_pack(const MlpPtrs& mp, int din, int dout, int ns, int fp16, unsigned char* blob, unsigned long long* state, cudaStream_t st) {
  if (ns != 1 && ns != 2) return "mlp_pack: nsplit must be 1 or 2";
  if (state) {
    tcs::ChecksumArgs c{}; c.count = 6;
    const int K[3] = {din, 256, 256}, N[3] = {256, 256, dout};
    for (int l = 0; l < 3; ++l) { c.p[2 * l] = mp.w[l]; c.n[2 * l] = (unsigned)(K[l] * N[l]); c.p[2 * l + 1] = mp.b[l]; c.n[2 * l + 1] = (unsigned)N[l]; }
    tcs::params_checksum_kernel<<<dim3(32, c.count), 256, 0, st>>>(c, state);
  }
  tcs::pack_mlp_kernel<<<dim3(32, 3), 256, 0, st>>>(mp, din, dout, ns, fp16, blob, state);
  return nullptr;
}

static long long* g_tc_trace = nullptr;
void mb_tc_set_trace(long long* buf) { g_tc_trace = buf; }
long long* mb_tc_get_trace() { return g_tc_trace; }

const char* mb_tc_step_launch(const StepArgs& a, const unsigned char* dynb, const unsigned char* polb, int ns, cudaStream_t st) {
  if (a.B <= 0) return nullptr;
  const int S = a.S, A = a.A;
  if (S < 2 || S > 64 || A < 1 || A > 16) return "tensor-core step kernel supports 2 <= S <= 64, 1 <= A <= 16";
  if (!dynb) return "tensor-core step needs dyn_pack (mobody_dyn_pack)";
  const bool has_policy = polb != nullptr;
  if (has_policy && !a.act_out) return "tensor-core step with a fused policy needs act_out";
  tcs::Cfg cfg{};
  const TcSched sc = tst::tc_step_sched(a, ns, has_policy, 32, &cfg.pol_bias_base);   // epilogue chunks of 32 columns
  const TcDynLayout DL = tc_dyn_layout(S, A, ns);
  cfg.obs_kp = (uint32_t)tc_rup16(S); cfg.sas_kp = (uint32_t)tc_rup16(2 * S + A);
  cfg.sa_off = (cfg.obs_kp / 8) * 2048u;
  uint32_t small = cfg.sa_off + 4 * 2048u, sasb = (cfg.sas_kp / 8) * 2048u;
  cfg.small_plane = small > sasb ? small : sasb;
  cfg.stage_bytes = (uint32_t)ns * 256u * 32u;
  cfg.dyn_bias_base = (uint32_t)DL.bias_base;
  cfg.has_policy = has_policy ? 1 : 0;
  cfg.trace = g_tc_trace;
  const size_t fixed = (size_t)ns * tcs::MAIN_PLANE + (size_t)ns * cfg.small_plane + (2 * 4 * 128 + tcs::NB * tcs::BSLOT) * sizeof(float) + sizeof(tcs::Bars) + 128;
  const size_t budget = 227 * 1024;
  if (fixed + 2 * cfg.stage_bytes > budget) return "tensor-core step kernel: shared memory budget exceeded for this (S, A)";
  if (!tst::tc_stats_scratch_fits((size_t)ns * tcs::MAIN_PLANE, tcs::TM, S))   // A_main is the scratch; single plane: S <= 63
    return "tensor-core step kernel: operand planes too small for the statistics scratch at this (S, A)";
  int nst = (int)((budget - fixed) / cfg.stage_bytes);
  if (nst > tcs::MAX_NST) nst = tcs::MAX_NST;
  cfg.nst = nst;
  const size_t bytes = fixed + (size_t)nst * cfg.stage_bytes;
  auto kern = ns == 2 ? tcs::step_tc_kernel<2> : tcs::step_tc_kernel<1>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
    return "cudaFuncSetAttribute(step_tc_kernel) failed";
  const dim3 grid((a.B + tcs::TM - 1) / tcs::TM), block(32 * (4 * tcs::NG + 2));
  if (tst::tc_launch_persisting(kern, grid, block, bytes, st, dynb, DL.total_bytes, a, dynb, polb ? polb : dynb, sc, cfg) != cudaSuccess)
    return "step_tc_kernel launch failed";
  return nullptr;
}
