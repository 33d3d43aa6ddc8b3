// Fused one-step model rollout on the tensor cores on 64-row tiles (2 <= S <= 128, 1 <= A <= 32), sm_100a.  The kernel is a
// template over its arithmetic:
//  * F16 = false: bf16x2's arithmetic (bf16 hi+lo split of both operands, 3 MMAs per K step, inside the 1e-4 bound) on the
//    two-plane images of mobody_dyn_pack / mobody_mlp_pack.  It serves bf16x2_wide (65 <= S <= 128) and bf16x2_t64 (S <= 64
//    with A > 16 or 2S+A > 96: the shapes the 128-row kernel cannot hold, such as Adroit's pen at 45 / 24).
//  * F16 = true: the fp16 mode's arithmetic (step_duo.cu): one fp16 plane per operand, one MMA per K step and the
//    packed-half epilogue of tc_epi.cuh, inside the stated looser bound 5e-3.  It serves fp16_t64: the shapes of the fp32
//    mode that the fp16 mode's 128-row kernel refuses.
// Swish layers arrive pre-scaled by the packer for the mode's plane count.  What differs from step_tc.cu is the row tile:
// one CTA owns 64 rows (UMMA M = 64), so every operand plane is half the size of step_tc.cu's and the planes of S <= 128,
// A <= 32 (the [s | a | s'] plane of the reward model reaches K = 288) fit in shared memory next to a weight ring of at
// least 4 stages (DESIGN.md 4.1c, 4.1e).  The ensemble statistics, noise, pick, penalty, termination, the reward head's
// operand and the final write are the fp32 code of tc_step.cuh, shared with step_tc.cu and step_duo.cu (as are the layer
// schedule, the launch and the bias staging).
//
//  * producer warp: per layer, its bias (ring of NB slots) and the weight K steps through the ring (1-D TMA bulk copies,
//    mbarrier complete_tx): bf16x2, one K step of both planes per stage; fp16, up to F16_KPS K steps of its plane;
//  * MMA warp: one elected thread issues tcgen05.mma 64 x N x 16 into TMEM (two 256-column accumulators, ping-pong); in
//    fp16 it waits and commits once per ring stage, since one MMA is shorter than the issuing thread's wait and commit;
//  * 16 epilogue warps (4 groups x 4 TMEM lane quadrants).  An M = 64 accumulator puts row i in TMEM lane
//    32 * (i / 16) + i % 16, so quadrant q holds rows 16q .. 16q+15 in its first 16 lanes.  tcgen05.ld 16x32bx2 gives
//    thread `lane` row 16q + lane % 16 and, per 64-column chunk, the 8 columns group * 16 + (lane / 16) * 8: one K group
//    of the next layer's operand per thread and chunk.  The 8 threads of a row (4 groups x 2 halves) are its `slot`s.
//    Chunks are announced in order (one mbarrier per 64 columns) and the next layer's MMAs trail the epilogue by a chunk.
#include "tc_step.cuh"

namespace tcw {
using namespace tst;

constexpr int TM = 64;                   // rows per CTA (UMMA M)
constexpr int NG = 4;                    // epilogue groups of 4 warps (one warp per TMEM lane quadrant)
constexpr int SLOTS = 2 * NG;            // epilogue threads per row
constexpr int CHUNK = 64;                // accumulator columns per announced chunk
constexpr uint32_t KG = TM * 16;         // bytes of one 8-wide K group of one plane (64 rows x 8 x 16 bits)
constexpr uint32_t MAIN_PLANE = 32 * KG; // 64 rows x 256 k x 16 bits
constexpr int F16_KPS = 4;               // fp16: K steps of a 256-wide layer per ring stage (one 64-column chunk)
constexpr int MAX_NST = 12;
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

// F16: one fp16 plane per operand and the packed-half epilogue instead of the bf16 hi + lo planes and fp32 epilogue math
template <bool F16>
__global__ void __launch_bounds__(32 * (4 * NG + 2), 1)
step_wide_kernel(const StepArgs a, const unsigned char* __restrict__ dynb, const unsigned char* __restrict__ polb,
                 const __grid_constant__ TcSched sched, const Cfg cfg) {
  constexpr int NS = F16 ? 1 : 2;          // operand planes: fp16, or bf16 hi + lo
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
        tc_stage_bias(li, L, dynb, polb, cfg.dyn_bias_base, cfg.pol_bias_base, bias_s, bars->b_full, bars->b_empty);
        if constexpr (F16) {   // as many K steps per stage as fit (F16_KPS of a 256-wide layer, all of a narrow one): one copy
          const int kps = max(1, min((int)L.ksteps, (int)(cfg.stage_bytes / bytes)));
          for (int s = 0; s < L.ksteps; s += kps) {
            const uint32_t nb = (uint32_t)min(kps, (int)L.ksteps - s) * bytes;
            tc::mbar_wait(&bars->w_empty[stage], phase ^ 1u);
            tc::mbar_arrive_expect_tx(&bars->w_full[stage], nb);
            tc::bulk_g2s(wst + (size_t)stage * cfg.stage_bytes, src + (size_t)s * bytes, nb, &bars->w_full[stage]);
            if (++stage == cfg.nst) { stage = 0; phase ^= 1u; }
          }
        } else {
          for (int s = 0; s < L.ksteps; ++s) {
            tc::mbar_wait(&bars->w_empty[stage], phase ^ 1u);
            tc::mbar_arrive_expect_tx(&bars->w_full[stage], bytes);
            tc::bulk_g2s(wst + (size_t)stage * cfg.stage_bytes, src + (size_t)s * bytes, bytes, &bars->w_full[stage]);
            if (++stage == cfg.nst) { stage = 0; phase ^= 1u; }
          }
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
        const uint32_t bplane = (uint32_t)L.n * 32u, blbo = (uint32_t)L.n * 16u;
        if constexpr (F16) {
          // one wait and one commit per ring stage (the producer's K-step grouping); operand chunks are awaited per K step
          const uint32_t idesc = tc::make_idesc_f16(TM, L.n);
          const int kps = max(1, min((int)L.ksteps, (int)(cfg.stage_bytes / bplane)));
          for (int s0 = 0; s0 < L.ksteps; s0 += kps) {
            tc::mbar_wait(&bars->w_full[stage], wphase);
            tc::tc_fence_after();
            const int ne = min(kps, (int)L.ksteps - s0);
            for (int j = 0; j < ne; ++j) {
              const int s = s0 + j;
              if ((s & 3) == 0 && (s >> 2) < L.a_wait) {   // a chunk is 64 columns = 4 K steps
                const int c = s >> 2;
                tc::mbar_wait(&bars->a_ready[c], (aph >> c) & 1u); aph ^= (1u << c);
                tc::tc_fence_after();
              }
              const uint32_t ao = abase + (uint32_t)s * 2u * KG, bo = wst0 + (uint32_t)stage * cfg.stage_bytes + (uint32_t)j * bplane;
              tc::umma_bf16(dcol, tc::make_smem_desc(ao, KG, 128), tc::make_smem_desc(bo, blbo, 128), idesc, s > 0 ? 1u : 0u);
            }
            tc::umma_commit(&bars->w_empty[stage]);
            if (++stage == cfg.nst) { stage = 0; wphase ^= 1u; }
          }
        } else {
          const uint32_t idesc = tc::make_idesc_bf16(TM, L.n);
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
    // 8 fp32 values -> this thread's K group of row r in an operand plane (fp16: saturating at +-65504)
    auto put8 = [&](unsigned char* base, uint32_t plane, uint32_t off, const float (&v)[8]) {
      if constexpr (F16) store8_f16(base, off, v); else store8<NS>(base, plane, off, v);
    };
    // the accumulator columns [c * 64 + col0, +8) of layer l, this thread's row
    auto ld_acc = [&](int l, int c, uint32_t (&x)[8]) { tc::tmem_ld16x2_8(lane_addr + (uint32_t)(l & 1) * 256u + (uint32_t)(c * CHUNK), x); };

    // 256-wide hidden layer: act(x + b) -> A_main planes; chunks complete in order, TMEM loads one chunk ahead
    auto epi_act256 = [&](int l, bool relu) {
      const float* bias = bias_of(l) + col0;
      wait_d(l);
      uint32_t xa[8], xb[8];
      auto chunk = [&](int c, const uint32_t (&x)[8]) {
        float bv[8];
        ld8(bias + c * CHUNK, bv);
        const uint32_t off = (uint32_t)((c * CHUNK + col0) / 8) * KG + roff;
        if constexpr (F16) {
          uint32_t o[4];
          act8_f16(x, bv, o, relu);
          *reinterpret_cast<uint4*>(A_main + off) = make_uint4(o[0], o[1], o[2], o[3]);
        } else {
          float v[8];
          act8<NS>(x, bv, v, relu);
          store8<NS>(A_main, MAIN_PLANE, off, v);
        }
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

    // ---------------- prologue: obs (and given actions) -> operand planes ----------------
    {
      const float* orow = a.obs + grow * a.obs_ld;
      for (int kg = slot; kg < (int)cfg.obs_kp / 8; kg += SLOTS) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { int j = kg * 8 + i; v[i] = (valid && j < S) ? __ldg(orow + j) : 0.f; }
        put8(A_small, sp, (uint32_t)kg * KG + roff, v);
      }
      if (!cfg.has_policy && 2 + slot < (int)cfg.sa_kp / 8) {   // [zs | a]: K groups 2 .. sa_kp/8 - 1 hold a, zero-padded
        const float* arow = a.act + grow * a.act_ld;
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { int j = slot * 8 + i; v[i] = (valid && j < A) ? __ldg(arow + j) : 0.f; }
        put8(A_small, sp, cfg.sa_off + (uint32_t)(2 + slot) * KG + roff, v);
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
          put8(A_small, sp, cfg.sa_off + (uint32_t)(2 + slot) * KG + roff, v);
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
          put8(A_small, sp, cfg.sa_off + (uint32_t)slot * KG + roff, zs);
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
          if constexpr (F16) {
            uint32_t o[4];
            act8_f16(x, bias + col0, o, false);
            *reinterpret_cast<uint4*>(A_main + (uint32_t)slot * KG + roff) = make_uint4(o[0], o[1], o[2], o[3]);
          } else {
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = swish_ns<NS>(__uint_as_float(x[i]) + bias[col0 + i]);
            store8<NS>(A_main, MAIN_PLANE, (uint32_t)slot * KG + roff, v);
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
          uint32_t x[8];
          ld_acc(l, 0, x);
          tc::tmem_ld_wait();
          float v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = zs[i] + (__uint_as_float(x[i]) + bias[col0 + i]);
          put8(A_main, MAIN_PLANE, (uint32_t)slot * KG + roff, v);
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

    // ---------------- ensemble statistics, noise, pick, penalty, termination (tc_step.cuh) ----------------
    // Every dynamics MMA has completed, so both operand regions (A_main and the small planes behind it, contiguous) serve
    // as fp32 scratch: at S = 128 that holds 3 members' squared deviations per batch in bf16x2 and 1 in fp16 (one plane).
    float* nobs_s = reinterpret_cast<float*>(A_main);
    const float row_pmax = tc_stats<TM, EPI_WARPS, SLOTS>(a, S, B, row0, live, r, slot, valid, nobs_s,
                                                          NS * MAIN_PLANE + NS * cfg.small_plane, [](int) {});
    pen = tc_penalty_terminal<TM, EPI_WARPS, SLOTS>(a, S, row_pmax, red, r, slot, valid, grow, nobs_s, [](int) {});
    // [s | a | s'] over the obs / sa planes
    tc_sas_operand<SLOTS>(a, S, A, cfg.has_policy, (int)cfg.sas_kp, r, slot, valid, grow, nobs_s,
                          [&](int kg, const float (&v)[8]) { put8(A_small, sp, (uint32_t)kg * KG + roff, v); });
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
          if constexpr (F16) {   // the packed-half swish, unpacked for the fp32 dot
            uint32_t o[4];
            float v[8];
            act8_f16(x, bv, o, false);
#pragma unroll
            for (int i = 0; i < 4; ++i) unpack_f16x2(o[i], v[2 * i], v[2 * i + 1]);
#pragma unroll
            for (int i = 0; i < 8; ++i) part = fmaf(v[i], wv[i], part);
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) part = fmaf(swish_ns<NS>(__uint_as_float(x[i]) + bv[i]), wv[i], part);
          }
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
    if (slot == 0 && valid) tc_write_reward(a, grow, racc, pen);
  }

  tc::tc_fence_before();
  __syncthreads();
  if (warp == PROD_WARP) tc::tmem_dealloc(tmem, 512);
}

}  // namespace tcw

// fp16 = 1: the single-plane fp16 image and arithmetic (fp16_t64); 0: bf16x2's (bf16x2_wide, bf16x2_t64)
const char* mb_tc_wide_step_launch(const StepArgs& a, const unsigned char* dynb, const unsigned char* polb, int fp16, cudaStream_t st) {
  if (a.B <= 0) return nullptr;
  const int S = a.S, A = a.A;
  if (S < 2 || S > 128 || A < 1 || A > 32) return "wide tensor-core step kernel supports 2 <= S <= 128, 1 <= A <= 32";
  if (!dynb) return "tensor-core step needs dyn_pack (mobody_dyn_pack)";
  const bool has_policy = polb != nullptr;
  if (has_policy && !a.act_out) return "tensor-core step with a fused policy needs act_out";
  const int ns = fp16 ? 1 : 2;
  tcw::Cfg cfg{};
  const TcSched sc = tst::tc_step_sched(a, ns, has_policy, tcw::CHUNK, &cfg.pol_bias_base);   // epilogue chunks of 64 columns
  const TcDynLayout DL = tc_dyn_layout(S, A, ns);
  cfg.obs_kp = (uint32_t)tc_rup16(S); cfg.sa_kp = (uint32_t)tc_rup16(MB_LATENT + A); cfg.sas_kp = (uint32_t)tc_rup16(2 * S + A);
  cfg.sa_off = (cfg.obs_kp / 8) * tcw::KG;
  const uint32_t small = cfg.sa_off + (cfg.sa_kp / 8) * tcw::KG, sasb = (cfg.sas_kp / 8) * tcw::KG;
  cfg.small_plane = small > sasb ? small : sasb;
  cfg.stage_bytes = (fp16 ? (uint32_t)tcw::F16_KPS : 1u) * (uint32_t)ns * 256u * 32u;   // 32 KB (fp16) / 16 KB (bf16x2)
  cfg.dyn_bias_base = (uint32_t)DL.bias_base;
  cfg.has_policy = has_policy ? 1 : 0;
  const size_t fixed = (size_t)ns * tcw::MAIN_PLANE + (size_t)ns * cfg.small_plane + (2 * tcw::SLOTS * tcw::TM + tcw::NB * tcw::BSLOT) * sizeof(float) +
                       sizeof(tcw::Bars) + 128;
  const size_t budget = 227 * 1024;
  if (fixed + 4 * cfg.stage_bytes > budget) return "wide tensor-core step kernel: shared memory budget exceeded for this (S, A)";
  // both operand regions are the scratch (in fp16 at S = 128 that is one member per batch)
  if (!tst::tc_stats_scratch_fits((size_t)ns * (tcw::MAIN_PLANE + cfg.small_plane), tcw::TM, S))
    return "wide tensor-core step kernel: operand planes too small for the statistics scratch at this (S, A)";
  int nst = (int)((budget - fixed) / cfg.stage_bytes);
  if (nst > tcw::MAX_NST) nst = tcw::MAX_NST;
  cfg.nst = nst;
  const size_t bytes = fixed + (size_t)nst * cfg.stage_bytes;
  auto kern = fp16 ? tcw::step_wide_kernel<true> : tcw::step_wide_kernel<false>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
    return "cudaFuncSetAttribute(step_wide_kernel) failed";
  const dim3 grid((a.B + tcw::TM - 1) / tcw::TM), block(32 * (4 * tcw::NG + 2));
  if (tst::tc_launch_persisting(kern, grid, block, bytes, st, dynb, DL.total_bytes, a, dynb, polb ? polb : dynb, sc, cfg) != cudaSuccess)
    return "step_wide_kernel launch failed";
  return nullptr;
}
