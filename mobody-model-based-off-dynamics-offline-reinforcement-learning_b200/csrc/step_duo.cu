// Fused one-step model rollout, TWO 128-row tiles in flight per CTA (single-pass bf16 mode).
//
// Same math and per-layer schedule as step_tc.cu (SURVEY.md Appendix A.1; reference
// algo/dynamics/mobody_dynamics.py:193-265, algo/dynamics/mobody_module.py:217-330,
// algo/offline_offline/mobody.py:60-72).  In step_tc.cu one tile walks a serial chain in which the tensor pipe and
// the epilogue warps mostly take turns.  With a single bf16 plane the A operand of a tile is 64 KB, so two tiles
// (X and Y) fit in one SM: each owns one 256-column TMEM accumulator and its own operand planes, and they are
// staggered by one layer — while the 16 epilogue warps turn tile X's layer-l accumulator into the layer-(l+1)
// operand, the tensor pipe runs tile Y's layer l, then X's layer l+1, and so on.  Every barrier is CTA-local (no
// cluster), so the hand-offs cost what they cost in step_tc.cu.  The bf16 hi+lo mode does not fit (2 x 128 KB of A).
//
// Units are processed in (layer, tile) order by the producer warp (weights: one K step per ring stage, streamed once
// per unit; biases: once per layer), the MMA warp and the 16 epilogue warps.  The layer schedule, the bias staging and each
// tile's statistics phase (ensemble statistics, noise, pick, penalty, termination, the reward head's operand) and final
// write are the code of tc_step.cuh, shared with step_tc.cu and step_wide.cu.
#include "tc_step.cuh"
#include <stdlib.h>

namespace tcd {
using namespace tst;

constexpr int TM = 128;
constexpr uint32_t MAIN_PLANE = 65536;     // 128 rows x 256 k x bf16
constexpr int MAX_NST = 12;
constexpr int EPI_WARPS = 16, PROD_WARP = 16, MMA_WARP = 17, NTHREADS = 32 * 18;
constexpr int NS = 1;                      // single bf16 plane

struct Cfg {
  int nst;
  uint32_t stage_bytes, small_plane, sa_off, obs_kp, sas_kp;
  uint32_t dyn_bias_base, pol_bias_base;
  int has_policy, first_dyn;
  long long* trace;     // debug: clock64 stamps of CTA 0, [(layer * 2 + tile)][8]; nullptr in production
};

struct Bars {
  uint64_t w_full[MAX_NST], w_empty[MAX_NST];
  uint64_t a_ready[2], d_full[2], d_empty[2], b_full[NB], b_empty[NB];
  uint32_t tmem_slot, pad;
};

// F16: fp16 operands and the packed-half epilogue (tc_epi.cuh) instead of bf16 operands and fp32 epilogue math.
template <bool F16>
__global__ void __launch_bounds__(NTHREADS, 1)
step_duo_kernel(const StepArgs a, const unsigned char* __restrict__ dynb, const unsigned char* __restrict__ polb,
                const __grid_constant__ TcSched sched, const Cfg cfg) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int S = a.S, A = a.A, B = a.B;
  const int live = a.n_rows_dev ? min(*a.n_rows_dev, B) : B;
  const int cta_row0 = (int)blockIdx.x * 2 * TM;
  if (cta_row0 >= live) return;

  unsigned char* A_main = smem;                                        // [tile][kgroup 0..31][128 rows][8 k]
  unsigned char* A_small = A_main + 2 * MAIN_PLANE;                    // [tile][small_plane]
  unsigned char* wst = A_small + 2 * cfg.small_plane;
  float* red = reinterpret_cast<float*>(wst + (size_t)cfg.nst * cfg.stage_bytes);      // [2][4][128]
  float* bias_s = red + 2 * 4 * TM;                                                    // [NB][BSLOT]
  Bars* bars = reinterpret_cast<Bars*>(bias_s + NB * BSLOT);
  auto main_of = [&](int u) { return A_main + (size_t)u * MAIN_PLANE; };
  auto small_of = [&](int u) { return A_small + (size_t)u * cfg.small_plane; };

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    for (int i = 0; i < cfg.nst; ++i) { tc::mbar_init(&bars->w_full[i], 1); tc::mbar_init(&bars->w_empty[i], 1); }
    for (int u = 0; u < 2; ++u) {
      tc::mbar_init(&bars->a_ready[u], EPI_WARPS); tc::mbar_init(&bars->d_full[u], 1); tc::mbar_init(&bars->d_empty[u], EPI_WARPS);
    }
    for (int i = 0; i < NB; ++i) { tc::mbar_init(&bars->b_full[i], 1); tc::mbar_init(&bars->b_empty[i], 2 * EPI_WARPS); }
    tc::mbar_fence_init();
  }
  if (warp == PROD_WARP) tc::tmem_alloc(&bars->tmem_slot, 512);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = bars->tmem_slot;

  if (warp == PROD_WARP) {
    // ================= producer: every unit's weight K steps through the ring, every layer's bias once =================
    if (tc::elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int li = 0; li < sched.n_layers; ++li) {
        const TcLayer L = sched.L[li];
        const unsigned char* src = (L.blob ? polb : dynb) + L.w_off;
        const uint32_t bytes = (uint32_t)L.n * 32u;
        tc_stage_bias(li, L, dynb, polb, cfg.dyn_bias_base, cfg.pol_bias_base, bias_s, bars->b_full, bars->b_empty);
        // a unit's MMAs wait for the tile's whole previous epilogue, so nothing hides the ring's load -> MMA -> commit ->
        // reload round trip here: narrow layers put as many K steps as fit into one stage (one copy, one round trip)
        const int kps = max(1, min((int)L.ksteps, (int)(cfg.stage_bytes / bytes)));
        for (int u = 0; u < 2; ++u)
          for (int s = 0; s < L.ksteps; s += kps) {
            const uint32_t nb = (uint32_t)min(kps, (int)L.ksteps - s) * bytes;
            tc::mbar_wait(&bars->w_empty[stage], phase ^ 1u);
            tc::mbar_arrive_expect_tx(&bars->w_full[stage], nb);
            tc::bulk_g2s(wst + (size_t)stage * cfg.stage_bytes, src + (size_t)s * bytes, nb, &bars->w_full[stage]);
            if (++stage == cfg.nst) { stage = 0; phase ^= 1u; }
          }
      }
    }
  } else if (warp == MMA_WARP) {
    // ================= MMA issuer: units in (layer, tile) order; a unit starts when its tile's previous epilogue is done =================
    if (tc::elect_one()) {
      int stage = 0; uint32_t wphase = 0, aph[2] = {0u, 0u};
      const uint32_t wst0 = tc::smem_u32(wst);
      for (int li = 0; li < sched.n_layers; ++li) {
        const TcLayer L = sched.L[li];
        const uint32_t idesc = F16 ? tc::make_idesc_f16(128, L.n) : tc::make_idesc_bf16(128, L.n);
        const uint32_t blbo = (uint32_t)L.n * 16u;
        const int kps = max(1, min((int)L.ksteps, (int)(cfg.stage_bytes / ((uint32_t)L.n * 32u))));     // K steps per ring stage (see the producer)
        for (int u = 0; u < 2; ++u) {
          const uint32_t dcol = tmem + (uint32_t)u * 256u;
          if (li >= 1) tc::mbar_wait(&bars->d_empty[u], (uint32_t)((li - 1) & 1));      // accumulator of this tile drained
          if (L.a_wait) { tc::mbar_wait(&bars->a_ready[u], aph[u]); aph[u] ^= 1u; }       // operand written by the last epilogue
          tc::tc_fence_after();
          if (cfg.trace && blockIdx.x == 0) cfg.trace[(li * 2 + u) * 8 + 0] = clock64();
          uint32_t abase;
          if (L.a_region == REG_MAIN) abase = tc::smem_u32(main_of(u));
          else abase = tc::smem_u32(small_of(u)) + (L.a_region == REG_SA ? cfg.sa_off : 0u);
          // one barrier wait and one commit per ring STAGE; inside a stage only descriptor increments and MMAs (the issuing
          // thread's serial latency per K step, ~230 cycles with a wait in it, exceeds the 128 cycles the MMA itself takes)
          const uint32_t kb16 = ((uint32_t)L.n * 32u) >> 4;
          const uint64_t b_tmpl = tc::make_smem_desc(0, blbo, 128);
          uint64_t ad = tc::make_smem_desc(abase, 2048, 128);
          uint32_t acc = 0u;
          for (int s0 = 0; s0 < L.ksteps; s0 += kps) {
            tc::mbar_wait(&bars->w_full[stage], wphase);
            tc::tc_fence_after();
            uint64_t bd = b_tmpl + (uint64_t)((wst0 + (uint32_t)stage * cfg.stage_bytes) >> 4);
            const int ne = min(kps, (int)L.ksteps - s0);
            for (int j = 0; j < ne; ++j) {
              tc::umma_bf16(dcol, ad, bd, idesc, acc);
              acc = 1u; ad += 256u; bd += kb16;                          // next K step: 4096 bytes of A, one K step of B
            }
            tc::umma_commit(&bars->w_empty[stage]);
            if (++stage == cfg.nst) { stage = 0; wphase ^= 1u; }
          }
          tc::umma_commit(&bars->d_full[u]);
          if (cfg.trace && blockIdx.x == 0) cfg.trace[(li * 2 + u) * 8 + 2] = clock64();
        }
      }
    }
  } else {
    // ================= epilogue warps =================
    const int q = warp & 3, group = warp >> 2;
    const int r = q * 32 + lane;                                // row of the tile
    const int col0 = group * 8;                                 // this warp's first column inside a 32-column chunk
    const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16);
    const uint32_t sp = cfg.small_plane;
    float zs[2][8];
    float racc[2] = {0.f, 0.f}, pen[2] = {0.f, 0.f};

    auto row0_of = [&](int u) { return (size_t)cta_row0 + (size_t)u * TM; };
    const bool tracer = cfg.trace && blockIdx.x == 0 && warp == 0 && lane == 0;
    auto wait_d = [&](int u, int l) {
      if (tracer) cfg.trace[(l * 2 + u) * 8 + 3] = clock64();
      tc::mbar_wait(&bars->d_full[u], (uint32_t)(l & 1)); tc::tc_fence_after();
      if (tracer) cfg.trace[(l * 2 + u) * 8 + 4] = clock64();
    };
    int cur_l = 0;
    auto release_d = [&](int u) {
      if (tracer) cfg.trace[(cur_l * 2 + u) * 8 + 5] = clock64();
      tc::tc_fence_before(); __syncwarp();
      if (lane == 0) tc::mbar_arrive(&bars->d_empty[u]);
    };
    auto signal_a = [&](int u) {
      tc::fence_proxy_async_smem(); __syncwarp();
      if (lane == 0) tc::mbar_arrive(&bars->a_ready[u]);
    };
    auto bias_of = [&](int l) -> const float* {
      tc::mbar_wait(&bars->b_full[l & (NB - 1)], (uint32_t)((l / NB) & 1));
      return bias_s + (l & (NB - 1)) * BSLOT;
    };
    auto bias_done = [&](int l) { __syncwarp(); if (lane == 0) tc::mbar_arrive(&bars->b_empty[l & (NB - 1)]); };
    auto put8 = [&](unsigned char* base, uint32_t off, const float (&v)[8]) {      // 8 fp32 values -> one 16-byte operand word group
      if (F16) store8_f16(base, off, v); else store8<NS>(base, 0u, off, v);
    };
    auto ld8s = [&](const float* b, float (&bv)[8]) {
      const float4 t0 = *reinterpret_cast<const float4*>(b), t1 = *(reinterpret_cast<const float4*>(b) + 1);
      bv[0] = t0.x; bv[1] = t0.y; bv[2] = t0.z; bv[3] = t0.w; bv[4] = t1.x; bv[5] = t1.y; bv[6] = t1.z; bv[7] = t1.w;
    };

    // 256-wide hidden layer of tile u: act(x + b) -> A_main[u].  Nothing trails this epilogue chunk by chunk (the tile's
    // next MMA waits for the whole unit), so warp group g simply owns the 64-column slab [64 g, 64 g + 64): four TMEM
    // loads of 16 columns, double buffered, 16 independent activations in flight per warp.
    auto epi_act256 = [&](int l, int u, bool relu) {
      const float* bias = bias_of(l) + group * 64;
      const uint32_t t0 = lane_base + (uint32_t)u * 256u + (uint32_t)(group * 64);
      unsigned char* Am = main_of(u);
      wait_d(u, l);
      uint32_t xa[16], xb[16];
      auto slab = [&](int c, const uint32_t (&x)[16]) {            // columns 64 g + 16 c .. + 15 = k-groups 8 g + 2 c, + 1
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float bv[8];
          ld8s(bias + c * 16 + h * 8, bv);
          const uint32_t off = (uint32_t)(group * 8 + c * 2 + h) * 2048u + (uint32_t)r * 16u;
          if (F16) {
            uint32_t o[4];
            act8_f16(&x[h * 8], bv, o, relu);
            *reinterpret_cast<uint4*>(Am + off) = make_uint4(o[0], o[1], o[2], o[3]);
          } else {
            float v[8];
            act8<NS>(&x[h * 8], bv, v, relu);
            store8<NS>(Am, MAIN_PLANE, off, v);
          }
        }
      };
      tc::tmem_ld16(t0, xa);
#pragma unroll 1
      for (int c = 0; c < 4; c += 2) {
        tc::tmem_ld_wait();
        tc::tmem_ld16(t0 + (uint32_t)(c + 1) * 16u, xb);
        slab(c, xa);
        tc::tmem_ld_wait();
        if (c + 2 < 4) tc::tmem_ld16(t0 + (uint32_t)(c + 2) * 16u, xa);
        slab(c + 1, xb);
      }
      signal_a(u);
      release_d(u);
      bias_done(l);
    };

    // ---------------- prologue: obs (and given actions) of both tiles -> bf16 operand planes ----------------
    for (int u = 0; u < 2; ++u) {
      const size_t grow = row0_of(u) + r;
      const bool valid = grow < (size_t)live;
      const float* orow = a.obs + grow * a.obs_ld;
      unsigned char* As = small_of(u);
      for (int kg = group; kg < (int)cfg.obs_kp / 8; kg += 4) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { int j = kg * 8 + i; v[i] = (valid && j < S) ? __ldg(orow + j) : 0.f; }
        put8(As, (uint32_t)kg * 2048u + (uint32_t)r * 16u, v);
      }
      if (!cfg.has_policy && group < 2) {
        const float* arow = a.act + grow * a.act_ld;
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { int j = group * 8 + i; v[i] = (valid && j < A) ? __ldg(arow + j) : 0.f; }
        put8(As, cfg.sa_off + (uint32_t)(2 + group) * 2048u + (uint32_t)r * 16u, v);
      }
      signal_a(u);
    }

    // ---------------- ensemble statistics, noise, pick, penalty, termination, reward-head operand (tile u; tc_step.cuh) ----------------
    // The tile's A_main serves as fp32 scratch (every dynamics MMA of the tile has completed); [s | a | s'] aliases its
    // obs / sa planes.
    auto stats = [&](int u) {
      float* nobs_s = reinterpret_cast<float*>(main_of(u));
      const size_t grow = row0_of(u) + r;
      const bool valid = grow < (size_t)live;
      const float row_pmax = tc_stats<TM, EPI_WARPS, 4>(a, S, B, row0_of(u), live, r, group, valid, nobs_s, MAIN_PLANE, [](int) {});
      pen[u] = tc_penalty_terminal<TM, EPI_WARPS, 4>(a, S, row_pmax, red + u * 4 * TM, r, group, valid, grow, nobs_s, [](int) {});
      unsigned char* As = small_of(u);
      tc_sas_operand<4>(a, S, A, cfg.has_policy, (int)cfg.sas_kp, r, group, valid, grow, nobs_s,
                        [&](int kg, const float (&v)[8]) { put8(As, (uint32_t)kg * 2048u + (uint32_t)r * 16u, v); });
      epi_bar<EPI_WARPS>();   // every sas plane is written (and nobs_s is no longer needed) before the operand is announced
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&bars->a_ready[u]);
    };

    // ---------------- units in (layer, tile) order: the same order the MMA issuer follows ----------------
#pragma unroll 1
    for (int l = 0; l < sched.n_layers; ++l) {
      const int kind = sched.L[l].kind, n = sched.L[l].n;
      cur_l = l;
      const int e = (l >= cfg.first_dyn && kind != EPI_REWARD) ? (l - cfg.first_dyn) >> 3 : 0;
#pragma unroll 1
      for (int u = 0; u < 2; ++u) {
        const size_t grow = row0_of(u) + r;
        const bool valid = grow < (size_t)live;
        const uint32_t tbase = lane_base + (uint32_t)u * 256u;
        switch (kind) {
          case EPI_SWISH256: epi_act256(l, u, false); break;
          case EPI_RELU256: epi_act256(l, u, true); break;
          case EPI_ACTION: {                                    // policy head: tanh * max_action -> [zs | act] operand, act_out
            const float* bias = bias_of(l);
            wait_d(u, l);
            if (col0 < n) {
              uint32_t x[8];
              tc::tmem_ld8(tbase + (uint32_t)col0, x); tc::tmem_ld_wait();
              float v[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const int j = col0 + i;
                v[i] = (j < A) ? tanhf(__uint_as_float(x[i]) + bias[j]) * a.max_action : 0.f;
                if (valid && j < A && a.act_out) a.act_out[grow * A + j] = v[i];
              }
              put8(small_of(u), cfg.sa_off + (uint32_t)(2 + group) * 2048u + (uint32_t)r * 16u, v);
            }
            release_d(u); bias_done(l);
          } break;
          case EPI_ZS: {                                        // zs3 mu half: keep zs, write the zs part of [zs | act]
            const float* bias = bias_of(l);
            wait_d(u, l);
            if (col0 < n) {
              uint32_t x[8];
              tc::tmem_ld8(tbase + (uint32_t)col0, x); tc::tmem_ld_wait();
              float v[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) { zs[u][i] = __uint_as_float(x[i]) + bias[col0 + i]; v[i] = zs[u][i]; }
              put8(small_of(u), cfg.sa_off + (uint32_t)group * 2048u + (uint32_t)r * 16u, v);
            }
            signal_a(u);
            release_d(u); bias_done(l);
          } break;
          case EPI_G: {                                         // za1: swish -> 32-wide operand (aliases A_main[u])
            const float* bias = bias_of(l);
            wait_d(u, l);
            if (col0 < n) {
              uint32_t x[8];
              tc::tmem_ld8(tbase + (uint32_t)col0, x); tc::tmem_ld_wait();
              float v[8];
              act8<NS>(x, bias + col0, v, false);
              put8(main_of(u), (uint32_t)group * 2048u + (uint32_t)r * 16u, v);
            }
            signal_a(u);
            release_d(u); bias_done(l);
          } break;
          case EPI_Z: {                                         // za2 mu half: z = zs + za -> 16-wide operand
            const float* bias = bias_of(l);
            wait_d(u, l);
            if (col0 < n) {
              uint32_t x[8];
              tc::tmem_ld8(tbase + (uint32_t)col0, x); tc::tmem_ld_wait();
              float v[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) v[i] = zs[u][i] + (__uint_as_float(x[i]) + bias[col0 + i]);
              put8(main_of(u), (uint32_t)group * 2048u + (uint32_t)r * 16u, v);
            }
            signal_a(u);
            release_d(u); bias_done(l);
          } break;
          case EPI_MEAN: {                                      // transition3 -> mean[e] (info['samples'])
            const float* bias = bias_of(l);
            wait_d(u, l);
            for (int c0 = col0; c0 < n; c0 += 32) {
              uint32_t x[8];
              tc::tmem_ld8(tbase + (uint32_t)c0, x); tc::tmem_ld_wait();
              if (valid) {
                float* mrow = a.mean + ((size_t)e * B + grow) * S;
#pragma unroll
                for (int i = 0; i < 8; ++i) { const int col = c0 + i; if (col < S) mrow[col] = __uint_as_float(x[i]) + bias[col]; }
              }
            }
            release_d(u); bias_done(l);
            if (e == MB_E - 1) stats(u);
          } break;
          case EPI_REWARD: {                                    // reward_model2 -> swish -> dot reward_model3[:,0]
            const float* bslot = bias_of(l);
            const float* bias = bslot + group * 64;
            const float* w3 = bslot + 256 + group * 64;
            const uint32_t t0 = tbase + (uint32_t)(group * 64);
            float part = 0.f;
            wait_d(u, l);
            uint32_t xa[16], xb[16];
            auto slab = [&](int c, const uint32_t (&x)[16]) {
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                float bv[8], wv[8], v[8];
                ld8s(bias + c * 16 + h * 8, bv); ld8s(w3 + c * 16 + h * 8, wv);
                if (F16) {
                  uint32_t o[4];
                  act8_f16(&x[h * 8], bv, o, false);
#pragma unroll
                  for (int i = 0; i < 4; ++i) unpack_f16x2(o[i], v[2 * i], v[2 * i + 1]);
                } else act8<NS>(&x[h * 8], bv, v, false);
#pragma unroll
                for (int i = 0; i < 8; ++i) part = fmaf(v[i], wv[i], part);
              }
            };
            tc::tmem_ld16(t0, xa);
#pragma unroll 1
            for (int c = 0; c < 4; c += 2) {
              tc::tmem_ld_wait();
              tc::tmem_ld16(t0 + (uint32_t)(c + 1) * 16u, xb);
              slab(c, xa);
              tc::tmem_ld_wait();
              if (c + 2 < 4) tc::tmem_ld16(t0 + (uint32_t)(c + 2) * 16u, xa);
              slab(c + 1, xb);
            }
            const float b3 = bslot[512];
            release_d(u); bias_done(l);
            float* redu = red + u * 4 * TM;
            redu[group * TM + r] = part;
            epi_bar<EPI_WARPS>();
            if (group == 0) {
              float sum = 0.f;
#pragma unroll
              for (int g2 = 0; g2 < 4; ++g2) sum += redu[g2 * TM + r];
              racc[u] += sum + b3;
            }
          } break;
          default: break;
        }
      }
    }
    if (group == 0) {
      for (int u = 0; u < 2; ++u) {
        const size_t grow = row0_of(u) + r;
        if (grow < (size_t)live) tc_write_reward(a, grow, racc[u], pen[u]);
      }
    }
  }

  tc::tc_fence_before();
  __syncthreads();
  if (warp == PROD_WARP) tc::tmem_dealloc(tmem, 512);
}

}  // namespace tcd

long long* mb_tc_get_trace();

// Single-pass modes only.  Returns "" (empty string) when this (S, A) does not fit two tiles, so the caller falls back.
const char* mb_tc_duo_step_launch(const StepArgs& a, const unsigned char* dynb, const unsigned char* polb, int fp16, cudaStream_t st, bool* launched) {
  *launched = false;
  if (a.B <= 0) { *launched = true; return nullptr; }
  const int S = a.S, A = a.A, ns = 1;
  if (S < 2 || S > 64 || A < 1 || A > 16) return "tensor-core step kernel supports 2 <= S <= 64, 1 <= A <= 16";
  if (!dynb) return "tensor-core step needs dyn_pack (mobody_dyn_pack)";
  const bool has_policy = polb != nullptr;
  if (has_policy && !a.act_out) return "tensor-core step with a fused policy needs act_out";
  tcd::Cfg cfg{};
  // a_wait = 1: a layer's whole A operand is announced at once, by the tile's preceding epilogue / prologue / statistics phase
  const TcSched sc = tst::tc_step_sched(a, ns, has_policy, 256, &cfg.pol_bias_base);
  const TcDynLayout DL = tc_dyn_layout(S, A, ns);
  cfg.obs_kp = (uint32_t)tc_rup16(S); cfg.sas_kp = (uint32_t)tc_rup16(2 * S + A);
  cfg.sa_off = (cfg.obs_kp / 8) * 2048u;
  uint32_t small = cfg.sa_off + 4 * 2048u, sasb = (cfg.sas_kp / 8) * 2048u;
  cfg.small_plane = small > sasb ? small : sasb;
  cfg.dyn_bias_base = (uint32_t)DL.bias_base;
  cfg.has_policy = has_policy ? 1 : 0;
  cfg.first_dyn = sc.first_dyn;
  cfg.trace = mb_tc_get_trace();
  const size_t fixed = 2 * ((size_t)tcd::MAIN_PLANE + (size_t)cfg.small_plane) +
                       (2 * 4 * tcd::TM + tcd::NB * tcd::BSLOT) * sizeof(float) + sizeof(tcd::Bars) + 128;
  const size_t budget = 227 * 1024;
  // ring stage: 16 KB (two K steps of a 256-wide layer, every K step of a narrow one) when three of them fit, else 8 KB
  cfg.stage_bytes = 2u * 256u * 32u;
  if (fixed + 3 * cfg.stage_bytes > budget) cfg.stage_bytes = 256u * 32u;
  if (fixed + 3 * cfg.stage_bytes > budget) return nullptr;    // two tiles do not fit for this (S, A): caller falls back
  int nst = (int)((budget - fixed) / cfg.stage_bytes);
  if (nst > tcd::MAX_NST) nst = tcd::MAX_NST;
  cfg.nst = nst;
  const size_t bytes = fixed + (size_t)nst * cfg.stage_bytes;
  auto kern = fp16 ? tcd::step_duo_kernel<true> : tcd::step_duo_kernel<false>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
    return "cudaFuncSetAttribute(step_duo_kernel) failed";
  const int grid = (a.B + 2 * tcd::TM - 1) / (2 * tcd::TM);
  kern<<<grid, tcd::NTHREADS, bytes, st>>>(a, dynb, polb ? polb : dynb, sc, cfg);
  *launched = true;
  return nullptr;
}
