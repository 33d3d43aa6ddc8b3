// Dynamics fitting step (SURVEY.md section 8f rank 3): one mini-batch of MOBODYEnsembleDynamics.learn
// (reference algo/dynamics/mobody_dynamics.py:594-653) = encoder_loss (:300-329) + transition_loss (:336-347) +
// reward_loss (:349-386) + backward + torch.optim.Adam, for the default configuration (no_vae = 0, latent_reward = 0,
// inverse_sep_reward_loss = 0, mopo = 0), on the 7-member ensemble with per-member (bootstrapped) batches [7, B, .].
//
// The reference runs encode_state five times per batch (each with fresh reparameterisation noise), the transition head
// four times, the action encoder three times and the reward head twice; every one of those is the SAME weights on
// different rows, so here each network runs ONCE over a row-stacked operand:
//   trunk   zs1 -> zs2 -> zs3            on [s ; s']                                     (2B rows per member)
//   action  za1 -> za2                   on [z3|a ; z5|a ; z6|a]                         (3B)
//   head    t1 -> t2 -> t3               on [z1 ; z2 ; z5 + za5 ; z6 + za6]              (4B)
//   reward  r1 -> r2 -> r3               on [s|a|fake' ; s|a|s']                         (2B)
// (z1..z6 = the six reparameterised latents in the reference's call order; z4 carries no gradient.)  Every layer is one
// launch of the tcgen05 GEMM tile kernel (umma_gemm.cuh, 3xTF32, one job per ensemble member): forward with a fused
// bias + Swish epilogue that also keeps the pre-activation, backward-data with a fused Swish-derivative epilogue writing in
// place over that pre-activation, weight gradients as K-split partials.  The glue between the GEMMs (reparameterisation,
// row stacking, the ensemble std of reward_loss and its gradient, loss gradients, loss scalars, Adam) is a handful of
// elementwise kernels below.  All launches are chained with programmatic dependent launch.
#include "umma_gemm.cuh"
#include "philox.cuh"
#include "../../include/mobody_b200.h"
#include <math.h>
#include <stdlib.h>

const char* mb_gemm_launch(const ug::Args& a, cudaStream_t st);     // train_tc.cu

#define MB_STREAM_FIT 0x66697473u

namespace dfit {
constexpr int E = MB_E, H = MB_H, L = MB_LATENT, ZH = MB_ZAH;
__host__ __device__ inline int r4(int x) { return (x + 3) & ~3; }

struct Ws {
  float *X0, *P1, *H1, *P2, *H2, *O3;                    // trunk      [E][2B][.]
  float *ZAin, *PG, *G, *ZA;                             // action     [E][3B][.]
  float *TrIn, *PU1, *U1, *PU2, *U2, *M;                 // head       [E][4B][.]
  float *RIn, *PV1, *V1, *PV2, *V2, *R;                  // reward     [E][2B][.]
  float *ZL, *Z4;                                        // [E][B][16]: z3 + za3 and the no-grad next-state latent
  float *EL, *EN;                                        // generated noise (when not injected): [6][E][B][16], [E][B][S]
  float *STD, *MBAR;                                     // [B][S4] ensemble statistics of the reward path's predicted mean
  float *dR, *dRIn, *dM, *dTrIn, *dZA, *dZAin, *dO3;     // gradients of the linear outputs / stacked inputs
  float *gw[11], *gb[11];                                // weight-gradient partials [E][nsplit][out][in], [E][nsplit][out]
  float *part;                                           // [E][8] loss partial sums
};
struct Dims { int S, A, B, S4, LA, LA4, RI, RI4; };

struct FitArgs {
  Dims d; Ws w;
  const float *obs, *act, *nobs, *rew;                   // [E][B][S], [E][B][A], [E][B][S], [E][B]
  const float *el, *en;                                  // noise actually used (injected or generated)
  long long ms;                                          // rows between members in obs / act / nobs / rew
  int gen_noise; unsigned long long seed; unsigned int draw;
  float c_enc, c_rew;                                    // encoder-loss weight in the total (5 or 1 times encoder_loss_coef), reward weight (1 / 0.01)
  float* scalars;
};

__device__ __forceinline__ float fit_normal(unsigned long long seed, unsigned int draw, unsigned int stream, unsigned long long i) {
  const unsigned long long blk = i >> 2;
  const Philox4 b = philox4x32_10((uint32_t)blk, (uint32_t)(blk >> 32), draw, stream, (uint32_t)seed, MB_STREAM_FIT);
  const float two_pi = 6.283185307179586f;
  const uint32_t xa = (i & 2) ? b.z : b.x, xb = (i & 2) ? b.w : b.y;
  const float r = sqrtf(-2.0f * logf(philox_u01(xa))), t = two_pi * philox_u01(xb);
  float s, c; sincosf(t, &s, &c);
  return (i & 1) ? r * s : r * c;
}

// stage 0: row-stack the batch into the GEMM operands, draw the noise when it is not injected
__global__ void __launch_bounds__(256) prep_kernel(const FitArgs a) {
  mb_pdl_begin();
  const Dims d = a.d; const int B = d.B, S = d.S, A = d.A;
  const long long n_rows = (long long)E * B;
  const long long gsz = (long long)gridDim.x * blockDim.x, g0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (long long i = g0; i < n_rows * S; i += gsz) {                       // states
    const int j = (int)(i % S); const long long eb = i / S; const int e = (int)(eb / B), b = (int)(eb % B);
    const size_t src = ((size_t)e * a.ms + b) * S + j;
    const float s = a.obs[src], n = a.nobs[src];
    a.w.X0[((size_t)e * 2 * B + b) * d.S4 + j] = s;
    a.w.X0[((size_t)e * 2 * B + B + b) * d.S4 + j] = n;
    a.w.RIn[((size_t)e * 2 * B + b) * d.RI4 + j] = s;
    a.w.RIn[((size_t)e * 2 * B + B + b) * d.RI4 + j] = s;
    a.w.RIn[((size_t)e * 2 * B + B + b) * d.RI4 + S + A + j] = n;
  }
  for (long long i = g0; i < n_rows * A; i += gsz) {                       // actions
    const int j = (int)(i % A); const long long eb = i / A; const int e = (int)(eb / B), b = (int)(eb % B);
    const float v = a.act[((size_t)e * a.ms + b) * A + j];
    a.w.RIn[((size_t)e * 2 * B + b) * d.RI4 + S + j] = v;
    a.w.RIn[((size_t)e * 2 * B + B + b) * d.RI4 + S + j] = v;
#pragma unroll
    for (int k = 0; k < 3; ++k) a.w.ZAin[((size_t)e * 3 * B + (size_t)k * B + b) * d.LA4 + L + j] = v;
  }
  if (a.gen_noise) {
    for (long long i = g0; i < 6 * n_rows * L; i += gsz) a.w.EL[i] = fit_normal(a.seed, a.draw, 1u, (unsigned long long)i);
    for (long long i = g0; i < n_rows * S; i += gsz) a.w.EN[i] = fit_normal(a.seed, a.draw, 2u, (unsigned long long)i);
  }
}

// stage 1 (after the trunk): the six reparameterised latents, in the reference's call order
//   0 encoder_decoder(s)  1 encoder_decoder(s')  2 encode_state(s) [latent consistency]  3 encode_state(s') [no grad]
//   4 forward_*(s, a) of transition_loss         5 forward_*(s, a) of reward_loss
__global__ void __launch_bounds__(256) reparam_kernel(const FitArgs a) {
  mb_pdl_begin();
  const Dims d = a.d; const int B = d.B;
  const long long n = (long long)E * B * L;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(i % L); const long long eb = i / L; const int e = (int)(eb / B), b = (int)(eb % B);
    const float* os = a.w.O3 + ((size_t)e * 2 * B + b) * 32; const float* on = a.w.O3 + ((size_t)e * 2 * B + B + b) * 32;
    const float mu_s = os[j], sd_s = expf(0.5f * os[L + j]), mu_n = on[j], sd_n = expf(0.5f * on[L + j]);
    float ep[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) ep[k] = a.el[(size_t)k * E * B * L + i];
    a.w.TrIn[((size_t)e * 4 * B + b) * L + j] = mu_s + ep[0] * sd_s;
    a.w.TrIn[((size_t)e * 4 * B + B + b) * L + j] = mu_n + ep[1] * sd_n;
    a.w.ZAin[((size_t)e * 3 * B + b) * d.LA4 + j] = mu_s + ep[2] * sd_s;
    a.w.Z4[i] = mu_n + ep[3] * sd_n;
    a.w.ZAin[((size_t)e * 3 * B + B + b) * d.LA4 + j] = mu_s + ep[4] * sd_s;
    a.w.ZAin[((size_t)e * 3 * B + 2 * B + b) * d.LA4 + j] = mu_s + ep[5] * sd_s;
  }
}

// stage 2 (after the action encoder): z + za for the three action-conditioned passes
__global__ void __launch_bounds__(256) combine_kernel(const FitArgs a) {
  mb_pdl_begin();
  const Dims d = a.d; const int B = d.B;
  const long long n = (long long)E * B * L;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(i % L); const long long eb = i / L; const int e = (int)(eb / B), b = (int)(eb % B);
    float z[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const size_t row = (size_t)e * 3 * B + (size_t)k * B + b;
      z[k] = a.w.ZAin[row * d.LA4 + j] + a.w.ZA[row * 32 + j];
    }
    a.w.ZL[i] = z[0];
    a.w.TrIn[((size_t)e * 4 * B + 2 * B + b) * L + j] = z[1];
    a.w.TrIn[((size_t)e * 4 * B + 3 * B + b) * L + j] = z[2];
  }
}

// stage 3 (after the head): fake_next_state = mean + randn * std(mean, axis = ensemble) (unbiased; :354) -> reward operand
__global__ void __launch_bounds__(256) fake_kernel(const FitArgs a) {
  mb_pdl_begin();
  const Dims d = a.d; const int B = d.B, S = d.S;
  const long long n = (long long)B * S;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(i % S), b = (int)(i / S);
    float m[E], mb = 0.f;
#pragma unroll
    for (int e = 0; e < E; ++e) { m[e] = a.w.M[((size_t)e * 4 * B + 3 * B + b) * d.S4 + j]; mb += m[e]; }
    mb *= (1.0f / E);
    float v = 0.f;
#pragma unroll
    for (int e = 0; e < E; ++e) { const float t = m[e] - mb; v = fmaf(t, t, v); }
    const float sd = sqrtf(v * (1.0f / (E - 1)));
    a.w.STD[(size_t)b * d.S4 + j] = sd; a.w.MBAR[(size_t)b * d.S4 + j] = mb;
#pragma unroll
    for (int e = 0; e < E; ++e)
      a.w.RIn[((size_t)e * 2 * B + b) * d.RI4 + S + d.A + j] = m[e] + a.en[((size_t)e * B + b) * S + j] * sd;
  }
}

// stage 4 (after the reward head): gradients of the losses with respect to the network outputs
__global__ void __launch_bounds__(256) lossgrad_kernel(const FitArgs a) {
  mb_pdl_begin();
  const Dims d = a.d; const int B = d.B, S = d.S;
  const long long gsz = (long long)gridDim.x * blockDim.x, g0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const float inv_bs = 1.0f / ((float)B * (float)S), inv_bl = 1.0f / ((float)B * (float)L), inv_b = 1.0f / (float)B;
  for (long long i = g0; i < (long long)E * 3 * B * S; i += gsz) {        // head outputs of passes 0, 1, 4 (blocks 0..2)
    const int j = (int)(i % S); const long long t = i / S; const int r = (int)(t % (3 * B)), e = (int)(t / (3 * B));
    const int blk = r / B, b = r % B;
    const size_t off = ((size_t)e * 4 * B + r) * d.S4 + j;
    const float tgt = blk == 0 ? a.obs[((size_t)e * a.ms + b) * S + j] : a.nobs[((size_t)e * a.ms + b) * S + j];
    const float w = blk == 2 ? 2.0f * inv_bs : a.c_enc * 100.0f * 2.0f * inv_bs;
    a.w.dM[off] = w * (a.w.M[off] - tgt);
  }
  for (long long i = g0; i < (long long)E * 2 * B; i += gsz) {            // reward outputs (mu column; the logvar column has no loss)
    const int r = (int)(i % (2 * B)), e = (int)(i / (2 * B)), b = r % B;
    const float g = a.c_rew * 2.0f * inv_b * (a.w.R[(size_t)i * 4] - a.rew[(size_t)e * a.ms + b]);
    *reinterpret_cast<float4*>(a.w.dR + (size_t)i * 4) = make_float4(g, 0.f, 0.f, 0.f);
  }
  for (long long i = g0; i < (long long)E * B * 32; i += gsz) {           // latent consistency (:322-325): d/d(z3 + za3)
    const int j = (int)(i % 32); const long long eb = i / 32; const int e = (int)(eb / B), b = (int)(eb % B);
    float g = 0.f;
    if (j < L) { const size_t k = ((size_t)e * B + b) * L + j; g = a.c_enc * 2.0f * inv_bl * (a.w.ZL[k] - a.w.Z4[k]); }
    a.w.dZA[((size_t)e * 3 * B + b) * 32 + j] = g;
  }
}

// loss scalars: one block per member, fixed summation order; [e][0..4] = recon, kl, latent, transition, reward (unweighted means)
__global__ void __launch_bounds__(256) loss_kernel(const FitArgs a) {
  mb_pdl_begin();
  const Dims d = a.d; const int B = d.B, S = d.S, e = blockIdx.x, tid = threadIdx.x;
  float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  for (int i = tid; i < 3 * B * S; i += 256) {
    const int j = i % S, r = i / S, blk = r / B, b = r % B;
    const float tgt = blk == 0 ? a.obs[((size_t)e * a.ms + b) * S + j] : a.nobs[((size_t)e * a.ms + b) * S + j];
    const float t = a.w.M[((size_t)e * 4 * B + r) * d.S4 + j] - tgt;
    acc[blk == 2 ? 3 : 0] += t * t;
  }
  for (int i = tid; i < 2 * B * L; i += 256) {
    const int j = i % L, r = i / L;
    const float* o = a.w.O3 + ((size_t)e * 2 * B + r) * 32;
    const float mu = o[j], lv = o[L + j];
    acc[1] += -0.5f * (1.0f + lv - mu * mu - expf(lv));
  }
  for (int i = tid; i < B * L; i += 256) { const float t = a.w.ZL[(size_t)e * B * L + i] - a.w.Z4[(size_t)e * B * L + i]; acc[2] += t * t; }
  for (int i = tid; i < 2 * B; i += 256) { const float t = a.w.R[((size_t)e * 2 * B + i) * 4] - a.rew[(size_t)e * a.ms + i % B]; acc[4] += t * t; }
  __shared__ float red[5][256];
#pragma unroll
  for (int k = 0; k < 5; ++k) red[k][tid] = acc[k];
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (tid < s) {
#pragma unroll
      for (int k = 0; k < 5; ++k) red[k][tid] += red[k][tid + s];
    }
    __syncthreads();
  }
  if (tid == 0) {
    const float inv_bs = 1.0f / ((float)B * (float)S), inv_bl = 1.0f / ((float)B * (float)L);
    float* p = a.w.part + e * 8;
    p[0] = red[0][0] * inv_bs; p[1] = 0.05f * red[1][0] * inv_bl; p[2] = red[2][0] * inv_bl; p[3] = red[3][0] * inv_bs; p[4] = red[4][0] / (float)B;
  }
}
__global__ void finish_kernel(const FitArgs a) {
  mb_pdl_begin();
  if (threadIdx.x != 0) return;
  float s[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  for (int e = 0; e < E; ++e)
    for (int k = 0; k < 5; ++k) s[k] += a.w.part[e * 8 + k];
  const float enc = 100.0f * s[0] + s[1] + s[2], rw = a.c_rew * s[4];
  a.scalars[0] = s[3] + a.c_enc * enc + rw;     // loss (:623-641)
  a.scalars[1] = s[3];                          // transition_loss
  a.scalars[2] = enc;                           // encoder_loss
  a.scalars[3] = s[0];                          // recon_loss
  a.scalars[4] = s[1];                          // kl_loss
  a.scalars[5] = rw;                            // reward_loss
}

// stage 5 (after the reward head's backward): gradient of pass 5's predicted mean through fake_next_state, including the
// shared ensemble std: d std / d m_e = (m_e - mbar) / ((E - 1) std)
__global__ void __launch_bounds__(256) dfake_kernel(const FitArgs a) {
  mb_pdl_begin();
  const Dims d = a.d; const int B = d.B, S = d.S;
  const long long n = (long long)B * S;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(i % S), b = (int)(i / S);
    float df[E], g = 0.f;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      df[e] = a.w.dRIn[((size_t)e * 2 * B + b) * d.RI4 + S + d.A + j];
      g = fmaf(df[e], a.en[((size_t)e * B + b) * S + j], g);
    }
    const float sd = a.w.STD[(size_t)b * d.S4 + j], mb = a.w.MBAR[(size_t)b * d.S4 + j];
    const float k = g / ((float)(E - 1) * sd);
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const size_t off = ((size_t)e * 4 * B + 3 * B + b) * d.S4 + j;
      a.w.dM[off] = df[e] + k * (a.w.M[off] - mb);
    }
  }
}

// stage 6 (after the head's backward): the action encoder's output gradients of passes 4 and 5 = the head's input gradients
__global__ void __launch_bounds__(256) dza_kernel(const FitArgs a) {
  mb_pdl_begin();
  const int B = a.d.B;
  const long long n = (long long)E * 2 * B * 32;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(i % 32); const long long t = i / 32; const int r = (int)(t % (2 * B)), e = (int)(t / (2 * B));
    a.w.dZA[((size_t)e * 3 * B + B + r) * 32 + j] = j < L ? a.w.dTrIn[((size_t)e * 4 * B + 2 * B + r) * L + j] : 0.f;
  }
}

// stage 7 (after the action encoder's backward): gradient of the trunk output (mu | logvar) from the five differentiable
// latents and the two KL terms (:330-333)
__global__ void __launch_bounds__(256) do3_kernel(const FitArgs a) {
  mb_pdl_begin();
  const Dims d = a.d; const int B = d.B;
  const long long n = (long long)E * B * L;
  const float kl_w = a.c_enc * 0.05f / ((float)B * (float)L);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(i % L); const long long eb = i / L; const int e = (int)(eb / B), b = (int)(eb % B);
    const float* os = a.w.O3 + ((size_t)e * 2 * B + b) * 32; const float* on = a.w.O3 + ((size_t)e * 2 * B + B + b) * 32;
    const float mu_s = os[j], lv_s = os[L + j], mu_n = on[j], lv_n = on[L + j];
    const float sd_s = expf(0.5f * lv_s), sd_n = expf(0.5f * lv_n);
    const size_t t0 = ((size_t)e * 4 * B + b) * L + j, za0 = (size_t)e * 3 * B + b;
    const float dz1 = a.w.dTrIn[t0], dz2 = a.w.dTrIn[t0 + (size_t)B * L];
    const float dz3 = a.w.dZA[za0 * 32 + j] + a.w.dZAin[za0 * d.LA4 + j];
    const float dz5 = a.w.dTrIn[t0 + (size_t)2 * B * L] + a.w.dZAin[(za0 + B) * d.LA4 + j];
    const float dz6 = a.w.dTrIn[t0 + (size_t)3 * B * L] + a.w.dZAin[(za0 + 2 * B) * d.LA4 + j];
    const float e1 = a.el[i], e2 = a.el[(size_t)E * B * L + i], e3 = a.el[(size_t)2 * E * B * L + i];
    const float e5 = a.el[(size_t)4 * E * B * L + i], e6 = a.el[(size_t)5 * E * B * L + i];
    float* gs = a.w.dO3 + ((size_t)e * 2 * B + b) * 32; float* gn = a.w.dO3 + ((size_t)e * 2 * B + B + b) * 32;
    gs[j] = ((dz1 + dz3) + (dz5 + dz6)) + kl_w * mu_s;
    gs[L + j] = 0.5f * sd_s * (((dz1 * e1 + dz3 * e3) + (dz5 * e5 + dz6 * e6))) - 0.5f * kl_w * (1.0f - expf(lv_s));
    gn[j] = dz2 + kl_w * mu_n;
    gn[L + j] = 0.5f * sd_n * dz2 * e2 - 0.5f * kl_w * (1.0f - expf(lv_n));
  }
}

// torch.optim.Adam (lr, betas (0.9, 0.999), eps 1e-8, no weight decay; train_mobody.py:801-804) over the trained tensors.
// Gradients arrive as K-split partials in [e][split][out][in] order (the GEMM computes dW transposed: its row sums are the
// bias gradient); parameters are [e][in][out].
struct AdamJob { float* p; float* m; float* v; const float* g; int in, out, is_bias; float lr_over_bc1, inv_sqrt_bc2; };
struct AdamArgs { AdamJob job[22]; int njobs, nsplit; float b1, b2, eps; };
__device__ __forceinline__ void adam_update(const AdamArgs& a, const AdamJob& jb, size_t i, float g) {
  const float m0 = jb.m[i], m = m0 + (g - m0) * (1.0f - a.b1);              // exp_avg.lerp_(grad, 1 - beta1)
  const float v = a.b2 * jb.v[i] + (1.0f - a.b2) * g * g;
  jb.m[i] = m; jb.v[i] = v;
  const float denom = sqrtf(v) * jb.inv_sqrt_bc2 + a.eps;
  jb.p[i] = jb.p[i] - jb.lr_over_bc1 * (m / denom);
}
// Weights: 32 x 32 tiles through shared memory -- the gradient is read along `in` (its contiguous axis), the parameter and
// its moments are touched along `out` (theirs); every access is a full 128-byte line.  block = (32, 8).
__global__ void __launch_bounds__(256) adam_kernel(const __grid_constant__ AdamArgs a) {
  mb_pdl_begin();
  const AdamJob& jb = a.job[blockIdx.y];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  if (jb.is_bias) {
    const int n = E * jb.out;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
      const int e = i / jb.out, o = i % jb.out;
      float g = 0.f;
      for (int s = 0; s < a.nsplit; ++s) g += jb.g[((size_t)e * a.nsplit + s) * jb.out + o];
      adam_update(a, jb, (size_t)i, g);
    }
    return;
  }
  __shared__ float tile[32][33];
  const int to = (jb.out + 31) / 32, ti = (jb.in + 31) / 32, per = to * ti;
  for (int t = blockIdx.x; t < E * per; t += gridDim.x) {
    const int e = t / per, o0 = ((t % per) / ti) * 32, i0 = ((t % per) % ti) * 32;
#pragma unroll
    for (int k = 0; k < 4; ++k) {                                           // tile[o][i] <- sum over the K splits, lanes along `in`
      const int o = o0 + ty + 8 * k, ii = i0 + tx;
      float g = 0.f;
      if (o < jb.out && ii < jb.in)
        for (int s = 0; s < a.nsplit; ++s) g += jb.g[(((size_t)e * a.nsplit + s) * jb.out + o) * jb.in + ii];
      tile[ty + 8 * k][tx] = g;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {                                           // lanes along `out`
      const int ii = i0 + ty + 8 * k, o = o0 + tx;
      if (ii < jb.in && o < jb.out) adam_update(a, jb, ((size_t)e * jb.in + ii) * jb.out + o, tile[tx][ty + 8 * k]);
    }
    __syncthreads();
  }
}

struct LayerDef { int idx, in, out; };

static size_t carve(Ws& w, float* base, const Dims& d, int nsplit, const LayerDef* ly, bool gen_noise) {
  size_t off = 0;
  auto take = [&](size_t n) { float* p = base ? base + off : nullptr; off += (n + 3) & ~(size_t)3; return p; };
  const size_t B = d.B, e = E;
  w.X0 = take(e * 2 * B * d.S4); w.P1 = take(e * 2 * B * H); w.H1 = take(e * 2 * B * H); w.P2 = take(e * 2 * B * H); w.H2 = take(e * 2 * B * H);
  w.O3 = take(e * 2 * B * 32);
  w.ZAin = take(e * 3 * B * d.LA4); w.PG = take(e * 3 * B * ZH); w.G = take(e * 3 * B * ZH); w.ZA = take(e * 3 * B * 32);
  w.TrIn = take(e * 4 * B * L); w.PU1 = take(e * 4 * B * H); w.U1 = take(e * 4 * B * H); w.PU2 = take(e * 4 * B * H); w.U2 = take(e * 4 * B * H);
  w.M = take(e * 4 * B * d.S4);
  w.RIn = take(e * 2 * B * d.RI4); w.PV1 = take(e * 2 * B * H); w.V1 = take(e * 2 * B * H); w.PV2 = take(e * 2 * B * H); w.V2 = take(e * 2 * B * H);
  w.R = take(e * 2 * B * 4);
  w.ZL = take(e * B * L); w.Z4 = take(e * B * L);
  w.EL = take(gen_noise ? 6 * e * B * L : 0); w.EN = take(gen_noise ? e * B * d.S : 0);
  w.STD = take(B * d.S4); w.MBAR = take(B * d.S4);
  w.dR = take(e * 2 * B * 4); w.dRIn = take(e * 2 * B * d.RI4); w.dM = take(e * 4 * B * d.S4); w.dTrIn = take(e * 4 * B * L);
  w.dZA = take(e * 3 * B * 32); w.dZAin = take(e * 3 * B * d.LA4); w.dO3 = take(e * 2 * B * 32);
  for (int i = 0; i < 11; ++i) { w.gw[i] = take(e * nsplit * ly[i].in * ly[i].out); w.gb[i] = take(e * nsplit * ly[i].out); }
  w.part = take(e * 8);
  return off * sizeof(float);
}
static void layer_table(LayerDef* ly, int S, int A, int use_trg) {
  const LayerDef t[11] = {{L_ZS1, S, H}, {L_ZS2, H, H}, {L_ZS3, H, 2 * L},
                          {use_trg ? L_ZATRG1 : L_ZASRC1, L + A, ZH}, {use_trg ? L_ZATRG2 : L_ZASRC2, ZH, 2 * L},
                          {L_T1, L, H}, {L_T2, H, H}, {L_T3, H, S}, {L_R1, 2 * S + A, H}, {L_R2, H, H}, {L_R3, H, 2}};
  for (int i = 0; i < 11; ++i) ly[i] = t[i];
}
static Dims make_dims(int B, int S, int A) { return Dims{S, A, B, r4(S), L + A, r4(L + A), 2 * S + A, r4(2 * S + A)}; }
}  // namespace dfit

// The eleven weight-gradient launches depend only on their layer's output gradient and input activation, not on each other or
// on the backward-data chain: they run on a side stream (fork by event after the kernel that produces the gradient, join
// before Adam), so the chain of dependent launches is 32 long instead of 43.  MOBODY_DYNFIT_SIDE=0 keeps one stream.
namespace dfit {
struct SideStream { cudaStream_t s = nullptr; cudaEvent_t fork[12] = {}, join = nullptr; bool ok = false, tried = false; };
static SideStream& side_stream() {
  static SideStream per_dev[64];
  int dev = 0; cudaGetDevice(&dev);
  SideStream& ss = per_dev[dev & 63];
  if (!ss.tried) {
    ss.tried = true;
    const char* e = getenv("MOBODY_DYNFIT_SIDE");
    if (!(e && e[0] == '0') && cudaStreamCreateWithFlags(&ss.s, cudaStreamNonBlocking) == cudaSuccess) {
      ss.ok = cudaEventCreateWithFlags(&ss.join, cudaEventDisableTiming) == cudaSuccess;
      for (int i = 0; i < 12 && ss.ok; ++i) ss.ok = cudaEventCreateWithFlags(&ss.fork[i], cudaEventDisableTiming) == cudaSuccess;
    }
  }
  return ss;
}
}  // namespace dfit

long long mb_dynfit_workspace_bytes(int B, int S, int A, int nsplit) {
  dfit::Ws w; dfit::LayerDef ly[11]; dfit::layer_table(ly, S, A, 1);
  return (long long)dfit::carve(w, nullptr, dfit::make_dims(B, S, A), nsplit, ly, true);
}

const char* mb_dynfit_step_launch(const mobody_dynfit_desc& dsc, cudaStream_t st) {
  using namespace dfit;
  const int B = dsc.B, S = dsc.S, A = dsc.A, ns = dsc.nsplit;
  if (S > 128 || A > 64 || 2 * S + A > 256) return "dynfit: obs_dim <= 128, action_dim <= 64 and 2 * obs_dim + action_dim <= 256";
  if (ns < 1 || ns > 16) return "dynfit: nsplit must be 1..16";
  LayerDef ly[11]; layer_table(ly, S, A, dsc.use_trg);
  FitArgs fa{};
  fa.d = make_dims(B, S, A);
  const bool gen = !dsc.eps_latent || !dsc.eps_next;
  if ((size_t)dsc.workspace_bytes < carve(fa.w, reinterpret_cast<float*>(dsc.workspace), fa.d, ns, ly, true)) return "dynfit: workspace too small (mobody_dynfit_workspace_bytes)";
  if ((reinterpret_cast<uintptr_t>(dsc.workspace) & 15) != 0) return "dynfit: workspace must be 16-byte aligned";
  fa.obs = dsc.obs; fa.act = dsc.act; fa.nobs = dsc.next_obs; fa.rew = dsc.reward;
  fa.ms = dsc.member_stride > 0 ? dsc.member_stride : B;
  fa.gen_noise = gen ? 1 : 0; fa.seed = dsc.seed; fa.draw = dsc.draw;
  fa.el = gen ? fa.w.EL : dsc.eps_latent; fa.en = gen ? fa.w.EN : dsc.eps_next;
  fa.c_enc = dsc.encoder_coef; fa.c_rew = dsc.reward_coef; fa.scalars = dsc.scalars_out;
  const Dims& d = fa.d; const Ws& w = fa.w;
  const char* err = nullptr;
#define EW(kern, n) do { const long long nb_ = ((long long)(n) + 255) / 256; \
    if (mb_launch(kern, dim3((unsigned)(nb_ < 1 ? 1 : (nb_ > 1184 ? 1184 : nb_))), dim3(256), 0, st, fa) != cudaSuccess) return #kern " launch failed"; } while (0)
#define GEMM(args) do { if ((err = mb_gemm_launch(args, st))) return err; } while (0)
  SideStream& ss = side_stream();
  // weight gradient of layer li: on the side stream, after everything enqueued on `st` so far (its operands are complete)
#define WGRAD(li, ...) do { \
    if (ss.ok) { \
      if (cudaEventRecord(ss.fork[li], st) != cudaSuccess || cudaStreamWaitEvent(ss.s, ss.fork[li], 0) != cudaSuccess) return "dynfit: side-stream fork failed"; \
      if ((err = mb_gemm_launch(wgrad(li, __VA_ARGS__), ss.s))) return err; \
    } else if ((err = mb_gemm_launch(wgrad(li, __VA_ARGS__), st))) return err; } while (0)

  // ---- GEMM job builders: one job per ensemble member ----
  auto fwd = [&](int li, const float* X, int ldx, int rows, float* C, int ldc, float* pre) {
    ug::Args g{}; g.njobs = E; g.nsplit = 1;
    const LayerDef& l = ly[li];
    for (int e = 0; e < E; ++e) {
      ug::Job& j = g.job[e];
      j.A = X + (size_t)e * rows * ldx; j.lda = ldx; j.a_src = ug::SRC_KCONTIG;
      j.B = dsc.params.w[l.idx] + (size_t)e * l.in * l.out; j.ldb = l.out; j.b_src = ug::SRC_RCONTIG;
      j.M = rows; j.N = l.out; j.K = l.in; j.bias = dsc.params.b[l.idx] + (size_t)e * l.out;
      j.epi = pre ? ug::EPI_SWISH : ug::EPI_STORE;
      j.C = C + (size_t)e * rows * ldc; j.ldc = ldc; j.pre = pre ? pre + (size_t)e * rows * ldc : nullptr;
    }
    return g;
  };
  // dX = dY * W^T (optionally times swish'(pre of the producing layer), written in place over that pre-activation)
  auto bwd = [&](int li, const float* dY, int ldy, int rows, float* C, int ldc, const float* pre) {
    ug::Args g{}; g.njobs = E; g.nsplit = 1;
    const LayerDef& l = ly[li];
    for (int e = 0; e < E; ++e) {
      ug::Job& j = g.job[e];
      j.A = dY + (size_t)e * rows * ldy; j.lda = ldy; j.a_src = ug::SRC_KCONTIG;
      j.B = dsc.params.w[l.idx] + (size_t)e * l.in * l.out; j.ldb = l.out; j.b_src = ug::SRC_KCONTIG;
      j.M = rows; j.N = l.in; j.K = l.out;
      j.epi = pre ? ug::EPI_DSWISH : ug::EPI_STORE;
      j.mask = pre ? pre + (size_t)e * rows * ldc : nullptr; j.ldmask = ldc;
      j.C = C + (size_t)e * rows * ldc; j.ldc = ldc;
    }
    return g;
  };
  auto wgrad = [&](int li, const float* dY, int ldy, const float* X, int ldx, int rows) {
    ug::Args g{}; g.njobs = E; g.nsplit = ns;
    const LayerDef& l = ly[li];
    for (int e = 0; e < E; ++e) {
      ug::Job& j = g.job[e];
      j.A = dY + (size_t)e * rows * ldy; j.lda = ldy; j.a_src = ug::SRC_RCONTIG;
      j.B = X + (size_t)e * rows * ldx; j.ldb = ldx; j.b_src = ug::SRC_RCONTIG;
      j.M = l.out; j.N = l.in; j.K = rows; j.epi = ug::EPI_PART;
      j.C = w.gw[li] + (size_t)e * ns * l.out * l.in; j.db = w.gb[li] + (size_t)e * ns * l.out;
    }
    return g;
  };

  // ---------------- forward ----------------
  EW(prep_kernel, (long long)E * B * (gen ? 6 * L : S));
  GEMM(fwd(0, w.X0, d.S4, 2 * B, w.H1, H, w.P1));
  GEMM(fwd(1, w.H1, H, 2 * B, w.H2, H, w.P2));
  GEMM(fwd(2, w.H2, H, 2 * B, w.O3, 32, nullptr));
  EW(reparam_kernel, (long long)E * B * L);
  GEMM(fwd(3, w.ZAin, d.LA4, 3 * B, w.G, ZH, w.PG));
  GEMM(fwd(4, w.G, ZH, 3 * B, w.ZA, 32, nullptr));
  EW(combine_kernel, (long long)E * B * L);
  GEMM(fwd(5, w.TrIn, L, 4 * B, w.U1, H, w.PU1));
  GEMM(fwd(6, w.U1, H, 4 * B, w.U2, H, w.PU2));
  GEMM(fwd(7, w.U2, H, 4 * B, w.M, d.S4, nullptr));
  EW(fake_kernel, (long long)B * S);
  GEMM(fwd(8, w.RIn, d.RI4, 2 * B, w.V1, H, w.PV1));
  GEMM(fwd(9, w.V1, H, 2 * B, w.V2, H, w.PV2));
  GEMM(fwd(10, w.V2, H, 2 * B, w.R, 4, nullptr));
  // ---------------- losses ----------------
  EW(lossgrad_kernel, (long long)E * 3 * B * S);
  {   // the loss scalars feed nothing downstream: off the critical path (side stream; they only read forward results)
    cudaStream_t ls = st;
    if (ss.ok) {
      if (cudaEventRecord(ss.fork[11], st) != cudaSuccess || cudaStreamWaitEvent(ss.s, ss.fork[11], 0) != cudaSuccess) return "dynfit: side-stream fork failed";
      ls = ss.s;
    }
    if (mb_launch(loss_kernel, dim3(E), dim3(256), 0, ls, fa) != cudaSuccess) return "loss_kernel launch failed";
    if (mb_launch(finish_kernel, dim3(1), dim3(32), 0, ls, fa) != cudaSuccess) return "finish_kernel launch failed";
  }
  // ---------------- backward: reward head ----------------
  WGRAD(10, w.dR, 4, w.V2, H, 2 * B);
  GEMM(bwd(10, w.dR, 4, 2 * B, w.PV2, H, w.PV2));           // PV2 <- dL/d(pre of r2)
  WGRAD(9, w.PV2, H, w.V1, H, 2 * B);
  GEMM(bwd(9, w.PV2, H, 2 * B, w.PV1, H, w.PV1));           // PV1 <- dL/d(pre of r1)
  WGRAD(8, w.PV1, H, w.RIn, d.RI4, 2 * B);
  GEMM(bwd(8, w.PV1, H, 2 * B, w.dRIn, d.RI4, nullptr));
  EW(dfake_kernel, (long long)B * S);
  // ---------------- transition head ----------------
  WGRAD(7, w.dM, d.S4, w.U2, H, 4 * B);
  GEMM(bwd(7, w.dM, d.S4, 4 * B, w.PU2, H, w.PU2));
  WGRAD(6, w.PU2, H, w.U1, H, 4 * B);
  GEMM(bwd(6, w.PU2, H, 4 * B, w.PU1, H, w.PU1));
  WGRAD(5, w.PU1, H, w.TrIn, L, 4 * B);
  GEMM(bwd(5, w.PU1, H, 4 * B, w.dTrIn, L, nullptr));
  EW(dza_kernel, (long long)E * 2 * B * 32);
  // ---------------- action encoder ----------------
  WGRAD(4, w.dZA, 32, w.G, ZH, 3 * B);
  GEMM(bwd(4, w.dZA, 32, 3 * B, w.PG, ZH, w.PG));
  WGRAD(3, w.PG, ZH, w.ZAin, d.LA4, 3 * B);
  GEMM(bwd(3, w.PG, ZH, 3 * B, w.dZAin, d.LA4, nullptr));
  EW(do3_kernel, (long long)E * B * L);
  // ---------------- trunk ----------------
  WGRAD(2, w.dO3, 32, w.H2, H, 2 * B);
  GEMM(bwd(2, w.dO3, 32, 2 * B, w.P2, H, w.P2));
  WGRAD(1, w.P2, H, w.H1, H, 2 * B);
  GEMM(bwd(1, w.P2, H, 2 * B, w.P1, H, w.P1));
  WGRAD(0, w.P1, H, w.X0, d.S4, 2 * B);
  // ---------------- Adam ----------------
  if (ss.ok && (cudaEventRecord(ss.join, ss.s) != cudaSuccess || cudaStreamWaitEvent(st, ss.join, 0) != cudaSuccess)) return "dynfit: side-stream join failed";
  AdamArgs aa{}; aa.nsplit = ns; aa.b1 = 0.9f; aa.b2 = 0.999f; aa.eps = 1e-8f;
  for (int i = 0; i < 11; ++i) {
    const int t = (i == 3 || i == 4) ? dsc.t_action : dsc.t_shared;
    const double bc1 = 1.0 - pow(0.9, (double)t), bc2 = 1.0 - pow(0.999, (double)t);
    for (int k = 0; k < 2; ++k) {
      AdamJob& j = aa.job[aa.njobs++];
      j.p = k ? dsc.params.b[ly[i].idx] : dsc.params.w[ly[i].idx];
      j.m = k ? dsc.adam_m.b[ly[i].idx] : dsc.adam_m.w[ly[i].idx];
      j.v = k ? dsc.adam_v.b[ly[i].idx] : dsc.adam_v.w[ly[i].idx];
      j.g = k ? w.gb[i] : w.gw[i]; j.in = ly[i].in; j.out = ly[i].out; j.is_bias = k;
      j.lr_over_bc1 = (float)((double)dsc.lr / bc1); j.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
    }
  }
  if (mb_launch(adam_kernel, dim3(112, aa.njobs), dim3(256), 0, st, aa) != cudaSuccess) return "dynfit adam_kernel launch failed";
#undef EW
#undef GEMM
#undef WGRAD
  return nullptr;
}
