// C-ABI entry points (include/mobody_b200.h).  Argument checking + kernel launches only.
#include <stdio.h>
#include <string.h>
#include "../../include/mobody_b200.h"
#include "common.cuh"
#include "tc_layout.h"

// launchers implemented in the kernel translation units
const char* mb_simt_step_launch(const StepArgs& a, const DynPtrs& dp, const MlpPtrs* pol, cudaStream_t st);
const char* mb_simt_policy_launch(const float* obs, int B, int S, int A, const MlpPtrs& pol, float max_action,
                                  float* act_out, cudaStream_t st);
void mb_gather_rows_launch(const float* rows, const int64_t* idx, long long n, int rw, float* out, cudaStream_t st);
void mb_philox_indices_launch(int64_t* idx, long long n, unsigned long long seed, unsigned int draw, unsigned int size, cudaStream_t st);
void mb_sample_rows_launch(const mobody_sample_job* jobs, int njobs, int rw, cudaStream_t st);
void mb_pack_rows_launch(const float* s, const float* a, const float* ns, const float* r, const float* d, long long n,
                         int S, int A, int rw, int done_is_terminal, float* out, cudaStream_t st);
void mb_ring_insert_launch(const float* src, long long n_cap, const int* n_dev, int rw, long long ptr, long long cap,
                           float* dst, cudaStream_t st);
void mb_termination_launch(const float* x, long long n, int S, int kind, unsigned char* out, cudaStream_t st);
void mb_compact_launch(int kind, const unsigned char* flags, const float* vals, float thr, long long n_cap, const int* n_dev,
                       int* scratch, int* pos, int* count_out, cudaStream_t st);
void mb_gather_pos_launch(const float* src, int w, int src_ld, const int* pos, const int* m_dev, long long m_cap,
                          float* dst, int dst_ld, cudaStream_t st);
void mb_gather_pos_i64_launch(const long long* src, const int* pos, const int* m_dev, long long m_cap, long long* dst, cudaStream_t st);

void mb_rollout_init_launch(long long* row_ids, unsigned long long row0, int B, int T, float* pens, unsigned char* terms,
                            int* counts, cudaStream_t st);
void mb_rollout_advance_launch(const float* nexts, const long long* ids_prev, int S, const int* pos, const int* m_dev,
                               long long m_cap, float* obs_next, long long* ids_next, cudaStream_t st);
void mb_rollout_pack_launch(const float* obss, const float* acts, const float* nexts, const float* rews, const unsigned char* terms,
                            const float* pens, int S, int A, const int* pos, const int* m_dev, long long m_cap, float* packed,
                            cudaStream_t st);
void mb_rollout_stats_launch(const float* rews, const unsigned char* terms, long long n, double* partial, unsigned int* ticket,
                             double* stats, cudaStream_t st);
void mb_model_eval_init_launch(long long* row_ids, unsigned long long row0, int B, double* ret, double* ret_disc, int* length,
                               int* counts, cudaStream_t st);
void mb_model_eval_accumulate_launch(const float* reward, const long long* row_ids, unsigned long long row0, const int* n_dev,
                                     long long n_cap, int t, double disc, double* ret, double* ret_disc, int* length, cudaStream_t st);

const char* mb_tc_dyn_pack(const DynPtrs& dp, int S, int A, int ns, int fp16, unsigned char* blob, unsigned long long* state, cudaStream_t st);
const char* mb_tc_mlp_pack(const MlpPtrs& mp, int din, int dout, int ns, int fp16, unsigned char* blob, unsigned long long* state, cudaStream_t st);
const char* mb_tc_step_launch(const StepArgs& a, const unsigned char* dynb, const unsigned char* polb, int ns, cudaStream_t st);
const char* mb_tc_wide_step_launch(const StepArgs& a, const unsigned char* dynb, const unsigned char* polb, int fp16, cudaStream_t st);
const char* mb_tc_duo_step_launch(const StepArgs& a, const unsigned char* dynb, const unsigned char* polb, int fp16, cudaStream_t st, bool* launched);
const char* mb_umma_selftest_launch(const float* A, const float* B, int K, int N, int nsplit, float* D, cudaStream_t st);
void mb_ring_insert_transitions_launch(const float* packed, long long n_cap, const int* n_dev, int S, int A, int rw, long long ptr, long long cap,
                                        float* dst, cudaStream_t st);
void mb_par_penalty_launch(float* rows, int n, int S, int A, int rw, const float* pred, float coef, float* mean_out, cudaStream_t st);

long long mb_peer_slot_floats(long long cap_rows, int W);
long long mb_peer_buffer_bytes(int world, long long cap_rows, int W);
const char* mb_peer_slot(const mobody_peer_desc* p, int r, float** rows, int** header);
const char* mb_peer_ack_launch(const mobody_peer_desc* p, unsigned int consumed, cudaStream_t st);
const char* mb_peer_wait_launch(const mobody_peer_desc* p, cudaStream_t st);
const char* mb_peer_header_launch(const mobody_peer_desc* p, const int* kept_dev, const double* stats_dev, cudaStream_t st);
const char* mb_peer_push_launch(const mobody_peer_desc* p, const int* kept_dev, const double* stats_dev, cudaStream_t st);
const char* mb_gemm_selftest_launch(const float* A, const float* B, int M, int N, int K, int a_src, int b_src, int lda, int ldb,
                                    float* C, cudaStream_t st);
void mb_tc_set_trace(long long* buf);
long long mb_train_workspace_bytes(int N, int S, int A, int nsplit);
long long mb_train_ex_workspace_bytes(int N, int S, int A, int nsplit);
const char* mb_train_step_launch(const mobody_train_ex_desc& d, cudaStream_t st);

long long mb_classifier_workspace_bytes(int N, int S, int A, int nsplit);
const char* mb_classifier_step_launch(const mobody_classifier_desc& d, cudaStream_t st);
const char* mb_dara_relabel_launch(float* rows, long long n, int S, int A, int rw, const MlpPtrs& sas, const MlpPtrs& sa,
                                   float coef, float* pen_out, cudaStream_t st);

long long mb_dynfit_workspace_bytes(int B, int S, int A, int nsplit);
const char* mb_dynfit_step_launch(const mobody_dynfit_desc& d, cudaStream_t st);

static thread_local char g_err[512] = "";

static int fail(int code, const char* msg) {
  snprintf(g_err, sizeof(g_err), "%s", msg);
  return code;
}
static int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return MOBODY_ERR_CUDA;
  }
  return MOBODY_OK;
}

static_assert(sizeof(mobody_dyn_params) == sizeof(DynPtrs), "DynPtrs layout");
static_assert(sizeof(mobody_mlp_params) == sizeof(MlpPtrs), "MlpPtrs layout");
static_assert(MOBODY_N_DYN_LAYERS == L_COUNT, "layer count");

extern "C" {

int mobody_abi_version(void) { return MOBODY_ABI_VERSION; }
const char* mobody_last_error(void) { return g_err; }

int mobody_step(const mobody_step_desc* d, void* stream) {
  if (!d) return fail(MOBODY_ERR_ARG, "mobody_step: null descriptor");
  if (d->B < 0 || d->S < 2 || d->A < 1) return fail(MOBODY_ERR_ARG, "mobody_step: bad B/S/A");
  if (d->B == 0) return MOBODY_OK;
  if (!d->obs || !d->dyn || !d->next_obs || !d->reward || !d->penalty || !d->terminal || !d->mean)
    return fail(MOBODY_ERR_ARG, "mobody_step: obs, dyn, next_obs, reward, penalty, terminal and mean are required");
  if (!d->act && !d->policy) return fail(MOBODY_ERR_ARG, "mobody_step: need act or policy");
  if (!d->idx && (!d->elites || d->n_elites < 1)) return fail(MOBODY_ERR_ARG, "mobody_step: need idx or elites");
  if (d->term_kind < 0 || d->term_kind > MOBODY_TERM_PEN) return fail(MOBODY_ERR_ARG, "mobody_step: bad term_kind");
  if (d->term_kind == MOBODY_TERM_PEN && d->S < 27) return fail(MOBODY_ERR_ARG, "mobody_step: pen termination needs S >= 27");
  if (d->precision == MOBODY_PREC_BF16X2 || d->precision == MOBODY_PREC_FP16) {
    const int max_sas = d->precision == MOBODY_PREC_FP16 ? MOBODY_TC_FP16_MAX_SAS : MOBODY_TC_BF16X2_MAX_SAS;
    if (d->S > MOBODY_TC_MAX_S || d->A > MOBODY_TC_MAX_A || 2 * d->S + d->A > max_sas)
      return fail(MOBODY_ERR_ARG, "mobody_step: tensor-core modes take S <= 64, A <= 16 and 2S+A <= 96 (bf16x2) / 112 (fp16)");
  }
  if (d->precision == MOBODY_PREC_BF16X2_WIDE &&
      (d->S < MOBODY_TC_WIDE_MIN_S || d->S > MOBODY_TC_WIDE_MAX_S || d->A > MOBODY_TC_WIDE_MAX_A))
    return fail(MOBODY_ERR_ARG, "mobody_step: bf16x2_wide takes 65 <= S <= 128 and A <= 32");
  if (d->precision == MOBODY_PREC_BF16X2_T64 &&
      (d->S > MOBODY_TC_T64_MAX_S || d->A > MOBODY_TC_T64_MAX_A ||
       (d->A <= MOBODY_TC_MAX_A && 2 * d->S + d->A <= MOBODY_TC_BF16X2_MAX_SAS)))
    return fail(MOBODY_ERR_ARG, "mobody_step: bf16x2_t64 takes S <= 64, A <= 32 with A > 16 or 2S+A > 96");
  if (d->precision == MOBODY_PREC_FP16_T64 &&
      (d->S > MOBODY_TC_WIDE_MAX_S || d->A > MOBODY_TC_WIDE_MAX_A ||
       (d->S <= MOBODY_TC_MAX_S && d->A <= MOBODY_TC_MAX_A && 2 * d->S + d->A <= MOBODY_TC_FP16_MAX_SAS)))
    return fail(MOBODY_ERR_ARG, "mobody_step: fp16_t64 takes S <= 128, A <= 32 outside fp16's S <= 64, A <= 16, 2S+A <= 112");
  StepArgs a;
  memset(&a, 0, sizeof(a));
  a.obs = d->obs; a.act = d->policy ? nullptr : d->act; a.eps = d->eps; a.idx = d->idx; a.elites = d->elites;
  a.n_elites = d->n_elites; a.B = d->B; a.S = d->S; a.A = d->A; a.n_rows_dev = d->n_rows_dev; a.row_ids = d->row_ids;
  a.obs_ld = d->obs_ld ? d->obs_ld : d->S; a.act_ld = d->act_ld ? d->act_ld : d->A;
  if (a.obs_ld < d->S || a.act_ld < d->A) return fail(MOBODY_ERR_ARG, "mobody_step: obs_ld / act_ld smaller than S / A");
  a.use_trg = d->use_trg; a.use_penalty = d->use_penalty; a.term_kind = d->term_kind;
  a.coef = d->penalty_coef; a.max_action = d->max_action; a.seed = d->seed; a.row0 = d->row0; a.step = d->step;
  a.act_out = d->act_out; a.next_obs = d->next_obs; a.reward = d->reward; a.raw_reward = d->raw_reward;
  a.penalty = d->penalty; a.terminal = d->terminal; a.mean = d->mean;
  DynPtrs dp; memcpy(&dp, d->dyn, sizeof(dp));
  for (int i = 0; i < L_COUNT; ++i)
    if (!dp.w[i] || !dp.b[i]) return fail(MOBODY_ERR_ARG, "mobody_step: null dynamics parameter pointer");
  MlpPtrs pol; const MlpPtrs* polp = nullptr;
  if (d->policy) { memcpy(&pol, d->policy, sizeof(pol)); polp = &pol; }
  const char* err = nullptr;
  switch (d->precision) {
    case MOBODY_PREC_FP32: err = mb_simt_step_launch(a, dp, polp, (cudaStream_t)stream); break;
    case MOBODY_PREC_FP16: {
      if (!d->dyn_pack) return fail(MOBODY_ERR_ARG, "mobody_step: tensor-core precision needs dyn_pack (mobody_dyn_pack)");
      if (d->policy && !d->policy_pack) return fail(MOBODY_ERR_ARG, "mobody_step: fused policy needs policy_pack (mobody_mlp_pack)");
      bool launched = false;
      err = mb_tc_duo_step_launch(a, (const unsigned char*)d->dyn_pack, d->policy ? (const unsigned char*)d->policy_pack : nullptr, 1,
                                  (cudaStream_t)stream, &launched);
      if (!err && !launched) err = "fp16 mode: two row tiles do not fit in shared memory for this (S, A); use bf16 or bf16x2";
    } break;
    case MOBODY_PREC_BF16X2:
    case MOBODY_PREC_BF16:
      if (!d->dyn_pack) return fail(MOBODY_ERR_ARG, "mobody_step: tensor-core precision needs dyn_pack (mobody_dyn_pack)");
      if (d->policy && !d->policy_pack) return fail(MOBODY_ERR_ARG, "mobody_step: fused policy needs policy_pack (mobody_mlp_pack)");
      {   // one CTA per 128-row tile; the single bf16 plane (diagnostic mode) fits two row tiles per SM -> two-tiles-in-flight kernel
        if (d->precision == MOBODY_PREC_BF16) {
          bool launched = false;
          err = mb_tc_duo_step_launch(a, (const unsigned char*)d->dyn_pack, d->policy ? (const unsigned char*)d->policy_pack : nullptr, 0,
                                      (cudaStream_t)stream, &launched);
          if (err) return fail(MOBODY_ERR_UNSUPPORTED, err);
          if (launched) return check_launch("mobody_step");
        }
        err = mb_tc_step_launch(a, (const unsigned char*)d->dyn_pack, d->policy ? (const unsigned char*)d->policy_pack : nullptr,
                                d->precision == MOBODY_PREC_BF16X2 ? 2 : 1, (cudaStream_t)stream);
      }
      break;
    case MOBODY_PREC_BF16X2_WIDE:
    case MOBODY_PREC_BF16X2_T64:
    case MOBODY_PREC_FP16_T64:
      if (!d->dyn_pack) return fail(MOBODY_ERR_ARG, "mobody_step: tensor-core precision needs dyn_pack (mobody_dyn_pack)");
      if (d->policy && !d->policy_pack) return fail(MOBODY_ERR_ARG, "mobody_step: fused policy needs policy_pack (mobody_mlp_pack)");
      err = mb_tc_wide_step_launch(a, (const unsigned char*)d->dyn_pack, d->policy ? (const unsigned char*)d->policy_pack : nullptr,
                                   d->precision == MOBODY_PREC_FP16_T64, (cudaStream_t)stream);
      break;
    default: return fail(MOBODY_ERR_UNSUPPORTED, "mobody_step: unknown precision mode");
  }
  if (err) return fail(MOBODY_ERR_UNSUPPORTED, err);
  return check_launch("mobody_step");
}

int mobody_policy_forward(const float* obs, int B, int S, int A, const mobody_mlp_params* policy, float max_action,
                          float* act_out, void* stream) {
  if (B < 0 || !policy || (B > 0 && (!obs || !act_out))) return fail(MOBODY_ERR_ARG, "mobody_policy_forward: bad arguments");
  MlpPtrs pol; memcpy(&pol, policy, sizeof(pol));
  const char* err = mb_simt_policy_launch(obs, B, S, A, pol, max_action, act_out, (cudaStream_t)stream);
  if (err) return fail(MOBODY_ERR_UNSUPPORTED, err);
  return check_launch("mobody_policy_forward");
}

int mobody_termination(const float* next_obs, long long n, int S, int term_kind, unsigned char* out, void* stream) {
  if (n < 0 || S < 1 || term_kind < 0 || term_kind > MOBODY_TERM_PEN) return fail(MOBODY_ERR_ARG, "mobody_termination: bad arguments");
  if (term_kind == MOBODY_TERM_PEN && S < 27) return fail(MOBODY_ERR_ARG, "mobody_termination: pen needs S >= 27");
  if ((term_kind == MOBODY_TERM_HOPPER || term_kind == MOBODY_TERM_WALKER2D) && S < 2)
    return fail(MOBODY_ERR_ARG, "mobody_termination: hopper/walker2d need S >= 2");
  if (n > 0 && (!next_obs || !out)) return fail(MOBODY_ERR_ARG, "mobody_termination: null pointer");
  mb_termination_launch(next_obs, n, S, term_kind, out, (cudaStream_t)stream);
  return check_launch("mobody_termination");
}

int mobody_row_width(int S, int A) { return (2 * S + A + 2 + 3) & ~3; }

int mobody_gather_rows(const float* rows, const int64_t* idx, long long n, int row_width, float* out, void* stream) {
  if (n < 0 || row_width <= 0 || (row_width & 3)) return fail(MOBODY_ERR_ARG, "mobody_gather_rows: row_width must be a positive multiple of 4");
  if (n > 0 && (!rows || !idx || !out)) return fail(MOBODY_ERR_ARG, "mobody_gather_rows: null pointer");
  mb_gather_rows_launch(rows, idx, n, row_width, out, (cudaStream_t)stream);
  return check_launch("mobody_gather_rows");
}

int mobody_philox_indices(int64_t* idx, long long n, unsigned long long seed, unsigned int draw, unsigned int size, void* stream) {
  if (n < 0 || size == 0 || (n > 0 && !idx)) return fail(MOBODY_ERR_ARG, "mobody_philox_indices: bad arguments (size must be > 0)");
  mb_philox_indices_launch(idx, n, seed, draw, size, (cudaStream_t)stream);
  return check_launch("mobody_philox_indices");
}

int mobody_sample_rows(const mobody_sample_job* jobs, int njobs, int row_width, void* stream) {
  if (!jobs || njobs < 1 || njobs > 4 || row_width <= 0 || (row_width & 3)) return fail(MOBODY_ERR_ARG, "mobody_sample_rows: bad arguments");
  for (int b = 0; b < njobs; ++b)
    if (jobs[b].n < 0 || (jobs[b].n > 0 && (!jobs[b].rows || !jobs[b].out || jobs[b].size == 0)))
      return fail(MOBODY_ERR_ARG, "mobody_sample_rows: null pointer or empty buffer");
  mb_sample_rows_launch(jobs, njobs, row_width, (cudaStream_t)stream);
  return check_launch("mobody_sample_rows");
}

int mobody_pack_rows(const float* s, const float* a, const float* ns, const float* r, const float* d, long long n,
                     int S, int A, int done_is_terminal, float* out_rows, void* stream) {
  if (n < 0 || S < 1 || A < 1 || S > 1024 || A > 1024) return fail(MOBODY_ERR_ARG, "mobody_pack_rows: bad arguments");
  if (n > 0 && (!s || !a || !ns || !r || !d || !out_rows)) return fail(MOBODY_ERR_ARG, "mobody_pack_rows: null pointer");
  mb_pack_rows_launch(s, a, ns, r, d, n, S, A, mobody_row_width(S, A), done_is_terminal, out_rows, (cudaStream_t)stream);
  return check_launch("mobody_pack_rows");
}

int mobody_ring_insert(const float* src_rows, long long n_cap, const int* n_dev, int row_width, long long ptr,
                       long long cap, float* dst_rows, void* stream) {
  if (n_cap < 0 || cap <= 0 || ptr < 0 || ptr >= cap || (row_width & 3) || row_width <= 0)
    return fail(MOBODY_ERR_ARG, "mobody_ring_insert: bad arguments");
  // the reference handles a single wrap only (utils.py:78-92); a longer batch is a shape error there
  if (n_cap > cap) return fail(MOBODY_ERR_ARG, "mobody_ring_insert: batch larger than buffer capacity");
  if (n_cap > 0 && (!src_rows || !dst_rows)) return fail(MOBODY_ERR_ARG, "mobody_ring_insert: null pointer");
  mb_ring_insert_launch(src_rows, n_cap, n_dev, row_width, ptr, cap, dst_rows, (cudaStream_t)stream);
  return check_launch("mobody_ring_insert");
}

int mobody_ring_insert_transitions(const float* packed, long long n_cap, const int* n_dev, int S, int A, long long ptr,
                                   long long cap, float* dst_rows, void* stream) {
  if (n_cap < 0 || cap <= 0 || ptr < 0 || ptr >= cap || S < 1 || A < 1) return fail(MOBODY_ERR_ARG, "mobody_ring_insert_transitions: bad arguments");
  if (n_cap > cap) return fail(MOBODY_ERR_ARG, "mobody_ring_insert_transitions: batch larger than buffer capacity");
  if (n_cap > 0 && (!packed || !dst_rows)) return fail(MOBODY_ERR_ARG, "mobody_ring_insert_transitions: null pointer");
  mb_ring_insert_transitions_launch(packed, n_cap, n_dev, S, A, mobody_row_width(S, A), ptr, cap, dst_rows, (cudaStream_t)stream);
  return check_launch("mobody_ring_insert_transitions");
}

int mobody_par_penalty(float* rows, int n, int S, int A, int row_width, const float* pred_next, float coef,
                       float* mean_out, void* stream) {
  if (n < 0 || S < 1 || A < 1 || row_width != mobody_row_width(S, A)) return fail(MOBODY_ERR_ARG, "mobody_par_penalty: bad arguments");
  if (n > 0 && (!rows || !pred_next)) return fail(MOBODY_ERR_ARG, "mobody_par_penalty: null pointer");
  if (n == 0) return MOBODY_OK;
  mb_par_penalty_launch(rows, n, S, A, row_width, pred_next, coef, mean_out, (cudaStream_t)stream);
  return check_launch("mobody_par_penalty");
}

long long mobody_compact_scratch_ints(long long n_cap) { return (n_cap + 1023) / 1024 + 1; }

int mobody_compact(int keep_kind, const unsigned char* flags, const float* vals, float thr, long long n_cap,
                   const int* n_dev, int* scratch, int* pos, int* count_out, void* stream) {
  if (n_cap < 0 || n_cap > 0x7fffffffLL || !count_out) return fail(MOBODY_ERR_ARG, "mobody_compact: bad arguments");
  const bool u8 = keep_kind == MOBODY_KEEP_U8_ZERO || keep_kind == MOBODY_KEEP_U8_VALID;
  if (u8 ? (n_cap > 0 && !flags) : (n_cap > 0 && !vals))
    return fail(MOBODY_ERR_ARG, "mobody_compact: predicate input missing");
  if (keep_kind < 0 || keep_kind > MOBODY_KEEP_U8_VALID) return fail(MOBODY_ERR_ARG, "mobody_compact: bad keep_kind");
  if (n_cap > 0 && (!scratch || !pos)) return fail(MOBODY_ERR_ARG, "mobody_compact: null pointer");
  mb_compact_launch(keep_kind, flags, vals, thr, n_cap, n_dev, scratch, pos, count_out, (cudaStream_t)stream);
  return check_launch("mobody_compact");
}

int mobody_gather_pos(const float* src, int w, int src_ld, const int* pos, const int* m_dev, long long m_cap,
                      float* dst, int dst_ld, void* stream) {
  if (m_cap < 0 || w < 1 || src_ld < w || dst_ld < w) return fail(MOBODY_ERR_ARG, "mobody_gather_pos: bad arguments");
  if (m_cap > 0 && (!src || !pos || !dst)) return fail(MOBODY_ERR_ARG, "mobody_gather_pos: null pointer");
  mb_gather_pos_launch(src, w, src_ld, pos, m_dev, m_cap, dst, dst_ld, (cudaStream_t)stream);
  return check_launch("mobody_gather_pos");
}

int mobody_gather_pos_i64(const long long* src, const int* pos, const int* m_dev, long long m_cap, long long* dst, void* stream) {
  if (m_cap < 0 || (m_cap > 0 && (!src || !pos || !dst))) return fail(MOBODY_ERR_ARG, "mobody_gather_pos_i64: bad arguments");
  mb_gather_pos_i64_launch(src, pos, m_dev, m_cap, dst, (cudaStream_t)stream);
  return check_launch("mobody_gather_pos_i64");
}

int mobody_rollout_stats_doubles(void) { return 2 + 2 * MB_STATS_BLOCKS; }

int mobody_rollout(const mobody_rollout_desc* d, void* stream) {
  if (!d) return fail(MOBODY_ERR_ARG, "mobody_rollout: null descriptor");
  const mobody_step_desc& s0 = d->step;
  const int B = s0.B, S = s0.S, A = s0.A, T = d->T;
  if (T < 1 || T > 200 || B < 0 || (long long)T * B > 0x7fffffffLL) return fail(MOBODY_ERR_ARG, "mobody_rollout: bad T / B");
  if (B == 0) return MOBODY_OK;
  if (!s0.policy) return fail(MOBODY_ERR_ARG, "mobody_rollout: the step template needs a policy (actions come from pi(s))");
  if (s0.obs_ld && s0.obs_ld != S) return fail(MOBODY_ERR_ARG, "mobody_rollout: start states must be dense [B,S]");
  if (!s0.obs || !d->obss || !d->acts || !d->nexts || !d->rews || !d->pens || !d->terms || !d->row_ids || !d->counts || !d->pos ||
      !d->scratch || !d->stats || !d->ticket || !d->packed)
    return fail(MOBODY_ERR_ARG, "mobody_rollout: null workspace pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (s0.obs != d->obss &&
      cudaMemcpyAsync(d->obss, s0.obs, (size_t)B * S * sizeof(float), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
    return fail(MOBODY_ERR_CUDA, "mobody_rollout: copy of the start states failed");
  mb_rollout_init_launch(d->row_ids, s0.row0, B, T, d->pens, d->terms, d->counts, st);
  for (int t = 0; t < T; ++t) {
    mobody_step_desc s = s0;
    const size_t o = (size_t)t * B;
    s.obs = d->obss + o * S; s.obs_ld = 0; s.act_ld = 0; s.act = nullptr; s.act_out = d->acts + o * A; s.next_obs = d->nexts + o * S;
    s.reward = d->rews + o; s.penalty = d->pens + o; s.terminal = d->terms + o;
    s.row_ids = d->row_ids + o; s.n_rows_dev = d->counts + t; s.step = s0.step + (unsigned)t;
    s.eps = d->eps_all ? d->eps_all + (size_t)t * MOBODY_E * B * S : nullptr;
    s.idx = d->idx_all ? d->idx_all + o : nullptr;
    if (int rc = mobody_step(&s, stream)) return rc;
    if (t + 1 < T) {   // nonterm_mask compaction (mobody.py:635-639): stable order, counts stay on the device
      mb_compact_launch(MOBODY_KEEP_U8_ZERO, s.terminal, nullptr, 0.f, B, d->counts + t, d->scratch, d->pos, d->counts + t + 1, st);
      mb_rollout_advance_launch(s.next_obs, s.row_ids, S, d->pos, d->counts + t + 1, B, d->obss + (o + B) * S, d->row_ids + o + B, st);
    }
  }
  // concat over steps + penalty filter (mobody.py:641-653): one stable compaction over the T*B slots
  if (d->filter_bad_rollout)
    mb_compact_launch(MOBODY_KEEP_F32_LE, nullptr, d->pens, d->env_filter, (long long)T * B, nullptr, d->scratch, d->pos, d->counts + T + 1, st);
  else
    mb_compact_launch(MOBODY_KEEP_U8_VALID, d->terms, nullptr, 0.f, (long long)T * B, nullptr, d->scratch, d->pos, d->counts + T + 1, st);
  mb_rollout_pack_launch(d->obss, d->acts, d->nexts, d->rews, d->terms, d->pens, S, A, d->pos, d->counts + T + 1, (long long)T * B,
                         d->packed, st);
  mb_rollout_stats_launch(d->rews, d->terms, (long long)T * B, d->stats + 2, d->ticket, d->stats, st);
  return check_launch("mobody_rollout");
}

// mobody_model_eval workspace: start-state ping-pong [2][B,S] | next_obs [B,S] | act [B,A] | mean [E,B,S] | reward [B] |
// penalty [B] | row ids [2][B] | compaction positions [B] | compaction scratch | terminal [B]; each region 256-byte aligned.
struct EvalWs {
  float *obs[2], *next, *act, *mean, *rew, *pen;
  long long* ids[2];
  int *pos, *scratch;
  unsigned char* term;
  long long bytes;
};
static EvalWs eval_ws_layout(void* base, int B, int S, int A) {
  EvalWs w;
  uintptr_t p = (uintptr_t)base;
  auto take = [&](size_t bytes) { void* r = (void*)p; p += (bytes + 255) & ~(size_t)255; return r; };
  const size_t b = (size_t)B;
  for (int k = 0; k < 2; ++k) w.obs[k] = (float*)take(b * S * sizeof(float));
  w.next = (float*)take(b * S * sizeof(float));
  w.act = (float*)take(b * A * sizeof(float));
  w.mean = (float*)take((size_t)MOBODY_E * b * S * sizeof(float));
  w.rew = (float*)take(b * sizeof(float));
  w.pen = (float*)take(b * sizeof(float));
  for (int k = 0; k < 2; ++k) w.ids[k] = (long long*)take(b * sizeof(long long));
  w.pos = (int*)take(b * sizeof(int));
  w.scratch = (int*)take((size_t)mobody_compact_scratch_ints(B) * sizeof(int));
  w.term = (unsigned char*)take(b);
  w.bytes = (long long)(p - (uintptr_t)base);
  return w;
}

long long mobody_model_eval_workspace_bytes(int B, int S, int A) {
  if (B < 1 || S < 1 || A < 1) return 0;
  return eval_ws_layout(nullptr, B, S, A).bytes;
}

int mobody_model_eval(const mobody_model_eval_desc* d, void* stream) {
  if (!d) return fail(MOBODY_ERR_ARG, "mobody_model_eval: null descriptor");
  const mobody_step_desc& s0 = d->step;
  const int B = s0.B, S = s0.S, A = s0.A, H = d->H;
  if (H < 1 || H > 100000) return fail(MOBODY_ERR_ARG, "mobody_model_eval: bad H (1 <= H <= 100000)");
  if ((unsigned long long)s0.step + (unsigned long long)H > 0x100000000ULL)
    return fail(MOBODY_ERR_ARG, "mobody_model_eval: step + H overflows the 32-bit Philox step word");
  if (B < 0) return fail(MOBODY_ERR_ARG, "mobody_model_eval: bad B");
  if (s0.eps || s0.idx) return fail(MOBODY_ERR_ARG, "mobody_model_eval: Philox draws only (eps and idx must be NULL)");
  if (!s0.policy) return fail(MOBODY_ERR_ARG, "mobody_model_eval: the step template needs a policy (actions come from pi(s))");
  if (s0.obs_ld && s0.obs_ld != S) return fail(MOBODY_ERR_ARG, "mobody_model_eval: start states must be dense [B,S]");
  if (!d->ret || !d->ret_disc || !d->length || !d->counts) return fail(MOBODY_ERR_ARG, "mobody_model_eval: null output pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (B == 0) {
    if (cudaMemsetAsync(d->counts, 0, (size_t)(H + 1) * sizeof(int), st) != cudaSuccess)
      return fail(MOBODY_ERR_CUDA, "mobody_model_eval: clearing counts failed");
    return MOBODY_OK;
  }
  if (!s0.obs) return fail(MOBODY_ERR_ARG, "mobody_model_eval: null start states");
  const long long need = mobody_model_eval_workspace_bytes(B, S, A);
  if (need <= 0) return fail(MOBODY_ERR_ARG, "mobody_model_eval: bad S / A");
  if (!d->workspace || d->workspace_bytes < need)
    return fail(MOBODY_ERR_ARG, "mobody_model_eval: workspace missing or smaller than mobody_model_eval_workspace_bytes(B, S, A)");
  const EvalWs w = eval_ws_layout(d->workspace, B, S, A);
  double disc = 1.0;
  for (int t = 0; t < H; ++t) {
    const int cur = t & 1, nxt = cur ^ 1;
    mobody_step_desc s = s0;
    // step 0 reads the caller's start states with the default keying row0 + i (what the ids of step 0 hold), so it is
    // enqueued first: mobody_step validates the template (shapes the precision takes, parameters) before anything runs
    s.obs = t == 0 ? s0.obs : w.obs[cur]; s.obs_ld = 0; s.act = nullptr; s.act_ld = 0; s.act_out = w.act;
    s.row_ids = t == 0 ? nullptr : w.ids[cur]; s.n_rows_dev = t == 0 ? nullptr : d->counts + t;
    s.next_obs = w.next; s.reward = w.rew; s.raw_reward = nullptr; s.penalty = w.pen; s.terminal = w.term; s.mean = w.mean;
    s.step = s0.step + (unsigned)t;
    if (int rc = mobody_step(&s, stream)) return rc;
    if (t == 0) mb_model_eval_init_launch(w.ids[0], s0.row0, B, d->ret, d->ret_disc, d->length, d->counts, st);
    mb_model_eval_accumulate_launch(w.rew, w.ids[cur], s0.row0, d->counts + t, B, t, disc, d->ret, d->ret_disc, d->length, st);
    mb_compact_launch(MOBODY_KEEP_U8_ZERO, w.term, nullptr, 0.f, B, d->counts + t, w.scratch, w.pos, d->counts + t + 1, st);
    if (t + 1 < H)
      mb_rollout_advance_launch(w.next, w.ids[cur], S, w.pos, d->counts + t + 1, B, w.obs[nxt], w.ids[nxt], st);
    disc *= d->gamma;
  }
  return check_launch("mobody_model_eval");
}

int mobody_peer_push(const mobody_peer_desc* p, const int* kept_dev, const double* stats_dev, void* stream) {
  if (const char* e = mb_peer_push_launch(p, kept_dev, stats_dev, (cudaStream_t)stream)) return fail(MOBODY_ERR_ARG, e);
  return check_launch("mobody_peer_push");
}
long long mobody_peer_slot_floats(long long cap_rows, int W) { return (cap_rows < 1 || W < 5) ? 0 : mb_peer_slot_floats(cap_rows, W); }
long long mobody_peer_buffer_bytes(int world, long long cap_rows, int W) {
  return (world < 1 || world > MOBODY_MAX_PEERS || cap_rows < 1 || W < 5) ? 0 : mb_peer_buffer_bytes(world, cap_rows, W);
}
int mobody_peer_header(const mobody_peer_desc* p, const int* kept_dev, const double* stats_dev, void* stream) {
  const char* err = mb_peer_header_launch(p, kept_dev, stats_dev, (cudaStream_t)stream);
  if (err) return fail(MOBODY_ERR_ARG, err);
  return check_launch("mobody_peer_header");
}
int mobody_peer_slot(const mobody_peer_desc* p, int r, float** rows, int** header) {
  if (const char* e = mb_peer_slot(p, r, rows, header)) return fail(MOBODY_ERR_ARG, e);
  return MOBODY_OK;
}
int mobody_peer_ack(const mobody_peer_desc* p, unsigned int consumed_epoch, void* stream) {
  if (const char* e = mb_peer_ack_launch(p, consumed_epoch, (cudaStream_t)stream)) return fail(MOBODY_ERR_ARG, e);
  return check_launch("mobody_peer_ack");
}
int mobody_peer_wait(const mobody_peer_desc* p, void* stream) {
  if (const char* e = mb_peer_wait_launch(p, (cudaStream_t)stream)) return fail(MOBODY_ERR_ARG, e);
  return check_launch("mobody_peer_wait");
}

long long mobody_train_workspace_bytes(int N, int S, int A, int nsplit) {
  if (N < 1 || S < 1 || A < 1 || nsplit < 1) return 0;
  return mb_train_workspace_bytes(N, S, A, nsplit);
}

static int fail_in(const char* fn, const char* msg) {
  snprintf(g_err, sizeof(g_err), "%s: %s", fn, msg);
  return MOBODY_ERR_ARG;
}
static bool mlp_state_null(const mobody_mlp_state& s) {
  for (int j = 0; j < 3; ++j)
    if (!s.w[j] || !s.b[j]) return true;
  return false;
}

// shared by mobody_train_step (default flags) and mobody_train_step_ex; `fn` names the entry point in messages
static int train_step(const mobody_train_ex_desc& x, void* stream, const char* fn) {
  const mobody_train_desc* d = &x.base;
  if (!d->rows) return fail_in(fn, "null descriptor / rows");
  if (d->row_width != mobody_row_width(d->S, d->A)) return fail_in(fn, "row_width does not match (S, A)");
  const mobody_mlp_state* all[11] = {&d->policy, &d->q1, &d->q2, &d->q1_target, &d->q2_target, &d->policy_m, &d->policy_v,
                                     &d->q1_m, &d->q1_v, &d->q2_m, &d->q2_v};
  for (int i = 0; i < 11; ++i)
    if (mlp_state_null(*all[i])) return fail_in(fn, "null parameter / moment pointer");
  if (d->t_q < 1 || d->t_pi < 1) return fail_in(fn, "optimiser step counts are 1-based");
  const char* err = mb_train_step_launch(x, (cudaStream_t)stream);
  if (err) return fail(MOBODY_ERR_UNSUPPORTED, err);
  return check_launch(fn);
}

int mobody_train_step(const mobody_train_desc* d, void* stream) {
  if (!d) return fail(MOBODY_ERR_ARG, "mobody_train_step: null descriptor / rows");
  mobody_train_ex_desc x{};
  x.base = *d; x.advantage = 0; x.scale_q = 1; x.q_weighted = 1;
  return train_step(x, stream, "mobody_train_step");
}

long long mobody_train_ex_workspace_bytes(int N, int S, int A, int nsplit) {
  if (N < 1 || S < 1 || A < 1 || nsplit < 1) return 0;
  return mb_train_ex_workspace_bytes(N, S, A, nsplit);
}

int mobody_train_step_ex(const mobody_train_ex_desc* d, void* stream) {
  if (!d) return fail(MOBODY_ERR_ARG, "mobody_train_step_ex: null descriptor / rows");
  for (int f : {d->advantage, d->scale_q, d->q_weighted})
    if (f != 0 && f != 1) return fail(MOBODY_ERR_ARG, "mobody_train_step_ex: advantage / scale_q / q_weighted must be 0 or 1");
  if (d->advantage) {
    if (mlp_state_null(d->value) || mlp_state_null(d->value_m) || mlp_state_null(d->value_v))
      return fail(MOBODY_ERR_ARG, "mobody_train_step_ex: advantage=1 needs the value function and its Adam moments");
    if (d->t_v < 1) return fail(MOBODY_ERR_ARG, "mobody_train_step_ex: the value optimiser step count is 1-based");
  }
  return train_step(*d, stream, "mobody_train_step_ex");
}

long long mobody_dynfit_workspace_bytes(int B, int S, int A, int nsplit) {
  if (B < 1 || S < 1 || A < 1 || nsplit < 1) return 0;
  return mb_dynfit_workspace_bytes(B, S, A, nsplit);
}

int mobody_dynfit_step(const mobody_dynfit_desc* d, void* stream) {
  if (!d || !d->obs || !d->act || !d->next_obs || !d->reward) return fail(MOBODY_ERR_ARG, "mobody_dynfit_step: null descriptor / batch pointer");
  if (d->B < 1 || d->S < 1 || d->A < 1) return fail(MOBODY_ERR_ARG, "mobody_dynfit_step: B >= 1, S >= 1, A >= 1");
  if ((d->eps_latent == nullptr) != (d->eps_next == nullptr)) return fail(MOBODY_ERR_ARG, "mobody_dynfit_step: inject both noise tensors or neither");
  for (int i = 0; i < MOBODY_N_DYN_LAYERS; ++i)
    if (!d->params.w[i] || !d->params.b[i] || !d->adam_m.w[i] || !d->adam_m.b[i] || !d->adam_v.w[i] || !d->adam_v.b[i])
      return fail(MOBODY_ERR_ARG, "mobody_dynfit_step: null parameter / moment pointer");
  if (d->t_shared < 1 || d->t_action < 1) return fail(MOBODY_ERR_ARG, "mobody_dynfit_step: optimiser step counts are 1-based");
  if (!d->workspace || !d->scalars_out) return fail(MOBODY_ERR_ARG, "mobody_dynfit_step: null workspace / scalars_out");
  const char* err = mb_dynfit_step_launch(*d, (cudaStream_t)stream);
  if (err) return fail(MOBODY_ERR_UNSUPPORTED, err);
  return check_launch("mobody_dynfit_step");
}

long long mobody_classifier_workspace_bytes(int N, int S, int A, int nsplit) {
  if (N < 1 || S < 1 || A < 1 || nsplit < 1) return 0;
  return mb_classifier_workspace_bytes(N, S, A, nsplit);
}

int mobody_classifier_step(const mobody_classifier_desc* d, void* stream) {
  if (!d || !d->rows || !d->label) return fail(MOBODY_ERR_ARG, "mobody_classifier_step: null descriptor / rows / label");
  if (d->row_width != mobody_row_width(d->S, d->A)) return fail(MOBODY_ERR_ARG, "mobody_classifier_step: row_width does not match (S, A)");
  const mobody_mlp_state* all[6] = {&d->sas, &d->sa, &d->sas_m, &d->sas_v, &d->sa_m, &d->sa_v};
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j < 3; ++j)
      if (!all[i]->w[j] || !all[i]->b[j]) return fail(MOBODY_ERR_ARG, "mobody_classifier_step: null parameter / moment pointer");
  if (d->t < 1) return fail(MOBODY_ERR_ARG, "mobody_classifier_step: optimiser step count is 1-based");
  const char* err = mb_classifier_step_launch(*d, (cudaStream_t)stream);
  if (err) return fail(MOBODY_ERR_UNSUPPORTED, err);
  return check_launch("mobody_classifier_step");
}

int mobody_dara_relabel(float* rows, long long n, int S, int A, int row_width, const mobody_mlp_params* sas,
                        const mobody_mlp_params* sa, float penalty_coef, float* penalty_out, void* stream) {
  if (n < 0 || !sas || !sa || (n > 0 && !rows)) return fail(MOBODY_ERR_ARG, "mobody_dara_relabel: bad arguments");
  if (row_width != mobody_row_width(S, A)) return fail(MOBODY_ERR_ARG, "mobody_dara_relabel: row_width does not match (S, A)");
  MlpPtrs p0, p1; memcpy(&p0, sas, sizeof(p0)); memcpy(&p1, sa, sizeof(p1));
  const char* err = mb_dara_relabel_launch(rows, n, S, A, row_width, p0, p1, penalty_coef, penalty_out, (cudaStream_t)stream);
  if (err) return fail(MOBODY_ERR_UNSUPPORTED, err);
  return check_launch("mobody_dara_relabel");
}

static int nsplit_of(int precision) { return (precision == MOBODY_PREC_BF16X2 || precision == MOBODY_PREC_BF16X2_WIDE || precision == MOBODY_PREC_BF16X2_T64) ? 2 : (precision == MOBODY_PREC_BF16 || precision == MOBODY_PREC_FP16 || precision == MOBODY_PREC_FP16_T64) ? 1 : 0; }
// the single fp16 plane of the fp16 modes (one image format for MOBODY_PREC_FP16 and MOBODY_PREC_FP16_T64)
static int is_fp16(int precision) { return precision == MOBODY_PREC_FP16 || precision == MOBODY_PREC_FP16_T64; }

long long mobody_dyn_pack_bytes(int S, int A, int precision) {
  int ns = nsplit_of(precision);
  if (!ns || S < 2 || A < 1) return 0;
  return (long long)tc_dyn_layout(S, A, ns).total_bytes;
}

int mobody_dyn_pack(const mobody_dyn_params* dyn, int S, int A, int precision, void* blob, unsigned long long* state, void* stream) {
  int ns = nsplit_of(precision);
  if (!ns || !dyn || !blob || S < 2 || A < 1) return fail(MOBODY_ERR_ARG, "mobody_dyn_pack: bad arguments");
  DynPtrs dp; memcpy(&dp, dyn, sizeof(dp));
  for (int i = 0; i < L_COUNT; ++i)
    if (!dp.w[i] || !dp.b[i]) return fail(MOBODY_ERR_ARG, "mobody_dyn_pack: null parameter pointer");
  const char* err = mb_tc_dyn_pack(dp, S, A, ns, is_fp16(precision), (unsigned char*)blob, state, (cudaStream_t)stream);
  if (err) return fail(MOBODY_ERR_ARG, err);
  return check_launch("mobody_dyn_pack");
}

long long mobody_mlp_pack_bytes(int din, int dout, int precision) {
  int ns = nsplit_of(precision);
  if (!ns || din < 1 || dout < 1) return 0;
  return (long long)tc_mlp_layout(din, dout, ns).total_bytes;
}

int mobody_mlp_pack(const mobody_mlp_params* mlp, int din, int dout, int precision, void* blob, unsigned long long* state, void* stream) {
  int ns = nsplit_of(precision);
  if (!ns || !mlp || !blob || din < 1 || dout < 1) return fail(MOBODY_ERR_ARG, "mobody_mlp_pack: bad arguments");
  MlpPtrs mp; memcpy(&mp, mlp, sizeof(mp));
  const char* err = mb_tc_mlp_pack(mp, din, dout, ns, is_fp16(precision), (unsigned char*)blob, state, (cudaStream_t)stream);
  if (err) return fail(MOBODY_ERR_ARG, err);
  return check_launch("mobody_mlp_pack");
}

int mobody_selftest_umma(const float* A, const float* B, int K, int N, int nsplit, float* D, void* stream) {
  if (!A || !B || !D) return fail(MOBODY_ERR_ARG, "mobody_selftest_umma: null pointer");
  const char* err = mb_umma_selftest_launch(A, B, K, N, nsplit, D, (cudaStream_t)stream);
  if (err) return fail(MOBODY_ERR_ARG, err);
  return check_launch("mobody_selftest_umma");
}

int mobody_selftest_gemm(const float* A, const float* B, int M, int N, int K, int a_src, int b_src, int lda, int ldb, float* C, void* stream) {
  if (!A || !B || !C) return fail(MOBODY_ERR_ARG, "mobody_selftest_gemm: null pointer");
  const char* err = mb_gemm_selftest_launch(A, B, M, N, K, a_src, b_src, lda, ldb, C, (cudaStream_t)stream);
  if (err) return fail(MOBODY_ERR_ARG, err);
  return check_launch("mobody_selftest_gemm");
}

/* debug hook (not in the public header): device int64[80*8] receiving per-layer clock64 stamps of CTA 0 */
int mobody_debug_set_trace(void* buf) { mb_tc_set_trace((long long*)buf); return MOBODY_OK; }

}  // extern "C"
