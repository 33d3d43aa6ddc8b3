/* mobody_b200 — C ABI of the B200-native MOBODY rollout / Q-weighted-BC hot path.
 *
 * Plain C: pointers and sizes only, no torch types.  Every pointer named "device" is a CUDA device
 * pointer owned by the caller (PyTorch) and valid for the duration of the call; the library never
 * allocates or frees.  All work is enqueued on `stream` (a cudaStream_t passed as void*) and is
 * asynchronous with respect to the host.  Every entry point returns 0 on success and a negative
 * code on failure; mobody_last_error() then holds a message (thread-local).  No exceptions cross
 * the boundary.
 *
 * The reference (guoyihonggyh/MOBODY...) has no FFI: its hot path is Python calling torch eager
 * ops.  Each export below names the reference Python interface it replaces; the Python-side
 * binding (ctypes) lives in mobody_b200/_ffi.py and INTEGRATION.md shows how train_mobody.py
 * binds to it.
 */
#ifndef MOBODY_B200_H
#define MOBODY_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define MOBODY_ABI_VERSION 2
#define MOBODY_TC_TRAIN_MIN_ROWS 1280  /* mobody_train_step runs on tcgen05 GEMM tiles from this many batch rows, below on mma.sync */
#define MOBODY_E 7            /* ensemble members      (train_mobody.py:795) */
#define MOBODY_H 256          /* hidden width          (train_mobody.py:794) */
#define MOBODY_N_DYN_LAYERS 13

/* error codes */
#define MOBODY_OK 0
#define MOBODY_ERR_ARG (-1)
#define MOBODY_ERR_UNSUPPORTED (-2)
#define MOBODY_ERR_CUDA (-3)

/* termination kinds (algo/mb_utils/terminal_funs.py:10-121; dispatcher :123-149 is host side) */
#define MOBODY_TERM_NEVER 0
#define MOBODY_TERM_HALFCHEETAH 1
#define MOBODY_TERM_HOPPER 2
#define MOBODY_TERM_WALKER2D 3
#define MOBODY_TERM_ANT 4
#define MOBODY_TERM_HUMANOID 5
#define MOBODY_TERM_PEN 6

/* precision modes of the fused step */
#define MOBODY_PREC_FP32 0    /* CUDA-core fp32 FMA; bit-faithful op order per row                  */
#define MOBODY_PREC_BF16X2 1  /* tcgen05 bf16 hi+lo split (3 MMAs), ~1e-5 rel: inside the 1e-4 bound */
#define MOBODY_PREC_BF16 2    /* tcgen05 single-pass bf16: DIAGNOSTIC ONLY, outside the stated bounds (measured 1.6e-2); the Python mirror does not offer it */
                              /* takes S <= 63 where two row tiles do not fit (2S+A > 112): the one-tile fallback has no
                                 statistics scratch at S = 64 and reports MOBODY_ERR_UNSUPPORTED */
#define MOBODY_PREC_FP16 3    /* tcgen05 single-pass fp16, two tiles per SM, packed-half epilogue; measured <= 4.6e-3, inside the stated looser bound 5e-3; |activations| < 6e4 */
#define MOBODY_PREC_BF16X2_WIDE 4  /* bf16x2's arithmetic on 64-row tiles for wide observations: MOBODY_TC_WIDE_MIN_S <= S <= MOBODY_TC_WIDE_MAX_S,
                                      A <= MOBODY_TC_WIDE_MAX_A (Ant's 111 / 8); packed images are bf16x2's */
#define MOBODY_PREC_BF16X2_T64 5   /* bf16x2's arithmetic on the same 64-row tiles for the S <= 64 shapes bf16x2 refuses
                                      (Adroit's pen 45 / 24, door 39 / 28, relocate 39 / 30, hammer 46 / 26); packed images are bf16x2's */
#define MOBODY_PREC_FP16_T64 6     /* fp16's arithmetic (single pass, packed-half epilogue, the stated looser bound 5e-3,
                                      |activations| < 6e4) on the same 64-row tiles for the shapes fp16 refuses (Ant's 111 / 8,
                                      Adroit); packed images are fp16's */
/* Shapes of the tensor-core modes: S <= 64, A <= 16, and the [s, a, s'] operand plane of the reward model must fit in
   shared memory next to the other planes: 2S+A <= 96 (bf16x2: hi and lo planes, one row tile per CTA) or 112 (fp16: two
   row tiles per CTA).  mobody_step rejects other shapes with MOBODY_ERR_ARG; the fp32 mode takes S <= 128, A <= 32. */
#define MOBODY_TC_MAX_S 64
#define MOBODY_TC_MAX_A 16
#define MOBODY_TC_BF16X2_MAX_SAS 96
#define MOBODY_TC_FP16_MAX_SAS 112
/* Shapes of MOBODY_PREC_BF16X2_WIDE: every shape the fp32 mode takes above MOBODY_TC_MAX_S. */
#define MOBODY_TC_WIDE_MIN_S 65
#define MOBODY_TC_WIDE_MAX_S 128
#define MOBODY_TC_WIDE_MAX_A 32
/* Shapes of MOBODY_PREC_BF16X2_T64: 2 <= S <= MOBODY_TC_T64_MAX_S, 1 <= A <= MOBODY_TC_T64_MAX_A, and A > MOBODY_TC_MAX_A or
   2S+A > MOBODY_TC_BF16X2_MAX_SAS -- exactly the shapes with S <= 64 that the fp32 mode takes and bf16x2 refuses.  So bf16x2,
   bf16x2_t64 and bf16x2_wide split the fp32 mode's shapes with no overlap: at most one of them takes a given (S, A). */
#define MOBODY_TC_T64_MAX_S 64
#define MOBODY_TC_T64_MAX_A 32
/* Shapes of MOBODY_PREC_FP16_T64: 2 <= S <= MOBODY_TC_WIDE_MAX_S, 1 <= A <= MOBODY_TC_WIDE_MAX_A, and not (S <= MOBODY_TC_MAX_S,
   A <= MOBODY_TC_MAX_A and 2S+A <= MOBODY_TC_FP16_MAX_SAS) -- exactly the shapes the fp32 mode takes and fp16 refuses.  So fp16
   and fp16_t64 split the fp32 mode's shapes with no overlap. */

/* compaction predicates */
#define MOBODY_KEEP_U8_ZERO 0 /* keep rows with flag == 0      (non-terminal rows, mobody.py:635)   */
#define MOBODY_KEEP_F32_LE 1  /* keep rows with value <= thr   (rollout filter, mobody.py:649)      */
#define MOBODY_KEEP_F32_LT 2  /* keep rows with value <  thr   (dataset-step filter, mobody.py:468) */
#define MOBODY_KEEP_U8_VALID 3 /* keep rows with flag != 0xFF  (rows a rollout step actually wrote) */

/* Live parameters of MOBODYModule (algo/dynamics/mobody_module.py:97-184), device fp32:
 * w[i] is weight [E,in,out], b[i] is bias [E,1,out], in the order
 * zs1 zs2 zs3 za_src1 za_src2 za_trg1 za_trg2 transition1 transition2 transition3
 * reward_model1 reward_model2 reward_model3. */
typedef struct mobody_dyn_params {
  const float* w[MOBODY_N_DYN_LAYERS];
  const float* b[MOBODY_N_DYN_LAYERS];
} mobody_dyn_params;

/* Live parameters of an MLPNetwork (algo/offline_offline/mobody.py:35-48): nn.Linear layout,
 * w[i] [out,in], b[i] [out], hidden 256. */
typedef struct mobody_mlp_params {
  const float* w[3];
  const float* b[3];
} mobody_mlp_params;

/* One imagined transition for a batch of rows.
 * Replaces MOBODYEnsembleDynamics.step (algo/dynamics/mobody_dynamics.py:193-265) and, when
 * `policy` is non-NULL, the Policy forward that precedes it in MOBODY.rollout
 * (algo/offline_offline/mobody.py:612).  Math: SURVEY.md Appendix A.1. */
typedef struct mobody_step_desc {
  int precision;             /* MOBODY_PREC_* */
  int B, S, A;               /* B = row capacity (stride of eps / mean); obs is [B,S]             */
  int obs_ld, act_ld;        /* row strides of obs / act in floats; 0 = dense (S / A).  Lets a step read the
                                state / action columns of packed replay-buffer rows in place (mobody.py:428-434) */
  const int* n_rows_dev;     /* NULL, or device int: live row count (<= B)                        */
  const long long* row_ids;  /* NULL, or device int64[B]: global row id per row (Philox counter)  */
  const float* obs;          /* device [B,S]                                                      */
  const float* act;          /* device [B,A], or NULL when `policy` computes it                   */
  const mobody_mlp_params* policy; /* NULL or host struct of device pointers                      */
  float max_action;
  const mobody_dyn_params* dyn;    /* host struct of device pointers (fp32 path reads them live)  */
  const void* dyn_pack;      /* device blob from mobody_dyn_pack (tensor-core precisions), or NULL */
  const void* policy_pack;   /* device blob from mobody_mlp_pack (tensor-core precisions), or NULL */
  int use_trg, use_penalty;  /* step(..., use_penalty, use_trg)                                   */
  float penalty_coef;        /* dynamics._penalty_coef                                            */
  int term_kind;             /* MOBODY_TERM_*                                                     */
  const float* eps;          /* NULL -> Philox; else device [E,B,S] N(0,1) (parity mode)          */
  const int64_t* idx;        /* NULL -> Philox pick among elites; else device int64[B] member ids */
  const int64_t* elites;     /* device int64[n_elites]  (model.elites)                            */
  int n_elites;
  unsigned long long seed;   /* Philox key                                                        */
  unsigned int step;         /* Philox counter word: rollout step                                 */
  unsigned long long row0;   /* global row id of obs[0] when row_ids is NULL                      */
  float* act_out;            /* NULL or device [B,A]                                              */
  float* next_obs;           /* device [B,S]                                                      */
  float* reward;             /* device [B]                                                        */
  float* raw_reward;         /* NULL or device [B]   (info['raw_reward'])                         */
  float* penalty;            /* device [B]           (info['penalty'])                            */
  unsigned char* terminal;   /* device [B], 0/1      (terminal_fn(next_obs))                      */
  float* mean;               /* device [E,B,S]       (info['samples']); always written            */
} mobody_step_desc;

int mobody_abi_version(void);
const char* mobody_last_error(void);

int mobody_step(const mobody_step_desc* d, void* stream);

/* Policy.forward / select_action (mobody.py:60-72, 138-144): act_out[B,A] = tanh(MLP(obs))*max_action */
int mobody_policy_forward(const float* obs, int B, int S, int A, const mobody_mlp_params* policy,
                          float max_action, float* act_out, void* stream);

/* terminal_fn(obs, act, next_obs) (terminal_funs.py:10-121) on device rows: out[n] in {0,1} */
int mobody_termination(const float* next_obs, long long n, int S, int term_kind, unsigned char* out, void* stream);

/* ---- replay buffer (algo/utils.py:13-193) on packed rows of row_width(S,A) floats:
 *      [state(S) | action(A) | next_state(S) | reward | not_done | pad to a multiple of 4] ---- */
int mobody_row_width(int S, int A);
/* ReplayBuffer.sample (utils.py:127-148) with indices given: out[i,:] = rows[idx[i],:] */
int mobody_gather_rows(const float* rows, const int64_t* idx, long long n, int row_width, float* out, void* stream);
/* np.random.randint(0, size, n) replacement (utils.py:128): Philox4x32-10, key (seed,'indx'), counter (i, draw) */
int mobody_philox_indices(int64_t* idx, long long n, unsigned long long seed, unsigned int draw,
                          unsigned int size, void* stream);
/* Fused draw + gather of up to 4 buffer samples in one launch (the three ReplayBuffer.sample calls of one
 * MOBODY.train step, mobody.py:399-400, 524): out[i,:] = rows[philox_index(i, draw, seed) , :], i < n. */
typedef struct mobody_sample_job {
  const float* rows; long long n; unsigned int size; unsigned int draw; unsigned long long seed; float* out;
} mobody_sample_job;
int mobody_sample_rows(const mobody_sample_job* jobs, int njobs, int row_width, void* stream);
/* convert_D4RL / add_batch packing (utils.py:43-92, 173-193): d is `terminals` when done_is_terminal (stores 1-d) */
int mobody_pack_rows(const float* s, const float* a, const float* ns, const float* r, const float* d,
                     long long n, int S, int A, int done_is_terminal, float* out_rows, void* stream);
/* ReplayBuffer.add_batch ring insert (utils.py:68-92): src row i -> dst row (ptr+i) % cap; n_dev optional device count */
int mobody_ring_insert(const float* src_rows, long long n_cap, const int* n_dev, int row_width, long long ptr,
                       long long cap, float* dst_rows, void* stream);

/* add_batch of a rollout result without an intermediate copy: packed rows [obs(S) | act(A) | next_obs(S) | reward |
 * terminal | penalty] (mobody_rollout's output layout) -> buffer rows [.. | reward | 1 - terminal | 0-pad] at ring
 * positions (ptr + i) % cap (utils.py:68-92 stores not_done = 1 - terminals). */
int mobody_ring_insert_transitions(const float* packed, long long n_cap, const int* n_dev, int S, int A, long long ptr,
                                   long long cap, float* dst_rows, void* stream);

/* `par` reward penalty of the steady-state train step (algo/offline_offline/mobody.py:428-434), in place on the
 * first n packed batch rows: rows[i].reward -= coef * mean_j (rows[i].next_state[j] - pred_next[i,j])^2, where
 * pred_next [n,S] is the next_obs of a dynamics step on the rows' (state, action).  mean_out (nullable device
 * float) receives the batch mean of the penalty ('train/reward_penalty_par', :433); fixed summation order. */
int mobody_par_penalty(float* rows, int n, int S, int A, int row_width, const float* pred_next, float coef,
                       float* mean_out, void* stream);

/* ---- stable stream compaction (mobody.py:635-639, 648-651, 468) ----
 * pos[0..count) = ascending indices i < n with keep(i); count_out is a device int.
 * scratch: device int[mobody_compact_scratch_ints(n_cap)]. */
long long mobody_compact_scratch_ints(long long n_cap);
int mobody_compact(int keep_kind, const unsigned char* flags, const float* vals, float thr, long long n_cap,
                   const int* n_dev, int* scratch, int* pos, int* count_out, void* stream);
/* dst[j,0:w] = src[pos[j],0:w] for j < count (count = *m_dev if given else m_cap) */
int mobody_gather_pos(const float* src, int w, int src_ld, const int* pos, const int* m_dev, long long m_cap,
                      float* dst, int dst_ld, void* stream);
int mobody_gather_pos_i64(const long long* src, const int* pos, const int* m_dev, long long m_cap,
                          long long* dst, void* stream);

/* ---- whole model rollout: MOBODY.rollout (algo/offline_offline/mobody.py:596-657) as ONE host call ----
 * T fused steps (policy forward + dynamics step) with device-side compaction of the non-terminal rows between
 * steps (:635-639), concatenation over steps and the penalty filter `penalty <= env_filter` (:641-653) — no host
 * round trip inside the rollout.  `step` is the template of every step: its obs is the start states [B,S], its
 * policy must be set, and its per-step fields (obs/act_out/next_obs/reward/penalty/terminal/row_ids/n_rows_dev/
 * step/eps/idx) are overridden from the workspace below.  Everything is caller-allocated device memory.
 * Outputs: packed[j,:] = [obs(S) | act(A) | next_obs(S) | reward | terminal(0/1) | penalty] for the kept
 * transitions j < counts[T+1] in the reference's order (step-major, rows ascending); counts[t] = live rows entering
 * step t (t < T); stats[0] = sum of rewards over all produced transitions, stats[1] = their number
 * (info['reward_mean'] = stats[0] / stats[1], info['num_transitions'] = stats[1]). */
typedef struct mobody_rollout_desc {
  mobody_step_desc step;
  int T;                      /* rollout_length (1 <= T <= 200)                                        */
  int filter_bad_rollout;     /* config['filter_bad_rollout']                                          */
  float env_filter;           /* config['env_filter']                                                  */
  const float* eps_all;       /* NULL -> Philox; else device [T,E,B,S]                                 */
  const int64_t* idx_all;     /* NULL -> Philox; else device int64 [T,B]                               */
  float* obss;                /* device [T,B,S]; obss[0] is filled from step.obs unless they alias     */
  float* acts;                /* device [T,B,A]                                                        */
  float* nexts;               /* device [T,B,S]                                                        */
  float* rews;                /* device [T,B]                                                          */
  float* pens;                /* device [T,B]                                                          */
  unsigned char* terms;       /* device [T,B]   0/1, 0xFF = slot never produced                        */
  long long* row_ids;         /* device int64 [T,B] global row ids (Philox counters)                   */
  int* counts;                /* device int [T+2]                                                      */
  int* pos;                   /* device int [T*B]                                                      */
  int* scratch;               /* device int [mobody_compact_scratch_ints(T*B)]                         */
  double* stats;              /* device double [mobody_rollout_stats_doubles()] (first 2 are the result) ... */
  unsigned int* ticket;       /* ... and one device unsigned, zero-initialised once by the caller      */
  float* packed;              /* device [T*B, 2S+A+3]                                                  */
} mobody_rollout_desc;
/* ---- multi-GPU assembly of the synthetic transitions (SURVEY.md section 8e) over peer memory ----
 * Every rank owns a receive buffer that its peers have mapped (symmetric memory / CUDA IPC; the host side only exchanges
 * handles): two `halves` (parity of the exchange number) of `world` slots, each slot = [cap_rows][W] packed transitions
 * followed by one header row, and a flag block behind them.  A rank's rollout packs into slot `rank` of its OWN buffer
 * (mobody_rollout with desc.packed = that slot); mobody_peer_push then streams exactly the kept rows into the same slot of
 * every peer's buffer with 128-bit NVLink stores -- or with ONE NVSwitch-replicated multicast store per 16 bytes when a
 * multicast mapping is given -- publishes the header {int32 kept, int64 produced, double reward sum} and raises
 * flag[rank] = epoch at every rank (system-scope release).  It replaces the NCCL all-gather of padded slabs: no
 * collective kernel, no padding on the wire, a few CTAs on a side stream beside the next rollout.  A rank may overwrite
 * half (epoch & 1) at a peer only after that peer acknowledged epoch - 2 (mobody_peer_ack, stream-ordered after the
 * peer's consumers); the push kernel waits for it.  mobody_peer_wait makes `stream` wait (device-side spin, no host
 * involvement) until every rank's rows of `epoch` have landed. */
#define MOBODY_MAX_PEERS 8
typedef struct mobody_peer_desc {
  int world, rank;
  void* base[MOBODY_MAX_PEERS];   /* base[r]: rank r's receive buffer as mapped in THIS process (base[rank] is local)   */
  void* multicast;                /* NULL, or the multicast mapping of the same buffers (NVLS)                          */
  long long cap_rows;             /* rows per slot (>= T*B of the largest shard)                                        */
  int W;                          /* floats per packed transition (2S+A+3)                                              */
  unsigned int epoch;             /* exchange number, 1, 2, 3, ... (monotone; same on every rank)                       */
  int ctas;                       /* CTAs of the push kernel (0 = default: 64 CTAs of 128 threads, small enough to sit beside a step tile) */
} mobody_peer_desc;
long long mobody_peer_slot_floats(long long cap_rows, int W);     /* floats per slot incl. header row, padded to 16 B   */
long long mobody_peer_buffer_bytes(int world, long long cap_rows, int W);   /* receive buffer: 2 halves + flag block    */
/* slot r of the half holding p->epoch in the LOCAL buffer: rows pointer and header pointer (host arithmetic only) */
int mobody_peer_slot(const mobody_peer_desc* p, int r, float** rows, int** header);
/* push slot `rank` (rows [0, *kept_dev)) of the local buffer to every peer; stats_dev = {reward sum, produced} doubles */
int mobody_peer_push(const mobody_peer_desc* p, const int* kept_dev, const double* stats_dev, void* stream);
/* Copy-engine variant of the push (no SM touches the payload): mobody_peer_header writes the header row of slot `rank` in the
 * LOCAL buffer; the host side then ships the whole slot (cap_rows + 1 rows) to every peer with stream-ordered device-to-device
 * copies and raises / awaits the flags with stream memory operations (cuStreamWriteValue32 / cuStreamWaitValue32 on the flag
 * block: word r = arrive[r], word 8 + r = ack[r], the block starts mobody_peer_buffer_bytes(...) - 128 bytes into a buffer). */
int mobody_peer_header(const mobody_peer_desc* p, const int* kept_dev, const double* stats_dev, void* stream);
int mobody_peer_ack(const mobody_peer_desc* p, unsigned int consumed_epoch, void* stream);
int mobody_peer_wait(const mobody_peer_desc* p, void* stream);

int mobody_rollout_stats_doubles(void);   /* size of mobody_rollout_desc.stats in doubles */
int mobody_rollout(const mobody_rollout_desc* d, void* stream);

/* ---- policy evaluation in the learned model: the episode return eval_policy reports (train_mobody.py:53-205), with the
 * dynamics model standing in for the environment, one episode per start state, as ONE host call ----
 * Step t (t < H) runs the fused step (policy forward + dynamics step) on the live rows with Philox step word
 * `step.step + t`, each row keyed on its global start id (step.row0 + its index in step.obs), exactly as mobody_rollout
 * keys them: a start state's episode does not depend on the batch it runs in.  The step reward is the step's `reward`
 * (raw reward, or reward - coef * penalty with use_penalty).  A row whose next state is terminal keeps that step's reward
 * and stops; survivors are compacted stably into the next step's input.  Memory is O(B) whatever H: nothing per step is
 * kept.  Returns accumulate in float64, one add per row and step in step order: ret += r; ret_disc += disc * r (product
 * rounded, then added), where disc starts at 1.0 and is multiplied by gamma after every step -- reproducible bit for bit
 * on a host.  Once every row has ended, the remaining steps launch kernels that exit at once.
 * `step` is the template as in mobody_rollout: obs = dense start states [B,S], policy required, eps / idx must be NULL
 * (Philox draws only); its per-step fields are overridden from the workspace. */
typedef struct mobody_model_eval_desc {
  mobody_step_desc step;
  int H;                      /* horizon, 1 .. 100000; step.step + H must not exceed 2^32                             */
  double gamma;
  void* workspace; long long workspace_bytes;   /* device, >= mobody_model_eval_workspace_bytes(B, S, A) (no H in it) */
  double* ret;                /* device [B] sum of the step rewards up to and including the terminating step (or H-1) */
  double* ret_disc;           /* device [B] sum over the same steps of gamma^t r_t                                     */
  int* length;                /* device [B] steps taken: t+1 for a row whose next state at step t is terminal, else H */
  int* counts;                /* device [H+1] live rows entering step t; counts[H] = rows still live after the last   */
} mobody_model_eval_desc;
long long mobody_model_eval_workspace_bytes(int B, int S, int A);
int mobody_model_eval(const mobody_model_eval_desc* d, void* stream);

/* ---- steady-state train step: twin-critic TD update + Polyak + Q-weighted BC actor update ----
 * Replaces MOBODY.update_q_functions / update_target / update_policy / bc_loss and the three
 * torch.optim.Adam steps inside MOBODY.train (algo/offline_offline/mobody.py:183-208, 246-276, 314-345,
 * 541-573; math in SURVEY.md Appendix A.3; defaults advantage=0, scale_Q=1, q_weighted=1).
 * `rows` is the concatenated batch [N, row_width] (src, tar, fake order; the first n_true rows are the
 * src+tar rows of the BC term).  Parameters and Adam moments are updated IN PLACE in the live
 * nn.Parameter storage.  scalars_out (device float[16]):
 *   [0] q_loss [1] mean q1 [2] policy loss [3] bc loss [4] mean q(s,pi(s)) [5] mean|q(s,pi(s))|
 *   [6] mean exp_adv [7] min exp_adv [8] max exp_adv [9] p_w [10] mean|q(s_t,a_t)| */
typedef struct mobody_mlp_state { float* w[3]; float* b[3]; } mobody_mlp_state;   /* writable twin of mobody_mlp_params */
typedef struct mobody_train_desc {
  const float* rows; int N, n_true, S, A, row_width;
  mobody_mlp_state policy, q1, q2, q1_target, q2_target;        /* parameters (updated in place)            */
  mobody_mlp_state policy_m, policy_v, q1_m, q1_v, q2_m, q2_v;  /* Adam first / second moments              */
  int t_q, t_pi;                 /* optimiser step counts AFTER this step (1-based), for bias correction    */
  float gamma, tau, critic_lr, actor_lr, weight, bc_coef, max_action;
  int nsplit;                    /* row splits of the weight-gradient GEMMs, 1..64 (any value: same update up to fp32 summation order) */
  void* workspace; long long workspace_bytes;   /* device scratch >= mobody_train_workspace_bytes(...)       */
  float* scalars_out;            /* device float[16]                                                        */
} mobody_train_desc;
long long mobody_train_workspace_bytes(int N, int S, int A, int nsplit);
int mobody_train_step(const mobody_train_desc* d, void* stream);

/* ---- the same train step with the reference's update-branch flags (mobody.py:210-310, 533-573) ----
 * advantage=1: first a value step -- adv = min(Q'1(s,a), Q'2(s,a)) - V(s) with the target critics before this step's
 *   Polyak update, v_loss = mean(|0.7 - 1[adv<0]| adv^2), Adam on `value` (lr = critic_lr, moments value_m / value_v);
 *   then the TD target r + nd * gamma * V(s') with the updated V, and BC weights exp(3 (min Q(s_t,a_t) - V(s_t))).
 * scale_q=0: p_w = 1 instead of weight / mean|q(s,pi(s))| (update_policy_1).   q_weighted=0: BC weights 1 (plain BC).
 * Flags 0/0/1/1 (advantage, scale_q, q_weighted = 0, 1, 1) are mobody_train_step, bit for bit.  The workspace must hold
 * mobody_train_ex_workspace_bytes(...).  scalars_out keeps slots [0..10]; with advantage=1 it adds [11] v_loss
 * [12] mean adv of the value step [13] mean V(s) before the step, and with any non-default flag [14] mean min Q(s,a)
 * after the critic step (all rows).  Other slots are not written. */
typedef struct mobody_train_ex_desc {
  mobody_train_desc base;
  int advantage, scale_q, q_weighted;          /* config flags, 0/1 */
  mobody_mlp_state value, value_m, value_v;    /* ValueFunc + Adam moments; required iff advantage */
  int t_v;                                     /* value optimiser step count AFTER this step (1-based) when advantage */
} mobody_train_ex_desc;
long long mobody_train_ex_workspace_bytes(int N, int S, int A, int nsplit);
int mobody_train_step_ex(const mobody_train_ex_desc* d, void* stream);

/* ---- DARA domain classifier (SURVEY.md section 8f rank 1) ----
 * mobody_classifier_step replaces the forward / double-softmax cross-entropy / backward / Adam of
 * MOBODY.update_classifier (algo/offline_offline/mobody.py:146-181) for Classifier (:11-33): `rows` [N,row_width]
 * is the concatenated (src, tar) and permuted batch, label[i] in {0,1} its domain.  noise_* inject the draws of
 * torch.randn_like (parity) or are NULL (Philox keyed on (seed, draw, row, column)); noise_std = gaussian_noise_std.
 * scalars_out: [0] loss_sa, [1] loss_sas.  Parameters and Adam moments are updated in place. */
typedef struct mobody_classifier_desc {
  const float* rows; int N, S, A, row_width;
  const int* label;                              /* device int32 [N]                                        */
  const float* noise_sas; const float* noise_sa; /* device [N,2S+A] / [N,S+A] or NULL                       */
  float noise_std; unsigned long long seed; unsigned int draw;
  mobody_mlp_state sas, sa, sas_m, sas_v, sa_m, sa_v;   /* sas_classifier / sa_classifier parameters + Adam moments */
  int t;                                         /* optimiser step count AFTER this step (1-based)          */
  float lr;                                      /* config['actor_lr'] (mobody.py:135)                      */
  int nsplit;
  void* workspace; long long workspace_bytes;    /* >= mobody_classifier_workspace_bytes(N, S, A, nsplit)   */
  float* scalars_out;                            /* device float[2]                                         */
} mobody_classifier_desc;
long long mobody_classifier_workspace_bytes(int N, int S, int A, int nsplit);
int mobody_classifier_step(const mobody_classifier_desc* d, void* stream);
/* One-off source-reward relabel (mobody.py:364-378) on packed buffer rows, in place:
 * reward += penalty_coef * clamp(log p_sas(tar)/p_sas(src) - log p_sa(tar)/p_sa(src), -10, 10); penalty_out optional [n]. */
int mobody_dara_relabel(float* rows, long long n, int S, int A, int row_width, const mobody_mlp_params* sas,
                        const mobody_mlp_params* sa, float penalty_coef, float* penalty_out, void* stream);

/* ---- dynamics fitting step (SURVEY.md section 8f rank 3) ----
 * One mini-batch of MOBODYEnsembleDynamics.learn (algo/dynamics/mobody_dynamics.py:594-653): encoder_loss (:300-329,
 * incl. get_kl_loss :330-333), transition_loss (:336-347), reward_loss (:349-386), loss.backward() and the
 * torch.optim.Adam step (train_mobody.py:801-804: lr = dynamics_lr, default betas / eps, no weight decay), for the default
 * configuration (no_vae = 0, latent_reward = 0, inverse_sep_reward_loss = 0, mopo = 0).  Batches are per ensemble member
 * (the reference indexes a bootstrapped [7, B, .] view, :607-610).  Trained layers: zs1-3, transition1-3, reward_model1-3
 * and za_trg1-2 (use_trg) or za_src1-2; every other parameter of MOBODYModule receives no gradient in the reference and is
 * left untouched (its Adam state is never created there).  Parameters and moments are updated IN PLACE.
 * eps_latent: the six torch.randn_like draws of MOBODYModule.reparameterize in the reference's call order
 *   [0] encoder_decoder(s) [1] encoder_decoder(s') [2] encode_state(s) [3] encode_state(s') under no_grad
 *   [4] forward_*(s, a) of transition_loss [5] forward_*(s, a) of reward_loss;  eps_next: randn_like(mean) of reward_loss (:354).
 * Both NULL -> Philox draws keyed on (seed, draw).
 * scalars_out (device float[8]): [0] loss [1] transition_loss [2] encoder_loss [3] recon_loss [4] kl_loss [5] reward_loss. */
typedef struct mobody_dyn_state { float* w[MOBODY_N_DYN_LAYERS]; float* b[MOBODY_N_DYN_LAYERS]; } mobody_dyn_state;   /* writable twin of mobody_dyn_params */
typedef struct mobody_dynfit_desc {
  int S, A, B;                    /* B = rows per ensemble member                                                  */
  int use_trg;                    /* 1: target-domain batch (za_trg*, encoder weight 5x, reward weight 1); 0: source (za_src*, 1x, 0.01) */
  const float* obs; const float* act; const float* next_obs; const float* reward;   /* device fp32 [7,B,S] [7,B,A] [7,B,S] [7,B,1] */
  long long member_stride;        /* rows between consecutive members in the four batch tensors (0 = B: contiguous); lets a batch be a
                                     row window [:, lo:lo+B] of epoch tensors [7,N,.] without a copy (:607-610)     */
  const float* eps_latent;        /* [6,7,B,16] or NULL                                                            */
  const float* eps_next;          /* [7,B,S] or NULL                                                               */
  unsigned long long seed; unsigned int draw;
  float encoder_coef;             /* weight of encoder_loss in the total: (use_trg ? 5 : 1) * config['encoder_loss_coef'] (:623-626) */
  float reward_coef;              /* use_trg ? 1 : 0.01 (:381-384)                                                 */
  mobody_dyn_state params, adam_m, adam_v;
  int t_shared, t_action;         /* Adam step counts AFTER this step (1-based): shared layers / this domain's action encoder */
  float lr;
  int nsplit;                     /* K splits of the weight-gradient GEMMs, 1..16                                  */
  void* workspace; long long workspace_bytes;   /* >= mobody_dynfit_workspace_bytes(B, S, A, nsplit), 16-byte aligned */
  float* scalars_out;
} mobody_dynfit_desc;
long long mobody_dynfit_workspace_bytes(int B, int S, int A, int nsplit);
int mobody_dynfit_step(const mobody_dynfit_desc* d, void* stream);

/* ---- tensor-core weight images (precision MOBODY_PREC_BF16X2, MOBODY_PREC_BF16X2_WIDE or MOBODY_PREC_BF16X2_T64: one format;
 *      MOBODY_PREC_FP16 or MOBODY_PREC_FP16_T64: another) ----
 * The reference keeps weights as fp32 nn.Parameters (mobody_module.py:371-391, mobody.py:35-48); the
 * tcgen05 path consumes them as 16-bit planes in the UMMA shared-memory layout (one launch per image).
 * `state`: NULL -> pack unconditionally.  Otherwise device uint64[4], zero-initialised ONCE by the caller and then
 * owned by the library: a position-dependent 64-bit checksum of the live fp32 parameters is computed on the device
 * and the pack is skipped when it equals the checksum the image was packed from -- so calling this before every
 * step keeps the image coherent with ANY write to the parameters (optimiser step, load_state_dict, the `.data.copy_`
 * of MOBODYModule.load_save, mobody_module.py:407-408) without a host round trip. */
long long mobody_dyn_pack_bytes(int S, int A, int precision);
int mobody_dyn_pack(const mobody_dyn_params* dyn, int S, int A, int precision, void* blob, unsigned long long* state, void* stream);
long long mobody_mlp_pack_bytes(int din, int dout, int precision);
int mobody_mlp_pack(const mobody_mlp_params* mlp, int din, int dout, int precision, void* blob, unsigned long long* state, void* stream);

/* Test hook: D[128,N] = A[128,K] * B[N,K]^T on one CTA through the same tcgen05 operand layout,
 * descriptors and TMEM read-back as the rollout kernel (nsplit 1 = bf16, 2 = bf16 hi+lo split). */
int mobody_selftest_umma(const float* A, const float* B, int K, int N, int nsplit, float* D, void* stream);

/* Test hook of the train step's tensor-core tiles (tcgen05.mma.kind::tf32, TF32 hi+lo split, 3 MMAs per K step):
 * C[M][N] = A * B in fp32-class precision.  a_src / b_src: 0 = element (row, k) at src[row*ld + k], 1 = at src[k*ld + row]
 * (row = m for A, n for B).  N <= 256. */
int mobody_selftest_gemm(const float* A, const float* B, int M, int N, int K, int a_src, int b_src, int lda, int ldb,
                         float* C, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MOBODY_B200_H */
