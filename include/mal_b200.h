/*
 * mal_b200.h -- C ABI of libmal_b200.so: the B200 (sm_100a) implementation of ma-league's
 * value-decomposition hot path.  Plain pointers and sizes only; no torch types.  Every device
 * pointer must live on the device that is current when the call is made; every call enqueues
 * work on `stream` (a cudaStream_t passed as void*) and returns without synchronising unless
 * stated otherwise.  Return value: 0 = ok, non-zero = error, text via mal_last_error().
 *
 * Each entry point names the reference interface it replaces (paths relative to
 * /root/reference/src).  The reference has no FFI of its own (it is 100 % Python on top of
 * PyTorch); the binding a maintainer would add is the ctypes stub shown in INTEGRATION.md and
 * shipped as ma_league_b200/_native.py.
 *
 * Fixed model constants of the path: rnn_hidden_dim == MAL_HID (config/default.yaml:45),
 * n_actions <= MAL_MAX_ACTIONS, mixing_embed_dim <= MAL_MAX_EMBED (config/algs/qmix.yaml:21).
 *
 * Agent input (basic_controller.py:80-101): the columns of fc1's input are
 *   [obs | one-hot(a_{t-1}) if obs_last_action | one-hot(agent id) if obs_agent_id]   (config/default.yaml:46-47),
 * d_in = OBS + A * obs_last_action + N * obs_agent_id.  The learner (mal_learner_cfg_t.agent_input), the fused
 * act-select (the dense_input argument of mal_agent_step / mal_dqn_step) and the rollout step
 * (mal_rollout_io_t.agent_input) take the two switches as MAL_IN_* bits; 0 = both on, the reference's default.
 */
#ifndef MAL_B200_H
#define MAL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MAL_ABI_VERSION 6
#define MAL_HID 64
#define MAL_MAX_ACTIONS 32
#define MAL_MAX_EMBED 32
#define MAL_MAX_POLICIES 1024   /* n_policies cap of the per-match policy entries (the schedule kernel's shared memory) */

/* A scheme field of an EpisodeBatch (marl/components/episode_batch.py:89-143):
 * tensor [B, TT, *inner] whose inner dims are contiguous; sb/st are the batch / time strides
 * in ELEMENTS of the field's dtype (views produced by slicing keep working). */
typedef struct mal_field {
    const void *ptr;
    int64_t sb;
    int64_t st;
} mal_field_t;

/* The scheme of runs/train/ma_experiment.py:99-118 plus the derived keys. */
typedef struct mal_batch {
    int32_t B, TT, N, A, OBS, S;      /* episodes, stored steps (T+1), agents, actions, obs dim, state dim */
    mal_field_t obs;                  /* f32 [B,TT,N,OBS] */
    mal_field_t onehot;               /* f32 [B,TT,N,A]   actions_onehot */
    mal_field_t actions;              /* i64 [B,TT,N,1] */
    mal_field_t avail;                /* i32 [B,TT,N,A] */
    mal_field_t state;                /* f32 [B,TT,S] */
    mal_field_t reward;               /* f32 [B,TT,1] */
    mal_field_t terminated;           /* u8  [B,TT,1] */
    mal_field_t filled;               /* i64 [B,TT,1] */
    mal_field_t weight;               /* f32 [B] importance weights of prioritized replay (sb = batch stride, st unused), or
                                         ptr = NULL: unweighted.  Weighted: loss = sum_b w_b sum_t (td*m)^2 / sum m, seed
                                         2 w_b td m^2; the other statistics are unweighted.  Rejected with cfg.unnormalized */
} mal_batch_t;

/* MAL_MIXER_NONE: independent Q-learners (IQL, `mixer: None`): no mixing network, every agent has its own TD error
 * against the transition's reward and the [B,T] mask broadcast over agents (q_learner.py:81-98 with self.mixer = None). */
enum { MAL_MIXER_VDN = 0, MAL_MIXER_QMIX2 = 1, MAL_MIXER_QMIX1 = 2, MAL_MIXER_NONE = 3 };

/* agent-input switches: a set bit leaves that column block out of fc1's input */
enum { MAL_IN_NO_LAST_ACTION = 1 /* obs_last_action = False */, MAL_IN_NO_AGENT_ID = 2 /* obs_agent_id = False */ };

/* Hyper-parameters read by QLearner / Learner (marl/learners/q_learner.py:18-24,70,86,104;
 * marl/learners/learner.py:25-31) and QMixer (marl/modules/mixers/qmix.py:12-21). */
typedef struct mal_learner_cfg {
    int32_t mixer;                    /* MAL_MIXER_* */
    int32_t double_q;
    int32_t embed;                    /* mixing_embed_dim */
    int32_t hyper_embed;              /* hypernet_embed */
    float gamma, lr, alpha, eps, clip;
    int32_t save_q;                   /* also materialise mac_out / target_mac_out (tests, debugging) */
    int32_t unnormalized;             /* data-parallel mode: mal_learner_backward leaves the gradient WITHOUT the
                                         1/mask.sum() factor so that ranks can all-reduce grads and mask sums first */
    int32_t freeze_agent;             /* the agent's parameters are frozen (multi_agent_controller.py:74-76, args.freeze_native):
                                         no agent gradient is computed, its grad slice is zero and left out of the clip norm,
                                         and clip + RMSprop skip its parameters and square_avg (only the mixer trains) */
    int32_t agent_kind;               /* MAL_AGENT_RNN (drqn_agent.py) or MAL_AGENT_DQN (dqn_agent.py: fc1 -> ReLU -> fc2) */
    int32_t agent_input;              /* MAL_IN_* bits (0: obs | last action | agent id); sets d_in and n_agent_params */
    int32_t returns;                  /* MAL_RETURNS_*: the TD targets (0, a zeroed tail: the 1-step target) */
    float td_lambda;                  /* MAL_RETURNS_TD_LAMBDA: lambda in [0, 1] (build_td_lambda_targets, coma_learner.py:10-21) */
    double target_tau;                /* 0 (a zeroed tail): no soft target update.  tau in (0, 1]: mal_learner_step and
                                         mal_learner_step_adam blend the target flats toward the updated parameters
                                         after the optimiser step (see mal_soft_target_t) */
} mal_learner_cfg_t;
enum { MAL_AGENT_RNN = 0, MAL_AGENT_DQN = 1 };
/* MAL_RETURNS_ONE_STEP: targets = r_t + gamma (1 - term_t) tq[t] (q_learner.py:86).
 * MAL_RETURNS_TD_LAMBDA: with tq[b,t] = target_q_tot of row (b,t) and the learner mask m,
 *     R[b,T] = tq[b,T-1] (1 - sum_{t<T} term[b,t])
 *     R[b,t] = lambda gamma R[b,t+1] + m[b,t] (r[b,t] + (1 - lambda) gamma (1 - term[b,t]) tq[b,t])   t = T-1 .. 0
 *     targets = R[:, 0:T]   (per (b, agent) for MAL_MIXER_NONE, with r, term and m broadcast over agents).
 * Everything downstream of the targets (td, loss, seeds, importance weights, statistics) is unchanged. */
enum { MAL_RETURNS_ONE_STEP = 0, MAL_RETURNS_TD_LAMBDA = 1 };

/* Byte offsets of every intermediate inside the caller-owned workspace (filled by mal_learner_plan).
 * Row index of the [TT*R, .] arrays is m = t*R + b*N + n; of the [B*T, .] arrays m = b*T + t.
 * MAL_MIXER_NONE: n_mixer_params = 0, y1 / a2 / d_a2 / d_y1 are empty and q_tot / target_q_tot / targets / td hold
 * [B,T,N] (one TD error per agent); mask stays [B,T]. */
typedef struct mal_plan {
    int64_t total_bytes;
    int64_t n_agent_params, n_mixer_params;
    int64_t x_on, x_tg;               /* f32 [TT*R,64]   relu(fc1) */
    int64_t gi_on, gi_tg;             /* f32 [TT*R,192]  W_ih x + b_ih */
    int64_t h_on, h_tg;               /* f32 [TT*R,64]   hidden states */
    int64_t gates;                    /* f32 [TT*R,256]  r|z|n|W_hn h+b_hn (online) */
    int64_t mac_out, target_mac_out;  /* f32 [B,TT,N,A]  (only when cfg.save_q) */
    int64_t chosen, target_max;       /* f32 [B,T,N] */
    int64_t argmax;                   /* i32 [B,T,N] */
    int64_t mask;                     /* f32 [B,T] */
    int64_t y1_on, y1_tg;             /* f32 [B*T, 2*HE+2*E]  h1|hf|b1|v1 */
    int64_t a2_on, a2_tg;             /* f32 [B*T, E*N+E]     a1|af (pre-abs) */
    int64_t q_tot, target_q_tot, targets, td;   /* f32 [B*T] ([B*T*N] for MAL_MIXER_NONE: chosen / target_max per agent) */
    int64_t d_a2, d_y1;               /* f32 like a2 / y1 */
    int64_t d_chosen;                 /* f32 [B,T,N] */
    int64_t d_g;                      /* f32 [TT*R,256]  d(gi_r)|d(gi_z)|d(gi_n)|d(gh_n) */
    int64_t d_x;                      /* f32 [TT*R,64] */
    int64_t dh_head;                  /* f32 [TT*R,64]  d_chosen * fc2.weight[a_t] (rows of t < T) */
    int64_t partials;                 /* f32 scratch for split reductions */
    int64_t partials_bytes;
    int64_t scalars;                  /* f32 [64]: see MAL_SC_* */
    int64_t w_t;                      /* f32: transposed copies of the weights the backward GEMMs read row-wise, written by the
                                         forward call: gru.weight_ih^T [64,192] | hyper_w_1.2.weight^T [HE,E*N] | hyper_w_final.2.weight^T [HE,E] */
} mal_plan_t;

/* indices into the scalars block (all float32 except where noted) */
enum {
    MAL_SC_MASK_SUM = 0, MAL_SC_LOSS = 1, MAL_SC_TD_ABS = 2, MAL_SC_Q_TAKEN = 3, MAL_SC_TARGET = 4,
    MAL_SC_GRAD_NORM = 5, MAL_SC_MASK_COUNT = 6 /* int32 bits */, MAL_SC_STATUS = 7 /* int32 bits */,
    /* raw (un-normalised) sums of this rank, for the data-parallel reduction:
       sum (td*mask)^2, sum |td*mask|, sum q_tot*mask, sum targets*mask, sum mask, count(mask != 0) */
    MAL_SC_RAW0 = 8
};

int mal_version(void);
const char *mal_last_error(void);

/* Accounting: number of kernels this library has launched so far (process-wide), and an opt-in profiler that
 * brackets every launch with CUDA events on the launching stream.  mal_profile_end synchronises and writes one
 * text line per kernel name: "<name> <launches> <total_ms>\n". */
uint64_t mal_launch_count(void);
/* kernels launched through a replayed CUDA graph that captured calls of this library (added to mal_launch_count) */
void mal_count_launches(uint64_t n);
int mal_profile_begin(void);
int mal_profile_end(char *out, int64_t out_len);
/* same, but one line per launch in issue order: "<name> <start_us> <end_us>\n" relative to the first recorded launch */
int mal_profile_end_timeline(char *out, int64_t out_len);

/* Parameter counts in state_dict order (drqn_agent.py:21-23, qmix.py:16-39). */
int64_t mal_agent_param_count(int32_t d_in, int32_t n_actions);
int64_t mal_agent_param_count_kind(int32_t agent_kind, int32_t d_in, int32_t n_actions);   /* MAL_AGENT_DQN: dqn_agent.py:24-25 */
int64_t mal_mixer_param_count(int32_t mixer, int32_t state_dim, int32_t n_agents, int32_t embed, int32_t hyper_embed);

int mal_learner_plan(const mal_batch_t *batch, const mal_learner_cfg_t *cfg, mal_plan_t *plan);

/* QLearner.train forward half, marl/learners/q_learner.py:36-98: unroll of the online and target
 * RNN agents, chosen-action gather, masked (double-Q) target max, mixers, TD error, masked loss.
 * Parameters are flat fp32 buffers in state_dict order. Results land in the workspace (plan offsets).
 * mixer / target_mixer may be NULL for MAL_MIXER_VDN and MAL_MIXER_NONE (no mixer parameters).
 * MAL_MIXER_NONE: the loss normaliser and every statistic use the mask expanded to [B,T,N] (q_learner.py:92,117-124):
 * scalars[MAL_SC_MASK_SUM] = N * mask.sum(), MAL_SC_MASK_COUNT counts N per live transition, and q_taken / target means
 * divide by that sum times N, as the reference's lines do. */
int mal_learner_forward(const mal_batch_t *batch, const mal_learner_cfg_t *cfg, const mal_plan_t *plan,
                        const float *agent, const float *target_agent, const float *mixer,
                        const float *target_mixer, void *workspace, void *stream);

/* loss.backward() of q_learner.py:103 for the state left by mal_learner_forward:
 * writes d loss / d params into grad[0 : n_agent_params + n_mixer_params] (agent first). */
int mal_learner_backward(const mal_batch_t *batch, const mal_learner_cfg_t *cfg, const mal_plan_t *plan,
                         const float *agent, const float *mixer, void *workspace, float *grad, void *stream);

/* clip_grad_norm_ + RMSprop.step of q_learner.py:104-105 / learner.py:25-31 over two flat
 * parameter buffers (agent, mixer) sharing one grad / square_avg buffer.  grad is scaled in place like
 * clip_grad_norm_ does; the unclipped global norm is written to scalars[MAL_SC_GRAD_NORM];
 * scratch needs ceil((n_agent+n_mixer)/256) floats. */
int mal_clip_rmsprop(float *agent, int64_t n_agent, float *mixer, int64_t n_mixer, float *grad,
                     float *square_avg, float lr, float alpha, float eps, float clip, float *scalars,
                     float *scratch, const float *denominator, int64_t n_frozen, void *stream);
/* denominator: NULL, or a DEVICE pointer to the global mask sum; the gradient is divided by it first (data-parallel
 * mode: grads and mask sums are all-reduced across ranks, then every rank applies the identical update).
 * n_frozen: the first n_frozen parameters are frozen (requires_grad = False): their gradient is zeroed and left out
 * of the norm, and neither they nor their square_avg are touched. */

/* Data-parallel mode, fused exchange: peer_bufs[r] = device pointer of rank r's symmetric buffer holding its UN-normalised
 * gradient [n_agent + n_mixer] followed by `tail` raw statistic sums (element 4 = its mask sum), all peer-mapped into
 * this process (torch symmetric memory / cudaIpc).  One kernel sums them in rank order over NVLink, normalises by the
 * global mask sum into the LOCAL grad_out, writes the reduced tail to tail_out, then clip + RMSprop run as usual.
 * The caller separates steps with a cross-rank barrier (nobody rewrites a buffer that a peer may still be reading). */
int mal_peer_allreduce_clip_rmsprop(const void *const *peer_bufs, int32_t world, float *agent, int64_t n_agent, float *mixer,
                                    int64_t n_mixer, float *grad_out, float *tail_out, int32_t tail, float *square_avg,
                                    float lr, float alpha, float eps, float clip, float *scalars, float *scratch,
                                    int64_t n_frozen, void *stream);

/* forward + backward + clip + RMSprop in one call (the whole of q_learner.py:34-105).  With cfg->target_tau > 0 the
 * step ends with the soft target update below and writes target_agent / target_mixer. */
int mal_learner_step(const mal_batch_t *batch, const mal_learner_cfg_t *cfg, const mal_plan_t *plan,
                     float *agent, const float *target_agent, float *mixer, const float *target_mixer,
                     void *workspace, float *grad, float *square_avg, void *stream);

/* Adam (torch.optim.Adam with amsgrad = False, maximize = False and L2 weight decay that is not decoupled) in place of
 * RMSprop.  For the trained parameters (a frozen prefix is skipped), after clip_grad_norm_ scaled grad in place:
 *     g' = g + weight_decay * p  (not written back) ; t = step + 1
 *     m = beta1 m + (1 - beta1) g' ; v = beta2 v + (1 - beta2) g'^2
 *     p -= (lr / (1 - beta1^t)) * m / (sqrt(v) / sqrt(1 - beta2^t) + eps) ; step = t
 * with the bias corrections computed in double.  The caller owns the optimiser state, MAL_ADAM_STATE_FLOATS(P) floats
 * for P = n_agent + n_mixer parameters, zeroed before the first step:
 *     exp_avg [P] | exp_avg_sq [P] | step (f32) | ticket (u32 bits, must stay 0 between calls)
 * The step counter lives in this buffer on the device, so a captured CUDA graph advances it on every replay.  As
 * torch's float32 `step` state, it counts exactly up to 2^24 steps. */
#define MAL_ADAM_STATE_FLOATS(P) (2 * (P) + 2)
typedef struct mal_adam {
    double lr, beta1, beta2, eps, weight_decay;   /* lr, betas, eps, weight_decay of the optimiser's param group */
    float clip;                                   /* grad_norm_clip (q_learner.py:104) */
} mal_adam_t;

/* mal_learner_step with Adam: cfg->lr / alpha / eps / clip are not read, `adam` holds the hyper-parameters. */
int mal_learner_step_adam(const mal_batch_t *batch, const mal_learner_cfg_t *cfg, const mal_plan_t *plan,
                          float *agent, const float *target_agent, float *mixer, const float *target_mixer,
                          void *workspace, float *grad, const mal_adam_t *adam, float *adam_state, void *stream);
/* mal_clip_rmsprop with Adam (same grad, scalars, scratch, denominator and n_frozen contract). */
int mal_clip_adam(float *agent, int64_t n_agent, float *mixer, int64_t n_mixer, float *grad, float *adam_state,
                  const mal_adam_t *adam, float *scalars, float *scratch, const float *denominator, int64_t n_frozen,
                  void *stream);
/* mal_peer_allreduce_clip_rmsprop with Adam. */
int mal_peer_allreduce_clip_adam(const void *const *peer_bufs, int32_t world, float *agent, int64_t n_agent, float *mixer,
                                 int64_t n_mixer, float *grad_out, float *tail_out, int32_t tail, float *adam_state,
                                 const mal_adam_t *adam, float *scalars, float *scratch, int64_t n_frozen, void *stream);

/* Soft target update (EPyMARL's `target_update_interval_or_tau` <= 1), in the optimiser kernel's pass over the
 * parameters: after the clip + RMSprop / Adam update, for every parameter p of agent | mixer, the frozen prefix included,
 *     c1 = (float)(1.0 - tau) (subtraction in double) ; c2 = (float)tau
 *     target[p] = fp32(fp32(target[p] * c1) + fp32(p_new * c2))   (no FMA contraction)
 * which is `target.data.copy_(target.data * (1.0 - tau) + param.data * tau)` on fp32 tensors; tau = 1 copies.  The target
 * flats have the layout of the online flats.  The *_soft entries are their namesakes followed by this update; they
 * reject a tau that is not a finite number in (0, 1] and a missing target buffer (target_mixer may be NULL when
 * n_mixer = 0). */
typedef struct mal_soft_target {
    double tau;
    float *target_agent;              /* [n_agent] */
    float *target_mixer;              /* [n_mixer] */
} mal_soft_target_t;
int mal_clip_rmsprop_soft(float *agent, int64_t n_agent, float *mixer, int64_t n_mixer, float *grad,
                          float *square_avg, float lr, float alpha, float eps, float clip, float *scalars,
                          float *scratch, const float *denominator, int64_t n_frozen, const mal_soft_target_t *soft,
                          void *stream);
int mal_peer_allreduce_clip_rmsprop_soft(const void *const *peer_bufs, int32_t world, float *agent, int64_t n_agent,
                                         float *mixer, int64_t n_mixer, float *grad_out, float *tail_out, int32_t tail,
                                         float *square_avg, float lr, float alpha, float eps, float clip, float *scalars,
                                         float *scratch, int64_t n_frozen, const mal_soft_target_t *soft, void *stream);
int mal_clip_adam_soft(float *agent, int64_t n_agent, float *mixer, int64_t n_mixer, float *grad, float *adam_state,
                       const mal_adam_t *adam, float *scalars, float *scratch, const float *denominator, int64_t n_frozen,
                       const mal_soft_target_t *soft, void *stream);
int mal_peer_allreduce_clip_adam_soft(const void *const *peer_bufs, int32_t world, float *agent, int64_t n_agent,
                                      float *mixer, int64_t n_mixer, float *grad_out, float *tail_out, int32_t tail,
                                      float *adam_state, const mal_adam_t *adam, float *scalars, float *scratch,
                                      int64_t n_frozen, const mal_soft_target_t *soft, void *stream);

/* update_targets, q_learner.py:127-131 (load_state_dict of the flat buffers). */
int mal_copy_f32(float *dst, const float *src, int64_t n, void *stream);

/* BasicMAC.forward for one timestep, basic_controller.py:38-54,80-92 + drqn_agent.py:29-35.
 * Row r = b*N + n (b-major).  obs = ep_batch["obs"][:, t] as [bs,N,OBS] with batch stride obs_sb (elements,
 * inner [N,OBS] contiguous), last_onehot = ep_batch["actions_onehot"][:, t-1] likewise or NULL (t == 0),
 * h_in [rows,64] or NULL (zeros), writes q [rows,A] and h_out [rows,64] (contiguous).
 * When `sel` is non-NULL the epsilon-greedy selection below is fused into the same launch. */
typedef struct mal_select {
    const int32_t *avail;             /* [bs,N,A] with batch stride avail_sb, inner [N,A] contiguous */
    int64_t avail_sb;
    float epsilon;                    /* already the schedule's value (0 in test mode) */
    int32_t rng_mode;                 /* 0: injected u/e, 1: Philox4x32-10 (seed, offset) */
    const float *u;                   /* [rows]      uniform draws  (mode 0) */
    const float *e;                   /* [rows,A]    Exp(1) draws   (mode 0) */
    uint64_t seed, offset;            /* mode 1 */
    int64_t *actions;                 /* [rows] out */
    int64_t *greedy;                  /* [rows] out: 1 - pick_random */
    int32_t *status;                  /* device int: set to 1 if a row has no available action */
} mal_select_t;

int mal_agent_step(const float *agent, int32_t rows, int32_t n_agents, int32_t obs_dim, int32_t n_actions,
                   int32_t dense_input, const float *obs, int64_t obs_sb, const float *last_onehot,
                   int64_t onehot_sb, const float *h_in, float *h_out, float *q, const mal_select_t *sel,
                   void *stream);
/* dense_input bit 0 set: `obs` is the already assembled agent input [rows, obs_dim] with row stride obs_sb
 * (DRQNAgentNetwork.forward(inputs, hidden_state), drqn_agent.py:29-35); obs_dim is then the full input width.
 * Bit 0 clear (fused input assembly): bits 1..2 are the agent-input switches, MAL_IN_* << 1 (last_onehot is not read
 * when MAL_IN_NO_LAST_ACTION is set).  Other bits are rejected. */

/* The same for the feed-forward DQNAgentNetwork (marl/modules/agents/dqn_agent.py:9-37: q = fc2(relu(fc1(inputs))), the
 * hidden state is passed through untouched); flat parameters fc1.weight | fc1.bias | fc2.weight | fc2.bias. */
int mal_dqn_step(const float *agent, int32_t rows, int32_t n_agents, int32_t obs_dim, int32_t n_actions,
                 int32_t dense_input, const float *obs, int64_t obs_sb, const float *last_onehot, int64_t onehot_sb,
                 float *q, const mal_select_t *sel, void *stream);

/* One rollout timestep of `bs` lock-step matches in ONE launch: the loop body of EpisodeStepper.run / SelfPlayStepper.run
 * (steppers/episode_stepper.py:110-142,177-186; steppers/self_play_stepper.py:64-106) for one team --
 *   EpisodeBatch.update(pre_transition_data, ts=t)   state / avail_actions / obs from the environment + filled = 1
 *   EpisodeBatch.update(post_transition_data, ts=t-1) reward / terminated of the previous step (when prev_reward != NULL)
 *   BasicMAC.select_actions(batch, t_ep=t, ...)       mal_agent_step + epsilon-greedy on the environment's obs / avail
 *   EpisodeBatch.update({"actions": ...}, ts=t)       actions + the derived actions_onehot
 * All `*_t` pointers address element [0, t] of the batch field (`*_tm1`: [0, t-1]); strides are batch strides in elements
 * of the field's dtype.  `alive` (optional, [bs] bytes): matches that have already ended select on a dummy avail row (no
 * ValueError from their all-zero rows); what they write past their end is cleared by the caller after the loop. */
typedef struct mal_rollout_io {
    int32_t state_dim;
    const float *env_state; int64_t env_state_sb;         /* [bs,S]      env.get_state()          */
    const int32_t *env_avail; int64_t env_avail_sb;       /* [bs,N,A]    env.get_avail_actions()  */
    const float *env_obs; int64_t env_obs_sb;             /* [bs,N,OBS]  env.get_obs()            */
    const uint8_t *alive;                                 /* [bs] or NULL */
    const float *prev_reward;                             /* [bs] or NULL (t == 0) */
    const uint8_t *prev_done;                             /* [bs] */
    float *state_t; int64_t state_sb;
    int32_t *avail_t; int64_t avail_sb;
    float *obs_t; int64_t obs_sb;
    int64_t *filled_t; int64_t filled_sb;
    int64_t *actions_t; int64_t actions_sb;
    float *onehot_t; int64_t onehot_sb;
    const float *onehot_tm1; int64_t onehot_tm1_sb;       /* actions_onehot[:, t-1] (agent input), NULL at t == 0 */
    float *reward_tm1; int64_t reward_sb;
    uint8_t *term_tm1; int64_t term_sb;
    int32_t agent_input;                                  /* MAL_IN_* bits of the agent's input (0: the default layout) */
} mal_rollout_io_t;

/* `sel` is required (sel->avail / avail_sb are ignored: the environment's avail rows of `io` are used).
 * onehot_t is written whatever io->agent_input says (actions_onehot is part of the batch scheme). */
int mal_rollout_step(const float *agent, int32_t bs, int32_t n_agents, int32_t obs_dim, int32_t n_actions,
                     const mal_rollout_io_t *io, const float *h_in, float *h_out, float *q, const mal_select_t *sel,
                     void *stream);

/* Per-match policies: one rollout / act-select launch over `bs` matches in which match b plays its own entry of a table of
 * agents (a league opponent per match, or every pairing of a population in cross-play).  `table` is [n_policies, table_ld]
 * fp32, row k = the flat parameters of agent k in state_dict order (DeviceAgentPool.pool, agent.flat_params()); table_ld
 * >= the agent's parameter count and may be odd (4-byte alignment is enough).  The table is read at every step, never
 * copied.  Recurrent agent (MAL_AGENT_RNN) only; 1 <= n_policies <= MAL_MAX_POLICIES.
 *
 * mal_policy_schedule_bytes: host-only (no device needed): size of the schedule buffer for (bs, n_agents, n_policies),
 *   -1 with mal_last_error set for arguments the entries reject.
 * mal_policy_schedule: ONE launch, once per assignment: match_policy [bs] (int32, device) -> `schedule` (a caller-owned,
 *   16-byte aligned device buffer of mal_policy_schedule_bytes; its content is internal to the library).  An id outside
 *   [0, n_policies) sets *status (device int, may be NULL) to 1 and its match is left out: no step reads its rows or
 *   anything outside the table.
 * mal_agent_step_pool / mal_rollout_step_pool: mal_agent_step / mal_rollout_step (every argument means what it means
 *   there; rows = bs * n_agents) with match b's rows computed from table row match_policy[b].  Row indices of inputs,
 *   hidden states, outputs, avail rows and Philox draws are unchanged, so each match gets bit for bit what the plain entry
 *   computes over the whole batch with its policy.  The schedule must have been built for the same bs, n_agents and
 *   n_policies (a CTA that finds another shape in it computes nothing). */
int64_t mal_policy_schedule_bytes(int32_t bs, int32_t n_agents, int32_t n_policies);
int mal_policy_schedule(const int32_t *match_policy, int32_t bs, int32_t n_agents, int32_t n_policies,
                        void *schedule, int32_t *status, void *stream);
int mal_agent_step_pool(const float *table, int64_t table_ld, int32_t n_policies, const void *schedule,
                        int32_t rows, int32_t n_agents, int32_t obs_dim, int32_t n_actions, int32_t dense_input,
                        const float *obs, int64_t obs_sb, const float *last_onehot, int64_t onehot_sb,
                        const float *h_in, float *h_out, float *q, const mal_select_t *sel, void *stream);
int mal_rollout_step_pool(const float *table, int64_t table_ld, int32_t n_policies, const void *schedule,
                          int32_t bs, int32_t n_agents, int32_t obs_dim, int32_t n_actions,
                          const mal_rollout_io_t *io, const float *h_in, float *h_out, float *q,
                          const mal_select_t *sel, void *stream);

/* Launch counters per kernel flavour since process start, for tests that assert which variant the launch heuristics
 * picked: "linear_tc2" (pipelined tcgen05 GEMM), "linear_tc", "reduce_tc", "reduce_tc_swap", "reduce_ffma",
 * "agent_in_fused", "rec_tc", "rec_tc_bwd", "reduce_fc1", "gru_balanced" (forward recurrence as 2 x SMs equal workers).
 * Unknown names return 0. */
uint64_t mal_stat(const char *name);

/* Library options (experiment switches; the defaults are the measured best).  They are PER CALLING THREAD, like the
 * library's side streams: a second thread driving another learner keeps its own settings.
 *   "tensor_cores"  1 (default): batched projections on tcgen05 (3xTF32, fp32-accurate); 0: fp32 FFMA panel GEMM
 *   "tc_pipelined"  0 / 1 (default, by launch size) / 2 (always): warp-specialised pipelined GEMM kernel
 *   "reduce_tc"     0 / 1 (default, by rows per CTA) / 2 (always): weight-gradient reductions on tcgen05
 *   "fuse_agent_in" 1 (default): fc1 + W_ih in one kernel; 0: two grouped GEMM launches
 *   "actsel_lat"    1 (default): rollout-sized act-select launches use the mma.sync latency kernel; 0: the lanes-along-k kernel
 *   "overlap"       1 (default): independent kernel chains of the learner step on side streams; 0: one stream
 *   "pdl"           1 (default): programmatic dependent launch along the main kernel chain; 0: full serialisation
 *   "time_chunks"   1 (default) / 2: time-chunked forward (input projection of the 2nd half beside the 1st half's recurrence)
 *   "gru_balance"   a forward recurrence of more than 2 and at most 3 chains per SM can run as 2 x SMs equal workers (a chain
 *                   may change workers once): 1 (default) when nothing runs beside it (VDN, no mixer), 2 always, 0 never
 *   "rec_carveout"  bit 0 / bit 1 (default 2 = backward only): the forward / backward recurrence kernel prefers the largest shared-memory
 *                   carve-out, so that the tcgen05 GEMMs of the side streams can be resident beside it (an SM keeps its L1 /
 *                   shared split while CTAs are resident); bit 2: the small kernels of the step too; 0: default carve-outs
 * Returns non-zero (and sets mal_last_error) for an unknown name. */
int mal_set_option(const char *name, int value);

/* Unit-test hook: Y = epi(A W^T + bias) on dense operands through the learner's own GEMM kernels
 * (epi 0 = bias, 1 = ReLU, 2 = multiply by (aux > 0); w_trans: W(n,k) = W[k*ldw + n]). */
int mal_debug_linear(int32_t M, int32_t K, int32_t Nout, const float *A, int64_t lda, const float *W, int64_t ldw,
                     int32_t w_trans, const float *bias, int32_t epi, const float *aux, int64_t ld_aux, float *Y,
                     int64_t ldy, int32_t use_tc, void *stream);

/* Unit-test hooks for the split-M weight-gradient reductions of the learner's backward, dW[n,k] = sum_m dY[m,n] A[m,k].
 * Each launches exactly the kernel instance the learner launches and writes the RAW per-chunk partials (no gather): chunk c
 * covers rows [c * rows_per_chunk, min((c + 1) * rows_per_chunk, M)), n_chunks = ceil(M / rows_per_chunk).  rows_per_chunk
 * must be a positive multiple of 64 and M < 2^31.  The mal_stat counters tick as in the learner.
 *
 * mal_debug_reduce: 1 to 3 problems as one grouped launch; part_w [n_chunks][Nout][K], part_b [n_chunks][Nout] (NULL: no
 * bias).  All problems share the A loader a_kind:
 *   MAL_RED_A_DENSE     row m reads A[(m - shift) * lda ..] (zero for m < shift);
 *   MAL_RED_A_STATE     row m = b*T + t reads batch->state[b, t + shift] (T = TT - 1, shift <= 1, K <= S, M <= B*T);
 *   MAL_RED_A_AGENT_IN  row m = t*R + b*N + n (R = B*N) reads [obs | one-hot(a_{t-1}) | agent id] as the MAL_IN_* bits of
 *                       agent_input select them (K = d_in, shift 0, M <= TT*R).
 *   batch is read by the last two only.  flavour: 0 fp32 FFMA (k_reduce_group); 1, 2, 3 tcgen05 k_reduce_tc with
 *   "reduce_mn" = 0, 1, 2; 4 the 512-thread k_reduce_tc3 ("reduce_mn" = 3, the default).
 * mal_debug_reduce_gru: the fused GRU weight gradients (k_reduce_gru) over M1 rows with h_{t-1}[m] = hout[m - R] (zero for
 *   m < R).  x, hout [M1,64], d_g [M1,256] contiguous and 16-byte aligned.  Per chunk: wih_w [192][64] = d_g[:, :192]^T x,
 *   whh_rz_w [128][64] = d_g[:, :128]^T h_{t-1}, whh_n_w [64][64] = d_g[:, 192:]^T h_{t-1}, the biases the column sums.
 * mal_debug_reduce_fc1: the fc1 weight gradient over the full input width (k_reduce_fc1), d_x [M,64] contiguous and 16-byte
 *   aligned, rows and input columns as MAL_RED_A_AGENT_IN; d_in <= 256.  part_w [n_chunks][64][d_in], part_b [n_chunks][64].
 * mal_debug_fc2_grad: the fc2 gradients (k_fc2_grad) over the T*R rows of the batch's actions, d_chosen [B,T,N] and hout
 *   [TT*R,64] (8-byte aligned) on `grid` CTAs: part_w [grid][A][64], part_b [grid][A]; CTA c sums the rows m whose
 *   m mod (8 grid) lies in [8c, 8c + 8). */
typedef struct mal_red_prob {
    int64_t M, rows_per_chunk;
    int32_t K, Nout, shift;
    const float *dY;
    int64_t ldy;
    const float *A;                   /* MAL_RED_A_DENSE only */
    int64_t lda;
    float *part_w, *part_b;
} mal_red_prob_t;
enum { MAL_RED_A_DENSE = 0, MAL_RED_A_AGENT_IN = 1, MAL_RED_A_STATE = 2 };
int mal_debug_reduce(int32_t flavour, int32_t a_kind, int32_t n_probs, const mal_red_prob_t *probs,
                     const mal_batch_t *batch, int32_t agent_input, void *stream);
int mal_debug_reduce_gru(const float *x, const float *hout, const float *d_g, int64_t M1, int32_t R, int64_t rows_per_chunk,
                         float *wih_w, float *wih_b, float *whh_rz_w, float *whh_rz_b, float *whh_n_w, float *whh_n_b,
                         void *stream);
int mal_debug_reduce_fc1(const mal_batch_t *batch, int32_t agent_input, const float *d_x, int64_t M, int64_t rows_per_chunk,
                         float *part_w, float *part_b, void *stream);
int mal_debug_fc2_grad(const mal_batch_t *batch, const float *d_chosen, const float *hout, int32_t grid, float *part_w,
                       float *part_b, void *stream);

/* QMixer.forward / VDNMixer.forward outside the learner, qmix.py:41-59 / vdn.py:9-10 (MAL_MIXER_NONE is rejected:
 * there is no mixer module to run).
 * agent_qs [B*T,N] contiguous, states [B,T,S] with strides in elements, scratch >= B*T*(2*HE+2*E + E*N+E)
 * floats (unused for VDN), q_tot [B*T]. */
int mal_mixer_forward(int32_t mixer, int32_t B, int32_t T, int32_t N, int32_t S, int32_t E, int32_t HE,
                      const float *params, const float *agent_qs, const float *states, int64_t state_sb,
                      int64_t state_st, float *scratch, float *q_tot, void *stream);

/* Autograd backward of the stand-alone module calls (BasicMAC.forward / DRQNAgentNetwork.forward / DQNAgentNetwork.forward for
 * one step, QMixer.forward), for callers that train through the modules with torch autograd instead of QLearner.train.
 * Both recompute what they need from the forward's inputs, write gradients (no accumulation: the caller adds them up) and
 * use no float atomics: two identical calls return bit-identical results.  Gradients with respect to obs / assembled inputs
 * and states are not computed.  The workspace queries are host-only (no device needed); they return the size in bytes,
 * or -1 (mal_last_error set) for arguments the backward rejects.
 *
 * mal_agent_step_backward: one step of mal_agent_step (agent_kind MAL_AGENT_RNN) or mal_dqn_step (MAL_AGENT_DQN).  agent,
 * rows ... onehot_sb and h_in mean exactly what they mean there (dense_input bit 0 = assembled input, bits 1..2 = MAL_IN_*
 * << 1; h_in NULL = zeros).  Upstream gradients: d_q [rows,A] and d_h_out [rows,64], either may be NULL (zeros).  Outputs:
 * d_h_in [rows,64] (NULL: not wanted) and d_agent, the step's gradient of the flat parameters in state_dict order (NULL:
 * frozen agent, only d_h_in is computed).  The feed-forward agent has no hidden state: h_in, d_h_out and d_h_in must be
 * NULL (its hidden state passes through, so is its gradient).  All outputs contiguous. */
int64_t mal_agent_step_backward_workspace(int32_t agent_kind, int32_t rows, int32_t n_agents, int32_t obs_dim,
                                          int32_t n_actions, int32_t dense_input);
int mal_agent_step_backward(int32_t agent_kind, const float *agent, int32_t rows, int32_t n_agents, int32_t obs_dim,
                            int32_t n_actions, int32_t dense_input, const float *obs, int64_t obs_sb,
                            const float *last_onehot, int64_t onehot_sb, const float *h_in, const float *d_q,
                            const float *d_h_out, float *d_h_in, float *d_agent, void *workspace, void *stream);

/* mal_mixer_backward: QMixer.forward backward for MAL_MIXER_QMIX2 / MAL_MIXER_QMIX1 (VDN's is d q_tot broadcast over the agents
 * and needs no kernel; other mixers are rejected).  Arguments as in mal_mixer_forward; `scratch` is the buffer that the
 * matching mal_mixer_forward call filled (raw hypernet outputs), d_q_tot [B*T].  Writes d_agent_qs [B*T,N] and d_params, the
 * gradient of the flat mixer parameters in state_dict order.  The derivative of abs() is the sign of the raw value (0 at 0),
 * as torch takes it. */
int64_t mal_mixer_backward_workspace(int32_t mixer, int32_t B, int32_t T, int32_t N, int32_t S, int32_t E, int32_t HE);
int mal_mixer_backward(int32_t mixer, int32_t B, int32_t T, int32_t N, int32_t S, int32_t E, int32_t HE,
                       const float *params, const float *agent_qs, const float *states, int64_t state_sb,
                       int64_t state_st, const float *scratch, const float *d_q_tot, float *d_agent_qs, float *d_params,
                       void *workspace, void *stream);

/* EpsilonGreedyActionSelector.select on existing Q-values, marl/components/action_selectors.py:44-62. */
int mal_eps_greedy_select(const float *q, int64_t q_ld, int32_t rows, int32_t n_agents, int32_t n_actions,
                          const mal_select_t *sel, void *stream);

/* Generator advance (in 32-bit Philox outputs) that th.rand_like([rows]) followed by exponential_([rows,A])
 * consume on this device (ATen/native/cuda/DistributionTemplates.h calc_execution_policy); rng_mode 1 uses the
 * same counter layout, so the caller adds this to torch's CUDA generator offset after each select. */
int mal_select_philox_advance(int32_t rows, int32_t n_actions, uint64_t *advance);

/* ReplayBuffer.sample / insert_episode_batch data movement, replay_buffer.py:22-53 /
 * episode_batch.py:226-238, over packed episode records: record i of dst (dst_ids ? dst_ids[i] : i)
 * receives `bytes` bytes of record (src_ids ? src_ids[i] : i) of src.  Strides and `bytes` must be
 * multiples of 16 and the bases 16-byte aligned (the host side pads records to 128 B). */
int mal_record_copy(void *dst, int64_t dst_stride, const int64_t *dst_ids, const void *src, int64_t src_stride,
                    const int64_t *src_ids, int32_t n, int64_t bytes, void *stream);

/* Compact wire form of an episode batch for the host <-> device path of a host-resident replay buffer
 * (`buffer_cpu_only`: runs/train/ma_experiment.py:238-239 moves the sampled batch to the device every step).  The wire
 * record of an episode holds, per stored step, state f32 | obs f32 | reward f32 | actions u8 [N] | avail bitmask u32 [N] |
 * flags u8 (bit 0 filled, bit 1 terminated); `actions_onehot` and `filled` are re-derived on the device (OneHot,
 * transforms.py:16-19: written for filled steps).  mal_wire_pack sets *status (device int, may be NULL) to 1 when a value
 * does not fit the encoding (actions outside [0, 255], avail flags other than 0 / 1, a one-hot row that is not the
 * OneHot of its action or all-zero); n_actions <= 32. */
typedef struct mal_wire_layout {
    int64_t record_bytes;             /* per episode, multiple of 128 */
    int64_t off_state, off_obs, off_reward, off_actions, off_avail, off_flags;
} mal_wire_layout_t;
int mal_wire_layout(int32_t TT, int32_t N, int32_t OBS, int32_t S, mal_wire_layout_t *out);
int mal_wire_pack(const mal_batch_t *batch, void *wire, const mal_wire_layout_t *layout, int32_t *status, void *stream);
int mal_wire_unpack(const mal_batch_t *batch, const void *wire, const mal_wire_layout_t *layout, void *stream);

/* Proportional prioritized episode replay (Schaul et al., 2016) over the live slots [0, n) of a replay buffer.
 *
 * mal_per_sample: ONE launch.  total = sum p_i, p_min = min p_i over the n slots (fixed reduction / scan order, fp64 prefix
 *   sums: identical inputs give bit-identical ids).  Draw j of B takes x_j = (j + u_j) * total / B and returns the first slot
 *   whose inclusive prefix sum exceeds x_j (sampling with replacement, stratified); ids [B] int64 can go straight into
 *   mal_record_copy as src_ids.  weights [B] f32: w_j = (p_min / p_{id_j})^beta (1 where p_{id_j} = 0).  Uniforms: u [B]
 *   (device) when non-NULL; otherwise Philox4x32-10 at (seed, offset) in exactly the layout th.rand(B) uses on this device,
 *   and *advance (may be NULL) receives what the caller adds to the generator's offset (0 for injected uniforms).
 *   priorities must be 16-byte aligned, >= 0 and finite.
 * mal_per_update: ONE launch after a learner step over the workspace's td ([B*T*n_q], row m = b*T + t; n_q = 1 with a mixer,
 *   N without) and mask ([B*T]): priorities[ids[b]] = (sum_{t,n} |td*m| / sum_{t,n} m + eps)^alpha (0 for the ratio when the
 *   episode has no live transition).  When a batch samples a slot twice the occurrence with the highest batch index wins;
 *   ids outside [0, capacity) are skipped.  *max_priority (device float) is raised to the largest new priority.
 * The _check queries are host-only (no device needed): 0, or non-zero with mal_last_error set for arguments the entries
 *   reject (n == 0, B < 1, a negative or non-finite alpha / beta / eps). */
int mal_per_sample_check(int64_t n, int32_t B, float beta);
int mal_per_sample(const float *priorities, int64_t n, int32_t B, float beta, const float *u, uint64_t seed,
                   uint64_t offset, int64_t *ids, float *weights, uint64_t *advance, void *stream);
int mal_per_update_check(int32_t B, int32_t T, int32_t n_q, float alpha, float eps);
int mal_per_update(const float *td, const float *mask, int32_t B, int32_t T, int32_t n_q, const int64_t *ids,
                   float alpha, float eps, float *priorities, int64_t capacity, float *max_priority, void *stream);

/* EpisodeBatch.max_t_filled, episode_batch.py:240-242: out[0] = max_b sum_t filled[b,t]. */
int mal_max_t_filled(const int64_t *filled, int64_t sb, int64_t st, int32_t B, int32_t TT, int32_t *out,
                     void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MAL_B200_H */
