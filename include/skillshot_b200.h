/*
 * skillshot_b200.h -- C ABI of libskillshot_b200.so (sm_100a).
 *
 * The reference (adrientremblay/Skillshot_Learning) has no FFI layer: its
 * boundary is the Python object surface of SkillshotGame / Player / Projectile
 * and SkillshotLearner.  The Python facade in skillshot_learning_b200/ keeps
 * that surface and binds these entry points with ctypes; each entry point names
 * the reference code it replaces (paths relative to the reference repo root).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller (PyTorch tensors in
 *    the facade) unless the name ends in _host; the library never allocates or
 *    frees caller memory and keeps no global state;
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *    the call returns without synchronising;
 *  - return value: 0 = success, SS_ERR_* (< 0) otherwise; nothing throws;
 *  - player index p is 0 or 1 (reference ids 1 and 2).
 */
#ifndef SKILLSHOT_B200_H
#define SKILLSHOT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SS_OK 0
#define SS_ERR_INVALID_ARG (-1)
#define SS_ERR_CUDA (-2)

/* ---- game state in HBM --------------------------------------------------
 * Structure of arrays, four 16-byte planes, plane k of env i at
 * state + (k * n_envs + i) * 16:
 *   plane 0  double2 { Player1.rotation, Player2.rotation }          (Player.py:21)
 *   plane 1  double2 { P1.projectile.rotation, P2.projectile.rotation } (Projectile.py:14)
 *   plane 2  int4    { player xy packed u8 (p1x | p1y<<8 | p2x<<16 | p2y<<24),
 *                      projectile xy packed u8 (same order),
 *                      P1.projectile.cooldown_current, P2...cooldown_current }
 *   plane 3  int4    { P1.projectile.age, P2.projectile.age, SkillshotGame.ticks,
 *                      flags: bit0/1 projectile.valid, bit2 game_live, bits 4-5 winner_id }
 * 64 bytes per env (the reference-natural widths of SURVEY.md 8(d) are 88). */
#define SS_STATE_BYTES_PER_ENV 64
#define SS_NUM_FEATURES 18   /* per-player keys of get_state, SkillshotGame.py:145-162 */
#define SS_NUM_OBS 12        /* prepare_states, SkillshotLearner.py:525-539 */

/* reward_mode */
#define SS_REWARD_NONE 0
#define SS_REWARD_LOOKING 1   /* calculate_rewards_looking, SkillshotLearner.py:575-588 */
#define SS_REWARD_TERMINAL 2  /* +1 / -1 / 0, readme.md:10 (no reference code) */
#define SS_REWARD_SIMPLE 3    /* calculate_rewards_simple, SkillshotLearner.py:590-603 */

/* reset_mode */
#define SS_RESET_FIXED 0      /* P1 [50,50], P2 [200,200], SkillshotGame.py:17-18 */
#define SS_RESET_RANDOM 1     /* uniform ints in [25,225), SkillshotGame.py:15; Philox4x32-10 */
#define SS_RESET_GIVEN 2      /* caller-supplied positions */

/* flags of ss_env_step */
#define SS_STEP_OBS_EVERY_TICK 1  /* obs_out is [n_ticks][n][2][12] instead of last tick only */
#define SS_STEP_EPISODE_STATS 2   /* `status` is the head of a block {uint32 status, uint32 pad, uint64 stats[SS_EPISODE_STATS]}:
                                   * every game that ENDS in this call is counted there (the per-episode ticks / winner log of
                                   * SkillshotLearner.py:164-180, 365-366, reduced on the device) */
/* stats[]: 0 episodes, 1 ended by a hit on player 1 (winner_id 1), 2 by a hit on player 2, 3 by the tick limit,
 * 4 sum of the episodes' tick counts, 5..7 reserved, 8..71 histogram of the tick counts in 64 bins of
 * ceil(tick_limit / 64) ticks (32 ticks when tick_limit <= 0; the last bin is open) */
#define SS_EPISODE_STATS 72

/* status bits OR-ed into *status by the kernels */
#define SS_STATUS_NAN 1       /* where the reference raises ValueError: int(round(nan)), Player.py:63 */
#define SS_STATUS_PEER_TIMEOUT 2   /* ss_peer_adam_tf gave up waiting for a peer's gradient */
#define SS_STATUS_ROLLOUT_TIMEOUT 4   /* ss_env_step_tiles gave up waiting for the actor forward kernel's actions */
#define SS_STATUS_SEAT_RANGE 8   /* ss_env_step_seated met a seat-table row outside [0, n_rows) (that env was not stepped) */

/* ops of ss_env_apply: the single-object methods of the reference */
#define SS_OP_MOVE_DIRECTION_FLOAT 0  /* Player.move_direction_float(value), Player.py:57-68 */
#define SS_OP_MOVE_LOOK_FLOAT 1       /* Player.move_look_float(value),     Player.py:33-39 */
#define SS_OP_SHOOT 2                 /* Player.move_shoot_projectile(),    Player.py:78-89 */
#define SS_OP_MOVE_FORWARDS 3         /* Player.move_forwards(),            Player.py:41-47 */
#define SS_OP_MOVE_BACKWARDS 4        /* Player.move_backwards(),           Player.py:49-55 */
#define SS_OP_LOOK_LEFT 5             /* Player.move_look_left(),           Player.py:27-28 */
#define SS_OP_LOOK_RIGHT 6            /* Player.move_look_right(),          Player.py:30-31 */
#define SS_OP_GAME_TICK 7             /* SkillshotGame.game_tick(),         SkillshotGame.py:115-122 */

int ss_version(void);

/* Bytes of `state` for n_envs games. */
int64_t ss_state_bytes(int64_t n_envs);

/* SkillshotGame.__init__ / game_reset (SkillshotGame.py:10-25, 168-169) for
 * every env whose mask byte is non-zero (mask == NULL: all).
 *   reset_mode SS_RESET_GIVEN reads positions int32 [n_envs][4] = p1x,p1y,p2x,p2y;
 *   SS_RESET_RANDOM draws them from Philox4x32-10(key = seed, counter = (env, counter)). */
int ss_env_reset(void *state, int64_t n_envs, const uint8_t *mask, int reset_mode,
                 const int32_t *positions, uint64_t seed, uint64_t counter, void *stream);

/* One or more ticks of the model_train inner loop for every env
 * (SkillshotLearner.py:304-315): both players act from the pre-tick state --
 * do_actions = move_direction_float, move_look_float, move_shoot_projectile
 * (SkillshotLearner.py:206-213), P1 then P2 -- then SkillshotGame.game_tick
 * (projectile advance, hit test, winner), then reward of the post-tick state
 * and the 12-float observation of each player (get_state + prepare_states).
 *
 *   actions     float32 [n_ticks][n_envs][2][2]   (player, (move, look))
 *   obs_out     float32 [n_envs][2][12] of the last tick (or [n_ticks]... with
 *               SS_STEP_OBS_EVERY_TICK); NULL = not computed
 *   reward_out  float32 [n_ticks][n_envs][2]; NULL or reward_mode 0 = not written
 *   done_out    uint8   [n_ticks][n_envs]  1 when the game ended (hit) or
 *               ticks >= tick_limit after the tick (tick_limit <= 0: no limit); NULL ok
 *   winner_out  uint8   [n_ticks][n_envs]  winner_id after the tick (the id of the
 *               player that was hit, SkillshotGame.py:77); NULL ok
 *   auto_reset  non-zero: a done env is reset (reset_mode FIXED or RANDOM) after
 *               its reward/done/winner are written; its obs is the post-reset one
 *   speeds      NULL (reference constants) or per-env constants, two 16-byte planes:
 *               plane 0 double2 {Player.speed_move, Player.speed_look},
 *               plane 1 {double Projectile.speed_move, int64 cooldown_max}
 *   status      NULL or uint32[1], SS_STATUS_* bits are OR-ed in (a larger block with SS_STEP_EPISODE_STATS)
 */
int ss_env_step(void *state, int64_t n_envs, const float *actions, float *obs_out,
                float *reward_out, uint8_t *done_out, uint8_t *winner_out,
                int n_ticks, int reward_mode, int64_t tick_limit, int auto_reset,
                int reset_mode, uint64_t seed, uint64_t counter, const void *speeds,
                uint32_t *status, int flags, void *stream);

/* ss_env_step with two extra outputs, so that a rollout can write its transitions straight into the
 * replay ring instead of copying them there afterwards (one tick per call when obs_out2 is given):
 *   obs_out2       second copy of the observation, float32 [n_envs][2][12] (the ring's NEXT segment:
 *                  the next tick's "obs" rows are this tick's "next_obs" rows), or NULL
 *   done_rows_out  the TERMINAL flag once per player row, uint8 [n_envs][2], or NULL: 1 when the game ended by a hit
 *                  (winner_id != 0), 0 otherwise -- a tick-limit restart is a truncation, not a termination, and must not
 *                  zero the TD bootstrap of r + gamma (1 - done) Q' (the reference itself has gamma = 0) */
int ss_env_step_ring(void *state, int64_t n_envs, const float *actions, float *obs_out, float *obs_out2,
                     float *reward_out, uint8_t *done_out, uint8_t *done_rows_out, uint8_t *winner_out,
                     int n_ticks, int reward_mode, int64_t tick_limit, int auto_reset,
                     int reset_mode, uint64_t seed, uint64_t counter, const void *speeds,
                     uint32_t *status, int flags, void *stream);

/* The physics-only step (reference speed constants, terminal +1 / -1 / 0 reward) with its three per-tick outputs packed
 * into ONE byte per env: packed_out uint8 [n_ticks][n_envs] = done | winner_id << 1 | hit << 3, where `hit` says that the
 * game ended by a hit on this very tick -- the tick on which the terminal reward is paid: reward of player p =
 * hit ? (winner_id - 1 == p ? -1 : +1) : 0.  Same trajectory, bit for bit, as ss_env_step with SS_REWARD_TERMINAL; built for
 * callers with HOST buffers, whose device-to-host traffic drops from 10 bytes per env-step to 1.
 * Requires 2 n_envs (n_ticks + 2) < 2^31. */
int ss_env_step_packed(void *state, int64_t n_envs, const float *actions, uint8_t *packed_out, int n_ticks,
                       int64_t tick_limit, int auto_reset, int reset_mode, uint64_t seed, uint64_t counter,
                       uint32_t *status, void *stream);

/* SkillshotGame.get_state (SkillshotGame.py:136-166) + prepare_states
 * (SkillshotLearner.py:512-543) in float64, formulas evaluated as written.
 *   feat_out    float64 [n_envs][2][18] in the dict's key order, or NULL
 *   obs_out     float64 [n_envs][2][12], or NULL
 *   general_out int32   [n_envs][3] = game_live, ticks, game_winner, or NULL */
int ss_env_features(const void *state, int64_t n_envs, double *feat_out, double *obs_out,
                    int32_t *general_out, const void *speeds, void *stream);

/* Unpack / pack `count` envs starting at `first` to natural-width arrays:
 *   ints  int32 [count][17] = px1,px2, py1,py2, qx1,qx2, qy1,qy2, cd1,cd2,
 *                             age1,age2, valid1,valid2, ticks, live, winner
 *   rots  float64 [count][4] = prot1, prot2, qrot1, qrot2                     */
#define SS_EXPORT_INTS 17
int ss_env_export(const void *state, int64_t n_envs, int64_t first, int64_t count,
                  int32_t *ints, double *rots, void *stream);
int ss_env_import(void *state, int64_t n_envs, int64_t first, int64_t count,
                  const int32_t *ints, const double *rots, void *stream);

/* One reference method call on one env (the object-style surface used by
 * skillshot_playable.py:51-64 and by do_actions). */
int ss_env_apply(void *state, int64_t n_envs, int64_t env, int player, int op, double value,
                 const void *speeds, uint32_t *status, void *stream);

/* ==== learner path =========================================================
 * The actor and critic of SkillshotLearner.model_define_actor / _critic
 * (SkillshotLearner.py:70-121).  A network's parameters are ONE flat float32
 * vector in Keras get_weights() order, Dense kernels stored [in][out]:
 *   actor   W1[12][256] b1[256] W2[256][128] b2[128] W3[128][2] b3[2]     36,482
 *   critic  W1[12][256] b1[256] W2[258][128] b2[128] W3[128][1] b3[1]     36,609
 * (critic W2 rows 0..255 take the dropped-out hidden layer, rows 256..257 the
 * action: concatenate([layer_model, actor_input]), SkillshotLearner.py:106).
 * Gradients, Adam moments and target networks use the same layout, so one
 * all-reduce over a flat buffer is the only exchange step of a multi-GPU update.
 * All matrices of samples are row-major float32: obs [n][12], act [n][2].
 * Parameter vectors must be 16-byte aligned. */
#define SS_DIM_STATE 12
#define SS_DIM_ACTION 2
#define SS_HIDDEN1 256
#define SS_HIDDEN2 128
#define SS_ACTOR_PARAMS 36482
#define SS_CRITIC_PARAMS 36609
#define SS_LEARNER_MAX_PARTS 512   /* most CTAs a gradient kernel will use */

/* Bytes of scratch the gradient entry points need (per-CTA gradient slices). */
int64_t ss_learner_workspace_bytes(void);

/* model_act / model_act_action_noise / model_act_param_noise
 * (SkillshotLearner.py:215-281) for n observations, without the env side effects
 * (do_actions is ss_env_step / ss_env_apply):  act_out[n][2] = actor(obs).
 *   param_noise_sd > 0: the actor is evaluated with w + w * N(0, sd) on all six
 *     arrays (SkillshotLearner.py:260-265); one draw is shared by `noise_group`
 *     consecutive rows (1 = the reference's fresh draw per call), drawn from
 *     Philox4x32-10(seed; parameter index, group index, counter);
 *   action_noise_sd > 0: act_out += N(0, sd)  (SkillshotLearner.py:238).
 * float32 arithmetic throughout (the exact path). */
int ss_actor_forward(const float *actor_params, const float *obs, float *act_out, int64_t n,
                     float param_noise_sd, int64_t noise_group, float action_noise_sd,
                     uint64_t seed, uint64_t counter, void *stream);

/* The same through the tensor cores: bf16 operands (observations split into a
 * bf16 high and low part so no input precision is lost), fp32 accumulation in
 * tensor memory, tcgen05.mma; the 128 -> 2 output layer and tanh in fp32.
 * `noise_group` must be a multiple of 128 when param_noise_sd > 0.  For the large
 * rollout batches (BASELINE.json configs 3-4); results agree with
 * ss_actor_forward to bf16 weight rounding (about 1e-2 absolute on the action). */
int ss_actor_forward_tc(const float *actor_params, const float *obs, float *act_out, int64_t n,
                        float param_noise_sd, int64_t noise_group, float action_noise_sd,
                        uint64_t seed, uint64_t counter, void *stream);

/* q = critic([obs, act]) on the tensor cores (Dropout off), any of:
 *   q_out[n]; neg_dq_da_out[n][2] = -dQ/da (the output_gradients of SkillshotLearner.py:410);
 *   y_out[n] = reward + gamma * (1 - done) * q  (the TD target when the parameters are the target critic's). */
int ss_critic_forward_tc(const float *critic_params, const float *obs, const float *act, int64_t n,
                         float *q_out, float *neg_dq_da_out, const float *reward, const uint8_t *done,
                         float gamma, float *y_out, void *stream);

/* Tensor-core versions of ss_critic_grad / ss_actor_grad / ss_ddpg_targets for large batches: the
 * layer GEMMs of the forward AND backward pass run as tcgen05.mma on bf16 operands with fp32
 * accumulation, the weight-gradient sums stay in tensor memory across the batch.  Same arguments
 * and outputs; gradients agree with the float32 entry points to about 1e-3 of their scale.
 * `workspace` must hold ss_learner_workspace_bytes() + 32 * n bytes. */
int ss_critic_grad_tc(const float *critic_params, const float *obs, const float *act, const float *target,
                      const uint8_t *dropout_keep, float dropout_rate, uint64_t seed, uint64_t counter,
                      int64_t n, int64_t n_global, int64_t row_offset, float *grad_out, float *sse_out,
                      void *workspace, int64_t workspace_bytes, void *stream);
int ss_actor_grad_tc(const float *actor_params, const float *critic_params, const float *obs, int64_t n,
                     float *grad_out, float *q_sum_out, void *workspace, int64_t workspace_bytes,
                     void *stream);
/* The same in two stages, for callers that have other work to put between them (ss_ddpg_update overlaps stage 1 with the
 * critic's gradient exchange): stage 1 = a = actor(s) only, into the scratch area of `workspace`; stage 2 = the rest,
 * reading those actions; stage 0 = ss_actor_grad_tc.  Same workspace and n in both stages. */
int ss_actor_grad_tc_staged(const float *actor_params, const float *critic_params, const float *obs, int64_t n,
                            float *grad_out, float *q_sum_out, void *workspace, int64_t workspace_bytes, int stage,
                            void *stream);
int ss_ddpg_targets_tc(const float *target_actor_params, const float *target_critic_params,
                       const float *reward, const float *next_obs, const uint8_t *done, float gamma,
                       float *y_out, int64_t n, void *workspace, int64_t workspace_bytes, void *stream);

/* out[p] = params[p] + params[p] * (sd * eps_p): the perturbed vector
 * ss_actor_forward uses for noise group `group` (introspection and tests). */
int ss_param_noise(const float *params, float *out, int64_t n_params, float sd, uint64_t seed,
                   uint64_t group, uint64_t counter, void *stream);

/* q_out[n] = critic([obs, act]), Dropout off (a model call / predict). */
int ss_critic_forward(const float *critic_params, const float *obs, const float *act, float *q_out,
                      int64_t n, void *stream);

/* y[n] = reward + gamma * (1 - done) * Q'(next_obs, mu'(next_obs)) with the target
 * networks.  The reference regresses the critic on the immediate reward
 * (SkillshotLearner.py:434): that is gamma = 0.  done may be NULL. */
int ss_ddpg_targets(const float *target_actor_params, const float *target_critic_params,
                    const float *reward, const float *next_obs, const uint8_t *done, float gamma,
                    float *y_out, int64_t n, void *stream);

/* Gradient of the critic's Keras "mse" loss for one batch (model_critic.fit,
 * SkillshotLearner.py:118, 434):  grad_out[36609] = d/dphi sum_i (q_i - target_i)^2 / n_global,
 * sse_out[1] = sum_i (q_i - target_i)^2  (may be NULL).
 *   dropout_rate  Dropout(0.2) of SkillshotLearner.py:105 as applied during fit; 0 = off.
 *   dropout_keep  NULL: mask from Philox(seed; row_offset + row, unit / 8, counter), 16 bits per unit;
 *                 else uint8 [n][256], 1 = keep (parity tests inject Keras' choice).
 *   n_global      divisor of the mean when n is one GPU's shard of a batch (<= 0: n).
 * The gradient is summed in a fixed order: bit-identical from run to run. */
int ss_critic_grad(const float *critic_params, const float *obs, const float *act, const float *target,
                   const uint8_t *dropout_keep, float dropout_rate, uint64_t seed, uint64_t counter,
                   int64_t n, int64_t n_global, int64_t row_offset, float *grad_out, float *sse_out,
                   void *workspace, int64_t workspace_bytes, void *stream);

/* model_actor_fit_step (SkillshotLearner.py:386-417) up to the optimiser:
 * a = actor(obs); q = critic([obs, a]) with Dropout off;
 * grad_out[36482] = d a / d theta contracted with -dq/da, summed over the batch
 * (tape.gradient of a non-scalar sums); q_sum_out[1] = sum q (may be NULL). */
int ss_actor_grad(const float *actor_params, const float *critic_params, const float *obs, int64_t n,
                  float *grad_out, float *q_sum_out, void *workspace, int64_t workspace_bytes,
                  void *stream);

/* tf.keras.optimizers.Adam.apply_gradients (SkillshotLearner.py:68, 118, 417), step t >= 1:
 *   g = grads * grad_scale; m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2;
 *   params -= lr * sqrt(1 - b2^t) / (1 - b1^t) * m / (sqrt(v) + eps)     (Keras: eps = 1e-7)
 * and, when target_params != NULL, the DDPG soft update
 *   target = tau * params + (1 - tau) * target                          (tau = 1: copy). */
int ss_adam_tf(float *params, const float *grads, float *m, float *v, float *target_params, int64_t n,
               int64_t step, float lr, float beta1, float beta2, float eps, float tau, float grad_scale,
               void *stream);

/* The fixed-order sum of the per-CTA gradient slices a gradient entry point left in `workspace` (called with
 * grad_out == NULL; `parts` = its return value) and ss_adam_tf on the result, in one kernel: the single-GPU form of
 * ss_peer_reduce_push + ss_peer_adam_tf.  aux_out[0] (may be NULL) = sum of the slices' extra slot (squared error /
 * Q sum); grad_out (may be NULL) receives the summed gradient. */
int ss_reduce_adam_tf(const void *workspace, int parts, int n_params, float *aux_out, float *grad_out, float *params,
                      float *m, float *v, float *target_params, int64_t step, float lr, float beta1, float beta2,
                      float eps, float tau, float grad_scale, void *stream);

/* n_ticks iterations of the rollout loop of model_train (SkillshotLearner.py:302-315) for n_envs games,
 * enqueued back to back from one host call: actor forward on both players' observations (2 n_envs rows;
 * tensor_cores != 0: ss_actor_forward_tc) -> ss_env_step with auto-reset -> ss_replay_push (skipped when
 * ring_obs == NULL).  obs_a / obs_b are a double buffer [n_envs][2][12]: obs_a holds the current
 * observation on entry, and after the call it is in obs_a if n_ticks is even, in obs_b otherwise (but see below).
 * actions [n_envs][2][2], reward [n_envs][2], done / winner [n_envs] hold the last tick's values on return.
 * Tick t uses Philox counters env_counter + t and noise_counter + t; ring rows advance by 2 n_envs per tick.
 * The ring's done flag is the TERMINAL flag (a hit, winner != 0; see ss_env_step_ring), so `winner` is required with a ring.
 * When capacity and write_pos are multiples of 2 n_envs (and the ring has at least two such segments, or n_ticks == 1)
 * the transitions are produced IN the ring (the actor
 * reads its observations from and writes its actions to the ring's rows, ss_env_step_ring writes reward, done
 * and both copies of the next observation there): no copy kernel runs, and the current observation is left
 * in obs_a whatever the parity of n_ticks.  Otherwise ss_replay_push copies each tick's rows.
 * step_flags: SS_STEP_EPISODE_STATS or 0, passed to every env step of the loop. */
int ss_selfplay_rollout(void *env_state, int64_t n_envs, const float *actor_params, float *obs_a, float *obs_b,
                        float *actions, float *reward, uint8_t *done, uint8_t *winner,
                        float *ring_obs, float *ring_act, float *ring_reward, float *ring_next_obs,
                        uint8_t *ring_done, int64_t capacity, int64_t write_pos, int n_ticks,
                        float param_noise_sd, int64_t noise_group, float action_noise_sd, int tensor_cores,
                        int reward_mode, int64_t tick_limit, int reset_mode, uint64_t env_seed,
                        uint64_t env_counter, uint64_t noise_seed, uint64_t noise_counter, const void *speeds,
                        uint32_t *status, int step_flags, void *stream);

/* ss_selfplay_rollout with the env step OVERLAPPED with the actor forward (tensor-core path, in-place ring form, reference
 * speeds, reward none / looking / terminal; anything else falls through to ss_selfplay_rollout): tile_ready = int32
 * [2 n_envs / 128 + noise_group / 128 + 1] zeroed once by the caller and left zero by every call, stream2 = a second
 * stream of the same device with HIGHER priority than `stream` (cudaStreamCreateWithPriority): per tick the forward kernel
 * runs on stream2 and ss_env_step_tiles on `stream` beside it (the forward kernel's CTAs must be placed first: it needs
 * whole SMs, the one-warp env CTAs fit in what it leaves); events order the two, and `stream` has caught up with stream2
 * when the call returns.  Same results, bit for bit. */
int ss_selfplay_rollout2(void *env_state, int64_t n_envs, const float *actor_params, float *obs_a, float *obs_b,
                         float *actions, float *reward, uint8_t *done, uint8_t *winner,
                         float *ring_obs, float *ring_act, float *ring_reward, float *ring_next_obs,
                         uint8_t *ring_done, int64_t capacity, int64_t write_pos, int n_ticks,
                         float param_noise_sd, int64_t noise_group, float action_noise_sd, int tensor_cores,
                         int reward_mode, int64_t tick_limit, int reset_mode, uint64_t env_seed,
                         uint64_t env_counter, uint64_t noise_seed, uint64_t noise_counter, const void *speeds,
                         uint32_t *status, int step_flags, int *tile_ready, void *stream2, void *stream);

/* One rollout tick as ONE kernel (tensor-core path): ss_actor_forward_tc on the players' observations (n_rows = 2 x envs,
 * row = 2 env + player) and, in its output stage, the env step of those players -- do_actions, game_tick, reward of the
 * post-tick state, auto-reset, next observation (SkillshotLearner.py:304-315) -- by the lane that has just computed the
 * player's action.  Same results, bit for bit, as ss_actor_forward_tc followed by ss_env_step_ring with auto_reset = 1:
 * act_out [n_rows][2]; obs_next (and obs_next2 if not NULL) [n_rows][12]; reward_out [n_rows]; done_out / winner_out
 * [n_rows / 2]; done_rows_out [n_rows] (the hit flag per row).  reward_mode none / looking / terminal, reference speeds.
 * ss_selfplay_rollout uses it for its in-place ring form. */
int ss_actor_forward_step_tc(const float *actor_params, const float *obs, float *act_out, int64_t n_rows,
                             float param_noise_sd, int64_t noise_group, float action_noise_sd, uint64_t seed,
                             uint64_t counter, void *env_state, float *obs_next, float *obs_next2, float *reward_out,
                             uint8_t *done_out, uint8_t *done_rows_out, uint8_t *winner_out, int reward_mode,
                             int64_t tick_limit, int reset_mode, uint64_t env_seed, uint64_t env_counter,
                             uint32_t *status, int flags, void *stream);

/* The two halves of the OVERLAPPED rollout tick (ss_selfplay_rollout with a second stream): ss_actor_forward_tc_signal is
 * ss_actor_forward_tc that also increments tile_ready[row / 128] (int32, zero-initialised by the caller) once per output warp
 * -- four times per 128-row tile -- when that tile's actions are in global memory, and reports its CTA count and tile count;
 * ss_env_step_tiles, enqueued on ANOTHER stream, is the env step with observations of ss_env_step_ring (one tick,
 * auto_reset = 1, reference speeds, reward none / looking / terminal) that walks the tiles in the order the forward
 * kernel completes them, waits for each tile's four arrivals, plays its 128 players' tick and takes the arrivals away
 * again.  It uses no shared memory and at most 64 registers, so it runs beside the forward kernel on the same SMs: the env
 * step ends a few microseconds after the forward does.  A tile that never arrives raises SS_STATUS_ROLLOUT_TIMEOUT. */
int ss_actor_forward_tc_signal(const float *actor_params, const float *obs, float *act_out, int64_t n,
                               float param_noise_sd, int64_t noise_group, float action_noise_sd,
                               uint64_t seed, uint64_t counter, int *tile_ready, int *grid_out, int64_t *units_out,
                               void *stream);
int ss_env_step_tiles(void *state, int64_t n_envs, const float *actions, float *obs_out, float *obs_out2,
                      float *reward_out, uint8_t *done_out, uint8_t *done_rows_out, uint8_t *winner_out,
                      int reward_mode, int64_t tick_limit, int reset_mode, uint64_t seed, uint64_t counter,
                      uint32_t *status, int flags, int *tile_ready, int64_t units, int grid_fwd, void *stream);

/* ---- frame-stacked ("planning") actor: readme.md:18-20, BASELINE.json configs[4]; no reference code ----
 * The actor reads the last `frames` observations of a player: first layer 12 * frames -> 256, the rest as
 * model_define_actor (SkillshotLearner.py:70-96); frames = 1 is the reference actor.  Parameters are one flat
 * vector [W1[12 frames][256] b1[256] W2[256][128] b2[128] W3[128][2] b3[2]] (ss_actor_frames_params floats).
 * The history is a ring per row, stack[n_rows][frames][12]; slot head % frames holds the newest frame, the
 * network input is ordered oldest -> newest.
 *   ss_obs_stack_push        newest observation -> slot head % frames; a row whose `done` flag is set (one flag
 *                            per done_div rows, NULL = none) gets it in every slot (the game restarted)
 *   ss_param_noise_groups    out[g][p] = params[p] + params[p] * sd * eps(p, g): one perturbed vector per noise group
 *                            (SkillshotLearner.py:260-265), g < n_groups, rows of `stride` floats (stride % 4 == 0);
 *                            the normals come from the hardware log / sincos units: within ~3e-6 of ss_param_noise's
 *   ss_actor_forward_frames  act_out[n][2]; param_stride = 0: every row uses `params`; else row i uses
 *                            params + (i / noise_group) * param_stride.  The exact float32 path.
 * Tensor-core path (tcgen05.mma: layer 1 in fp16, layer 2 in bf16, fp32 accumulation, the output layer and
 * tanh in fp32; agrees with the float32 path to about 1e-2 on the action).  Its history ring is a separate
 * buffer of ss_obs_stack_tc_bytes(n_rows, frames) bytes, zero-initialised by the caller: fp16 tiles of 128 rows
 * already in the tensor core's operand layout [tile][K / 8][128][8] with K = 12 frames + 2 padded to 16, columns
 * in ring-slot order (column 12 slot + j), a constant {1, 1} pair behind them.
 *   ss_obs_stack_push_tc        as ss_obs_stack_push, into that buffer (observations rounded to fp16)
 *   ss_actor_forward_frames_tc  as ss_actor_forward_frames, from that buffer.  noise_group must be a multiple
 *                            of 128 when param_stride > 0; `workspace` (16-byte aligned) holds
 *                            ss_actor_frames_tc_workspace_bytes(n, noise_group) bytes: hidden layer 1 of every
 *                            128-row tile between the two kernels of the call */
#define SS_MAX_FRAMES 20
int64_t ss_actor_frames_params(int frames);
int ss_obs_stack_push(float *stack, int64_t n_rows, int frames, int64_t head, const float *obs, const uint8_t *done,
                      int done_div, void *stream);
int ss_param_noise_groups(const float *params, float *out, int64_t n_params, int64_t n_groups, int64_t stride, float sd,
                          uint64_t seed, uint64_t counter, void *stream);
int ss_actor_forward_frames(const float *params, int64_t param_stride, int64_t noise_group, const float *stack, int frames,
                            int64_t head, float *act_out, int64_t n, void *stream);
int64_t ss_actor_frames_tc_workspace_bytes(int64_t n, int64_t noise_group);
int64_t ss_obs_stack_tc_bytes(int64_t n_rows, int frames);
int ss_obs_stack_push_tc(void *stack_tc, int64_t n_rows, int frames, int64_t head, const float *obs, const uint8_t *done,
                         int done_div, void *stream);
int ss_actor_forward_frames_tc(const float *params, int64_t param_stride, int64_t noise_group, const void *stack_tc, int frames,
                               int64_t head, float *act_out, int64_t n, void *workspace, int64_t workspace_bytes,
                               void *stream);

/* ---- the learner of the frame-stacked networks (readme.md:18-20; no reference code, parity unpinned) ----
 * The update of SkillshotLearner.py:386-443 (critic fit step, model_actor_fit_step) for an actor and a critic whose first
 * Dense layer reads 12 * frames inputs: actor as above, critic [W1[12 frames][256] b1 W2[258][128] b2 W3[128][1] b3]
 * (ss_critic_frames_params floats).  Observations are dense float32 rows [n][12 frames], oldest frame first
 * (ss_obs_stack_ordered writes them from the history ring).  The exact float32 kernels of the 12-input entry points with
 * a run-time input width: frames = 1 IS ss_critic_forward / ss_ddpg_targets / ss_critic_grad / ss_actor_grad, argument
 * for argument.  Workspace: ss_learner_frames_workspace_bytes(frames) bytes hold SS_LEARNER_MAX_PARTS gradient slices
 * (fewer bytes = fewer CTAs).  The replay ring of these transitions is ss_replay_push_frames / ss_replay_sample_frames:
 * ss_replay_push / ss_replay_sample with observation rows of 12 * frames floats. */
int64_t ss_critic_frames_params(int frames);
int64_t ss_learner_frames_workspace_bytes(int frames);
int ss_obs_stack_ordered(const float *stack, int64_t n_rows, int frames, int64_t head, float *out, void *stream);
int ss_critic_forward_frames(const float *critic_params, int frames, const float *obs, const float *act, float *q_out,
                             int64_t n, void *stream);
int ss_ddpg_targets_frames(const float *target_actor_params, const float *target_critic_params, int frames,
                           const float *reward, const float *next_obs, const uint8_t *done, float gamma, float *y_out,
                           int64_t n, void *stream);
int ss_critic_grad_frames(const float *critic_params, int frames, const float *obs, const float *act, const float *target,
                          const uint8_t *dropout_keep, float dropout_rate, uint64_t seed, uint64_t counter,
                          int64_t n, int64_t n_global, int64_t row_offset, float *grad_out, float *sse_out,
                          void *workspace, int64_t workspace_bytes, void *stream);
int ss_actor_grad_frames(const float *actor_params, const float *critic_params, int frames, const float *obs, int64_t n,
                         float *grad_out, float *q_sum_out, void *workspace, int64_t workspace_bytes, void *stream);
/* The same four calls on the tensor cores (tcgen05.mma), argument for argument, with a workspace of
 * ss_learner_frames_tc_workspace_bytes(frames, n) bytes (16-byte aligned) that holds the gradient slices and the tiles
 * passed between the kernels of a call.  Precision: observations fp16 in the forward layer 1 and bf16 high + low halves
 * in dW1; W1 fp16; hidden activations, dz1 / dz2 and W2 bf16; biases and the critic's action as high + low bf16 pairs;
 * fp32 accumulation; the output layer, loss and tanh in fp32.  Results agree with the float32 path to about 2e-2 of
 * their scale.  The gradient calls leave slices of n_params + 1 floats and return their number when grad_out is NULL,
 * like ss_critic_grad_tc / ss_actor_grad_tc.  Dropout keep bits are those of ss_critic_grad_frames.  neg_dq_da_out
 * [n][2] (may be NULL) receives -dQ/da. */
int64_t ss_learner_frames_tc_workspace_bytes(int frames, int64_t n);
int ss_critic_forward_frames_tc(const float *critic_params, int frames, const float *obs, const float *act, float *q_out,
                                float *neg_dq_da_out, int64_t n, void *workspace, int64_t workspace_bytes, void *stream);
int ss_ddpg_targets_frames_tc(const float *target_actor_params, const float *target_critic_params, int frames,
                              const float *reward, const float *next_obs, const uint8_t *done, float gamma, float *y_out,
                              int64_t n, void *workspace, int64_t workspace_bytes, void *stream);
int ss_critic_grad_frames_tc(const float *critic_params, int frames, const float *obs, const float *act, const float *target,
                             const uint8_t *dropout_keep, float dropout_rate, uint64_t seed, uint64_t counter,
                             int64_t n, int64_t n_global, int64_t row_offset, float *grad_out, float *sse_out,
                             void *workspace, int64_t workspace_bytes, void *stream);
int ss_actor_grad_frames_tc(const float *actor_params, const float *critic_params, int frames, const float *obs, int64_t n,
                            float *grad_out, float *q_sum_out, void *workspace, int64_t workspace_bytes, void *stream);

/* ---- TD3 target (twin critics, target policy smoothing; no reference code, DESIGN.md section 6.14) ----
 *   a~[i] = clamp(mu'(s'_i) + clamp(noise_sd * eps_i, -noise_clip, noise_clip), -1, 1)
 *   y_out[i] = reward[i] + gamma * (1 - done[i]) * min(Q1'(s'_i, a~[i]), Q2'(s'_i, a~[i]))
 * target_critic2_params NULL: the minimum is over Q1' alone.  eps_i: the first two of the four Box-Muller normals of
 * Philox4x32-10(seed; row_offset + i, (row_offset + i) >> 32, counter) with tag SS_TAG_TARGET_NOISE (the keying of the
 * action noise of ss_actor_forward, by the GLOBAL row as dropout is: a shard of a batch draws what the whole batch draws);
 * noise_sd == 0 draws nothing.  With target_critic2_params == NULL and noise_sd == 0 each entry point returns, bit for
 * bit, what its ss_ddpg_targets* counterpart returns.  Every argument is checked before anything is enqueued; a bad one
 * (NULL pointer, n <= 0, frames out of range, noise_sd < 0, noise_clip < 0, row_offset < 0, a misaligned parameter vector,
 * a short workspace) returns SS_ERR_INVALID_ARG.
 *   ss_td3_targets_frames     float32 CUDA cores, frames 1..SS_MAX_FRAMES (frames = 1: the 12-input networks).
 *                             The workspace is not used (may be NULL).
 *   ss_td3_targets_tc         tcgen05, the 12-input networks: ss_ddpg_targets_tc's forwards; workspace (16-byte aligned)
 *                             of at least SS_TD3_TC_WORKSPACE_BYTES(n) bytes (8 n rounded up to 16 is enough for one critic).
 *   ss_td3_targets_frames_tc  tcgen05, frames 2..SS_MAX_FRAMES: ss_ddpg_targets_frames_tc's forwards with its workspace,
 *                             ss_learner_frames_tc_workspace_bytes(frames, n). */
#define SS_TAG_TARGET_NOISE 5
#define SS_TD3_TC_WORKSPACE_BYTES(n) (((int64_t)(n) * 8 + 15) / 16 * 16 + 2 * (((int64_t)(n) * 4 + 15) / 16 * 16))
int ss_td3_targets_frames(const float *target_actor_params, const float *target_critic_params, const float *target_critic2_params,
                          int frames, const float *reward, const float *next_obs, const uint8_t *done, float gamma,
                          float noise_sd, float noise_clip, uint64_t seed, uint64_t counter, int64_t row_offset, float *y_out,
                          int64_t n, void *workspace, int64_t workspace_bytes, void *stream);
int ss_td3_targets_tc(const float *target_actor_params, const float *target_critic_params, const float *target_critic2_params,
                      const float *reward, const float *next_obs, const uint8_t *done, float gamma, float noise_sd, float noise_clip,
                      uint64_t seed, uint64_t counter, int64_t row_offset, float *y_out, int64_t n, void *workspace,
                      int64_t workspace_bytes, void *stream);
int ss_td3_targets_frames_tc(const float *target_actor_params, const float *target_critic_params, const float *target_critic2_params,
                             int frames, const float *reward, const float *next_obs, const uint8_t *done, float gamma, float noise_sd,
                             float noise_clip, uint64_t seed, uint64_t counter, int64_t row_offset, float *y_out, int64_t n,
                             void *workspace, int64_t workspace_bytes, void *stream);

int ss_replay_push_frames(float *ring_obs, float *ring_act, float *ring_reward, float *ring_next_obs, uint8_t *ring_done,
                          int64_t capacity, int64_t write_pos, int frames, const float *obs, const float *act,
                          const float *reward, const float *next_obs, const uint8_t *done, int done_div, int64_t n,
                          void *stream);
int ss_replay_sample_frames(const float *ring_obs, const float *ring_act, const float *ring_reward,
                            const float *ring_next_obs, const uint8_t *ring_done, int64_t capacity, int64_t size, int frames,
                            const int64_t *indices, uint64_t seed, uint64_t counter, int64_t batch,
                            float *obs, float *act, float *reward, float *next_obs, uint8_t *done, int64_t *indices_out,
                            void *stream);

/* ---- n-step rows of the replay ring (no reference code, DESIGN.md section 6.15) ----
 * A ring written one block of tick_rows rows per tick (2 n_envs for self-play, the learner's rows of a pool) holds the same
 * player's next transition after row r at row (r + tick_rows) mod capacity.  Row r is drawn uniformly from the eligible rows:
 * the runs [start, start + length) of ring positions in runs_host[2 n_runs] = {start_0, length_0, start_1, ...}, taken in
 * order; the draw is ss_replay_sample's Philox word x (tag kTagReplay, row b, counter) as j = (x * total) >> 32 with total
 * = the sum of the lengths, and j picks the j-th row of the runs.  With one run [0, size) the rows are ss_replay_sample's,
 * bit for bit.  The walk then visits r_t = (r + t tick_rows) mod capacity, t = 0 .. n_step - 1, and stops after the first
 * row whose done flag is set; k rows visited.
 *   obs, act, indices_out  row r's (indices_out may be NULL)
 *   reward                 sum over t < k of g_t reward[r_t] in float32, increasing t, each product and sum rounded
 *                          (no FMA); g_0 = 1, g_{t+1} = g_t * gamma in float32
 *   next_obs, done         row r_{k-1}'s
 *   steps_out              k (uint8, may be NULL)
 * The TD target is then reward + g_n (1 - done) Q'(next_obs, .) with g_n of the same recurrence: pass it as the gamma of
 * ss_ddpg_targets* / ss_td3_targets* / ss_ddpg_update.  Which rows are eligible (no walk passes the newest stored tick or a
 * break in the players' trajectories) is the caller's; the library checks only that every run lies inside the ring.
 * Every argument is checked before anything is enqueued: NULL pointers (but indices_out, steps_out), frames out of
 * 1..SS_MAX_FRAMES, n_step out of 1..SS_REPLAY_MAX_NSTEP, tick_rows < 1, n_step * tick_rows > capacity, n_runs out of
 * 1..SS_REPLAY_MAX_RUNS, a run with start < 0, length < 1 or past the capacity, a total of 2^32 rows or more, a gamma that
 * is not finite and observation pointers that are not 16-byte aligned return SS_ERR_INVALID_ARG. */
#define SS_REPLAY_MAX_RUNS 16
#define SS_REPLAY_MAX_NSTEP 32
int ss_replay_sample_nstep(const float *ring_obs, const float *ring_act, const float *ring_reward, const float *ring_next_obs,
                           const uint8_t *ring_done, int64_t capacity, int frames, int64_t tick_rows, int n_step, float gamma,
                           const int64_t *runs_host, int n_runs, uint64_t seed, uint64_t counter, int64_t batch, float *obs,
                           float *act, float *reward, float *next_obs, uint8_t *done, int64_t *indices_out, uint8_t *steps_out,
                           void *stream);

/* ---- prioritized replay (Schaul et al. 2016, proportional; no reference code, DESIGN.md section 6.16) ----
 * A prioritized ring keeps one float32 leaf per ring position, priority[capacity] = p^alpha, and a device scalar
 * priority_max (1.0 at the start).  Every row written gets the leaf priority_max (ss_replay_priority_fill); a priority update
 * sets leaf[idx_b] = powf(|delta_b| + eps, alpha) and raises priority_max to the largest leaf it wrote.
 *
 * ss_replay_sample_prioritized: ss_replay_sample_nstep's arguments (n_step = 1: one-step rows; pass one run [0, size) for
 * the rows ss_replay_sample draws from) and
 *   priority               the leaves (4-byte aligned)
 *   scratch                at least ss_replay_priority_scratch_bytes(capacity) bytes, 8-byte aligned (float64 prefix)
 *   beta                   importance-weight exponent in [0, 1]
 *   weights_out[batch]     w_b = (leaf_min / leaf[src_b])^beta in float64, rounded to float32; leaf_min is the smallest
 *                          non-zero eligible leaf, so every w is in (0, 1]
 * The eligible rows are those of the runs, in run order; eligible row j maps to its ring position as in
 * ss_replay_sample_nstep.  P[j] is the float64 inclusive prefix of their leaves, summed in a fixed order (bit-identical from
 * run to run) and total = P[last].  Row b of B draws the smallest j with P[j] > u_b, where
 *   u_b = ((double)b + x_b * 2^-32) / (double)B * total,   x_b = word b & 3 of Philox4x32-10 with tag SS_TAG_PRIORITY,
 *         keyed (b / 4, (b / 4) >> 32, counter) like ss_replay_sample's draw,
 * or, when u_b rounds up to total, the last eligible row with a non-zero leaf.  The row is then gathered (and walked for
 * n_step > 1) exactly as by ss_replay_sample_nstep.  (Every eligible leaf 0: row 0 of the runs, weight 1.)  The draw is
 * three launches: a block scan of the leaves, one block over the blocks' sums, and the search + gather.
 * ss_replay_priority_update: leaf[indices[b]] = powf(|td_abs[b]| + eps, alpha) for b < batch; when an index occurs more than
 * once, the largest b wins.  scratch: int32[capacity] (contents need not be set).  Indices outside [0, capacity) are skipped.
 * ss_replay_priority_fill: leaf[(pos + i) mod capacity] = *priority_max for i < n.
 * Every argument is checked before anything is enqueued: NULL pointers (but indices_out, steps_out), the ranges of
 * ss_replay_sample_nstep, a beta outside [0, 1], an alpha < 0, an eps <= 0, any of them not finite, runs holding more
 * rows than the ring, a short scratch and misaligned pointers return SS_ERR_INVALID_ARG. */
#define SS_TAG_PRIORITY 6
int64_t ss_replay_priority_scratch_bytes(int64_t capacity);
int ss_replay_sample_prioritized(const float *ring_obs, const float *ring_act, const float *ring_reward, const float *ring_next_obs,
                                 const uint8_t *ring_done, int64_t capacity, int frames, int64_t tick_rows, int n_step, float gamma,
                                 const int64_t *runs_host, int n_runs, uint64_t seed, uint64_t counter, int64_t batch, float *obs,
                                 float *act, float *reward, float *next_obs, uint8_t *done, int64_t *indices_out, uint8_t *steps_out,
                                 const float *priority, void *scratch, int64_t scratch_bytes, float beta, float *weights_out,
                                 void *stream);
int ss_replay_priority_update(float *priority, float *priority_max, int64_t capacity, const int64_t *indices, const float *td_abs,
                              int64_t batch, float alpha, float eps, int32_t *scratch, void *stream);
int ss_replay_priority_fill(float *priority, const float *priority_max, int64_t capacity, int64_t pos, int64_t n, void *stream);

/* ss_critic_grad_weighted: the critic gradient of the row-weighted loss (prioritized replay's importance weights):
 * d_b = (2 e_b / n_global) * row_weight[b], the weight multiplied last, so that row_weight = 1 gives the unweighted d bit
 * for bit; sse_out stays the unweighted sum of e_b^2.  td_abs_out[b] = |e_b| = |q_b - target_b| of the same forward
 * (with its dropout mask).  Either may be NULL (row_weight NULL: weight 1).  One entry point for the three families:
 *   tensor_cores = 0        float32 CUDA cores, frames 1..SS_MAX_FRAMES (ss_critic_grad_frames)
 *   tensor_cores, frames 1  tcgen05, 12 inputs (ss_critic_grad_tc, its workspace)
 *   tensor_cores, frames>1  tcgen05, frame-stacked (ss_critic_grad_frames_tc, ss_learner_frames_tc_workspace_bytes)
 * The other arguments, the return value and the checks are those of the family's unweighted entry point; row_weight and
 * td_abs_out must be 4-byte aligned. */
int ss_critic_grad_weighted(const float *critic_params, int frames, int tensor_cores, const float *obs, const float *act,
                            const float *target, const float *row_weight, float *td_abs_out, const uint8_t *dropout_keep,
                            float dropout_rate, uint64_t seed, uint64_t counter, int64_t n, int64_t n_global, int64_t row_offset,
                            float *grad_out, float *sse_out, void *workspace, int64_t workspace_bytes, void *stream);

/* ---- matches: two actors against each other (no reference code; the readme's "does the planning actor play better" question) ----
 * A match is n_envs games between policy A and policy B, ONE game per env (no auto-reset: every game starts at tick 0 and
 * is played to a hit or to tick_limit ticks, so no outcome is sampled by its length).  Seat map, split index 0 <= split <= n_envs:
 *   env j <  split: A is player 1, B is player 2
 *   env j >= split: B is player 1, A is player 2
 * The seats are not symmetric -- check_collision tests player 1 first and a double hit records id 1 (SkillshotGame.py:58-94)
 * -- so a fair match seats each policy in both.  The policies' inputs and outputs are POLICY-MAJOR, env j at row j of its half:
 *   obs float32 [2][n_envs][12]   half 0 = A's observations, half 1 = B's
 *   act float32 [2][n_envs][2]    the same layout for the actions
 * so each policy's forward reads one contiguous block of rows; only the env step knows the seat map.
 *
 *   ss_env_step_match     one tick of every env: each env's two actions are read from `act` through the seat map, both next
 *                         observations written to `obs_out` (policy-major).  No reward, no auto-reset; per-env speeds as for
 *                         ss_env_step; SS_STATUS_NAN as ss_env_step raises it.  A game still live with ticks >= tick_limit
 *                         (> 0) is NOT stepped (its observation is rewritten unchanged), so an outcome cannot change after the
 *                         limit however many ticks are enqueued.  For up to tick_limit ticks from a fresh reset the state and
 *                         the observations are bit-identical to ss_env_step(reward_mode NONE, auto_reset 0) under the seat
 *                         permutation.
 *   ss_actor_forward_groups_tc  ss_actor_forward_tc (no noise) with one parameter vector per group of rows: row i uses
 *                         params + (i / group_rows) * param_stride (param_stride % 4 == 0; 0 = one vector for all rows).
 *                         Each row's action is bit-identical to ss_actor_forward_tc run on its group's rows alone.
 *   ss_match_summary      out uint64 [SS_MATCH_STATS] = [2][8] from the state (ticks, live, winner), OVERWRITTEN: block 0 = the
 *                         envs where A is player 1 (j < split), block 1 = where A is player 2; per block
 *                         { games, A wins (B was hit), B wins (A was hit), draws (live, ticks >= tick_limit),
 *                           unfinished (live, ticks < tick_limit), sum of the ticks of the decided games, 0, 0 }.
 *                         winner_id is the id of the player that was HIT (SkillshotGame.py:77).  Exact integer counts. */
#define SS_MATCH_STATS 16
int ss_env_step_match(void *state, int64_t n_envs, int64_t split, const float *actions, float *obs_out, int64_t tick_limit,
                      const void *speeds, uint32_t *status, void *stream);
int ss_actor_forward_groups_tc(const float *params, int64_t param_stride, int64_t group_rows, const float *obs, float *act_out,
                               int64_t n, void *stream);
int ss_match_summary(const void *state, int64_t n_envs, int64_t split, int64_t tick_limit, uint64_t *out, void *stream);

/* n_ticks match ticks enqueued from one host call (as ss_selfplay_rollout does for self-play).  Per tick: the policies'
 * forwards from `obs` (and their histories), then ss_env_step_match, then the newest observation of each frames > 1 policy
 * pushed into its history at slot head + 1.  The forwards:
 *   both frames 1, tensor_cores     ONE ss_actor_forward_groups_tc over 2 n_envs rows, group_rows = n_envs
 *   a policy with frames > 1        ss_actor_forward_frames_tc (float32: ss_actor_forward_frames) on its half, param_stride 0
 *   a frames-1 policy otherwise     ss_actor_forward_tc (float32: ss_actor_forward) on its half
 * Histories: stack_a / stack_b (NULL for frames 1) are the layout of ss_obs_stack_push_tc (tensor_cores) or ss_obs_stack_push
 * (float32) for n_envs rows; `head` is the slot counter of the newest frame on entry, the same for both; after the call it is
 * head + n_ticks.  On return `obs` holds the current observations and `act` the last tick's actions.  Parameters: A's vector at
 * `params`, B's at params + param_stride (param_stride % 4 == 0, at least the larger of the two vectors' lengths).
 * `workspace` holds ss_match_workspace_bytes(n_envs, frames_a, frames_b, tensor_cores) bytes (16-byte aligned; NULL when 0).
 * Every argument is checked before anything is enqueued. */
typedef struct ss_match_args {
    void *state;
    int64_t n_envs, split, tick_limit;
    const void *speeds;                        /* NULL or the per-env speeds of ss_env_step */
    uint32_t *status;                          /* NULL or uint32[1] */
    float *obs, *act;
    const float *params;
    int64_t param_stride;
    int frames_a, frames_b;
    void *stack_a, *stack_b;
    int64_t head;
    void *workspace;
    int64_t workspace_bytes;
    int tensor_cores;
    int n_ticks;
} ss_match_args;
int64_t ss_match_workspace_bytes(int64_t n_envs, int frames_a, int frames_b, int tensor_cores);
int ss_match_play(const ss_match_args *args, void *stream);

/* ---- leagues: up to SS_LEAGUE_MAX_POLICIES actors in one batch (a match generalised to any schedule of pairings) ----
 * One game per env from tick 0 as in a match.  The rows of the policies' inputs and outputs are grouped in SEGMENTS, one
 * per policy, contiguous and in order: segment s = rows [seg_start[s], seg_start[s + 1]), one row for every env in which
 * its policy plays, and n_rows = 2 n_envs.  Which rows an env's two players read and write is device data:
 *   seat_rows   int32 [n_envs][2]  {row of player 1, row of player 2}  (an int2 per env, 8-byte aligned)
 *   seat_policy uint8 [n_envs][2]  {policy of player 1, policy of player 2}  (2-byte aligned; for the summary only)
 *   obs float32 [n_rows][12], act float32 [n_rows][2]
 *
 *   ss_env_step_seated    ss_env_step_match with the rows taken from seat_rows instead of the split rule: no reward, no
 *                         auto-reset, a live game with ticks >= tick_limit (> 0) is not stepped (its observation is written
 *                         again), SS_STATUS_NAN as ss_env_step raises it.  An env with a row outside [0, n_rows) is neither
 *                         read, stepped nor written and raises SS_STATUS_SEAT_RANGE.  n_rows < 2^31.
 *   ss_actor_forward_segments_tc  ss_actor_forward_tc (no noise) over n_segs (1..SS_LEAGUE_MAX_POLICIES) consecutive
 *                         segments of seg_rows_host[s] >= 1 rows each (a HOST array): segment s reads and writes the rows
 *                         from sum_{t<s} seg_rows_host[t] on and uses the vector params + s param_stride (param_stride % 4
 *                         == 0, 0 or >= SS_ACTOR_PARAMS).  Each row's action is bit-identical to ss_actor_forward_tc run
 *                         on its segment alone.
 *   ss_league_summary     out uint64 [n_policies][n_policies][8], OVERWRITTEN: cell (i, j) counts the envs with policy i in
 *                         seat 1 and policy j in seat 2 { games, seat-1 wins (player 2 was hit), seat-2 wins, draws (live,
 *                         ticks >= tick_limit), unfinished (live, ticks < tick_limit), sum of the ticks of the decided
 *                         games, 0, 0 }.  winner_id is the id of the player that was HIT.  Exact integer counts; an env
 *                         with a policy index >= n_policies is not counted.  2 <= n_policies <= SS_LEAGUE_MAX_POLICIES. */
#define SS_LEAGUE_MAX_POLICIES 64
int ss_env_step_seated(void *state, int64_t n_envs, const void *seat_rows, int64_t n_rows, const float *actions, float *obs_out,
                       int64_t tick_limit, const void *speeds, uint32_t *status, void *stream);
int ss_actor_forward_segments_tc(const float *params, int64_t param_stride, const int64_t *seg_rows_host, int n_segs,
                                 const float *obs, float *act_out, void *stream);
int ss_league_summary(const void *state, int64_t n_envs, const uint8_t *seat_policy, int n_policies, int64_t tick_limit,
                      uint64_t *out, void *stream);

/* n_ticks league ticks from one host call (as ss_match_play for two policies).  The arrays seg_start [n_policies + 1],
 * frames [n_policies] and stacks [n_policies] are HOST arrays indexed by segment; segment s uses the vector
 * params + s param_stride (param_stride % 4 == 0, at least every segment's ss_actor_frames_params).  Per tick:
 *   tensor_cores   one ss_actor_forward_segments_tc per maximal run of consecutive frames-1 segments, and
 *                  ss_actor_forward_frames_tc (param_stride 0) on each frames > 1 segment
 *   float32        ss_actor_forward or ss_actor_forward_frames on each segment
 * then ss_env_step_seated, then the newest observation of each frames > 1 segment pushed into its history stacks[s]
 * (the layout of ss_obs_stack_push_tc / ss_obs_stack_push for that segment's rows; NULL for frames 1) at slot head + 1.
 * `workspace` holds ss_league_workspace_bytes(args) bytes (16-byte aligned; NULL when 0; that call reads n_policies,
 * seg_start, frames and tensor_cores and returns -1 when they are invalid).  Every argument is checked before anything is
 * enqueued: 2 <= n_policies <= SS_LEAGUE_MAX_POLICIES, seg_start[0] == 0, every segment >= 1 row, seg_start[n_policies]
 * == 2 n_envs. */
typedef struct ss_league_args {
    void *state;
    int64_t n_envs, tick_limit;
    const void *speeds;                        /* NULL or the per-env speeds of ss_env_step */
    uint32_t *status;                          /* NULL or uint32[1] */
    const void *seat_rows;                     /* int32 [n_envs][2] */
    float *obs, *act;
    const float *params;
    int64_t param_stride;
    int n_policies;
    const int64_t *seg_start;                  /* host [n_policies + 1] */
    const int *frames;                         /* host [n_policies] */
    void *const *stacks;                       /* host [n_policies] */
    int64_t head;
    void *workspace;
    int64_t workspace_bytes;
    int tensor_cores;
    int n_ticks;
} ss_league_args;
int64_t ss_league_workspace_bytes(const ss_league_args *args);
int ss_league_play(const ss_league_args *args, void *stream);

/* ---- training against a pool: the self-play learner also plays frozen opponents ----
 * The last M = pool_envs of the n_envs envs are POOL envs: the learner against one of K = n_opponents frozen 1-frame actors.
 * Opponent k owns the b = M / K consecutive envs from S + k b (S = n_envs - M); the learner is player 1 in the first b / 2
 * of them and player 2 in the others, so M % (2K) == 0.  The rows, a fixed formula of (S, M, K):
 *   learner rows   L = 2S + M:  self-play env i < S: player p is row 2i + p (the layout of ss_env_step_ring);
 *                               pool env j >= S: the learner's player is row 2S + (j - S)
 *   opponent rows  M:           pool env j: the opponent's player is row j - S; opponent k's rows are one segment of b rows
 *
 *   ss_env_step_pool   one tick of ss_env_step_ring (auto-reset, reward none / looking / terminal, reference speeds) with the
 *                      rows above: actions float32 [L][2] and opp_actions [M][2] in; obs_out (and obs_out2 when not NULL)
 *                      [L][12], reward_out [L] (NULL or reward none: not written), done_rows_out uint8 [L] (the terminal
 *                      flag of ss_env_step_ring, NULL ok) for the learner's rows; opp_obs_out [M][12] for the opponents';
 *                      done_out / winner_out uint8 [n_envs] per env (NULL ok).  flags: SS_STEP_EPISODE_STATS or 0 (every env
 *                      counts).  pool_stats: NULL or uint64 [K][SS_POOL_STATS] ADDED TO per finished pool game: {episodes, learner wins
 *                      (the opponent was hit), learner losses (the learner was hit), tick-limit endings, sum of episode
 *                      ticks, 0, 0, 0}; winner_id is the player that was HIT, and a double hit records player 1 as hit.
 *                      M = 0 (n_opponents ignored) is the self-play step of ss_env_step_ring, bit for bit.
 *
 * ss_pool_rollout: n_ticks training ticks from one host call (as ss_selfplay_rollout).  Per tick:
 *   tensor_cores  ss_actor_forward_tc on the L learner rows (the rollout's noise, counter noise_counter + t), then
 *                 ss_actor_forward_segments_tc on the M opponent rows (K segments of b rows, no noise; skipped when M = 0)
 *   float32       ss_actor_forward on the learner rows and on each opponent segment
 * then ss_env_step_pool with counter env_counter + t.  The tensor-core launches form the dependent-launch chain of
 * ss_selfplay_rollout (ss_set_dependent_launch).  Opponent k acts with opp_params + k opp_param_stride.
 *   obs [L][12]        the learner rows' current observation on entry and on return
 *   opp_obs [M][12]    the opponent rows' current observation on entry and on return (updated in place)
 *   act [L][2], reward [L], opp_act [M][2], done / winner [n_envs]: the last tick's values on return
 * With a ring (ring_obs != NULL) the learner's transitions are produced IN the ring as in ss_selfplay_rollout: tick t owns
 * the L rows from write_pos + t L (mod capacity).  capacity and write_pos must be multiples of L, with capacity >= 2 L or
 * n_ticks == 1.  Without a ring the learner's rows are rewritten in obs / act / reward.  The opponents' transitions are not
 * stored.  Every argument is checked before anything is enqueued: besides the rules of ss_env_step_pool, speeds must be
 * NULL (per-env speeds: ss_pool_rollout_speeds below), K <= SS_LEAGUE_MAX_POLICIES and pointers aligned
 * as ss_selfplay_rollout's.  M = 0 gives ss_selfplay_rollout's results bit for bit. */
#define SS_POOL_STATS 8        /* uint64 counters per opponent in pool_stats */
int ss_env_step_pool(void *state, int64_t n_envs, int64_t pool_envs, int n_opponents, const float *actions,
                     const float *opp_actions, float *obs_out, float *obs_out2, float *reward_out, uint8_t *done_rows_out,
                     float *opp_obs_out, uint8_t *done_out, uint8_t *winner_out, int reward_mode, int64_t tick_limit,
                     int reset_mode, uint64_t seed, uint64_t counter, uint32_t *status, int flags, uint64_t *pool_stats,
                     void *stream);

/* Blocks of any size: opponent k owns the b_k consecutive pool envs from S + B_k, B_k = b_0 + ... + b_{k-1}, with the
 * learner player 1 in the first b_k / 2 of them and player 2 in the others.  The rows keep the formula above (learner row
 * 2S + (j - S), opponent row j - S of pool env j), so opponent k's rows are one segment of b_k rows from B_k.  Every b_k
 * = M / K is the layout above.  A block table opp_envs is a HOST int64 [K] of pool envs per opponent, each even and >= 2,
 * summing to M (M < 2^31); NULL means M / K each.  An invalid table returns -1 before anything is enqueued.
 *   ss_env_step_pool_blocks  ss_env_step_pool under the table (M = 0 takes no table).  Bit-identical to ss_env_step_pool
 *                            for the uniform table.
 *   ss_pool_restart          every pool env starts a new game: reset_mode FIXED or RANDOM, Philox4x32-10(key = seed,
 *                            counter = (env, counter)) as the auto-reset of a step with that counter.  The self-play envs are
 *                            untouched.  obs [L][12] (learner rows) and opp_obs [M][12] receive the new games' observations
 *                            under the table, the bytes an auto-reset tick writes.  No game ended, so nothing is counted;
 *                            status is not written (NULL ok). */
int ss_env_step_pool_blocks(void *state, int64_t n_envs, int64_t pool_envs, int n_opponents, const float *actions,
                            const float *opp_actions, float *obs_out, float *obs_out2, float *reward_out, uint8_t *done_rows_out,
                            float *opp_obs_out, uint8_t *done_out, uint8_t *winner_out, int reward_mode, int64_t tick_limit,
                            int reset_mode, uint64_t seed, uint64_t counter, uint32_t *status, int flags, uint64_t *pool_stats,
                            const int64_t *opp_envs, void *stream);
int ss_pool_restart(void *state, int64_t n_envs, int64_t pool_envs, int n_opponents, const int64_t *opp_envs, int reset_mode,
                    uint64_t seed, uint64_t counter, float *obs, float *opp_obs, uint32_t *status, void *stream);
/* Per-env speeds: ss_env_step_pool_blocks with the per-env constants of ss_env_step (`speeds`, required: not NULL, 16-byte
 * aligned, two 16-byte planes of n_envs entries, SkillshotEnvs.set_speeds).  Every other rule is ss_env_step_pool_blocks'
 * (opp_envs NULL: M / K each; reward none / looking / terminal).  Env i plays with the speeds of entry i whichever block
 * it is in, and its bytes are those of ss_env_step_ring with the same speeds under the layout's rows.  Without per-env
 * speeds the step is ss_env_step_pool / ss_env_step_pool_blocks.  ss_pool_restart serves both: a new game has cooldown 0,
 * so its observation does not depend on the speeds, and no start draw reads them. */
int ss_env_step_pool_speeds(void *state, int64_t n_envs, int64_t pool_envs, int n_opponents, const float *actions,
                            const float *opp_actions, float *obs_out, float *obs_out2, float *reward_out, uint8_t *done_rows_out,
                            float *opp_obs_out, uint8_t *done_out, uint8_t *winner_out, int reward_mode, int64_t tick_limit,
                            int reset_mode, uint64_t seed, uint64_t counter, uint32_t *status, int flags, uint64_t *pool_stats,
                            const int64_t *opp_envs, const void *speeds, void *stream);
typedef struct ss_pool_rollout_args {
    void *state;
    int64_t n_envs, pool_envs;
    int n_opponents;
    const float *params;                       /* the learner's actor */
    const float *opp_params;                   /* K opponent vectors, opp_param_stride floats apart */
    int64_t opp_param_stride;
    float *obs, *act, *reward;                 /* learner rows */
    float *opp_obs, *opp_act;                  /* opponent rows */
    uint8_t *done, *winner;                    /* [n_envs] */
    float *ring_obs, *ring_act, *ring_reward, *ring_next_obs;
    uint8_t *ring_done;
    int64_t capacity, write_pos;
    int n_ticks;
    float param_noise_sd;
    int64_t noise_group;
    float action_noise_sd;
    int tensor_cores, reward_mode;
    int64_t tick_limit;
    int reset_mode;
    uint64_t env_seed, env_counter, noise_seed, noise_counter;
    const void *speeds;                        /* must be NULL (per-env speeds: ss_pool_rollout_speeds) */
    uint32_t *status;                          /* NULL or the status block of ss_env_step */
    int step_flags;                            /* SS_STEP_EPISODE_STATS or 0 */
    uint64_t *pool_stats;                      /* NULL or uint64 [K][SS_POOL_STATS], added to */
} ss_pool_rollout_args;
int ss_pool_rollout(const ss_pool_rollout_args *args, void *stream);

/* The same training against a pool with frame-stacked networks: the learner reads its last `frames` (F_l, 1..20)
 * observations and opponent k its last opp_frames[k] (F_k, 1..20).  Histories are those of ss_obs_stack_push_tc
 * (tensor_cores) / ss_obs_stack_push (float32); `head` is the slot counter of the newest frame of every history on entry
 * (after the call: head + n_ticks).
 *
 *   ss_obs_stack_push_pool  the learner's history step of one pool tick, for its L = 2S + M rows (S = n_envs - pool_envs):
 *                           row r belongs to env r < 2S ? r / 2 : S + (r - 2S) and restarts when done[env] is set (any
 *                           episode end, the per-env done_out of ss_env_step_pool).  obs[r] goes to slot head % frames of
 *                           stack_tc (NULL: none) and stack32, or to every slot on a restart, with the bytes of
 *                           ss_obs_stack_push_tc and ss_obs_stack_push; the ordered row [12 frames] (oldest frame first, as
 *                           ss_obs_stack_ordered) is written to rows_out and, when not NULL, to rows_out2.  M = 0 is the
 *                           self-play rule (row r <-> env r / 2).  One launch; every history slot is read at most once.
 *
 * ss_pool_rollout_frames: ss_pool_rollout (whose all-frames-1 case it is, launch for launch) with these histories.  Per tick:
 *   learner, F_l > 1    ss_param_noise_groups (counter noise_counter + t; skipped without parameter noise), then
 *                       ss_actor_forward_frames_tc (float32: ss_actor_forward_frames) over the L rows, one vector per group
 *   learner, F_l = 1    as ss_pool_rollout
 *   opponents           one ss_actor_forward_segments_tc per maximal run of consecutive 1-frame opponents, and
 *                       ss_actor_forward_frames_tc (parameter stride 0) on each F_k > 1 opponent's b rows; float32: the
 *                       exact forward of each opponent
 *   ss_env_step_pool    reward and hit flag into the ring segment; observations into it too when F_l = 1, into the staging
 *                       obs [L][12] when F_l > 1
 *   pushes              F_l > 1: ss_obs_stack_push_pool, writing the ring's next_obs of segment t and obs of segment t + 1
 *                       (the caller's `rows` on the last tick; without a ring only `rows`); each F_k > 1 opponent:
 *                       ss_obs_stack_push_tc / ss_obs_stack_push on its stack with done + S + k b, done_div 1
 * With F_l > 1 the ring rows hold 12 F_l floats of observation (ss_replay_push_frames' layout) and segment t's obs is filled
 * from `rows` on entry.  The ring, speed and reward rules are ss_pool_rollout's; action_noise_sd must be 0 when F_l > 1.
 *   rows [L][12 F_l]    the learner's current ordered rows on entry and on return (F_l > 1)
 *   opp_frames [K]      HOST array; NULL: every opponent has 1 frame.  opp_stacks [K] HOST array, NULL entries for F_k = 1
 *   opp_param_stride    % 4 == 0 and (K > 1) at least every opponent's ss_actor_frames_params(F_k)
 *   workspace           ss_pool_rollout_frames_workspace_bytes(args) bytes, 16-byte aligned (NULL when 0): the learner's
 *                       noisy parameter vectors and the frame-stacked forward's layer-1 tiles.  That call reads n_envs,
 *                       pool_envs, n_opponents, frames, opp_frames, tensor_cores, param_noise_sd and noise_group and returns
 *                       -1 when they are invalid.
 *   opp_envs [K]        HOST block table of ss_env_step_pool_blocks (it also reads this); NULL: M / K each, launch for launch
 *                       the rollout above.  With a table, opponent k's forward, history and workspace use its b_k rows from
 *                       B_k, and the step is ss_env_step_pool_blocks.
 *
 * ss_pool_rollout_speeds: ss_pool_rollout_frames with per-env speeds -- args->speeds (required, the layout of ss_env_step)
 * -- and the env step ss_env_step_pool_speeds in place of ss_env_step_pool / ss_env_step_pool_blocks.  Every other launch,
 * rule, ring layout and the workspace (ss_pool_rollout_frames_workspace_bytes) are ss_pool_rollout_frames'. */
typedef struct ss_pool_rollout_frames_args {
    void *state;
    int64_t n_envs, pool_envs;
    int n_opponents;
    const float *params;
    const float *opp_params;
    int64_t opp_param_stride;
    float *obs, *act, *reward;
    float *opp_obs, *opp_act;
    uint8_t *done, *winner;
    float *ring_obs, *ring_act, *ring_reward, *ring_next_obs;
    uint8_t *ring_done;
    int64_t capacity, write_pos;
    int n_ticks;
    float param_noise_sd;
    int64_t noise_group;
    float action_noise_sd;
    int tensor_cores, reward_mode;
    int64_t tick_limit;
    int reset_mode;
    uint64_t env_seed, env_counter, noise_seed, noise_counter;
    const void *speeds;                        /* ss_pool_rollout_speeds: the per-env speeds; ss_pool_rollout_frames: NULL */
    uint32_t *status;
    int step_flags;
    uint64_t *pool_stats;
    int frames;                                /* the learner's F_l */
    void *stack_tc;                            /* learner history, tensor-core layout (tensor_cores, F_l > 1) */
    float *stack32;                            /* learner history, float32 [L][F_l][12] (F_l > 1) */
    float *rows;                               /* [L][12 F_l] (F_l > 1) */
    int64_t head;
    const int *opp_frames;                     /* host [K] or NULL */
    void *const *opp_stacks;                   /* host [K] or NULL */
    void *workspace;
    int64_t workspace_bytes;
    const int64_t *opp_envs;                   /* host [K]: pool envs per opponent; NULL: M / K each */
} ss_pool_rollout_frames_args;
int ss_obs_stack_push_pool(void *stack_tc, float *stack32, int64_t n_envs, int64_t pool_envs, int frames, int64_t head,
                           const float *obs, const uint8_t *done, float *rows_out, float *rows_out2, void *stream);
int64_t ss_pool_rollout_frames_workspace_bytes(const ss_pool_rollout_frames_args *args);
int ss_pool_rollout_frames(const ss_pool_rollout_frames_args *args, void *stream);
int ss_pool_rollout_speeds(const ss_pool_rollout_frames_args *args, void *stream);

/* ---- multi-GPU: the gradient all-reduce fused with its neighbours over NVLink peer memory ----
 * One exchange allocation per rank = flags[2][world] | inbox[2][world][capacity floats], made by
 * ss_peer_alloc and shared between the processes of one node through CUDA IPC (export on the owner,
 * import on every other rank; these five helpers are the library's only allocating calls).
 *
 * A sharded update step (ranks hold equal shards of the batch):
 *   1. ss_critic_grad / ss_actor_grad / *_tc with grad_out == NULL: only the per-CTA gradient
 *      slices are left in `workspace`; the call returns their number (> 0) instead of 0;
 *   2. ss_peer_reduce_push: sums the slices in a fixed order and stores the result into slot `rank`
 *      of EVERY rank's inbox (peer stores), then raises this rank's flag for `epoch` everywhere;
 *      aux_out[0] = sum of the slices' extra slot (the shard's squared error / Q sum), or NULL;
 *   3. ss_peer_adam_tf: waits for all `world` flags of `epoch`, sums the inbox slots in rank order
 *      (bit-identical on every rank), then does exactly what ss_adam_tf does; grad_out (may be NULL)
 *      receives the summed gradient.  A peer that never arrives sets SS_STATUS_PEER_TIMEOUT.
 * `epoch` starts at 1 and increases by 1 per exchange, identically on all ranks; `done_counter` is a
 * zero-initialised uint32 on the device.  peer_bases_host[world] are the exchange allocations as
 * mapped in this process (own allocation at index rank). */
#define SS_PEER_MAX_WORLD 8
#define SS_PEER_HANDLE_BYTES 64
int64_t ss_peer_bytes(int world, int64_t capacity);
int ss_peer_alloc(int world, int64_t capacity, void **base_out);
int ss_peer_free(void *base);
int ss_peer_export(void *base, void *handle_out_host);          /* 64-byte CUDA IPC handle */
int ss_peer_import(const void *handle_host, void **base_out);
int ss_peer_close(void *imported_base);
int ss_peer_reduce_push(const void *workspace, int parts, int n_params, float *aux_out,
                        void *const *peer_bases_host, int world, int rank, int64_t capacity,
                        uint32_t epoch, uint32_t *done_counter, void *stream);
int ss_peer_adam_tf(void *own_base, int world, int64_t capacity, uint32_t epoch, float *params, float *m,
                    float *v, float *target_params, float *grad_out, int64_t n, int64_t step, float lr,
                    float beta1, float beta2, float eps, float tau, float grad_scale, uint32_t *status,
                    void *stream);
/* ss_peer_reduce_push + ss_peer_adam_tf as ONE kernel: each 64-parameter CTA sums the slices, pushes its sums to every
 * rank's inbox, raises its own flag there, waits for the same CTA's flag of every rank, and applies Adam to the sum taken
 * in rank order.  Same results as the two calls, bit for bit; one launch and no grid-wide completion counter per exchange.
 * (The allocation of ss_peer_alloc holds these per-CTA flags behind the inboxes.) */
int ss_peer_reduce_adam_tf(const void *workspace, int parts, int n_params, float *aux_out, void *const *peer_bases_host,
                           int world, int rank, int64_t capacity, uint32_t epoch, float *params, float *m, float *v,
                           float *target_params, float *grad_out, int64_t step, float lr, float beta1, float beta2, float eps,
                           float tau, float grad_scale, uint32_t *status, void *stream);

/* Device-resident replay ring, structure of arrays with `capacity` rows:
 * obs [cap][12], act [cap][2], reward [cap], next_obs [cap][12], done [cap] u8.
 * The reference's "buffer" is one episode used once (SkillshotLearner.py:334-361);
 * a ring of that size consumed in order reproduces it.
 * push: rows write_pos .. write_pos+n-1 (mod capacity) <- the n transitions; done
 *       has one entry per `done_div` rows (2 when it is the per-env flag of ss_env_step). */
int ss_replay_push(float *ring_obs, float *ring_act, float *ring_reward, float *ring_next_obs,
                   uint8_t *ring_done, int64_t capacity, int64_t write_pos, const float *obs,
                   const float *act, const float *reward, const float *next_obs, const uint8_t *done,
                   int done_div, int64_t n, void *stream);

/* sample: batch rows gathered from the first `size` rows; indices int64 [batch]
 * given (parity: np.random.shuffle order, SkillshotLearner.py:426-431) or NULL =
 * uniform with replacement from Philox(seed; counter). indices_out may be NULL. */
int ss_replay_sample(const float *ring_obs, const float *ring_act, const float *ring_reward,
                     const float *ring_next_obs, const uint8_t *ring_done, int64_t capacity, int64_t size,
                     const int64_t *indices, uint64_t seed, uint64_t counter, int64_t batch,
                     float *obs, float *act, float *reward, float *next_obs, uint8_t *done,
                     int64_t *indices_out, void *stream);

/* One update step of the batched learner from a single host call: ss_replay_sample (Philox indices)
 * -> TD target (skipped when gamma == 0: the critic regresses on the reward, SkillshotLearner.py:434)
 * -> critic gradient -> [exchange] -> Adam + soft target update -> actor gradient with the UPDATED critic
 * (model_actor_fit_step, SkillshotLearner.py:386-417, follows the critic fit, 434-443) -> [exchange] -> Adam.
 * The same launches, in the same order and with the same arguments, as calling those entry points one by
 * one; it exists because that sequence costs ~150 us of interpreter time per update from Python.
 * All pointers are device pointers except peer_bases (host array, as for ss_peer_reduce_push).
 *   tensor_cores != 0   the *_tc gradient / target kernels (workspace as they require)
 *   peer_bases == NULL  single GPU (ss_reduce_adam_tf): grad_actor / grad_critic (may be NULL) receive the gradients
 *   peer_bases != NULL  sharded batch with the fused NVLink exchange: the critic exchange is epoch
 *                       `epoch`, the actor's `epoch + 1`; grad_* (may be NULL) receive the summed gradients
 *   stats[2]            sum of squared errors of the critic batch, sum of Q of the actor batch (this shard's)
 *   step_critic/actor   Adam step numbers of THIS update (>= 1) */
typedef struct ss_ddpg_update_args {
    const float *ring_obs, *ring_act, *ring_reward, *ring_next_obs;
    const uint8_t *ring_done;
    int64_t capacity, size;
    uint64_t replay_seed, replay_counter;
    int64_t batch;
    float *obs, *act, *reward, *next_obs;      /* minibatch buffers of `batch` rows, filled by the call */
    uint8_t *done;
    int64_t *indices;                          /* may be NULL */
    float *y;                                  /* TD targets [batch]; unused when gamma == 0 */
    float *actor, *critic, *target_actor, *target_critic;    /* targets may be NULL when gamma == 0 (no soft update) */
    float *m_actor, *v_actor, *m_critic, *v_critic;
    float *grad_actor, *grad_critic;
    float *stats;
    float gamma, tau, lr_actor, lr_critic, beta1, beta2, eps, dropout_rate;
    uint64_t seed, counter;                    /* dropout stream (ss_critic_grad) */
    int64_t step_critic, step_actor;
    int64_t n_global, row_offset;              /* as for ss_critic_grad */
    void *workspace;
    int64_t workspace_bytes;
    int tensor_cores;
    int world, rank;
    void *const *peer_bases;
    int64_t peer_capacity;
    uint32_t epoch;
    uint32_t *done_counter, *status;
    void *pair_mail;                           /* ss_actor_critic_forward_tc's mailbox for `batch` rows, or NULL: the
                                                  actor -> critic forward pairs then run as two launches each */
    int sample_early;                          /* 1: the caller guarantees that the launch preceding this call on the stream
                                                  neither writes the replay ring nor touches THIS call's minibatch buffers
                                                  (obs .. y, indices) -- e.g. the previous ss_ddpg_update used another set of
                                                  buffers and no rollout came between: the minibatch is then gathered while
                                                  that launch still runs.  0: the gather waits for it */
    int n_step;                                /* 0 or 1: one-step rows (ss_replay_sample), the fields below unused;
                                                  2..SS_REPLAY_MAX_NSTEP: n-step rows (ss_replay_sample_nstep), and gamma
                                                  above is then the bootstrap factor g_n of that recurrence */
    int64_t tick_rows;                         /* ring rows per tick (ss_replay_sample_nstep) */
    int n_runs;                                /* eligible runs: runs_host[2 n_runs] = {start, length, ...} (host memory) */
    const int64_t *runs_host;
    float step_gamma;                          /* the per-tick gamma of the n-step reward sum's weights */
    int prioritized;                           /* 0: the uniform draw, the fields below unused.  1: prioritized replay
                                                  (DESIGN.md section 6.16): ss_replay_sample_prioritized over [0, size) (or the
                                                  n-step runs), the critic gradient weighted by `weights` with |e| into
                                                  td_abs (ss_critic_grad_weighted), and after the critic's Adam
                                                  ss_replay_priority_update at `indices`.  Refused with sample_early. */
    float *priority;                           /* leaves [capacity] */
    float *priority_max;
    void *priority_scratch;                    /* ss_replay_priority_scratch_bytes(capacity) bytes */
    int64_t priority_scratch_bytes;
    int32_t *priority_update_scratch;          /* int32[capacity] */
    float priority_alpha, priority_beta, priority_eps;
    float *weights;                            /* [batch] importance weights out */
    float *td_abs;                             /* [batch] |q - y| out */
} ss_ddpg_update_args;
int ss_ddpg_update(const ss_ddpg_update_args *args, void *stream);

/* ss_ddpg_update and ss_selfplay_rollout launch their kernels as a programmatic-dependent-launch chain (each grid is placed
 * while its predecessor drains and waits, griddepcontrol.wait, before its first dependent access; csrc/ss_launch.cuh).
 * enabled = 0: ordinary launches; 1: chained; -1: back to the default (chained).  Returns the previous setting (-1 / 0 / 1).
 * Results are bit-identical either way. */
int ss_set_dependent_launch(int enabled);

/* a = actor(s) -> act_out [n][2], then critic([s, a]) -> any of q_out [n] / neg_dq_da_out [n][2] / y_out [n] (the TD target
 * reward + gamma (1 - done) q, as ss_critic_forward_tc), in ONE launch: half of the CTAs play the actor, the other half the
 * critic, which takes each row's actions as soon as the actor half has written them.  The two steps of
 * model_actor_fit_step's forward pass (SkillshotLearner.py:395-400) and of the TD target.  Bit-identical to
 * ss_actor_forward_tc (no noise) followed by ss_critic_forward_tc.
 * pair_mail: 8 bytes per row (8-byte aligned), every 32-bit word SS_PAIR_MAIL_EMPTY before the first call; every call
 * leaves it so.  The actor half writes a row's two actions there, the critic half polls the row until neither word is the
 * empty mark (the data is its own flag), takes them and puts the mark back. */
#define SS_PAIR_MAIL_EMPTY 0x7fc0dead          /* a NaN payload no arithmetic produces */
int ss_actor_critic_forward_tc(const float *actor_params, const float *critic_params, const float *obs, float *act_out,
                               int64_t n, float *q_out, float *neg_dq_da_out, const float *reward, const uint8_t *done,
                               float gamma, float *y_out, void *pair_mail, void *stream);
/* ss_actor_grad_tc_staged / ss_ddpg_targets_tc with the forward pair as one launch when pair_mail != NULL (stage 0 only) */
int ss_actor_grad_tc_paired(const float *actor_params, const float *critic_params, const float *obs, int64_t n,
                            float *grad_out, float *q_sum_out, void *workspace, int64_t workspace_bytes, int stage,
                            void *pair_mail, void *stream);
int ss_ddpg_targets_tc_paired(const float *target_actor_params, const float *target_critic_params, const float *reward,
                              const float *next_obs, const uint8_t *done, float gamma, float *y_out, int64_t n,
                              void *workspace, int64_t workspace_bytes, void *pair_mail, void *stream);

/* Measurement aid (no reference counterpart): instruction-rate ceilings of this GPU for the roofline record of the fused
 * step kernel, which is bound by the warp schedulers and the float64 pipe rather than by HBM once K ticks are played per
 * launch.  Runs two register-only kernels, times them with CUDA events and SYNCHRONISES (the one entry point that does).
 *   out_host[0]  warp-instructions per second of an alternating LOP3 / IMAD stream (the issue ceiling: SMs x 4 schedulers x clock)
 *   out_host[1]  warp-instructions per second of a DFMA stream (the float64 pipe)
 *   out_host[2]  number of SMs;  out_host[3] reserved
 *   scratch      any device buffer of >= 8 bytes (never written in practice) */
int ss_probe_rates(double *out_host, void *scratch, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SKILLSHOT_B200_H */
