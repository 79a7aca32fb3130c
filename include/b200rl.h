/*
 * b200rl.h — C ABI of libb200rl.so: the collect -> store -> sample -> update hot path
 * of TF-Agents, as hand-written sm_100a CUDA.
 *
 * The reference (tensorflow/agents @ eb24cf5f) has no FFI for this path: it is plain
 * Python over TensorFlow ops (SURVEY.md §8b).  This header therefore *defines* the
 * boundary a reference maintainer would bind with ctypes (see INTEGRATION.md); every
 * entry point cites the reference function whose device work it replaces.  All
 * file:line citations are relative to /root/reference/tf_agents/.
 *
 * Conventions
 *   - Every pointer named *_dev / documented "device" is a CUDA device pointer owned by the
 *     caller (PyTorch in this repo).  The library never allocates persistent memory.
 *   - `stream` is a cudaStream_t passed as void*.  Every call only ENQUEUES work on that
 *     stream and returns; ordering on one stream replaces the reference's
 *     tf.CriticalSection (replay_buffers/tf_uniform_replay_buffer.py:154,582-601).
 *   - Return value: 0 = ok, <0 = error; b200rl_last_error() gives the message
 *     (thread-local).  No entry point falls back to the CPU.
 *   - Counters that the reference keeps in tf.Variables (last_id, train_step, Periodically
 *     counter, optimizer iterations) live in device memory so that a whole
 *     collect/train step can be captured in one CUDA graph and replayed.  Counter blocks
 *     named step_dev / counter_dev (int64[2]) and the rng_call_dev of the env / policy
 *     kernels (uint64[2]) are {value, ticket}: the second word is scratch for the
 *     last-block-done update and must start at 0.  b200rl_rb_sample / b200rl_rb_draw use
 *     ring->ticket instead, so their rng_call_dev is a single uint64.
 */
#ifndef B200RL_H_
#define B200RL_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200RL_OK 0
#define B200RL_ERR_INVALID (-1)
#define B200RL_ERR_CUDA (-2)
#define B200RL_ERR_UNSUPPORTED (-3)

#define B200RL_MAX_LEAVES 24

/* activation codes for dense / conv epilogues */
#define B200RL_ACT_NONE 0
#define B200RL_ACT_RELU 1
#define B200RL_ACT_TANH 2

/* element-wise TD loss kinds (utils/common.py:1199-1208) */
#define B200RL_LOSS_HUBER 0
#define B200RL_LOSS_SQUARED 1

const char* b200rl_last_error(void);
int b200rl_version(void);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t b200rl_launch_count(void);
/* Programmatic dependent launch: when enabled (the default; B200RL_PDL=0 in the environment or
 * b200rl_set_pdl(0) switches it off) every kernel
 * is launched with cudaLaunchAttributeProgrammaticStreamSerialization, so inside a captured step
 * (common.function, utils/common.py:128 in the reference) the next node's launch overlaps the
 * running one; every kernel orders itself with griddepcontrol.wait. */
int b200rl_set_pdl(int enabled);
int b200rl_get_pdl(void);

/* ------------------------------------------------------------------------------------
 * Ring storage — replaces Table (replay_buffers/table.py:32-137) + the variables of
 * TFUniformReplayBuffer (replay_buffers/tf_uniform_replay_buffer.py:132-161).
 * One leaf == one slot of the Table: a [capacity, row_bytes] byte matrix.
 * Segment b occupies rows [b*max_length, (b+1)*max_length).
 * ------------------------------------------------------------------------------------ */
typedef struct {
  void* storage;     /* device, [capacity * row_bytes] bytes */
  int64_t row_bytes; /* bytes of one item of this leaf */
} b200rl_leaf_t;

typedef struct {
  int32_t num_leaves;
  int32_t _pad;
  int64_t batch_size; /* B_env: number of segments */
  int64_t max_length; /* L: rows per segment */
  int64_t* id_table;  /* device, [capacity] int64 (id table, tf_uniform_replay_buffer.py:152) */
  int64_t* last_id;   /* device scalar int64, -1 when empty (:153) */
  uint32_t* ticket;   /* device scalar uint32 scratch, zero-initialised by the caller */
  b200rl_leaf_t leaves[B200RL_MAX_LEAVES];
} b200rl_ring_t;

/* Selects the row-copy kernel used by every ring read/write: 0 = 16-byte LDG/STG kernel,
 * 1 = TMA bulk-copy (cp.async.bulk) kernel.  Default: env B200RL_COPY_VARIANT, else 1 (TMA:
 * 5.7 TB/s vs 3.6 TB/s at batch 4096, profiles/r1_gather_sweep.jsonl). */
int b200rl_set_copy_variant(int variant);

/* _add_batch (tf_uniform_replay_buffer.py:182-209): id = ++last_id; rows[b] = b*L + id % L;
 * scatter every leaf row and the id.  items[i] is a device pointer to [B_env, row_bytes_i]. */
int b200rl_rb_add_batch(const b200rl_ring_t* ring, const void* const* items, void* stream);

/* _get_next (tf_uniform_replay_buffer.py:211-310), time_stacked form.
 *   B = sample_batch_size (>=1; pass 1 for the unbatched form), T = num_steps (>=1).
 *   ids_dev/offs_dev: when both non-NULL the kernel uses these externally supplied draws
 *     (ids in [min,max), offs in [0,B_env)) — "oracle mode"; otherwise it draws with
 *     Philox4x32-10 keyed by `seed`, call index *rng_call_dev (then increments it).
 *   out[i]: device pointer to [B, T, row_bytes_i]; out_ids: [B,T] int64 (id table values);
 *   out_rows: optional [B,T] int64 row indices; out_prob: [B] f32.
 *   status_dev: optional device int32, set to 1 when the valid id range is empty. */
int b200rl_rb_sample(const b200rl_ring_t* ring, int64_t B, int64_t T, const int64_t* ids_dev,
                     const int64_t* offs_dev, uint64_t seed, uint64_t* rng_call_dev,
                     void* const* out, int64_t* out_ids, int64_t* out_rows, float* out_prob,
                     int32_t* status_dev, void* stream);

/* Table.read(rows) (table.py:86-110) for explicit row ids rows_dev[n] (already < capacity). */
int b200rl_rb_read_rows(const b200rl_ring_t* ring, const int64_t* rows_dev, int64_t n,
                        void* const* out, int64_t* out_ids, void* stream);

/* Table.write(rows, values) (table.py:112-137) for explicit row ids. */
int b200rl_rb_write_rows(const b200rl_ring_t* ring, const int64_t* rows_dev, int64_t n,
                         const void* const* items, void* stream);

/* _gather_all (tf_uniform_replay_buffer.py:533-557): out[i] is [B_env, n_valid, row_bytes_i],
 * items in age order; n_valid is the host's copy of max_val-min_val. */
int b200rl_rb_gather_all(const b200rl_ring_t* ring, int64_t n_valid, void* const* out,
                         void* stream);

/* _clear (tf_uniform_replay_buffer.py:559-579): last_id = -1; zero tables when clear_all. */
int b200rl_rb_clear(const b200rl_ring_t* ring, int clear_all, void* stream);

/* Frame-dedup gather (no TFUniformReplayBuffer counterpart; the reference de-duplicates frames
 * only in the host-side PyHashedReplayBuffer, replay_buffers/py_hashed_replay_buffer.py:37-181).
 * frames: [batch_size*max_length, frame_bytes] uint8 ring leaf holding ONE frame per slot;
 * step_type: the ring's int32 step_type leaf.  For every sampled window start ids_dev[b] in segment
 * offsets_dev[b] and every t < T, out[b, t] (frame_bytes * K bytes, pixel-major / channel-minor,
 * i.e. [H, W, K]) receives the K most recent frames of the item's episode: channel c = frame of id
 * max(id - (K-1-c), id of the episode's FIRST step) (semantics: oracle/frame_stack.py).
 * frame_bytes must be a multiple of 4, 1 <= K <= 4.  The caller keeps ids whose look-back would
 * reach overwritten slots out of ids_dev. */
int b200rl_rb_gather_frame_stack(const void* frames, const int32_t* step_type,
                                 int64_t frame_bytes, int64_t max_length,
                                 const int64_t* ids_dev, const int64_t* offsets_dev, int64_t B,
                                 int64_t T, int32_t K, void* out, void* stream);

/* Philox draw alone (tf_uniform_replay_buffer.py:265-272) — same stream as b200rl_rb_sample. */
int b200rl_rb_draw(const b200rl_ring_t* ring, int64_t B, int64_t T, uint64_t seed,
                   uint64_t* rng_call_dev, int64_t* out_ids, int64_t* out_offs, void* stream);

/* ------------------------------------------------------------------------------------
 * Scans — utils/value_ops.py
 * ------------------------------------------------------------------------------------ */
/* discounted_return (value_ops.py:21-99).  Inputs [T,B] when time_major else [B,T].
 * final_value may be NULL (zeros).  provide_all: out has the input layout; else out is [B]. */
int b200rl_discounted_return(const float* rewards, const float* discounts,
                             const float* final_value, float* out, int64_t B, int64_t T,
                             int time_major, int provide_all, void* stream);

/* generalized_advantage_estimation (value_ops.py:102-164). */
int b200rl_gae(const float* values, const float* final_value, const float* discounts,
               const float* rewards, float td_lambda, float* out_adv, int64_t B, int64_t T,
               int time_major, void* stream);

/* Batch-major variants over the first T columns of [B, ld] arrays (PPO: T-1 of T steps). */
int b200rl_discounted_return_ld(const float* rewards, const float* discounts,
                                const float* final_value, float* out, int64_t B, int64_t T,
                                int64_t ld_in, int64_t ld_out, int64_t fv_stride, void* stream);
int b200rl_gae_ld(const float* values, const float* final_value, const float* discounts,
                  const float* rewards, float td_lambda, float* out_adv, int64_t B, int64_t T,
                  int64_t ld_in, int64_t ld_out, int64_t fv_stride, void* stream);

/* to_n_step_transition reward/discount reduction (trajectories/trajectory.py:815-832):
 * reward,discount are [B,T] (T = n+1, last column ignored). */
int b200rl_nstep_reduce(const float* reward, const float* discount, double gamma,
                        float* out_reward, float* out_discount, int64_t B, int64_t T,
                        void* stream);

/* ------------------------------------------------------------------------------------
 * DQN loss epilogue — agents/dqn/dqn_agent.py:462-579 (+ :75-78, :451-460, :604-645,
 * DdqnAgent :659-700), utils/common.py:367-411 (index_with_actions), :1199-1208 (losses),
 * :1400-1476 (aggregate_losses).
 *   q[B,A]          online Q(s_0)
 *   next_q_tgt[B,A] target Q(s_n)          (value taken here)
 *   next_q_sel[B,A] net that picks argmax  (== next_q_tgt for DQN, online Q(s_n) for DDQN)
 *   next_mask[B,A]  optional int32 action mask for the argmax (1 = allowed)
 *   step_type0[B]   int32 step type of the first frame (LAST=2 zeroes the loss)
 *   action_stride / step_stride: element strides of `actions` / `step_type0`, so the [:, 0]
 *                   columns of [B, T] trajectory tensors are read in place (1 when packed);
 *                   actions outside [0, A) are clamped before they index q
 *   traj_reward/traj_discount [B,T] raw trajectory fields (T = n+1); n-step reduction fused.
 *   weights[B] optional.  global_batch: divisor of the loss sum (B * replicas).
 * Outputs: loss[0] (= sum(td_loss*w)/global_batch, no reg), td_loss[B], td_error[B],
 *          dq[B,A] = dLoss/dq (zero except at the taken action), nan_flag (optional int32,
 *          set when loss is not finite; dqn_agent.py:422 check_numerics).
 * ------------------------------------------------------------------------------------ */
int b200rl_dqn_td_loss(const float* q, const float* next_q_tgt, const float* next_q_sel,
                       const int32_t* next_mask, const int32_t* actions,
                       const int32_t* step_type0, const float* traj_reward,
                       const float* traj_discount, const float* weights, int64_t action_stride,
                       int64_t step_stride, int64_t B, int64_t A, int64_t T, double gamma,
                       double reward_scale, int loss_kind,
                       float global_batch, float* loss, float* td_loss, float* td_error,
                       float* dq, int32_t* nan_flag, void* stream);

/* ------------------------------------------------------------------------------------
 * Episodic replay buffer bookkeeping -- replay_buffers/episodic_replay_buffer.py.
 * An episode slot owns rows [slot*max_len, (slot+1)*max_len) of the leaf storage; row
 * capacity*max_len is a trash row for items whose episode id is stale.
 * ------------------------------------------------------------------------------------ */
/* One launch = `_get_batch_episode_ids` (:1109-1187: ids < 0 or with begin[i] get consecutive new
 * ids in item order, their slots are reset) + `_maybe_end_batch_episodes` (:1015-1045) + the
 * length bump of add_batch / add_sequence / extend_episodes (:332-463, :1336-1414).  steps (per
 * item) or steps_all rows are reserved per valid item and their first storage row is returned in
 * out_rows (the trash row for stale ids or when max_len would be exceeded; *overflow = 1 then).
 * All arrays are device pointers; begin / end / mask / steps / num_writes / out_rows / overflow
 * may be NULL. */
int b200rl_ep_assign(int64_t* episode_ids, const uint8_t* begin, const uint8_t* end,
                     const uint8_t* mask, const int64_t* steps, int64_t steps_all, int64_t N,
                     int64_t capacity, int64_t max_len, int64_t* last_episode, int64_t* loc_to_id,
                     int64_t* lengths, uint8_t* completed, int64_t* num_writes, int bump_writes,
                     int set_completed_from_end, int64_t* out_rows, int32_t* overflow,
                     void* stream);

/* ------------------------------------------------------------------------------------
 * PPO update math — agents/ppo/ppo_agent.py, ppo_utils.py, utils/tensor_normalizer.py
 * ------------------------------------------------------------------------------------ */
/* Fused clipped-surrogate / value / entropy losses + gradients over N = B*T elements
 * (ppo_agent.py:1159-1201 entropy, :1203-1327 value, :1329-1512 policy gradient; each is
 * sum(loss*w) / (T * global_batch), utils/common.py:1400-1476).  The current policy is a diagonal
 * Normal(loc, scale) given as [N, A] views with row stride ld_ls; gradients are written with row
 * stride ld_g.  clip_eps <= 0, value_clip <= 0, logp_clip <= 0 disable the respective clipping.
 * losses[6] = {policy_gradient, value_estimation (x vf_coef), entropy_regularization (x ent_coef),
 * clip_fraction, total (without l2), kl_penalty}.
 * kl (NULL: no KL penalty, what PPOClipAgent configures, ppo_clip_agent.py:226-232): the
 * behaviour policy's Normal(old_loc, old_scale) and the device scalars written by
 * b200rl_ppo_kl_terms; the gradient of kl_cutoff_loss + adaptive_kl_loss (ppo_agent.py:1514-1630)
 * is added to dloc/dscale and their sum to the total. */
typedef struct {
  const float* old_loc;   /* device [N, A], row stride ld_old */
  const float* old_scale;
  int64_t ld_old;
  const float* terms;     /* device float[3] from b200rl_ppo_kl_terms */
  float grad_scale;       /* d(mean_kl)/d(sum_n w_n kl_n) = 1 / N_global */
} b200rl_ppo_kl_t;
int b200rl_ppo_loss(const float* loc, const float* scale, int64_t ld_ls, const float* action,
                    const float* old_logp, const float* adv, const float* ret, const float* v,
                    const float* v_old, const float* w, int64_t N, int64_t A, int64_t T,
                    float global_batch, float clip_eps, float value_clip, float vf_coef,
                    float ent_coef, float logp_clip, float* losses, float* dloc, float* dscale,
                    int64_t ld_g, float* dv, int32_t* nan_flag, const b200rl_ppo_kl_t* kl,
                    void* workspace, int64_t ws_bytes, void* stream);
/* out_sum = out_scale * sum_n w_n * KL(Normal(old_loc, old_scale)_n || Normal(loc, scale)_n), the
 * KL summed over action dims (ppo_utils.nested_kl_divergence, ppo_utils.py:194-227; per-dimension
 * closed form of tfp Normal); out_kl (optional) keeps the weighted per-element values
 * (kl_penalty_loss, ppo_agent.py:1613-1617).  w may be NULL. */
int b200rl_ppo_kl(const float* loc, const float* scale, int64_t ld, const float* old_loc,
                  const float* old_scale, int64_t ld_old, const float* w, int64_t N, int64_t A,
                  float out_scale, float* out_kl, float* out_sum, void* workspace,
                  int64_t ws_bytes, void* stream);
/* terms[3] = {kl_cutoff_loss = coef * max(mean_kl - factor*target, 0)^2 (ppo_agent.py:1514-1539;
 * 0 when factor <= 0), adaptive_kl_loss = beta * mean_kl (:1541-1558; beta_dev NULL -> 0), and the
 * derivative of their sum w.r.t. mean_kl}. */
int b200rl_ppo_kl_terms(const float* mean_kl_dev, const float* beta_dev, float kl_cutoff_factor,
                        float adaptive_kl_target, float kl_cutoff_coef, float* terms_dev,
                        void* stream);
/* update_adaptive_kl_beta (ppo_agent.py:1632-1675) on the device-resident beta. */
int b200rl_ppo_kl_beta_update(const float* mean_kl_dev, float* beta_dev, float adaptive_kl_target,
                              float adaptive_kl_tolerance, void* stream);
/* log-prob of actions under Normal(loc, scale), summed over action dims (common.py:682-717). */
int b200rl_normal_logp(const float* loc, const float* scale, int64_t ld, const float* action,
                       int64_t N, int64_t A, float* out, void* stream);
/* action = clip(loc + scale * z, amin, amax), z ~ N(0,1) (Philox + Box-Muller);
 * rng_call_dev is uint64[2] {call, ticket}. */
int b200rl_normal_sample(const float* loc, const float* scale, int64_t ld, int64_t N, int64_t A,
                         const float* amin, const float* amax, uint64_t seed,
                         uint64_t* rng_call_dev, float* out, void* stream);
/* NormalProjectionNetwork head (networks/normal_projection_network.py): loc = tanh-squash of the
 * mean layer to [amin, amax], scale = softplus(bias) broadcast; bwd returns dm_raw and the
 * per-element d(scale bias) terms (column-sum them with b200rl_colsum). */
int b200rl_normal_proj_fwd(const float* m_raw, const float* s_raw, const float* amin,
                           const float* amax, int64_t N, int64_t A, float* loc, float* scale,
                           void* stream);
int b200rl_normal_proj_bwd(const float* m_raw, const float* s_raw, const float* amin,
                           const float* amax, const float* dloc, const float* dscale, int64_t N,
                           int64_t A, float* dm_raw, float* ds_part, void* stream);
/* out[c] = scale * sum_r f(x[r,c]), f = identity or (x - center[c])^2 — the two passes of
 * tf.nn.moments (ppo_agent.py:100-110) and of the streaming normaliser. Deterministic. */
int b200rl_colsum(const float* x, const float* center, int squared, int64_t rows, int64_t cols,
                  float scale, float* out, void* workspace, int64_t ws_bytes, void* stream);
/* tf.nn.batch_normalization without offset/scale: out = x*inv - mean*inv, inv = rsqrt(var+eps),
 * var = m2/count (count NULL: m2 is the variance); mean NULL -> 0; clip > 0 clips to +-clip
 * (utils/tensor_normalizer.py:134-205). */
int b200rl_normalize(const float* x, float* out, int64_t rows, int64_t cols, const float* mean,
                     const float* m2, const float* count, float eps, float clip, void* stream);
/* StreamingTensorNormalizer update: Chan merge + Kahan carry (tensor_normalizer.py:397-470). */
int b200rl_normalizer_update(float* count, float* avg, float* m2, float* carry,
                             const float* avg_a, const float* m2_a, float n_a, int64_t cols,
                             void* stream);
/* gamma * discount * (next_step_type != LAST) (ppo_agent.py:632-660). */
int b200rl_ppo_discounts(const float* discount, const int32_t* next_step_type, float gamma,
                         int64_t n, float* out, void* stream);
/* make_trajectory_mask (ppo_utils.py:35-59) times optional weights. */
int b200rl_ppo_weights(const int32_t* step_type, const float* ret, const float* adv,
                       const float* weights, int64_t n, float* out, void* stream);

/* ------------------------------------------------------------------------------------
 * SAC update math — agents/sac/sac_agent.py, sac/tanh_normal_projection_network.py,
 * distributions/utils.py (SquashToSpecNormal), distributions/tanh_bijector_stable.py
 * ------------------------------------------------------------------------------------ */
/* _actions_and_log_probs (sac_agent.py:537-557) for the tanh-Normal policy: head [N, 2A] =
 * (loc | log_std); u = loc + exp(log_std)*eps, action = tanh-squash of u to [amin, amax] (written
 * with row stride ld_action), logp = log pi(action).  eps_in (oracle mode) or Philox+Box-Muller
 * (rng_call_dev uint64[2]).  u_out / eps_out (optional) are saved for the backward. */
int b200rl_sac_sample(const float* head, int64_t N, int64_t A, const float* amin,
                      const float* amax, const float* eps_in, uint64_t seed,
                      uint64_t* rng_call_dev, float* action, int64_t ld_action, float* logp,
                      float* u_out, float* eps_out, void* stream);
/* dL/dhead from dL/daction (da1 + da2, [N, ld_da] views, either may be NULL) and dL/dlogp. */
int b200rl_sac_sample_bwd(const float* head, const float* u_saved, const float* eps_saved,
                          const float* amin, const float* amax, const float* da1,
                          const float* da2, int64_t ld_da, const float* dlogp, int64_t N,
                          int64_t A, float* dhead, void* stream);
/* critic_loss (sac_agent.py:559-643) with squared TD error: y = rs*r + gamma*d*(min(tq1,tq2) -
 * exp(log_alpha)*next_logp); loss = loss_weight * sum(w*((y-q1)^2 + (y-q2)^2)) / global_batch. */
int b200rl_sac_critic_loss(const float* q1, const float* q2, const float* tq1, const float* tq2,
                           const float* next_logp, const float* reward, const float* discount,
                           const float* weights, const float* log_alpha_dev, int64_t B,
                           float gamma, float reward_scale, float loss_weight,
                           float global_batch, float* loss, float* dq1, float* dq2,
                           float* td_targets, int32_t* nan_flag, void* stream);
/* actor_loss (sac_agent.py:645-694): sum(w*(exp(log_alpha)*logp - min(q1,q2))) / global_batch. */
int b200rl_sac_actor_loss(const float* q1, const float* q2, const float* logp,
                          const float* weights, const float* log_alpha_dev, int64_t B,
                          float loss_weight, float global_batch, float* loss, float* dlogp,
                          float* dq1, float* dq2, int32_t* nan_flag, void* stream);
/* alpha_loss (sac_agent.py:696-739). */
int b200rl_sac_alpha_loss(const float* logp, const float* weights, const float* log_alpha_dev,
                          int64_t B, float target_entropy, int use_log_alpha, float loss_weight,
                          float global_batch, float* loss, float* dlog_alpha, int32_t* nan_flag,
                          void* stream);
/* out[N, da+db] = (a[N, :da] | b[N, :db]) — the critic's concat(observation, action) input
 * (agents/ddpg/critic_network.py:163-178). */
int b200rl_concat2(const float* a, int64_t lda, int64_t da, const float* b, int64_t ldb,
                   int64_t db, int64_t N, float* out, void* stream);

/* ------------------------------------------------------------------------------------
 * Network layers (fp32).  Replace Keras Dense/Conv2D fwd+bwd that the reference executes
 * through TensorFlow (networks/encoding_network.py:224-312, q_network.py:126-135).
 * All matrices are row-major.
 * ------------------------------------------------------------------------------------ */
/* GEMM engine for every dense / conv entry point below: 0 = fp32 FFMA register-tiled kernel,
 * 1 = tcgen05 tensor cores with the 3xTF32 split (fp32-grade accuracy, TMEM accumulators),
 * 2 = tcgen05 single-pass TF32 (~1e-3 relative; NOT within the 1e-5 parity bar).
 * Default: env B200RL_GEMM_MODE, else 1.  In modes 1 and 2 a GEMM takes the tensor cores when
 * N >= 16, M >= 32, K >= 8 and both operands can be read as aligned 16-byte chunks (reduction
 * length and leading dimensions multiples of 4, 16-byte aligned bases; uint8 conv inputs with
 * KW*C, stride*C, W*C and the image stride multiples of 16); every other GEMM runs on the FFMA
 * kernel.  Heads of <= 16 outputs and inputs of <= 32 features have kernels of their own in
 * modes 1 and 2. */
int b200rl_set_gemm_mode(int mode);
/* Tensor-core GEMM kernel (tc2_gemm.cuh) switches.  bit 0: store an explicitly masked TF32 "hi"
 * plane instead of using the raw fp32 operand tile for it (the tensor core ignores the low 13
 * mantissa bits; both settings are bit-identical, the default saves the store).  bit 1: unused.
 * bit 2: load plain 2-D operands with cp.async like the im2col views instead of TMA tensor
 * tiles.  bits 3-5: timing ablations (profiles/tc2_ablate.py; results are garbage).  bit 6: poll
 * mbarriers with test_wait instead of try_wait.  B200RL_TC2_FLAGS in the environment sets the
 * initial value. */
int b200rl_set_tc2_flags(int flags);
/* Work distribution of the persistent tcgen05 GEMM: 0 (default) static striding over the CTAs,
 * 1 dynamic (global tile counter) -- set by the data-parallel Learner (train/learner.py:104-143 in
 * the reference is where the strategy is attached) so that CTAs whose SM is held by the gradient
 * all-reduce take fewer tiles; B200RL_TILE_SCHED=0/1 in the environment sets the initial value. */
int b200rl_set_tile_scheduler(int dynamic);
/* Profiling aid: CTA 0 of every tc2 GEMM stamps %globaltimer at the start/end of each pipeline
 * step of each role into dev_buf[4 roles][256 steps][2] (int64); NULL switches it off. */
int b200rl_tc2_trace_buffer(long long* dev_buf);

/* Y[M,N] = act(X[M,K] @ W[K,N] + bias[N]).  ldx = row stride of X in elements (0 -> K), so a
 * [B,T,K] batch can be read at a fixed t without a copy.  workspace: device scratch of
 * ws_bytes (may be NULL when ws_bytes==0; then split-K is disabled). */
int b200rl_dense_fwd(const float* X, int64_t ldx, const float* W, const float* bias, float* Y,
                     int64_t M, int64_t K, int64_t N, int act, void* workspace,
                     int64_t ws_bytes, void* stream);
/* Two dense layers of identical shape (X1 @ W1 + b1 -> Y1, X2 @ W2 + b2 -> Y2; biases both given
 * or both NULL) in ONE launch of the persistent tensor-core kernel; two launches when that kernel
 * does not take the shape.  DqnAgent evaluates the online network on obs[:, 0] and the target
 * network on obs[:, T-1] this way (agents/dqn/dqn_agent.py:488-520, :575-579 in the reference are
 * the two independent forward passes).  Workspace as b200rl_dense_fwd (split-K needs room for both). */
int b200rl_dense_fwd_pair(const float* X1, const float* X2, int64_t ldx, const float* W1,
                          const float* W2, const float* bias1, const float* bias2, float* Y1,
                          float* Y2, int64_t M, int64_t K, int64_t N, int act, void* workspace,
                          int64_t ws_bytes, void* stream);
/* Given dY[M,N] (already multiplied by act'), compute dX[M,K] (optional, NULL to skip),
 * dW[K,N] (optional) and db[N] (optional).  accumulate!=0 adds into dW/db instead of
 * overwriting.  x_act: activation code of the layer whose OUTPUT is X (B200RL_ACT_NONE when X is
 * a raw input): dX is then multiplied by act'(X) in the GEMM epilogue, i.e. it is the gradient
 * w.r.t. that layer's pre-activation and no b200rl_act_bwd pass is needed (Keras composes
 * Dense(activation=...) the same way, networks/encoding_network.py:287-300).  In tensor-core
 * mode db is accumulated by the operand producers of the dW GEMM (no separate column-sum
 * launches; B200RL_FUSE_BIAS_GRAD=0 restores them). */
int b200rl_dense_bwd(const float* X, int64_t ldx, const float* W, const float* dY, float* dX,
                     float* dW, float* db, int64_t M, int64_t K, int64_t N, int accumulate,
                     int x_act, void* workspace, int64_t ws_bytes, void* stream);
/* dZ = dY * act'(Y) element-wise (in place allowed). */
int b200rl_act_bwd(const float* Y, const float* dY, float* dZ, int64_t n, int act,
                   void* stream);

/* conv2d, NHWC, VALID padding, square stride.  X is [N,H,W,C] f32, or u8 when x_is_u8
 * (then each element is converted to f32 and DIVIDED by x_scale — the reference's
 * cast+/255 preprocessing layer, examples/dqn/mnih15/dqn_train_eval_atari.py:104).
 * Wt is [KH,KW,C,F] (Keras HWIO), Y is [N,OH,OW,F]. */
typedef struct {
  int32_t N, H, W, C, KH, KW, F, stride;
  int64_t x_batch_stride; /* elements between consecutive images of X (0 -> H*W*C) */
} b200rl_conv_t;
int b200rl_conv2d_fwd(const void* X, int x_is_u8, float x_scale, const float* Wt,
                      const float* bias, float* Y, const b200rl_conv_t* g, int act,
                      void* workspace, int64_t ws_bytes, void* stream);
/* Two convolutions of identical geometry in one launch (see b200rl_dense_fwd_pair). */
int b200rl_conv2d_fwd_pair(const void* X1, const void* X2, int x_is_u8, float x_scale,
                           const float* Wt1, const float* Wt2, const float* bias1,
                           const float* bias2, float* Y1, float* Y2, const b200rl_conv_t* c,
                           int act, void* workspace, int64_t ws_bytes, void* stream);
/* dX, dW and db may each be NULL (that gradient is skipped), so the parameter gradients and the
 * input gradient of one layer can be issued on different streams.  x_act as in
 * b200rl_dense_bwd: the col2im scatter-add is linear, so act'(X) is applied to every
 * contribution at its destination element. */
int b200rl_conv2d_bwd(const void* X, int x_is_u8, float x_scale, const float* Wt,
                      const float* dY, float* dX, float* dW, float* db,
                      const b200rl_conv_t* g, int accumulate, int x_act, void* workspace,
                      int64_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Optimisers and target updates on flat fp32 parameter buffers.
 * ------------------------------------------------------------------------------------ */
/* TF Adam (tf.compat.v1.train.AdamOptimizer / Keras Adam):
 *   t = ++(*step_dev); lr_t = lr*sqrt(1-b2^t)/(1-b1^t);
 *   m = b1*m+(1-b1)*g; v = b2*v+(1-b2)*g*g; p -= lr_t*m/(sqrt(v)+eps).
 * grad_scale multiplies g first (1.0 normally; used for global-norm clipping when
 * grad_scale_dev != NULL, in which case *grad_scale_dev is read on device). */
int b200rl_adam_tf(float* p, const float* g, float* m, float* v, int64_t n, float lr,
                   float b1, float b2, float eps, int64_t* step_dev,
                   const float* grad_scale_dev, void* stream);
/* TF RMSProp (tf.compat.v1.train.RMSPropOptimizer; Mnih'15 config
 * examples/dqn/mnih15/dqn_train_eval_atari.py:176-182): centered optional. */
int b200rl_rmsprop_tf(float* p, const float* g, float* ms, float* mg, float* mom, int64_t n,
                      float lr, float decay, float momentum, float eps, int centered,
                      const float* grad_scale_dev, void* stream);
/* soft_variables_update (utils/common.py:250-346): t = (1-tau)*t + tau*s, gated on device by
 * Periodically (utils/common.py:450-507): if period>1 the kernel does
 * c = ++(*counter_dev); update only when c % period == 0.  period<=1: always. */
int b200rl_soft_update(float* target, const float* source, int64_t n, float tau,
                       int64_t period, int64_t* counter_dev, void* stream);
/* Per-variable clip_by_norm (utils/eager_utils.py:227-246): segments given by
 * offsets[nseg+1] (device int64). */
int b200rl_clip_by_norm_segments(float* g, const int64_t* offsets_dev, int64_t nseg,
                                 float max_norm, void* stream);
/* tf.clip_by_global_norm scale factor: *scale_dev = clip/max(norm,clip); *norm_dev=norm. */
int b200rl_global_norm_scale(const float* g, int64_t n, float clip, float* scale_dev,
                             float* norm_dev, void* workspace, int64_t ws_bytes,
                             void* stream);
/* Generic helpers used by the host glue. */
int b200rl_add_scaled(float* dst, const float* src, int64_t n, float alpha, void* stream);
int b200rl_l2_sum(const float* x, int64_t n, float coef, float* out_accum, void* stream);
int b200rl_counter_add(int64_t* counter_dev, int64_t inc, void* stream);

/* Emission order of a tf.data-style `shuffle(buffer)` over a stream of n elements, as used by
 * PPOLearner's minibatch pipeline `cache().repeat(epochs).unbatch().shuffle(buffer).batch(mb)`
 * (train/ppo_learner.py:220-250).  A reservoir holds the first min(buffer, n) stream elements;
 * output i emits slot j = Philox4x32-10(counter=(i, call), key=seed) -> lo + u64 % fill and
 * refills that slot with the next stream element (or with the last slot once the stream is
 * exhausted).  HOST function (the reference's input pipeline is host-side too): out_host[n]
 * receives stream indices; the rows themselves are gathered on the device
 * (b200rl_rb_read_rows).  The reference leaves the order unpinned (tf.data RNG). */
int b200rl_shuffle_order(int64_t n, int64_t buffer, uint64_t seed, uint64_t call,
                         int64_t* out_host);

/* ------------------------------------------------------------------------------------
 * Collect — environments + policies
 * ------------------------------------------------------------------------------------ */
/* EpsilonGreedyPolicy._action (policies/epsilon_greedy_policy.py:120-145) over
 * GreedyPolicy(QPolicy) (greedy_policy.py:70-89, q_policy.py:150-194):
 *   a = (u >= eps) ? argmax_a q[b,a] (masked) : uniform{0..A-1 | mask}.  u, random action from
 *   Philox (seed, *rng_call_dev, element b); when u_dev/rand_dev are non-NULL they are used
 *   instead (oracle mode). */
int b200rl_epsilon_greedy(const float* q, const int32_t* mask, int64_t B, int64_t A, float eps,
                          uint64_t seed, uint64_t* rng_call_dev, const float* u_dev,
                          const int32_t* rand_dev, int32_t* out_action, void* stream);

/* RandomTFEnvironment-style synthetic env (environments/random_tf_environment.py:96-129)
 * with per-env termination and the TFEnvironment auto-reset contract
 * (environments/tf_environment.py:211-241; trajectories/time_step.py:135-195):
 *   if step_type[b]==LAST: -> FIRST, reward 0, discount 1, fresh obs
 *   else: reward~U[0,1), terminate w.p. p_term -> LAST/discount 0 else MID/discount 1.
 * obs is [B, obs_bytes] u8 (uniform 0..255) when obs_is_u8 else [B, obs_elems] f32 ~ N(0,1).
 * State (step_type) is read and written in place; out_step_type (optional) receives a copy of
 * the new step types so the caller can ping-pong its TimeStep output buffers. */
int b200rl_env_random_step(int32_t* step_type, int32_t* out_step_type, void* obs,
                           int64_t obs_elems, int obs_is_u8, float* reward, float* discount,
                           int64_t B, float p_term, uint64_t seed, uint64_t* rng_call_dev,
                           void* stream);

/* Vectorised CartPole-v1 dynamics (gym classic_control formulae; the reference loads it via
 * suite_gym, agents/dqn/examples/v2/train_eval.py:151): state[B,4] f32, steps[B] int32. */
int b200rl_env_cartpole_step(float* state, int32_t* steps, int32_t* step_type,
                             const int32_t* action, float* obs, float* reward, float* discount,
                             int64_t B, int32_t max_steps, uint64_t seed,
                             uint64_t* rng_call_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200RL_H_ */
