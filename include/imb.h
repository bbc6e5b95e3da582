/* imb.h -- C ABI of libimb.so: the B200-native (sm_100a) GAIL/AIRL inner loop.
 *
 * The reference (HumanCompatibleAI/imitation) has no FFI/plugin registry; its boundary
 * for this path is the Python class API (SURVEY.md section 8b).  This header is the C-ABI
 * that sits directly under our Python mirror of that API (imitation_b200/): every entry
 * point below names the reference function(s) it replaces (paths relative to
 * /root/reference/src/imitation).  INTEGRATION.md shows the ctypes stub a maintainer
 * would add to the reference to call these.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer owned by the caller
 *    (e.g. torch tensor .data_ptr()); nothing is allocated or freed inside the library;
 *  - every call is asynchronous on `stream` (a cudaStream_t passed as void*), never
 *    synchronises, and is CUDA-graph capturable; per-call scalars that change from call to
 *    call live in the device-resident `imb_state` block so captured graphs can be replayed;
 *  - return value: 0 = ok, <0 = error (imb_last_error() gives the text, thread-local);
 *  - float32 arithmetic throughout; indices are int64 on the API, done masks uint8.
 *
 * Data layouts in HBM
 *  - transition TABLE (expert set, generator ring): AoS rows, row-major [capacity][tw],
 *    row = [obs(d_obs) | act(d_act; Discrete -> one-hot) | next_obs(d_obs) | done(1)],
 *    tw = 2*d_obs + d_act + 1.  Random row gathers read whole contiguous rows.
 *  - disc BATCH: SoA / feature-major [bw][ld], bw = tw + 1 (last feature row = log pi(a|s)),
 *    ld = row count rounded up to IMB_TILE_ROWS (padding zero).  Streaming kernels read it
 *    in [feature][128-row] tiles staged into shared memory by cp.async.bulk (TMA unit).
 *  - ROLLOUT table (PPO): row-major [E*T][rw], row index = env*T + step,
 *    row = [obs(d_obs) | act(da_store) | logp | value | reward | adv | ret].
 *  - parameters: one flat fp32 vector per network in torch nn.Linear order
 *    (weight [out][in] row-major, then bias), so nn.Parameters can alias it.
 */
#ifndef IMB_H_
#define IMB_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IMB_TILE_ROWS 128
#define IMB_MAX_HIDDEN 64   /* hidden widths 1..64, at most 2 hidden layers */
#define IMB_MAX_DIN 64      /* MLP input width 1..64 */
#define IMB_F_ZERO_GRAD 1    /* imb_disc_fwd_bwd: clear the gradient accumulator first */
#define IMB_F_TRAIN_NORM 2   /* imb_disc_fwd_bwd: Phi(s') uses the mid-update norm snapshot */
#define IMB_F_NO_TENSOR 4    /* imb_disc_fwd_bwd: force the fp32-FFMA kernel (A/B measurements; default = tcgen05 when the shape fits) */
#define IMB_RF_DETERMINISTIC 1 /* imb_rollout flags: act = mean / argmax (policy.predict(deterministic=True)) */

/* One MLP: [RunningNorm?] -> Linear(din,h1) -> act -> [Linear(h1,h2) -> act] -> Linear(h_last,n_out).
 * util/networks.py:204-283 (build_mlp).  Parameter block (at `param_off` floats into the
 * owning flat vector): W1[h1][din] b1[h1] W2[h2][h1] b2[h2] Wf[n_out][h_last] bf[n_out].  */
typedef struct imb_mlp {
  int32_t din;
  int32_t n_hidden;   /* 0, 1 or 2 */
  int32_t h1, h2;
  int32_t n_out;      /* 1 for reward/potential/value nets; d_act for the policy head */
  int32_t has_norm;   /* RunningNorm input layer (util/networks.py:98-134) */
  int32_t param_off;  /* float offset of this MLP's block in the flat parameter vector */
  int32_t norm_off;   /* float offset of [mean(din) | var(din)] in the norm-state vector */
  int32_t count_idx;  /* index of this norm's int32 count in the norm-count vector */
  float norm_eps;     /* 1e-5 */
} imb_mlp;

/* Discriminator / reward network description.
 * rewards/reward_nets.py:383-457 (BasicRewardNet), :674-736 (ShapedRewardNet),
 * :739-839 (BasicShapedRewardNet/BasicPotentialMLP); adversarial/gail.py:135-160,
 * adversarial/airl.py:67-119 (logit = r - log pi). */
typedef struct imb_disc_desc {
  int32_t d_obs, d_act;                       /* flattened widths (Discrete -> one-hot width) */
  int32_t use_state, use_action, use_next_state, use_done;
  imb_mlp base;
  int32_t shaped;                             /* 1: + gamma*(1-done)*Phi(s') - Phi(s) */
  imb_mlp potential;
  float gamma;
  int32_t subtract_logp;                      /* AIRL */
  int32_t n_params;                           /* total floats in the flat parameter vector */
} imb_disc_desc;

/* Adam hyper-parameters (torch.optim.Adam defaults: adversarial/common.py:123).  weight_decay > 0 = torch.optim.AdamW's
 * decoupled decay, param *= 1 - lr * weight_decay before the step (the reward trainer of preference comparisons,
 * algorithms/preference_comparisons.py:1182-1185); 0 = plain Adam. */
typedef struct imb_adam {
  float lr, beta1, beta2, eps, weight_decay;
} imb_adam;

/* Device-resident counters (int64 words) so that captured graphs replay correctly. */
enum {
  IMB_ST_RING_IDX = 0,    /* data/buffer.py Buffer._idx */
  IMB_ST_RING_N = 1,      /* Buffer._n_data */
  IMB_ST_EP_STEP = 2,     /* steps since the (lock-step) episode start */
  IMB_ST_EPISODE = 3,     /* episode counter (Philox reset stream) */
  IMB_ST_GLOBAL_STEP = 4, /* env steps taken per env since construction (noise stream) */
  IMB_ST_REPLAY_DRAW = 5, /* replay-sample draw counter */
  IMB_ST_EXPERT_POS = 6,  /* position inside the current expert permutation */
  IMB_ST_EXPERT_EPOCH = 7,
  IMB_ST_PPO_EPOCH = 8,   /* PPO permutation draw counter */
  IMB_ST_DISC_STEP = 9,   /* Adam step count of the discriminator */
  IMB_ST_PPO_STEP = 10,   /* Adam step count of the policy */
  IMB_ST_WORDS = 16
};

int imb_version(void);
const char* imb_last_error(void);
/* number of floats of workspace the discriminator kernels need (partials, accumulators) */
int64_t imb_disc_workspace_floats(const imb_disc_desc* d);

/* ---- stage 3: discriminator ------------------------------------------------------------ */

/* RunningNorm.update_stats on a feature-major batch (util/networks.py:111-134; order of
 * operations BaseNorm.forward :79-91).  For a shaped net the potential norm is updated twice
 * (next_obs rows, then obs rows; SURVEY Appendix A.5) and the intermediate stats are kept in
 * `ws` for the forward pass.  batch: [bw][ld], rows [0,n) valid. */
int imb_disc_norm_update(const imb_disc_desc* d, const float* batch, int64_t ld, int64_t n,
                         float* norm_state, int32_t* norm_count, float* ws, void* stream);

/* RunningNorm.update_stats (util/networks.py:111-134) over `din` consecutive feature rows [row0, row0 + din) of a
 * feature-major batch, for a normaliser that is NOT the discriminator's own: the generator policy's
 * NormalizeFeaturesExtractor, which the reference updates as a side effect of `policy.evaluate_actions` on every
 * discriminator minibatch (algorithms/adversarial/common.py:606-615 with the policy left in train mode by SB3's
 * PPO.train).  defer == NULL: fold into (norm_state = [mean | var], norm_count) immediately.  defer != NULL: append the
 * batch moments to the slot list `defer` ([0] = number of slots in use, [4 + k * (2 din + 1) ...] = mean | var | n) so that
 * the update can be computed on a stream that runs beside the PPO update and applied afterwards, in order, by
 * imb_norm_fold.  `d` / `ws`: any discriminator descriptor + its workspace (chunk partials live there). */
int imb_norm_batch_stats(const imb_disc_desc* d, const float* batch, int64_t ld, int64_t n, int row0, int din,
                                 float* norm_state, int32_t* norm_count, float* defer, int defer_cap, float* ws,
                                 void* stream);
int imb_norm_fold(int din, float* defer, float* norm_state, int32_t* norm_count, int n_slots /* <= 0: the list's own
                  counter, which is then reset; > 0: exactly that many slots (an all-gathered list), no reset */,
                  void* stream);
/* `train_disc` returns Mapping[str, float] (common.py:79-92): copy the n <= 15 statistics into HOST-MAPPED pinned memory
 * (16 floats) and then store the current value of state[state_idx] (the Adam step) as int32 into word 15; the host polls that
 * word -- no D2H memcpy, no event synchronisation on the critical path of the synchronous API. */
int imb_stats_publish(const float* stats_dev, int n, float* host_mapped, const int64_t* state, int state_idx, void* stream);
/* multi-GPU discriminator step (SURVEY 8e): after the [gradient | statistic sums] block at the start of the workspace
 * (n_params rounded up to 32 floats, then 5 sums) has been all-reduced over the ranks, record the GLOBAL row counts that
 * imb_disc_adam's statistics divide by (common.py:52-77 over the global 2 * minibatch rows). */
int imb_disc_set_rows(const imb_disc_desc* d, float* ws, int64_t n_rows_total, int64_t n_expert_total, void* stream);

/* Fused forward + BCE-with-logits + backward over one minibatch of n = 2*mb rows (expert rows
 * first: label 1, generator rows second: label 0), gradients ACCUMULATED into ws (scaled by
 * loss_scale = 1/(2*B), common.py:360-369).  Replaces RewardNet.forward + F.binary_cross_
 * entropy_with_logits + loss.backward() (common.py:353-369).  If grad_out != NULL the BCE is
 * skipped and grad_out[n] is used as dL/dlogit (autograd backward of RewardNet.forward).
 * logits_out[n] (optional) receives the logits.  flags: IMB_F_ZERO_GRAD clears the accumulator
 * first (common.py:346); IMB_F_TRAIN_NORM = the norm stats were just updated by
 * imb_disc_norm_update (training mode). */
int imb_disc_fwd_bwd(const imb_disc_desc* d, const float* params, const float* norm_state,
                     const float* batch, int64_t ld, int64_t n, int64_t n_expert,
                     float loss_scale, const float* grad_out, float* logits_out,
                     int flags, float* ws, void* stream);

/* Finish the update: deterministic reduction of the per-CTA partials, optional copy of the
 * gradient to grad_out_flat (for external optimisers / all-reduce), optional Adam step
 * (common.py:372) and the 9 train stats of the LAST minibatch (common.py:27-92) into
 * stats_out[16] = {loss, acc, acc_expert, acc_gen, entropy, prop_expert_true,
 * prop_expert_pred, n_expert, n_generated}.  state[IMB_ST_DISC_STEP] is incremented. */
int imb_disc_reduce(const imb_disc_desc* d, float* ws, float* grad_out_flat, void* stream);
int imb_disc_adam(const imb_disc_desc* d, const imb_adam* opt, float* params, float* exp_avg,
                  float* exp_avg_sq, const float* grad_flat_or_null, float grad_div, float* ws,
                  int64_t* state, float* stats_out, void* stream);

/* Forward only (RewardNet.predict_th in eval mode, reward_nets.py:120-153; out_mode 0 = raw
 * net output, 1 = logits (AIRL subtracts log pi), 2 = GAIL reward -logsigmoid(-x),
 * gail.py:83). */
int imb_reward_forward(const imb_disc_desc* d, const float* params, const float* norm_state,
                       const float* batch, int64_t ld, int64_t n, int out_mode, float* out,
                       void* stream);

/* NormalizedRewardNet.predict_processed over T consecutive env steps of E rewards
 * (reward_nets.py:637-671): normalise step t with the running stats, THEN merge step t. */
int imb_reward_norm_scan(float* rews, int64_t n_envs, int64_t n_steps, int64_t step_stride,
                         int64_t env_stride, float* norm_state2, int32_t* norm_count, float eps,
                         int update_stats, void* stream);

/* ---- stage 2: tables, ring buffer, sampling --------------------------------------------- */

/* Build AoS table rows from separate row-major arrays (ReplayBuffer.store, data/buffer.py:
 * 397-412, Buffer.store :147-214 with truncate_ok).  acts_f (float [n][d_act]) or acts_i
 * (int64 [n], one-hot encoded, RewardNet.preprocess reward_nets.py:88-111).  Rows are written
 * at ring positions (state[RING_IDX] + i) mod capacity for the LAST min(n,capacity) rows;
 * use_ring = 0 writes rows at i (expert table).  Ring header advanced by imb_ring_advance. */
int imb_table_store(float* table, int64_t capacity, int32_t d_obs, int32_t d_act,
                    const float* obs, const float* acts_f, const int64_t* acts_i,
                    const float* next_obs, const uint8_t* dones, int64_t n, int use_ring,
                    const int64_t* state, void* stream);
int imb_ring_advance(int64_t* state, int64_t capacity, int64_t n_stored, void* stream);

/* Index generation on device ("perf mode"; parity mode uploads host indices instead).
 * kind 0: with replacement in [0, state[RING_N]) -- Buffer.sample, buffer.py:216-232;
 * kind 1: next n entries of an endless sequence of Feistel permutations of [0,size) with
 * drop_last semantics -- make_data_loader(shuffle, drop_last) + endless_iter,
 * algorithms/base.py:272-282, util/util.py:215-241. */
int imb_sample_indices(int kind, int64_t* idx_out, int64_t n, int64_t size, uint64_t seed,
                       int64_t* state, void* stream);

/* Device sampling + gather of one discriminator minibatch in ONE launch: batch columns [0, mb) =
 * expert rows drawn like imb_sample_indices(kind 1), columns [mb, 2 mb) = generator-ring rows drawn
 * like kind 0, both at offset `start` of the update's draws (common.py:552 `sample` + :592-595
 * concatenate + the DataLoader batch of :208-216).  The draw counters advance once per update:
 * imb_sample_advance2(demo_batch_size, ...).  Bit-identical to the unfused calls. */
int imb_disc_sample_gather(const float* expert_table, int64_t n_expert, const float* ring,
                           int64_t ring_capacity, int32_t tw, int64_t mb, int64_t start,
                           uint64_t seed, const int64_t* expert_state, const int64_t* ring_state,
                           float* batch, int64_t ld, void* stream);
int imb_sample_advance2(int64_t n, int64_t n_expert, int64_t* expert_state, int64_t* ring_state,
                        void* stream);

/* Gather table rows by index into the feature-major batch at column col0 (idx == NULL ->
 * rows 0..n-1).  A warp loads 32 indices coalesced, then walks them by warp shuffle so that
 * each row is read by consecutive lanes; the 32x tw tile is transposed through shared memory
 * so batch writes are coalesced too.  Buffer.sample gather (buffer.py:231-232) + the
 * concatenate of common.py:592-595. */
int imb_gather_rows(const float* table, int64_t capacity, int32_t tw, const int64_t* idx,
                    int64_t n, float* batch, int64_t ld, int64_t col0, void* stream);

/* ---- stage 1: generator rollouts (GPU-resident VecEnv + policy + reward relabel) ---------- */

/* Actor-critic policy (SB3 ActorCriticPolicy with separate pi / vf towers, tanh;
 * imitation policies/base.py:92-104 FeedForward32Policy; optional feature RunningNorm,
 * policies/base.py:123-149).  Flat parameter vector: pi tower | vf tower | action head
 * (imb_mlp with n_hidden = 0 semantics: Linear(h, d_act)) | value head | log_std[d_act]. */
typedef struct imb_policy_desc {
  int32_t d_obs, d_act;     /* d_act: action dim (Box) or number of actions (Discrete) */
  int32_t discrete;
  int32_t hidden;           /* tower width (two tanh layers of this width) */
  int32_t has_norm;         /* NormalizeFeaturesExtractor */
  float norm_eps;
  int32_t off_pi_w1, off_pi_b1, off_pi_w2, off_pi_b2;
  int32_t off_vf_w1, off_vf_b1, off_vf_w2, off_vf_b2;
  int32_t off_act_w, off_act_b, off_val_w, off_val_b, off_log_std;
  int32_t n_params;
} imb_policy_desc;

/* Synthetic MuJoCo-shaped environment (defined by this repo, SURVEY section 8d):
 * obs' = tanh(A obs + Bm u + c), reward = w.obs' - 0.1|u|^2, fixed horizon, auto-reset. */
typedef struct imb_env_desc {
  int32_t d_obs, d_act, discrete, horizon;
  uint64_t seed;
  int64_t env_id_offset;    /* global id of this rank's env 0 (multi-GPU sharding) */
} imb_env_desc;

typedef struct imb_ppo_hparams {
  float gamma, gae_lambda, clip_range, ent_coef, vf_coef, max_grad_norm, lr, adam_eps;
  int32_t n_epochs, batch_size, normalize_advantage;
} imb_ppo_hparams;

/* One generator rollout of T steps for E envs in ONE launch (thread per env): policy
 * forward + sampling (OnPolicyAlgorithm.collect_rollouts), env step with auto-reset and
 * terminal-observation handling (data/wrappers.py:69-91, data/rollout.py:120-187), learned
 * reward relabel on (old_obs, clipped act, terminal-fixed next obs, done)
 * (rewards/reward_wrapper.py:92-133 -> RewardNet.predict_processed), time-limit bootstrap,
 * rollout rows, GAE, and the flattened transition rows in reference order
 * (pop_trajectories + flatten_trajectories, wrappers.py:132-148, rollout.py:563-621) written
 * straight into the generator ring with Buffer.store truncation (buffer.py:174-192).
 * reward_mode: 0 = env reward (debug_use_ground_truth), 1 = GAIL -logsigmoid(-logit),
 * 2 = raw reward-net output (AIRL; normalise afterwards with imb_reward_norm_scan).
 * noise (optional, [T][E][d_act] normals or [T][E] uniforms) pins sampling for parity;
 * flags: IMB_RF_DETERMINISTIC for evaluation rollouts (data/rollout.py:382-506). */
int imb_rollout(const imb_env_desc* env, const float* env_params, float* env_obs,
                const imb_policy_desc* pol, const float* pol_params, const float* pol_norm,
                const imb_disc_desc* disc, const float* disc_params, const float* disc_norm,
                int reward_mode, const imb_ppo_hparams* hp, int64_t n_envs, int64_t n_steps,
                float* rollout, float* ring, int64_t ring_capacity, float* flat_out, float* aux,
                const float* noise, int flags, const int64_t* state, void* stream);
/* floats per rollout row: d_obs + (discrete ? 1 : d_act) + 5 (logp, value, reward, adv, ret), padded
 * to a multiple of 4 (16-byte aligned rows: imb_ppo_update stages each minibatch row with one bulk copy);
 * aux needs 2*E + 2*E*T floats (V(last obs), last done, per-step time-limit bootstrap,
 * per-step ground-truth env reward). */
int imb_rollout_row_width(const imb_policy_desc* pol);
/* GAE over the rollout table once rewards are final (SB3 RolloutBuffer.compute_returns_and_
 * advantage); call BEFORE imb_rollout_advance (it needs the pre-rollout episode step). */
int imb_gae(float* rollout, int32_t rw, int32_t col_value, int64_t n_envs, int64_t n_steps,
            const float* aux, float gamma, float gae_lambda, const int64_t* state_before,
            int32_t horizon, void* stream);
/* advance EP_STEP/EPISODE/GLOBAL_STEP (+ ring header when ring_capacity > 0) after a rollout */
int imb_rollout_advance(int64_t* state, int64_t n_envs, int64_t n_steps, int32_t horizon,
                        int64_t ring_capacity, void* stream);
/* VecEnv.reset(): env_obs[d_obs][E] = 0.1 * N(0,1) from Philox(seed, env id, episode). */
int imb_env_reset(float* env_obs, int64_t n_envs, const imb_env_desc* env, const int64_t* state,
                  void* stream);

/* PPO.train as ONE persistent launch of an 8-CTA thread-block cluster: n_epochs x (N/batch)
 * sequential minibatch steps (gather by permutation, evaluate_actions, clipped surrogate + value +
 * entropy loss, backward, clip_grad_norm_, Adam).  Two kernels behind this entry point: k_ppo_update for tower width <= 32
 * and batch_size <= 64 (the reference's FeedForward32Policy with SB3's default minibatch: the minibatch is resident in
 * shared memory, one lane per hidden unit), k_ppo_update_gen for tower widths up to 64 (SB3 MlpPolicy 64x64) and
 * minibatches up to 4096 rows (tuned_hps airl_seals_walker: 128, airl_seals_hopper: 512).  perm == NULL -> device Feistel
 * permutations.  loss_log (optional) [n_steps_total][4] = pg_loss, value_loss, entropy_loss, total. */
int imb_ppo_update(const imb_policy_desc* pol, float* pol_params, float* pol_norm,
                   int32_t* pol_norm_count, float* exp_avg, float* exp_avg_sq,
                   const float* rollout, int64_t n_rows, const imb_ppo_hparams* hp,
                   const int64_t* perm, uint64_t seed, float* loss_log, int64_t* state,
                   void* stream);

/* log pi(a|s) of the generator policy for the disc batch (common.py:476-519 ->
 * ActorCriticPolicy.evaluate_actions), written into the batch's last feature row. */
int imb_policy_logp(const imb_policy_desc* pol, const float* pol_params, const float* pol_norm,
                    float* batch, int64_t ld, int64_t n, int32_t row_logp, void* stream);

/* imb_disc_reduce + imb_disc_adam in one launch (last minibatch of an update; gradient taken from
 * the workspace accumulator). */
int imb_disc_reduce_adam(const imb_disc_desc* d, const imb_adam* opt, float* params, float* exp_avg,
                         float* exp_avg_sq, float grad_div, float* ws, int64_t* state,
                         float* stats_out, void* stream);

/* ---- preference comparisons (SURVEY 8 row f1) --------------------------------------------------
 * One minibatch of P fragment pairs of L transitions each: rews[2][P][L] are the reward network's outputs for the first
 * fragments, then the second fragments (row f * L + t).  PreferenceModel.probability (algorithms/preference_comparisons.py:
 * 487-530): d = clip(sum_t discount^t (r2 - r1), -threshold, threshold), p = noise_prob / 2 + (1 - noise_prob) / (1 + e^d);
 * CrossEntropyRewardLoss (:1043-1090): loss = mean_P BCE(p, pref) with torch's log clamp at -100, accuracy = mean((p > .5)
 * == (pref > .5)).  Outputs (each optional): grad_rews[2][P][L] = grad_scale * d loss / d rews (autograd's result, incl.
 * the zero gradient of clipped pairs and torch's BCE backward denominator clamp 1e-12) -- the upstream gradient for
 * imb_disc_fwd_bwd(grad_out=...); probs_out[P]; statistics slot `stats_slot` = the four floats at stats_acc + 4 * stats_slot:
 * [0] += loss, [1] += accuracy, [2] += 1 (so the per-minibatch means of an epoch -- one slot per epoch and per quantity
 * group -- are read back once).  The reference computes this with a Python loop over the pairs (:441-454). */
int imb_pref_loss(const float* rews, int64_t n_pairs, int32_t frag_len, const float* prefs, float noise_prob,
                  float discount, float threshold, float grad_scale, float* grad_rews, float* probs_out,
                  float* stats_acc, int32_t stats_slot, void* stream);

/* ---- multi-GPU: replica state around the ONE all-reduce of a round ---------------------------
 * (SURVEY.md section 8e; the reference is single-process, so there is no reference interface to
 * cite: the merge restates RunningNorm's Chan update, util/networks.py:96-134, in its additive
 * sufficient-statistics form).  avg[i] (avg_n[i] floats) are averaged over the ranks; norm i is
 * (mean[k], var[k], int32 count) and is merged exactly relative to the round-start snapshot.
 * Staging buffers are float64: buf has imb_sync_buffer_doubles() entries, start the norm part. */
#define IMB_SYNC_MAX_AVG 8
#define IMB_SYNC_MAX_NORM 4
typedef struct imb_sync_desc {
  int32_t n_avg, n_norm;
  float* avg[IMB_SYNC_MAX_AVG];
  int64_t avg_n[IMB_SYNC_MAX_AVG];
  float* mean[IMB_SYNC_MAX_NORM];
  float* var[IMB_SYNC_MAX_NORM];
  int32_t* count[IMB_SYNC_MAX_NORM];
  int32_t k[IMB_SYNC_MAX_NORM];
} imb_sync_desc;
int64_t imb_sync_buffer_doubles(const imb_sync_desc* d);
int imb_sync_snapshot(const imb_sync_desc* d, double* start, void* stream);
int imb_sync_pack(const imb_sync_desc* d, double* buf, void* stream);
int imb_sync_unpack(const imb_sync_desc* d, const double* buf, const double* start, int32_t world,
                    void* stream);

/* zero the device-resident counter block */
int imb_state_init(int64_t* state, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IMB_H_ */
