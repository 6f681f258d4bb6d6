/* pearl_b200.h — C ABI of libpearlb200.so: the B200-native learner hot path of
 * facebookresearch/Pearl (`ReplayBuffer.sample -> PolicyLearner.learn()`).
 *
 * Conventions
 *   - extern "C", plain ints / pointers / sizes; no C++ or torch types.
 *   - every entry point returns 0 on success or a negative PRL_E* code; the
 *     message for the calling thread is available from prl_last_error().
 *   - the CALLER (PyTorch in pearl_b200/, or any other host) allocates and owns
 *     every device buffer; the library owns only its opaque handles, a pinned
 *     staging area for host pushes and small workspaces.  Pointers registered
 *     by *_create / *_bind stay referenced until *_destroy.
 *   - all device work is enqueued on the `stream` argument (a cudaStream_t
 *     passed as void*; NULL = legacy default stream).  No hidden
 *     synchronisation except where stated.
 *   - one handle is used from one host thread at a time (thread-compatible).
 *
 * Each group cites the reference interface it replaces (paths relative to
 * /root/reference/pearl, commit 48f1fbb).
 */
#ifndef PEARL_B200_H
#define PEARL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PRL_OK 0
#define PRL_EINVAL (-1)    /* contract violation (reference raises ValueError / assert) */
#define PRL_ECUDA (-2)     /* CUDA runtime error */
#define PRL_ENOMEM (-3)
#define PRL_ESTATE (-4)    /* call not valid in the handle's current state */
#define PRL_EUNSUPPORTED (-5)

#define PRL_ABI_VERSION 1

/* ---- library ----------------------------------------------------------- */
int prl_abi_version(void);
/* Select `device` for the calling thread and check it is sm_100 (B200).
 * There is no CPU fallback: without a B200 this returns PRL_EUNSUPPORTED. */
int prl_init(int device);
const char *prl_last_error(void);
/* multiprocessor count of the current device (grid sizing, reported by bench) */
int prl_sm_count(void);

/* ---- replay buffer ------------------------------------------------------
 * Replaces BasicReplayBuffer / TensorBasedReplayBuffer
 * (replay_buffers/basic_replay_buffer.py:17-48,
 *  replay_buffers/tensor_based_replay_buffer.py:55-133,253-288).
 *
 * Storage is ONE caller-allocated device array of `capacity` fixed-size
 * records ("array of transitions": sampling touches whole random transitions,
 * so a transition is contiguous, 16-byte aligned, and moves with one bulk
 * copy).  Record layout in 32-bit words (see prl_buf_layout):
 *     [off_state      .. +obs_dim)   state        f32
 *     [off_next_state .. +obs_dim)   next_state   f32
 *     [off_action     .. +act_words) action       i32 (discrete) | f32[act_dim]
 *     [off_reward]                   reward       f32
 *     [off_flags]                    bit0 terminated, bit1 truncated,
 *                                    bits 8..23 number of next available actions
 *     [off_avail .. ) (PRL_BUF_DYNAMIC_ACTIONS only) n_actions u8 ids of the
 *                     next available actions (padded with 0), as the reference
 *                     pads `next_available_actions` (tensor_based_replay_buffer.py:179-251)
 * FIFO eviction like deque(maxlen=capacity): logical index 0 = oldest.
 */
#define PRL_BUF_DISCRETE 0x1          /* action is one int32 id in [0, n_actions) */
#define PRL_BUF_CONTINUOUS 0x2        /* action is act_dim floats */
#define PRL_BUF_DYNAMIC_ACTIONS 0x4   /* per-transition next-available-action sets */

typedef struct prl_buf_desc {
    int64_t capacity;
    int32_t obs_dim;
    int32_t act_dim;     /* continuous: action dimension; discrete: 1 */
    int32_t n_actions;   /* discrete: max_number_actions; continuous: 0 */
    int32_t flags;       /* PRL_BUF_* */
} prl_buf_desc;

typedef struct prl_buf_layout {
    int32_t record_words;   /* record stride in 32-bit words (multiple of 4) */
    int32_t off_state, off_next_state, off_action, off_reward, off_flags, off_avail;
    int32_t act_words;
    int64_t storage_bytes;  /* capacity * record_words * 4 */
} prl_buf_layout;

typedef struct prl_buf prl_buf;

int prl_buf_layout_of(const prl_buf_desc *desc, prl_buf_layout *out);
/* `storage_dev`: device memory of layout.storage_bytes bytes, 16-byte aligned.
 * `mt_state_dev`: device uint32[625], the MT19937 state in the layout of
 * CPython's random.getstate()[1] (624 words + position). */
int prl_buf_create(prl_buf **out, const prl_buf_desc *desc, void *storage_dev,
                   uint32_t *mt_state_dev);
int prl_buf_destroy(prl_buf *buf);
int64_t prl_buf_len(const prl_buf *buf);          /* __len__  (:284-285) */
int64_t prl_buf_capacity(const prl_buf *buf);
int64_t prl_buf_head(const prl_buf *buf);         /* physical slot of logical index 0 */
int prl_buf_clear(prl_buf *buf);                  /* clear()  (:287-288) */
/* Restore occupancy after the caller refilled `storage_dev` itself
 * (checkpoint load): `len` valid records, oldest at physical slot `head`. */
int prl_buf_set_occupancy(prl_buf *buf, int64_t len, int64_t head);

/* Multi-GPU: `buf` is rank `rank`'s shard of ONE logical replay buffer of `world * capacity` transitions
 * (SURVEY.md 8e; the reference has no sharded buffer — its BasicReplayBuffer is the world == 1 case,
 * basic_replay_buffer.py:21-48).  The transition with global write counter g lives on rank g mod world at
 * local slot (g div world) mod capacity, so FIFO eviction and age-uniform sampling stay balanced.
 * `global_pushed` = pushes to the logical buffer so far; the shard must hold exactly its share.  A sharded
 * buffer samples from the LOGICAL population: every rank runs the same MT19937 stream and draws the same
 * `batch` global indices as one GPU would (random.sample over the whole deque,
 * tensor_based_replay_buffer.py:276); prl_dqn_learn then works on the rows the rank owns. */
int prl_buf_set_shard(prl_buf *buf, int rank, int world, int64_t global_pushed);
int64_t prl_buf_global_len(const prl_buf *buf);

/* The same host push for `count` buffers of one record layout in ONE call (a vectorised environment feeding
 * a learner group): every source is a [count][n][...] host array; no per-transition action sets.  Records
 * are packed by a few worker threads and copied with one cudaMemcpyAsync per buffer. */
int prl_buf_push_host_multi(prl_buf *const *bufs, int count, int64_t n, const float *state, const void *action,
                            const float *reward, const float *next_state, const uint8_t *terminated,
                            const uint8_t *truncated, void *stream);

/* push n transitions given as HOST arrays (struct-of-arrays, C order):
 * state/next_state f32[n][obs_dim]; action int32[n] or f32[n][act_dim];
 * reward f32[n]; terminated/truncated u8[n]; next_avail_ids u8[n][n_actions]
 * and next_avail_cnt i32[n] (both NULL => all n_actions available).
 * Records are packed into the handle's pinned staging area and copied with
 * at most two cudaMemcpyAsync (ring wrap).  Replaces push() (:55-133) +
 * _store_transition (basic_replay_buffer.py:21-48), batched. */
int prl_buf_push_host(prl_buf *buf, int64_t n, const float *state, const void *action,
                      const float *reward, const float *next_state, const uint8_t *terminated,
                      const uint8_t *truncated, const uint8_t *next_avail_ids,
                      const int32_t *next_avail_cnt, void *stream);
/* same, sources already on the device (pack kernel, no host round trip) */
int prl_buf_push_device(prl_buf *buf, int64_t n, const float *state, const void *action,
                        const float *reward, const float *next_state, const uint8_t *terminated,
                        const uint8_t *truncated, const uint8_t *next_avail_ids,
                        const int32_t *next_avail_cnt, void *stream);

/* RNG state hand-off with CPython's global `random` module
 * (the reference samples with random.sample, tensor_based_replay_buffer.py:276;
 * state = random.getstate()[1]).  Host pointers, uint32[625].  get synchronises
 * `stream`. */
int prl_rng_set_state(prl_buf *buf, const uint32_t *state625_host, void *stream);
int prl_rng_get_state(prl_buf *buf, uint32_t *state625_host, void *stream);
/* random.seed(int): abs(seed) as little-endian 32-bit key words */
int prl_rng_seed(prl_buf *buf, const uint32_t *key_host, int key_len, void *stream);

/* Draw `rounds` consecutive samples of `k` distinct logical indices, exactly
 * the values `random.sample(range(len), k)` would return `rounds` times in a
 * row from the current MT19937 state (both CPython branches), advancing the
 * state.  out_logical_dev / out_slot_dev: device int32[rounds][k] (either may
 * be NULL); slot = physical record index.  PRL_EINVAL if k > len
 * (reference: ValueError, :271-275). */
int prl_buf_sample_indices(prl_buf *buf, int rounds, int k, int32_t *out_logical_dev,
                           int32_t *out_slot_dev, void *stream);

/* Gather k records into the reference's TransitionBatch field layout
 * (_create_transition_batch :290-400; dtypes of SURVEY.md §8 a4), all device
 * pointers, any of them may be NULL:
 *   state/next_state f32[k][obs_dim]; action i64[k] (discrete) or
 *   f32[k][act_dim]; reward f32[k]; terminated/truncated u8[k] (bool);
 *   next_avail f32[k][n_actions] (action ids, 0-padded);
 *   next_unavail_mask u8[k][n_actions] (1 = unavailable). */
int prl_buf_gather(const prl_buf *buf, const int32_t *slot_dev, int k, float *state, void *action,
                   float *reward, float *next_state, uint8_t *terminated, uint8_t *truncated,
                   float *next_avail, uint8_t *next_unavail_mask, void *stream);

/* ---- DQN / DoubleDQN learner ---------------------------------------------
 * Replaces DeepTDLearning.learn_batch + DeepQLearning / DoubleDQN
 * .get_next_state_values + VanillaQValueNetwork.get_q_values + AdamW(amsgrad)
 * + update_target_network, driven by PolicyLearner.learn's training_rounds
 * loop (policy_learners/policy_learner.py:162-195,
 * policy_learners/sequential_decision_making/deep_td_learning.py:269-360,
 * deep_q_learning.py:130-167, double_dqn.py:29-57,
 * neural_networks/sequential_decision_making/q_value_networks.py:152-174,
 * neural_networks/common/utils.py:214-226, torch/optim/adam.py).
 *
 * Network: VanillaQValueNetwork with two hidden layers,
 *   x = [state | one_hot(action)]  ->  Linear(H1) ReLU Linear(H2) ReLU Linear(1).
 * Parameters are ONE flat fp32 array in torch's own parameter order and
 * layout (nn.Linear weight [out][in] row-major, then bias):
 *   W1[H1][obs+A] b1[H1] W2[H2][H1] b2[H2] W3[1][H2] b3[1]
 * so the caller can expose views of it as the module's state_dict.
 */
typedef struct prl_dqn_cfg {
    int32_t obs_dim, n_actions, hidden1, hidden2;
    int32_t double_dqn;            /* 0: DeepQLearning, 1: DoubleDQN */
    int32_t target_update_freq;    /* soft update when (training_steps+1) % freq == 0 */
    int32_t max_batch;             /* largest batch learn()/learn_batch() will be given */
    int32_t max_rounds;            /* largest `rounds` per prl_dqn_learn call */
    int32_t rows_per_cta;          /* 0 = choose automatically */
    /* AdamW (amsgrad always on), discount, soft-update coefficient: doubles,
     * because the reference evaluates these scalars in Python floats */
    double lr, beta1, beta2, eps, weight_decay;
    double gamma, tau;
} prl_dqn_cfg;

typedef struct prl_dqn prl_dqn;

int64_t prl_dqn_param_count(const prl_dqn_cfg *cfg);
/* bytes of device workspace the caller must provide to prl_dqn_create */
int64_t prl_dqn_workspace_bytes(const prl_dqn_cfg *cfg);
/* w, w_target, exp_avg, exp_avg_sq, max_exp_avg_sq: device f32[param_count].
 * adam_step: number of optimizer steps already taken (torch's `step`). */
int prl_dqn_create(prl_dqn **out, const prl_dqn_cfg *cfg, float *w, float *w_target,
                   float *exp_avg, float *exp_avg_sq, float *max_exp_avg_sq, int64_t adam_step,
                   void *workspace_dev);
int prl_dqn_destroy(prl_dqn *dqn);
int64_t prl_dqn_adam_step(const prl_dqn *dqn);
int prl_dqn_set_adam_step(prl_dqn *dqn, int64_t step);
int prl_dqn_set_lr(prl_dqn *dqn, double lr);

/* PolicyLearner.learn(replay_buffer) for `rounds` training rounds in ONE call:
 * draws rounds x batch indices (bit-exact with random.sample), then runs a
 * persistent kernel that per round gathers the batch, applies the scheduled
 * soft target update, computes Q(s,a), the Bellman target, the MSE gradient,
 * and the AdamW(amsgrad) step.  `training_steps0` is the learner's
 * `_training_steps` BEFORE the call (round r uses training_steps0 + r + 1).
 * out_mae_dev: device f32[rounds], the reference's reported "loss"
 * (mean |q - y|, deep_td_learning.py:358-360).  Optional device outputs for
 * parity tests (NULL to skip): out_q / out_y f32[rounds][batch],
 * out_logical i32[rounds][batch].  Asynchronous on `stream`. */
int prl_dqn_learn(prl_dqn *dqn, prl_buf *buf, int rounds, int batch, int64_t training_steps0,
                  float *out_mae_dev, float *out_q_dev, float *out_y_dev,
                  int32_t *out_logical_dev, void *stream);

/* DeepTDLearning.learn_batch(batch) on a caller-supplied TransitionBatch
 * (PearlAgent.learn_batch / offline learning, pearl_agent.py:222-231): device
 * arrays in prl_buf_gather's output layout; next_avail / mask may be NULL
 * (all actions available).  `do_target_update` = the caller's evaluation of
 * (training_steps+1) % freq == 0.  out_mae_dev: f32[1]. */
int prl_dqn_learn_batch(prl_dqn *dqn, int batch, const float *state, const int64_t *action,
                        const float *reward, const float *next_state, const uint8_t *terminated,
                        const float *next_avail, const uint8_t *next_unavail_mask,
                        int do_target_update, float *out_mae_dev, float *out_q_dev,
                        float *out_y_dev, void *stream);

/* Q(s, a) for every action (act(): deep_td_learning.py:200-254): device
 * state f32[n][obs_dim] -> out_q f32[n][n_actions], online (target=0) or
 * target network. */
int prl_dqn_q_values(prl_dqn *dqn, int n, const float *state, int target, float *out_q_dev,
                     void *stream);

/* how the last prl_dqn_learn was executed (bench / tests): number of kernel
 * launches, CTAs of the persistent learner kernel, rows per CTA */
int prl_dqn_last_launch_info(const prl_dqn *dqn, int32_t *launches, int32_t *ctas,
                             int32_t *rows_per_cta);

/* ---- multi-GPU data-parallel learner -------------------------------------
 * One process per GPU (torch.distributed provides the rendezvous only).  Each rank owns a replay
 * shard and samples its own batch; inside the persistent learner kernel the per-rank gradient
 * (P floats) is exchanged between phase A and the AdamW step by ONE-SHOT PUSH over NVLink peer
 * memory: every rank stores (gradient value, round sequence number) as one 8-byte word into every
 * peer's inbox (double-buffered by round parity); the owner of parameter i polls the W sequence
 * numbers of element i, sums the W values in rank order and divides by W — one-way NVLink latency,
 * no fence / flag round trip, no host involvement.  All ranks therefore apply bit-identical updates
 * (the mean gradient of the W*B sampled transitions).  The reference has no counterpart: no RL
 * learner in Pearl is distributed (SURVEY.md §5, §8e); this is the "all-reduce on the gradient
 * only" of the north star, fused into the step kernel instead of a separate NCCL launch.
 *
 * The communicator's buffers are library-allocated (cudaMalloc) so that they can be shared with
 * CUDA IPC: exchange the 128-byte blob of prl_comm_local_handles between all ranks (any byte
 * all-gather), then prl_comm_open_peers with the W blobs in rank order. */
typedef struct prl_comm prl_comm;
#define PRL_COMM_HANDLE_BYTES 128
int prl_comm_create(prl_comm **out, int rank, int world, int64_t max_param_count);
int prl_comm_local_handles(prl_comm *comm, uint8_t out_blob[PRL_COMM_HANDLE_BYTES]);
int prl_comm_open_peers(prl_comm *comm, const uint8_t *blobs /* [world][PRL_COMM_HANDLE_BYTES] */);
int prl_comm_destroy(prl_comm *comm);
/* attach (or detach with NULL) a communicator to a learner; every rank must then call
 * prl_dqn_learn with the same `rounds` */
int prl_dqn_set_comm(prl_dqn *dqn, prl_comm *comm);

/* ---- tensor-core learner, one SM per learner (aggregate mode) -----------------------------
 * PolicyLearner.learn() for `count` INDEPENDENT learners (seeds / agents; the reference runs those
 * as separate OS processes, utils/scripts/benchmark.py:80-116) in one launch: CTA i trains learner
 * dqns[i] on buffer bufs[i] for `rounds` gradient steps with every dense contraction on tcgen05
 * (3xTF32, fp32 accumulation in TMEM).  Same arithmetic contract and outputs as prl_dqn_learn, per
 * learner; out_mae (required) / out_q / out_y / out_logical are arrays of `count` device pointers
 * (the optional arrays and their entries may be NULL).  Shape class: hidden [64,64], obs % 8 == 0
 * and <= 128, n_actions in {1,2,4,8,16}, DeepQLearning (not DoubleDQN), batch 128 or 256, all
 * learners with one configuration and one record layout; otherwise PRL_EUNSUPPORTED (use
 * prl_dqn_learn).  prl_dqn_tc_supported answers that question for one learner. */
int prl_dqn_tc_supported(const prl_dqn *dqn, int batch);
int prl_dqn_learn_multi(prl_dqn *const *dqns, prl_buf *const *bufs, int count, int rounds, int batch,
                        const int64_t *training_steps0, float *const *out_mae_dev, float *const *out_q_dev,
                        float *const *out_y_dev, int32_t *const *out_logical_dev, void *stream);

/* ---- prioritized replay (sum tree) ----------------------------------------------------------
 * NOT in the reference (no prioritized replay exists in Pearl @ 48f1fbb, SURVEY.md §0.3): parity is
 * pinned against oracle/per_oracle.py, the restatement of proportional prioritization (Schaul et al.
 * 2016) that both sides implement with bit-identical fp32 trees.  Leaves are the physical ring slots
 * of a replay buffer of `capacity` records.  The caller provides two device arrays of
 * prl_per_tree_floats(capacity) floats (sum tree, min tree) and one device float (running maximum
 * priority); prl_per_create initialises them on `stream`. */
typedef struct prl_per_cfg {
    int64_t capacity;
    double alpha, beta, eps;   /* p = (|td| + eps)^alpha ; w = (p_min / p)^beta */
    uint64_t seed;             /* Philox4x32-10 key of the stratified draws */
} prl_per_cfg;
typedef struct prl_per prl_per;
int64_t prl_per_tree_floats(int64_t capacity);
int prl_per_create(prl_per **out, const prl_per_cfg *cfg, float *sum_tree_dev, float *min_tree_dev,
                   float *max_priority_dev, void *stream);
int prl_per_destroy(prl_per *per);
int prl_per_set_beta(prl_per *per, double beta);
int64_t prl_per_draws(const prl_per *per);
/* transitions just written to ring slots [first_slot, first_slot + count) (wrapping) enter at the
 * running maximum priority */
int prl_per_push(prl_per *per, int64_t first_slot, int64_t count, void *stream);
/* k <= 1024 stratified draws: out_slots_dev i32[k] (ring slots), out_weights_dev f32[k] (IS weights) */
int prl_per_sample(prl_per *per, int k, int32_t *out_slots_dev, float *out_weights_dev, void *stream);
/* new priorities (|td| + eps)^alpha for k <= 1024 sampled slots; out_priority_dev (optional) f32[k] */
int prl_per_set_priorities(prl_per *per, const int32_t *slots_dev, const float *td_dev, int k,
                           float *out_priority_dev, void *stream);
/* PolicyLearner.learn() over a prioritized buffer: per round sample -> weighted MSE step (the IS weight
 * multiplies the squared TD error) -> priority update from |q - y|.  Same outputs as prl_dqn_learn;
 * out_slots_dev (optional) i32[rounds][batch] receives the sampled ring slots. */
int prl_dqn_learn_per(prl_dqn *dqn, prl_buf *buf, prl_per *per, int rounds, int batch, int64_t training_steps0,
                      float *out_mae_dev, float *out_q_dev, float *out_y_dev, int32_t *out_slots_dev,
                      float *out_weights_dev, void *stream);

/* ---- PPO preprocessing: GAE + truncated lambda returns --------------------------------------
 * Replaces the per-transition loop of ProximalPolicyOptimization.preprocess_replay_buffer
 * (policy_learners/sequential_decision_making/ppo.py:271-293).  All arrays are device pointers in
 * TIME order (index 0 = oldest stored transition): values[i] = critic(state_i), last_next_value =
 * critic(next_state of the newest transition), reward f32, terminated / truncated u8.  Outputs gae[i],
 * lam_return[i] are bit-identical to the reference loop (same fp32 operation order); episodes
 * (chains between terminated / truncated transitions) are processed in parallel.  scratch_dev: device int32[n + 1]
 * owned by the caller (the compacted chain heads and their count; contents are overwritten). */
int prl_ppo_gae(int n, const float *values_dev, float last_next_value, const float *reward_dev,
                const uint8_t *terminated_dev, const uint8_t *truncated_dev, double gamma, double lam,
                float *out_gae_dev, float *out_lam_return_dev, int32_t *scratch_dev, void *stream);

/* ---- continuous Soft Actor-Critic ---------------------------------------------------------------
 * Replaces ContinuousSoftActorCritic.learn_batch (policy_learners/sequential_decision_making/
 * actor_critic_base.py:309-366, soft_actor_critic_continuous.py:131-231) driven by PolicyLearner.learn
 * (policy_learner.py:162-204) over a continuous-action ring: per round sample -> actor step
 * (GaussianActorNetwork.sample_action, actor_networks.py:551-591, twin-critic minimum) -> critic step
 * with the updated actor (twin MSE against the entropy-regularised target, critic_utils.py:170-203)
 * -> soft target update (tau every step) -> entropy-coefficient step.  Three AdamW(amsgrad) states.
 * Flat parameter layouts (fp32, row-major [out][in] like nn.Linear):
 *   actor : W1[h1][obs] b1 W2[h2][h1] b2 Wmu[A][h2] bmu Wstd[A][h2] bstd
 *   critic: TWO consecutive copies (q1 then q2) of W1[c1][obs+A] b1 W2[c2][c1] b2 W3[1][c2] b3
 * The reparameterisation noise is an input (device f32[rounds][2][batch][A]: first draw on `state`
 * for the actor loss, second on `next_state` for the target), as torch's Normal.rsample consumes it. */
typedef struct prl_sac_cfg {
    int32_t obs_dim, act_dim, actor_h1, actor_h2, critic_h1, critic_h2;
    int32_t autotune;     /* entropy_autotune */
    int32_t max_batch, max_rounds;
    double actor_lr, critic_lr, beta1, beta2, eps, weight_decay, gamma, tau;
} prl_sac_cfg;
typedef struct prl_sac prl_sac;
int64_t prl_sac_actor_param_count(const prl_sac_cfg *cfg);
int64_t prl_sac_critic_param_count(const prl_sac_cfg *cfg);   /* ONE critic */
int64_t prl_sac_workspace_bytes(const prl_sac_cfg *cfg);
/* All pointers are device memory owned by the caller: actor vectors f32[actor_param_count], critic
 * vectors f32[2 * critic_param_count], log_alpha4 = {log_alpha, exp_avg, exp_avg_sq, max_exp_avg_sq},
 * alpha1 = the entropy coefficient in use, low/high f32[act_dim] action-space bounds. */
int prl_sac_create(prl_sac **out, const prl_sac_cfg *cfg, float *actor_w, float *actor_m, float *actor_v,
                   float *actor_vmax, float *critic_w, float *critic_m, float *critic_v, float *critic_vmax,
                   float *critic_target_w, float *log_alpha4, float *alpha1, const float *low_dev,
                   const float *high_dev, int64_t adam_step, void *workspace);
int prl_sac_destroy(prl_sac *sac);
int64_t prl_sac_adam_step(const prl_sac *sac);
/* out_*_loss: device f32[rounds]; out_logical_dev (optional) i32[rounds][batch] = sampled indices */
int prl_sac_learn(prl_sac *sac, prl_buf *buf, int rounds, int batch, const float *noise_dev,
                  float *out_actor_loss_dev, float *out_critic_loss_dev, float *out_entropy_loss_dev,
                  int32_t *out_logical_dev, void *stream);
/* The round is a fixed sequence of kernel launches replayed from a CUDA graph (default on; 0 = plain
 * stream launches, e.g. under a profiler).  prl_sac_last_launches: kernels launched by the last learn. */
int prl_sac_set_graph(prl_sac *sac, int enable);
int64_t prl_sac_last_launches(const prl_sac *sac);

/* ---- discrete Soft Actor-Critic -----------------------------------------------------------------
 * Replaces SoftActorCritic.learn_batch (policy_learners/sequential_decision_making/soft_actor_critic.py:151-286 on
 * actor_critic_base.py:309-366) driven by PolicyLearner.learn (policy_learner.py:162-204) over a discrete-action ring with a
 * fixed action space: per round sample -> actor step (p = softmax(actor(s)), loss = mean over B x A of
 * p (alpha log(p + 1e-8) - min(Q1, Q2)(s, .)), :247-286) -> critic step with the updated actor (y = r + gamma (1 - terminated)
 * sum_a p'(min(Q1t, Q2t)(s', a) - alpha log(p' + 1e-8)), twin MSE, :180-245, critic_utils.py:170-203) -> soft target update
 * (tau every round, critic_utils.py:103-122) -> [autotune] entropy step: loss = exp(log_alpha) (H - target_entropy),
 * H = -mean_b sum_a p log(p + 1e-8) of the actor step's p, torch.optim.Adam(eps = entropy_eps) (:137-142, 151-178).
 * Actor and critics: AdamW(amsgrad), one step count.  The step draws no random numbers.
 * Flat parameter layouts (fp32, row-major [out][in] like nn.Linear):
 *   actor : W1[h1][obs] b1 W2[h2][h1] b2 W3[A][h2] b3
 *   critic: TWO consecutive copies (q1 then q2) of W1[c1][obs+A] b1 W2[c2][c1] b2 W3[1][c2] b3   (input = state || one_hot(a)) */
typedef struct prl_dsac_cfg {
    int32_t obs_dim, n_actions, actor_h1, actor_h2, critic_h1, critic_h2;
    int32_t autotune;     /* entropy_autotune */
    int32_t max_batch, max_rounds;
    double actor_lr, critic_lr, entropy_lr, beta1, beta2, eps, weight_decay, gamma, tau;
    double target_entropy; /* -target_entropy_scale * log(1 / n_actions), as the reference evaluates it in fp32 */
    double entropy_eps;    /* eps of the entropy optimizer (the reference: 1e-4) */
} prl_dsac_cfg;
typedef struct prl_dsac prl_dsac;
int64_t prl_dsac_actor_param_count(const prl_dsac_cfg *cfg);
int64_t prl_dsac_critic_param_count(const prl_dsac_cfg *cfg);   /* ONE critic */
int64_t prl_dsac_workspace_bytes(const prl_dsac_cfg *cfg);
/* All pointers are device memory owned by the caller: actor vectors f32[actor_param_count], critic vectors
 * f32[2 * critic_param_count], log_alpha4 = {log_alpha, Adam exp_avg, Adam exp_avg_sq, unused}, alpha1 = the entropy
 * coefficient in use (fixed when autotune = 0).  adam_step: optimizer steps already taken (all three optimizers). */
int prl_dsac_create(prl_dsac **out, const prl_dsac_cfg *cfg, float *actor_w, float *actor_m, float *actor_v,
                    float *actor_vmax, float *critic_w, float *critic_m, float *critic_v, float *critic_vmax,
                    float *critic_target_w, float *log_alpha4, float *alpha1, int64_t adam_step, void *workspace);
int prl_dsac_destroy(prl_dsac *dsac);
int64_t prl_dsac_adam_step(const prl_dsac *dsac);
/* New actor / critic learning rates, used from the next prl_dsac_learn on (the per-round optimizer scalars are computed
 * at every call, so a captured round is kept): SoftActorCritic.reset steps an ExponentialLR of the actor every episode. */
int prl_dsac_set_lr(prl_dsac *dsac, double actor_lr, double critic_lr);
/* out_*_loss: device f32[rounds] (out_entropy_loss: the entropy loss of autotune rounds, untouched otherwise);
 * out_logical_dev (optional) i32[rounds][batch] = sampled indices.  PRL_EINVAL without device work for a continuous-action
 * buffer, a buffer with PRL_BUF_DYNAMIC_ACTIONS, a sharded buffer or mismatched dimensions. */
int prl_dsac_learn(prl_dsac *dsac, prl_buf *buf, int rounds, int batch, float *out_actor_loss_dev, float *out_critic_loss_dev,
                   float *out_entropy_loss_dev, int32_t *out_logical_dev, void *stream);
/* CUDA-graph replay of the round (default on; 0 = plain stream launches).  Kernels launched by the last learn. */
int prl_dsac_set_graph(prl_dsac *dsac, int enable);
int64_t prl_dsac_last_launches(const prl_dsac *dsac);

/* ---- TD3 / DDPG ----------------------------------------------------------------------------------
 * Replaces TD3.learn_batch (policy_learners/sequential_decision_making/td3.py:106-202) and, with
 * actor_update_freq = 1 and no noise, DeepDeterministicPolicyGradient (ddpg.py:105-157 on
 * actor_critic_base.py:309-366), driven by PolicyLearner.learn (policy_learner.py:162-204) over a
 * continuous-action ring: per round sample -> [if training_steps % actor_update_freq == 0: actor step,
 * maximise Q1(s, pi(s)), VanillaContinuousActorNetwork tanh head + action_scaling, actor_networks.py:29-51,448-485]
 * -> twin-critic step against min(Q1', Q2')(s', clamp(pi'(s') + clipped noise)) -> [on the same rounds: soft
 * update of the critic targets and of the actor target].  The actor optimizer's step count advances only on its
 * update rounds.  Flat layouts (fp32, row-major [out][in]):
 *   actor : W1[h1][obs] b1 W2[h2][h1] b2 W3[A][h2] b3       critic: as prl_sac (q1 then q2)
 * noise_dev: device f32[rounds][batch][A] = the torch.normal(0, actor_update_noise, ...) draws (null: DDPG). */
typedef struct prl_td3_cfg {
    int32_t obs_dim, act_dim, actor_h1, actor_h2, critic_h1, critic_h2;
    int32_t actor_update_freq;
    int32_t max_batch, max_rounds;
    double actor_lr, critic_lr, beta1, beta2, eps, weight_decay, gamma, actor_tau, critic_tau, noise_clip;
} prl_td3_cfg;
typedef struct prl_td3 prl_td3;
int64_t prl_td3_actor_param_count(const prl_td3_cfg *cfg);
int64_t prl_td3_critic_param_count(const prl_td3_cfg *cfg);   /* ONE critic */
int64_t prl_td3_workspace_bytes(const prl_td3_cfg *cfg);
int prl_td3_create(prl_td3 **out, const prl_td3_cfg *cfg, float *actor_w, float *actor_m, float *actor_v,
                   float *actor_vmax, float *actor_target_w, float *critic_w, float *critic_m, float *critic_v,
                   float *critic_vmax, float *critic_target_w, const float *low_dev, const float *high_dev,
                   int64_t actor_adam_step, int64_t critic_adam_step, void *workspace);
int prl_td3_destroy(prl_td3 *td3);
int64_t prl_td3_actor_adam_step(const prl_td3 *td3);
int64_t prl_td3_critic_adam_step(const prl_td3 *td3);
/* training_steps0 = learner._training_steps before the call; out_*_loss: device f32[rounds] */
int prl_td3_learn(prl_td3 *td3, prl_buf *buf, int rounds, int batch, int64_t training_steps0, const float *noise_dev,
                  float *out_actor_loss_dev, float *out_critic_loss_dev, int32_t *out_logical_dev, void *stream);
int prl_td3_set_graph(prl_td3 *td3, int enable);
int64_t prl_td3_last_launches(const prl_td3 *td3);

/* ---- PPO learner ------------------------------------------------------------------------------
 * Replaces ProximalPolicyOptimization.learn (policy_learners/sequential_decision_making/ppo.py:195-293):
 * prl_ppo_preprocess = preprocess_replay_buffer (state values, taken-action probabilities under the current
 * policy, GAE and truncated lambda returns over the whole rollout, time order), prl_ppo_learn =
 * PolicyLearner.learn (policy_learner.py:162-204) x ActorCriticBase.learn_batch (actor_critic_base.py:309-349):
 * clipped-surrogate actor step (ppo.py:152-184; VanillaActorNetwork softmax policy) then the state-value critic
 * step (critic_utils.py:139-167).  Flat parameter layouts (row-major [out][in]):
 *   actor : W1[h1][obs] b1 W2[h2][h1] b2 W3[A][h2] b3      critic: W1[c1][obs] b1 W2[c2][c1] b2 W3[1][c2] b3 */
typedef struct prl_ppo_cfg {
    int32_t obs_dim, n_actions, actor_h1, actor_h2, critic_h1, critic_h2;
    int32_t max_batch, max_rounds;
    int64_t max_rollout;
    double actor_lr, critic_lr, beta1, beta2, eps, weight_decay, gamma, lam, epsilon, entropy_bonus;
} prl_ppo_cfg;
typedef struct prl_ppo prl_ppo;
int64_t prl_ppo_actor_param_count(const prl_ppo_cfg *cfg);
int64_t prl_ppo_critic_param_count(const prl_ppo_cfg *cfg);
int64_t prl_ppo_workspace_bytes(const prl_ppo_cfg *cfg);
int prl_ppo_create(prl_ppo **out, const prl_ppo_cfg *cfg, float *actor_w, float *actor_m, float *actor_v, float *actor_vmax,
                   float *critic_w, float *critic_m, float *critic_v, float *critic_vmax, int64_t adam_step,
                   void *workspace);
int prl_ppo_destroy(prl_ppo *ppo);
int64_t prl_ppo_adam_step(const prl_ppo *ppo);
int prl_ppo_set_graph(prl_ppo *ppo, int enable);
int64_t prl_ppo_last_launches(const prl_ppo *ppo);
/* outputs: device f32[len(buf)] each, index 0 = oldest stored transition; out_cut_dev (optional) u8[len]:
 * 1 where the transition is terminated or truncated (ends a GAE chain) */
int prl_ppo_preprocess(prl_ppo *ppo, prl_buf *buf, float *out_values_dev, float *out_action_probs_dev,
                       float *out_gae_dev, float *out_lam_return_dev, uint8_t *out_cut_dev, void *stream);
/* Rollout sharded over ranks by contiguous time chunks: re-run this chunk's GAE chains with V(next) of its newest
 * transition = `next_value` (first state value of the next, newer chunk) and the chain entering from there =
 * `incoming_gae` (that chunk's first gae).  Uses the rewards / flags staged by the last prl_ppo_preprocess.
 * Bit-identical to the unsharded computation. */
int prl_ppo_gae_redo(prl_ppo *ppo, const float *values_dev, float next_value, float incoming_gae,
                     float *out_gae_dev, float *out_lam_return_dev, void *stream);
/* gae / lam_return / action_probs: the arrays prl_ppo_preprocess produced; out_*_loss: device f32[rounds] */
int prl_ppo_learn(prl_ppo *ppo, prl_buf *buf, int rounds, int batch, const float *gae_dev,
                  const float *lam_return_dev, const float *action_probs_dev, float *out_actor_loss_dev,
                  float *out_critic_loss_dev, int32_t *out_logical_dev, void *stream);

/* Device timing of the persistent learner kernel alone (CUDA events recorded on
 * the launch stream around the kernel); used by bench.py for the roofline line.
 * prl_dqn_last_kernel_ms synchronises on the end event. */
int prl_dqn_set_timing(prl_dqn *dqn, int enable);
/* Developer profiling: device int64[rounds][16] receiving SM-clock stamps of one CTA at
 * the phase boundaries of every round of the next prl_dqn_learn calls (NULL = off).  The
 * tensor-core group kernel stamps CTA $PRL_TC_PROF_CTA (default 0), the cooperative kernel CTA 0. */
int prl_dqn_set_profile(prl_dqn *dqn, long long *stamps_dev);
int prl_dqn_last_kernel_ms(prl_dqn *dqn, float *ms);

/* Self-test of the tcgen05 / TMEM building block used by the learner kernels: one CTA computes
 * D[128][n] = A[128][k] * B[n][k]^T (device fp32 row-major arrays) with plain TF32 (passes = 1) or
 * the 3xTF32 split the learner uses for fp32 parity (passes = 3).  Test infrastructure hook. */
int prl_test_umma_gemm(const float *a_dev, const float *b_dev, float *d_dev, int n, int k, int passes,
                       void *stream);
/* Same product with the A operand in tensor memory (written by tcgen05.st), B in shared memory;
 * k <= 64; reps > 1 prints a throughput probe. */
int prl_test_umma_gemm_ts(const float *a_dev, const float *b_dev, float *d_dev, int n, int k, int reps, void *stream);
/* General self-test: D[m][n] = A[m][k] * B[n][k]^T with m in {64,128} and a free operand chunk pitch
 * `lbo` (128 dense / 144 transposed-write friendly, see csrc/umma.cuh).  draw_dev receives the raw
 * accumulator: 128 TMEM lanes x n columns (for m = 64, row i is lane 32*(i/16) + i%16). */
int prl_test_umma_gemm2(const float *a_dev, const float *b_dev, float *draw_dev, int m, int n, int k, int lbo,
                        void *stream);

/* ---- contraction engine of the actor-critic learners (SAC, PPO, TD3 / DDPG) --------------------------------
 * The dense layers of those learners (the torch matmuls of pearl/neural_networks/common/utils.py:mlp_block as used by
 * actor_networks.py / value_networks.py, forward and autograd backward) run as 3xTF32 tcgen05 tiles or as fp32 SIMT tiles:
 * engine 1 (default) picks per product whichever is faster on a B200 (profiles/r2_gemm_tc.md), 0 = SIMT only,
 * 2 = tcgen05 always.  Process-wide; read when a learner's round is launched or captured into its CUDA graph, so set it
 * before the first learn() of a learner. */
int prl_set_contraction_engine(int engine);
int prl_get_contraction_engine(void);
/* Test hook: one contraction of the three kinds the learners use, `nets` stacked problems contiguous in every operand.
 *   op 0  c[M x N]   = act(x W^T + bias)      a = x [M x K] (or [M x split] and a2 = [M x (K - split)]), b = W [N x K]
 *   op 1  c[M x K] (+)= dy W, masked          a = dy [M x N], b = W [N x K], mask [M x K] (keep where mask > 0)
 *   op 2  c[N x K]   = dy^T x, c_tail = dy^T 1  a = dy [M x N], b = x [M x K] (or split with a2)
 * engine: -1 library default, 0 SIMT, 1 automatic, 2 tcgen05 always; 64 / 32: the shared-memory-operand form with that tile
 * width, 164 / 132: the tensor-memory-operand form with tile width 64 / 32. */
int prl_test_contraction(int op, int engine, int M, int N, int K, const float *a, const float *b, const float *a2, int split,
                         const float *bias, const float *mask, int relu, int accumulate, float *c, float *c_tail, int nets,
                         void *stream);
/* Developer profiling of the tcgen05 contraction: device int64[33][8] receiving SM-clock stamps of CTA 0 (per 32-deep
 * chunk: loader warp 0 at iteration start / loads issued / stage free / tile stored, issuer at operands ready / MMAs
 * issued) for the following prl_test_contraction calls; NULL = off. */
int prl_test_contraction_stamps(long long *stamps_dev);

#ifdef __cplusplus
}
#endif
#endif /* PEARL_B200_H */
