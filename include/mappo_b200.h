/*
 * mappo_b200.h -- C ABI of the B200-native MAPPO rollout-and-update engine (libmappo_b200.so).
 *
 * The reference (marlbenchmark/on-policy) has no FFI on this path: all arithmetic is PyTorch/NumPy
 * called from four Python classes.  This ABI is the boundary *introduced* beneath those classes
 * (SURVEY.md section 8b); each entry point names the reference code it replaces
 * (paths relative to /root/reference/onpolicy/).  Style follows the reference's only C ABI,
 * envs/hanabi/pyhanabi.h:24-60 (extern "C", opaque handles, plain pointers and sizes).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to fp32 unless the name says otherwise (host structs are
 *     `const mappo_*_t*`); storage is allocated and owned by the caller ("tensors in, tensors out");
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), performs no host
 *     synchronisation and no allocation, and is CUDA-graph capturable;
 *   - return value: 0 = ok, negative = mappo_status; text via mappo_last_error() (thread local);
 *   - row-major everywhere; a "row" is one (t, n, m) sample: row = (t*N + n)*M + m, E = N*M rows per step.
 */
#ifndef MAPPO_B200_H_
#define MAPPO_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MAPPO_MAX_HEADS 4      /* MultiDiscrete heads per actor */
#define MAPPO_MAX_LAYERS 2     /* layer_N hidden (H->H) blocks per MLP base */
#define MAPPO_ABI_VERSION 5

typedef enum mappo_status {
  MAPPO_OK = 0,
  MAPPO_ERR_INVALID = -1,      /* bad argument / unsupported configuration */
  MAPPO_ERR_CUDA = -2,         /* CUDA runtime error (launch, attribute, ...) */
  MAPPO_ERR_UNSUPPORTED = -3   /* valid in the reference, not built yet (fails loudly, never falls back) */
} mappo_status;

/* One network (actor or critic).  Mirrors what R_Actor / R_Critic build
 * (algorithms/r_mappo/algorithm/r_actor_critic.py:12-43, 120-154; algorithms/utils/mlp.py:6-57;
 * rnn.py:7-22; act.py:12-42): [LayerNorm(in)] -> Linear(in,H) -> act -> LN -> layer_n x [Linear(H,H) -> act -> LN]
 * -> [GRU(H,H) -> LN] -> heads.  Critic: n_heads = 1, head_dim[0] = 1 (v_out). */
typedef struct mappo_net_desc {
  int32_t in_dim;              /* obs_dim (actor) or share_obs_dim (critic) */
  int32_t hidden;              /* hidden_size H */
  int32_t layer_n;             /* layer_N */
  int32_t use_feature_norm;    /* use_feature_normalization */
  int32_t use_relu;            /* 1 ReLU, 0 Tanh (config.py:203) */
  int32_t recurrent;           /* 1 = GRU block present (recurrent_N == 1 only) */
  int32_t n_heads;
  int32_t head_dim[MAPPO_MAX_HEADS];
  int32_t is_critic;
} mappo_net_desc_t;

/* Offsets (in floats) of every tensor inside the flat parameter vector of a net; -1 = absent.
 * Matrix layouts are the PyTorch ones ([out, in] row-major), so a state_dict copies in verbatim
 * (key names: SURVEY.md App. A.8). */
typedef struct mappo_net_layout {
  int32_t fn_w, fn_b;                                   /* base.feature_norm.{weight,bias}            [in]     */
  int32_t fc1_w, fc1_b, ln1_w, ln1_b;                   /* base.mlp.fc1.0 [H,in],[H]; fc1.2 [H],[H]              */
  int32_t fc2_w[MAPPO_MAX_LAYERS], fc2_b[MAPPO_MAX_LAYERS];   /* base.mlp.fc2.i.0 [H,H],[H]                      */
  int32_t ln2_w[MAPPO_MAX_LAYERS], ln2_b[MAPPO_MAX_LAYERS];   /* base.mlp.fc2.i.2                                */
  int32_t gru_wih, gru_whh, gru_bih, gru_bhh;           /* rnn.rnn.{weight,bias}_{ih,hh}_l0 [3H,H],[3H] (r,z,n)  */
  int32_t rnn_ln_w, rnn_ln_b;                           /* rnn.norm.{weight,bias}                               */
  int32_t head_w, head_b;                               /* heads stacked: [sum(head_dim), H], [sum(head_dim)]   */
  int32_t total;                                        /* parameter count                                      */
} mappo_net_layout_t;

/* Hyper-parameters of one optimiser step (R_MAPPO.__init__, algorithms/r_mappo/r_mappo.py:24-41). */
typedef struct mappo_loss_cfg {
  float clip_param, entropy_coef, value_loss_coef, huber_delta;
  int32_t use_clipped_value_loss, use_huber_loss, use_value_active_masks, use_policy_active_masks;
  int32_t use_valuenorm;       /* normalise return targets with the ValueNorm state */
  int32_t update_actor;        /* ppo_update(sample, update_actor) r_mappo.py:91,145 */
  int32_t gemm_mode;           /* MAPPO_GEMM_FP32 (exact fp32 FFMA tiles) or MAPPO_GEMM_TF32 (tcgen05 tensor cores) */
  int32_t happo;               /* 1: actor loss of HAPPO (algorithms/happo/happo_trainer.py:129-141): one importance weight per row
                                  (product over the action heads) times mappo_batch_t.factor inside the clipped surrogate */
  int32_t inputs_prepared;     /* hidden >= 128 nets only: the workspace already holds the normalised input rows of THIS batch
                                  (same rows, same order) from an earlier mappo_update_fwd_bwd on it -- e.g. the later PPO epochs
                                  of one train() over an unchanged buffer -- so the feature-norm pass is skipped */
  int32_t image_ready;         /* MAPPO_GEMM_TF32 hidden-64 nets only: the workspace already holds the folded weight image of the
                                  CURRENT parameters (left there by mappo_update_tail of the previous optimiser step) */
} mappo_loss_cfg_t;

#define MAPPO_GEMM_FP32 0
#define MAPPO_GEMM_TF32 1

/* One minibatch as the update kernels see it.  Either a view of the rollout storage read through
 * an index list (`rows` != NULL: fused gather, replaces shared_buffer.py:377-396 / 557-604) or a
 * materialised sample (`rows` == NULL: arrays are already [n_rows, .]).
 * Recurrent minibatches are time-major [L, n_seq] (position p = l*n_seq + c) with one initial
 * hidden state per sequence; feed-forward: seq_len = 1, n_seq = n_rows. */
typedef struct mappo_batch {
  const float* obs;            /* [.,Do]  actor input rows                       */
  const float* share_obs;      /* [.,Ds]  critic input rows                      */
  const float* actions;        /* [.,as]  stored as fp32 (shared_buffer.py:77)   */
  const float* old_logp;       /* [.,as]                                         */
  const float* value_preds;    /* [.,1]                                          */
  const float* returns;        /* [.,1]                                          */
  const float* advantages;     /* [.,1]   raw advantages (normalised on the fly) */
  const float* masks;          /* [.,1]                                          */
  const float* active_masks;   /* [.,1]                                          */
  const float* avail;          /* [.,A] or NULL                                  */
  const float* h0_actor;       /* [.,H]   rnn_states        rows (recurrent only) */
  const float* h0_critic;      /* [.,H]   rnn_states_critic rows (recurrent only) */
  const int32_t* rows;         /* [n_rows] storage row feeding position p, or NULL */
  const int32_t* seq_first;    /* [n_seq] storage row whose rnn state starts sequence c, or NULL */
  const float* factor;         /* [.,1]   HAPPO importance factor of the row (separated_buffer.py:62-63) or NULL (= 1) */
  int32_t n_rows, seq_len, n_seq;
} mappo_batch_t;

/* ---- library ------------------------------------------------------------------------------- */
int32_t mappo_abi_version(void);
const char* mappo_last_error(void);
/* SM count / arch check of the current device; fails unless compute capability is 10.x. */
int32_t mappo_device_check(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor);

/* ---- parameter layout (host only) ---------------------------------------------------------- */
int32_t mappo_net_layout(const mappo_net_desc_t* desc, mappo_net_layout_t* out);

/* ---- a8: rollout inference ------------------------------------------------------------------
 * R_MAPPOPolicy.get_actions / get_values / act (rMAPPOPolicy.py:48-127) -> R_Actor.forward
 * (r_actor_critic.py:44-71), R_Critic.forward (:156-175), ACTLayer.forward (act.py:44-91),
 * FixedCategorical.sample/mode/log_probs (distributions.py:14-28).
 * Either net may be skipped by passing params == NULL (get_values: actor NULL; act: critic NULL).
 * Sampling: action = argmax_j softmax(logits)_j / q_j with q ~ Exp(1) (== torch multinomial).
 *   exp_noise != NULL : q read from exp_noise[row, sum(head_dim)] (parity mode, host-drawn noise)
 *   exp_noise == NULL : q = -log(u), u from Philox4x32-10 keyed by (rng_seed, *rng_offset_dev + row)
 * deterministic != 0 : argmax of the probabilities.
 * Outputs go straight into the caller's storage slots: values [E,1], actions [E,as] (fp32, the
 * buffer dtype) and optionally actions_i64 [E,as], logp [E,as], h_out [E,H] (recurrent). */
int32_t mappo_policy_step(const mappo_net_desc_t* actor_desc, const float* actor_params,
                          const mappo_net_desc_t* critic_desc, const float* critic_params,
                          const float* obs, const float* share_obs,
                          const float* h_actor_in, const float* h_critic_in, const float* masks,
                          const float* avail, const float* exp_noise,
                          uint64_t rng_seed, const uint64_t* rng_offset_dev, int32_t deterministic,
                          int32_t n_rows,
                          float* values, float* actions, int64_t* actions_i64, float* logp,
                          float* h_actor_out, float* h_critic_out,
                          const float* actor_image, const float* critic_image, void* stream);
/* Optional: the rollout weights do not change during the T collect steps of an iteration.  Packing them once into
 * the kernel's shared-memory layout lets every policy_step CTA fetch them with one TMA bulk copy
 * (cp.async.bulk + mbarrier) -- pass the images to mappo_policy_step (NULL = load from the flat parameters). */
/* The whole collect phase of one iteration as ONE launch, for the device-resident pipeline where the env outputs of
 * the iteration are already staged in HBM (synthetic / on-device environments): T x (policy_step + env_insert) + the
 * bootstrap get_values of Runner.compute (runner/shared/mpe_runner.py:26-40, base_runner.py:120-134).  Rows never
 * interact, so each CTA keeps its 32 rows, the weights and the recurrent state on chip and walks t = 0..T.
 * Storage pointers address slot 0 (slots are E*dim floats apart); f_* are the staged env outputs, index t = what the env
 * returned after step t (written to slot t+1; rewards to slot t).  Sampling as in mappo_policy_step (per-step noise
 * [T, E, sum A] or Philox; the device offset advances by T*E).
 * f_share may be NULL for feed-forward nets when share_obs is the concatenation of the obs of the agents of a rollout
 * thread (use_centralized_V in the MPE runner, mpe_runner.py:133-135; requires share_dim = k * obs_dim and rows ordered
 * thread-major): the critic then reads its rows straight from f_obs and only obs needs staging (4x fewer H2D bytes
 * for 3 agents); the share_obs storage slots are still written. */
int32_t mappo_rollout_persistent(const mappo_net_desc_t* actor_desc, const float* actor_params, const float* actor_image,
                                 const mappo_net_desc_t* critic_desc, const float* critic_params, const float* critic_image,
                                 float* obs, float* share_obs, float* h_actor, float* h_critic, float* masks, float* avail,
                                 float* value_preds, float* actions, float* logp, float* rewards, float* active_masks,
                                 const float* f_obs, const float* f_share, const float* f_rew, const float* f_done,
                                 const float* f_active, const float* f_avail, const float* exp_noise, uint64_t rng_seed,
                                 uint64_t* rng_offset_dev, int32_t T, int32_t E, void* stream);
/* The CLOSED rollout loop of one iteration as one launch (feed-forward policies, MPE simple_spread worlds on the device):
 * T x [mappo_policy_step -> mappo_mpe_spread_step -> mappo_env_insert] + the bootstrap value, i.e. the reference's
 * `for step in range(episode_length): collect; envs.step; insert` followed by compute()'s get_values
 * (runner/shared/mpe_runner.py:26-40, base_runner.py:120-134) with the environment inside the kernel -- the observation of
 * step t + 1 is computed from the action of step t, nothing is staged.  Storage pointers address slot 0 (slot 0 must hold the
 * current observations, e.g. from mappo_mpe_spread_step(actions = NULL) or the previous iteration's after_update); world state as
 * in mappo_mpe_spread_step; reset_states [T, n_envs, 2 (agents + landmarks)] (nullable): the state a world restarts from
 * when its episode ends at step t (NULL: Philox; *env_counter_dev advances by T * n_envs).  Images from
 * mappo_pack_rollout_weights; sampling as in mappo_rollout_persistent. */
int32_t mappo_rollout_closed_loop(const mappo_net_desc_t* actor_desc, const float* actor_image,
                                  const mappo_net_desc_t* critic_desc, const float* critic_image, float* obs, float* share_obs,
                                  float* masks, float* value_preds, float* actions, float* logp, float* rewards,
                                  double* agent_pos, double* agent_vel, double* landmark_pos, int32_t* step_count,
                                  const double* reset_states, uint64_t env_seed, uint64_t* env_counter_dev,
                                  const float* exp_noise, uint64_t rng_seed, uint64_t* rng_offset_dev, int32_t T, int32_t E,
                                  int32_t num_agents, int32_t num_landmarks, int32_t episode_length, void* stream);
/* The same closed loop for either MPE world and for recurrent policies.  world: MAPPO_WORLD_SPREAD (state and reset_states as
 * above; goal / comm NULL) or MAPPO_WORLD_REFERENCE (simple_reference, state as in mappo_mpe_reference_step: num_agents 2,
 * num_landmarks 3, goal / comm [n_envs, 2]; reset_states [T, n_envs, 12]).  The actor must match the world's action space
 * (Discrete(5) / MultiDiscrete(5, 10)) and observation width, the critic its share_obs width (MAPPO_ERR_INVALID otherwise).
 * Feed-forward nets: h_actor / h_critic NULL.  Recurrent (GRU) nets: h_actor / h_critic = the rnn-state storage [T + 1, E, hidden]
 * (slot 0 read; slots 1..T written with the state after step t, zero for rows whose episode ended at step t, as
 * mappo_policy_step followed by mappo_env_insert leaves them); each world group then runs on a 2-CTA cluster (actor CTA with the
 * worlds, critic CTA).  Nets off the warp-per-row kernels (hidden 64, in_dim <= 64, <= 32 head outputs) or needing more than
 * 227 KB of shared memory per CTA: MAPPO_ERR_UNSUPPORTED.  Counters advance as in mappo_rollout_closed_loop. */
#define MAPPO_WORLD_SPREAD 0
#define MAPPO_WORLD_REFERENCE 1
int32_t mappo_rollout_closed_loop_ex(const mappo_net_desc_t* actor_desc, const float* actor_image,
                                     const mappo_net_desc_t* critic_desc, const float* critic_image, float* obs,
                                     float* share_obs, float* h_actor, float* h_critic, float* masks, float* value_preds,
                                     float* actions, float* logp, float* rewards, int32_t world, double* agent_pos,
                                     double* agent_vel, double* landmark_pos, int32_t* goal, int32_t* comm,
                                     int32_t* step_count, const double* reset_states, uint64_t env_seed,
                                     uint64_t* env_counter_dev, const float* exp_noise, uint64_t rng_seed,
                                     uint64_t* rng_offset_dev, int32_t T, int32_t E, int32_t num_agents,
                                     int32_t num_landmarks, int32_t episode_length, void* stream);
int32_t mappo_rollout_image_floats(const mappo_net_desc_t* desc);
int32_t mappo_pack_rollout_weights(const mappo_net_desc_t* desc, const float* params, float* image, void* stream);

/* ---- hidden_size >= 128 MLP nets (BASELINE c5: hidden 512, layer_N 2; algorithms/utils/mlp.py:6-57) ---------------------
 * Weights no longer fit in shared memory: every Linear is its own GEMM (TMA-fed tcgen05 tiles in MAPPO_GEMM_TF32, FFMA tiles
 * in MAPPO_GEMM_FP32) with LayerNorm / activation / loss fused into the epilogues, activations in a per-net workspace.
 * mappo_big_net: 1 if `desc` takes that path (MLP, hidden a multiple of 128 up to 1024, sum(head_dim) <= 32).
 * For such nets the rollout "image" IS the workspace: size from mappo_rollout_workspace_floats(desc, n_rows) (other nets:
 * = mappo_rollout_image_floats), weights packed by mappo_pack_rollout_weights_ex (gemm_mode decides tf32 rounding), and the
 * step is mappo_policy_step_ex (= mappo_policy_step + gemm_mode; the persistent / closed-loop kernels do not cover them).
 * Training uses the same entry points as every net: mappo_update_workspace_floats / mappo_update_fwd_bwd /
 * mappo_update_finish (one gradient slot: the pipeline leaves the complete flat gradient). */
int32_t mappo_big_net(const mappo_net_desc_t* desc);
/* Diagnostic: CUDA-event device time (ms) and launch count of each kernel family of the pipeline since the last call --
 * [0] weight pack, [1] feature norm, [2] forward GEMMs, [3] head + loss, [4] input-gradient GEMMs, [5] weight-gradient
 * GEMMs, [6] slot reduction + unfold -- accumulated over eager (non-captured) launches while `enable` was set; reading
 * synchronises on the recorded events.  Host pointers (7 entries each, nullable). */
int32_t mappo_debug_big_timing(int32_t enable, double* ms_out7, int64_t* launches_out7);
/* Same for the tcgen05 pipeline of recurrent (GRU) hidden-64 nets (MAPPO_GEMM_TF32; replaces the per-segment nn.GRU calls of
 * algorithms/utils/rnn.py:43-77 and their autograd): [0] weight images, [1] base MLP forward, [2] sequence forward, [3] heads + loss,
 * [4] BPTT, [5] gate gradients, [6] base MLP backward, [7] slot sums + unfold.  Host pointers (8 entries each, nullable). */
int32_t mappo_debug_gru_timing(int32_t enable, double* ms_out8, int64_t* launches_out8);
/* clock64 stamps inside one step of the two sequence kernels (CTA 0, thread 0; update_gru_tc.cu lists the points): where does a step's
 * latency go.  Host pointer, 16 entries. */
int32_t mappo_debug_gru_cycles(int64_t* out16);
/* Kernel-level test entries: the two GEMM kernels of the pipeline in isolation (tests/test_gpu_bignet.py compares them with
 * torch.matmul).  mappo_debug_big_lin: out[rows, N] (leading dimension N + 32; columns N, N + 1 = row mean / sigma) =
 * relu(A[rows, K] W[N, K]^T + colvec[N + o]) and stats[rows] = (mean, 1 / sigma), K and N multiples of 32; scratch [rows, N]
 * (fp32 build only).  mappo_debug_big_grad: gsum[M, Qw] = P[rows, :M]^T Q[rows, :Qw] via partial[splits, M, Qw]
 * (splits from mappo_debug_big_grad_splits). */
int32_t mappo_debug_big_lin(const float* A, int32_t lda, const float* W, int32_t ldw, float* out, float* stats, const float* colvec,
                            float* scratch, int32_t rows, int32_t K, int32_t N, int32_t gemm_mode, void* stream);
int32_t mappo_debug_big_grad(const float* P, int32_t ldp, int32_t Pw, int32_t M, const float* Q, int32_t ldq, int32_t Qw, int32_t rows,
                             float* partial, float* gsum, int32_t gemm_mode, void* stream);
int32_t mappo_debug_big_grad_splits(int32_t rows, int32_t M, int32_t Pw, int32_t Qw);
/* Diagnostic: float offsets of the regions of a hidden >= 128 net's update workspace for n_rows rows (64 values, host pointer;
 * layout in csrc/big_net.cu debug_plan) -- scripts/diag_big.py checks the stored intermediates against float64 algebra. */
int32_t mappo_debug_big_plan(const mappo_net_desc_t* desc, int32_t n_rows, int64_t* out64);
int64_t mappo_rollout_workspace_floats(const mappo_net_desc_t* desc, int32_t n_rows);
int32_t mappo_pack_rollout_weights_ex(const mappo_net_desc_t* desc, const float* params, float* image, int32_t gemm_mode,
                                      void* stream);
int32_t mappo_policy_step_ex(const mappo_net_desc_t* actor_desc, const float* actor_params,
                             const mappo_net_desc_t* critic_desc, const float* critic_params,
                             const float* obs, const float* share_obs,
                             const float* h_actor_in, const float* h_critic_in, const float* masks,
                             const float* avail, const float* exp_noise, uint64_t rng_seed,
                             const uint64_t* rng_offset_dev, int32_t deterministic, int32_t n_rows,
                             float* values, float* actions, int64_t* actions_i64, float* logp,
                             float* h_actor_out, float* h_critic_out, const float* actor_image,
                             const float* critic_image, int32_t gemm_mode, void* stream);

/* ---- f1 (SURVEY 8f): device-side environment -------------------------------------------------------------------
 * One step of n_envs vectorised MPE `simple_spread` worlds (envs/env_wrappers.py:140-154 -> envs/mpe/environment.py:115-146
 * -> envs/mpe/core.py:207-323 + scenarios/simple_spread.py:32-103): action decoding, action and contact forces, damped
 * integration, shared reward, observations, done = step >= episode_length, auto-reset (the reset observation replaces the
 * terminal one).  State (float64, the reference's precision; owned by the caller): agent_pos / agent_vel
 * [n_envs, num_agents, 2], landmark_pos [n_envs, num_landmarks, 2], step_count [n_envs].
 * actions [n_envs * num_agents]: integer-valued floats in 0..4 exactly as mappo_policy_step stores them; NULL = reset all
 * worlds (writes obs only).  reset_states [n_envs, 2 (agents + landmarks)] (nullable): the positions a world restarts
 * from -- NumPy's global Mersenne stream cannot be reproduced on a device, so parity tests inject the reference's draws;
 * NULL draws uniform(-1, 1) / 0.8 uniform(-1, 1) from Philox (rng_seed, *rng_counter_dev; the counter advances).
 * Outputs in the layout mappo_env_insert / mappo_rollout_persistent consume: obs [E, D] (D = 4 + 2 L + 4 (M - 1)),
 * share_obs [E, M D] (nullable; the thread's obs concatenated, mpe_runner.py:133-135), rewards [E], dones [E] (1.0 / 0.0). */
int32_t mappo_mpe_spread_step(double* agent_pos, double* agent_vel, double* landmark_pos, int32_t* step_count,
                              const float* actions, const double* reset_states, uint64_t rng_seed,
                              uint64_t* rng_counter_dev, int32_t n_envs, int32_t num_agents, int32_t num_landmarks,
                              int32_t episode_length, float* obs_out, float* share_obs_out, float* rewards_out,
                              float* dones_out, void* stream);

/* The same for MPE `simple_reference` (BASELINE configs[2]'s scenario; scenarios/simple_reference.py:8-97): 2 agents, 3
 * landmarks, 10 communication symbols, no contacts.  Extra state: goal [n_envs, 2] (the landmark agent m wants the OTHER agent
 * on), comm [n_envs, 2] (the symbol agent m uttered last step, -1 = silent after a reset).  actions [n_envs * 2, 2]: the
 * MultiDiscrete([[0,4],[0,9]]) pair (move, symbol) as integer-valued floats, the layout mappo_policy_step stores.
 * reset_states [n_envs, 12] (nullable): goal_0, goal_1, agent positions, landmark positions.  obs [E, 21] = velocity,
 * landmarks - pos, goal colour, other agent's symbol one-hot; share_obs [E, 42] (nullable); rewards = r_0 + r_1 for both
 * agents, r_m = -|pos[1 - m] - landmark[goal_m]|^2. */
int32_t mappo_mpe_reference_step(double* agent_pos, double* agent_vel, double* landmark_pos, int32_t* goal, int32_t* comm,
                                 int32_t* step_count, const float* actions, const double* reset_states, uint64_t rng_seed,
                                 uint64_t* rng_counter_dev, int32_t n_envs, int32_t episode_length, float* obs_out,
                                 float* share_obs_out, float* rewards_out, float* dones_out, void* stream);

/* Advance the device-side Philox offset after a sampling step (no host round trip). */
int32_t mappo_counter_add(uint64_t* counter_dev, uint64_t inc, void* stream);

/* ---- a2: insert / after_update --------------------------------------------------------------
 * SharedReplayBuffer.insert (utils/shared_buffer.py:90-123) fused with the runner's done handling
 * (runner/shared/mpe_runner.py:125-139): writes the env outputs of one step into slot t+1 / t,
 * masks = 1 - done, zeroes both rnn states of done rows.  NULL sources are skipped.  rng_counter_dev (optional):
 * *rng_counter_dev += rng_inc, i.e. the Philox offset consumed by the preceding mappo_policy_step. */
int32_t mappo_env_insert(const float* next_obs, const float* next_share_obs, const float* rewards,
                         const float* dones, const float* next_active, const float* next_avail,
                         int32_t n_rows, int32_t obs_dim, int32_t share_dim, int32_t hidden, int32_t n_act,
                         float* obs_slot, float* share_obs_slot, float* rewards_slot, float* masks_slot,
                         float* h_actor_slot, float* h_critic_slot, float* active_slot, float* avail_slot,
                         uint64_t* rng_counter_dev, uint64_t rng_inc, void* stream);

/* ---- a3 + a4(denormalise) + a5(statistics): compute_returns ---------------------------------
 * SharedReplayBuffer.compute_returns (shared_buffer.py:179-262, non-MAT branches) as one backward
 * scan, one thread per (n,m) lane; ValueNorm.denormalize (utils/valuenorm.py:68-79) folded in
 * (vn_state = {running_mean, running_mean_sq, debiasing_term} or NULL); also emits the raw
 * advantages returns - denorm(value_preds) and accumulates {sum, sum^2, count} over active entries
 * into adv_stats (3 doubles, caller zeroes) for R_MAPPO.train's normalisation (r_mappo.py:179-187).
 * value_preds must already hold next_value in slot T (shared_buffer.py:218). */
int32_t mappo_compute_returns(const float* rewards, const float* value_preds, const float* masks,
                              const float* bad_masks, const float* active_masks, const float* vn_state,
                              int32_t T, int32_t E, float gamma, float gae_lambda,
                              int32_t use_gae, int32_t use_proper_time_limits,
                              float* returns, float* advantages, double* adv_stats, void* stream);

/* Stand-alone a5 for callers that wrote `returns` themselves: advantages[i] = returns[i] -
 * denorm(value_preds[i]) over n entries + the same masked statistics (r_mappo.py:179-187). */
int32_t mappo_advantages(const float* returns, const float* value_preds, const float* active_masks,
                         const float* vn_state, int32_t n, float* advantages, double* adv_stats, void* stream);

/* ---- a4: ValueNorm.update + per-minibatch loss normalisers ----------------------------------
 * Reduces one minibatch: stats[0]=sum(active), [1]=sum(returns), [2]=sum(returns^2), [3]=n_rows
 * (doubles; caller zeroes).  Multi-GPU: the caller all-reduces `stats` before applying them. */
int32_t mappo_minibatch_stats(const float* returns, const float* active_masks, const int32_t* rows,
                              int32_t n_rows, double* stats, void* stream);
/* Kernels this library has launched (or recorded into a CUDA graph capture) since it was loaded. */
int64_t mappo_debug_launch_count(void);
/* The same for every minibatch of a train() call in one launch: rows of update u start at rows + u*rows_stride, its
 * statistics land in stats[4u .. 4u+3]. */
int32_t mappo_minibatch_stats_batch(const float* returns, const float* active_masks, const int32_t* rows,
                                    int64_t rows_stride, int32_t n_rows, int32_t n_batches, double* stats, void* stream);
/* ValueNorm.update (utils/valuenorm.py:38-55) from reduced statistics: vn_state <- beta-blend. */
int32_t mappo_valuenorm_update(float* vn_state, const double* stats, void* stream);

/* ---- a6 / a7: materialising gathers (only for callers that want the 12-tuples) --------------
 * dst[p, :] = src[rows[p], :]  (feed_forward_generator shared_buffer.py:377-396; the chunked
 * recurrent_generator :557-604 and naive_recurrent_generator :409-497 reduce to the same gather
 * once `rows` is built by mappo_chunk_rows / host arithmetic). */
int32_t mappo_gather_rows(const float* src, const int32_t* rows, int32_t n_rows, int32_t dim, float* dst,
                          void* stream);
/* Row list of recurrent_generator for the chunk ids in `chunks` [n_chunks]: rows[l*n_chunks + c] =
 * storage row of (n,m,t)-ordered position chunks[c]*L + l, first[c] = rows[0*n_chunks + c]
 * (shared_buffer.py:505-569, _cast :11-12; chunks may straddle trajectories when T % L != 0). */
int32_t mappo_chunk_rows(const int32_t* chunks, int32_t n_chunks, int32_t L, int32_t T, int32_t E,
                         int32_t* rows, int32_t* first, void* stream);
/* Device-side random permutation of [0, n) (stand-in for torch.randperm when the host RNG stream
 * is not being reproduced): keyed Feistel network with cycle walking, seed + *counter_dev. */
int32_t mappo_randperm(int32_t n, uint64_t seed, const uint64_t* counter_dev, int32_t* out, void* stream);
/* n_perms independent permutations (one per ppo epoch) in one launch: out[e*n .. (e+1)*n). */
int32_t mappo_randperm_batch(int32_t n, int32_t n_perms, uint64_t seed, const uint64_t* counter_dev, int32_t* out,
                             void* stream);

/* ---- a9 - a12: training forward + losses + backward -----------------------------------------
 * policy.evaluate_actions (rMAPPOPolicy.py:88-114; r_actor_critic.py:73-117, 156-175;
 * act.py:115-178) + the surrogate / entropy / value losses (r_mappo.py:52-89, 129-146, 156-160)
 * + their gradients (what autograd computes at :146 and :160), for one net per call.
 *   norm_stats : the reduced minibatch statistics (4 doubles, see mappo_minibatch_stats)
 *   adv_stats  : {sum, sum^2, count} of raw advantages over active entries (3 doubles)
 *   vn_state   : ValueNorm state AFTER this minibatch's update (critic only; r_mappo.py:65)
 *   grad_part  : workspace [n_slots, layout.total]; slot s receives the partial gradient of the
 *                tiles handled by CTA s (deterministic two-stage reduction; zeroed by this call)
 *   loss_out   : 6 doubles accumulated: [0] value_loss [1] policy_loss [2] dist_entropy
 *                [5] ratio mean (caller zeroes; [3],[4] are the grad norms written by the optimiser)
 *   workspace  : >= mappo_update_workspace_floats() floats, 16-byte aligned (recurrent nets: activations between
 *                the four launches; MAPPO_GEMM_TF32: the folded tf32 weight image fetched by TMA). */
int64_t mappo_update_workspace_floats(const mappo_net_desc_t* desc, int32_t n_rows, int32_t gemm_mode);
int32_t mappo_update_grad_slots(const mappo_net_desc_t* desc, int32_t n_rows, int32_t gemm_mode);
/* 1 if the tcgen05 (MAPPO_GEMM_TF32) kernels cover this net, else 0 (callers then use MAPPO_GEMM_FP32). */
int32_t mappo_tf32_supported(const mappo_net_desc_t* desc);
/* Diagnostic: clock64() phase stamps of CTA 0 of the last tcgen05 update launch (16 values, host pointer; syncs). */
int32_t mappo_debug_tc_timing(int64_t* out16);
/* Accumulated clock64 cycles of the rollout kernels' CTA 0, [8*net + phase] (phase 0 row load, 1 MLP base, 2 GRU cell,
 * 3 head GEMM, 4 sampling + outputs); `reset` != 0 zeroes the counters after reading. */
int32_t mappo_debug_pol_timing(int64_t* out16, int32_t reset);
int32_t mappo_update_fwd_bwd(const mappo_net_desc_t* desc, const float* params, const mappo_batch_t* batch,
                             const mappo_loss_cfg_t* loss, const double* norm_stats,
                             const double* adv_stats, const float* vn_state,
                             float* grad_part, int32_t n_slots, double* loss_out, float* workspace,
                             void* stream);

/* Gradient-free half of the same kernels = policy.evaluate_actions (rMAPPOPolicy.py:88-114):
 * actor -> out[n_rows, as] log-probs of batch->actions, loss_out[2] += dist_entropy (act.py:170-176);
 * critic -> out[n_rows, 1] values.  Loss-only inputs of `batch` may be NULL. */
int32_t mappo_evaluate_actions(const mappo_net_desc_t* desc, const float* params, const mappo_batch_t* batch,
                               const mappo_loss_cfg_t* loss, const double* norm_stats, float* out,
                               double* loss_out, float* workspace, void* stream);

/* ---- C1: the multi-GPU exchange (none in the reference: single process) ---------------------------------------
 * One-shot all-reduce over peer-mapped memory (NVLink 5 / NVSwitch) as ONE kernel per rank -- no host involvement, so
 * the whole multi-GPU iteration stays a single CUDA graph.  peer_bufs[p] / peer_signals[p] (HOST arrays of `world`
 * device pointers, world <= 8): rank p's symmetric buffer and its signal pad uint32[world] (zero-initialised), both
 * mapped into this process.  out[i] = sum_p peer_bufs[p][offset_bytes + i] in rank order (bit-identical on every
 * rank).  round_dev: device uint32[2] = {completed rounds, scratch}, zero-initialised, private to this rank; every
 * rank must issue the same sequence of calls.  A region of the symmetric buffer may be rewritten once a LATER call has
 * completed locally (each call is a full barrier): alternate two regions for back-to-back reductions.
 * f32 only: sumsq_part (nullable) receives *n_sumsq_blocks_out per-CTA sums of squares of the reduced vector -- exactly
 * what mappo_clip_adam takes, so no separate mappo_grad_sumsq launch follows the collective. */
int32_t mappo_p2p_allreduce_f32(const void* const* peer_bufs, void* const* peer_signals, int32_t world, int32_t rank,
                                int64_t offset_bytes, int32_t n, float* out, uint32_t* round_dev, float* sumsq_part,
                                int32_t* n_sumsq_blocks_out, void* stream);
int32_t mappo_p2p_allreduce_f64(const void* const* peer_bufs, void* const* peer_signals, int32_t world, int32_t rank,
                                int64_t offset_bytes, int32_t n, double* out, uint32_t* round_dev, void* stream);

/* ---- a13: gradient reduction + clip_grad_norm_ + Adam ----------------------------------------
 * Sums the partial-gradient slots into `grad` [n_params] (the buffer a multi-GPU caller
 * all-reduces), nn.utils.clip_grad_norm_ (r_mappo.py:148-151, 162-165; SURVEY App. A.6) and
 * torch.optim.Adam(lr, eps, betas=(0.9,0.999), weight_decay=0) (rMAPPOPolicy.py:31-37).
 *   mappo_grad_reduce : grad = sum_s grad_part[s]; sumsq_part[b] = per-block sum(grad^2)
 *   mappo_clip_adam   : total = sqrt(sum sumsq_part); coef = min(1, max_norm/(total+1e-6)) when
 *                       use_max_grad_norm; Adam step with g*coef; ++step_dev[0]; *grad_norm_out += total.
 *                       step_dev points to TWO ints: {Adam step count, scratch ticket (keep 0)}.
 *                       beta_pow_dev (nullable): THREE doubles {0.9^t, 0.999^t, t}, a cache of the bias-correction powers
 *                       the kernel keeps itself (any content is safe: a stale tag just recomputes with pow()).
 * lr is read from device memory (lr_dev[0]) so lr_decay (utils/util.py:17-21) needs no re-capture. */
/* Floats per gradient slot (`grad_part` holds n_slots of them): n_params for the fp32 build; the tcgen05 build
 * parks its still-folded TMEM accumulators (dW', db' columns) instead. */
int32_t mappo_update_slot_floats(const mappo_net_desc_t* desc, int32_t gemm_mode);
/* Slot reduction for either build: sums the slots into the flat gradient `grad` [n_params] (tcgen05 build: sums the raw
 * accumulators into the workspace, then unfolds the LayerNorm/bias folding once) and leaves *n_blocks_out partial sums
 * of squares in sumsq_part for mappo_clip_adam. */
int32_t mappo_update_finish(const mappo_net_desc_t* desc, const float* params, const float* grad_part, int32_t n_slots,
                            int32_t gemm_mode, float* grad, float* sumsq_part, int32_t* n_blocks_out, float* workspace,
                            void* stream);
/* The optimiser tail of one MAPPO_GEMM_TF32 hidden-64 net as ONE launch (one 8-CTA thread-block cluster, stages separated by
 * cluster barriers): `stages` bit 0 = mappo_update_finish (slot sum + unfold -> grad, 12 partial sums of squares in sumsq_part);
 * bit 1 = mappo_clip_adam on `grad` (reading n_sumsq_blocks partials; 12 when bit 0 ran in the same launch) followed by the
 * folded weight image of the NEW parameters into `workspace` -- so the next mappo_update_fwd_bwd may be called with
 * mappo_loss_cfg_t.image_ready = 1 and launches no pack kernel.  Bit-identical to the separate calls.  A multi-GPU caller
 * runs stages = 1, its all-reduce of `grad`, then stages = 2 -- or stages = 7: bit 2 puts the exchange INSIDE the launch
 * (mappo_p2p_allreduce_f32's protocol, arguments and summation order: the local gradient is written at sym_offset_bytes of this
 * rank's symmetric buffer, every rank sums all peers' copies into `grad`), so a data-parallel optimiser step is the update kernel
 * plus this one launch.  peer_* / world / rank / round_dev as in mappo_p2p_allreduce_f32 (ignored unless bit 2 is set).
 * workspace as for mappo_update_fwd_bwd / mappo_update_finish. */
int32_t mappo_update_tail(const mappo_net_desc_t* desc, float* params, const float* grad_part, int32_t n_slots, float* grad,
                          float* exp_avg, float* exp_avg_sq, float* sumsq_part, int32_t n_sumsq_blocks, const float* lr_dev,
                          int32_t* step_dev, float eps, float max_grad_norm, int32_t use_max_grad_norm, double* grad_norm_out,
                          double* beta_pow_dev, float* workspace, int32_t stages, const void* const* peer_bufs,
                          void* const* peer_signals, int32_t world, int32_t rank, int64_t sym_offset_bytes, uint32_t* round_dev,
                          void* stream);
int32_t mappo_grad_reduce(const float* grad_part, int32_t n_slots, int32_t n_params, float* grad,
                          float* sumsq_part, int32_t* n_sumsq_blocks_out, void* stream);
/* Per-block sums of squares of an already reduced (e.g. all-reduced) gradient vector. */
int32_t mappo_grad_sumsq(const float* grad, int32_t n_params, float* sumsq_part, int32_t* n_sumsq_blocks_out,
                         void* stream);
int32_t mappo_clip_adam(float* params, const float* grad, float* exp_avg, float* exp_avg_sq,
                        int32_t n_params, const float* sumsq_part, int32_t n_sumsq_blocks,
                        const float* lr_dev, int32_t* step_dev, float eps, float max_grad_norm,
                        int32_t use_max_grad_norm, double* grad_norm_out, double* beta_pow_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MAPPO_B200_H_ */
