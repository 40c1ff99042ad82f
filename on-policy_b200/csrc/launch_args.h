// launch_args.h -- argument blocks shared between api.cu and the kernel translation units.
#pragma once
#include "common.cuh"

namespace mappo {

struct PolArgs {
  const float* params[2];      // [0] actor, [1] critic
  const float* image[2];       // optional pre-packed shared-memory weight images (mappo_pack_rollout_weights)
  const float* in[2];          // obs, share_obs
  const float* h_in[2];
  float* h_out[2];
  const float* masks;
  const float* avail;
  const float* exp_noise;
  uint64_t rng_seed;
  const uint64_t* rng_offset;
  int deterministic, n_rows, n_avail;
  float* values;
  float* actions;
  int64_t* actions_i64;
  float* logp;
};

struct InsertArgs {
  const float *next_obs, *next_share, *rewards, *dones, *next_active, *next_avail;
  int E, Do, Ds, H, A;
  float *obs, *share, *rew, *masks, *ha, *hc, *active, *avail;
  uint64_t* rng_counter;
  uint64_t rng_inc;
};

struct RolloutArgs {
  const float* params[2];
  const float* image[2];
  float *obs, *share_obs, *h_actor, *h_critic, *masks, *avail, *value_preds, *actions, *logp, *rewards, *active;
  const float *f_obs, *f_share, *f_rew, *f_done, *f_active, *f_avail;
  const float* exp_noise;
  uint64_t rng_seed;
  uint64_t* rng_offset;
  int T, E, n_avail;
  int share_agents;            // > 0: no staged share_obs -- a critic row is the concatenation of the obs rows of the
                               // `share_agents` agents of its rollout thread (mpe_runner.py:133-135), read from f_obs
};
// f1: vectorised MPE simple_spread worlds (mpe_env.cu)
struct MpeArgs {
  double *apos, *avel, *lpos;            // [N][M][2], [N][M][2], [N][L][2]
  int32_t* step_count;                   // [N]
  const float* actions;                  // [N*M] integer-valued (Discrete(5)); NULL = reset only
  const double* reset_states;            // [N][2 (M + L)] or NULL (device RNG)
  uint64_t rng_seed;
  const uint64_t* rng_counter;
  int N, M, L, episode_length;
  float *obs, *share_obs, *rewards, *dones;   // [N*M][D], [N*M][M*D] (nullable), [N*M], [N*M]
};
int mpe_spread_launch(const MpeArgs& a, cudaStream_t st);
struct MpeRefArgs {                      // `simple_reference`: 2 agents, 3 landmarks, 10 symbols
  double *apos, *avel, *lpos;            // [N][2][2], [N][2][2], [N][3][2]
  int32_t *goal, *comm, *step_count;     // [N][2] goal landmark, [N][2] last symbol (-1 = silent), [N]
  const float* actions;                  // [N*2][2] integer-valued (move 0..4, symbol 0..9); NULL = reset only
  const double* reset_states;            // [N][12]: goal_0, goal_1, agent positions, landmark positions; or NULL (device RNG)
  uint64_t rng_seed;
  const uint64_t* rng_counter;
  int N, episode_length;
  float *obs, *share_obs, *rewards, *dones;   // [N*2][21], [N*2][42] (nullable), [N*2], [N*2]
};
int mpe_reference_launch(const MpeRefArgs& a, cudaStream_t st);

// closed rollout loop with the device-side MPE worlds (rollout_closed.cuh)
struct ClosedArgs {
  RolloutArgs r;                     // storage pointers (h_actor / h_critic: recurrent nets), images, sampling noise / RNG, T, E
                                     // (f_* unused)
  int world;                         // MAPPO_WORLD_SPREAD / MAPPO_WORLD_REFERENCE
  double *apos, *avel, *lpos;        // world state [N][M][2], [N][M][2], [N][L][2]
  int32_t *goal, *comm;              // simple_reference only: [N][2] each (NULL for simple_spread)
  int32_t* step_count;               // [N]
  const double* reset_states;        // [T][N][per-world doubles] episode starts to use when a world ends at step t, or NULL (Philox)
  uint64_t env_seed;
  const uint64_t* env_counter;
  int M, L, episode_length;
};
int rollout_closed_launch(const NetDev& na, const NetDev& nc, const ClosedArgs& ca, cudaStream_t st);
int rollout_persistent_launch(const NetDev& na, const NetDev& nc, const RolloutArgs& a, cudaStream_t st);
int policy_step_launch(const NetDev* na, const NetDev* nc, const PolArgs& a, cudaStream_t st);
int env_insert_launch(const InsertArgs& a, cudaStream_t st);

}  // namespace mappo
