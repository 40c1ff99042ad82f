// mpe_env.cu -- N vectorised MPE `simple_spread` / `simple_reference` worlds stepped on the device (SURVEY.md section 8(f), row f1).
//
// Replaces, for this scenario, SubprocVecEnv.step -> MultiAgentEnv.step -> World.step + the scenario callbacks
// (envs/env_wrappers.py:140-154, envs/mpe/environment.py:115-146, envs/mpe/core.py:207-323,
// envs/mpe/scenarios/simple_spread.py:32-103): action decoding, action + contact forces, damping / integration, reward
// (minimum agent distance per landmark, collision penalties incl. the reference's self-"collision", summed over the
// agents of the world), observation, done = step >= episode_length, auto-reset with the reset observation replacing the
// terminal one.  The state is float64 and every expression keeps the reference's order of operations (mpe_world.cuh), so a
// trajectory follows the NumPy one to the last bits of exp / log1p (the only non-IEEE-exact operations involved).
// One thread per world: a world is 6 entities, the work per step is a few hundred flops -- pure latency; what this buys
// is a rollout without a host round trip (the reference pays a pipe round trip + NumPy physics per env step).
#include "launch_args.h"
#include "mpe_world.cuh"

namespace mappo {

template <int MT, int LT>
__global__ void __launch_bounds__(128) mpe_spread_kernel(const MpeArgs a) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.N) return;
  const int M = a.M, L = a.L;
  MpeWorld w;
  mpe_world_load<MT, LT>(w, M, L, a.apos, a.avel, a.lpos, a.step_count, e);
  const double* rs = a.reset_states ? a.reset_states + (size_t)e * 2 * (M + L) : nullptr;
  const uint64_t ctr = a.reset_states ? 0ull : *a.rng_counter + (uint64_t)e;
  double reward = 0.0;
  bool done = false;
  if (!a.actions) {                      // envs.reset()
    mpe_world_reset<MT, LT>(w, M, L, rs, a.rng_seed, ctr);
  } else {
    int act[kMpeMaxAgents];
    for (int m = 0; m < M; ++m) act[m] = (int)a.actions[(size_t)e * M + m];
    reward = mpe_world_step<MT, LT>(w, M, L, act, a.episode_length, &done);
    if (done) mpe_world_reset<MT, LT>(w, M, L, rs, a.rng_seed, ctr);   // env_wrappers.py:146-152: the reset obs replaces the terminal one
  }
  mpe_world_store<MT, LT>(w, M, L, a.apos, a.avel, a.lpos, a.step_count, e);
  const int D = 4 + 2 * L + 4 * (M - 1);
  for (int m = 0; m < M; ++m) {
    mpe_world_obs<MT, LT>(w, M, L, m, a.obs + ((size_t)e * M + m) * D);
    if (a.actions) {
      a.rewards[(size_t)e * M + m] = (float)reward;
      a.dones[(size_t)e * M + m] = done ? 1.f : 0.f;
    }
  }
  if (a.share_obs) {                     // share_obs = all agents' obs of the world (mpe_runner.py:133-135)
    const float* src = a.obs + (size_t)e * M * D;            // written above by this thread
    for (int m = 0; m < M; ++m) {
      float* s = a.share_obs + ((size_t)e * M + m) * (size_t)(M * D);
      for (int i = 0; i < M * D; ++i) s[i] = src[i];
    }
  }
}

int mpe_spread_launch(const MpeArgs& a, cudaStream_t st) {
  if (a.M < 1 || a.M > kMpeMaxAgents || a.L < 1 || a.L > kMpeMaxLandmarks) { set_error("mpe_spread: %d agents / %d landmarks outside [1,8]", a.M, a.L); return MAPPO_ERR_UNSUPPORTED; }
  if (a.M == 3 && a.L == 3) mpe_spread_kernel<3, 3><<<(a.N + 127) / 128, 128, 0, st>>>(a);      // the reference's default shape
  else mpe_spread_kernel<0, 0><<<(a.N + 127) / 128, 128, 0, st>>>(a);
  return check_launch("mpe_spread_kernel");
}

// ---- `simple_reference` (BASELINE configs[2]'s scenario; the world functions are in mpe_world.cuh) -------------------
__global__ void __launch_bounds__(128) mpe_reference_kernel(const MpeRefArgs a) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.N) return;
  constexpr int M = kRefAgents;
  MpeRefWorld w;
  ref_world_load(w, a.apos, a.avel, a.lpos, a.goal, a.comm, a.step_count, e);
  double reward = 0.0;
  bool done = false;
  if (a.actions) {
    int mv[M], sym[M];
    for (int m = 0; m < M; ++m) { mv[m] = (int)a.actions[((size_t)e * M + m) * 2]; sym[m] = (int)a.actions[((size_t)e * M + m) * 2 + 1]; }
    reward = ref_world_step(w, mv, sym, a.episode_length, &done);
  }
  if (!a.actions || done)                  // reset_world; env_wrappers.py:146-152
    ref_world_reset(w, a.reset_states ? a.reset_states + (size_t)e * kRefResetDoubles : nullptr, a.rng_seed,
                    a.reset_states ? 0ull : *a.rng_counter + (uint64_t)e);
  ref_world_store(w, a.apos, a.avel, a.lpos, a.goal, a.comm, a.step_count, e);
  for (int m = 0; m < M; ++m) {
    ref_world_obs(w, m, a.obs + ((size_t)e * M + m) * kRefObs);
    if (a.actions) {
      a.rewards[(size_t)e * M + m] = (float)reward;
      a.dones[(size_t)e * M + m] = done ? 1.f : 0.f;
    }
  }
  if (a.share_obs) {
    const float* src = a.obs + (size_t)e * M * kRefObs;
    for (int m = 0; m < M; ++m) {
      float* s = a.share_obs + ((size_t)e * M + m) * (size_t)(M * kRefObs);
      for (int i = 0; i < M * kRefObs; ++i) s[i] = src[i];
    }
  }
}

int mpe_reference_launch(const MpeRefArgs& a, cudaStream_t st) {
  mpe_reference_kernel<<<(a.N + 127) / 128, 128, 0, st>>>(a);
  return check_launch("mpe_reference_kernel");
}

}  // namespace mappo
