// mpe_world.cuh -- one MPE `simple_spread` or `simple_reference` world in registers: load / reset / step / observation /
// store (device functions shared by the standalone env kernels, mpe_env.cu, and the closed-loop rollout kernels,
// rollout_closed.cuh).
//
// Mirrors envs/mpe/core.py:207-323, envs/mpe/environment.py:115-262 and envs/mpe/scenarios/simple_spread.py:32-103 in
// float64 with the reference's order of operations.  Every arithmetic step is an explicit round-to-nearest intrinsic
// (__dmul_rn / __dadd_rn / ...): those are never contracted into fused multiply-adds, so the results do not depend on
// the translation unit's -fmad setting and follow NumPy bit for bit up to exp / log1p of the contact term.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "rng.cuh"

namespace mappo {

constexpr int kMpeMaxAgents = 8, kMpeMaxLandmarks = 8;
constexpr double kAgentSize = 0.15;      // simple_spread.py:22
constexpr double kContactForce = 1e2;    // core.py:128
constexpr double kContactMargin = 1e-3;  // core.py:129
constexpr double kDamping = 0.25;        // core.py:126
constexpr double kDt = 0.1;              // core.py:124
constexpr double kSensitivity = 5.0;     // environment.py:243

struct MpeWorld {
  double ap[kMpeMaxAgents][2], av[kMpeMaxAgents][2], lp[kMpeMaxLandmarks][2];
  int step;
};

__device__ __forceinline__ double d_add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double d_sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double d_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double d_div(double a, double b) { return __ddiv_rn(a, b); }
// np.sqrt(np.sum(np.square(delta))) for a 2-vector
__device__ __forceinline__ double d_norm2(double dx, double dy) { return __dsqrt_rn(d_add(d_mul(dx, dx), d_mul(dy, dy))); }

// np.logaddexp(0, y) (numpy/core/src/npymath/npy_math_internal.h.src: npy_logaddexp)
__device__ __forceinline__ double logaddexp0(double y) {
  if (y == 0.0) return 0.6931471805599453094172321214581766;
  const double tmp = d_sub(0.0, y);
  if (tmp > 0) return d_add(0.0, log1p(exp(-tmp)));
  if (tmp <= 0) return d_add(y, log1p(exp(tmp)));
  return tmp;
}

// scenario.reset_world (simple_spread.py:32-45): positions from `s` (agents then landmarks, 2 (M + L) doubles) or, when s is
// NULL, uniform(-1, 1) / 0.8 uniform(-1, 1) from Philox keyed by (seed, ctr)
// MT / LT: compile-time agent / landmark counts (0 = use the runtime M / L).  With constants every loop unrolls and the world
// lives in registers; the arithmetic and its order are the same.
template <int MT = 0, int LT = 0>
__device__ __forceinline__ void mpe_world_reset(MpeWorld& w, int Mr, int Lr, const double* __restrict__ s, uint64_t seed,
                                                uint64_t ctr) {
  const int M = MT ? MT : Mr, L = LT ? LT : Lr;
  if (s) {
    for (int m = 0; m < M; ++m) { w.ap[m][0] = s[2 * m]; w.ap[m][1] = s[2 * m + 1]; }
    for (int l = 0; l < L; ++l) { w.lp[l][0] = s[2 * (M + l)]; w.lp[l][1] = s[2 * (M + l) + 1]; }
  } else {
    for (int q = 0; q < (2 * (M + L) + 3) / 4; ++q) {
      const uint4 r = philox4x32_10(make_uint4((uint32_t)ctr, (uint32_t)(ctr >> 32), 0x4d504500u + q, 0u),
                                    make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
      const uint32_t v[4] = {r.x, r.y, r.z, r.w};
      for (int j = 0; j < 4; ++j) {
        const int i = 4 * q + j;
        if (i >= 2 * (M + L)) break;
        const double u = d_add(-1.0, d_mul(2.0, d_mul(d_add((double)v[j], 0.5), 2.3283064365386962890625e-10)));
        if (i < 2 * M) w.ap[i >> 1][i & 1] = u;
        else w.lp[(i - 2 * M) >> 1][i & 1] = d_mul(0.8, u);
      }
    }
  }
  for (int m = 0; m < M; ++m) w.av[m][0] = w.av[m][1] = 0.0;
  w.step = 0;
}

// MultiAgentEnv.step for integer actions act[m] in 0..4 (what the one-hot the runner sends decodes to): returns the shared
// reward; *done = the episode ended (the caller resets, env_wrappers.py:146-152).
template <int MT = 0, int LT = 0>
__device__ __forceinline__ double mpe_world_step(MpeWorld& w, int Mr, int Lr, const int* act, int episode_length, bool* done) {
  const int M = MT ? MT : Mr, L = LT ? LT : Lr;
  double f[kMpeMaxAgents][2];
#pragma unroll
  for (int m = 0; m < M; ++m) {          // environment.py:232-246 (_set_action), core.py:229-238 (apply_action_force)
    double u0 = 0.0, u1 = 0.0;
    u0 = d_add(u0, d_sub(act[m] == 1 ? 1.0 : 0.0, act[m] == 2 ? 1.0 : 0.0));
    u1 = d_add(u1, d_sub(act[m] == 3 ? 1.0 : 0.0, act[m] == 4 ? 1.0 : 0.0));
    u0 = d_mul(u0, kSensitivity); u1 = d_mul(u1, kSensitivity);
    f[m][0] = d_add(d_mul(1.0, u0), 0.0);
    f[m][1] = d_add(d_mul(1.0, u1), 0.0);
  }
#pragma unroll
  for (int ia = 0; ia < M; ++ia)         // core.py:241-265, 293-323: contacts between agents (landmarks do not collide)
#pragma unroll
    for (int ib = ia + 1; ib < M; ++ib) {
      const double dx = d_sub(w.ap[ia][0], w.ap[ib][0]), dy = d_sub(w.ap[ia][1], w.ap[ib][1]);
      const double dist = d_norm2(dx, dy);
      const double k = kContactMargin;
      const double pen = d_mul(logaddexp0(d_div(-d_sub(dist, d_add(kAgentSize, kAgentSize)), k)), k);
      const double fx = d_mul(d_div(d_mul(kContactForce, dx), dist), pen);
      const double fy = d_mul(d_div(d_mul(kContactForce, dy), dist), pen);
      f[ia][0] = d_add(fx, f[ia][0]); f[ia][1] = d_add(fy, f[ia][1]);
      f[ib][0] = d_add(-fx, f[ib][0]); f[ib][1] = d_add(-fy, f[ib][1]);
    }
#pragma unroll
  for (int m = 0; m < M; ++m)            // core.py:267-281 (integrate_state)
#pragma unroll
    for (int d = 0; d < 2; ++d) {
      double v = d_mul(w.av[m][d], 1 - kDamping);
      v = d_add(v, d_mul(d_div(f[m][d], 1.0), kDt));
      w.av[m][d] = v;
      w.ap[m][d] = d_add(w.ap[m][d], d_mul(v, kDt));
    }
  w.step += 1;
  double reward = 0.0;                   // simple_spread.py:72-85, shared reward = sum over agents (environment.py:139-142)
#pragma unroll
  for (int m = 0; m < M; ++m) {
    double rew = 0.0;
#pragma unroll
    for (int l = 0; l < L; ++l) {
      double mn = 0.0;
#pragma unroll
      for (int q = 0; q < M; ++q) {
        const double d = d_norm2(d_sub(w.ap[q][0], w.lp[l][0]), d_sub(w.ap[q][1], w.lp[l][1]));
        mn = (q == 0 || d < mn) ? d : mn;
      }
      rew = d_sub(rew, mn);
    }
#pragma unroll
    for (int q = 0; q < M; ++q)          // q == m included: an agent "collides" with itself in the reference
      if (d_norm2(d_sub(w.ap[q][0], w.ap[m][0]), d_sub(w.ap[q][1], w.ap[m][1])) < d_add(kAgentSize, kAgentSize))
        rew = d_sub(rew, 1.0);
    reward = m == 0 ? rew : d_add(reward, rew);
  }
  *done = w.step >= episode_length;
  return reward;
}

// scenario.observation of agent m (simple_spread.py:87-103) as float32 (what the rollout storage keeps):
// vel, pos, landmarks - pos, other agents - pos, other agents' (silent => zero) communication
template <int MT = 0, int LT = 0>
__device__ __forceinline__ void mpe_world_obs(const MpeWorld& w, int Mr, int Lr, int m, float* __restrict__ o) {
  const int M = MT ? MT : Mr, L = LT ? LT : Lr;
  int c = 0;
  o[c++] = (float)w.av[m][0]; o[c++] = (float)w.av[m][1];
  o[c++] = (float)w.ap[m][0]; o[c++] = (float)w.ap[m][1];
  for (int l = 0; l < L; ++l) { o[c++] = (float)d_sub(w.lp[l][0], w.ap[m][0]); o[c++] = (float)d_sub(w.lp[l][1], w.ap[m][1]); }
  for (int q = 0; q < M; ++q)
    if (q != m) { o[c++] = (float)d_sub(w.ap[q][0], w.ap[m][0]); o[c++] = (float)d_sub(w.ap[q][1], w.ap[m][1]); }
  for (int q = 0; q < M; ++q)
    if (q != m) { o[c++] = 0.f; o[c++] = 0.f; }
}

template <int MT = 0, int LT = 0>
__device__ __forceinline__ void mpe_world_load(MpeWorld& w, int Mr, int Lr, const double* __restrict__ apos,
                                               const double* __restrict__ avel, const double* __restrict__ lpos,
                                               const int32_t* __restrict__ step_count, int e) {
  const int M = MT ? MT : Mr, L = LT ? LT : Lr;
  for (int m = 0; m < M; ++m)
    for (int d = 0; d < 2; ++d) { w.ap[m][d] = apos[((size_t)e * M + m) * 2 + d]; w.av[m][d] = avel[((size_t)e * M + m) * 2 + d]; }
  for (int l = 0; l < L; ++l)
    for (int d = 0; d < 2; ++d) w.lp[l][d] = lpos[((size_t)e * L + l) * 2 + d];
  w.step = step_count[e];
}
template <int MT = 0, int LT = 0>
__device__ __forceinline__ void mpe_world_store(const MpeWorld& w, int Mr, int Lr, double* __restrict__ apos,
                                                double* __restrict__ avel, double* __restrict__ lpos,
                                                int32_t* __restrict__ step_count, int e) {
  const int M = MT ? MT : Mr, L = LT ? LT : Lr;
  for (int m = 0; m < M; ++m)
    for (int d = 0; d < 2; ++d) { apos[((size_t)e * M + m) * 2 + d] = w.ap[m][d]; avel[((size_t)e * M + m) * 2 + d] = w.av[m][d]; }
  for (int l = 0; l < L; ++l)
    for (int d = 0; d < 2; ++d) lpos[((size_t)e * L + l) * 2 + d] = w.lp[l][d];
  step_count[e] = w.step;
}

// ---- `simple_reference` (BASELINE configs[2]'s scenario) -------------------------------------------------------------
// envs/mpe/scenarios/simple_reference.py:8-97: 2 agents, 3 landmarks, 10 communication symbols, nothing collides.  Agent m
// wants the OTHER agent on landmark goal[m]; both receive r_0 + r_1, r_m = -|pos[1 - m] - landmark[goal_m]|^2 (:62-67 with
// shared_reward, environment.py:139-142).  Action = MultiDiscrete([[0,4],[0,9]]) (environment.py:55-63): a movement head
// decoded like simple_spread's and a symbol head that becomes the agent's communication state (core.py:283-290, c_noise
// None).  Observation (:69-97) = velocity, landmarks - pos, colour of the goal landmark, the other agent's communication.
constexpr int kRefAgents = 2, kRefLandmarks = 3, kRefSymbols = 10, kRefObs = 2 + 2 * kRefLandmarks + 3 + kRefSymbols;
constexpr int kRefResetDoubles = 2 + 2 * (kRefAgents + kRefLandmarks);   // goal_0, goal_1, agent positions, landmark positions

struct MpeRefWorld {
  double ap[kRefAgents][2], av[kRefAgents][2], lp[kRefLandmarks][2];
  int goal[kRefAgents], comm[kRefAgents];   // comm: the symbol uttered last step, -1 = silent
  int step;
};

__device__ __forceinline__ void ref_world_load(MpeRefWorld& w, const double* __restrict__ apos, const double* __restrict__ avel,
                                               const double* __restrict__ lpos, const int32_t* __restrict__ goal,
                                               const int32_t* __restrict__ comm, const int32_t* __restrict__ step_count, int e) {
  constexpr int M = kRefAgents, L = kRefLandmarks;
  for (int m = 0; m < M; ++m)
    for (int d = 0; d < 2; ++d) { w.ap[m][d] = apos[((size_t)e * M + m) * 2 + d]; w.av[m][d] = avel[((size_t)e * M + m) * 2 + d]; }
  for (int l = 0; l < L; ++l)
    for (int d = 0; d < 2; ++d) w.lp[l][d] = lpos[((size_t)e * L + l) * 2 + d];
  for (int m = 0; m < M; ++m) { w.goal[m] = goal[(size_t)e * M + m]; w.comm[m] = comm[(size_t)e * M + m]; }
  w.step = step_count[e];
}
__device__ __forceinline__ void ref_world_store(const MpeRefWorld& w, double* __restrict__ apos, double* __restrict__ avel,
                                                double* __restrict__ lpos, int32_t* __restrict__ goal, int32_t* __restrict__ comm,
                                                int32_t* __restrict__ step_count, int e) {
  constexpr int M = kRefAgents, L = kRefLandmarks;
  for (int m = 0; m < M; ++m)
    for (int d = 0; d < 2; ++d) { apos[((size_t)e * M + m) * 2 + d] = w.ap[m][d]; avel[((size_t)e * M + m) * 2 + d] = w.av[m][d]; }
  for (int l = 0; l < L; ++l)
    for (int d = 0; d < 2; ++d) lpos[((size_t)e * L + l) * 2 + d] = w.lp[l][d];
  for (int m = 0; m < M; ++m) { goal[(size_t)e * M + m] = w.goal[m]; comm[(size_t)e * M + m] = w.comm[m]; }
  step_count[e] = w.step;
}

// reset_world (:35-60; env_wrappers.py:146-152): goals and positions from `s` (kRefResetDoubles doubles) or, when s is NULL,
// from Philox keyed by (seed, ctr); at rest and silent (state.c = zeros)
__device__ __forceinline__ void ref_world_reset(MpeRefWorld& w, const double* __restrict__ s, uint64_t seed, uint64_t ctr) {
  constexpr int M = kRefAgents, L = kRefLandmarks;
  if (s) {
    w.goal[0] = (int)s[0]; w.goal[1] = (int)s[1];
    for (int m = 0; m < M; ++m) { w.ap[m][0] = s[2 + 2 * m]; w.ap[m][1] = s[3 + 2 * m]; }
    for (int l = 0; l < L; ++l) { w.lp[l][0] = s[2 + 2 * (M + l)]; w.lp[l][1] = s[3 + 2 * (M + l)]; }
  } else {
    double uu[12];
    for (int q = 0; q < 3; ++q) {
      const uint4 r = philox4x32_10(make_uint4((uint32_t)ctr, (uint32_t)(ctr >> 32), 0x52454600u + q, 0u),
                                    make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
      const uint32_t v[4] = {r.x, r.y, r.z, r.w};
      for (int j = 0; j < 4; ++j) uu[4 * q + j] = d_mul(d_add((double)v[j], 0.5), 2.3283064365386962890625e-10);
    }
    w.goal[0] = min(L - 1, (int)d_mul(uu[10], (double)L)); w.goal[1] = min(L - 1, (int)d_mul(uu[11], (double)L));
    for (int i = 0; i < 2 * M; ++i) w.ap[i >> 1][i & 1] = d_add(-1.0, d_mul(2.0, uu[i]));
    for (int i = 0; i < 2 * L; ++i) w.lp[i >> 1][i & 1] = d_mul(0.8, d_add(-1.0, d_mul(2.0, uu[2 * M + i])));
  }
  for (int m = 0; m < M; ++m) { w.av[m][0] = w.av[m][1] = 0.0; w.comm[m] = -1; }
  w.step = 0;
}

// MultiAgentEnv.step for the (move, symbol) pairs mv[m], sym[m] (environment.py:184-250, core.py:229-238, :267-281, no
// contacts): returns the shared reward; *done = the episode ended (the caller resets)
__device__ __forceinline__ double ref_world_step(MpeRefWorld& w, const int* mv, const int* sym, int episode_length, bool* done) {
  constexpr int M = kRefAgents;
#pragma unroll
  for (int m = 0; m < M; ++m) {
    double u[2];
    u[0] = d_mul(d_add(0.0, d_sub(mv[m] == 1 ? 1.0 : 0.0, mv[m] == 2 ? 1.0 : 0.0)), kSensitivity);
    u[1] = d_mul(d_add(0.0, d_sub(mv[m] == 3 ? 1.0 : 0.0, mv[m] == 4 ? 1.0 : 0.0)), kSensitivity);
#pragma unroll
    for (int d = 0; d < 2; ++d) {
      const double f = d_add(d_mul(1.0, u[d]), 0.0);
      double v = d_mul(w.av[m][d], 1 - kDamping);
      v = d_add(v, d_mul(d_div(f, 1.0), kDt));
      w.av[m][d] = v;
      w.ap[m][d] = d_add(w.ap[m][d], d_mul(v, kDt));
    }
    w.comm[m] = sym[m] < 0 ? 0 : (sym[m] >= kRefSymbols ? kRefSymbols - 1 : sym[m]);
  }
  w.step += 1;
  double reward = 0.0;
#pragma unroll
  for (int m = 0; m < M; ++m) {            // simple_reference.py:62-67
    const double dx = d_sub(w.ap[1 - m][0], w.lp[w.goal[m]][0]), dy = d_sub(w.ap[1 - m][1], w.lp[w.goal[m]][1]);
    const double r = -d_add(d_mul(dx, dx), d_mul(dy, dy));
    reward = m == 0 ? r : d_add(reward, r);
  }
  *done = w.step >= episode_length;
  return reward;
}

// scenario.observation of agent m (:69-97) as float32: velocity, landmarks - pos, goal colour, the other agent's symbol one-hot
__device__ __forceinline__ void ref_world_obs(const MpeRefWorld& w, int m, float* __restrict__ o) {
  int c = 0;
  o[c++] = (float)w.av[m][0]; o[c++] = (float)w.av[m][1];
  for (int l = 0; l < kRefLandmarks; ++l) { o[c++] = (float)d_sub(w.lp[l][0], w.ap[m][0]); o[c++] = (float)d_sub(w.lp[l][1], w.ap[m][1]); }
  for (int k = 0; k < 3; ++k) o[c++] = k == w.goal[m] ? 0.75f : 0.25f;        // simple_reference.py:46-48
  for (int k = 0; k < kRefSymbols; ++k) o[c++] = k == w.comm[1 - m] ? 1.f : 0.f;
}

}  // namespace mappo
