// rollout_closed.cuh -- the CLOSED rollout loop of one iteration as ONE launch: policy step -> MPE world step -> insert,
// T times, plus the bootstrap value (SURVEY.md section 8(f) row f1 on top of a8 / a2).
// (included by policy_step.cu only, after rollout_mlp.cuh and rollout_gru.cuh)
//
// Unlike the persistent rollout kernels there is no staged feed: the observation of step t + 1 is produced from the action of
// step t inside the kernel, so the sequential dependence of on-policy rollouts is real here.  The world (`simple_spread` with
// M agents / L landmarks, or `simple_reference`) is a template parameter; its float64 state lives in the registers of ONE
// environment thread per world (mpe_world.cuh).  The critic's share_obs row is the world's M observations back to back
// (mpe_runner.py:133-135).
//
// Feed-forward policies (rollout_closed_kernel): a CTA owns kCG worlds -- for every world M actor warps and M critic warps (one
// row each, the warp-per-row path of rollout_mlp.cuh, both weight images in shared memory) and the environment thread.  Per step:
//   actor / critic warps: forward, sample, write values / actions / log-probs (and the row into its storage slot)
//   __syncthreads
//   environment thread: read the world's actions (every head), step the physics, reward / done -> storage, reset if the
//                       episode ended, new observations -> shared memory
//   __syncthreads
//   every warp picks its next row from shared memory.
//
// Recurrent (GRU) policies (rollout_closed_gru_kernel): the two weight images (~130 KB each) do not fit one CTA, so a world group
// runs on a 2-CTA CLUSTER.  CTA rank 0 holds the actor image, the actor warps (two rows each, gru_fast_step of rollout_gru.cuh)
// and the environment threads (lanes of warp 0, one per world); CTA rank 1 holds the critic image and the critic warps of the same
// rows.  Per step t:
//   actor CTA:  forward + sample step t -> __syncthreads -> environment threads step the worlds and write the observations of
//               t + 1 and the done flags into slot (t + 1) & 1 of their own shared memory AND, through DSMEM, of the critic CTA's
//               -> cluster barrier (arrive + wait)
//   critic CTA: arrive (its rows of step t are already in registers) -> forward step t -> wait
//   both:       read the next rows and done flags from slot (t + 1) & 1; done rows zero their state; store rnn_states[t + 1].
// The slot is double-buffered, so one cluster barrier per step orders everything: the environment overwrites a slot two steps
// later, after the critic has arrived past its read.  The critic never holds up the actor with its arithmetic.
// The done flag of env step t exists only after the actions of step t have been sampled, so the state reset that the per-step path
// does in mappo_env_insert happens here after the world step, and rnn_states[t + 1] gets the same values.
#pragma once
#include "rollout_mlp.cuh"
#include "rollout_gru.cuh"
#include "mpe_world.cuh"

namespace mappo {

constexpr int kCG = 2;               // worlds per CTA (feed-forward kernel)

// the world of the closed kernels: load / step / reset / obs / store of one world through the ClosedArgs it lives in
template <int MT, int LT>            // simple_spread; MT / LT: compile-time agent / landmark counts (0 = runtime)
struct SpreadClosedWorld {
  static constexpr int kM = MT;      // agents (0 = runtime ca.M)
  MpeWorld w;
  __device__ static int reset_doubles(const ClosedArgs& ca) { return 2 * (ca.M + ca.L); }
  __device__ void load(const ClosedArgs& ca, int e) { mpe_world_load<MT, LT>(w, ca.M, ca.L, ca.apos, ca.avel, ca.lpos, ca.step_count, e); }
  __device__ void store(const ClosedArgs& ca, int e) const { mpe_world_store<MT, LT>(w, ca.M, ca.L, ca.apos, ca.avel, ca.lpos, ca.step_count, e); }
  // act: the world's action rows [M][as]
  __device__ double step(const ClosedArgs& ca, const float* act, int as, bool* done) {
    const int M = MT ? MT : ca.M;
    int a[kMpeMaxAgents];
    for (int q = 0; q < M; ++q) a[q] = (int)act[q * as];
    return mpe_world_step<MT, LT>(w, ca.M, ca.L, a, ca.episode_length, done);
  }
  __device__ void reset(const ClosedArgs& ca, const double* s, uint64_t ctr) { mpe_world_reset<MT, LT>(w, ca.M, ca.L, s, ca.env_seed, ctr); }
  __device__ void obs(const ClosedArgs& ca, int m, float* o) const { mpe_world_obs<MT, LT>(w, ca.M, ca.L, m, o); }
};

struct ReferenceClosedWorld {        // simple_reference: 2 agents, actions (move, symbol)
  static constexpr int kM = kRefAgents;
  MpeRefWorld w;
  __device__ static int reset_doubles(const ClosedArgs&) { return kRefResetDoubles; }
  __device__ void load(const ClosedArgs& ca, int e) { ref_world_load(w, ca.apos, ca.avel, ca.lpos, ca.goal, ca.comm, ca.step_count, e); }
  __device__ void store(const ClosedArgs& ca, int e) const { ref_world_store(w, ca.apos, ca.avel, ca.lpos, ca.goal, ca.comm, ca.step_count, e); }
  __device__ double step(const ClosedArgs& ca, const float* act, int as, bool* done) {
    int mv[kRefAgents], sym[kRefAgents];
    for (int q = 0; q < kRefAgents; ++q) { mv[q] = (int)act[q * as]; sym[q] = (int)act[q * as + 1]; }
    return ref_world_step(w, mv, sym, ca.episode_length, done);
  }
  __device__ void reset(const ClosedArgs& ca, const double* s, uint64_t ctr) { ref_world_reset(w, s, ca.env_seed, ctr); }
  __device__ void obs(const ClosedArgs&, int m, float* o) const { ref_world_obs(w, m, o); }
};

// Env step t of world `env` (the insert of mpe_*_step + mappo_env_insert): reads the world's actions of slot t, writes rewards
// of slot t and masks of slot t + 1, resets the world when the episode ended (reset_states of step t, or Philox counter
// ctr0 + t N + env), writes its M new observation rows to o [M][D].  Returns done.
template <class World>
__device__ __forceinline__ bool closed_env_step(World& w, const ClosedArgs& ca, int t, int env, int N, int M, int D, int as,
                                                uint64_t ctr0, float* o) {
  const RolloutArgs& a = ca.r;
  const int E = a.E;
  bool done;
  const double reward = w.step(ca, a.actions + ((size_t)t * E + (size_t)env * M) * as, as, &done);
  if (done)                                                   // env_wrappers.py:146-152
    w.reset(ca, ca.reset_states ? ca.reset_states + ((size_t)t * N + env) * World::reset_doubles(ca) : nullptr,
            ctr0 + (uint64_t)t * N + env);
  for (int q = 0; q < M; ++q) {
    a.rewards[(size_t)t * E + (size_t)env * M + q] = (float)reward;                   // insert: rewards of slot t,
    a.masks[(size_t)(t + 1) * E + (size_t)env * M + q] = done ? 0.f : 1.f;            // masks of slot t + 1
    w.obs(ca, q, o + (size_t)q * D);
  }
  return done;
}

template <class World>
__global__ void __launch_bounds__(64 * kCG * (World::kM ? World::kM : kMpeMaxAgents))
rollout_closed_kernel(const NetDev na, const NetDev nc, const ClosedArgs ca) {
  extern __shared__ __align__(16) float smem[];
  __shared__ uint64_t wbar;
  const RolloutArgs& a = ca.r;
  const int tid = threadIdx.x, lane = tid & 31, wq = tid >> 5;
  const int M = World::kM ? World::kM : ca.M, E = a.E, T = a.T, N = E / M;
  const int rows = kCG * M;                                   // actor warps [0, rows), critic warps [rows, 2 rows)
  const int which = wq >= rows ? 1 : 0;
  const int rl = which ? wq - rows : wq, env_local = rl / M, m = rl - env_local * M;
  const int env = blockIdx.x * kCG + env_local;
  const int g = env < N ? env * M + m : -1;
  const NetDev& n = which == 0 ? na : nc;
  const FastImg fa = make_fast_img(na), fc = make_fast_img(nc);
  const int D = na.in_dim;                                    // the world's observation width
  float* obs_s = smem + fa.total + fc.total + 2 * rows * kFWarpScratch;     // [kCG][M][D]

  // ---- both weight images by TMA, one mbarrier ----
  if (tid == 0) {
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&wbar);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)((fa.total + fc.total) * 4)) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(a.image[0]), "r"((uint32_t)(fa.total * 4)), "r"(bar) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"((uint32_t)__cvta_generic_to_shared(smem + fa.total)), "l"(a.image[1]), "r"((uint32_t)(fc.total * 4)), "r"(bar) : "memory");
  }
  FastCtx c;
  c.f = which == 0 ? fa : fc;
  c.sW = smem + (which == 0 ? 0 : fa.total);
  c.bufA = smem + fa.total + fc.total + wq * kFWarpScratch;
  c.bufB = c.bufA + 64;
  // slot 0 of the storage holds the observations the env produced last (warm-up / previous iteration)
  float* store_in = which == 0 ? a.obs : a.share_obs;
  const int in = n.in_dim;
  float x[2];
  load_row_lane(store_in, g, in, lane, x);
  // the environment thread of a world: lane 0 of its first actor warp
  const bool env_thread = which == 0 && m == 0 && lane == 0 && env < N;
  World w;
  if (env_thread) w.load(ca, env);
  const uint64_t env_ctr0 = (env_thread && !ca.reset_states) ? *ca.env_counter : 0ull;
  __syncthreads();
  {
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&wbar);
    uint32_t ok = 0;
    while (!ok)
      asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                   : "=r"(ok) : "r"(bar), "r"(0u) : "memory");
  }
  const int Atot = na.head_total, as = na.n_heads;
  const uint64_t rng0 = (!a.exp_noise && which == 0) ? *a.rng_offset : 0ull;
  long long t_last = clock64();
#pragma unroll 1
  for (int t = 0; t <= T; ++t) {
    PolStep p;
    p.in = nullptr;
    p.in_copy = t == 0 ? nullptr : store_in + (size_t)t * E * in;
    p.h_in = nullptr; p.h_out = nullptr; p.done_now = nullptr; p.done_prev = nullptr;
    p.masks = a.masks; p.masks_copy = nullptr;
    p.avail = nullptr; p.avail_copy = nullptr;
    p.exp_noise = (a.exp_noise && t < T) ? a.exp_noise + (size_t)t * E * Atot : nullptr;
    p.rng_ctr = rng0 + (uint64_t)t * (uint64_t)E;
    p.values = a.value_preds + (size_t)t * E;
    p.actions = t < T ? a.actions + (size_t)t * E * as : nullptr;
    p.actions_i64 = nullptr;
    p.logp = t < T ? a.logp + (size_t)t * E * as : nullptr;
    p.forward = (t < T) || which == 1;                            // slot T: only the critic's bootstrap value
    fast_step(n, which, c, p, x, g, lane, 0, 0, a.rng_seed, t_last, tid);
    if (t == T) break;
    __syncthreads();                                              // the world's actions of step t are visible
    if (env_thread) closed_env_step(w, ca, t, env, N, M, D, as, env_ctr0, obs_s + (size_t)env_local * M * D);
    __syncthreads();                                              // the next observations are in shared memory
    {
      const float* src = obs_s + (size_t)env_local * M * D + (which == 0 ? m * D : 0);   // critic: the world's M rows
      x[0] = (g >= 0 && lane < in) ? src[lane] : 0.f;
      x[1] = (g >= 0 && lane + 32 < in) ? src[lane + 32] : 0.f;
    }
  }
  if (env_thread) w.store(ca, env);
}

inline size_t closed_smem_bytes(const NetDev& na, const NetDev& nc, int M) {
  return (size_t)(make_fast_img(na).total + make_fast_img(nc).total + 2 * kCG * M * kFWarpScratch + kCG * M * na.in_dim + 4) *
         sizeof(float);
}

// ---- recurrent policies: one 2-CTA cluster per group of `W` worlds ----
constexpr int kCGruRows = 2 * kGW;   // rows per CTA at most (16 warps x 2 rows)

struct ClosedGruPlan { int worlds, rows, warps, clusters; };
// Worlds per cluster: rows per CTA (worlds x M) even -- two rows per warp, a world may straddle two warps -- and at most 32; as
// few as let the clusters cover at most one per SM pair (a step is one long dependent chain per warp, so spreading the rows over
// the SMs beats stacking warps on a scheduler).
inline ClosedGruPlan closed_gru_plan(int N, int M, int sm_count) {
  const int step = (M & 1) ? 2 : 1;
  int wmax = kCGruRows / M;
  wmax -= wmax % step;
  const int pairs = sm_count / 2 > 0 ? sm_count / 2 : 1;
  int w = (N + pairs - 1) / pairs;
  w = (w + step - 1) / step * step;
  if (w > wmax) w = wmax;
  if (w < step) w = step;
  ClosedGruPlan p;
  p.worlds = w;
  p.rows = w * M;
  p.warps = p.rows / 2;
  p.clusters = (N + w - 1) / w;
  return p;
}
// dynamic shared memory, both CTAs alike: the larger image | warp scratch | observation slots [2][rows][D] | done flags [2][W]
__host__ __device__ inline size_t closed_gru_smem_floats_before_slots(const NetDev& na, const NetDev& nc, int warps) {
  const int ta = make_gru_fast_img(na).total, tc = make_gru_fast_img(nc).total;
  return (size_t)(ta > tc ? ta : tc) + (size_t)warps * kGWarpScratch;
}
inline size_t closed_gru_smem_bytes(const NetDev& na, const NetDev& nc, const ClosedGruPlan& p) {
  return (closed_gru_smem_floats_before_slots(na, nc, p.warps) + 2 * (size_t)p.rows * na.in_dim + 2 * (size_t)p.worlds) * sizeof(float);
}

template <class World>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGT)
rollout_closed_gru_kernel(const NetDev na, const NetDev nc, const ClosedArgs ca, const int W) {
  extern __shared__ __align__(16) float smem[];
  __shared__ uint64_t wbar;
  const RolloutArgs& a = ca.r;
  const int tid = threadIdx.x, lane = tid & 31, wq = tid >> 5;
  const int which = (int)cluster_cta_rank();                  // 0: actor + worlds, 1: critic
  const int cluster = blockIdx.x >> 1;
  const int M = World::kM ? World::kM : ca.M, E = a.E, T = a.T, N = E / M;
  const int R = W * M;                                        // rows of this cluster's worlds
  const NetDev& n = which == 0 ? na : nc;
  const int D = na.in_dim, in = n.in_dim;
  float* obs_s = smem + closed_gru_smem_floats_before_slots(na, nc, blockDim.x >> 5);    // [2][R][D]
  float* done_s = obs_s + 2 * R * D;                                                     // [2][W]
  float* store_in = which == 0 ? a.obs : a.share_obs;
  float* h_store = which == 0 ? a.h_actor : a.h_critic;
  int g[2], rl[2];
  float x[2][2], h[2][2], mask[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    rl[r] = 2 * wq + r;
    g[r] = cluster * R + rl[r] < E ? cluster * R + rl[r] : -1;
    load_row_lane(store_in, g[r], in, lane, x[r]);            // slot 0
    h[r][0] = g[r] >= 0 ? h_store[(size_t)g[r] * 64 + lane] : 0.f;
    h[r][1] = g[r] >= 0 ? h_store[(size_t)g[r] * 64 + lane + 32] : 0.f;
    mask[r] = g[r] >= 0 ? a.masks[g[r]] : 0.f;
  }
  // the environment thread of world `tid` of the cluster: lane tid of warp 0 of the actor CTA
  const int env = cluster * W + tid;
  const bool env_thread = which == 0 && tid < W && env < N;
  World w;
  if (env_thread) w.load(ca, env);
  const uint64_t env_ctr0 = (env_thread && !ca.reset_states) ? *ca.env_counter : 0ull;
  const GruFastCtx c = gru_fast_setup(n, smem, a.image[which], &wbar, tid);
  cluster_arrive();                                           // both CTAs run before any DSMEM store
  cluster_wait();
  const int Atot = na.head_total, as = na.n_heads;
  const uint64_t rng0 = (!a.exp_noise && which == 0) ? *a.rng_offset : 0ull;
#pragma unroll 1
  for (int t = 0; t <= T; ++t) {
    if (which == 1 && t < T) cluster_arrive();                // the critic's rows of step t are in registers
    PolStep p;
    p.in = nullptr;
    p.in_copy = t == 0 ? nullptr : store_in + (size_t)t * E * in;
    p.h_in = nullptr; p.h_out = nullptr; p.done_now = nullptr; p.done_prev = nullptr;   // state stored below, after the world step
    p.masks = a.masks; p.masks_copy = nullptr;
    p.avail = nullptr; p.avail_copy = nullptr;
    p.exp_noise = (a.exp_noise && t < T) ? a.exp_noise + (size_t)t * E * Atot : nullptr;
    p.rng_ctr = rng0 + (uint64_t)t * (uint64_t)E;
    p.values = a.value_preds + (size_t)t * E;
    p.actions = t < T ? a.actions + (size_t)t * E * as : nullptr;
    p.actions_i64 = nullptr;
    p.logp = t < T ? a.logp + (size_t)t * E * as : nullptr;
    p.forward = (t < T) || which == 1;                        // slot T: only the critic's bootstrap value
    gru_fast_step(n, which, c, p, x, g, h, mask, lane, 0, 0, a.rng_seed);
    if (t == T) break;
    const int buf = (t + 1) & 1;
    float* ob = obs_s + (size_t)buf * R * D;
    float* dn = done_s + buf * W;
    if (which == 0) {
      __syncthreads();                                        // the actions of step t are visible to the environment threads
      if (env_thread) {
        float* o = ob + (size_t)tid * M * D;
        const bool done = closed_env_step(w, ca, t, env, N, M, D, as, env_ctr0, o);
        for (int i = 0; i < M * D; ++i) st_cluster_f32(o + i, 1u, o[i]);
        dn[tid] = done ? 1.f : 0.f;
        st_cluster_f32(dn + tid, 1u, done ? 1.f : 0.f);
      }
      cluster_arrive();
    }
    cluster_wait();                                           // observations / done flags of env step t are in both CTAs
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int wl = rl[r] / M;
      const float* src = ob + (size_t)wl * M * D + (which == 0 ? (rl[r] - wl * M) * D : 0);   // critic: the world's M rows
      x[r][0] = (g[r] >= 0 && lane < in) ? src[lane] : 0.f;
      x[r][1] = (g[r] >= 0 && lane + 32 < in) ? src[lane + 32] : 0.f;
      const bool d = g[r] >= 0 && dn[wl] != 0.f;
      mask[r] = d ? 0.f : 1.f;
      if (d) { h[r][0] = 0.f; h[r][1] = 0.f; }                // env done: the next episode starts from zeros (mpe_runner.py:128-131)
      if (g[r] >= 0) {
        h_store[((size_t)(t + 1) * E + g[r]) * 64 + lane] = h[r][0];
        h_store[((size_t)(t + 1) * E + g[r]) * 64 + lane + 32] = h[r][1];
      }
    }
  }
  if (env_thread) w.store(ca, env);
}

}  // namespace mappo
