// policy_step.cu -- rollout inference for one env step over E = N*M rows (a8 of SURVEY.md section 8).
// Replaces R_MAPPOPolicy.get_actions / get_values / act (algorithms/r_mappo/algorithm/rMAPPOPolicy.py:48-127):
// actor = feature LN -> MLP -> [GRU step + LN] -> categorical heads -> sample/mode + log-prob,
// critic = the same trunk -> value.  blockIdx.y picks the net, blockIdx.x the 32-row tile; results are
// written straight into the rollout-storage slots handed in by the caller.
#include "net_tiles.cuh"
#include "launch_args.h"
#include "rng.cuh"

namespace mappo {

constexpr int kPolTR = 32;

// ---- packed weight image: the shared-memory weight layout (odd leading dimensions), pre-built in global memory so a
//      CTA fetches it with ONE TMA bulk copy instead of ~70 address-computing cp.async per thread ----
__device__ __forceinline__ int simt_image_offset(const NetDev& n, const SmemW& s, int i) {
  const int H = n.hid, I = n.in_dim;
  auto mat = [&](int base, int rows_cols, int img, int ld, int cols) { const int t = i - base; const int r = t / cols; return img + r * ld + (t - r * cols); };
  (void)mat;
  const mappo_net_layout_t& g = n.g;
  if (n.use_fn) {
    if (i >= g.fn_w && i < g.fn_w + I) return s.fn_w + (i - g.fn_w);
    if (i >= g.fn_b && i < g.fn_b + I) return s.fn_b + (i - g.fn_b);
  }
  if (i >= g.fc1_w && i < g.fc1_w + H * I) { const int t = i - g.fc1_w, r = t / I; return s.fc1_w + r * s.ld1 + (t - r * I); }
  if (i >= g.fc1_b && i < g.fc1_b + H) return s.fc1_b + (i - g.fc1_b);
  if (i >= g.ln1_w && i < g.ln1_w + H) return s.ln1_w + (i - g.ln1_w);
  if (i >= g.ln1_b && i < g.ln1_b + H) return s.ln1_b + (i - g.ln1_b);
  for (int l = 0; l < n.layer_n; ++l) {
    if (i >= g.fc2_w[l] && i < g.fc2_w[l] + H * H) { const int t = i - g.fc2_w[l], r = t / H; return s.fc2_w[l] + r * s.ldh + (t - r * H); }
    if (i >= g.fc2_b[l] && i < g.fc2_b[l] + H) return s.fc2_b[l] + (i - g.fc2_b[l]);
    if (i >= g.ln2_w[l] && i < g.ln2_w[l] + H) return s.ln2_w[l] + (i - g.ln2_w[l]);
    if (i >= g.ln2_b[l] && i < g.ln2_b[l] + H) return s.ln2_b[l] + (i - g.ln2_b[l]);
  }
  if (n.recurrent) {
    if (i >= g.gru_wih && i < g.gru_wih + 3 * H * H) { const int t = i - g.gru_wih, r = t / H; return s.wih + r * s.ldh + (t - r * H); }
    if (i >= g.gru_whh && i < g.gru_whh + 3 * H * H) { const int t = i - g.gru_whh, r = t / H; return s.whh + r * s.ldh + (t - r * H); }
    if (i >= g.gru_bih && i < g.gru_bih + 3 * H) return s.bih + (i - g.gru_bih);
    if (i >= g.gru_bhh && i < g.gru_bhh + 3 * H) return s.bhh + (i - g.gru_bhh);
    if (i >= g.rnn_ln_w && i < g.rnn_ln_w + H) return s.rln_w + (i - g.rnn_ln_w);
    if (i >= g.rnn_ln_b && i < g.rnn_ln_b + H) return s.rln_b + (i - g.rnn_ln_b);
  }
  if (i >= g.head_w && i < g.head_w + n.head_total * H) { const int t = i - g.head_w, r = t / H; return s.head_w + r * s.ldh + (t - r * H); }
  if (i >= g.head_b && i < g.head_b + n.head_total) return s.head_b + (i - g.head_b);
  return -1;
}

__global__ void __launch_bounds__(256) pack_rollout_kernel(const NetDev n, const float* __restrict__ p, float* __restrict__ img) {
  const SmemW s = make_smem_w(n, true);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n.g.total; i += gridDim.x * blockDim.x) {
    const int o = simt_image_offset(n, s, i);
    if (o >= 0) img[o] = p[i];
  }
}

struct PolSmem { int w, x0, xh0, s0, s1, h, gi, gh, stats, red, rowid, total; };

__host__ __device__ inline PolSmem make_pol_smem(const NetDev& n, const SmemW& s) {
  constexpr int LD = Tile<kPolTR>::LD;
  PolSmem u;
  int o = 0;
  const int inT = ((n.in_dim + 3) & ~3) * LD, hT = n.hid * LD;
  u.w = o; o += s.total;
  u.x0 = o; o += inT;
  u.xh0 = o; o += n.use_fn ? inT : 0;
  u.s0 = o; o += hT;
  u.s1 = o; o += hT;
  u.h = o; o += n.recurrent ? hT : 0;
  u.gi = o; o += n.recurrent ? 3 * hT : 0;      // r, z pre-activations (input + hidden parts summed), n input part
  u.gh = o; o += n.recurrent ? hT : 0;          // n hidden part (multiplied by r before the tanh)
  const int lg = ((n.head_total + 3) & ~3) * LD;     // logits share the gi area when recurrent
  if (!n.recurrent) { u.gi = o; o += lg; }
  u.stats = o; o += 2 * (kMaxLayers + 3) * kPolTR;
  u.red = o; o += 8 * kPolTR;
  u.rowid = o; o += kPolTR;
  u.total = o;
  return u;
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// Per-step operands of one net for the rows [row0, row0 + TR) of a step.
struct PolStep {
  const float* in;            // [E, in_dim] input rows of this step
  float* in_copy;             // optional: also store the rows here (persistent rollout: the insert of slot t)
  const float* h_in;          // [E, H] recurrent state of this step, or NULL to use the state carried in shared memory
  const float* masks;         // [E] or NULL (persistent rollout passes mask_from_done)
  const float* done_prev;     // [E] done flags of the previous env step: mask = 1 - done (persistent rollout)
  float* masks_copy;          // optional: store the masks of this step (insert)
  float* h_out;               // [E, H] new state (slot t+1), optional
  const float* done_now;      // [E] done flags of THIS env step: zero the new state of done rows (mpe_runner.py:128-131)
  const float* avail;         // [E, A] or NULL
  float* avail_copy;
  const float* exp_noise;     // [E, sum A] or NULL
  uint64_t rng_ctr;           // Philox counter base of this step (device value + step offset)
  float* values;              // critic out [E]
  float* actions;             // actor outs
  int64_t* actions_i64;
  float* logp;
  bool forward;               // false: only the copies (last slot of the actor in the persistent rollout)
};

struct PolCtx {
  float* sW;
  BaseTiles<kPolTR> t;
  SmemW s;
  PolSmem u;
  int* rowid;
  float* smem;
  float* hcarry;              // [H][LD] recurrent state carried between steps (persistent rollout)
};

// accumulated clock64 deltas of CTA x = 0 (thread 0): [8 * net + phase], phases: 0 row load/copy, 1 base forward,
// 2 recurrent cell, 3 head GEMM, 4 sampling + outputs; read by mappo_debug_pol_timing()
__device__ long long g_pol_timing[16];
#define POL_T(i) do { if (blockIdx.x == 0 && tid == 0) { const long long now_ = clock64(); \
    g_pol_timing[8 * which + (i)] += now_ - t_last; t_last = now_; } } while (0)

template <int NJH>
__device__ __forceinline__ void pol_step(const NetDev& n, int which, const PolCtx& c, const PolStep& p, int n_rows,
                                         int row0, int deterministic, uint64_t rng_seed, int n_avail, int tid) {
  constexpr int TR = kPolTR;
  constexpr int LD = Tile<TR>::LD;
  constexpr int NT = Tile<TR>::NT;
  const int H = n.hid;
  const SmemW& s = c.s;
  const PolSmem& u = c.u;
  float* smem = c.smem;
  float* sW = c.sW;
  const int* rowid = c.rowid;
  long long t_last = clock64();
  // ---- rows of this step: coalesced (a warp walks a row), optional copy into the storage slot ----
  {
    const int warp = tid >> 5, lane = tid & 31, nw = NT >> 5;
    for (int r = warp; r < TR; r += nw) {
      const int g = rowid[r];
      for (int k = lane; k < n.in_dim; k += 32) {
        const float v = g >= 0 ? p.in[(size_t)g * n.in_dim + k] : 0.f;
        c.t.x0[k * LD + r] = v;
        if (p.in_copy && g >= 0) p.in_copy[(size_t)g * n.in_dim + k] = v;
      }
    }
    if (which == 0 && p.avail_copy && p.avail)
      for (int i = tid; i < TR * n_avail; i += NT) {
        const int r = i / n_avail, k = i - r * n_avail, g = rowid[r];
        if (g >= 0) p.avail_copy[(size_t)g * n_avail + k] = p.avail[(size_t)g * n_avail + k];
      }
    if (which == 0 && p.masks_copy && tid < TR && rowid[tid] >= 0)
      p.masks_copy[rowid[tid]] = p.done_prev ? (p.done_prev[rowid[tid]] != 0.f ? 0.f : 1.f) : p.masks[rowid[tid]];
  }
  if (!p.forward) { __syncthreads(); return; }
  POL_T(0);
  base_forward<TR, NJH>(n, s, sW, c.t, tid);
  const float* feat = c.t.Y[n.layer_n];
  POL_T(1);

  if (n.recurrent) {
    // h <- h * mask (rnn.py:27), one GRU step (torch gate order r,z,n; SURVEY App. A.2), LN (rnn.py:79)
    float* hT = smem + u.h;
    float* gi = smem + u.gi;
    float* gh = smem + u.gh;
    for (int i = tid; i < TR * H; i += NT) {
      const int r = i / H, cc = i - r * H;
      const int g = rowid[r];
      float m = 0.f, h = 0.f;
      if (g >= 0) {
        m = p.done_prev ? (p.done_prev[g] != 0.f ? 0.f : 1.f) : p.masks[g];
        h = p.h_in ? p.h_in[(size_t)g * H + cc] : c.hcarry[cc * LD + r];
      }
      hT[cc * LD + r] = h * m;
    }
    __syncthreads();
    // r and z gates: x part and state part in one k loop (same summation order and rounding as two passes), then the n gate's two halves
#pragma unroll 1
    for (int gate = 0; gate < 2; ++gate)
      tile_mm2<TR, NJH>(feat, sW + s.wih + gate * H * s.ldh, sW + s.bih + gate * H, hT, sW + s.whh + gate * H * s.ldh,
                        sW + s.bhh + gate * H, H, s.ldh, gi + gate * H * LD, nullptr, true, tid);
    tile_mm2<TR, NJH>(feat, sW + s.wih + 2 * H * s.ldh, sW + s.bih + 2 * H, hT, sW + s.whh + 2 * H * s.ldh, sW + s.bhh + 2 * H, H, s.ldh,
                      gi + 2 * H * LD, gh, false, tid);
    __syncthreads();
    float* hn = (feat == smem + u.s0) ? smem + u.s1 : smem + u.s0;      // new hidden state (pre-LN): the free tile
    for (int i = tid; i < TR * H; i += NT) {
      const int cc = i / TR, r = i - cc * TR;
      const int o = cc * LD + r;
      const float rg = sigmoidf_(gi[o]);
      const float zg = sigmoidf_(gi[H * LD + o]);
      const float ng = tanhf(gi[2 * H * LD + o] + rg * gh[o]);
      hn[o] = (1.f - zg) * ng + zg * hT[o];
    }
    __syncthreads();
    for (int i = tid; i < TR * H; i += NT) {
      const int r = i / H, cc = i - r * H;
      const int g = rowid[r];
      float v = hn[cc * LD + r];
      if (g >= 0 && p.done_now && p.done_now[g] != 0.f) v = 0.f;       // env done: next episode starts from zeros
      if (g >= 0 && p.h_out) p.h_out[(size_t)g * H + cc] = v;
      if (c.hcarry) c.hcarry[cc * LD + r] = v;
    }
    float* ln_out = (hn == smem + u.s0) ? smem + u.s1 : smem + u.s0;    // old feat tile: gates are done with it
    tile_layernorm<TR>(hn, H, sW + s.rln_w, sW + s.rln_b, ln_out, c.t.mean[kMaxLayers + 1] + 2 * TR,
                       c.t.rstd[kMaxLayers + 1] + 2 * TR, c.t.red, tid);
    feat = ln_out;
  }

  float* lgT = smem + u.gi;
  const int Atot = n.head_total;
  __syncthreads();
  POL_T(2);
  tile_mm<TR, 2>(feat, H, sW + s.head_w, s.ldh, 1, Atot, sW + s.head_b, ACT_NONE, lgT, tid);
  __syncthreads();
  POL_T(3);
  if (tid < TR && rowid[tid] >= 0) {
    const int r = tid, g = rowid[r];
    if (which == 1) {
      if (p.values) p.values[g] = lgT[r];
    } else {
      const float* av = (p.avail && n.n_heads == 1) ? p.avail + (size_t)g * n_avail : nullptr;
      const int as = n.n_heads;
      const uint64_t ctr = p.rng_ctr + (uint64_t)g;
      int off = 0;
      for (int k = 0; k < as; ++k) {
        const int A = n.head_dim[k];
        float lse;
        head_lse<LD>(lgT, off, A, r, av, lse);
        int best = 0;
        float bestv = -INFINITY, best_lp = 0.f;
        uint4 rnd = make_uint4(0, 0, 0, 0);
        for (int j = 0; j < A; ++j) {
          float lgt = lgT[(off + j) * LD + r];
          if (av && av[j] == 0.f) lgt = -1e10f;
          const float lp = lgt - lse;
          const float pr = expf(lp);
          float score = pr;
          if (!deterministic) {
            float q;
            if (p.exp_noise) {
              q = p.exp_noise[(size_t)g * Atot + off + j];
            } else {
              if ((j & 3) == 0)
                rnd = philox4x32_10(make_uint4((uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)(k * 64 + (j >> 2)), 0u),
                                    make_uint2((uint32_t)rng_seed, (uint32_t)(rng_seed >> 32)));
              const uint32_t x = (j & 3) == 0 ? rnd.x : ((j & 3) == 1 ? rnd.y : ((j & 3) == 2 ? rnd.z : rnd.w));
              q = -logf(((float)x + 0.5f) * 2.3283064365386963e-10f);
            }
            score = pr / q;                                  // torch multinomial: argmax(p / Exp(1))
          }
          if (score > bestv) { bestv = score; best = j; best_lp = lp; }
        }
        if (p.actions) p.actions[(size_t)g * as + k] = (float)best;
        if (p.actions_i64) p.actions_i64[(size_t)g * as + k] = (int64_t)best;
        if (p.logp) p.logp[(size_t)g * as + k] = best_lp;
        off += A;
      }
    }
  }
  __syncthreads();
  POL_T(4);
}

}  // namespace mappo
#include "rollout_mlp.cuh"
#include "rollout_gru.cuh"       // warp-per-two-rows kernels of the recurrent policies
#include "rollout_closed.cuh"
namespace mappo {

// shared setup of both kernels: carve shared memory, start the weight fetch, fill rowid; returns the context
template <int NJH>
__device__ __forceinline__ PolCtx pol_setup(const NetDev& n, float* smem, const float* params, const float* image,
                                            int n_rows, uint64_t* wbar, int tid) {
  constexpr int TR = kPolTR;
  constexpr int NT = Tile<TR>::NT;
  PolCtx c;
  c.s = make_smem_w(n, true);
  c.u = make_pol_smem(n, c.s);
  c.smem = smem;
  c.sW = smem + c.u.w;
  c.t.xh0 = smem + c.u.xh0;
  c.t.x0 = smem + c.u.x0;
  // fused layers read Y[l-1] and write Y[l]: ping-pong between the two scratch tiles
  for (int l = 0; l <= kMaxLayers; ++l) { c.t.A[l] = nullptr; c.t.Y[l] = smem + ((l & 1) ? c.u.s0 : c.u.s1); }
  c.t.keep_act = false;
  for (int l = 0; l < kMaxLayers + 2; ++l) { c.t.mean[l] = smem + c.u.stats + 2 * l * TR; c.t.rstd[l] = c.t.mean[l] + TR; }
  c.t.red = smem + c.u.red;
  c.rowid = reinterpret_cast<int*>(smem + c.u.rowid);
  c.hcarry = nullptr;
  if (image) {                                        // one TMA bulk copy of the pre-packed image (UBLKCP)
    if (tid == 0) {
      const uint32_t bar = (uint32_t)__cvta_generic_to_shared(wbar);
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)(c.s.total * 4)) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"((uint32_t)__cvta_generic_to_shared(c.sW)), "l"(image), "r"((uint32_t)(c.s.total * 4)), "r"(bar) : "memory");
    }
  } else {
    load_weights(c.sW, c.s, n, params, true, tid, NT);
  }
  const int row0 = blockIdx.x * TR;
  if (tid < TR) c.rowid[tid] = row0 + tid < n_rows ? row0 + tid : -1;
  __syncthreads();
  if (image) {                                        // every thread waits for the image (init ordered by the barrier)
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(wbar);
    uint32_t ok = 0;
    while (!ok)
      asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                   : "=r"(ok) : "r"(bar), "r"(0u) : "memory");
  }
  return c;
}

template <int NJH>
__global__ void __launch_bounds__(4 * kPolTR)
policy_step_kernel(const NetDev na, const NetDev nc, const PolArgs a, int first_net) {
  extern __shared__ __align__(16) float smem[];
  __shared__ uint64_t wbar;
  const int tid = threadIdx.x;
  const int which = first_net + blockIdx.y;           // 0 actor, 1 critic
  const NetDev& n = which == 0 ? na : nc;
  const PolCtx c = pol_setup<NJH>(n, smem, a.params[which], a.image[which], a.n_rows, &wbar, tid);
  PolStep p;
  p.in = a.in[which]; p.in_copy = nullptr; p.h_in = a.h_in[which]; p.masks = a.masks; p.done_prev = nullptr;
  p.masks_copy = nullptr; p.h_out = a.h_out[which]; p.done_now = nullptr; p.avail = a.avail; p.avail_copy = nullptr;
  p.exp_noise = a.exp_noise;
  p.rng_ctr = (!a.exp_noise && !a.deterministic && which == 0) ? *a.rng_offset : 0ull;
  p.values = a.values; p.actions = a.actions; p.actions_i64 = a.actions_i64; p.logp = a.logp; p.forward = true;
  pol_step<NJH>(n, which, c, p, a.n_rows, blockIdx.x * kPolTR, a.deterministic, a.rng_seed, a.n_avail, tid);
}

// ---------------------------------------------------------------------------------------------------------------
// Persistent rollout: the T collect steps + inserts of one iteration as ONE launch.  Rows never interact (an MLP / GRU
// policy is row-wise, compute_returns works per lane), and in the device-resident pipeline the env outputs of the whole
// iteration are already staged in HBM -- so a CTA keeps its 32 rows AND the weights in shared memory and walks
// t = 0..T: read the step's rows (slot 0 of the storage for t = 0, the staged env output afterwards), store them into
// slot t (= SharedReplayBuffer.insert), forward, sample, write values / actions / log-probs / states; the critic CTA
// finishes with the bootstrap value of slot T (= Runner.compute's get_values).
// Replaces T x (mappo_policy_step + mappo_env_insert) + the get_values launch: 2T + 1 launches -> 1.
// ---------------------------------------------------------------------------------------------------------------
template <int NJH>
__global__ void __launch_bounds__(4 * kPolTR)
rollout_persistent_kernel(const NetDev na, const NetDev nc, const RolloutArgs a) {
  constexpr int TR = kPolTR;
  constexpr int LD = Tile<TR>::LD;
  constexpr int NT = Tile<TR>::NT;
  extern __shared__ __align__(16) float smem[];
  __shared__ uint64_t wbar;
  const int tid = threadIdx.x;
  const int which = blockIdx.y;
  const NetDev& n = which == 0 ? na : nc;
  PolCtx c = pol_setup<NJH>(n, smem, a.params[which], a.image[which], a.E, &wbar, tid);
  const int H = n.hid, E = a.E, T = a.T;
  const int Atot = na.head_total;
  if (n.recurrent) {                                    // carried state lives behind the regular tiles
    c.hcarry = smem + c.u.total;
    const float* h0 = which == 0 ? a.h_actor : a.h_critic;
    for (int i = tid; i < TR * H; i += NT) {
      const int r = i / H, cc = i - r * H, g = c.rowid[r];
      c.hcarry[cc * LD + r] = g >= 0 ? h0[(size_t)g * H + cc] : 0.f;
    }
  }
  const uint64_t rng0 = (!a.exp_noise && which == 0) ? *a.rng_offset : 0ull;
  const int in_dim = n.in_dim;
  float* store_in = which == 0 ? a.obs : a.share_obs;
  const float* feed_in = which == 0 ? a.f_obs : a.f_share;
  float* h_store = which == 0 ? a.h_actor : a.h_critic;
  __syncthreads();
#pragma unroll 1
  for (int t = 0; t <= T; ++t) {
    PolStep p;
    p.in = t == 0 ? store_in : feed_in + (size_t)(t - 1) * E * in_dim;
    p.in_copy = t == 0 ? nullptr : store_in + (size_t)t * E * in_dim;
    p.h_in = nullptr;                                   // carried in shared memory
    p.masks = a.masks;                                  // t == 0: slot 0
    p.done_prev = t == 0 ? nullptr : a.f_done + (size_t)(t - 1) * E;
    p.masks_copy = t == 0 ? nullptr : a.masks + (size_t)t * E;
    p.h_out = (n.recurrent && t < T) ? h_store + (size_t)(t + 1) * E * H : nullptr;
    p.done_now = t < T ? a.f_done + (size_t)t * E : nullptr;
    p.avail = a.avail ? (t == 0 ? a.avail : a.f_avail + (size_t)(t - 1) * E * a.n_avail) : nullptr;
    p.avail_copy = (a.avail && t > 0) ? a.avail + (size_t)t * E * a.n_avail : nullptr;
    p.exp_noise = (a.exp_noise && t < T) ? a.exp_noise + (size_t)t * E * Atot : nullptr;
    p.rng_ctr = rng0 + (uint64_t)t * (uint64_t)E;
    p.values = a.value_preds + (size_t)t * E;
    p.actions = t < T ? a.actions + (size_t)t * E * na.n_heads : nullptr;
    p.actions_i64 = nullptr;
    p.logp = t < T ? a.logp + (size_t)t * E * na.n_heads : nullptr;
    p.forward = (t < T) || which == 1;                  // slot T: only the critic's bootstrap value
    // rewards / active masks of env step t-1 -> slot t-1 / t (the rest of insert), done by the actor CTAs
    if (which == 0 && t > 0 && tid < TR && c.rowid[tid] >= 0) {
      const int g = c.rowid[tid];
      a.rewards[(size_t)(t - 1) * E + g] = a.f_rew[(size_t)(t - 1) * E + g];
      if (a.f_active) a.active[(size_t)t * E + g] = a.f_active[(size_t)(t - 1) * E + g];
    }
    pol_step<NJH>(n, which, c, p, E, blockIdx.x * TR, 0, a.rng_seed, a.n_avail, tid);
  }
}

int debug_pol_timing(long long* out16, int reset) {
  if (cudaMemcpyFromSymbol(out16, g_pol_timing, sizeof(long long) * 16) != cudaSuccess) return MAPPO_ERR_CUDA;
  if (reset) {
    long long z[16] = {0};
    if (cudaMemcpyToSymbol(g_pol_timing, z, sizeof(z)) != cudaSuccess) return MAPPO_ERR_CUDA;
  }
  return MAPPO_OK;
}

__global__ void counter_add_kernel(uint64_t* c, uint64_t inc) { *c += inc; }

static int device_sm_count() {
  static thread_local int sm[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  int& v = sm[dev & 63];
  if (v == 0) { cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev); if (v <= 0) v = 148; }
  return v;
}

// A net that qualifies for a warp-per-row kernel has its image packed in that kernel's layout (pack_rollout_launch), and
// that image can be smaller than the tile layout.  When the OTHER net sends both onto the 32-row tile kernels, such a net
// loads its weights from the flat parameters instead.
static inline const float* tile_image(const NetDev& n, const float* image) {
  return (fast_rollout_supported(n) || gru_fast_supported(n)) ? nullptr : image;
}

int policy_step_launch(const NetDev* na, const NetDev* nc, const PolArgs& a, cudaStream_t st) {
  const NetDev& ref = na ? *na : *nc;
  {   // feed-forward nets with a packed image: the warp-per-two-rows path (rollout_mlp.cuh)
    bool fast = true;
    size_t fb = 0;
    for (int w = 0; w < 2; ++w) {
      const NetDev* n = w == 0 ? na : nc;
      if (!n) continue;
      if (!fast_rollout_supported(*n) || !a.image[w]) fast = false;
      else { const size_t b = fast_smem_bytes(*n); fb = b > fb ? b : fb; }
    }
    if (fast) {
      static thread_local SmemConfig configured_f_dev = {};
  size_t& configured_f = configured_f_dev.slot();
      if (fb > configured_f) {
        if (cudaFuncSetAttribute(policy_step_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fb) != cudaSuccess)
          return check_launch("policy_step_fast: cudaFuncSetAttribute");
        configured_f = fb;
      }
      const dim3 grid((a.n_rows + kFR - 1) / kFR, (na && nc) ? 2 : 1);
      policy_step_fast_kernel<<<grid, kFT, fb, st>>>(na ? *na : ref, nc ? *nc : ref, a, na ? 0 : 1);
      return check_launch("policy_step_fast_kernel");
    }
  }
  {   // recurrent nets with a packed image: two rows per warp, state in registers (rollout_gru.cuh)
    bool fast = true;
    size_t fb = 0;
    for (int w = 0; w < 2; ++w) {
      const NetDev* n = w == 0 ? na : nc;
      if (!n) continue;
      if (!gru_fast_supported(*n) || !a.image[w] || !a.h_in[w]) fast = false;
    }
    const int n_nets = (na && nc) ? 2 : 1;
    const int warps = gru_fast_warps(a.n_rows, n_nets, device_sm_count());
    for (int w = 0; w < 2 && fast; ++w) {
      const NetDev* n = w == 0 ? na : nc;
      if (n) { const size_t b = gru_fast_smem_bytes(*n, warps); fb = b > fb ? b : fb; }
    }
    if (fast && fb <= 227 * 1024) {
      static thread_local SmemConfig configured_g_dev = {};
      size_t& configured_g = configured_g_dev.slot();
      if (fb > configured_g) {
        if (cudaFuncSetAttribute(policy_step_gru_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fb) != cudaSuccess)
          return check_launch("policy_step_gru_fast: cudaFuncSetAttribute");
        configured_g = fb;
      }
      const dim3 grid((a.n_rows + 2 * warps - 1) / (2 * warps), n_nets);
      policy_step_gru_fast_kernel<<<grid, 32 * warps, fb, st>>>(na ? *na : ref, nc ? *nc : ref, a, na ? 0 : 1);
      return check_launch("policy_step_gru_fast_kernel");
    }
  }
  size_t bytes = 0;
  for (const NetDev* n : {na, nc}) {
    if (!n) continue;
    if (n->hid != 64) { set_error("policy_step: hidden_size %d not built in the fused SIMT path (64 only)", n->hid); return MAPPO_ERR_UNSUPPORTED; }
    if (n->head_total > 32) { set_error("policy_step: sum(head_dim) > 32"); return MAPPO_ERR_UNSUPPORTED; }
    const SmemW s = make_smem_w(*n, true);
    const size_t b = (size_t)make_pol_smem(*n, s).total * sizeof(float);
    bytes = b > bytes ? b : bytes;
  }
  if (bytes > 227 * 1024) { set_error("policy_step: %zu B shared memory per CTA > 227 KB (in_dim too large)", bytes); return MAPPO_ERR_UNSUPPORTED; }
  PolArgs ta = a;
  for (int w = 0; w < 2; ++w) {
    const NetDev* n = w == 0 ? na : nc;
    if (n) ta.image[w] = tile_image(*n, ta.image[w]);
  }
  auto kern = policy_step_kernel<4>;
  static thread_local SmemConfig configured_dev = {};
  size_t& configured = configured_dev.slot();
  if (bytes > configured) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
      return check_launch("policy_step: cudaFuncSetAttribute");
    configured = bytes;
  }
  const dim3 grid((a.n_rows + kPolTR - 1) / kPolTR, (na && nc) ? 2 : 1);
  kern<<<grid, 4 * kPolTR, bytes, st>>>(na ? *na : ref, nc ? *nc : ref, ta, na ? 0 : 1);
  return check_launch("policy_step_kernel");
}

int rollout_persistent_launch(const NetDev& na, const NetDev& nc, const RolloutArgs& a, cudaStream_t st) {
  if (fast_rollout_supported(na) && fast_rollout_supported(nc) && a.image[0] && a.image[1]) {
    const size_t ba = fast_smem_bytes(na), bc = fast_smem_bytes(nc), fb = ba > bc ? ba : bc;
    static thread_local SmemConfig configured_f_dev = {};
  size_t& configured_f = configured_f_dev.slot();
    if (fb > configured_f) {
      if (cudaFuncSetAttribute(rollout_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fb) != cudaSuccess)
        return check_launch("rollout_fast: cudaFuncSetAttribute");
      configured_f = fb;
    }
    rollout_fast_kernel<<<dim3((a.E + kFR - 1) / kFR, 2), kFT, fb, st>>>(na, nc, a);
    return check_launch("rollout_fast_kernel");
  }
  if (gru_fast_supported(na) && gru_fast_supported(nc) && a.image[0] && a.image[1]) {
    const int warps = gru_fast_warps(a.E, 2, device_sm_count());
    const size_t ba = gru_fast_smem_bytes(na, warps), bc = gru_fast_smem_bytes(nc, warps), fb = ba > bc ? ba : bc;
    if (fb <= 227 * 1024) {
      static thread_local SmemConfig configured_g_dev = {};
      size_t& configured_g = configured_g_dev.slot();
      if (fb > configured_g) {
        if (cudaFuncSetAttribute(rollout_gru_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fb) != cudaSuccess)
          return check_launch("rollout_gru_fast: cudaFuncSetAttribute");
        configured_g = fb;
      }
      rollout_gru_fast_kernel<<<dim3((a.E + 2 * warps - 1) / (2 * warps), 2), 32 * warps, fb, st>>>(na, nc, a);
      return check_launch("rollout_gru_fast_kernel");
    }
  }
  if (a.share_agents > 0) { set_error("rollout: share_obs derived from obs is only built for the feed-forward and the two-rows-per-warp recurrent path"); return MAPPO_ERR_UNSUPPORTED; }
  size_t bytes = 0;
  for (const NetDev* n : {&na, &nc}) {
    if (n->hid != 64) { set_error("rollout: hidden_size %d not built in the fused SIMT path (64 only)", n->hid); return MAPPO_ERR_UNSUPPORTED; }
    if (n->head_total > 32) { set_error("rollout: sum(head_dim) > 32"); return MAPPO_ERR_UNSUPPORTED; }
    const SmemW s = make_smem_w(*n, true);
    size_t b = (size_t)make_pol_smem(*n, s).total * sizeof(float);
    if (n->recurrent) b += (size_t)n->hid * Tile<kPolTR>::LD * sizeof(float);
    bytes = b > bytes ? b : bytes;
  }
  if (bytes > 227 * 1024) { set_error("rollout: %zu B shared memory per CTA > 227 KB", bytes); return MAPPO_ERR_UNSUPPORTED; }
  RolloutArgs ta = a;
  ta.image[0] = tile_image(na, a.image[0]);
  ta.image[1] = tile_image(nc, a.image[1]);
  auto kern = rollout_persistent_kernel<4>;
  static thread_local SmemConfig configured_dev = {};
  size_t& configured = configured_dev.slot();
  if (bytes > configured) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
      return check_launch("rollout: cudaFuncSetAttribute");
    configured = bytes;
  }
  const dim3 grid((a.E + kPolTR - 1) / kPolTR, 2);
  kern<<<grid, 4 * kPolTR, bytes, st>>>(na, nc, ta);
  return check_launch("rollout_persistent_kernel");
}

// raise the kernel's dynamic shared-memory limit once per device
template <class K>
static int closed_set_smem(K kern, size_t bytes, SmemConfig& conf) {
  size_t& c = conf.slot();
  if (bytes > c) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
      return check_launch("rollout_closed: cudaFuncSetAttribute");
    c = bytes;
  }
  return MAPPO_OK;
}

template <class World>
static int closed_mlp_launch(const NetDev& na, const NetDev& nc, const ClosedArgs& ca, int M, size_t bytes, cudaStream_t st) {
  static thread_local SmemConfig conf = {};
  if (int rc = closed_set_smem(rollout_closed_kernel<World>, bytes, conf)) return rc;
  const int N = ca.r.E / M;
  rollout_closed_kernel<World><<<(N + kCG - 1) / kCG, 64 * kCG * M, bytes, st>>>(na, nc, ca);
  return check_launch("rollout_closed_kernel");
}

template <class World>
static int closed_gru_launch(const NetDev& na, const NetDev& nc, const ClosedArgs& ca, const ClosedGruPlan& p, size_t bytes,
                             cudaStream_t st) {
  static thread_local SmemConfig conf = {};
  if (int rc = closed_set_smem(rollout_closed_gru_kernel<World>, bytes, conf)) return rc;
  rollout_closed_gru_kernel<World><<<2 * p.clusters, 32 * p.warps, bytes, st>>>(na, nc, ca, p.worlds);
  return check_launch("rollout_closed_gru_kernel");
}

int rollout_closed_launch(const NetDev& na, const NetDev& nc, const ClosedArgs& ca, cudaStream_t st) {
  const bool ref = ca.world == MAPPO_WORLD_REFERENCE;
  const int M = ref ? kRefAgents : ca.M, L = ref ? kRefLandmarks : ca.L;
  const bool images = ca.r.image[0] && ca.r.image[1];
  const bool mlp = fast_rollout_supported(na) && fast_rollout_supported(nc);
  const bool gru = gru_fast_supported(na) && gru_fast_supported(nc) && ca.r.h_actor && ca.r.h_critic;
  if (!images || !(mlp || gru)) { set_error("rollout_closed: needs two feed-forward or two recurrent nets on the warp-per-row path (hidden 64, in_dim <= 64, <= 32 head outputs; recurrent: with state storage) and packed weight images"); return MAPPO_ERR_UNSUPPORTED; }
  if (M < 1 || M > kMpeMaxAgents || L < 1 || L > kMpeMaxLandmarks || ca.r.E % M != 0) { set_error("rollout_closed: %d agents / %d landmarks / %d rows", M, L, ca.r.E); return MAPPO_ERR_UNSUPPORTED; }
  if (ref) {
    if (na.n_heads != 2 || na.head_dim[0] != 5 || na.head_dim[1] != kRefSymbols || na.in_dim != kRefObs || nc.in_dim != M * kRefObs) { set_error("rollout_closed: policy shapes do not match simple_reference (MultiDiscrete(5, 10), obs %d, share_obs %d)", kRefObs, M * kRefObs); return MAPPO_ERR_INVALID; }
  } else {
    const int D = 4 + 2 * L + 4 * (M - 1);
    if (na.n_heads != 1 || na.head_dim[0] != 5 || na.in_dim != D || nc.in_dim != M * D) { set_error("rollout_closed: policy shapes do not match simple_spread (Discrete(5), obs %d, share_obs %d)", D, M * D); return MAPPO_ERR_INVALID; }
  }
  const bool spread33 = !ref && M == 3 && L == 3;             // the reference's default shape: compile-time counts
  if (mlp) {
    const size_t bytes = closed_smem_bytes(na, nc, M);
    if (bytes > 227 * 1024) { set_error("rollout_closed: %zu B shared memory", bytes); return MAPPO_ERR_UNSUPPORTED; }
    if (ref) return closed_mlp_launch<ReferenceClosedWorld>(na, nc, ca, M, bytes, st);
    if (spread33) return closed_mlp_launch<SpreadClosedWorld<3, 3>>(na, nc, ca, M, bytes, st);
    return closed_mlp_launch<SpreadClosedWorld<0, 0>>(na, nc, ca, M, bytes, st);
  }
  const ClosedGruPlan p = closed_gru_plan(ca.r.E / M, M, device_sm_count());
  const size_t bytes = closed_gru_smem_bytes(na, nc, p);
  if (bytes > 227 * 1024) { set_error("rollout_closed: %zu B shared memory per CTA of the recurrent closed loop > 227 KB", bytes); return MAPPO_ERR_UNSUPPORTED; }
  if (ref) return closed_gru_launch<ReferenceClosedWorld>(na, nc, ca, p, bytes, st);
  if (spread33) return closed_gru_launch<SpreadClosedWorld<3, 3>>(na, nc, ca, p, bytes, st);
  return closed_gru_launch<SpreadClosedWorld<0, 0>>(na, nc, ca, p, bytes, st);
}

int pack_rollout_launch(const NetDev& n, const float* params, float* image, cudaStream_t st) {
  if (fast_rollout_supported(n)) {        // feed-forward nets: the [k][tx][4] image of rollout_mlp.cuh
    pack_fast_kernel<<<(make_fast_img(n).total + 255) / 256, 256, 0, st>>>(n, params, image);
    return check_launch("pack_fast_kernel");
  }
  if (gru_fast_supported(n)) {            // recurrent nets: the feed-forward image + the gate matrices as [gate][k][lane][2]
    pack_gru_fast_kernel<<<(make_gru_fast_img(n).total + 255) / 256, 256, 0, st>>>(n, params, image);
    return check_launch("pack_gru_fast_kernel");
  }
  pack_rollout_kernel<<<(n.g.total + 255) / 256, 256, 0, st>>>(n, params, image);
  return check_launch("pack_rollout_kernel");
}
int rollout_image_floats(const NetDev& n) {
  if (gru_fast_supported(n)) return make_gru_fast_img(n).total;
  return fast_rollout_supported(n) ? make_fast_img(n).total : make_smem_w(n, true).total;
}

int counter_add_launch(uint64_t* c, uint64_t inc, cudaStream_t st) {
  counter_add_kernel<<<1, 1, 0, st>>>(c, inc);
  return check_launch("counter_add_kernel");
}

}  // namespace mappo
