// update_mlp.cu -- fused training step for feed-forward (MLP) actor / critic nets:
//   index-driven gather -> base forward -> heads -> PPO / value loss -> backward -> per-CTA gradient slot.
// One launch per net per optimiser step; activations never leave the SM.
// Replaces: feed_forward_generator's gather (utils/shared_buffer.py:377-396), policy.evaluate_actions
// (algorithms/r_mappo/algorithm/rMAPPOPolicy.py:88-114), the losses of R_MAPPO.ppo_update / cal_value_loss
// (algorithms/r_mappo/r_mappo.py:52-89, 129-146) and autograd's backward (:146, :160).
#include "net_tiles.cuh"

namespace mappo {

template <int TR>
struct UpdSmem {
  // offsets in floats
  int w, xh0, x0, A[kMaxLayers + 1], Y[kMaxLayers + 1], gA, gB, lg, stats, red, rowid, rowf, sred, total;
};

template <int TR>
__host__ __device__ inline UpdSmem<TR> make_upd_smem(const NetDev& n, const SmemW& s) {
  constexpr int LD = Tile<TR>::LD;
  UpdSmem<TR> u;
  int o = 0;
  const int inT = ((n.in_dim + 3) & ~3) * LD, hT = n.hid * LD;
  const int gT = (n.in_dim > n.hid ? ((n.in_dim + 3) & ~3) : n.hid) * LD;
  u.w = o; o += s.total;
  u.xh0 = o; o += n.use_fn ? inT : 0;
  u.x0 = o; o += inT;
  for (int l = 0; l <= kMaxLayers; ++l) {
    const bool on = l <= n.layer_n;
    u.A[l] = o; o += on ? hT : 0;
    u.Y[l] = o; o += on ? hT : 0;
  }
  u.gA = o; o += gT;
  u.gB = o; o += gT;
  u.lg = o; o += ((n.head_total + 3) & ~3) * LD;
  u.stats = o; o += 2 * (kMaxLayers + 2) * TR;
  u.red = o; o += 8 * TR;
  u.rowid = o; o += TR;
  u.rowf = o; o += 8 * TR;          // per-row scalars: adv, active, v_old, ret, (spare)
  o = (o + 1) & ~1;
  u.sred = o; o += 2 * 6 * 32;      // doubles
  u.total = o;
  return u;
}

template <int TR, int NJH, int NJIN>
__global__ void __launch_bounds__(4 * TR, 1)
update_mlp_kernel(const NetDev n, const float* __restrict__ params, const BatchDev b, const LossDev L,
                  const double* __restrict__ norm_stats, const double* __restrict__ adv_stats,
                  const float* __restrict__ vn_state, float* __restrict__ grad_part, double* __restrict__ loss_out,
                  int n_tiles, float* __restrict__ feat_out, const float* __restrict__ dfeat_in, int n_slots_zero) {
  constexpr int LD = Tile<TR>::LD;
  constexpr int NT = Tile<TR>::NT;
  extern __shared__ __align__(16) float smem[];
  const int tid = threadIdx.x;
  const SmemW s = make_smem_w(n, false);
  const UpdSmem<TR> u = make_upd_smem<TR>(n, s);
  float* sW = smem + u.w;
  BaseTiles<TR> t;
  t.xh0 = smem + u.xh0;
  t.x0 = smem + u.x0;
  for (int l = 0; l <= kMaxLayers; ++l) { t.A[l] = smem + u.A[l]; t.Y[l] = smem + u.Y[l]; }
  for (int l = 0; l < kMaxLayers + 2; ++l) { t.mean[l] = smem + u.stats + 2 * l * TR; t.rstd[l] = t.mean[l] + TR; }
  t.red = smem + u.red;
  t.keep_act = true;
  float* gA = smem + u.gA;
  float* gB = smem + u.gB;
  float* lgT = smem + u.lg;
  int* rowid = reinterpret_cast<int*>(smem + u.rowid);
  float* rowf = smem + u.rowf;
  double* sred = reinterpret_cast<double*>(smem + u.sred);

  load_weights(sW, s, n, params, false, tid, NT);
  // Gradient slot of this CTA.  Feed-forward nets: zeroed here, filled below.  Recurrent nets run this kernel
  // twice around the sequence kernels (update_gru.cu): the forward-only pass (feat_out) zeroes ALL slots, the
  // backward pass (dfeat_in) only accumulates.
  float* g = (b.eval_only || feat_out) ? nullptr : grad_part + (size_t)blockIdx.x * n.g.total;
  if (g && !dfeat_in) for (int i = tid; i < n.g.total; i += NT) g[i] = 0.f;
  if (feat_out && grad_part && !b.eval_only)
    for (int sl = blockIdx.x; sl < n_slots_zero; sl += gridDim.x) {
      float* z = grad_part + (size_t)sl * n.g.total;
      for (int i = tid; i < n.g.total; i += NT) z[i] = 0.f;
    }

  const LossConsts lc = make_loss_consts(n, L, norm_stats, adv_stats, vn_state);
  const double n_rows_d = lc.n_rows_d;
  const int H = n.hid;
  const int Atot = n.head_total;
  double acc[3] = {0.0, 0.0, 0.0};      // critic: value_loss | actor: policy_loss, entropy, ratio

  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    __syncthreads();
    if (tid < TR) {
      const int p = tile * TR + tid;
      rowid[tid] = p < b.n_rows ? (b.rows ? b.rows[p] : p) : -1;
    }
    __syncthreads();
    load_rows_T<TR>(n.is_critic ? b.share_obs : b.obs, n.in_dim, rowid, t.x0, tid);
    base_forward<TR, NJH>(n, s, sW, t, tid);
    const float* feat = t.Y[n.layer_n];
    if (feat_out) {                       // recurrent nets, pass 1: features of every position -> workspace
      for (int i = tid; i < TR * H; i += NT) {
        const int r = i / H, c = i - r * H;
        const int p = tile * TR + r;
        if (p < b.n_rows) feat_out[(size_t)p * H + c] = feat[c * LD + r];
      }
      continue;
    }
    if (dfeat_in) {                       // recurrent nets, pass 4: dL/dfeatures from the sequence backward
      for (int i = tid; i < TR * H; i += NT) {
        const int r = i / H, c = i - r * H;
        const int p = tile * TR + r;
        gA[c * LD + r] = p < b.n_rows ? dfeat_in[(size_t)p * H + c] : 0.f;
      }
      __syncthreads();
      base_backward<TR, NJH, NJIN>(n, s, sW, t, gA, gB, g, tid);
      continue;
    }
    tile_mm<TR, 2>(feat, H, sW + s.head_w, s.ldh, 1, Atot, sW + s.head_b, ACT_NONE, lgT, tid);
    __syncthreads();

    // ---- per-row loss and d(loss)/d(logits | value), in place in lgT ----
    if (tid < TR) row_loss<LD>(n, b, L, lc, lgT, tid, rowid[tid], tile * TR + tid, acc);
    __syncthreads();
    if (b.eval_only) continue;

    // ---- head backward ----
    tile_colsum<TR>(lgT, Atot, g + n.g.head_b, tid);
    tile_dw<TR, 2, NJH>(lgT, Atot, feat, H, g + n.g.head_w, H, tid);        // NI=2: Atot <= 32 with NTY=16
    tile_mm<TR, NJH>(lgT, Atot, sW + s.head_w, 1, s.ldh, H, nullptr, ACT_NONE, gA, tid);
    __syncthreads();
    base_backward<TR, NJH, NJIN>(n, s, sW, t, gA, gB, g, tid);
  }

  if (feat_out || dfeat_in) return;
  // loss scalars: [0] value_loss [1] policy_loss [2] dist_entropy [5] ratio
  double v[3];
  if (n.is_critic) { v[0] = acc[0]; v[1] = 0.0; v[2] = 0.0; }
  else { v[0] = acc[0]; v[1] = acc[1]; v[2] = acc[2] / (n_rows_d * (double)b.act_shape); }
  __syncthreads();
  if (n.is_critic) {
    double one[1] = {v[0]};
    block_accumulate<1>(one, loss_out + 0, sred, tid, NT);
  } else {
    double two[2] = {v[0], v[1]};
    block_accumulate<2>(two, loss_out + 1, sred, tid, NT);
    double rt[1] = {v[2]};
    block_accumulate<1>(rt, loss_out + 5, sred, tid, NT);
  }
}

// -------------------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------------------
constexpr int kUpdTR = 64;

static int upd_grid(int n_rows, int sm) {
  const int n_tiles = (n_rows + kUpdTR - 1) / kUpdTR;
  return n_tiles < 2 * sm ? n_tiles : 2 * sm;
}

int update_mlp_slots(const NetDev& n, int n_rows, int sm_count) { return upd_grid(n_rows, sm_count); }

template <int NJIN>
static int launch_upd(const NetDev& n, const float* params, const BatchDev& b, const LossDev& L,
                      const double* norm_stats, const double* adv_stats, const float* vn_state, float* grad_part,
                      int n_slots, double* loss_out, float* feat_out, const float* dfeat_in, cudaStream_t st) {
  const SmemW s = make_smem_w(n, false);
  const UpdSmem<kUpdTR> u = make_upd_smem<kUpdTR>(n, s);
  const size_t bytes = (size_t)u.total * sizeof(float);
  if (bytes > 227 * 1024) {
    set_error("update_mlp: net needs %zu B of shared memory per CTA (> 227 KB): in_dim=%d hidden=%d layer_N=%d",
              bytes, n.in_dim, n.hid, n.layer_n);
    return MAPPO_ERR_UNSUPPORTED;
  }
  auto kern = update_mlp_kernel<kUpdTR, 4, NJIN>;
  static thread_local SmemConfig configured_dev = {};
  size_t& configured = configured_dev.slot();
  if (bytes > configured) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
      return check_launch("update_mlp: cudaFuncSetAttribute");
    configured = bytes;
  }
  const int n_tiles = (b.n_rows + kUpdTR - 1) / kUpdTR;
  kern<<<n_slots, 4 * kUpdTR, bytes, st>>>(n, params, b, L, norm_stats, adv_stats, vn_state, grad_part, loss_out,
                                           n_tiles, feat_out, dfeat_in, n_slots);
  return check_launch("update_mlp_kernel");
}

int update_mlp_launch(const NetDev& n, const float* params, const BatchDev& b, const LossDev& L,
                      const double* norm_stats, const double* adv_stats, const float* vn_state, float* grad_part,
                      int n_slots, double* loss_out, cudaStream_t st, float* feat_out, const float* dfeat_in) {
  if (n.hid != 64) {
    set_error("update_mlp: hidden_size %d not built in the fused SIMT path (64 only)", n.hid);
    return MAPPO_ERR_UNSUPPORTED;
  }
  if (n.head_total > 32) { set_error("update_mlp: sum(head_dim)=%d > 32", n.head_total); return MAPPO_ERR_UNSUPPORTED; }
  if (n.in_dim <= 64)
    return launch_upd<4>(n, params, b, L, norm_stats, adv_stats, vn_state, grad_part, n_slots, loss_out, feat_out, dfeat_in, st);
  // <64, 4, 8> is instantiated for inputs up to 128, but its 64-row tiles fit in 227 KB of shared memory only up to in_dim 96
  // (layer_N 1): from 97 the shared-memory check in launch_upd refuses the net before launching
  if (n.in_dim <= 128)
    return launch_upd<8>(n, params, b, L, norm_stats, adv_stats, vn_state, grad_part, n_slots, loss_out, feat_out, dfeat_in, st);
  set_error("update_mlp: in_dim %d > 128 not built in the fused SIMT path", n.in_dim);
  return MAPPO_ERR_UNSUPPORTED;
}

}  // namespace mappo
