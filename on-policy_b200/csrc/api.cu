// api.cu -- the extern "C" surface of libmappo_b200.so (declared in include/mappo_b200.h).
// No torch types, no allocation, no host synchronisation: every call validates its arguments on the host,
// launches on the caller's stream and returns.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "net_tiles.cuh"
#include "launch_args.h"
#include "big_net.h"

namespace mappo {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static std::atomic<long long> g_launches{0};

// every kernel launch of the library reports here under its kernel name ("x: attribute" strings are not launches)
int check_launch(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return MAPPO_ERR_CUDA;
  }
  if (!strchr(what, ':')) g_launches.fetch_add(1, std::memory_order_relaxed);
  return MAPPO_OK;
}

static int validate_desc(const mappo_net_desc_t* d) {
  if (!d) { set_error("net desc is NULL"); return MAPPO_ERR_INVALID; }
  if (d->in_dim <= 0 || d->hidden <= 0 || d->hidden % 16 != 0) { set_error("bad in_dim/hidden (%d/%d)", d->in_dim, d->hidden); return MAPPO_ERR_INVALID; }
  if (d->layer_n < 0 || d->layer_n > MAPPO_MAX_LAYERS) { set_error("layer_N %d outside [0,%d]", d->layer_n, MAPPO_MAX_LAYERS); return MAPPO_ERR_UNSUPPORTED; }
  if (d->n_heads < 1 || d->n_heads > MAPPO_MAX_HEADS) { set_error("n_heads %d outside [1,%d]", d->n_heads, MAPPO_MAX_HEADS); return MAPPO_ERR_UNSUPPORTED; }
  for (int k = 0; k < d->n_heads; ++k)
    if (d->head_dim[k] <= 0) { set_error("head_dim[%d] = %d", k, d->head_dim[k]); return MAPPO_ERR_INVALID; }
  if (d->is_critic && (d->n_heads != 1 || d->head_dim[0] != 1)) { set_error("critic must have one head of width 1"); return MAPPO_ERR_INVALID; }
  return MAPPO_OK;
}

static void fill_layout(const mappo_net_desc_t* d, mappo_net_layout_t* L) {
  const int H = d->hidden, I = d->in_dim;
  int o = 0, A = 0;
  for (int k = 0; k < d->n_heads; ++k) A += d->head_dim[k];
  auto take = [&](int n) { const int at = o; o += n; return at; };
  L->fn_w = d->use_feature_norm ? take(I) : -1;
  L->fn_b = d->use_feature_norm ? take(I) : -1;
  L->fc1_w = take(H * I); L->fc1_b = take(H); L->ln1_w = take(H); L->ln1_b = take(H);
  for (int l = 0; l < MAPPO_MAX_LAYERS; ++l) {
    const bool on = l < d->layer_n;
    L->fc2_w[l] = on ? take(H * H) : -1; L->fc2_b[l] = on ? take(H) : -1;
    L->ln2_w[l] = on ? take(H) : -1;     L->ln2_b[l] = on ? take(H) : -1;
  }
  const bool r = d->recurrent != 0;
  L->gru_wih = r ? take(3 * H * H) : -1; L->gru_whh = r ? take(3 * H * H) : -1;
  L->gru_bih = r ? take(3 * H) : -1;     L->gru_bhh = r ? take(3 * H) : -1;
  L->rnn_ln_w = r ? take(H) : -1;        L->rnn_ln_b = r ? take(H) : -1;
  L->head_w = take(A * H); L->head_b = take(A);
  L->total = o;
}

NetDev make_net_dev(const mappo_net_desc_t* d) {
  NetDev n;
  memset(&n, 0, sizeof(n));
  n.in_dim = d->in_dim; n.hid = d->hidden; n.layer_n = d->layer_n; n.use_fn = d->use_feature_norm;
  n.use_relu = d->use_relu; n.recurrent = d->recurrent; n.n_heads = d->n_heads; n.is_critic = d->is_critic;
  n.head_total = 0;
  for (int k = 0; k < d->n_heads; ++k) { n.head_dim[k] = d->head_dim[k]; n.head_total += d->head_dim[k]; }
  fill_layout(d, &n.g);
  return n;
}

// launchers implemented in the other translation units
int update_mlp_slots(const NetDev& n, int n_rows, int sm_count);
int update_mlp_launch(const NetDev&, const float*, const BatchDev&, const LossDev&, const double*, const double*,
                      const float*, float*, int, double*, cudaStream_t, float* feat_out = nullptr,
                      const float* dfeat_in = nullptr);
bool update_mlp_tc_supported(const NetDev& n);
int debug_tc_timing(long long* out16);
int debug_pol_timing(long long* out16, int reset);
int update_mlp_tc_slot_floats(const NetDev& n);
int update_mlp_tc_unfold_launch(const NetDev&, const float*, const float*, float*, float*, cudaStream_t);
int64_t update_mlp_tc_workspace_floats(const NetDev& n);
int update_mlp_tc_slots(const NetDev& n, int n_rows, int sm_count);
int update_mlp_tc_launch(const NetDev&, const float*, const BatchDev&, const LossDev&, const double*, const double*,
                         const float*, float*, int, double*, float*, cudaStream_t, bool image_ready);
int update_mlp_tc_tail_launch(const NetDev&, const float*, int, float*, float*, float*, float*, float*, float*, int, const float*, int*,
                              float, float, int, double*, double*, float*, int, cudaStream_t, const void* const*, void* const*, int, int,
                              long long, uint32_t*);
int update_gru_slots(const NetDev& n, int n_rows, int seq_len, int sm_count);
int64_t update_gru_workspace_floats(const NetDev& n, int n_rows);
bool update_gru_tc_supported(const NetDev& n);
int debug_gru_timing(int enable, double* ms_out, long long* n_out);
int debug_gru_cycles(long long* out16);
int64_t update_gru_tc_workspace_floats(const NetDev& n, int n_rows, int sm_count);
int update_gru_tc_launch(const NetDev&, const float*, const BatchDev&, const LossDev&, const double*, const double*, const float*,
                         float* grad_out, double* loss_out, float* workspace, int sm_count, cudaStream_t);
int update_gru_launch(const NetDev&, const float*, const BatchDev&, const LossDev&, const double*, const double*,
                      const float*, float*, int, double*, float*, cudaStream_t);
int gae_launch(const float*, const float*, const float*, const float*, const float*, const float*, int, int, float,
               float, int, int, float*, float*, double*, cudaStream_t);
int advantages_launch(const float*, const float*, const float*, const float*, int, float*, double*, cudaStream_t);
int minibatch_stats_launch(const float*, const float*, const int32_t*, int, double*, cudaStream_t);
int valuenorm_update_launch(float*, const double*, cudaStream_t);
int gather_rows_launch(const float*, const int32_t*, int, int, float*, cudaStream_t);
int chunk_rows_launch(const int32_t*, int, int, int, int, int32_t*, int32_t*, cudaStream_t);
int randperm_launch(int, uint64_t, const uint64_t*, int32_t*, cudaStream_t, int n_perms = 1);
int minibatch_stats_batch_launch(const float*, const float*, const int32_t*, long long, int, int, double*, cudaStream_t);
int grad_reduce_launch(const float*, int, int, float*, float*, int*, cudaStream_t);
int sumsq_launch(const float*, int, float*, int*, cudaStream_t);
int copy_sumsq_launch(const float*, float*, int, float*, int*, cudaStream_t);
int clip_adam_launch(float*, const float*, float*, float*, int, const float*, int, const float*, int*, float, float,
                     int, double*, double*, cudaStream_t);
int counter_add_launch(uint64_t*, uint64_t, cudaStream_t);
int p2p_allreduce_f32_launch(const void* const*, void* const*, int, int, long long, int, float*, uint32_t*, float*, int*,
                             cudaStream_t);
int p2p_allreduce_f64_launch(const void* const*, void* const*, int, int, long long, int, double*, uint32_t*, cudaStream_t);
int pack_rollout_launch(const NetDev&, const float*, float*, cudaStream_t);
int rollout_image_floats(const NetDev&);
namespace big {
int policy_launch(const NetDev& n, float* ws, const float* input, int n_rows, const EpiSample::Args& sample_in, bool tf32, int sm,
                  cudaStream_t st);
bool supported(const NetDev& n);
int debug_timing(int enable, double* ms_out, long long* n_out);
int debug_lin(const float* A, int lda, const float* W, int ldw, float* out, float* stats, const float* colvec, float* scratch,
              int rows, int K, int N, bool tf32, int sm, cudaStream_t st);
int debug_grad(const float* P, int ldp, int Pw, int M, const float* Q, int ldq, int Qw, int rows, float* partial, float* gsum,
               bool tf32, int sm, cudaStream_t st);
int debug_grad_splits(int rows, int M, int Pw, int Qw, int sm);
int debug_plan(const NetDev& n, int rows, int sm, long long* out);
int64_t workspace_floats(const NetDev& n, int rows, int sm);
int pack_launch(const NetDev& n, const float* params, float* ws, int rows, bool round_tf32, int sm, cudaStream_t st);
int update_launch(const NetDev& n, const float* params, const BatchDev& b, const LossDev& L, const double* norm_stats,
                  const double* adv_stats, const float* vn_state, float* grad, double* loss_out, float* ws, bool tf32, int sm,
                  cudaStream_t st, bool inputs_prepared = false);
}  // namespace big

static int g_sm_count = 0;
static int sm_count() {
  if (g_sm_count == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_sm_count, cudaDevAttrMultiProcessorCount, dev);
    if (g_sm_count <= 0) g_sm_count = 148;
  }
  return g_sm_count;
}

}  // namespace mappo

using namespace mappo;


namespace mappo {
bool pdl_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("MAPPO_B200_PDL"); v = (e && e[0] == '1') ? 1 : 0; }
  return v != 0;
}
}  // namespace mappo
extern "C" {
int32_t mappo_abi_version(void) { return MAPPO_ABI_VERSION; }
const char* mappo_last_error(void) { return g_err; }

int32_t mappo_device_check(int32_t* sm, int32_t* major, int32_t* minor) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return check_launch("cudaGetDevice");
  cudaDeviceProp p;
  if (cudaGetDeviceProperties(&p, dev) != cudaSuccess) return check_launch("cudaGetDeviceProperties");
  if (sm) *sm = p.multiProcessorCount;
  if (major) *major = p.major;
  if (minor) *minor = p.minor;
  if (p.major != 10) {
    set_error("libmappo_b200 is built for sm_100a only; device %d is sm_%d%d", dev, p.major, p.minor);
    return MAPPO_ERR_UNSUPPORTED;
  }
  return MAPPO_OK;
}

int32_t mappo_net_layout(const mappo_net_desc_t* desc, mappo_net_layout_t* out) {
  int rc = validate_desc(desc);
  if (rc) return rc;
  if (!out) { set_error("layout out pointer is NULL"); return MAPPO_ERR_INVALID; }
  fill_layout(desc, out);
  return MAPPO_OK;
}

int32_t mappo_policy_step(const mappo_net_desc_t* ad, const float* ap, const mappo_net_desc_t* cd, const float* cp,
                          const float* obs, const float* share_obs, const float* h_a_in, const float* h_c_in,
                          const float* masks, const float* avail, const float* exp_noise, uint64_t rng_seed,
                          const uint64_t* rng_offset_dev, int32_t deterministic, int32_t n_rows, float* values,
                          float* actions, int64_t* actions_i64, float* logp, float* h_a_out, float* h_c_out,
                          const float* actor_image, const float* critic_image, void* stream) {
  return mappo_policy_step_ex(ad, ap, cd, cp, obs, share_obs, h_a_in, h_c_in, masks, avail, exp_noise, rng_seed, rng_offset_dev,
                              deterministic, n_rows, values, actions, actions_i64, logp, h_a_out, h_c_out, actor_image,
                              critic_image, MAPPO_GEMM_FP32, stream);
}

int32_t mappo_policy_step_ex(const mappo_net_desc_t* ad, const float* ap, const mappo_net_desc_t* cd, const float* cp,
                             const float* obs, const float* share_obs, const float* h_a_in, const float* h_c_in,
                             const float* masks, const float* avail, const float* exp_noise, uint64_t rng_seed,
                             const uint64_t* rng_offset_dev, int32_t deterministic, int32_t n_rows, float* values,
                             float* actions, int64_t* actions_i64, float* logp, float* h_a_out, float* h_c_out,
                             const float* actor_image, const float* critic_image, int32_t gemm_mode, void* stream) {
  const bool has_a = ap != nullptr, has_c = cp != nullptr;
  if (!has_a && !has_c) { set_error("policy_step: both nets are NULL"); return MAPPO_ERR_INVALID; }
  if (n_rows <= 0) return MAPPO_OK;
  NetDev na, nc;
  if (has_a) {
    int rc = validate_desc(ad); if (rc) return rc;
    if (ad->is_critic) { set_error("policy_step: actor desc has is_critic set"); return MAPPO_ERR_INVALID; }
    if (!obs) { set_error("policy_step: obs is NULL"); return MAPPO_ERR_INVALID; }
    if (!deterministic && !exp_noise && !rng_offset_dev) { set_error("policy_step: sampling needs exp_noise or rng_offset_dev"); return MAPPO_ERR_INVALID; }
    if (ad->recurrent && (!h_a_in || !masks)) { set_error("policy_step: recurrent actor needs h_actor_in and masks"); return MAPPO_ERR_INVALID; }
    na = make_net_dev(ad);
  }
  if (has_c) {
    int rc = validate_desc(cd); if (rc) return rc;
    if (!cd->is_critic) { set_error("policy_step: critic desc lacks is_critic"); return MAPPO_ERR_INVALID; }
    if (!share_obs) { set_error("policy_step: share_obs is NULL"); return MAPPO_ERR_INVALID; }
    if (cd->recurrent && (!h_c_in || !masks)) { set_error("policy_step: recurrent critic needs h_critic_in and masks"); return MAPPO_ERR_INVALID; }
    nc = make_net_dev(cd);
  }
  if ((has_a && big::supported(na)) || (has_c && big::supported(nc))) {
    // hidden >= 128: layer-by-layer GEMM pipeline; the "image" is the net's workspace with the packed weights in front
    // (mappo_rollout_workspace_floats / mappo_pack_rollout_weights_ex)
    const bool tf32 = gemm_mode == MAPPO_GEMM_TF32;
    if (has_a) {
      if (!actor_image) { set_error("policy_step: hidden >= 128 actor needs its workspace (actor_image)"); return MAPPO_ERR_INVALID; }
      big::EpiSample::Args ea;
      memset(&ea, 0, sizeof(ea));
      ea.avail = avail; ea.exp_noise = exp_noise; ea.rng_seed = rng_seed; ea.rng_offset = exp_noise || deterministic ? nullptr : rng_offset_dev;
      ea.deterministic = deterministic; ea.n_avail = na.head_dim[0];
      ea.actions = actions; ea.actions_i64 = actions_i64; ea.logp = logp;
      int rc = big::policy_launch(na, const_cast<float*>(actor_image), obs, n_rows, ea, tf32, sm_count(), (cudaStream_t)stream);
      if (rc) return rc;
    }
    if (has_c) {
      if (!critic_image) { set_error("policy_step: hidden >= 128 critic needs its workspace (critic_image)"); return MAPPO_ERR_INVALID; }
      big::EpiSample::Args ea;
      memset(&ea, 0, sizeof(ea));
      ea.values = values; ea.deterministic = 1;
      int rc = big::policy_launch(nc, const_cast<float*>(critic_image), share_obs, n_rows, ea, tf32, sm_count(), (cudaStream_t)stream);
      if (rc) return rc;
    }
    return MAPPO_OK;
  }
  PolArgs a;
  memset(&a, 0, sizeof(a));
  a.params[0] = ap; a.params[1] = cp;
  a.image[0] = actor_image; a.image[1] = critic_image;
  a.in[0] = obs; a.in[1] = share_obs;
  a.h_in[0] = h_a_in; a.h_in[1] = h_c_in;
  a.h_out[0] = h_a_out; a.h_out[1] = h_c_out;
  a.masks = masks; a.avail = avail; a.exp_noise = exp_noise;
  a.rng_seed = rng_seed; a.rng_offset = rng_offset_dev;
  a.deterministic = deterministic; a.n_rows = n_rows;
  a.n_avail = has_a ? na.head_dim[0] : 0;
  a.values = values; a.actions = actions; a.actions_i64 = actions_i64; a.logp = logp;
  return policy_step_launch(has_a ? &na : nullptr, has_c ? &nc : nullptr, a, (cudaStream_t)stream);
}

int32_t mappo_rollout_persistent(const mappo_net_desc_t* ad, const float* ap, const float* a_img,
                                 const mappo_net_desc_t* cd, const float* cp, const float* c_img,
                                 float* obs, float* share_obs, float* h_actor, float* h_critic, float* masks, float* avail,
                                 float* value_preds, float* actions, float* logp, float* rewards, float* active_masks,
                                 const float* f_obs, const float* f_share, const float* f_rew, const float* f_done,
                                 const float* f_active, const float* f_avail, const float* exp_noise, uint64_t rng_seed,
                                 uint64_t* rng_offset_dev, int32_t T, int32_t E, void* stream) {
  int rc = validate_desc(ad); if (rc) return rc;
  rc = validate_desc(cd); if (rc) return rc;
  if (ad->is_critic || !cd->is_critic) { set_error("rollout_persistent: actor/critic descriptors swapped"); return MAPPO_ERR_INVALID; }
  if (!ap || !cp || !obs || !share_obs || !masks || !value_preds || !actions || !logp || !rewards || !f_obs ||
      !f_rew || !f_done || T <= 0 || E <= 0) { set_error("rollout_persistent: NULL / bad argument"); return MAPPO_ERR_INVALID; }
  int share_agents = 0;
  if (!f_share) {             // centralized V in the MPE runner's sense: share_obs = all agents' obs of the thread
    if (cd->in_dim % ad->in_dim != 0 || E % (cd->in_dim / ad->in_dim) != 0) { set_error("rollout_persistent: f_share is NULL but share_obs is not a concatenation of obs rows (%d vs %d, E = %d)", cd->in_dim, ad->in_dim, E); return MAPPO_ERR_INVALID; }
    share_agents = cd->in_dim / ad->in_dim;
  }
  if ((ad->recurrent && !h_actor) || (cd->recurrent && !h_critic)) { set_error("rollout_persistent: recurrent net without state storage"); return MAPPO_ERR_INVALID; }
  if (!exp_noise && !rng_offset_dev) { set_error("rollout_persistent: sampling needs exp_noise or rng_offset_dev"); return MAPPO_ERR_INVALID; }
  if ((avail != nullptr) != (f_avail != nullptr)) { set_error("rollout_persistent: avail storage and staged avail must come together"); return MAPPO_ERR_INVALID; }
  if (f_active && !active_masks) { set_error("rollout_persistent: staged active masks without storage"); return MAPPO_ERR_INVALID; }
  RolloutArgs a;
  a.params[0] = ap; a.params[1] = cp; a.image[0] = a_img; a.image[1] = c_img;
  a.obs = obs; a.share_obs = share_obs; a.h_actor = h_actor; a.h_critic = h_critic; a.masks = masks; a.avail = avail;
  a.value_preds = value_preds; a.actions = actions; a.logp = logp; a.rewards = rewards; a.active = active_masks;
  a.f_obs = f_obs; a.f_share = f_share; a.f_rew = f_rew; a.f_done = f_done; a.f_active = f_active; a.f_avail = f_avail;
  a.exp_noise = exp_noise; a.rng_seed = rng_seed; a.rng_offset = rng_offset_dev; a.T = T; a.E = E;
  a.n_avail = ad->head_dim[0];
  a.share_agents = share_agents;
  rc = rollout_persistent_launch(make_net_dev(ad), make_net_dev(cd), a, (cudaStream_t)stream);
  if (rc) return rc;
  if (!exp_noise) return counter_add_launch(rng_offset_dev, (uint64_t)T * (uint64_t)E, (cudaStream_t)stream);
  return MAPPO_OK;
}

int32_t mappo_rollout_closed_loop(const mappo_net_desc_t* ad, const float* a_img, const mappo_net_desc_t* cd, const float* c_img,
                                  float* obs, float* share_obs, float* masks, float* value_preds, float* actions, float* logp,
                                  float* rewards, double* agent_pos, double* agent_vel, double* landmark_pos,
                                  int32_t* step_count, const double* reset_states, uint64_t env_seed,
                                  uint64_t* env_counter_dev, const float* exp_noise, uint64_t rng_seed,
                                  uint64_t* rng_offset_dev, int32_t T, int32_t E, int32_t num_agents, int32_t num_landmarks,
                                  int32_t episode_length, void* stream) {
  return mappo_rollout_closed_loop_ex(ad, a_img, cd, c_img, obs, share_obs, nullptr, nullptr, masks, value_preds, actions, logp,
                                      rewards, MAPPO_WORLD_SPREAD, agent_pos, agent_vel, landmark_pos, nullptr, nullptr, step_count,
                                      reset_states, env_seed, env_counter_dev, exp_noise, rng_seed, rng_offset_dev, T, E,
                                      num_agents, num_landmarks, episode_length, stream);
}

int32_t mappo_rollout_closed_loop_ex(const mappo_net_desc_t* ad, const float* a_img, const mappo_net_desc_t* cd, const float* c_img,
                                     float* obs, float* share_obs, float* h_actor, float* h_critic, float* masks, float* value_preds,
                                     float* actions, float* logp, float* rewards, int32_t world, double* agent_pos,
                                     double* agent_vel, double* landmark_pos, int32_t* goal, int32_t* comm, int32_t* step_count,
                                     const double* reset_states, uint64_t env_seed, uint64_t* env_counter_dev,
                                     const float* exp_noise, uint64_t rng_seed, uint64_t* rng_offset_dev, int32_t T, int32_t E,
                                     int32_t num_agents, int32_t num_landmarks, int32_t episode_length, void* stream) {
  int rc = validate_desc(ad); if (rc) return rc;
  rc = validate_desc(cd); if (rc) return rc;
  if (ad->is_critic || !cd->is_critic) { set_error("rollout_closed_loop: actor/critic descriptors swapped"); return MAPPO_ERR_INVALID; }
  if (!a_img || !c_img || !obs || !share_obs || !masks || !value_preds || !actions || !logp || !rewards || !agent_pos ||
      !agent_vel || !landmark_pos || !step_count || T <= 0 || E <= 0 || episode_length <= 0) { set_error("rollout_closed_loop: NULL / bad argument"); return MAPPO_ERR_INVALID; }
  if (world != MAPPO_WORLD_SPREAD && world != MAPPO_WORLD_REFERENCE) { set_error("rollout_closed_loop: unknown world %d", world); return MAPPO_ERR_INVALID; }
  if (world == MAPPO_WORLD_REFERENCE && (!goal || !comm || num_agents != 2 || num_landmarks != 3)) { set_error("rollout_closed_loop: simple_reference needs goal / comm state, 2 agents and 3 landmarks"); return MAPPO_ERR_INVALID; }
  if ((ad->recurrent && !h_actor) || (cd->recurrent && !h_critic)) { set_error("rollout_closed_loop: recurrent net without state storage"); return MAPPO_ERR_INVALID; }
  if (!exp_noise && !rng_offset_dev) { set_error("rollout_closed_loop: sampling needs exp_noise or rng_offset_dev"); return MAPPO_ERR_INVALID; }
  if (!reset_states && !env_counter_dev) { set_error("rollout_closed_loop: resets need reset_states or env_counter_dev"); return MAPPO_ERR_INVALID; }
  ClosedArgs ca;
  memset(&ca, 0, sizeof(ca));
  RolloutArgs& a = ca.r;
  a.image[0] = a_img; a.image[1] = c_img;
  a.obs = obs; a.share_obs = share_obs; a.masks = masks; a.value_preds = value_preds; a.actions = actions; a.logp = logp;
  a.h_actor = ad->recurrent ? h_actor : nullptr; a.h_critic = cd->recurrent ? h_critic : nullptr;
  a.rewards = rewards; a.exp_noise = exp_noise; a.rng_seed = rng_seed; a.rng_offset = rng_offset_dev; a.T = T; a.E = E;
  ca.world = world;
  ca.apos = agent_pos; ca.avel = agent_vel; ca.lpos = landmark_pos; ca.goal = goal; ca.comm = comm; ca.step_count = step_count;
  ca.reset_states = reset_states; ca.env_seed = env_seed; ca.env_counter = env_counter_dev; ca.M = num_agents; ca.L = num_landmarks;
  ca.episode_length = episode_length;
  rc = rollout_closed_launch(make_net_dev(ad), make_net_dev(cd), ca, (cudaStream_t)stream);
  if (rc) return rc;
  if (!exp_noise) { rc = counter_add_launch(rng_offset_dev, (uint64_t)T * (uint64_t)E, (cudaStream_t)stream); if (rc) return rc; }
  if (!reset_states) return counter_add_launch(env_counter_dev, (uint64_t)T * (uint64_t)(E / num_agents), (cudaStream_t)stream);
  return MAPPO_OK;
}

int32_t mappo_rollout_image_floats(const mappo_net_desc_t* desc) {
  if (validate_desc(desc)) return -1;
  return rollout_image_floats(make_net_dev(desc));
}

int32_t mappo_debug_gru_cycles(int64_t* out16) { return debug_gru_cycles(reinterpret_cast<long long*>(out16)); }

int32_t mappo_debug_gru_timing(int32_t enable, double* ms_out8, int64_t* launches_out8) {
  return debug_gru_timing(enable, ms_out8, reinterpret_cast<long long*>(launches_out8));
}

int32_t mappo_debug_big_timing(int32_t enable, double* ms_out7, int64_t* launches_out7) {
  return big::debug_timing(enable, ms_out7, reinterpret_cast<long long*>(launches_out7));
}

int32_t mappo_debug_big_lin(const float* A, int32_t lda, const float* W, int32_t ldw, float* out, float* stats, const float* colvec,
                            float* scratch, int32_t rows, int32_t K, int32_t N, int32_t gemm_mode, void* stream) {
  if (!A || !W || !out || !stats || !colvec || rows <= 0 || K <= 0 || K % 32 || N <= 0 || N % 32 || N > 1024) { set_error("debug_big_lin: bad arguments"); return MAPPO_ERR_INVALID; }
  return big::debug_lin(A, lda, W, ldw, out, stats, colvec, scratch, rows, K, N, gemm_mode == MAPPO_GEMM_TF32, sm_count(), (cudaStream_t)stream);
}
int32_t mappo_debug_big_grad(const float* P, int32_t ldp, int32_t Pw, int32_t M, const float* Q, int32_t ldq, int32_t Qw, int32_t rows,
                             float* partial, float* gsum, int32_t gemm_mode, void* stream) {
  if (!P || !Q || !partial || !gsum || rows <= 0 || Pw % 32 || Qw % 32 || M <= 0 || M > Pw) { set_error("debug_big_grad: bad arguments"); return MAPPO_ERR_INVALID; }
  return big::debug_grad(P, ldp, Pw, M, Q, ldq, Qw, rows, partial, gsum, gemm_mode == MAPPO_GEMM_TF32, sm_count(), (cudaStream_t)stream);
}
int32_t mappo_debug_big_grad_splits(int32_t rows, int32_t M, int32_t Pw, int32_t Qw) { return big::debug_grad_splits(rows, M, Pw, Qw, sm_count()); }
int32_t mappo_debug_big_plan(const mappo_net_desc_t* desc, int32_t n_rows, int64_t* out64) {
  int rc = validate_desc(desc);
  if (rc) return rc;
  if (!out64) { set_error("debug_big_plan: NULL output"); return MAPPO_ERR_INVALID; }
  const NetDev n = make_net_dev(desc);
  if (!big::supported(n)) { set_error("debug_big_plan: not a hidden >= 128 MLP"); return MAPPO_ERR_UNSUPPORTED; }
  return big::debug_plan(n, n_rows, sm_count(), reinterpret_cast<long long*>(out64));
}

int32_t mappo_big_net(const mappo_net_desc_t* desc) {
  if (validate_desc(desc)) return 0;
  return big::supported(make_net_dev(desc)) ? 1 : 0;
}

int64_t mappo_rollout_workspace_floats(const mappo_net_desc_t* desc, int32_t n_rows) {
  if (validate_desc(desc) || n_rows <= 0) return -1;
  const NetDev n = make_net_dev(desc);
  return big::supported(n) ? big::workspace_floats(n, n_rows, sm_count()) : (int64_t)rollout_image_floats(n);
}

int32_t mappo_pack_rollout_weights(const mappo_net_desc_t* desc, const float* params, float* image, void* stream) {
  return mappo_pack_rollout_weights_ex(desc, params, image, MAPPO_GEMM_FP32, stream);
}

int32_t mappo_pack_rollout_weights_ex(const mappo_net_desc_t* desc, const float* params, float* image, int32_t gemm_mode,
                                      void* stream) {
  int rc = validate_desc(desc);
  if (rc) return rc;
  if (!params || !image || (reinterpret_cast<uintptr_t>(image) & 15)) { set_error("pack_rollout_weights: NULL or unaligned image"); return MAPPO_ERR_INVALID; }
  const NetDev n = make_net_dev(desc);
  if (big::supported(n)) return big::pack_launch(n, params, image, 128, gemm_mode == MAPPO_GEMM_TF32, sm_count(), (cudaStream_t)stream);
  return pack_rollout_launch(n, params, image, (cudaStream_t)stream);
}

int32_t mappo_p2p_allreduce_f32(const void* const* peer_bufs, void* const* peer_signals, int32_t world, int32_t rank,
                                int64_t offset_bytes, int32_t n, float* out, uint32_t* round_dev, float* sumsq_part,
                                int32_t* n_sumsq_blocks_out, void* stream) {
  return p2p_allreduce_f32_launch(peer_bufs, peer_signals, world, rank, offset_bytes, n, out, round_dev, sumsq_part,
                                  n_sumsq_blocks_out, (cudaStream_t)stream);
}
int32_t mappo_p2p_allreduce_f64(const void* const* peer_bufs, void* const* peer_signals, int32_t world, int32_t rank,
                                int64_t offset_bytes, int32_t n, double* out, uint32_t* round_dev, void* stream) {
  return p2p_allreduce_f64_launch(peer_bufs, peer_signals, world, rank, offset_bytes, n, out, round_dev, (cudaStream_t)stream);
}

int32_t mappo_mpe_spread_step(double* agent_pos, double* agent_vel, double* landmark_pos, int32_t* step_count,
                              const float* actions, const double* reset_states, uint64_t rng_seed,
                              uint64_t* rng_counter_dev, int32_t n_envs, int32_t num_agents, int32_t num_landmarks,
                              int32_t episode_length, float* obs_out, float* share_obs_out, float* rewards_out,
                              float* dones_out, void* stream) {
  if (!agent_pos || !agent_vel || !landmark_pos || !step_count || !obs_out || n_envs <= 0 || episode_length <= 0) { set_error("mpe_spread_step: NULL / bad argument"); return MAPPO_ERR_INVALID; }
  if (!reset_states && !rng_counter_dev) { set_error("mpe_spread_step: resets need reset_states or rng_counter_dev"); return MAPPO_ERR_INVALID; }
  if (actions && (!rewards_out || !dones_out)) { set_error("mpe_spread_step: a step needs rewards_out and dones_out"); return MAPPO_ERR_INVALID; }
  MpeArgs a;
  a.apos = agent_pos; a.avel = agent_vel; a.lpos = landmark_pos; a.step_count = step_count; a.actions = actions;
  a.reset_states = reset_states; a.rng_seed = rng_seed; a.rng_counter = rng_counter_dev;
  a.N = n_envs; a.M = num_agents; a.L = num_landmarks; a.episode_length = episode_length;
  a.obs = obs_out; a.share_obs = share_obs_out; a.rewards = rewards_out; a.dones = dones_out;
  const int rc = mpe_spread_launch(a, (cudaStream_t)stream);
  if (rc) return rc;
  if (!reset_states) return counter_add_launch(rng_counter_dev, (uint64_t)n_envs, (cudaStream_t)stream);
  return MAPPO_OK;
}

int32_t mappo_mpe_reference_step(double* agent_pos, double* agent_vel, double* landmark_pos, int32_t* goal, int32_t* comm,
                                 int32_t* step_count, const float* actions, const double* reset_states, uint64_t rng_seed,
                                 uint64_t* rng_counter_dev, int32_t n_envs, int32_t episode_length, float* obs_out,
                                 float* share_obs_out, float* rewards_out, float* dones_out, void* stream) {
  if (!agent_pos || !agent_vel || !landmark_pos || !goal || !comm || !step_count || !obs_out || n_envs <= 0 || episode_length <= 0) { set_error("mpe_reference_step: NULL / bad argument"); return MAPPO_ERR_INVALID; }
  if (!reset_states && !rng_counter_dev) { set_error("mpe_reference_step: resets need reset_states or rng_counter_dev"); return MAPPO_ERR_INVALID; }
  if (actions && (!rewards_out || !dones_out)) { set_error("mpe_reference_step: a step needs rewards_out and dones_out"); return MAPPO_ERR_INVALID; }
  MpeRefArgs a;
  a.apos = agent_pos; a.avel = agent_vel; a.lpos = landmark_pos; a.goal = goal; a.comm = comm; a.step_count = step_count;
  a.actions = actions; a.reset_states = reset_states; a.rng_seed = rng_seed; a.rng_counter = rng_counter_dev;
  a.N = n_envs; a.episode_length = episode_length;
  a.obs = obs_out; a.share_obs = share_obs_out; a.rewards = rewards_out; a.dones = dones_out;
  const int rc = mpe_reference_launch(a, (cudaStream_t)stream);
  if (rc) return rc;
  if (!reset_states) return counter_add_launch(rng_counter_dev, (uint64_t)n_envs, (cudaStream_t)stream);
  return MAPPO_OK;
}

int32_t mappo_counter_add(uint64_t* counter_dev, uint64_t inc, void* stream) {
  if (!counter_dev) { set_error("counter_add: NULL"); return MAPPO_ERR_INVALID; }
  return counter_add_launch(counter_dev, inc, (cudaStream_t)stream);
}

int32_t mappo_env_insert(const float* next_obs, const float* next_share_obs, const float* rewards, const float* dones,
                         const float* next_active, const float* next_avail, int32_t n_rows, int32_t obs_dim,
                         int32_t share_dim, int32_t hidden, int32_t n_act, float* obs_slot, float* share_obs_slot,
                         float* rewards_slot, float* masks_slot, float* h_actor_slot, float* h_critic_slot,
                         float* active_slot, float* avail_slot, uint64_t* rng_counter_dev, uint64_t rng_inc,
                         void* stream) {
  if (n_rows <= 0) return MAPPO_OK;
  if ((next_obs && !obs_slot) || (next_share_obs && !share_obs_slot) || (rewards && !rewards_slot) ||
      (next_avail && !avail_slot)) { set_error("env_insert: source given without destination slot"); return MAPPO_ERR_INVALID; }
  InsertArgs a;
  a.next_obs = next_obs; a.next_share = next_share_obs; a.rewards = rewards; a.dones = dones;
  a.next_active = next_active; a.next_avail = next_avail;
  a.E = n_rows; a.Do = obs_dim; a.Ds = share_dim; a.H = hidden; a.A = n_act;
  a.obs = obs_slot; a.share = share_obs_slot; a.rew = rewards_slot; a.masks = masks_slot;
  a.ha = h_actor_slot; a.hc = h_critic_slot; a.active = active_slot; a.avail = avail_slot;
  a.rng_counter = rng_counter_dev; a.rng_inc = rng_inc;
  return env_insert_launch(a, (cudaStream_t)stream);
}

int32_t mappo_compute_returns(const float* rewards, const float* value_preds, const float* masks,
                              const float* bad_masks, const float* active_masks, const float* vn_state, int32_t T,
                              int32_t E, float gamma, float gae_lambda, int32_t use_gae,
                              int32_t use_proper_time_limits, float* returns, float* advantages, double* adv_stats,
                              void* stream) {
  if (!rewards || !value_preds || !masks || !active_masks || !returns) { set_error("compute_returns: NULL array"); return MAPPO_ERR_INVALID; }
  if (use_proper_time_limits && !bad_masks) { set_error("compute_returns: use_proper_time_limits needs bad_masks"); return MAPPO_ERR_INVALID; }
  if (T <= 0 || E <= 0) { set_error("compute_returns: T=%d E=%d", T, E); return MAPPO_ERR_INVALID; }
  return gae_launch(rewards, value_preds, masks, bad_masks, active_masks, vn_state, T, E, gamma, gae_lambda, use_gae,
                    use_proper_time_limits, returns, advantages, adv_stats, (cudaStream_t)stream);
}

int32_t mappo_advantages(const float* returns, const float* value_preds, const float* active_masks,
                         const float* vn_state, int32_t n, float* advantages, double* adv_stats, void* stream) {
  if (!returns || !value_preds || !active_masks || !advantages || !adv_stats || n <= 0) { set_error("advantages: bad arguments"); return MAPPO_ERR_INVALID; }
  return advantages_launch(returns, value_preds, active_masks, vn_state, n, advantages, adv_stats, (cudaStream_t)stream);
}

int32_t mappo_minibatch_stats(const float* returns, const float* active_masks, const int32_t* rows, int32_t n_rows,
                              double* stats, void* stream) {
  if (!returns || !active_masks || !stats || n_rows <= 0) { set_error("minibatch_stats: bad arguments"); return MAPPO_ERR_INVALID; }
  return minibatch_stats_launch(returns, active_masks, rows, n_rows, stats, (cudaStream_t)stream);
}

int32_t mappo_debug_pol_timing(int64_t* out16, int32_t reset) {
  if (!out16) { set_error("debug_pol_timing: NULL"); return MAPPO_ERR_INVALID; }
  return debug_pol_timing(reinterpret_cast<long long*>(out16), reset);
}

int64_t mappo_debug_launch_count(void) { return (int64_t)g_launches.load(std::memory_order_relaxed); }

int32_t mappo_minibatch_stats_batch(const float* returns, const float* active_masks, const int32_t* rows,
                                    int64_t rows_stride, int32_t n_rows, int32_t n_batches, double* stats, void* stream) {
  if (!returns || !active_masks || !rows || !stats || n_rows <= 0 || n_batches <= 0) { set_error("minibatch_stats_batch: bad arguments"); return MAPPO_ERR_INVALID; }
  return minibatch_stats_batch_launch(returns, active_masks, rows, rows_stride, n_rows, n_batches, stats, (cudaStream_t)stream);
}

int32_t mappo_randperm_batch(int32_t n, int32_t n_perms, uint64_t seed, const uint64_t* counter_dev, int32_t* out, void* stream) {
  if (n < 0 || n_perms < 0 || (n > 0 && n_perms > 0 && !out)) { set_error("randperm_batch: bad arguments"); return MAPPO_ERR_INVALID; }
  return randperm_launch(n, seed, counter_dev, out, (cudaStream_t)stream, n_perms);
}

int32_t mappo_valuenorm_update(float* vn_state, const double* stats, void* stream) {
  if (!vn_state || !stats) { set_error("valuenorm_update: NULL"); return MAPPO_ERR_INVALID; }
  return valuenorm_update_launch(vn_state, stats, (cudaStream_t)stream);
}

int32_t mappo_gather_rows(const float* src, const int32_t* rows, int32_t n_rows, int32_t dim, float* dst, void* stream) {
  if (n_rows < 0 || dim <= 0) { set_error("gather_rows: n_rows=%d dim=%d", n_rows, dim); return MAPPO_ERR_INVALID; }
  if (n_rows == 0) return MAPPO_OK;
  if (!src || !rows || !dst) { set_error("gather_rows: NULL pointer"); return MAPPO_ERR_INVALID; }
  return gather_rows_launch(src, rows, n_rows, dim, dst, (cudaStream_t)stream);
}

int32_t mappo_chunk_rows(const int32_t* chunks, int32_t n_chunks, int32_t L, int32_t T, int32_t E, int32_t* rows,
                         int32_t* first, void* stream) {
  if (n_chunks < 0 || L <= 0 || T <= 0 || E <= 0) { set_error("chunk_rows: bad sizes"); return MAPPO_ERR_INVALID; }
  if (n_chunks == 0) return MAPPO_OK;
  if (!chunks || !rows) { set_error("chunk_rows: NULL pointer"); return MAPPO_ERR_INVALID; }
  return chunk_rows_launch(chunks, n_chunks, L, T, E, rows, first, (cudaStream_t)stream);
}

int32_t mappo_randperm(int32_t n, uint64_t seed, const uint64_t* counter_dev, int32_t* out, void* stream) {
  if (n < 0 || (n > 0 && !out)) { set_error("randperm: bad arguments"); return MAPPO_ERR_INVALID; }
  return randperm_launch(n, seed, counter_dev, out, (cudaStream_t)stream);
}

static int fill_batch(const mappo_net_desc_t* d, const mappo_batch_t* b, BatchDev* o) {
  if (!b) { set_error("batch is NULL"); return MAPPO_ERR_INVALID; }
  if (b->n_rows <= 0) { set_error("batch has %d rows", b->n_rows); return MAPPO_ERR_INVALID; }
  if (b->seq_len < 1 || b->n_seq < 1 || (int64_t)b->seq_len * b->n_seq != b->n_rows) { set_error("batch: seq_len*n_seq != n_rows (%d*%d vs %d)", b->seq_len, b->n_seq, b->n_rows); return MAPPO_ERR_INVALID; }
  if (!b->active_masks) { set_error("batch: active_masks is NULL"); return MAPPO_ERR_INVALID; }
  if (d->is_critic) {
    if (!b->share_obs || !b->value_preds || !b->returns) { set_error("batch: critic needs share_obs, value_preds, returns"); return MAPPO_ERR_INVALID; }
  } else {
    if (!b->obs || !b->actions || !b->old_logp || !b->advantages) { set_error("batch: actor needs obs, actions, old_logp, advantages"); return MAPPO_ERR_INVALID; }
  }
  if (d->recurrent && (!b->masks || !(d->is_critic ? b->h0_critic : b->h0_actor))) { set_error("batch: recurrent net needs masks and h0"); return MAPPO_ERR_INVALID; }
  o->obs = b->obs; o->share_obs = b->share_obs; o->actions = b->actions; o->old_logp = b->old_logp;
  o->value_preds = b->value_preds; o->returns = b->returns; o->advantages = b->advantages; o->masks = b->masks;
  o->active_masks = b->active_masks; o->avail = b->avail; o->h0_actor = b->h0_actor; o->h0_critic = b->h0_critic;
  o->factor = b->factor;
  o->rows = b->rows; o->seq_first = b->seq_first; o->n_rows = b->n_rows; o->seq_len = b->seq_len; o->n_seq = b->n_seq;
  o->act_shape = d->n_heads; o->n_avail = d->head_dim[0];
  o->eval_out = nullptr; o->eval_only = 0;
  return MAPPO_OK;
}

int32_t mappo_debug_tc_timing(int64_t* out16) { return debug_tc_timing(reinterpret_cast<long long*>(out16)); }

int32_t mappo_tf32_supported(const mappo_net_desc_t* desc) {
  if (validate_desc(desc)) return 0;
  const NetDev n = make_net_dev(desc);
  return (update_mlp_tc_supported(n) || update_gru_tc_supported(n) || big::supported(n)) ? 1 : 0;
}

int64_t mappo_update_workspace_floats(const mappo_net_desc_t* desc, int32_t n_rows, int32_t gemm_mode) {
  if (validate_desc(desc)) return -1;
  const NetDev n = make_net_dev(desc);
  if (desc->recurrent)
    return (gemm_mode == MAPPO_GEMM_TF32 && update_gru_tc_supported(n)) ? update_gru_tc_workspace_floats(n, n_rows, sm_count())
                                                                         : update_gru_workspace_floats(n, n_rows);
  if (big::supported(n)) return big::workspace_floats(n, n_rows, sm_count());
  // tf32: [folded weight image][slot-summed raw accumulators]
  return (gemm_mode == MAPPO_GEMM_TF32 && update_mlp_tc_supported(n))
             ? update_mlp_tc_workspace_floats(n) + update_mlp_tc_slot_floats(n) : 0;
}

int32_t mappo_update_slot_floats(const mappo_net_desc_t* desc, int32_t gemm_mode) {
  if (validate_desc(desc)) return -1;
  const NetDev n = make_net_dev(desc);
  if (!desc->recurrent && gemm_mode == MAPPO_GEMM_TF32 && update_mlp_tc_supported(n)) return update_mlp_tc_slot_floats(n);
  return n.g.total;
}

int32_t mappo_update_finish(const mappo_net_desc_t* desc, const float* params, const float* grad_part, int32_t n_slots,
                            int32_t gemm_mode, float* grad, float* sumsq_part, int32_t* n_blocks_out, float* workspace,
                            void* stream) {
  int rc = validate_desc(desc);
  if (rc) return rc;
  if (!params || !grad_part || !grad || !sumsq_part || n_slots <= 0) { set_error("update_finish: bad arguments"); return MAPPO_ERR_INVALID; }
  const NetDev n = make_net_dev(desc);
  if (!desc->recurrent && gemm_mode == MAPPO_GEMM_TF32 && update_mlp_tc_supported(n)) {
    if (!workspace) { set_error("update_finish: tf32 mode needs the workspace"); return MAPPO_ERR_INVALID; }
    float* raw_sum = workspace + update_mlp_tc_workspace_floats(n);
    rc = grad_reduce_launch(grad_part, n_slots, update_mlp_tc_slot_floats(n), raw_sum, nullptr, nullptr, (cudaStream_t)stream);
    if (rc) return rc;
    if (n_blocks_out) *n_blocks_out = 12;
    return update_mlp_tc_unfold_launch(n, params, raw_sum, grad, sumsq_part, (cudaStream_t)stream);
  }
  if (n_slots == 1 && n.g.total >= 65536 && ((reinterpret_cast<uintptr_t>(grad_part) | reinterpret_cast<uintptr_t>(grad)) & 15) == 0)
    return copy_sumsq_launch(grad_part, grad, n.g.total, sumsq_part, n_blocks_out, (cudaStream_t)stream);
  return grad_reduce_launch(grad_part, n_slots, n.g.total, grad, sumsq_part, n_blocks_out, (cudaStream_t)stream);
}

int32_t mappo_update_tail(const mappo_net_desc_t* desc, float* params, const float* grad_part, int32_t n_slots, float* grad,
                          float* exp_avg, float* exp_avg_sq, float* sumsq_part, int32_t n_sumsq_blocks, const float* lr_dev,
                          int32_t* step_dev, float eps, float max_grad_norm, int32_t use_max_grad_norm, double* grad_norm_out,
                          double* beta_pow_dev, float* workspace, int32_t stages, const void* const* peer_bufs,
                          void* const* peer_signals, int32_t world, int32_t rank, int64_t sym_offset_bytes, uint32_t* round_dev,
                          void* stream) {
  int rc = validate_desc(desc);
  if (rc) return rc;
  if (!params || !grad || !sumsq_part || !workspace) { set_error("update_tail: NULL argument"); return MAPPO_ERR_INVALID; }
  const NetDev n = make_net_dev(desc);
  if (desc->recurrent || !update_mlp_tc_supported(n)) { set_error("update_tail: built for the MAPPO_GEMM_TF32 hidden-64 MLP path only"); return MAPPO_ERR_UNSUPPORTED; }
  return update_mlp_tc_tail_launch(n, grad_part, n_slots, workspace + update_mlp_tc_workspace_floats(n), params, grad, exp_avg, exp_avg_sq,
                                   sumsq_part, n_sumsq_blocks, lr_dev, step_dev, eps, max_grad_norm, use_max_grad_norm, grad_norm_out,
                                   beta_pow_dev, workspace, stages, (cudaStream_t)stream, peer_bufs, peer_signals, world, rank,
                                   (long long)sym_offset_bytes, round_dev);
}

int32_t mappo_update_grad_slots(const mappo_net_desc_t* desc, int32_t n_rows, int32_t gemm_mode) {
  if (validate_desc(desc)) return -1;
  const NetDev n = make_net_dev(desc);
  if (desc->recurrent) {
    if (gemm_mode == MAPPO_GEMM_TF32 && update_gru_tc_supported(n)) return 1;      // the tcgen05 GRU pipeline leaves the flat gradient in slot 0
    return update_gru_slots(n, n_rows, 1, sm_count());
  }
  if (big::supported(n)) return 1;                     // the GEMM pipeline leaves the complete flat gradient in slot 0
  if (gemm_mode == MAPPO_GEMM_TF32 && update_mlp_tc_supported(n)) return update_mlp_tc_slots(n, n_rows, sm_count());
  return update_mlp_slots(n, n_rows, sm_count());
}

int32_t mappo_update_fwd_bwd(const mappo_net_desc_t* desc, const float* params, const mappo_batch_t* batch,
                             const mappo_loss_cfg_t* loss, const double* norm_stats, const double* adv_stats,
                             const float* vn_state, float* grad_part, int32_t n_slots, double* loss_out,
                             float* workspace, void* stream) {
  int rc = validate_desc(desc);
  if (rc) return rc;
  if (!params || !loss || !norm_stats || !grad_part || !loss_out || n_slots <= 0) { set_error("update_fwd_bwd: NULL / bad argument"); return MAPPO_ERR_INVALID; }
  BatchDev b;
  rc = fill_batch(desc, batch, &b);
  if (rc) return rc;
  LossDev L;
  L.clip = loss->clip_param; L.ent_coef = loss->entropy_coef; L.vl_coef = loss->value_loss_coef;
  L.huber_delta = loss->huber_delta; L.use_clipped_value_loss = loss->use_clipped_value_loss;
  L.use_huber = loss->use_huber_loss; L.use_value_active = loss->use_value_active_masks;
  L.use_policy_active = loss->use_policy_active_masks; L.use_valuenorm = loss->use_valuenorm;
  L.update_actor = loss->update_actor;
  L.happo = loss->happo;
  if (desc->is_critic && L.use_valuenorm && !vn_state) { set_error("update_fwd_bwd: use_valuenorm needs vn_state"); return MAPPO_ERR_INVALID; }
  const NetDev n = make_net_dev(desc);
  if (desc->recurrent) {
    if (!workspace) { set_error("update_fwd_bwd: recurrent net needs a workspace"); return MAPPO_ERR_INVALID; }
    if (loss->gemm_mode == MAPPO_GEMM_TF32 && !b.eval_only) {
      if (!update_gru_tc_supported(n)) { set_error("update_fwd_bwd: MAPPO_GEMM_TF32 is not built for this recurrent net (hidden 64, layer_N 1, in_dim <= 63)"); return MAPPO_ERR_UNSUPPORTED; }
      return update_gru_tc_launch(n, params, b, L, norm_stats, adv_stats, vn_state, grad_part, loss_out, workspace, sm_count(),
                                  (cudaStream_t)stream);
    }
    return update_gru_launch(n, params, b, L, norm_stats, adv_stats, vn_state, grad_part, n_slots, loss_out, workspace,
                             (cudaStream_t)stream);
  }
  if (b.seq_len != 1) { set_error("update_fwd_bwd: feed-forward net with seq_len %d", b.seq_len); return MAPPO_ERR_INVALID; }
  if (big::supported(n)) {
    if (!workspace) { set_error("update_fwd_bwd: hidden >= 128 net needs its workspace"); return MAPPO_ERR_INVALID; }
    return big::update_launch(n, params, b, L, norm_stats, adv_stats, vn_state, grad_part, loss_out, workspace,
                              loss->gemm_mode == MAPPO_GEMM_TF32, sm_count(), (cudaStream_t)stream, loss->inputs_prepared != 0);
  }
  if (n.hid != 64) { set_error("update_fwd_bwd: hidden_size %d is not built (64, or a multiple of 128 up to 1024)", n.hid); return MAPPO_ERR_UNSUPPORTED; }
  if (loss->gemm_mode == MAPPO_GEMM_TF32) {
    if (!update_mlp_tc_supported(n)) { set_error("update_fwd_bwd: MAPPO_GEMM_TF32 is not built for this net (hidden 64, layer_N 1, in_dim <= 63, MLP only)"); return MAPPO_ERR_UNSUPPORTED; }
    return update_mlp_tc_launch(n, params, b, L, norm_stats, adv_stats, vn_state, grad_part, n_slots, loss_out, workspace,
                                (cudaStream_t)stream, loss->image_ready != 0);
  }
  return update_mlp_launch(n, params, b, L, norm_stats, adv_stats, vn_state, grad_part, n_slots, loss_out,
                           (cudaStream_t)stream);
}

int32_t mappo_evaluate_actions(const mappo_net_desc_t* desc, const float* params, const mappo_batch_t* batch,
                               const mappo_loss_cfg_t* loss, const double* norm_stats, float* out, double* loss_out,
                               float* workspace, void* stream) {
  int rc = validate_desc(desc);
  if (rc) return rc;
  if (!params || !loss || !norm_stats || !out || !loss_out) { set_error("evaluate_actions: NULL argument"); return MAPPO_ERR_INVALID; }
  BatchDev b;
  mappo_batch_t bb = *batch;
  // evaluation needs no targets: let absent loss inputs alias always-present arrays
  if (!desc->is_critic) { if (!bb.old_logp) bb.old_logp = bb.actions; if (!bb.advantages) bb.advantages = bb.active_masks; }
  else { if (!bb.value_preds) bb.value_preds = bb.active_masks; if (!bb.returns) bb.returns = bb.active_masks; }
  rc = fill_batch(desc, &bb, &b);
  if (rc) return rc;
  if (!desc->is_critic && bb.old_logp == bb.actions && desc->n_heads != 1 && false) return MAPPO_ERR_INVALID;
  b.eval_out = out; b.eval_only = 1;
  LossDev L;
  memset(&L, 0, sizeof(L));
  L.clip = loss->clip_param; L.use_policy_active = loss->use_policy_active_masks;
  L.use_value_active = loss->use_value_active_masks; L.huber_delta = loss->huber_delta;
  const NetDev n = make_net_dev(desc);
  if (!desc->recurrent && big::supported(n)) {
    if (!workspace) { set_error("evaluate_actions: hidden >= 128 net needs its workspace"); return MAPPO_ERR_INVALID; }
    return big::update_launch(n, params, b, L, norm_stats, nullptr, nullptr, nullptr, loss_out, workspace,
                              loss->gemm_mode == MAPPO_GEMM_TF32, sm_count(), (cudaStream_t)stream);
  }
  const int slots = mappo_update_grad_slots(desc, b.n_rows, MAPPO_GEMM_FP32);
  if (desc->recurrent) {
    if (!workspace) { set_error("evaluate_actions: recurrent net needs a workspace"); return MAPPO_ERR_INVALID; }
    return update_gru_launch(n, params, b, L, norm_stats, nullptr, nullptr, nullptr, slots, loss_out, workspace, (cudaStream_t)stream);
  }
  return update_mlp_launch(n, params, b, L, norm_stats, nullptr, nullptr, nullptr, slots, loss_out, (cudaStream_t)stream);
}

int32_t mappo_grad_reduce(const float* grad_part, int32_t n_slots, int32_t n_params, float* grad, float* sumsq_part,
                          int32_t* n_blocks_out, void* stream) {
  if (!grad_part || !grad || !sumsq_part || n_slots <= 0 || n_params <= 0) { set_error("grad_reduce: bad arguments"); return MAPPO_ERR_INVALID; }
  return grad_reduce_launch(grad_part, n_slots, n_params, grad, sumsq_part, n_blocks_out, (cudaStream_t)stream);
}

int32_t mappo_grad_sumsq(const float* grad, int32_t n_params, float* sumsq_part, int32_t* n_blocks_out, void* stream) {
  if (!grad || !sumsq_part || n_params <= 0) { set_error("grad_sumsq: bad arguments"); return MAPPO_ERR_INVALID; }
  return sumsq_launch(grad, n_params, sumsq_part, n_blocks_out, (cudaStream_t)stream);
}

int32_t mappo_clip_adam(float* params, const float* grad, float* exp_avg, float* exp_avg_sq, int32_t n_params,
                        const float* sumsq_part, int32_t n_sumsq_blocks, const float* lr_dev, int32_t* step_dev,
                        float eps, float max_grad_norm, int32_t use_max_grad_norm, double* grad_norm_out,
                        double* beta_pow_dev, void* stream) {
  if (!params || !grad || !exp_avg || !exp_avg_sq || !sumsq_part || !lr_dev || !step_dev || n_params <= 0 || n_sumsq_blocks <= 0) { set_error("clip_adam: bad arguments"); return MAPPO_ERR_INVALID; }
  return clip_adam_launch(params, grad, exp_avg, exp_avg_sq, n_params, sumsq_part, n_sumsq_blocks, lr_dev, step_dev, eps,
                          max_grad_norm, use_max_grad_norm, grad_norm_out, beta_pow_dev, (cudaStream_t)stream);
}

}  // extern "C"
