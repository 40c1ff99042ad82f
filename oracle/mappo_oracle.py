"""CPU oracle for the MAPPO hot path  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference`
legs may import this module; the product path (`on-policy_b200/`) never does and fails loudly
when its CUDA library is missing.

This is an independent restatement (NumPy for the buffer / scan / gather arithmetic, torch-CPU
autograd + torch.optim.Adam for the network arithmetic -- PyTorch is the third-party library in
which the reference's own arithmetic lives, SURVEY.md section 8c) of the reference path

    collect xT -> compute_returns (GAE) -> minibatch generator -> ppo_update x(ppo_epoch*num_mini_batch)
    -> after_update

Every function cites the reference file:line (relative to /root/reference/onpolicy/) it follows.
Parity pin: the reference holds no tests or golden vectors for this path (SURVEY.md section 4), so the
oracle is pinned against outputs of the reference itself, generated in the build container by
`tests/golden/make_golden.py` / `make_golden_separated.py` (committed together with the fixtures they wrote;
`tests/test_oracle_golden.py` checks the oracle against every one of them).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field, asdict
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F


# --------------------------------------------------------------------------------------------
# configuration
# --------------------------------------------------------------------------------------------
@dataclass
class PathConfig:
    """Effective hyper-parameters of one run (defaults = config.py:156-307)."""
    episode_length: int = 25           # T
    n_rollout_threads: int = 8         # N
    num_agents: int = 3                # M
    obs_dim: int = 18                  # Do
    share_obs_dim: int = 54            # Ds
    act_dims: Sequence[int] = (5,)     # [A] Discrete, [A0, A1, ...] MultiDiscrete
    multi_discrete: bool = False
    hidden_size: int = 64
    layer_N: int = 1
    recurrent_N: int = 1
    use_ReLU: bool = True
    use_feature_normalization: bool = True
    use_recurrent_policy: bool = False
    use_naive_recurrent_policy: bool = False
    data_chunk_length: int = 10
    gamma: float = 0.99
    gae_lambda: float = 0.95
    use_gae: bool = True
    use_valuenorm: bool = True
    use_proper_time_limits: bool = False
    clip_param: float = 0.2
    ppo_epoch: int = 15
    num_mini_batch: int = 1
    value_loss_coef: float = 1.0
    entropy_coef: float = 0.01
    max_grad_norm: float = 10.0
    huber_delta: float = 10.0
    use_max_grad_norm: bool = True
    use_clipped_value_loss: bool = True
    use_huber_loss: bool = True
    use_value_active_masks: bool = True
    use_policy_active_masks: bool = True
    lr: float = 5e-4
    critic_lr: float = 5e-4
    opti_eps: float = 1e-5
    gain: float = 0.01

    @property
    def act_shape(self) -> int:            # utils/util.py:41-51
        return len(self.act_dims) if self.multi_discrete else 1

    @property
    def has_avail(self) -> bool:           # shared_buffer.py:69-73: only Discrete spaces get the array
        return not self.multi_discrete

    @property
    def recurrent(self) -> bool:
        return self.use_recurrent_policy or self.use_naive_recurrent_policy

    def to_dict(self):
        d = asdict(self)
        d["act_dims"] = list(self.act_dims)
        return d


# --------------------------------------------------------------------------------------------
# ValueNorm  (utils/valuenorm.py:8-79)
# --------------------------------------------------------------------------------------------
class ValueNormState:
    """Debiased running first/second moment of the returns, fp32 like the reference."""
    BETA = np.float32(0.99999)
    EPS = np.float32(1e-5)

    def __init__(self):
        self.running_mean = np.float32(0.0)
        self.running_mean_sq = np.float32(0.0)
        self.debiasing_term = np.float32(0.0)

    def mean_var(self):                                     # valuenorm.py:32-36
        d = max(self.debiasing_term, self.EPS)
        mean = np.float32(self.running_mean / d)
        mean_sq = np.float32(self.running_mean_sq / d)
        var = np.float32(max(np.float32(mean_sq - np.float32(mean * mean)), np.float32(1e-2)))
        return mean, var

    def update(self, x):                                    # valuenorm.py:38-55
        xt = torch.as_tensor(np.asarray(x, dtype=np.float32)).reshape(-1)
        bm = np.float32(xt.mean().item())
        bsq = np.float32((xt ** 2).mean().item())
        w = self.BETA
        one_m = np.float32(1.0 - 0.99999)      # the reference forms (1.0 - weight) in double, then casts
        self.running_mean = np.float32(self.running_mean * w + bm * one_m)
        self.running_mean_sq = np.float32(self.running_mean_sq * w + bsq * one_m)
        self.debiasing_term = np.float32(self.debiasing_term * w + np.float32(1.0) * one_m)

    def normalize(self, x):                                 # valuenorm.py:57-66
        mean, var = self.mean_var()
        return (np.asarray(x, dtype=np.float32) - mean) / np.float32(np.sqrt(var))

    def denormalize(self, x):                               # valuenorm.py:68-79
        mean, var = self.mean_var()
        return np.asarray(x, dtype=np.float32) * np.float32(np.sqrt(var)) + mean

    def state(self):
        return np.array([self.running_mean, self.running_mean_sq, self.debiasing_term], dtype=np.float32)

    def load(self, s):
        self.running_mean, self.running_mean_sq, self.debiasing_term = (np.float32(v) for v in s)


# --------------------------------------------------------------------------------------------
# rollout storage  (utils/shared_buffer.py:31-177; separated_buffer.py is the M==1 special case
# of the same memory layout: [T+1, N, D] == [T+1, N, 1, D])
# --------------------------------------------------------------------------------------------
class RolloutStore:
    def __init__(self, cfg: PathConfig):
        T, N, M, H = cfg.episode_length, cfg.n_rollout_threads, cfg.num_agents, cfg.hidden_size
        f = lambda *s: np.zeros(s, dtype=np.float32)
        self.cfg = cfg
        self.share_obs = f(T + 1, N, M, cfg.share_obs_dim)           # :54-56
        self.obs = f(T + 1, N, M, cfg.obs_dim)
        self.rnn_states = f(T + 1, N, M, cfg.recurrent_N, H)          # :58-61
        self.rnn_states_critic = f(T + 1, N, M, cfg.recurrent_N, H)
        self.value_preds = f(T + 1, N, M, 1)                          # :63-67
        self.returns = f(T + 1, N, M, 1)
        self.available_actions = (np.ones((T + 1, N, M, cfg.act_dims[0]), np.float32)
                                  if cfg.has_avail else None)         # :69-73
        self.actions = f(T, N, M, cfg.act_shape)                      # :77-82
        self.action_log_probs = f(T, N, M, cfg.act_shape)
        self.rewards = f(T, N, M, 1)
        self.masks = np.ones((T + 1, N, M, 1), np.float32)            # :84-86
        self.bad_masks = np.ones_like(self.masks)
        self.active_masks = np.ones_like(self.masks)
        self.step = 0

    def insert(self, share_obs, obs, rnn_a, rnn_c, actions, logp, values, rewards, masks,
               bad_masks=None, active_masks=None, available_actions=None):   # :90-123
        s = self.step
        self.share_obs[s + 1] = share_obs
        self.obs[s + 1] = obs
        self.rnn_states[s + 1] = rnn_a
        self.rnn_states_critic[s + 1] = rnn_c
        self.actions[s] = actions
        self.action_log_probs[s] = logp
        self.value_preds[s] = values
        self.rewards[s] = rewards
        self.masks[s + 1] = masks
        if bad_masks is not None:
            self.bad_masks[s + 1] = bad_masks
        if active_masks is not None:
            self.active_masks[s + 1] = active_masks
        if available_actions is not None:
            self.available_actions[s + 1] = available_actions
        self.step = (s + 1) % self.cfg.episode_length

    def after_update(self):                                           # :160-170
        for name in ("share_obs", "obs", "rnn_states", "rnn_states_critic", "masks", "bad_masks",
                     "active_masks", "available_actions"):
            a = getattr(self, name)
            if a is not None:
                a[0] = a[-1].copy()


# --------------------------------------------------------------------------------------------
# compute_returns  (shared_buffer.py:179-262, non-MAT branches)
# --------------------------------------------------------------------------------------------
def compute_returns(store: RolloutStore, next_value, vn: Optional[ValueNormState]):
    """T sequential vector steps, each of them like the reference does it (per-step denormalise)."""
    cfg = store.cfg
    T = cfg.episode_length
    g, lam = np.float32(cfg.gamma), np.float32(cfg.gae_lambda)
    den = (lambda v: vn.denormalize(v)) if (cfg.use_valuenorm and vn is not None) else (lambda v: v)
    r, v, m, bad, ret = store.rewards, store.value_preds, store.masks, store.bad_masks, store.returns
    if cfg.use_gae:
        v[-1] = next_value                                           # :186 / :218
        gae = 0
        for t in reversed(range(T)):
            v_t, v_n = den(v[t]), den(v[t + 1])
            delta = r[t] + g * v_n * m[t + 1] - v_t                   # :190-192 / :236-238
            gae = delta + g * lam * m[t + 1] * gae                    # :193 / :239
            if cfg.use_proper_time_limits:
                gae = gae * bad[t + 1]                                # :194
            ret[t] = gae + v_t                                        # :195 / :240
    else:
        ret[-1] = next_value                                         # :204 / :260
        for t in reversed(range(T)):
            if cfg.use_proper_time_limits:                            # :206-215
                ret[t] = (ret[t + 1] * g * m[t + 1] + r[t]) * bad[t + 1] + (1 - bad[t + 1]) * den(v[t])
            else:                                                     # :261-262
                ret[t] = ret[t + 1] * g * m[t + 1] + r[t]


def normalized_advantages(store: RolloutStore, vn: Optional[ValueNormState]):
    """r_mappo.py:179-187: raw advantage, stats over active entries only, normalise all entries."""
    cfg = store.cfg
    v = store.value_preds[:-1]
    adv = store.returns[:-1] - (vn.denormalize(v) if (cfg.use_valuenorm and vn is not None) else v)
    c = adv.copy()
    c[store.active_masks[:-1] == 0.0] = np.nan
    return ((adv - np.nanmean(c)) / (np.nanstd(c) + 1e-5)).astype(np.float32)


# --------------------------------------------------------------------------------------------
# minibatch index arithmetic  (the integer part of the generators: bit-exact contract)
# --------------------------------------------------------------------------------------------
def ff_minibatch_rows(perm: np.ndarray, B: int, num_mini_batch: int) -> List[np.ndarray]:
    """shared_buffer.py:358-361. Row id = (t*N + n)*M + m of the [:-1] flattened arrays."""
    mb = B // num_mini_batch
    return [np.asarray(perm[i * mb:(i + 1) * mb], dtype=np.int64) for i in range(num_mini_batch)]


def chunk_minibatch_rows(perm: np.ndarray, T: int, N: int, M: int, L: int, num_mini_batch: int):
    """shared_buffer.py:505-512, 557-604.  Rows are re-ordered (n, m, t) (`_cast`, :11-12), cut every L
    rows regardless of T (chunks may straddle trajectories, SURVEY App. B-3), chunks permuted, and
    the minibatch is laid out time-major [L, Nc].  Returns per minibatch
      rows  int64 [L*Nc]  natural (t*N+n)*M+m row id feeding position l*Nc + c
      first int64 [Nc]    natural row id whose stored rnn state starts chunk c
    """
    B = T * N * M
    data_chunks = B // L
    mb = data_chunks // num_mini_batch
    out = []
    for i in range(num_mini_batch):
        chunks = np.asarray(perm[i * mb:(i + 1) * mb], dtype=np.int64)
        j = chunks[None, :] * L + np.arange(L, dtype=np.int64)[:, None]     # (n,m,t)-ordered position
        t = j % T
        nm = j // T                                                          # = n*M + m
        rows = t * (N * M) + nm
        out.append((rows.reshape(-1), rows[0].copy()))
    return out


def naive_minibatch_rows(perm: np.ndarray, T: int, N: int, M: int, num_mini_batch: int):
    """shared_buffer.py:409-447: whole trajectories, [T, Nc] time-major, initial state = slot 0."""
    E = N * M
    per = E // num_mini_batch
    out = []
    for start in range(0, E, per):
        lanes = np.asarray(perm[start:start + per], dtype=np.int64)
        if len(lanes) < per:
            break
        rows = np.arange(T, dtype=np.int64)[:, None] * E + lanes[None, :]
        out.append((rows.reshape(-1), lanes.copy()))
    return out


_GEN_FIELDS = ("share_obs", "obs", "rnn_states", "rnn_states_critic", "actions", "value_preds", "returns",
               "masks", "active_masks", "action_log_probs", "advantages", "available_actions")


def _flat_tables(store: RolloutStore, advantages):
    c = store.cfg
    B = c.episode_length * c.n_rollout_threads * c.num_agents
    tab = {
        "share_obs": store.share_obs[:-1].reshape(B, -1),
        "obs": store.obs[:-1].reshape(B, -1),
        "rnn_states": store.rnn_states[:-1].reshape(B, c.recurrent_N, c.hidden_size),
        "rnn_states_critic": store.rnn_states_critic[:-1].reshape(B, c.recurrent_N, c.hidden_size),
        "actions": store.actions.reshape(B, -1),
        "value_preds": store.value_preds[:-1].reshape(B, 1),
        "returns": store.returns[:-1].reshape(B, 1),
        "masks": store.masks[:-1].reshape(B, 1),
        "active_masks": store.active_masks[:-1].reshape(B, 1),
        "action_log_probs": store.action_log_probs.reshape(B, -1),
        "advantages": advantages.reshape(B, 1),
        "available_actions": (store.available_actions[:-1].reshape(B, -1)
                              if store.available_actions is not None else None),
    }
    return tab, B


def minibatches(store: RolloutStore, advantages, perm: np.ndarray, factor=None):
    """Yield the reference's 12-tuples (order of shared_buffer.py:397-400 / :602-604) for one epoch (13-tuples with the
    gathered `factor` rows when given, separated_buffer.py:197-227).
    `perm` is the permutation the reference would have drawn with torch.randperm at :360 / :415 / :511."""
    c = store.cfg
    tab, B = _flat_tables(store, advantages)
    T, N, M = c.episode_length, c.n_rollout_threads, c.num_agents
    if c.use_recurrent_policy:
        plan = chunk_minibatch_rows(perm, T, N, M, c.data_chunk_length, c.num_mini_batch)
    elif c.use_naive_recurrent_policy:
        plan = naive_minibatch_rows(perm, T, N, M, c.num_mini_batch)
    else:
        plan = [(r, r) for r in ff_minibatch_rows(perm, B, c.num_mini_batch)]
    for rows, first in plan:
        sample = []
        for name in _GEN_FIELDS:
            a = tab[name]
            if a is None:
                sample.append(None)
            elif name in ("rnn_states", "rnn_states_critic"):
                sample.append(a[first])
            else:
                sample.append(a[rows])
        if factor is not None:
            sample.append(np.asarray(factor).reshape(B, -1)[rows])
        yield tuple(sample)


# --------------------------------------------------------------------------------------------
# networks  (algorithms/utils/{mlp,rnn,act,distributions}.py, r_actor_critic.py) as pure functions of
# a {state_dict key: tensor} mapping, so reference weights drop in unchanged (SURVEY App. A.8)
# --------------------------------------------------------------------------------------------
def init_params(cfg: PathConfig, critic: bool, seed: Optional[int] = None) -> Dict[str, torch.Tensor]:
    """Orthogonal weights / zero biases with the reference's gains (mlp.py:12-16, rnn.py:14-21,
    distributions.py:58-62, r_actor_critic.py:146-152)."""
    g = torch.Generator().manual_seed(seed) if seed is not None else None
    H, Din = cfg.hidden_size, (cfg.share_obs_dim if critic else cfg.obs_dim)
    act_gain = math.sqrt(2.0) if cfg.use_ReLU else 5.0 / 3.0
    p: Dict[str, torch.Tensor] = {}

    def ortho(rows, cols, gain):
        w = torch.empty(rows, cols)
        if g is None:
            torch.nn.init.orthogonal_(w, gain=gain)
        else:
            torch.nn.init.orthogonal_(w, gain=gain, generator=g)
        return w

    if cfg.use_feature_normalization:
        p["base.feature_norm.weight"], p["base.feature_norm.bias"] = torch.ones(Din), torch.zeros(Din)
    p["base.mlp.fc1.0.weight"], p["base.mlp.fc1.0.bias"] = ortho(H, Din, act_gain), torch.zeros(H)
    p["base.mlp.fc1.2.weight"], p["base.mlp.fc1.2.bias"] = torch.ones(H), torch.zeros(H)
    for i in range(cfg.layer_N):
        p[f"base.mlp.fc2.{i}.0.weight"], p[f"base.mlp.fc2.{i}.0.bias"] = ortho(H, H, act_gain), torch.zeros(H)
        p[f"base.mlp.fc2.{i}.2.weight"], p[f"base.mlp.fc2.{i}.2.bias"] = torch.ones(H), torch.zeros(H)
    if cfg.recurrent:
        for l in range(cfg.recurrent_N):
            p[f"rnn.rnn.weight_ih_l{l}"] = ortho(3 * H, H, 1.0)
            p[f"rnn.rnn.weight_hh_l{l}"] = ortho(3 * H, H, 1.0)
            p[f"rnn.rnn.bias_ih_l{l}"] = torch.zeros(3 * H)
            p[f"rnn.rnn.bias_hh_l{l}"] = torch.zeros(3 * H)
        p["rnn.norm.weight"], p["rnn.norm.bias"] = torch.ones(H), torch.zeros(H)
    if critic:
        p["v_out.weight"], p["v_out.bias"] = ortho(1, H, 1.0), torch.zeros(1)
    elif cfg.multi_discrete:
        for k, A in enumerate(cfg.act_dims):
            p[f"act.action_outs.{k}.linear.weight"] = ortho(A, H, cfg.gain)
            p[f"act.action_outs.{k}.linear.bias"] = torch.zeros(A)
    else:
        p["act.action_out.linear.weight"] = ortho(cfg.act_dims[0], H, cfg.gain)
        p["act.action_out.linear.bias"] = torch.zeros(cfg.act_dims[0])
    return p


def _mlp_base(cfg: PathConfig, p, x):
    """mlp.py:52-57 (feature LN) then mlp.py:26-30 (Linear -> act -> LN stack)."""
    act = F.relu if cfg.use_ReLU else torch.tanh
    H = cfg.hidden_size
    if cfg.use_feature_normalization:
        x = F.layer_norm(x, (x.shape[-1],), p["base.feature_norm.weight"], p["base.feature_norm.bias"])
    x = F.layer_norm(act(F.linear(x, p["base.mlp.fc1.0.weight"], p["base.mlp.fc1.0.bias"])), (H,),
                     p["base.mlp.fc1.2.weight"], p["base.mlp.fc1.2.bias"])
    for i in range(cfg.layer_N):
        x = F.layer_norm(act(F.linear(x, p[f"base.mlp.fc2.{i}.0.weight"], p[f"base.mlp.fc2.{i}.0.bias"])),
                         (H,), p[f"base.mlp.fc2.{i}.2.weight"], p[f"base.mlp.fc2.{i}.2.bias"])
    return x


def _gru_cell(p, l, x, h):
    """torch GRU equations (SURVEY App. A.2), gate order (r, z, n)."""
    gi = F.linear(x, p[f"rnn.rnn.weight_ih_l{l}"], p[f"rnn.rnn.bias_ih_l{l}"])
    gh = F.linear(h, p[f"rnn.rnn.weight_hh_l{l}"], p[f"rnn.rnn.bias_hh_l{l}"])
    i_r, i_z, i_n = gi.chunk(3, -1)
    h_r, h_z, h_n = gh.chunk(3, -1)
    r = torch.sigmoid(i_r + h_r)
    z = torch.sigmoid(i_z + h_z)
    n = torch.tanh(i_n + r * h_n)
    return (1.0 - z) * n + z * h


def _rnn_layer(cfg: PathConfig, p, x, hxs, masks):
    """rnn.py:24-80.  Equivalent per-step form of the segment loop: before every step the carried
    state is multiplied by that step's mask (rnn.py:27 single step; :62-69 training segments --
    inside a segment all masks are 1, at a segment start the state is multiplied by masks[start])."""
    H, R = cfg.hidden_size, cfg.recurrent_N
    Nb = hxs.shape[0]
    L = x.shape[0] // Nb
    xs = x.view(L, Nb, H)
    ms = masks.view(L, Nb, 1)
    h = [hxs[:, l] for l in range(R)]
    outs = []
    for t in range(L):
        inp = xs[t]
        for l in range(R):
            h[l] = _gru_cell(p, l, inp, h[l] * ms[t])
            inp = h[l]
        outs.append(inp)
    y = torch.stack(outs, 0).reshape(L * Nb, H)
    y = F.layer_norm(y, (H,), p["rnn.norm.weight"], p["rnn.norm.bias"])           # rnn.py:79
    return y, torch.stack(h, 1)


def _features(cfg, p, x, hxs, masks):
    f = _mlp_base(cfg, p, x)
    if cfg.recurrent:
        f, hxs = _rnn_layer(cfg, p, f, hxs, masks)
    return f, hxs


def _head_logits(cfg: PathConfig, p, feat, avail):
    """distributions.py:64-68 (masked fill with -1e10 before normalisation)."""
    if cfg.multi_discrete:
        return [F.linear(feat, p[f"act.action_outs.{k}.linear.weight"], p[f"act.action_outs.{k}.linear.bias"])
                for k in range(len(cfg.act_dims))]
    lg = F.linear(feat, p["act.action_out.linear.weight"], p["act.action_out.linear.bias"])
    if avail is not None:
        lg = torch.where(avail == 0, torch.full_like(lg, -1e10), lg)
    return [lg]


def critic_forward(cfg, p, share_obs, hxs, masks):
    """r_actor_critic.py:156-175."""
    f, hxs = _features(cfg, p, share_obs, hxs, masks)
    return F.linear(f, p["v_out.weight"], p["v_out.bias"]), hxs


def actor_act(cfg, p, obs, hxs, masks, avail=None, deterministic=False, exp_noise=None):
    """r_actor_critic.py:44-71 + act.py:44-91.  Sampling: Categorical.sample == argmax(p / Exp(1))
    (torch multinomial, probe in SURVEY 8c); `exp_noise` [rows, sum(act_dims)] injects the Exp(1)
    draws so a device implementation can be compared bit-exactly; None draws them from the global
    CPU generator exactly like the reference would (one exponential_ per head, in head order)."""
    f, hxs = _features(cfg, p, obs, hxs, masks)
    acts, lps, off = [], [], 0
    for k, lg in enumerate(_head_logits(cfg, p, f, avail)):
        logp = lg - lg.logsumexp(-1, keepdim=True)
        probs = logp.exp()
        if deterministic:
            a = probs.argmax(-1, keepdim=True)                                    # distributions.py:27-28
        else:
            A = lg.shape[-1]
            q = (torch.empty_like(probs).exponential_(1) if exp_noise is None else exp_noise[:, off:off + A])
            a = (probs / q).argmax(-1, keepdim=True)
            off += A
        acts.append(a)
        lps.append(logp.gather(-1, a))
    return torch.cat(acts, -1), torch.cat(lps, -1), hxs


def actor_evaluate(cfg, p, obs, hxs, actions, masks, avail=None, active=None):
    """r_actor_critic.py:73-117 + act.py:115-178 (Discrete :170-176, MultiDiscrete :147-160)."""
    f, _ = _features(cfg, p, obs, hxs, masks)
    lps, ents = [], []
    use_active = active is not None and cfg.use_policy_active_masks
    for k, lg in enumerate(_head_logits(cfg, p, f, avail)):
        logp = lg - lg.logsumexp(-1, keepdim=True)
        probs = logp.exp()
        a = actions[:, k:k + 1].long()
        lps.append(logp.gather(-1, a))
        ent = -(probs * logp.clamp(min=torch.finfo(logp.dtype).min)).sum(-1)      # torch Categorical.entropy
        ents.append((ent * active.squeeze(-1)).sum() / active.sum() if use_active else ent.mean())
    return torch.cat(lps, -1), sum(ents) / len(ents)


# --------------------------------------------------------------------------------------------
# trainer  (algorithms/r_mappo/r_mappo.py)
# --------------------------------------------------------------------------------------------
def _huber(e, d):                                                                 # utils/util.py:23-26
    a = (e.abs() <= d).to(e.dtype)
    return a * e ** 2 / 2 + (1 - a) * d * (e.abs() - d / 2)


class Learner:
    """Actor + critic parameter sets, two Adam optimisers (rMAPPOPolicy.py:31-37), ValueNorm,
    and the reference update rule (r_mappo.py:52-224)."""

    def __init__(self, cfg: PathConfig, actor: Dict[str, torch.Tensor], critic: Dict[str, torch.Tensor], happo: bool = False,
                 dtype: torch.dtype = torch.float32):
        """`dtype`: parameters and inputs are cast to it (float64 gives a high-precision reference of the same update)."""
        self.cfg = cfg
        self.dtype = dtype
        self.happo = happo            # algorithms/happo/happo_trainer.py instead of r_mappo.py (see ppo_update / train)
        self.actor = {k: v.detach().clone().to(dtype).requires_grad_(True) for k, v in actor.items()}
        self.critic = {k: v.detach().clone().to(dtype).requires_grad_(True) for k, v in critic.items()}
        self.opt_a = torch.optim.Adam(list(self.actor.values()), lr=cfg.lr, eps=cfg.opti_eps, weight_decay=0)
        self.opt_c = torch.optim.Adam(list(self.critic.values()), lr=cfg.critic_lr, eps=cfg.opti_eps,
                                      weight_decay=0)
        self.vn = ValueNormState() if cfg.use_valuenorm else None

    # ---- rollout side (rMAPPOPolicy.py:48-86) ----
    @torch.no_grad()
    def get_actions(self, share_obs, obs, h_a, h_c, masks, avail=None, deterministic=False, exp_noise=None):
        t = lambda a: None if a is None else torch.as_tensor(np.asarray(a), dtype=self.dtype)
        acts, lps, h_a2 = actor_act(self.cfg, self.actor, t(obs), t(h_a), t(masks), t(avail), deterministic,
                                    None if exp_noise is None else torch.as_tensor(exp_noise, dtype=self.dtype))
        vals, h_c2 = critic_forward(self.cfg, self.critic, t(share_obs), t(h_c), t(masks))
        return vals, acts, lps, h_a2, h_c2

    @torch.no_grad()
    def get_values(self, share_obs, h_c, masks):
        t = lambda a: torch.as_tensor(np.asarray(a), dtype=self.dtype)
        return critic_forward(self.cfg, self.critic, t(share_obs), t(h_c), t(masks))[0]

    # ---- one optimiser step (r_mappo.py:91-169) ----
    def ppo_update(self, sample, update_actor=True, keep_grads=False):
        c = self.cfg
        t = lambda a: None if a is None else torch.as_tensor(np.asarray(a), dtype=self.dtype)
        (share_obs, obs, h_a, h_c, actions, v_old, ret, masks, active, lp_old, adv, avail) = map(t, sample[:12])

        values, _ = critic_forward(c, self.critic, share_obs, h_c, masks)
        logp, ent = actor_evaluate(c, self.actor, obs, h_a, actions, masks, avail, active)

        if self.happo:                                     # happo_trainer.py:129-141: joint ratio, per-row factor
            factor = t(sample[12])
            ratio = torch.prod(torch.exp(logp - lp_old), dim=-1, keepdim=True)
            s1 = ratio * adv
            s2 = torch.clamp(ratio, 1.0 - c.clip_param, 1.0 + c.clip_param) * adv
            per_row = -torch.sum(factor * torch.min(s1, s2), dim=-1, keepdim=True)
        else:
            ratio = torch.exp(logp - lp_old)                                      # :129
            s1 = ratio * adv
            s2 = torch.clamp(ratio, 1.0 - c.clip_param, 1.0 + c.clip_param) * adv
            per_row = -torch.sum(torch.min(s1, s2), dim=-1, keepdim=True)
        pol = (per_row * active).sum() / active.sum() if c.use_policy_active_masks else per_row.mean()  # :134-139

        self.opt_a.zero_grad()
        if update_actor:
            (pol - ent * c.entropy_coef).backward()                               # :146
        a_gn = self._clip(self.actor, c)                                          # :148-151
        a_grads = {k: (v.grad.clone() if v.grad is not None else torch.zeros_like(v))
                   for k, v in self.actor.items()} if keep_grads else None
        self.opt_a.step()                                                         # :153

        v_clip = v_old + (values - v_old).clamp(-c.clip_param, c.clip_param)      # :62-63
        if self.vn is not None:
            if not self.happo:                 # happo_trainer.py:56-66 normalises with the state as is (never updates it)
                self.vn.update(ret.numpy())                                       # :65
            mean, var = self.vn.mean_var()
            target = (ret - torch.tensor(mean)) / torch.sqrt(torch.tensor(var))    # fp32, valuenorm.py:63-64
        else:
            target = ret
        e_c, e_o = target - v_clip, target - values
        if c.use_huber_loss:
            l_c, l_o = _huber(e_c, c.huber_delta), _huber(e_o, c.huber_delta)
        else:
            l_c, l_o = e_c ** 2 / 2, e_o ** 2 / 2
        vl = torch.max(l_o, l_c) if c.use_clipped_value_loss else l_o
        vl = (vl * active).sum() / active.sum() if c.use_value_active_masks else vl.mean()   # :83-86

        self.opt_c.zero_grad()
        (vl * c.value_loss_coef).backward()                                       # :160
        c_gn = self._clip(self.critic, c)
        c_grads = {k: v.grad.clone() for k, v in self.critic.items()} if keep_grads else None
        self.opt_c.step()                                                         # :167

        out = dict(value_loss=float(vl.detach()), policy_loss=float(pol.detach()), dist_entropy=float(ent.detach()),
                   actor_grad_norm=float(a_gn), critic_grad_norm=float(c_gn), ratio=float(ratio.mean().detach()))
        if keep_grads:
            out["actor_grads"], out["critic_grads"] = a_grads, c_grads
        return out

    @staticmethod
    def _clip(params, c):
        ps = [v for v in params.values() if v.grad is not None]
        if not ps:
            return 0.0
        if c.use_max_grad_norm:
            return torch.nn.utils.clip_grad_norm_(ps, c.max_grad_norm)
        return math.sqrt(sum(float(v.grad.norm()) ** 2 for v in ps))            # utils/util.py:9-15

    # ---- r_mappo.py:171-224 ----
    def train(self, store: RolloutStore, perms: Optional[List[np.ndarray]] = None, update_actor=True, factor=None):
        """`factor` [T, N, M, 1]: the separated buffers' importance factor (separated_buffer.py:62-63), yielded as the 13th
        element of every minibatch (:197-227); MAPPO ignores it (r_mappo.py:108-111), HAPPO multiplies it in."""
        c = self.cfg
        # happo_trainer.py:181-184 denormalises the value predictions only under use_popart (never with ValueNorm)
        adv = normalized_advantages(store, None if self.happo else self.vn)
        info = dict(value_loss=0.0, policy_loss=0.0, dist_entropy=0.0, actor_grad_norm=0.0,
                    critic_grad_norm=0.0, ratio=0.0)
        for e in range(c.ppo_epoch):
            perm = perms[e] if perms is not None else torch.randperm(perm_length(c)).numpy()
            for sample in minibatches(store, adv, perm, factor):
                o = self.ppo_update(sample, update_actor)
                for k in info:
                    info[k] += o[k]
        n = c.ppo_epoch * c.num_mini_batch
        return {k: v / n for k, v in info.items()}


def perm_length(c: PathConfig) -> int:
    """Argument of the torch.randperm call of the selected generator (shared_buffer.py:360, 415, 511)."""
    B = c.episode_length * c.n_rollout_threads * c.num_agents
    if c.use_recurrent_policy:
        return B // c.data_chunk_length
    if c.use_naive_recurrent_policy:
        return c.n_rollout_threads * c.num_agents
    return B


# --------------------------------------------------------------------------------------------
# synthetic environment feed (SURVEY section 8d) and the full iteration (mpe_runner.py:26-40,
# base_runner.py:120-141) -- used by tests (parity) and by bench.py's CPU legs (timing)
# --------------------------------------------------------------------------------------------
@dataclass
class SyntheticFeed:
    """Pre-generated env outputs for one iteration: obs/share_obs for slots 0..T, rewards, dones, masks."""
    obs: np.ndarray           # [T+1, N, M, Do]
    share_obs: np.ndarray     # [T+1, N, M, Ds]
    rewards: np.ndarray       # [T, N, M, 1]
    dones: np.ndarray         # [T, N, M] bool (agent-level, mpe_runner.py:128-131)
    active_masks: Optional[np.ndarray] = None     # [T, N, M, 1] value for slot t+1
    available_actions: Optional[np.ndarray] = None  # [T+1, N, M, A]


def make_feed(cfg: PathConfig, seed: int = 0, kind: str = "mpe") -> SyntheticFeed:
    rng = np.random.RandomState(seed)
    T, N, M = cfg.episode_length, cfg.n_rollout_threads, cfg.num_agents
    obs = rng.randn(T + 1, N, M, cfg.obs_dim).astype(np.float32)
    if kind == "mpe" and cfg.share_obs_dim == cfg.obs_dim * M:
        share = np.repeat(obs.reshape(T + 1, N, 1, M * cfg.obs_dim), M, axis=2)     # mpe_runner.py:133-135
        rew = np.repeat(rng.randn(T, N, 1, 1).astype(np.float32), M, axis=2)        # shared reward
    else:
        share = rng.randn(T + 1, N, M, cfg.share_obs_dim).astype(np.float32)
        rew = rng.randn(T, N, M, 1).astype(np.float32)
    dones = np.zeros((T, N, M), dtype=bool)
    active = avail = None
    if kind == "mpe":
        dones[T - 1] = True                                                          # world_length == T
    else:                                                                            # smac / hanabi shaped
        env_done = rng.rand(T, N) < (1.0 / 60.0)
        dones[:] = env_done[:, :, None]
        active = (rng.rand(T, N, M, 1) < 0.9).astype(np.float32)
        active[dones] = 1.0
        if cfg.has_avail:
            avail = (rng.rand(T + 1, N, M, cfg.act_dims[0]) < 0.7).astype(np.float32)
            avail[..., 0] = np.maximum(avail[..., 0], (avail.sum(-1) == 0))
    return SyntheticFeed(obs, share, rew, dones, active, avail)


def run_iteration(cfg: PathConfig, learner: Learner, store: RolloutStore, feed: SyntheticFeed,
                  noise: Optional[np.ndarray] = None, perms: Optional[List[np.ndarray]] = None):
    """collect xT -> insert xT -> compute -> train -> after_update, on host arrays like the reference."""
    T, N, M = cfg.episode_length, cfg.n_rollout_threads, cfg.num_agents
    E = N * M
    cat = lambda a: a.reshape(E, *a.shape[2:])
    if store.step == 0 and not np.any(store.obs[0]):                                 # warmup (mpe_runner.py:81-93)
        store.obs[0], store.share_obs[0] = feed.obs[0], feed.share_obs[0]
        if feed.available_actions is not None:
            store.available_actions[0] = feed.available_actions[0]
    for t in range(T):
        avail = cat(store.available_actions[t]) if (feed.available_actions is not None) else None
        vals, acts, lps, h_a, h_c = learner.get_actions(
            cat(store.share_obs[t]), cat(store.obs[t]), cat(store.rnn_states[t]), cat(store.rnn_states_critic[t]),
            cat(store.masks[t]), avail, exp_noise=None if noise is None else noise[t])
        un = lambda x: x.numpy().reshape(N, M, *x.shape[1:])
        h_a, h_c = un(h_a).copy(), un(h_c).copy()
        d = feed.dones[t]
        h_a[d] = 0.0                                                                 # mpe_runner.py:128-131
        h_c[d] = 0.0
        masks = np.ones((N, M, 1), np.float32)
        masks[d] = 0.0
        store.insert(feed.share_obs[t + 1], feed.obs[t + 1], h_a, h_c, un(acts).astype(np.float32), un(lps),
                     un(vals), feed.rewards[t], masks,
                     active_masks=None if feed.active_masks is None else feed.active_masks[t],
                     available_actions=None if feed.available_actions is None else feed.available_actions[t + 1])
    nv = learner.get_values(cat(store.share_obs[-1]), cat(store.rnn_states_critic[-1]), cat(store.masks[-1]))
    compute_returns(store, nv.numpy().reshape(N, M, 1), learner.vn)                  # base_runner.py:120-134
    info = learner.train(store, perms)                                               # base_runner.py:136-141
    store.after_update()
    return info
