"""Device-side vectorised MPE `simple_spread` / `simple_reference` (SURVEY.md section 8(f), row f1): bindings of
mappo_mpe_spread_step / mappo_mpe_reference_step.

`DeviceSpreadEnv` owns the float64 world state on the GPU and writes observations / rewards / dones straight into the
buffers the rollout kernels consume -- a collect step then has no host round trip (the reference pays a SubprocVecEnv pipe
round trip plus NumPy physics per step, envs/env_wrappers.py:257-266).  `DeviceSpreadVecEnv` wraps it in the reference's
vec-env interface (reset() / step(one-hot actions) -> obs, rews, dones, infos as NumPy) so the unchanged runner can use it.
Either env can also be stepped inside the one-launch closed rollout loop (engine.RolloutEngine(device_env=...)), which reads
and writes the same state tensors.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check, ptr
from .core import stream_ptr


class DeviceSpreadEnv:
    WORLD = _lib.WORLD_SPREAD              # world kind of the one-launch closed loop (engine.RolloutEngine)

    def __init__(self, n_envs: int, num_agents: int = 3, num_landmarks: int = 3, episode_length: int = 25,
                 device="cuda", seed: int = 1):
        self.lib = _lib.load()
        self.N, self.M, self.L, self.EP = int(n_envs), int(num_agents), int(num_landmarks), int(episode_length)
        self.dev = torch.device(device)
        self.seed = int(seed)
        self.obs_dim = 4 + 2 * self.L + 4 * (self.M - 1)
        self.share_dim = self.M * self.obs_dim
        z = lambda *s: torch.zeros(*s, dtype=torch.float64, device=self.dev)
        self.apos, self.avel, self.lpos = z(self.N, self.M, 2), z(self.N, self.M, 2), z(self.N, self.L, 2)
        self.step_count = torch.zeros(self.N, dtype=torch.int32, device=self.dev)
        self.rng_counter = torch.zeros(1, dtype=torch.int64, device=self.dev)

    def _call(self, actions, reset_states, obs_out, share_out, rew_out, done_out):
        if reset_states is not None:
            reset_states = torch.as_tensor(reset_states, dtype=torch.float64, device=self.dev).contiguous()
            assert reset_states.numel() == self.N * 2 * (self.M + self.L)
            self._keep = reset_states                      # alive until the kernel has run (stream-ordered free otherwise)
        check(self.lib.mappo_mpe_spread_step(
            ptr(self.apos), ptr(self.avel), ptr(self.lpos), ptr(self.step_count), ptr(actions), ptr(reset_states),
            self.seed, ptr(self.rng_counter), self.N, self.M, self.L, self.EP, ptr(obs_out), ptr(share_out),
            ptr(rew_out), ptr(done_out), stream_ptr()))

    def reset(self, obs_out: torch.Tensor, share_out: torch.Tensor = None, reset_states=None):
        """envs.reset(): (re)draw every world, write obs [N*M, D] (and share_obs [N*M, M*D])."""
        self._call(None, reset_states, obs_out, share_out, None, None)

    def step(self, actions: torch.Tensor, obs_out, share_out, rew_out, done_out, reset_states=None):
        """envs.step(): `actions` float [N*M(, 1)] with integer values 0..4 (what mappo_policy_step stores)."""
        assert actions.is_contiguous() and actions.numel() == self.N * self.M
        self._call(actions, reset_states, obs_out, share_out, rew_out, done_out)


class DeviceSpreadVecEnv:
    """The reference's ShareVecEnv surface (envs/env_wrappers.py) over DeviceSpreadEnv, NumPy in / NumPy out."""

    def __init__(self, n_envs, num_agents=3, num_landmarks=3, episode_length=25, device="cuda", seed=1):
        self.env = DeviceSpreadEnv(n_envs, num_agents, num_landmarks, episode_length, device, seed)
        e = self.env
        f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=e.dev)
        self._obs, self._rew, self._done = f(e.N * e.M, e.obs_dim), f(e.N * e.M), f(e.N * e.M)
        self.num_envs = e.N
        Box = type("Box", (), {})
        Discrete = type("Discrete", (), {})
        self.observation_space, self.share_observation_space, self.action_space = [], [], []
        for _ in range(e.M):
            o, s, a = Box(), Box(), Discrete()
            o.shape, s.shape, a.n = (e.obs_dim,), (e.share_dim,), 5
            self.observation_space.append(o); self.share_observation_space.append(s); self.action_space.append(a)

    def reset(self):
        self.env.reset(self._obs)
        return self._obs.reshape(self.env.N, self.env.M, -1).cpu().numpy()

    def step(self, actions_env):
        e = self.env
        a = np.asarray(actions_env)
        if a.ndim == 3 and a.shape[-1] == 5:                      # one-hot, as the runner sends it (mpe_runner.py:112-119)
            a = a.argmax(-1)
        act = torch.as_tensor(a.reshape(-1), dtype=torch.float32).to(e.dev)
        e.step(act, self._obs, None, self._rew, self._done)
        obs = self._obs.reshape(e.N, e.M, -1).cpu().numpy()
        rew = self._rew.reshape(e.N, e.M, 1).cpu().numpy()
        done = self._done.reshape(e.N, e.M).cpu().numpy() != 0
        # (the kernel exports the shared reward only; the reference logs the per-agent term here)
        infos = [[{"individual_reward": float(rew[i, m, 0])} for m in range(e.M)] for i in range(e.N)]
        return obs, rew, done, infos

    def close(self):
        pass


class DeviceReferenceEnv:
    """N `simple_reference` worlds on the device (mappo_mpe_reference_step): 2 agents, 3 landmarks, 10 symbols;
    actions [N*2, 2] = (move, symbol) as the policy stores a MultiDiscrete sample; obs [N*2, 21]."""
    M, L, DIM_C = 2, 3, 10
    WORLD = _lib.WORLD_REFERENCE

    def __init__(self, n_envs: int, episode_length: int = 25, device="cuda", seed: int = 1):
        self.lib = _lib.load()
        self.N, self.EP = int(n_envs), int(episode_length)
        self.dev = torch.device(device)
        self.seed = int(seed)
        self.obs_dim = 2 + 2 * self.L + 3 + self.DIM_C
        self.share_dim = self.M * self.obs_dim
        z = lambda *s: torch.zeros(*s, dtype=torch.float64, device=self.dev)
        zi = lambda *s: torch.zeros(*s, dtype=torch.int32, device=self.dev)
        self.apos, self.avel, self.lpos = z(self.N, 2, 2), z(self.N, 2, 2), z(self.N, 3, 2)
        self.goal, self.comm, self.step_count = zi(self.N, 2), zi(self.N, 2), zi(self.N)
        self.rng_counter = torch.zeros(1, dtype=torch.int64, device=self.dev)

    def _call(self, actions, reset_states, obs_out, share_out, rew_out, done_out):
        if reset_states is not None:
            reset_states = torch.as_tensor(reset_states, dtype=torch.float64, device=self.dev).contiguous()
            assert reset_states.numel() == self.N * 12
            self._keep = reset_states
        check(self.lib.mappo_mpe_reference_step(
            ptr(self.apos), ptr(self.avel), ptr(self.lpos), ptr(self.goal), ptr(self.comm), ptr(self.step_count),
            ptr(actions), ptr(reset_states), self.seed, ptr(self.rng_counter), self.N, self.EP, ptr(obs_out),
            ptr(share_out), ptr(rew_out), ptr(done_out), stream_ptr()))

    def reset(self, obs_out, share_out=None, reset_states=None):
        self._call(None, reset_states, obs_out, share_out, None, None)

    def step(self, actions, obs_out, share_out, rew_out, done_out, reset_states=None):
        assert actions.is_contiguous() and actions.dtype == torch.float32 and actions.numel() == self.N * 4
        self._call(actions, reset_states, obs_out, share_out, rew_out, done_out)


class DeviceReferenceVecEnv:
    """ShareVecEnv surface over DeviceReferenceEnv; step() takes what the runner sends for a MultiDiscrete space: the two
    heads one-hot and concatenated, [N, 2, 15] (mpe_runner.py:112-119), or the integer pairs [N, 2, 2]."""

    def __init__(self, n_envs, episode_length=25, device="cuda", seed=1):
        self.env = e = DeviceReferenceEnv(n_envs, episode_length, device, seed)
        f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=e.dev)
        self._obs, self._rew, self._done = f(e.N * 2, e.obs_dim), f(e.N * 2), f(e.N * 2)
        self.num_envs = e.N
        Box = type("Box", (), {})
        MultiDiscrete = type("MultiDiscrete", (), {})
        self.observation_space, self.share_observation_space, self.action_space = [], [], []
        for _ in range(2):
            o, s, a = Box(), Box(), MultiDiscrete()
            o.shape, s.shape = (e.obs_dim,), (e.share_dim,)
            a.high, a.low, a.shape = np.array([4, 9]), np.array([0, 0]), 2
            self.observation_space.append(o); self.share_observation_space.append(s); self.action_space.append(a)

    def reset(self):
        self.env.reset(self._obs)
        return self._obs.reshape(self.env.N, 2, -1).cpu().numpy()

    def step(self, actions_env):
        e = self.env
        a = np.asarray(actions_env)
        if a.shape[-1] == 15:
            a = np.stack([a[..., :5].argmax(-1), a[..., 5:].argmax(-1)], axis=-1)
        act = torch.as_tensor(np.ascontiguousarray(a.reshape(-1, 2)), dtype=torch.float32).to(e.dev)
        e.step(act, self._obs, None, self._rew, self._done)
        obs = self._obs.reshape(e.N, 2, -1).cpu().numpy()
        rew = self._rew.reshape(e.N, 2, 1).cpu().numpy()
        done = self._done.reshape(e.N, 2).cpu().numpy() != 0
        infos = [[{"individual_reward": float(rew[i, m, 0])} for m in range(2)] for i in range(e.N)]
        return obs, rew, done, infos

    def close(self):
        pass
