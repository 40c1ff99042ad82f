"""RolloutEngine: one whole iteration of the hot path as a single CUDA graph.

    collect x T  ->  insert x T  ->  get_values + compute_returns  ->  R_MAPPO update x (ppo_epoch * num_mini_batch)
    ->  after_update                                  (runner/shared/mpe_runner.py:26-40, base_runner.py:120-141)

Every launch goes through the C ABI of libmappo_b200 on the current stream; the graph is captured once and
replayed per iteration, so the host's share of an iteration is: refresh the pinned staging buffers (env outputs,
and -- in "host" RNG mode -- the reference's sampling noise / permutations), one graph launch, one 48-byte read.
The rollout kernels write values / actions / log-probs / rnn states STRAIGHT into the storage slots.  Three collect modes:
  * staged feed, persistent (default): all T steps + inserts + the bootstrap value in ONE launch (mappo_rollout_persistent),
  * staged feed, per step: T x (mappo_policy_step + mappo_env_insert)  (MAPPO_B200_PERSISTENT_ROLLOUT=0),
  * closed loop (device_env=DeviceSpreadEnv or DeviceReferenceEnv): the MPE worlds are stepped on the device between policy
    and insert -- inside one persistent kernel (mappo_rollout_closed_loop_ex; feed-forward and GRU policies, default) or as
    one extra launch per step (MAPPO_B200_PERSISTENT_ROLLOUT=0).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check, ptr
from .core import stream_ptr

class SegmentedGraph:
    """A CUDA graph cut at every collective: [graph][all_reduce][graph][all_reduce]...[graph].

    NCCL calls made through torch.distributed are kept OUT of stream capture (their watchdog / event bookkeeping is
    not capture-safe in every build); the kernels between two collectives are still one graph launch each.  All
    segments share one memory pool, so tensors allocated while capturing stay valid across segments."""

    def __init__(self):
        self.items, self.pool, self.cur = [], torch.cuda.graph_pool_handle(), None

    def begin(self):
        self.cur = torch.cuda.CUDAGraph()
        self.cur.capture_begin(pool=self.pool)

    def end(self):
        self.cur.capture_end()
        self.items.append(("graph", self.cur))
        self.cur = None

    def collective(self, t):
        """Called in place of dist.all_reduce while capturing."""
        self.end()
        self.items.append(("allreduce", t))
        self.begin()

    def replay(self):
        import torch.distributed as dist
        for kind, x in self.items:
            if kind == "graph":
                x.replay()
            else:
                dist.all_reduce(x, op=dist.ReduceOp.SUM)


INFO_KEYS = ("value_loss", "policy_loss", "dist_entropy", "actor_grad_norm", "critic_grad_norm", "ratio")


def warp_per_row_rollout(*descs) -> bool:
    """True when every net qualifies for the warp-per-row rollout kernels: hidden 64, in_dim <= 64 and at most 32 head
    outputs (csrc/rollout_mlp.cuh fast_rollout_supported, csrc/rollout_gru.cuh gru_fast_supported).  The persistent
    rollout takes that path only when BOTH nets qualify; otherwise it runs the 32-row tile kernels, which read share_obs
    from its own staging buffer, and the one-launch closed loop (mappo_rollout_closed_loop_ex) is not built at all."""
    return all(d.hidden == 64 and d.in_dim <= 64 and sum(d.head_dim[k] for k in range(d.n_heads)) <= 32 for d in descs)


class RolloutEngine:
    def __init__(self, args, policy, trainer, buffer, rng: str = "device", seed: int = 1,
                 share_obs_from_obs: bool = False, device_env=None):
        """share_obs_from_obs: the env's share_obs is the concatenation of the obs of the agents of a rollout thread
        (what the MPE runner builds on the host, mpe_runner.py:133-135): only obs is staged / uploaded and the critic
        reads its rows from it on the device (feed-forward policies, persistent rollout).
        device_env: a mappo_b200.mpe_env.DeviceSpreadEnv or DeviceReferenceEnv -- CLOSED LOOP: every collect step is
        policy_step -> env step -> insert on the device (no staged feed, no upload).  By default the whole collect is one launch
        with the worlds inside the rollout kernel; with MAPPO_B200_PERSISTENT_ROLLOUT=0 the env writes into the staging buffers
        the per-step insert reads."""
        self.args, self.policy, self.trainer, self.buffer = args, policy, trainer, buffer
        self.dev = policy.device
        self.rng = rng
        self.seed = int(seed)
        self.lib = _lib.load()
        b = buffer
        self.T, self.E = b.episode_length, b._E
        self.H = b.hidden_size
        self.Do, self.Ds = b.obs.shape[-1], b.share_obs.shape[-1]
        self.A = b.available_actions.shape[-1] if b.available_actions is not None else 0
        self.sumA = sum(policy.actor.head_dims)
        self.recurrent = bool(policy.actor.desc.recurrent)
        T, E = self.T, self.E
        f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=self.dev)
        import os
        self.env = device_env
        self.env_reset_states = None        # optional [T, N, reset doubles per world] float64: injected episode starts (parity tests)
        want_persistent = os.environ.get("MAPPO_B200_PERSISTENT_ROLLOUT", "1") == "1"
        # hidden >= 128 nets run the layer-by-layer GEMM pipeline per step (the persistent kernels keep weights in shared memory)
        self.big = bool(self.lib.mappo_big_net(C.byref(policy.actor.desc)))
        self.gemm = getattr(trainer, "gemm_mode", _lib.GEMM_FP32)
        if self.big:
            if device_env is not None:
                raise NotImplementedError("closed-loop device env with hidden >= 128 nets")
            want_persistent = False
        self.persistent_rollout = want_persistent and device_env is None
        # closed loop as ONE launch (mappo_rollout_closed_loop_ex): feed-forward or GRU policies whose nets both take the
        # warp-per-row path (a wider critic, e.g. 4-agent simple_spread's share_obs of 96, steps the env per step instead)
        fast = warp_per_row_rollout(policy.actor.desc, policy.critic.desc)
        self.closed_persistent = want_persistent and device_env is not None and fast
        if device_env is not None and (device_env.N * device_env.M != E or device_env.obs_dim != self.Do
                                       or device_env.share_dim != self.Ds):
            raise ValueError("device_env does not match the rollout storage (rows / obs_dim / share_obs_dim)")
        # (wider nets stage share_obs like any other input)
        self.share_from_obs = bool(share_obs_from_obs) and self.persistent_rollout and not self.recurrent and fast \
            and self.Ds % self.Do == 0 and E % (self.Ds // self.Do) == 0
        # device staging of one iteration of env outputs (next obs for slots 1..T, rewards, dones, ...): ONE flat buffer
        # (= one H2D copy per iteration) with views per field
        n_obs, n_share = T * E * self.Do, (0 if self.share_from_obs else T * E * self.Ds)
        self.d_stage = f(n_obs + n_share + 2 * T * E)
        self.h_stage = None
        o = 0
        self.d_obs = self.d_stage[o:o + n_obs].view(T, E, self.Do); o += n_obs
        self.d_share = self.d_stage[o:o + n_share].view(T, E, self.Ds) if n_share else None; o += n_share
        self.d_rew = self.d_stage[o:o + T * E].view(T, E, 1); o += T * E
        self.d_done = self.d_stage[o:o + T * E].view(T, E)
        self.d_active = None
        self.d_avail = None
        self.d_noise = f(T, E, self.sumA) if rng == "host" else None
        self.perm_len = trainer.perm_length(buffer)
        self.n_epochs = trainer.ppo_epoch
        self.d_perm = torch.zeros(self.n_epochs, self.perm_len, dtype=torch.int32, device=self.dev)
        self.perm_ctr = torch.zeros(1, dtype=torch.int64, device=self.dev)
        self.loss_out = torch.zeros(6, dtype=torch.float64, device=self.dev)
        self.h_loss = torch.zeros(6, dtype=torch.float64).pin_memory()
        # rollout weight images (shared-memory layout), re-packed once per iteration, fetched by TMA in policy_step
        # (hidden >= 128 nets: the image is the workspace of the layer-by-layer GEMM pipeline for E rows)
        self.img_actor = torch.zeros(int(self.lib.mappo_rollout_workspace_floats(C.byref(policy.actor.desc), self.E)),
                                     dtype=torch.float32, device=self.dev)
        self.img_critic = torch.zeros(int(self.lib.mappo_rollout_workspace_floats(C.byref(policy.critic.desc), self.E)),
                                      dtype=torch.float32, device=self.dev)
        self.host = {}
        self.graph = None
        self._allreduce = "auto"        # "auto": torch.distributed when a multi-rank group exists
        self._epoch_i = 0
        self.launches_per_iteration = 0

    # -- host staging ----------------------------------------------------------------------------
    def stage_feed(self, feed):
        """Pin one iteration of synthetic env outputs (oracle.SyntheticFeed layout) in host memory."""
        T, E = self.T, self.E
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).pin_memory()
        if self.share_from_obs:
            M = self.Ds // self.Do
            want = np.repeat(feed.obs.reshape(T + 1, E // M, 1, M * self.Do), M, axis=2).reshape(feed.share_obs.shape)
            if not np.array_equal(want, feed.share_obs):
                raise ValueError("share_obs_from_obs: the feed's share_obs is not the concatenation of its obs rows")
        # obs | [share_obs] | rewards | dones in one pinned buffer, mirrored by d_stage
        if self.h_stage is None:
            self.h_stage = torch.zeros(self.d_stage.numel(), dtype=torch.float32).pin_memory()
        parts = [feed.obs[1:]] + ([] if self.share_from_obs else [feed.share_obs[1:]]) + \
                [feed.rewards, feed.dones.astype(np.float32)]
        flat = np.concatenate([np.ascontiguousarray(a, dtype=np.float32).reshape(-1) for a in parts])
        assert flat.size == self.h_stage.numel()
        self.h_stage.copy_(torch.from_numpy(flat))
        self.host = dict(stage=self.h_stage)
        if feed.active_masks is not None:
            self.host["active"] = pin(feed.active_masks.reshape(T, E, 1))
            if self.d_active is None:
                self.d_active = torch.zeros(T, E, 1, dtype=torch.float32, device=self.dev)
        if feed.available_actions is not None:
            self.host["avail"] = pin(feed.available_actions[1:].reshape(T, E, -1))
            if self.d_avail is None:
                self.d_avail = torch.zeros(T, E, self.A, dtype=torch.float32, device=self.dev)
        # warm-up slot 0 (mpe_runner.py:81-93)
        b = self.buffer                                  # (separated buffers have no agent axis: reshape, same row order)
        b.obs[0].copy_(torch.from_numpy(feed.obs[0]).reshape(b.obs[0].shape))
        b.share_obs[0].copy_(torch.from_numpy(feed.share_obs[0]).reshape(b.share_obs[0].shape))
        if feed.available_actions is not None:
            b.available_actions[0].copy_(torch.from_numpy(feed.available_actions[0]).reshape(b.available_actions[0].shape))
        if self.rng == "host":
            self.host["noise"] = torch.zeros(T, E, self.sumA).pin_memory()
            self.host["perm"] = torch.zeros(self.n_epochs, self.perm_len, dtype=torch.int32).pin_memory()

    def h2d_bytes(self):
        return int(sum(v.numel() * v.element_size() for v in self.host.values()))

    def reset_env(self, reset_states=None):
        """Closed loop: envs.reset() into storage slot 0 (the runner's warmup, mpe_runner.py:81-93)."""
        self.env.reset(self.buffer.obs[0].view(self.E, self.Do), self.buffer.share_obs[0].view(self.E, self.Ds),
                       reset_states=reset_states)

    def upload(self):
        """Host -> device copy of this iteration's inputs (async, current stream)."""
        if self.env is not None:
            return                                             # closed loop: nothing comes from the host
        h = self.host
        self.d_stage.copy_(h["stage"], non_blocking=True)
        if "active" in h:
            self.d_active.copy_(h["active"], non_blocking=True)
        if "avail" in h:
            self.d_avail.copy_(h["avail"], non_blocking=True)
        if self.rng == "host":
            self.draw_host_rng()
            self.d_noise.copy_(h["noise"], non_blocking=True)
            self.d_perm.copy_(h["perm"], non_blocking=True)

    def draw_host_rng(self):
        """Consume torch's CPU generator exactly like one reference iteration does (SURVEY App. B-8):
        T x one exponential_ per head, then one randperm per epoch."""
        noise, perm = self.host["noise"], self.host["perm"]
        for t in range(self.T):
            off = 0
            for a in self.policy.actor.head_dims:
                noise[t, :, off:off + a] = torch.empty(self.E, a).exponential_(1)
                off += a
        for e in range(self.n_epochs):
            perm[e] = torch.randperm(self.perm_len).to(torch.int32)

    # -- device work -------------------------------------------------------------------------------
    def _collect_and_insert(self, t):
        b, pol, lib, st = self.buffer, self.policy, self.lib, stream_ptr()
        rec = self.recurrent
        noise = self.d_noise[t] if self.d_noise is not None else None
        check(lib.mappo_policy_step_ex(
            C.byref(pol.actor.desc), ptr(pol.actor.flat), C.byref(pol.critic.desc), ptr(pol.critic.flat),
            ptr(b.obs[t]), ptr(b.share_obs[t]), ptr(b.rnn_states[t]) if rec else None,
            ptr(b.rnn_states_critic[t]) if rec else None, ptr(b.masks[t]),
            ptr(b.available_actions[t]) if b.available_actions is not None else None, ptr(noise),
            self.seed, ptr(pol.rng_offset), 0, self.E,
            ptr(b.value_preds[t]), ptr(b.actions[t]), None, ptr(b.action_log_probs[t]),
            ptr(b.rnn_states[t + 1]) if rec else None, ptr(b.rnn_states_critic[t + 1]) if rec else None,
            ptr(self.img_actor), ptr(self.img_critic), self.gemm, st))
        if self.env is not None:             # closed loop: the env consumes the actions just written to slot t
            rs = self.env_reset_states[t] if self.env_reset_states is not None else None
            self.env.step(b.actions[t], self.d_obs[t], self.d_share[t], self.d_rew[t], self.d_done[t], reset_states=rs)
        check(lib.mappo_env_insert(
            ptr(self.d_obs[t]), ptr(self.d_share[t]), ptr(self.d_rew[t]), ptr(self.d_done[t]),
            ptr(self.d_active[t]) if self.d_active is not None else None,
            ptr(self.d_avail[t]) if self.d_avail is not None else None,
            self.E, self.Do, self.Ds, self.H, self.A,
            ptr(b.obs[t + 1]), ptr(b.share_obs[t + 1]), ptr(b.rewards[t]), ptr(b.masks[t + 1]),
            ptr(b.rnn_states[t + 1]) if rec else None, ptr(b.rnn_states_critic[t + 1]) if rec else None,
            ptr(b.active_masks[t + 1]) if self.d_active is not None else None,
            ptr(b.available_actions[t + 1]) if self.d_avail is not None else None,
            ptr(pol.rng_offset) if noise is None else None, self.E, st))

    def _rollout_persistent(self):
        """All T collect steps + inserts + the bootstrap value as ONE launch (mappo_rollout_persistent)."""
        b, pol, lib = self.buffer, self.policy, self.lib
        rec = self.recurrent
        check(lib.mappo_rollout_persistent(
            C.byref(pol.actor.desc), ptr(pol.actor.flat), ptr(self.img_actor),
            C.byref(pol.critic.desc), ptr(pol.critic.flat), ptr(self.img_critic),
            ptr(b.obs), ptr(b.share_obs), ptr(b.rnn_states) if rec else None, ptr(b.rnn_states_critic) if rec else None,
            ptr(b.masks), ptr(b.available_actions) if self.d_avail is not None else None,
            ptr(b.value_preds), ptr(b.actions), ptr(b.action_log_probs), ptr(b.rewards),
            ptr(b.active_masks) if self.d_active is not None else None,
            ptr(self.d_obs), ptr(self.d_share), ptr(self.d_rew), ptr(self.d_done),          # d_share None: from d_obs
            ptr(self.d_active) if self.d_active is not None else None,
            ptr(self.d_avail) if self.d_avail is not None else None,
            ptr(self.d_noise), self.seed, ptr(pol.rng_offset), self.T, self.E, stream_ptr()))

    def _rollout_closed(self):
        """Closed loop, all T steps + the bootstrap value as ONE launch (policy -> world step -> insert inside the kernel); the
        world kind comes from the env (simple_spread / simple_reference)."""
        b, pol, lib, env = self.buffer, self.policy, self.lib, self.env
        rs = self.env_reset_states
        rec = self.recurrent
        ref = env.WORLD == _lib.WORLD_REFERENCE
        check(lib.mappo_rollout_closed_loop_ex(
            C.byref(pol.actor.desc), ptr(self.img_actor), C.byref(pol.critic.desc), ptr(self.img_critic),
            ptr(b.obs), ptr(b.share_obs), ptr(b.rnn_states) if rec else None, ptr(b.rnn_states_critic) if rec else None,
            ptr(b.masks), ptr(b.value_preds), ptr(b.actions), ptr(b.action_log_probs), ptr(b.rewards), env.WORLD,
            ptr(env.apos), ptr(env.avel), ptr(env.lpos), ptr(env.goal) if ref else None, ptr(env.comm) if ref else None,
            ptr(env.step_count), ptr(rs) if rs is not None else None, env.seed, ptr(env.rng_counter), ptr(self.d_noise),
            self.seed, ptr(pol.rng_offset), self.T, self.E, env.M, env.L, env.EP, stream_ptr()))

    def _returns(self):
        b, lib, st, T = self.buffer, self.lib, stream_ptr(), self.T
        vn = self.trainer.value_normalizer
        b._adv_stats.zero_()
        check(lib.mappo_compute_returns(ptr(b.rewards), ptr(b.value_preds), ptr(b.masks), ptr(b.bad_masks),
                                        ptr(b.active_masks), ptr(vn.state) if vn is not None else None, T, self.E,
                                        float(b.gamma), float(b.gae_lambda), int(bool(b._use_gae)),
                                        int(bool(b._use_proper_time_limits)), ptr(b.returns), ptr(b.advantages),
                                        ptr(b._adv_stats), st))
        b._adv_version = id(vn) if vn is not None else 0

    def _compute(self):
        b, pol, lib, st, T = self.buffer, self.policy, self.lib, stream_ptr(), self.T
        rec = self.recurrent
        check(lib.mappo_policy_step_ex(
            C.byref(pol.actor.desc), None, C.byref(pol.critic.desc), ptr(pol.critic.flat),
            None, ptr(b.share_obs[T]), None, ptr(b.rnn_states_critic[T]) if rec else None, ptr(b.masks[T]),
            None, None, 0, None, 1, self.E, ptr(b.value_preds[T]), None, None, None, None, None,
            None, ptr(self.img_critic), self.gemm, st))
        vn = self.trainer.value_normalizer
        b._adv_stats.zero_()
        check(lib.mappo_compute_returns(ptr(b.rewards), ptr(b.value_preds), ptr(b.masks), ptr(b.bad_masks),
                                        ptr(b.active_masks), ptr(vn.state) if vn is not None else None, T, self.E,
                                        float(b.gamma), float(b.gae_lambda), int(bool(b._use_gae)),
                                        int(bool(b._use_proper_time_limits)), ptr(b.returns), ptr(b.advantages),
                                        ptr(b._adv_stats), st))
        b._adv_version = id(vn) if vn is not None else 0

    def _draw_perm(self, n):
        e = self._epoch_i
        self._epoch_i += 1
        out = self.d_perm[e]
        if self.rng != "host":
            # one counter bump per iteration (launch_iteration); epochs are told apart by the seed
            # (mappo_randperm_batch adds the same golden-ratio multiple per permutation)
            if self.d_perm.shape[0] > 1 and n == self.d_perm.shape[1]:
                if e == 0:          # every epoch's permutation in one launch
                    check(self.lib.mappo_randperm_batch(n, self.d_perm.shape[0], self.seed, ptr(self.perm_ctr),
                                                        ptr(self.d_perm), stream_ptr()))
            else:
                seed = (self.seed + 0x9E3779B97F4A7C15 * (e + 1)) & 0xFFFFFFFFFFFFFFFF
                check(self.lib.mappo_randperm(n, seed, ptr(self.perm_ctr), ptr(out), stream_ptr()))
        return out

    def launch_iteration(self):
        """Enqueue one full iteration on the current stream (no host synchronisation)."""
        n0 = self.lib.mappo_debug_launch_count()
        pol = self.policy
        check(self.lib.mappo_pack_rollout_weights_ex(C.byref(pol.actor.desc), ptr(pol.actor.flat), ptr(self.img_actor), self.gemm, stream_ptr()))
        check(self.lib.mappo_pack_rollout_weights_ex(C.byref(pol.critic.desc), ptr(pol.critic.flat), ptr(self.img_critic), self.gemm, stream_ptr()))
        if self.persistent_rollout:
            self._rollout_persistent()
            self._returns()
        elif self.closed_persistent:
            self._rollout_closed()
            self._returns()
        else:
            for t in range(self.T):
                self._collect_and_insert(t)
            self._compute()
        self._epoch_i = 0
        tr = self.trainer
        n_upd = tr.ppo_epoch * tr.num_mini_batch
        tr.launch_train(self.buffer, True, self._draw_perm, self.loss_out, allreduce=self._allreduce)
        if self.rng != "host":
            check(self.lib.mappo_counter_add(ptr(self.perm_ctr), 1, stream_ptr()))
        self.buffer.after_update()
        # kernels of OUR library enqueued by one iteration, counted by the library itself (memsets / torch copies excluded)
        self.launches_per_iteration = int(self.lib.mappo_debug_launch_count() - n0)

    def phase_breakdown(self, reps: int = 20):
        """Device time of the three phases of an iteration, each captured as its own CUDA graph and replayed `reps`
        times (single process only; diagnostic for bench.py)."""
        def timed(fn):
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                fn()
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                fn()
            torch.cuda.synchronize()
            g.replay()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                g.replay()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / reps

        def collect():
            pol = self.policy
            if self.persistent_rollout:
                check(self.lib.mappo_pack_rollout_weights_ex(C.byref(pol.actor.desc), ptr(pol.actor.flat), ptr(self.img_actor), self.gemm, stream_ptr()))
                check(self.lib.mappo_pack_rollout_weights_ex(C.byref(pol.critic.desc), ptr(pol.critic.flat), ptr(self.img_critic), self.gemm, stream_ptr()))
                self._rollout_persistent()
                return
            if self.closed_persistent:
                check(self.lib.mappo_pack_rollout_weights_ex(C.byref(pol.actor.desc), ptr(pol.actor.flat), ptr(self.img_actor), self.gemm, stream_ptr()))
                check(self.lib.mappo_pack_rollout_weights_ex(C.byref(pol.critic.desc), ptr(pol.critic.flat), ptr(self.img_critic), self.gemm, stream_ptr()))
                self._rollout_closed()
                return
            check(self.lib.mappo_pack_rollout_weights_ex(C.byref(pol.actor.desc), ptr(pol.actor.flat), ptr(self.img_actor), self.gemm, stream_ptr()))
            check(self.lib.mappo_pack_rollout_weights_ex(C.byref(pol.critic.desc), ptr(pol.critic.flat), ptr(self.img_critic), self.gemm, stream_ptr()))
            for t in range(self.T):
                self._collect_and_insert(t)

        def train():
            self._epoch_i = 0
            self.trainer.launch_train(self.buffer, True, self._draw_perm, self.loss_out, allreduce=None)

        # cycle split of one rollout pass inside CTA 0 of each net (clock64 accumulators of the kernel)
        buf = (C.c_int64 * 16)()
        torch.cuda.synchronize()
        self.lib.mappo_debug_pol_timing(buf, 1)
        collect()
        torch.cuda.synchronize()
        self.lib.mappo_debug_pol_timing(buf, 1)
        names = ["rows", "mlp_base", "gru_cell", "head_gemm", "sample_store"]
        cyc = {net: {nm: int(buf[8 * k + i]) for i, nm in enumerate(names)} for k, net in enumerate(("actor", "critic"))}
        return {"rollout_cycles_cta0": cyc, "collect_insert_ms": timed(collect),
                "values_gae_ms": timed(self._returns if (self.persistent_rollout or self.closed_persistent) else self._compute), "train_ms": timed(train),
                "after_update_ms": timed(self.buffer.after_update)}

    def capture(self, warmup: int = 2):
        """Warm up eagerly (lazy workspace allocation, cudaFuncSetAttribute) then capture the iteration."""
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(warmup):
                self.launch_iteration()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        import torch.distributed as dist
        multi = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        if multi and getattr(self.trainer, "_p2p", None) is None:
            seg = SegmentedGraph()
            self._allreduce = seg.collective
            try:
                with torch.cuda.stream(s):
                    seg.begin()
                    self.launch_iteration()
                    seg.end()
            finally:
                self._allreduce = "auto"
            torch.cuda.current_stream().wait_stream(s)
            self.graph = seg
        else:
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.launch_iteration()
        torch.cuda.synchronize()

    def step_resident(self):
        """One iteration with inputs already resident in HBM (device staging reused as is)."""
        if self.graph is not None:
            self.graph.replay()
        else:
            self.launch_iteration()

    def enable_input_prefetch(self):
        """Double-buffered input staging for step_e2e(): the host -> device copy of the NEXT iteration's env outputs runs on a copy
        stream underneath this iteration's graph (into shadow buffers; a device-to-device copy moves them into the staging the
        graph reads at the start of the next step).  Every step still performs one full H2D of pinned host inputs; it just no
        longer sits on the critical path.  Host buffers must not change between the prefetch and the step that consumes it
        (bench.py's staged feed; tests that rewrite the host buffers per step keep the synchronous path)."""
        if self.env is not None or self.rng == "host":
            return False
        self._pf = {"stream": torch.cuda.Stream(device=self.dev), "ready": torch.cuda.Event(), "consumed": torch.cuda.Event(),
                    "primed": False, "shadow": {}}
        pairs = {"stage": self.d_stage, "active": self.d_active, "avail": self.d_avail}
        for k, d in pairs.items():
            if k in self.host and d is not None:
                self._pf["shadow"][k] = (torch.empty_like(d), d)
        return True

    def _prefetch_issue(self):
        pf = self._pf
        with torch.cuda.stream(pf["stream"]):
            for k, (shadow, _) in pf["shadow"].items():
                shadow.view(-1).copy_(self.host[k].view(-1), non_blocking=True)
            pf["ready"].record(pf["stream"])

    def step_e2e(self):
        """One iteration from HOST buffers: H2D of the env outputs, the graph, D2H of train_info (+ sync)."""
        pf = getattr(self, "_pf", None)
        if pf is None:
            self.upload()
            self.step_resident()
        else:
            main = torch.cuda.current_stream()
            if not pf["primed"]:
                self._prefetch_issue()
                pf["primed"] = True
            main.wait_event(pf["ready"])                       # this step's inputs have landed in the shadow buffers
            for shadow, dst in pf["shadow"].values():
                dst.copy_(shadow, non_blocking=True)           # device-to-device
            pf["consumed"].record(main)
            self.step_resident()
            pf["stream"].wait_event(pf["consumed"])            # the shadows are free again: fetch the next step's inputs now
            self._prefetch_issue()
        self.h_loss.copy_(self.loss_out, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        n = float(self.trainer.ppo_epoch * self.trainer.num_mini_batch)
        return dict(zip(INFO_KEYS, (self.h_loss / n).tolist()))
