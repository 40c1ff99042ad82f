"""The one-launch closed rollout loop (mappo_rollout_closed_loop_ex, csrc/rollout_closed.cuh) for GRU policies on a 2-CTA cluster,
and for the simple_reference world with feed-forward and GRU policies: bit-for-bit against the per-step path
(T x [policy_step -> mpe_*_step -> env_insert]), replayed through the oracle environments, under CUDA-graph replay, and the
refusals of nets the kernels do not cover."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import mappo_oracle as O
from oracle.mpe_oracle import ReferenceVecEnv, SpreadVecEnv
from test_gpu_mpe_env import ATOL, RTOL


def _cfg(world, recurrent, N, M=3, L=3):
    if world == "reference":
        obs, share, acts, md, M = 21, 42, (5, 10), True, 2
    else:
        obs = 4 + 2 * L + 4 * (M - 1)
        obs, share, acts, md = obs, M * obs, (5,), False
    return O.PathConfig(episode_length=25, n_rollout_threads=N, num_agents=M, obs_dim=obs, share_obs_dim=share, act_dims=acts,
                        multi_discrete=md, use_ReLU=world == "reference", use_recurrent_policy=recurrent,
                        data_chunk_length=10, ppo_epoch=2, num_mini_batch=1, lr=7e-4, critic_lr=7e-4)


def _env(world, N, ep, seed, M=3, L=3):
    from mappo_b200.mpe_env import DeviceReferenceEnv, DeviceSpreadEnv
    if world == "reference":
        return DeviceReferenceEnv(N, ep, device="cuda", seed=seed)
    return DeviceSpreadEnv(N, M, L, ep, device="cuda", seed=seed)


def _engine(cfg, world, ep, fused, monkeypatch, env_seed=9, M=3, L=3):
    import test_gpu_parity as TP
    from mappo_b200.engine import RolloutEngine
    monkeypatch.setenv("MAPPO_B200_PERSISTENT_ROLLOUT", "1" if fused else "0")
    torch.manual_seed(1)
    args, policy, trainer, buf = TP.build(cfg)
    env = _env(world, cfg.n_rollout_threads, ep, env_seed, M, L)
    eng = RolloutEngine(args, policy, trainer, buf, rng="device", seed=4, device_env=env)
    assert eng.closed_persistent == fused
    return eng, policy, buf, env


def _state(policy, buf, env):
    t = [buf.obs, buf.share_obs, buf.rnn_states, buf.rnn_states_critic, buf.rewards, buf.masks, buf.actions,
         buf.value_preds, buf.action_log_probs, env.apos, env.avel, env.lpos, env.step_count, env.rng_counter,
         policy.rng_offset, policy.actor.flat, policy.critic.flat]
    if hasattr(env, "goal"):
        t += [env.goal, env.comm]
    return [x.clone() for x in t]


# (world, recurrent, N, agents, landmarks, episode length): 3/3 spread runs the compile-time world, 3/2 spread the runtime one
# (obs 16, share_obs 48; with 17 worlds some straddle two warps and the last cluster is partly filled); episode length 10 ends
# episodes inside the 25-step rollout
CASES = [("spread", True, 33, 3, 3, 25), ("spread", True, 17, 3, 2, 10), ("reference", True, 33, 2, 3, 10),
         ("reference", False, 33, 2, 3, 25)]


@pytest.mark.gpu
@pytest.mark.parametrize("world,recurrent,N,M,L,ep", CASES)
def test_one_launch_equals_the_per_step_closed_loop_bit_for_bit(world, recurrent, N, M, L, ep, monkeypatch):
    """Two iterations with device-RNG resets: storage (both rnn-state tensors included), world state, both counters and the
    trained weights are identical."""
    cfg = _cfg(world, recurrent, N, M, L)
    outs = []
    for fused in (True, False):
        eng, policy, buf, env = _engine(cfg, world, ep, fused, monkeypatch, M=M, L=L)
        eng.reset_env()
        for _ in range(2):
            eng.step_resident()
        torch.cuda.synchronize()
        outs.append(_state(policy, buf, env))
    for i, (a, b) in enumerate(zip(*outs)):
        assert torch.equal(a, b), i
    T = cfg.episode_length
    assert env.rng_counter.item() == 2 * T * N + N             # reset_env + two iterations of T steps
    assert policy.rng_offset.item() == 2 * T * N * cfg.num_agents


@pytest.mark.gpu
@pytest.mark.parametrize("world", ["spread", "reference"])
def test_episodes_ending_inside_a_rollout_replay_through_the_oracle(world, monkeypatch):
    """Episode length 10 with T = 25: replaying the stored actions through the oracle environment from the injected starts
    reproduces obs, share_obs, rewards and masks (simple_reference bit for bit), and the stored states of rows whose episode
    ended are zero."""
    N, T, ep = 21, 25, 10
    cfg = _cfg(world, True, N)
    eng, policy, buf, env = _engine(cfg, world, ep, True, monkeypatch)
    ref = ReferenceVecEnv(N, ep, seed=11) if world == "reference" else SpreadVecEnv(N, 3, 3, ep, seed=11)
    starts = ref.draw_reset_states(N)
    rs = np.stack([ref.draw_reset_states(N) for _ in range(T)])          # a different restart state per step
    eng.env_reset_states = torch.from_numpy(rs).cuda()
    eng.reset_env(reset_states=starts)
    eng.step_resident()
    torch.cuda.synchronize()
    M = cfg.num_agents
    ref.reset(starts)
    acts = buf.actions.cpu().numpy().reshape(T, N, M, -1).astype(np.int64)
    want = [ref.step(acts[t] if world == "reference" else acts[t, ..., 0], rs[t]) for t in range(T)]
    want_obs = np.array([w[0] for w in want]).astype(np.float32)
    want_rew = np.array([w[1] for w in want]).astype(np.float32)
    want_mask = 1.0 - np.array([w[2] for w in want]).astype(np.float32)
    got_obs, got_rew = buf.obs.cpu().numpy()[1:], buf.rewards.cpu().numpy()
    if world == "reference":
        np.testing.assert_array_equal(got_obs, want_obs)
        np.testing.assert_array_equal(got_rew, want_rew)
    else:
        np.testing.assert_allclose(got_obs, want_obs, rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(got_rew, want_rew, rtol=RTOL, atol=ATOL)
    masks = buf.masks.cpu().numpy()[1:, ..., 0]
    np.testing.assert_array_equal(masks, want_mask)
    assert (masks == 0).any(axis=(1, 2)).tolist() == [(t + 1) % ep == 0 for t in range(T)]
    np.testing.assert_array_equal(buf.share_obs.cpu().numpy()[1:], np.repeat(got_obs.reshape(T, N, 1, -1), M, axis=2))
    for h in (buf.rnn_states, buf.rnn_states_critic):
        h = h.cpu().numpy()[1:].reshape(T, N, M, -1)
        done = masks == 0
        assert np.all(h[done] == 0)
        assert np.all(np.abs(h[~done]).max(axis=-1) > 0)
    assert np.isfinite(policy.actor.flat.cpu().numpy()).all()


@pytest.mark.gpu
@pytest.mark.parametrize("world", ["spread", "reference"])
def test_graph_replay_of_the_recurrent_closed_loop_equals_eager(world, monkeypatch):
    """A captured iteration computes what the eager one does (world state, storage, counters, weights)."""
    N, ep = 19, 10
    cfg = _cfg(world, True, N)
    outs = []
    for graph in (False, True):
        eng, policy, buf, env = _engine(cfg, world, ep, True, monkeypatch)
        eng.reset_env()
        if graph:
            eng.capture(warmup=1)
            eng.step_resident()
        else:
            eng.launch_iteration()
            eng.launch_iteration()
        torch.cuda.synchronize()
        assert eng.launches_per_iteration > 0
        outs.append(_state(policy, buf, env))
    for i, (a, b) in enumerate(zip(*outs)):
        assert torch.equal(a, b), i


def _desc(in_dim, heads, critic, recurrent=1):
    from mappo_b200 import _lib
    d = _lib.NetDesc()
    d.in_dim, d.hidden, d.layer_n, d.use_feature_norm, d.use_relu, d.recurrent = in_dim, 64, 1, 1, 1, recurrent
    d.n_heads = len(heads)
    for k, a in enumerate(heads):
        d.head_dim[k] = a
    d.is_critic = int(critic)
    return d


def test_refusals_name_the_mismatch_before_any_launch():
    """Shapes that do not match the world are MAPPO_ERR_INVALID, nets off the warp-per-row kernels MAPPO_ERR_UNSUPPORTED; both
    are refused on the host before anything is launched (the pointers here are host buffers that are never dereferenced)."""
    from mappo_b200 import _lib
    lib = _lib.load()
    buf = (C.c_double * 64)()
    p = C.addressof(buf)

    def call(actor, critic, world, M, L):
        return lib.mappo_rollout_closed_loop_ex(C.byref(actor), p, C.byref(critic), p, p, p, p, p, p, p, p, p, p, world,
                                                p, p, p, p, p, p, None, 1, p, None, 1, p, 25, 4 * M, M, L, 25, None)

    ref_a, ref_c = _desc(21, (5, 10), False), _desc(42, (1,), True)
    spr_a, spr_c = _desc(18, (5,), False), _desc(54, (1,), True)
    assert call(ref_a, ref_c, _lib.WORLD_SPREAD, 3, 3) == -1                         # reference nets, spread world
    assert b"do not match simple_spread" in lib.mappo_last_error()
    assert call(spr_a, spr_c, _lib.WORLD_REFERENCE, 2, 3) == -1                      # spread nets, reference world
    assert b"do not match simple_reference" in lib.mappo_last_error()
    assert call(_desc(21, (5,), False), ref_c, _lib.WORLD_REFERENCE, 2, 3) == -1     # one action head only
    assert call(spr_a, _desc(65, (1,), True), _lib.WORLD_SPREAD, 3, 3) == -3         # in_dim 65 critic: tile kernels only
    assert b"warp-per-row" in lib.mappo_last_error()
    assert call(_desc(18, (5,), False, 0), spr_c, _lib.WORLD_SPREAD, 3, 3) == -3     # feed-forward actor, GRU critic
    assert call(ref_a, ref_c, 7, 2, 3) == -1
    assert b"unknown world" in lib.mappo_last_error()
    assert lib.mappo_rollout_closed_loop_ex(C.byref(ref_a), p, C.byref(ref_c), p, p, p, None, p, p, p, p, p, p,
                                            _lib.WORLD_REFERENCE, p, p, p, p, p, p, None, 1, p, None, 1, p, 25, 8, 2, 3, 25,
                                            None) == -1                              # GRU nets without state storage
    assert b"without state storage" in lib.mappo_last_error()
