"""Hidden-64 policies whose input is wider than 64 (or exactly 64), against float64 evaluations of the oracle's network.

Which kernel runs depends on the input width: up to 64 the warp-per-row rollout kernels (csrc/rollout_mlp.cuh,
rollout_gru.cuh), from 65 the 32-row tile kernels of csrc/policy_step.cu with their own packed image; the fp32 update runs
update_mlp_kernel<64, 4, 4> up to 64 and <64, 4, 8> above (also the base MLP of the fp32 GRU pipeline); from 97 inputs its
tiles no longer fit in shared memory, and from 129 it is not built: both are refused before launch.
The persistent rollout takes the warp-per-row path only when BOTH nets qualify, so one wide critic moves the actor onto the
tile kernels too.  4-agent simple_spread (obs 24, share_obs 96) and SMAC states are such shapes.

Reference: O.actor_act / O.actor_evaluate / O.critic_forward / O.Learner in float64, with every LayerNorm affine and bias
perturbed away from its initial value (at initialisation the LayerNorm biases are 0, which hides terms of the backward).
Tolerances: forward (values, log-probs, GRU states one step from the kernel's own stored state) rtol 1e-4 / atol 1e-5; actions
equal wherever the float64 margin between the best and second-best p / q exceeds 1e-5 relative, one of the tied candidates
inside it; first-update gradients as tests/helpers.py grad_agreement (fp32 build), losses 1e-4.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import mappo_oracle as O
from helpers import assert_close, grad_agreement, rollout_image_floats
from argsutil import make_args
import test_gpu_parity as TP
from test_gpu_bignet import _perturb, _sample

pytestmark = pytest.mark.gpu

F64 = torch.float64


def _perturb_all(policy, seed):
    """test_gpu_bignet._perturb (LayerNorm affines, Linear biases, heads) plus the GRU biases (bias_ih_l0 / bias_hh_l0)."""
    _perturb(policy, seed)
    g = torch.Generator().manual_seed(seed + 1000)
    for net in (policy.actor, policy.critic):
        for k, v in net.state_dict().items():
            if ".bias_" in k:
                v.copy_((0.1 * torch.randn(v.shape, generator=g)).to(v.device))


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _gru_fast_warps(n_rows, n_nets, sm_count):
    """csrc/rollout_gru.cuh gru_fast_warps: warps (two rows each) per CTA of the two-rows-per-warp GRU kernels."""
    ctas = max(sm_count // n_nets, 1)
    return min(max((n_rows + 2 * ctas - 1) // (2 * ctas), 2), 16)


def _params64(net):
    return {k: v.detach().cpu().to(F64) for k, v in net.state_dict().items()}


def _feed(cfg, seed):
    """Staged env outputs: dones in the middle of episodes, and (Discrete heads) availability masks where every 4th row
    allows exactly one action."""
    rng = np.random.RandomState(seed)
    T, N, M = cfg.episode_length, cfg.n_rollout_threads, cfg.num_agents
    obs = (rng.randn(T + 1, N, M, cfg.obs_dim) * 1.5 + 0.3).astype(np.float32)
    share = (rng.randn(T + 1, N, M, cfg.share_obs_dim) * 1.5 - 0.2).astype(np.float32)
    rew = rng.randn(T, N, M, 1).astype(np.float32)
    dones = rng.rand(T, N, M) < 0.15
    avail = None
    if cfg.has_avail:
        A = cfg.act_dims[0]
        avail = (rng.rand(T + 1, N, M, A) < 0.6).astype(np.float32)
        avail[..., 0] = np.maximum(avail[..., 0], avail.sum(-1) == 0)
        one = np.zeros((T + 1, N, M, A), np.float32)
        np.put_along_axis(one, rng.randint(0, A, size=(T + 1, N, M, 1)), 1.0, axis=-1)
        avail.reshape(-1, A)[::4] = one.reshape(-1, A)[::4]
    return O.SyntheticFeed(obs, share, rew, dones, None, avail)


def _noise(cfg, seed):
    E = cfg.n_rollout_threads * cfg.num_agents
    return np.random.RandomState(seed).exponential(size=(cfg.episode_length, E, sum(cfg.act_dims))).astype(np.float32)


def _run_rollout(cfg, policy, trainer, buf, feed, noise, persistent, monkeypatch):
    """Per step: policy._step + buffer.insert (T x mappo_policy_step).  Persistent: the engine's one-launch rollout with the
    staged feed and injected noise.  Returns the engine (persistent) or None."""
    if not persistent:
        TP.warm(buf, feed)
        TP.collect_and_returns(cfg, policy, trainer, buf, feed, noise)
        torch.cuda.synchronize()
        return None
    from mappo_b200.engine import RolloutEngine
    from mappo_b200._lib import check, ptr
    from mappo_b200.core import stream_ptr
    monkeypatch.setenv("MAPPO_B200_PERSISTENT_ROLLOUT", "1")
    args = make_args(cfg)
    eng = RolloutEngine(args, policy, trainer, buf, rng="host", seed=1)
    assert eng.persistent_rollout
    eng.stage_feed(feed)
    eng.draw_host_rng = lambda: None
    eng.host["noise"].copy_(torch.from_numpy(noise))
    eng.upload()
    for net, img in ((policy.actor, eng.img_actor), (policy.critic, eng.img_critic)):
        check(eng.lib.mappo_pack_rollout_weights_ex(C.byref(net.desc), ptr(net.flat), ptr(img), eng.gemm, stream_ptr()))
    eng._rollout_persistent()
    eng._returns()
    torch.cuda.synchronize()
    return eng


def _check_rollout(cfg, policy, buf, feed, noise, what):
    """Every stored step against one float64 step of the oracle from the kernel's own stored inputs (teacher-forced)."""
    T, N, M, H = cfg.episode_length, cfg.n_rollout_threads, cfg.num_agents, cfg.hidden_size
    E = N * M
    pa, pc = _params64(policy.actor), _params64(policy.critic)
    g = lambda x: x.detach().cpu().numpy()
    obs, share = g(buf.obs), g(buf.share_obs)
    np.testing.assert_array_equal(obs, feed.obs)                    # the insert: rows stored bit for bit
    np.testing.assert_array_equal(share, feed.share_obs)
    ha, hc, masks = g(buf.rnn_states), g(buf.rnn_states_critic), g(buf.masks)
    acts, lps, vals = g(buf.actions), g(buf.action_log_probs), g(buf.value_preds)
    avail = g(buf.available_actions) if feed.available_actions is not None else None
    np.testing.assert_array_equal(masks[1:, ..., 0], 1.0 - feed.dones.astype(np.float32))
    d = lambda a, t, *s: torch.from_numpy(a[t].reshape(E, *s)).to(F64)
    err = dict(value=0.0, logp=0.0, state=0.0)
    near_ties = 0
    for t in range(T + 1):
        h_c = d(hc, t, 1, H)
        v_ref, hc_ref = O.critic_forward(cfg, pc, d(share, t, -1), h_c, d(masks, t, 1))
        # (the perturbed value head has weights ~2.5: a value is a sum of 64 O(1) terms, compared relative to the values' scale)
        assert_close(vals[t].reshape(E, 1), v_ref.numpy(), 1e-4, 1e-5 * max(1.0, float(v_ref.abs().max())), f"{what}: values t={t}")
        err["value"] = max(err["value"], float(np.abs(vals[t].reshape(E, 1) - v_ref.numpy()).max()))
        if t == T:
            break                                                   # slot T: the bootstrap value only
        x, h_a, m = d(obs, t, -1), d(ha, t, 1, H), d(masks, t, 1)
        av = d(avail, t, -1) if avail is not None else None
        a_t = torch.from_numpy(acts[t].reshape(E, -1)).to(F64)
        lp_ref, _ = O.actor_evaluate(cfg, pa, x, h_a, a_t, m, av)
        assert_close(lps[t].reshape(E, -1), lp_ref.numpy(), 1e-4, 1e-5, f"{what}: log-probs t={t}")
        err["logp"] = max(err["logp"], float(np.abs(lps[t].reshape(E, -1) - lp_ref.numpy()).max()))
        # sampled actions: argmax(p / q) of the float64 scores, or one of the near-tied candidates
        feat, ha_ref = O._features(cfg, pa, x, h_a, m)
        off = 0
        q = torch.from_numpy(noise[t]).to(F64)
        for k, lg in enumerate(O._head_logits(cfg, pa, feat, av)):
            A = lg.shape[-1]
            score = (lg - lg.logsumexp(-1, keepdim=True)).exp() / q[:, off:off + A]
            off += A
            top = score.topk(2, -1).values
            best = score.argmax(-1).numpy()
            got = acts[t].reshape(E, -1)[:, k].astype(np.int64)
            tie = ((top[:, 0] - top[:, 1]) <= 1e-5 * top[:, 0]).numpy()
            near_ties += int(tie.sum())
            assert np.array_equal(got[~tie], best[~tie]), f"{what}: actions t={t} head {k}"
            cand = (score >= top[:, :1] * (1 - 1e-5)).numpy()
            assert cand[np.arange(E), got].all(), f"{what}: action outside the near-tied candidates, t={t} head {k}"
        if cfg.recurrent:
            done = feed.dones[t].reshape(E)
            for h_store, h_ref, nm in ((ha, ha_ref, "actor"), (hc, hc_ref, "critic")):
                nxt = h_store[t + 1].reshape(E, H)
                assert np.all(nxt[done] == 0.0), f"{what}: {nm} state of a done row is not zero, t={t}"
                want = h_ref.reshape(E, H).numpy()
                assert_close(nxt[~done], want[~done], 1e-4, 1e-5, f"{what}: {nm} GRU state t={t + 1}")
                err["state"] = max(err["state"], float(np.abs(nxt[~done] - want[~done]).max(initial=0.0)))
    print(f"\n{what}: max |err| value {err['value']:.2e}, log-prob {err['logp']:.2e}, GRU state {err['state']:.2e}; "
          f"near-ties {near_ties}")
    return err, near_ties


def _image_path_is(policy, lib):
    """Per net: the rollout image the library builds -- 'fast' (warp-per-row layout) up to in_dim 64, 'tile' (32-row tiles)
    above -- checked against both layouts' sizes."""
    out = []
    for net in (policy.actor, policy.critic):
        dsc = net.desc
        fast, tile = rollout_image_floats(dsc.in_dim, dsc.layer_n, dsc.use_feature_norm, dsc.recurrent,
                                          sum(dsc.head_dim[k] for k in range(dsc.n_heads)))
        kind = "fast" if dsc.in_dim <= 64 else "tile"
        assert lib.mappo_rollout_image_floats(C.byref(dsc)) == (fast if kind == "fast" else tile), (dsc.in_dim, fast, tile)
        out.append(kind)
    return out


# (obs, share_obs) widths x the net's switches; every width pair runs for MLP and GRU nets
ROLLOUT_CASES = {
    "24-96": dict(obs_dim=24, share_obs_dim=96, act_dims=(5,), use_ReLU=False),           # 4-agent simple_spread widths
    "64-64": dict(obs_dim=64, share_obs_dim=64, act_dims=(6,), layer_N=2),
    "65-65": dict(obs_dim=65, share_obs_dim=65, act_dims=(7,), use_feature_normalization=False),
    "30-128": dict(obs_dim=30, share_obs_dim=128, act_dims=(9,), layer_N=2, use_ReLU=False),
    "100-127": dict(obs_dim=100, share_obs_dim=127, act_dims=(5, 7), multi_discrete=True),
    # one net on the warp-per-row layout, the other on the tile kernels, GRU included (the narrow net then loads its weights
    # from the flat parameters: its packed image has the warp-per-row layout and is smaller than the tile layout)
    "24-72": dict(obs_dim=24, share_obs_dim=72, act_dims=(5,), use_ReLU=False),
    "30-88": dict(obs_dim=30, share_obs_dim=88, act_dims=(9,), use_feature_normalization=False),
}
# Recurrent nets on the tile kernels keep the GRU matrices in shared memory too (make_smem_w + make_pol_smem, 227 KB per CTA).
# With feature normalisation the persistent kernel fits no width above 64, and the per-step kernel none above 80 for a critic
# (1 output) or 77 for a 7-action actor; without it the persistent kernel fits a critic up to 88.  Wider nets are refused before
# launch: (case, persistent) pairs that must raise.
GRU_TOO_WIDE = {(name, p) for name in ("24-96", "30-128", "100-127") for p in (False, True)} | {("24-72", True)}


def _rollout_cfg(name, recurrent, T=12, N=13, M=3):
    return O.PathConfig(episode_length=T, n_rollout_threads=N, num_agents=M, use_recurrent_policy=recurrent,
                        ppo_epoch=1, **ROLLOUT_CASES[name])


@pytest.mark.parametrize("persistent", [False, True], ids=["per_step", "persistent"])
@pytest.mark.parametrize("recurrent", [False, True], ids=["mlp", "gru"])
@pytest.mark.parametrize("name", list(ROLLOUT_CASES))
def test_rollout_matches_float64_at_wide_inputs(name, recurrent, persistent, monkeypatch):
    monkeypatch.setenv("MAPPO_B200_GEMM", "fp32")
    cfg = _rollout_cfg(name, recurrent)
    torch.manual_seed(3)
    args, policy, trainer, buf = TP.build(cfg)
    _perturb_all(policy, 4)
    from mappo_b200 import _lib
    paths = _image_path_is(policy, _lib.load())
    assert paths == ["fast" if w <= 64 else "tile" for w in (cfg.obs_dim, cfg.share_obs_dim)]
    feed, noise = _feed(cfg, 1), _noise(cfg, 2)
    if recurrent and (name, persistent) in GRU_TOO_WIDE:
        with pytest.raises(RuntimeError, match="shared memory"):
            _run_rollout(cfg, policy, trainer, buf, feed, noise, persistent, monkeypatch)
        torch.cuda.synchronize()
        return
    _run_rollout(cfg, policy, trainer, buf, feed, noise, persistent, monkeypatch)
    _check_rollout(cfg, policy, buf, feed, noise, f"{'gru' if recurrent else 'mlp'} {name} "
                   f"{'persistent' if persistent else 'per step'} ({'/'.join(paths)} images)")


def _gru_launch_rows(regime, sm):
    """Row counts E that put the persistent two-rows-per-warp GRU rollout (two nets) into each launch regime on `sm` SMs."""
    rows_per_warp_row = 2 * max(sm // 2, 1)                        # rows covered by one warp in every CTA
    if regime == "one_row":
        return 1
    if regime == "odd_partial_cta":                                # 7 warps, odd E, last CTA partly filled
        E = rows_per_warp_row * 6 + 1
        while _gru_fast_warps(E, 2, sm) != 7 or E % 14 == 0 or E % 2 == 0:
            E += 2
        return E
    return rows_per_warp_row * 17 + 1                              # above the 16-warp cap


@pytest.mark.parametrize("regime", ["one_row", "odd_partial_cta", "warp_cap"])
def test_gru_warp_per_row_rollout_launch_shapes(regime, monkeypatch):
    monkeypatch.setenv("MAPPO_B200_GEMM", "fp32")
    sm = _sm_count()
    E = _gru_launch_rows(regime, sm)
    w = _gru_fast_warps(E, 2, sm)
    if regime == "odd_partial_cta":
        assert w >= 3 and E % 2 == 1 and E % (2 * w) != 0
    if regime == "warp_cap":
        assert w == 16 and E > 2 * 16 * (sm // 2)
    cfg = O.PathConfig(episode_length=6, n_rollout_threads=E, num_agents=1, obs_dim=30, share_obs_dim=45, act_dims=(9,),
                       use_recurrent_policy=True, use_ReLU=False, ppo_epoch=1)
    torch.manual_seed(5)
    args, policy, trainer, buf = TP.build(cfg)
    _perturb_all(policy, 6)
    from mappo_b200 import _lib
    assert _image_path_is(policy, _lib.load()) == ["fast", "fast"]
    feed, noise = _feed(cfg, 7), _noise(cfg, 8)
    _run_rollout(cfg, policy, trainer, buf, feed, noise, True, monkeypatch)
    _check_rollout(cfg, policy, buf, feed, noise, f"gru warp-per-row E={E} ({w} warps per CTA, {sm} SMs)")


def _grad_report(policy, ref, smooth, report):
    """grad_agreement per tensor + whole-gradient relative L2 / cosine per net; returns (failing tensors, worst numbers)."""
    bad, worst = [], dict(elem=0.0, l2=0.0, whole_l2=0.0, cos=1.0)
    for net, key in ((policy.actor, "actor_grads"), (policy.critic, "critic_grads")):
        gv, rv = [], []
        for k, v in net.named_grads().items():
            want = ref[key][k].numpy().astype(np.float64)
            got = v.cpu().numpy().astype(np.float64)
            gv.append(got.reshape(-1)); rv.append(want.reshape(-1))
            ok, l2 = grad_agreement(got, want, f"{key} {k}", smooth, False, report)
            worst["elem"] = max(worst["elem"], float(np.abs(got - want).max() / (np.abs(want).max() + 1e-300)))
            worst["l2"] = max(worst["l2"], l2)
            if not ok:
                bad.append(f"{key} {k}")
        gv, rv = np.concatenate(gv), np.concatenate(rv)
        l2 = float(np.linalg.norm(gv - rv) / np.linalg.norm(rv))
        cos = float(gv @ rv / (np.linalg.norm(gv) * np.linalg.norm(rv)))
        report.append(f"{key}: whole-gradient relative L2 error {l2:.3e}, cosine {cos:.8f}")
        worst["whole_l2"], worst["cos"] = max(worst["whole_l2"], l2), min(worst["cos"], cos)
        if smooth:
            if l2 > 1e-4:
                bad.append(f"{key} whole gradient")
        elif l2 > 1e-2 or cos < 0.999:
            bad.append(f"{key} whole gradient")
    return bad, worst


def _check_losses(out, ref, what):
    vl, cgn, pl, ent, agn, ratio = [float(x.reshape(-1)[0]) if torch.is_tensor(x) else float(x) for x in out]
    assert_close(vl, ref["value_loss"], 1e-4, 1e-6, f"{what}: value_loss")
    assert_close(pl, ref["policy_loss"], 1e-4, 1e-6, f"{what}: policy_loss")
    assert_close(ent, ref["dist_entropy"], 1e-4, 1e-6, f"{what}: dist_entropy")
    assert_close(ratio, ref["ratio"], 1e-4, 1e-6, f"{what}: ratio")
    assert_close([agn, cgn], [ref["actor_grad_norm"], ref["critic_grad_norm"]], 1e-3, 1e-7, f"{what}: grad norms")


def _update_cfg(width, relu, recurrent, **kw):
    return O.PathConfig(obs_dim=width, share_obs_dim=width, act_dims=(5, 7) if recurrent else (9,), multi_discrete=recurrent,
                        hidden_size=64, layer_N=1, use_ReLU=relu, use_recurrent_policy=recurrent, use_max_grad_norm=False,
                        entropy_coef=0.015, lr=7e-4, critic_lr=1e-3, **kw)


@pytest.mark.parametrize("relu", [False, True], ids=["tanh", "relu"])
@pytest.mark.parametrize("rows", ["ragged", "several_tiles_per_cta"])
@pytest.mark.parametrize("width", [64, 65, 80, 96])
def test_mlp_first_update_gradients_match_float64(width, rows, relu, monkeypatch):
    """fp32 build, update_mlp_kernel<64, 4, 4> at 64 and <64, 4, 8> above (the whole NJIN = 8 backward over the input), up to
    96, the widest input whose 64-row tiles fit in 227 KB of shared memory."""
    monkeypatch.setenv("MAPPO_B200_GEMM", "fp32")
    n_rows = 333 if rows == "ragged" else 2 * _sm_count() * 64 + 333
    cfg = _update_cfg(width, relu, False, episode_length=4, n_rollout_threads=4, num_agents=2)
    torch.manual_seed(11)
    args, policy, trainer, buf = TP.build(cfg)
    _perturb_all(policy, 5)
    vn = [0.3e-4, 1.7e-4, 1.2e-4]
    trainer.value_normalizer.state.copy_(torch.tensor(vn))
    sample = _sample(cfg, n_rows, 17)
    learner = O.Learner(cfg, _params64(policy.actor), _params64(policy.critic), dtype=F64)
    learner.vn.load(vn)
    ref = learner.ppo_update(sample, keep_grads=True)
    out = trainer.ppo_update(sample)
    torch.cuda.synchronize()
    what = f"mlp width {width} {'relu' if relu else 'tanh'} {n_rows} rows"
    _check_losses(out, ref, what)
    report = []
    bad, worst = _grad_report(policy, ref, not relu, report)
    print(f"\n{what}: worst max|err|/scale {worst['elem']:.2e}, tensor rel L2 {worst['l2']:.2e}, whole rel L2 "
          f"{worst['whole_l2']:.2e}, cosine {worst['cos']:.8f}")
    assert not bad, "\n".join(report)


@pytest.mark.parametrize("relu", [False, True], ids=["tanh", "relu"])
@pytest.mark.parametrize("width", [64, 65, 80, 96])
def test_gru_chunked_first_update_gradients_match_float64(width, relu, monkeypatch):
    """fp32 GRU pipeline (update_gru.cu): base forward and base backward through update_mlp_kernel (NJIN = 8 above 64) around
    the sequence kernels, on one chunked minibatch of recurrent_generator."""
    monkeypatch.setenv("MAPPO_B200_GEMM", "fp32")
    T, N, M, L = 20, 8, 3, 10
    cfg = _update_cfg(width, relu, True, episode_length=T, n_rollout_threads=N, num_agents=M, data_chunk_length=L,
                      num_mini_batch=2)
    torch.manual_seed(12)
    args, policy, trainer, buf = TP.build(cfg)
    _perturb_all(policy, 6)
    vn = [0.3e-4, 1.7e-4, 1.2e-4]
    trainer.value_normalizer.state.copy_(torch.tensor(vn))
    store = O.RolloutStore(cfg)
    rng = np.random.RandomState(width)
    store.obs[:] = rng.randn(*store.obs.shape) * 1.5 + 0.3
    store.share_obs[:] = rng.randn(*store.share_obs.shape) * 1.5 - 0.2
    store.rnn_states[:] = 0.5 * rng.randn(*store.rnn_states.shape)
    store.rnn_states_critic[:] = 0.5 * rng.randn(*store.rnn_states_critic.shape)
    store.actions[:] = np.stack([rng.randint(0, a, size=(T, N, M)) for a in cfg.act_dims], -1)
    store.action_log_probs[:] = -1.5 + 0.3 * rng.randn(*store.action_log_probs.shape)
    store.value_preds[:] = rng.randn(*store.value_preds.shape)
    store.returns[:] = rng.randn(*store.returns.shape) * 2 + 0.5
    store.masks[:] = rng.rand(*store.masks.shape) > 0.1
    store.active_masks[:] = rng.rand(*store.active_masks.shape) > 0.2
    for nm in ("share_obs", "obs", "rnn_states", "rnn_states_critic", "actions", "action_log_probs", "value_preds", "returns",
               "masks", "active_masks"):
        getattr(buf, nm).copy_(torch.from_numpy(getattr(store, nm)))
    adv = rng.randn(T, N, M, 1).astype(np.float32)
    perm = np.random.RandomState(1).permutation(T * N * M // L)
    monkeypatch.setattr(torch, "randperm", TP.FakeRandperm([perm]))
    sample = next(buf.recurrent_generator(adv, cfg.num_mini_batch, L))
    learner = O.Learner(cfg, _params64(policy.actor), _params64(policy.critic), dtype=F64)
    learner.vn.load(vn)
    ref = learner.ppo_update(next(iter(O.minibatches(store, adv, perm))), keep_grads=True)
    out = trainer.ppo_update(sample)
    torch.cuda.synchronize()
    what = f"gru width {width} {'relu' if relu else 'tanh'} {T * N * M // cfg.num_mini_batch} rows in chunks of {L}"
    _check_losses(out, ref, what)
    report = []
    bad, worst = _grad_report(policy, ref, not relu, report)
    print(f"\n{what}: worst max|err|/scale {worst['elem']:.2e}, tensor rel L2 {worst['l2']:.2e}, whole rel L2 "
          f"{worst['whole_l2']:.2e}, cosine {worst['cos']:.8f}")
    assert not bad, "\n".join(report)


def test_tf32_actor_and_fp32_critic_in_one_trainer_match_float64(monkeypatch):
    """MAPPO_B200_GEMM=tf32 with an actor of width 30 (tcgen05 update) and a critic of width 96 (not offered in tf32: the fp32
    update_mlp_kernel<64, 4, 8>), through a full 2-epoch train()."""
    from mappo_b200 import _lib
    monkeypatch.setenv("MAPPO_B200_GEMM", "tf32")
    cfg = O.PathConfig(episode_length=10, n_rollout_threads=8, num_agents=3, obs_dim=30, share_obs_dim=96, act_dims=(5,),
                       use_ReLU=False, ppo_epoch=2, lr=7e-4, critic_lr=7e-4)
    torch.manual_seed(13)
    args, policy, trainer, buf = TP.build(cfg)
    _perturb_all(policy, 7)
    feed = O.make_feed(cfg, seed=3, kind="smac")
    noise = _noise(cfg, 4)
    TP.warm(buf, feed)
    TP.collect_and_returns(cfg, policy, trainer, buf, feed, noise)
    learner = O.Learner(cfg, _params64(policy.actor), _params64(policy.critic), dtype=F64)
    learner.vn.load(trainer.value_normalizer.state.cpu().numpy())
    store = O.RolloutStore(cfg)                        # the kernel's rollout, teacher-forced into the oracle's storage
    for nm in ("share_obs", "obs", "actions", "action_log_probs", "value_preds", "returns", "rewards", "masks", "bad_masks",
               "active_masks", "available_actions"):
        getattr(store, nm)[:] = getattr(buf, nm).cpu().numpy().reshape(getattr(store, nm).shape)
    perms = [np.random.RandomState(20 + e).permutation(O.perm_length(cfg)) for e in range(cfg.ppo_epoch)]
    monkeypatch.setattr(torch, "randperm", TP.FakeRandperm(perms))
    info = trainer.train(buf)
    # the workspaces train() ran with: the actor's tf32 (tcgen05) build, the critic's fp32 update_mlp_kernel<64, 4, 8>
    assert trainer._ws and all(ws_a.gemm_mode == _lib.GEMM_TF32 and ws_c.gemm_mode == _lib.GEMM_FP32
                               for ws_a, ws_c in trainer._ws.values())
    want = learner.train(store, perms)
    for k in ("policy_loss", "dist_entropy", "ratio"):
        assert_close(info[k], want[k], 2e-2, 2e-4, f"train_info[{k}] (tf32 actor)")
    assert_close(info["actor_grad_norm"], want["actor_grad_norm"], 5e-3, 1e-6, "actor grad norm (tf32)")
    assert_close(info["value_loss"], want["value_loss"], 2e-3, 2e-5, "value_loss (fp32 critic)")
    assert_close(info["critic_grad_norm"], want["critic_grad_norm"], 2e-3, 2e-5, "critic grad norm (fp32 critic)")
    steps = cfg.ppo_epoch * cfg.num_mini_batch
    worst = {}
    for net, ref, rtol, atol, nm in ((policy.actor, learner.actor, 2e-2, 2.1 * steps * cfg.lr, "actor"),
                                     (policy.critic, learner.critic, 2e-2, 2.1 * steps * cfg.critic_lr, "critic")):
        for k, v in net.state_dict().items():
            got, w = v.cpu().numpy(), ref[k].detach().numpy()
            assert_close(got, w, rtol, atol, f"{nm} {k} after train()")
            worst[nm] = max(worst.get(nm, 0.0), float(np.abs(got - w).max()))
    print(f"\nmixed tf32 actor (30) / fp32 critic (96): max |weight err| actor {worst['actor']:.2e}, critic {worst['critic']:.2e}")


@pytest.mark.parametrize("width,message", [(97, "shared memory"), (128, "shared memory"), (129, "in_dim 129")])
def test_too_wide_update_is_refused_before_launch(width, message, monkeypatch):
    """The fused update is not built for hidden-64 nets wider than 128 inputs, and from 97 inputs its 64-row tiles need more than
    227 KB of shared memory: the library refuses with the reason in the message before launching anything, so the CUDA context
    stays usable."""
    monkeypatch.setenv("MAPPO_B200_GEMM", "fp32")
    cfg = _update_cfg(width, False, False, episode_length=4, n_rollout_threads=4, num_agents=2)
    with pytest.raises(RuntimeError, match=message):
        torch.manual_seed(1)
        args, policy, trainer, buf = TP.build(cfg)
        trainer.ppo_update(_sample(cfg, 64, 1))
        torch.cuda.synchronize()
    ok = _update_cfg(18, False, False, episode_length=4, n_rollout_threads=4, num_agents=2)
    torch.manual_seed(1)
    args, policy, trainer, buf = TP.build(ok)
    out = trainer.ppo_update(_sample(ok, 64, 1))
    torch.cuda.synchronize()
    assert all(np.isfinite(float(x.reshape(-1)[0]) if torch.is_tensor(x) else float(x)) for x in out)


def _spread_cfg(N, M, T=10, **kw):
    od = 4 + 2 * M + 4 * (M - 1)                     # simple_spread with M agents and M landmarks
    return O.PathConfig(episode_length=T, n_rollout_threads=N, num_agents=M, obs_dim=od, share_obs_dim=M * od, act_dims=(5,),
                        use_ReLU=False, ppo_epoch=2, lr=7e-4, critic_lr=7e-4, **kw)


def _engine_iteration(cfg, share_obs_from_obs, monkeypatch):
    from mappo_b200.engine import RolloutEngine
    monkeypatch.setenv("MAPPO_B200_PERSISTENT_ROLLOUT", "1")
    torch.manual_seed(1)
    args, policy, trainer, buf = TP.build(cfg)
    eng = RolloutEngine(args, policy, trainer, buf, rng="host", seed=1, share_obs_from_obs=share_obs_from_obs)
    eng.stage_feed(O.make_feed(cfg, seed=0, kind="mpe"))
    torch.manual_seed(7)
    eng.step_e2e()
    torch.cuda.synchronize()
    return eng, policy, buf


def test_four_agent_spread_stages_share_obs(monkeypatch):
    """share_obs_from_obs with a 96-wide critic (4-agent simple_spread): the persistent rollout runs the tile kernels, which do
    not derive share_obs, so the engine stages it; the iteration equals one run without the option."""
    monkeypatch.setenv("MAPPO_B200_GEMM", "fp32")
    cfg = _spread_cfg(13, 4)
    assert (cfg.obs_dim, cfg.share_obs_dim) == (24, 96)
    eng, policy, buf = _engine_iteration(cfg, True, monkeypatch)
    assert not eng.share_from_obs
    eng2, policy2, buf2 = _engine_iteration(cfg, False, monkeypatch)
    for nm in ("obs", "share_obs", "actions", "action_log_probs", "value_preds", "returns", "rewards", "masks"):
        np.testing.assert_array_equal(getattr(buf, nm).cpu().numpy(), getattr(buf2, nm).cpu().numpy(), err_msg=nm)
    assert_close(policy.actor.flat.cpu().numpy(), policy2.actor.flat.cpu().numpy(), 1e-5, 1e-7, "actor weights")
    assert_close(policy.critic.flat.cpu().numpy(), policy2.critic.flat.cpu().numpy(), 1e-5, 1e-7, "critic weights")


def test_three_agent_spread_still_derives_share_obs(monkeypatch):
    """c1 / c2 shapes (obs 18, share_obs 54): share_obs stays derived on the device, so only obs crosses the bus."""
    monkeypatch.setenv("MAPPO_B200_GEMM", "fp32")
    cfg = _spread_cfg(16, 3)
    eng, policy, buf = _engine_iteration(cfg, True, monkeypatch)
    assert eng.share_from_obs
    eng2, _, buf2 = _engine_iteration(cfg, False, monkeypatch)
    T, E = cfg.episode_length, cfg.n_rollout_threads * cfg.num_agents
    assert eng2.h2d_bytes() - eng.h2d_bytes() == 4 * T * E * cfg.share_obs_dim
    np.testing.assert_array_equal(buf.share_obs.cpu().numpy(), buf2.share_obs.cpu().numpy())
    np.testing.assert_array_equal(buf.actions.cpu().numpy(), buf2.actions.cpu().numpy())


def test_four_agent_device_spread_runs_per_step_and_matches_the_oracle_env(monkeypatch):
    """DeviceSpreadEnv with 4 agents / 4 landmarks: mappo_rollout_closed_loop needs both nets on the warp-per-row path, so the
    engine steps policy -> env -> insert per step; replaying the stored actions through the oracle environment reproduces the
    stored observations, rewards and masks."""
    from mappo_b200.engine import RolloutEngine
    from mappo_b200.mpe_env import DeviceSpreadEnv
    from oracle.mpe_oracle import SpreadVecEnv
    monkeypatch.setenv("MAPPO_B200_PERSISTENT_ROLLOUT", "1")
    monkeypatch.setenv("MAPPO_B200_GEMM", "fp32")
    N, M, T = 11, 4, 25
    cfg = _spread_cfg(N, M, T)
    torch.manual_seed(1)
    args, policy, trainer, buf = TP.build(cfg)
    env = DeviceSpreadEnv(N, M, M, T, device="cuda", seed=5)
    ref = SpreadVecEnv(N, M, M, T, seed=11)
    starts = ref.draw_reset_states(N)
    nxt = ref.draw_reset_states(N)
    eng = RolloutEngine(args, policy, trainer, buf, rng="device", seed=2, device_env=env)
    assert not eng.closed_persistent
    eng.env_reset_states = torch.from_numpy(np.repeat(nxt[None], T, axis=0)).cuda()
    eng.reset_env(reset_states=starts)
    eng.step_resident()
    torch.cuda.synchronize()
    ref.reset(starts)
    acts = buf.actions.cpu().numpy().reshape(T, N, M).astype(np.int64)
    want_obs, want_rew, want_done = [], [], []
    for t in range(T):
        o, r, d = ref.step(acts[t], nxt)
        want_obs.append(o); want_rew.append(r); want_done.append(d)
    got_obs = buf.obs.cpu().numpy()
    np.testing.assert_allclose(got_obs[1:], np.array(want_obs).astype(np.float32), rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(buf.rewards.cpu().numpy(), np.array(want_rew).astype(np.float32), rtol=1e-6, atol=1e-6)
    np.testing.assert_array_equal(buf.masks.cpu().numpy()[1:, :, :, 0], 1.0 - np.array(want_done).astype(np.float32))
    np.testing.assert_array_equal(buf.share_obs.cpu().numpy()[1:],
                                  np.repeat(got_obs[1:].reshape(T, N, 1, M * cfg.obs_dim), M, axis=2))
    assert want_done[-1].all()
    assert np.isfinite(policy.actor.flat.cpu().numpy()).all() and np.isfinite(policy.critic.flat.cpu().numpy()).all()
