"""closed_loop_bench.py -- the closed MPE rollout loop (device worlds) with GRU policies: one launch
(mappo_rollout_closed_loop_ex, a 2-CTA cluster per world group) against the per-step path (T x [mappo_policy_step ->
mappo_mpe_*_step -> mappo_env_insert]), both inside a full training iteration.

    python scripts/closed_loop_bench.py [--iters 50] [--rounds 5] [--out FILE]

Shapes (the reference's rmappo MPE scripts):
    c3      simple_reference, 2 agents, 128 rollout threads, T 25, GRU (ReLU), data_chunk_length 10, ppo_epoch 15
    spread  train_mpe_spread.sh: simple_spread 3 agents / 3 landmarks, 128 rollout threads, T 25, GRU (ReLU), ppo_epoch 10
Both train with the tcgen05 (tf32) update kernels; the rollout is fp32 either way.  For each shape the two modes are built in
this one process and timed alternately (`--rounds` rounds of `--iters` CUDA-graph replays each; the median round is
reported).  Per mode: collect ms (RolloutEngine.phase_breakdown: the collect phase alone, as its own graph), graph-replayed
ms per iteration, env-steps/s (threads x T / iteration time) and library launches per iteration.  The working set fits in L2
and is not flushed between iterations.  Prints one JSON line with the GPU name and power limit; --out also writes it to FILE.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "on-policy_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def shape(name):
    from oracle import mappo_oracle as O
    if name == "c3":
        cfg = O.PathConfig(episode_length=25, n_rollout_threads=128, num_agents=2, obs_dim=21, share_obs_dim=42,
                           act_dims=(5, 10), multi_discrete=True, use_recurrent_policy=True, data_chunk_length=10,
                           ppo_epoch=15, num_mini_batch=1, lr=7e-4, critic_lr=7e-4)
        return cfg, "reference"
    cfg = O.PathConfig(episode_length=25, n_rollout_threads=128, num_agents=3, obs_dim=18, share_obs_dim=54, act_dims=(5,),
                       use_recurrent_policy=True, data_chunk_length=10, ppo_epoch=10, num_mini_batch=1, lr=7e-4,
                       critic_lr=7e-4)
    return cfg, "spread"


def engine(cfg, world, fused):
    import torch
    from argsutil import make_args, make_spaces
    from onpolicy.algorithms.r_mappo.algorithm.rMAPPOPolicy import R_MAPPOPolicy
    from onpolicy.algorithms.r_mappo.r_mappo import R_MAPPO
    from onpolicy.utils.shared_buffer import SharedReplayBuffer
    from mappo_b200.engine import RolloutEngine
    from mappo_b200.mpe_env import DeviceReferenceEnv, DeviceSpreadEnv
    os.environ["MAPPO_B200_PERSISTENT_ROLLOUT"] = "1" if fused else "0"
    os.environ["MAPPO_B200_GEMM"] = "tf32"
    args = make_args(cfg)
    obs_s, share_s, act_s = make_spaces(cfg)
    torch.manual_seed(1)
    dev = torch.device("cuda:0")
    policy = R_MAPPOPolicy(args, obs_s, share_s, act_s, device=dev)
    trainer = R_MAPPO(args, policy, device=dev)
    buf = SharedReplayBuffer(args, cfg.num_agents, obs_s, share_s, act_s)
    N, T = cfg.n_rollout_threads, cfg.episode_length
    env = DeviceReferenceEnv(N, T, seed=3) if world == "reference" else DeviceSpreadEnv(N, 3, 3, T, seed=3)
    eng = RolloutEngine(args, policy, trainer, buf, rng="device", seed=2, device_env=env)
    assert eng.closed_persistent == fused
    eng.reset_env()
    eng.capture(warmup=2)
    return eng


def time_graph(eng, iters):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eng.step_resident()
    a.record()
    for _ in range(iters):
        eng.step_resident()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0), "sm_count": torch.cuda.get_device_properties(0).multi_processor_count}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"not read: {e}"
    return info


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--iters", type=int, default=50, help="graph replays per timed round")
    ap.add_argument("--rounds", type=int, default=5, help="alternating rounds per mode")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("closed_loop_bench.py measures on a CUDA device; none is visible")
    line = dict(gpu_info(), script="scripts/closed_loop_bench.py", iters_per_round=a.iters, rounds=a.rounds, l2_flush=False)
    for name in ("c3", "spread"):
        cfg, world = shape(name)
        engines = {"one_launch": engine(cfg, world, True), "per_step": engine(cfg, world, False)}
        ms = {k: [] for k in engines}
        for _ in range(a.rounds):
            for k, e in engines.items():
                ms[k].append(time_graph(e, a.iters))
        res = {"world": world, "threads": cfg.n_rollout_threads, "agents": cfg.num_agents, "T": cfg.episode_length,
               "ppo_epoch": cfg.ppo_epoch, "gemm": "tf32"}
        for k, e in engines.items():
            it = statistics.median(ms[k])
            pb = e.phase_breakdown()
            res[k] = {"collect_ms": round(pb["collect_insert_ms"], 4), "iteration_ms": round(it, 4),
                      "iteration_ms_rounds": [round(x, 4) for x in ms[k]],
                      "env_steps_per_s": round(cfg.n_rollout_threads * cfg.episode_length / (it * 1e-3), 1),
                      "launches_per_iteration": e.launches_per_iteration}
        res["one_launch_faster"] = res["one_launch"]["iteration_ms"] < res["per_step"]["iteration_ms"]
        line[name] = res
        del engines
        torch.cuda.synchronize()
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
