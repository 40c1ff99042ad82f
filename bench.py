#!/usr/bin/env python
"""bench.py -- env-steps/s through collect -> GAE -> ppo_update on synthetic rollouts of the BASELINE.json configs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2|c3|c4|c5] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

Default workload = BASELINE.json configs[1] ("c2", the configuration the metric is quoted on): MPE simple_spread-shaped,
3 agents, 128 rollout threads PER GPU (weak scaling), episode_length 25, shared MLP policy (Tanh, hidden 64), ppo_epoch 10.
One "step" = one full iteration
    T x (policy forward + sample + insert) -> get_values + compute_returns -> ppo_epoch x (actor + critic update) -> after_update
and processes threads * T env steps per GPU.  `--config` selects the other BASELINE configs (SURVEY.md App. C):
    c3  MPE simple_reference-shaped, 2 agents, 128 threads, GRU policy, recurrent_generator L = 10, ppo_epoch 15
    c4  SMAC 3m-shaped, 3 agents, 512 threads IN TOTAL (strong scaling: 512 / N per GPU), episode_length 400, GRU, ppo_epoch 15
    c5  Hanabi-Full-shaped, 2 players with SEPARATE policies, 1024 threads in total (1024 / N per GPU), episode_length 80,
        MLP hidden 512 / layer_N 2 (the TMA-fed tcgen05 GEMM pipeline), ppo_epoch 15
With --config c2 (the default) and one GPU the line also carries compact results of c3 and c5 under "other_configs"
(--no-extras skips them).

`value`  : K = --steps iterations replayed from inputs already resident in HBM, each device-timed with its own pair of CUDA
           events, L2 flushed between iterations; `ms_per_step` is the mean.
`e2e`    : then K more iterations driven from HOST buffers (pinned env outputs -> H2D, D2H of train_info) per step, wall clock.
`--dump-outputs DIR` : after the timed iterations, run one more iteration of the timed path from the seeded starting
           state and write what it hands its caller as DIR/<name>.npy (dump_outputs).  Inputs, initial weights and RNG
           seeds are fixed, so two builds run with the same arguments can be compared array by array.
`--impl reference` : the CPU restatement of the reference path (oracle/, see its header) on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "on-policy_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

UNIT = "env-steps/s"


# ------------------------------------------------------------------------------------------------
# workloads (SURVEY.md section 8 header + App. C)
# ------------------------------------------------------------------------------------------------
def workload(name, world=1, threads=None):
    """-> dict(cfg = PathConfig of ONE policy on ONE GPU, n_policies, feed, scaling, label, total_threads)."""
    from oracle import mappo_oracle as O
    if name == "c2":
        n = threads or 128
        cfg = O.PathConfig(episode_length=25, n_rollout_threads=n, num_agents=3, obs_dim=18, share_obs_dim=54,
                           act_dims=(5,), use_ReLU=False, ppo_epoch=10, num_mini_batch=1, lr=7e-4, critic_lr=7e-4)
        return dict(cfg=cfg, n_policies=1, feed="mpe", scaling="weak", total_threads=n * world,
                    label=f"c2: MPE simple_spread-shaped, 3 agents x {n} rollout threads per GPU x 25 steps, shared MLP "
                          "(tanh, H=64), ppo_epoch 10, 1 minibatch")
    if name == "c3":
        n = threads or 128
        cfg = O.PathConfig(episode_length=25, n_rollout_threads=n, num_agents=2, obs_dim=21, share_obs_dim=42,
                           act_dims=(5, 10), multi_discrete=True, use_recurrent_policy=True, data_chunk_length=10,
                           ppo_epoch=15, num_mini_batch=1, lr=7e-4, critic_lr=7e-4)
        return dict(cfg=cfg, n_policies=1, feed="mpe", scaling="weak", total_threads=n * world,
                    label=f"c3: MPE simple_reference-shaped, 2 agents x {n} rollout threads per GPU x 25 steps, shared GRU policy "
                          "(ReLU, H=64, MultiDiscrete[5,10]), recurrent_generator L=10, ppo_epoch 15")
    if name == "c4":
        tot = threads or 512
        n = max(tot // world, 1)
        cfg = O.PathConfig(episode_length=400, n_rollout_threads=n, num_agents=3, obs_dim=30, share_obs_dim=48,
                           act_dims=(9,), use_recurrent_policy=True, data_chunk_length=10, ppo_epoch=15, num_mini_batch=1,
                           lr=5e-4, critic_lr=5e-4, use_value_active_masks=False)
        return dict(cfg=cfg, n_policies=1, feed="smac", scaling="strong", total_threads=n * world,
                    label=f"c4: SMAC 3m-shaped (obs 30, state 48, 9 actions, avail + active masks), 3 agents x {n * world} rollout "
                          f"threads in total ({n} per GPU) x 400 steps, shared GRU policy, L=10, ppo_epoch 15")
    if name == "c5":
        tot = threads or 1024
        n = max(tot // world, 1)
        cfg = O.PathConfig(episode_length=80, n_rollout_threads=n, num_agents=1, obs_dim=660, share_obs_dim=785,
                           act_dims=(20,), hidden_size=512, layer_N=2, ppo_epoch=15, num_mini_batch=1, entropy_coef=0.015,
                           lr=7e-4, critic_lr=1e-3)
        return dict(cfg=cfg, n_policies=2, feed="smac", scaling="strong", total_threads=n * world,
                    label=f"c5: Hanabi-Full-shaped (obs 658+2, share 783+2, 20 actions, avail masks), 2 players with separate "
                          f"policies x {n * world} rollout threads in total ({n} per GPU) x 80 steps, MLP hidden 512 / layer_N 2 "
                          "(ReLU), ppo_epoch 15")
    raise SystemExit(f"unknown config {name}")


def metric_name(name):
    return {"c2": "env-steps/sec through collect->GAE->ppo_update (MAPPO, MPE simple_spread-shaped c2)",
            "c3": "env-steps/sec through collect->GAE->ppo_update (rMAPPO GRU, MPE simple_reference-shaped c3)",
            "c4": "env-steps/sec through collect->GAE->ppo_update (rMAPPO GRU, SMAC 3m-shaped c4)",
            "c5": "env-steps/sec through collect->GAE->ppo_update (MAPPO separated, Hanabi-Full-shaped c5)"}[name]


def workload_dict(w, n_gpus):
    cfg = w["cfg"]
    return {"workload": w["label"], "rollout_threads_per_gpu": cfg.n_rollout_threads, "global_rollout_threads": w["total_threads"],
            "episode_length": cfg.episode_length, "num_agents": cfg.num_agents * w["n_policies"], "ppo_epoch": cfg.ppo_epoch,
            "parallelism": f"dp{n_gpus} over rollout threads", "l2_flush_between_steps": True}


# ------------------------------------------------------------------------------------------------
# CPU legs (the only place bench.py executes oracle/)
# ------------------------------------------------------------------------------------------------
def cpu_iteration_rate(w, iters, warmup, threads):
    """env-steps/s of the CPU port on `threads` torch threads: all policies of the workload, `iters` timed iterations."""
    import torch
    from oracle import mappo_oracle as O
    cfg = w["cfg"]
    torch.set_num_threads(threads)
    torch.manual_seed(1)
    jobs = []
    for a in range(w["n_policies"]):
        learner = O.Learner(cfg, O.init_params(cfg, False, seed=1 + 2 * a), O.init_params(cfg, True, seed=2 + 2 * a))
        jobs.append((learner, O.RolloutStore(cfg), O.make_feed(cfg, seed=a, kind=w["feed"])))
    times = []
    for i in range(warmup + iters):
        t0 = time.perf_counter()
        for learner, store, feed in jobs:
            O.run_iteration(cfg, learner, store, feed)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    tot = sum(times)
    return cfg.n_rollout_threads * cfg.episode_length * len(times) / tot, tot / len(times)


def cpu_sample_workload(name):
    """A bounded sample of the workload for the CPU legs (same nets, horizon, epochs; fewer rollout threads where one
    iteration of the full batch would take minutes on the host)."""
    full = workload(name)
    n = {"c2": 128, "c3": 128, "c4": 8, "c5": 8}[name]
    return workload(name, 1, threads=n), full["total_threads"], n


def best_cpu_threads(w):
    """The port (like the reference) is many small torch ops: more intra-op threads is not always faster.  Probe a few
    counts with one iteration each and keep the fastest ("all the host threads it can USE")."""
    cores = os.cpu_count() or 1
    best, best_rate = 1, 0.0
    for th in sorted({1, min(4, cores), min(8, cores), min(16, cores), min(32, cores)}):
        rate, _ = cpu_iteration_rate(w, 1, 1, th)
        if rate > best_rate:
            best, best_rate = th, rate
    return best


def cpu_baseline(name, iters):
    w, full_threads, n = cpu_sample_workload(name)
    cores = best_cpu_threads(w)
    rate, per = cpu_iteration_rate(w, iters, 1, cores)
    sample = (f"{iters} full iterations of {name} " +
              (f"on a {n}-thread sample of the {full_threads} rollout threads " if n != full_threads else "") +
              f"({n * w['cfg'].episode_length} env steps each, all {w['cfg'].ppo_epoch} PPO epochs) of oracle/mappo_oracle.py on "
              f"{cores} torch threads (fastest of 1/4/8/16/32; host has {os.cpu_count()} cores), {per * 1e3:.0f} ms each")
    return {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}, per


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = workload(a.config, 1)
    steps = min(a.steps, {"c2": 60, "c3": 20, "c4": 3, "c5": 5}[a.config])
    base, per = cpu_baseline(a.config, steps)
    base["sample"] += ("; oracle/mappo_oracle.py = CPU restatement of the reference (the Python reference cannot travel to the "
                       "GPU box, and `pip install --target baseline/_ref /root/reference` yields a package without "
                       "algorithms/utils, r_mappo/algorithm and runner -- DESIGN.md section 5)")
    line = {"impl": "reference", "metric": metric_name(a.config), "value": base["value"], "unit": UNIT, "n_gpus": a.gpus,
            "steps": steps, "warmup": 1, "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": w["scaling"],
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_dict(w, 1), "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(int(r[1]) for r in self.rows if len(r) > 8 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) > 8 and r[2].isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) > 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def update_flops(cfg):
    """Algorithmic GEMM FLOPs of one optimiser step per net (SURVEY section 8a9/a12: 3F - 2*in*H per row; GRU adds 2*2*6H^2
    per row forward)."""
    H, L, B = cfg.hidden_size, cfg.layer_N, cfg.episode_length * cfg.n_rollout_threads * cfg.num_agents
    gru = 2 * 6 * H * H if cfg.recurrent else 0
    fa = 2 * (cfg.obs_dim * H + L * H * H + H * sum(cfg.act_dims)) + gru
    fc = 2 * (cfg.share_obs_dim * H + L * H * H + H) + gru
    return B * (3 * fa - 2 * cfg.obs_dim * H), B * (3 * fc - 2 * cfg.share_obs_dim * H)


def measure_tf32_peak(dev):
    """torch.matmul with TF32 inputs (cuBLAS, 8192^3), best of 5: the tensor-pipe denominator for kind::tf32 kernels."""
    import torch
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn(8192, 8192, device=dev)
        b = torch.randn(8192, 8192, device=dev)
        best = 1e9
        for i in range(7):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            torch.matmul(a, b)
            e.record()
            torch.cuda.synchronize()
            if i >= 2:
                best = min(best, s.elapsed_time(e))
        return 2 * 8192 ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


class Job:
    """One policy + trainer + rollout storage + engine on this rank (a separated-policy workload has several)."""

    def __init__(self, w, idx, dev, rank, a):
        import torch
        from oracle import mappo_oracle as O
        from argsutil import make_args, make_spaces
        from onpolicy.algorithms.r_mappo.algorithm.rMAPPOPolicy import R_MAPPOPolicy
        from onpolicy.algorithms.r_mappo.r_mappo import R_MAPPO
        from onpolicy.utils.shared_buffer import SharedReplayBuffer
        from onpolicy.utils.separated_buffer import SeparatedReplayBuffer
        from mappo_b200.engine import RolloutEngine
        cfg = w["cfg"]
        self.cfg = cfg
        args = make_args(cfg)
        obs_s, share_s, act_s = make_spaces(cfg)
        torch.manual_seed(1 + idx)                         # identical replicas on every rank
        self.policy = R_MAPPOPolicy(args, obs_s, share_s, act_s, device=dev)
        self.trainer = R_MAPPO(args, self.policy, device=dev)
        if w["n_policies"] > 1:
            self.buf = SeparatedReplayBuffer(args, obs_s, share_s, act_s)
        else:
            self.buf = SharedReplayBuffer(args, cfg.num_agents, obs_s, share_s, act_s)
        feed = O.make_feed(cfg, seed=100 + 17 * idx + rank, kind=w["feed"])     # each rank owns its own rollout threads
        if a.env == "device":
            from mappo_b200.mpe_env import DeviceSpreadEnv
            env = DeviceSpreadEnv(cfg.n_rollout_threads, cfg.num_agents, 3, cfg.episode_length, device=dev, seed=100 + rank)
            self.eng = RolloutEngine(args, self.policy, self.trainer, self.buf, rng="device", seed=1 + rank, device_env=env)
            self.eng.reset_env()
        else:
            self.eng = RolloutEngine(args, self.policy, self.trainer, self.buf, rng="device", seed=1 + rank + 101 * idx,
                                     share_obs_from_obs=(w["feed"] == "mpe"))
            self.eng.stage_feed(feed)
            self.eng.upload()


def run_config(name, a, world, rank, dev, dist, sampler=None):
    """Build the workload, time a.steps iterations."""
    import torch
    w = workload(name, world)
    cfg = w["cfg"]
    os.environ["MAPPO_B200_GEMM"] = a.gemm               # update-kernel GEMM engine: tcgen05 tf32 or exact fp32 FFMA
    jobs = [Job(w, i, dev, rank, a) for i in range(w["n_policies"])]
    torch.cuda.synchronize()
    graph_ok = not a.eager
    try:
        if a.eager:
            raise RuntimeError("--eager")
        for j in jobs:
            j.eng.capture(warmup=2)
    except Exception as e:                                 # e.g. a collective that refuses capture: run eagerly
        graph_ok = False
        for j in jobs:
            j.eng.graph = None
        torch.cuda.synchronize()
        if rank == 0 and not a.eager:
            print(f"[bench] CUDA graph capture unavailable ({type(e).__name__}: {e}); running eager", file=sys.stderr)
    if world > 1:                                          # every rank must run the same mode
        ok = torch.tensor([1 if graph_ok else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            graph_ok = False
            for j in jobs:
                j.eng.graph = None
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)       # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        for j in jobs:
            j.eng.step_resident()

    def step_e2e():
        info = None
        for j in jobs:
            info = j.eng.step_e2e()
        return info

    # ---- device-timed resident loop: exactly K steps, each between its own pair of events ----
    K = a.steps
    W = max(a.warmup, 3)
    for _ in range(W):
        step_resident()
    barrier()
    if sampler is not None:
        sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    t_wall0 = time.perf_counter()
    for s, e in evs:
        flush.zero_()                                      # L2 flush between timed iterations (outside the events)
        s.record()
        step_resident()
        e.record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = sum(j.eng.launches_per_iteration for j in jobs) * K

    # ---- end to end from host buffers (same flush discipline; its ~40 us of device time is inside the wall clock) ----
    # double-buffered staging: the H2D of the next iteration's inputs overlaps this iteration's graph (engine.enable_input_prefetch)
    prefetch = all([j.eng.enable_input_prefetch() for j in jobs]) if not getattr(a, "no_prefetch", False) else False
    for _ in range(3):
        step_e2e()
    info = None
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        flush.zero_()
        info = step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop() if sampler is not None else None

    # max over ranks of every step (and of the e2e loop), then the mean over steps
    t = torch.tensor([s.elapsed_time(e) for s, e in evs] + [e2e_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t = t.tolist()
    sm = t[:K]
    ms_step = sum(sm) / K
    e2e_ms_step = t[K] / K
    steps_env = cfg.n_rollout_threads * cfg.episode_length * world
    res = {"workload": w, "cfg": cfg, "jobs": jobs, "graph_ok": graph_ok, "ms_per_step": ms_step, "value": steps_env / (ms_step * 1e-3),
           "e2e_ms_per_step": e2e_ms_step, "e2e_value": steps_env / (e2e_ms_step * 1e-3),
           "step_ms": {"min": min(sm), "median": sorted(sm)[K // 2], "max": max(sm)},
           "launches": launches, "h2d": sum(j.eng.h2d_bytes() for j in jobs), "d2h": 48 * len(jobs), "clocks": clocks,
           "wall_s_timed_region": t_wall, "info": info, "flush": flush, "steps_env": steps_env, "prefetch": bool(prefetch)}
    return res


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(w, a, rank, dev, out_dir):
    """One iteration of the timed path (engine.launch_iteration, the launch sequence its CUDA graph replays) from the seeded
    starting state of the timed jobs -- same initial weights, staged inputs and RNG seeds -- and DIR/<name>.npy of what it
    hands its caller, per policy (prefix `policy<i>_` when there are several): train_info (float64, engine.INFO_KEYS
    order), the trained actor / critic parameter vectors, the value normaliser's state, and the rollout storage the
    iteration filled (actions, log-probs, value predictions, returns, advantages).
    Not the last timed iteration itself: float atomics in the update sum in a different order from run to run, and over
    tens of iterations the sampled actions turn those last-bit differences into different trajectories."""
    import numpy as np
    import torch
    jobs = [Job(w, i, dev, rank, a) for i in range(w["n_policies"])]
    for j in jobs:
        j.eng.step_resident()                              # no graph captured: launch_iteration()
    torch.cuda.synchronize()
    if rank != 0:
        return
    arrays = {}
    for i, j in enumerate(jobs):
        pre = f"policy{i}_" if len(jobs) > 1 else ""
        n = j.trainer.ppo_epoch * j.trainer.num_mini_batch
        arrays[pre + "train_info"] = (j.eng.loss_out / n).cpu().numpy()
        arrays[pre + "actor_params"] = j.policy.actor.flat
        arrays[pre + "critic_params"] = j.policy.critic.flat
        if j.trainer.value_normalizer is not None:
            arrays[pre + "value_normalizer"] = j.trainer.value_normalizer.state
        for k in ("actions", "action_log_probs", "value_preds", "returns", "advantages"):
            arrays[pre + k] = getattr(j.buf, k)
    arrays = {k: v if isinstance(v, np.ndarray) else v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def kernel_roofline(res, a, peaks, tf32_peak):
    """Live CUDA-event timing of the dominant kernel in one eager train() per job (events on the launching stream)."""
    import ctypes as C
    import torch
    from mappo_b200 import core
    jobs, cfg = res["jobs"], res["cfg"]
    lib = core._lib.load()
    big = bool(jobs[0].eng.big)
    fa, fc = update_flops(cfg)
    out = {}
    if big:
        # hidden >= 128: the update is a pipeline of GEMM launches; the library times each kernel family with events
        lib.mappo_debug_big_timing(1, None, None)
        saved = [(j.eng.graph, j.trainer.overlap_nets) for j in jobs]
        try:
            for j in jobs:
                j.eng.graph, j.trainer.overlap_nets = None, False
            res["flush"].zero_()
            for j in jobs:
                j.eng._epoch_i = 0
                j.trainer.launch_train(j.buf, True, j.eng._draw_perm, j.eng.loss_out, allreduce=None)
            torch.cuda.synchronize()
        finally:
            for j, (g, o) in zip(jobs, saved):
                j.eng.graph, j.trainer.overlap_nets = g, o
        ms = (C.c_double * 7)()
        cnt = (C.c_int64 * 7)()
        lib.mappo_debug_big_timing(0, ms, cnt)
        fam = ["pack", "feature_norm", "fwd_gemm", "head_loss", "bwd_gemm", "grad_gemm", "reduce_unfold"]
        table = {f: {"ms_total": ms[i], "launches": int(cnt[i])} for i, f in enumerate(fam)}
        H, L, B = cfg.hidden_size, cfg.layer_N, cfg.episode_length * cfg.n_rollout_threads
        n_upd = cfg.ppo_epoch * cfg.num_mini_batch * len(jobs)            # per net kind
        ins = (cfg.obs_dim, cfg.share_obs_dim)
        heads = (sum(cfg.act_dims), 1)
        fl = {"fwd_gemm": sum(2 * B * (i * H + L * H * H) for i in ins) * n_upd,
              "bwd_gemm": sum(2 * B * (L * H * H + H * h) for h in heads) * n_upd,
              "grad_gemm": sum(2 * B * (i * H + L * H * H + H * h) for i, h in zip(ins, heads)) * n_upd,
              "head_loss": sum(2 * B * H * h for h in heads) * n_upd}
        for f, v in fl.items():
            table[f]["algorithmic_tflop"] = v / 1e12
            table[f]["tflops"] = v / 1e12 / (table[f]["ms_total"] * 1e-3) if table[f]["ms_total"] > 0 else None
        # the same launches against the HBM roofline: every [B, 512] fp32 activation (168 MB at c5) is larger than L2, so each GEMM
        # streams its operands from and its result to HBM once (DESIGN.md 3b: algorithmic bytes per row)
        Hx, pad = H + 64, lambda k: (k + 1 + 63) // 64 * 64
        by = {"fwd_gemm": sum(4 * B * (pad(i) + Hx + L * (H + Hx)) for i in ins) * n_upd,
              "bwd_gemm": sum(4 * B * (32 + 2 * H + L * 3 * H) for _ in ins) * n_upd,
              "grad_gemm": sum(4 * B * ((H + pad(i)) + L * (H + Hx) + (Hx + 32)) for i in ins) * n_upd,
              "head_loss": sum(4 * B * (H + 32) for _ in ins) * n_upd}
        hbm_peak = float(peaks.get("hbm_gbs", 6580.0))
        for f, v in by.items():
            table[f]["algorithmic_gbyte"] = v / 1e9
            table[f]["hbm_gbs"] = v / 1e9 / (table[f]["ms_total"] * 1e-3) if table[f]["ms_total"] > 0 else None
            table[f]["hbm_frac"] = table[f]["hbm_gbs"] / hbm_peak if table[f]["hbm_gbs"] else None
        dom = max(("fwd_gemm", "bwd_gemm", "grad_gemm"), key=lambda f: table[f]["ms_total"])
        d = table[dom]
        avg_ms = d["ms_total"] / max(d["launches"], 1)
        ach = d["tflops"]
        kern = {"fwd_gemm": "big_lin_kernel<EpiFwd>", "bwd_gemm": "big_lin_kernel<EpiBwd>", "grad_gemm": "big_grad_kernel"}[dom]
        peak = tf32_peak if a.gemm == "tf32" else float(peaks.get("bf16_tflops", 1590.0))
        pipeline_ms = sum(table[f]["ms_total"] for f in fam)
        out = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak if ach else None,
               "kernel": f"{kern} (TMA-fed tcgen05 kind::tf32 GEMM, {dom})" if a.gemm == "tf32" else f"{dom} (fp32 FFMA build)",
               "peak_source": "torch.matmul TF32 8192^3 measured beside this run (cuBLAS, best of 5); "
                              f"MEASURED_PEAKS.json bf16_tflops = {peaks.get('bf16_tflops')}" if a.gemm == "tf32" else "MEASURED_PEAKS.json bf16_tflops",
               "avg_launch_ms": avg_ms, "launches_timed": d["launches"],
               "algorithmic_gflop_per_launch": d["algorithmic_tflop"] * 1e3 / max(d["launches"], 1),
               "kernel_share_of_step": d["ms_total"] / res["ms_per_step"],
               "hbm": {"achieved": d.get("hbm_gbs"), "peak": hbm_peak, "unit": "GB/s", "frac": d.get("hbm_frac"),
                       "note": "same launches against the HBM roofline (algorithmic operand + result bytes, MEASURED_PEAKS hbm_gbs): the "
                               "GEMMs of this pipeline sit between both roofs"},
               "pipeline_families": table, "update_pipeline_ms_per_step": pipeline_ms,
               "update_pipeline_tflops": (fa + fc) * n_upd / 1e12 / (pipeline_ms * 1e-3) if pipeline_ms > 0 else None}
    elif cfg.recurrent and a.gemm == "tf32":
        # tcgen05 GRU pipeline: the library times every kernel family with CUDA events on the launching stream (one eager train());
        # the sequence kernels stream 64-float rows per position per plane: the honest bound of the dominant ones is HBM
        lib.mappo_debug_gru_timing(1, None, None)
        j = jobs[0]
        saved_graph, saved_overlap = j.eng.graph, j.trainer.overlap_nets
        j.eng.graph, j.trainer.overlap_nets = None, False
        try:
            res["flush"].zero_()
            j.eng.step_resident()
            torch.cuda.synchronize()
        finally:
            j.eng.graph, j.trainer.overlap_nets = saved_graph, saved_overlap
        ms = (C.c_double * 8)()
        cnt = (C.c_int64 * 8)()
        lib.mappo_debug_gru_timing(0, ms, cnt)
        cyc = (C.c_int64 * 16)()
        lib.mappo_debug_gru_cycles(cyc)
        fam = ["pack", "base_fwd", "seq_fwd", "heads_loss", "bptt", "gate_grad", "base_bwd", "reduce_unfold"]
        table = {f: {"ms_total": ms[i], "launches": int(cnt[i])} for i, f in enumerate(fam)}
        P = cfg.episode_length * cfg.n_rollout_threads * cfg.num_agents // cfg.data_chunk_length * cfg.data_chunk_length \
            if cfg.use_recurrent_policy else cfg.episode_length * cfg.n_rollout_threads * cfg.num_agents
        H = cfg.hidden_size
        plane = 4 * P * H                                      # bytes of one [position][64] fp32 workspace plane
        ins = (cfg.obs_dim, cfg.share_obs_dim)
        heads = (sum(cfg.act_dims), 1)
        n_upd = cfg.ppo_epoch * cfg.num_mini_batch             # per net kind; the table sums actor + critic launches
        # algorithmic bytes per optimiser step, actor + critic (DESIGN.md 3c: planes read + written by each kernel, gathered rows once)
        by = {"base_fwd": sum(4 * P * i for i in ins) + 2 * plane, "seq_fwd": 2 * 6 * plane, "heads_loss": 2 * 2 * plane,
              "bptt": 2 * 9 * plane, "gate_grad": 2 * 7 * plane, "base_bwd": sum(4 * P * i for i in ins) + 2 * plane}
        fl = {"base_fwd": sum(2 * P * (i * H + H * H) for i in ins), "seq_fwd": 2 * 2 * P * 6 * H * H,
              "heads_loss": sum(3 * 2 * P * H * h for h in heads), "bptt": 2 * 2 * P * 3 * H * H,
              "gate_grad": 2 * 2 * P * (3 * H * H + 6 * H * H), "base_bwd": sum(2 * P * (3 * H * H + 2 * i * H) for i in ins)}
        hbm_peak = float(peaks.get("hbm_gbs", 6580.0))
        for f in by:
            t = table[f]["ms_total"] * 1e-3
            table[f]["algorithmic_gbyte"] = by[f] * n_upd / 1e9
            table[f]["hbm_gbs"] = by[f] * n_upd / 1e9 / t if t > 0 else None
            table[f]["hbm_frac"] = table[f]["hbm_gbs"] / hbm_peak if t > 0 else None
            table[f]["tflops"] = fl[f] * n_upd / 1e12 / t if t > 0 else None
        dom = max(by, key=lambda f: table[f]["ms_total"])
        d = table[dom]
        kern = {"base_fwd": "update_mlp_tc_kernel<TC_BASE_FWD>", "seq_fwd": "gru_tc_fwd_kernel", "heads_loss": "update_mlp_tc_kernel<TC_HEAD>",
                "bptt": "gru_tc_bwd_kernel", "gate_grad": "gru_tc_grad_kernel", "base_bwd": "update_mlp_tc_kernel<TC_BASE_BWD>"}[dom]
        pipeline_ms = sum(table[f]["ms_total"] for f in fam)
        avg_ms = d["ms_total"] / max(d["launches"], 1)
        out = {"bound": "hbm", "achieved": d["hbm_gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": d["hbm_frac"],
               "kernel": f"{kern} ({dom}: the slowest kernel family of the tcgen05 GRU pipeline, update_gru_tc.cu)",
               "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6580 GB/s (B200_PROFILING.md)",
               "avg_launch_ms": avg_ms, "launches_timed": d["launches"],
               "algorithmic_mbyte_per_launch": d["algorithmic_gbyte"] * 1e3 / max(d["launches"], 1),
               "kernel_share_of_step": d["ms_total"] / res["ms_per_step"],
               "tensor": {"achieved": (fa + fc) * n_upd / 1e12 / (pipeline_ms * 1e-3) if pipeline_ms > 0 else None, "peak": tf32_peak,
                          "unit": "TFLOP/s", "note": "whole pipeline (algorithmic GEMM FLOPs of one optimiser step / summed kernel time) "
                                                      "against cuBLAS tf32 measured beside the run: the GEMMs are 64 wide, the planes set the pace"},
               "pipeline_families": table, "update_pipeline_ms_per_step": pipeline_ms,
               "seq_step_cycles": {"fwd": {nm: int(cyc[i + 1] - cyc[i]) for i, nm in enumerate(
                                       ["wait_state_mma", "cell_math_stores", "operand_tiles", "barrier", "mma_issue", "prefetch_issue"])},
                                   "bwd": {nm: int(cyc[9 + i] - cyc[8 + i]) for i, nm in enumerate(
                                       ["loads_gate_math_stores", "operand_tile", "barrier", "mma_issue", "mma_wait", "dh_update"])}}}
    else:
        orig = lib.mappo_update_fwd_bwd
        pairs = []

        class TimedCall:
            def __call__(self, *args):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                rc = orig(*args)
                e.record()
                pairs.append((s, e))
                return rc

        j = jobs[0]
        saved_graph, saved_overlap = j.eng.graph, j.trainer.overlap_nets
        j.eng.graph, j.trainer.overlap_nets = None, False    # one launch at a time: the events see this kernel alone
        try:
            lib.mappo_update_fwd_bwd = TimedCall()
            res["flush"].zero_()
            j.eng.step_resident()
            torch.cuda.synchronize()
        finally:
            lib.mappo_update_fwd_bwd = orig
            j.eng.graph, j.trainer.overlap_nets = saved_graph, saved_overlap
        msl = [s.elapsed_time(e) for s, e in pairs]
        avg_ms = sum(msl) / max(len(msl), 1)
        tc = a.gemm == "tf32"
        peak = tf32_peak if tc else float(peaks.get("bf16_tflops", 1590.0))
        ach = (fa + fc) / 2 / (avg_ms * 1e-3) / 1e12
        kname = ("tcgen05 GRU pipeline (update_gru_tc.cu: base fwd -> sequence fwd -> heads + loss -> BPTT -> gate gradients -> base bwd, "
                 "kind::tf32 + TMEM; the timed call includes weight packing, slot sums and unfold)" if (tc and cfg.recurrent) else
                 "update_mlp_tc_kernel (fused fwd+loss+bwd, tcgen05 kind::tf32 + TMEM; launch incl. its weight-pack kernel)" if tc else
                 ("gru_seq_fwd/bwd kernels (4-launch fused GRU fwd+loss+BPTT pipeline, fp32 FFMA)" if cfg.recurrent else
                  "update_mlp_kernel (fused fwd+loss+bwd, fp32 FFMA tiles)"))
        out = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "kernel": kname,
               "peak_source": ("torch.matmul TF32 8192^3 measured beside this run (cuBLAS, best of 5); "
                               f"MEASURED_PEAKS.json bf16_tflops = {peaks.get('bf16_tflops')}") if tc else
                              "MEASURED_PEAKS.json bf16_tflops (burst): the GEMM FLOPs run on fp32 FFMA here",
               "avg_launch_ms": avg_ms, "launches_timed": len(msl), "algorithmic_gflop_per_launch": (fa + fc) / 2 / 1e9,
               # actor and critic chains run concurrently (two graph branches): share of the critical path = one chain
               "kernel_share_of_step": avg_ms * cfg.ppo_epoch * cfg.num_mini_batch / res["ms_per_step"],
               "kernel_time_sum_over_step": avg_ms * 2 * cfg.ppo_epoch * cfg.num_mini_batch / res["ms_per_step"]}
    return out


def result_line(name, res, a, world, roof, cpu, clocks, extra_cfg):
    cfg, w, jobs = res["cfg"], res["workload"], res["jobs"]
    eng = jobs[0].eng
    tr = jobs[0].trainer
    tc = a.gemm == "tf32"
    line = {"metric": metric_name(name), "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": a.steps,
            "warmup": max(a.warmup, 3), "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": w["scaling"],
            "vs_baseline": None,
            "dtype": "tf32 tensor-core GEMMs (fp32 accumulate / fp32 elsewhere)" if tc else "f32",
            "data": "synthetic",
            "config": {**workload_dict(w, world), "cuda_graph": res["graph_ok"], "gemm": a.gemm,
                       "collective": ("none (1 GPU)" if world == 1 else
                                      "one-shot peer-memory all-reduce kernel over NVLink, in-graph"
                                      if getattr(tr, "_p2p", None) is not None else
                                      "NCCL all-reduce via torch.distributed between graph segments"),
                       "rng": "device (Philox sampling, Feistel permutations)",
                       "rollout": ("persistent kernel, one launch per iteration" if (eng.persistent_rollout or eng.closed_persistent)
                                   else ("layer-by-layer GEMM pipeline per env step" if eng.big else "one launch per env step")),
                       "env": ("device-side simple_spread, closed loop " + ("inside one persistent rollout kernel" if eng.closed_persistent
                               else "(policy_step -> env step -> insert per step)")) if a.env == "device" else "synthetic staged env outputs",
                       "h2d": "obs, rewards, dones (share_obs = concat of the thread's agents' obs is formed on the device)"
                              if eng.share_from_obs else "obs, share_obs, rewards, dones (+ active / avail masks)",
                       **extra_cfg},
            "timing": {"timed_steps": a.steps, "step_ms": res["step_ms"], "e2e_timed_steps": a.steps,
                       "wall_s_timed_region": res["wall_s_timed_region"]},
            "e2e": {"value": res["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": res["h2d"], "d2h_bytes_per_step": res["d2h"],
                    "ms_per_step": res["e2e_ms_per_step"],
                    "input_staging": "double buffered: the H2D of step i + 1 overlaps the graph of step i" if res.get("prefetch") else "synchronous"},
            "gpu_launches": res["launches"], "roofline": roof, "clocks": clocks, "train_info_last": res["info"]}
    if cpu is not None:
        line["cpu_baseline"] = cpu
    return line


def run_gpu(a):
    if os.environ.get("BENCH_WATCHDOG"):
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["BENCH_WATCHDOG"]), exit=True)
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.gpus > 1 and world != a.gpus:
        raise SystemExit(f"--gpus {a.gpus} needs torchrun with {a.gpus} ranks (WORLD_SIZE={world})")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    peaks = {}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    try:
        tf32_peak = measure_tf32_peak(dev)
    except Exception as e:                                 # never lose the headline to a side measurement
        print(f"[bench] tf32 peak measurement failed ({type(e).__name__}: {e}); using bf16 / 2", file=sys.stderr)
        tf32_peak = float(peaks.get("bf16_tflops", 1590.0)) / 2

    sampler = ClockSampler(local)
    res = run_config(a.config, a, world, rank, dev, dist, sampler)
    if a.dump_outputs:
        dump_outputs(res["workload"], a, rank, dev, a.dump_outputs)
    cfg = res["cfg"]
    eng0 = res["jobs"][0].eng

    # replicas must stay bit-identical: checksum of every parameter vector over ranks (min == max)
    extra_cfg = {}
    if world > 1:
        for j in res["jobs"]:
            j.trainer.check_collectives()                  # no peer-memory all-reduce timed out
        ck = torch.stack([torch.stack([j.policy.actor.flat.double().sum(), j.policy.critic.flat.double().sum(),
                                       (j.policy.actor.flat.double() ** 2).sum(), (j.policy.critic.flat.double() ** 2).sum()])
                          for j in res["jobs"]]).reshape(-1)
        lo, hi = ck.clone(), ck.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        same = bool(torch.equal(lo, hi))
        extra_cfg["replica_checksums_identical_across_ranks"] = same
        if not same:
            raise SystemExit(f"[bench] rank {rank}: parameter checksums differ across ranks after the timed loop: {lo.tolist()} vs {hi.tolist()}")

    breakdown = None
    if rank == 0 and a.breakdown and res["workload"]["n_policies"] == 1:
        try:
            breakdown = eng0.phase_breakdown()
        except Exception as e:
            print(f"[bench] phase breakdown failed ({type(e).__name__}: {e})", file=sys.stderr)
            breakdown = {"error": f"{type(e).__name__}: {e}"}
        if a.gemm == "tf32" and not eng0.big and not cfg.recurrent and "error" not in breakdown:
            import ctypes as C
            from mappo_b200 import _lib
            t = (C.c_int64 * 16)()
            torch.cuda.synchronize()
            _lib.load().mappo_debug_tc_timing(t)
            names = ["setup", "S1", "fc1_mma", "S3", "fc2_mma", "S5", "head_mma", "S7_loss", "dx2_Gh_mma", "S9", "dx1_G2_mma",
                     "S11", "dump_G2", "G1_wait", "tail"]
            breakdown["tc_tile_cycles_warm"] = {nm: int(t[i + 1] - t[i]) for i, nm in enumerate(names)}
            breakdown["tc_tile_cycles_warm"]["total"] = int(t[15] - t[0])
    roof = None
    if rank == 0:
        try:
            roof = kernel_roofline(res, a, peaks, tf32_peak)
        except Exception as e:
            print(f"[bench] roofline leg failed ({type(e).__name__}: {e})", file=sys.stderr)
            roof = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            key = ("big_lin_kernel" if eng0.big else ("update_mlp_tc_kernel" if a.gemm == "tf32" else "update_mlp_kernel"))
            if cfg.recurrent and a.gemm == "tf32" and "kernel" in roof:
                key = roof["kernel"].split(" ")[0] if a.config == "c4" else "-"      # per-kernel captures of the GRU pipeline at c4's size
            traffic = tj.get(key)
        roof["traffic"] = traffic
        roof["traffic_unit"] = "bytes/launch (ncu --set full, profiles/)"
        cpu = None
        if world == 1 and a.cpu_iters > 0:
            try:
                cpu, _ = cpu_baseline(a.config, min(a.cpu_iters, {"c2": 100, "c3": 10, "c4": 2, "c5": 3}[a.config]))
            except Exception as e:
                print(f"[bench] cpu_baseline leg failed ({type(e).__name__}: {e})", file=sys.stderr)
        line = result_line(a.config, res, a, world, roof, cpu, res["clocks"], extra_cfg)
        line["phase_breakdown_ms"] = breakdown
        line["tf32_peak_tflops_measured"] = tf32_peak
        # fp32-mode companion (same workload, exact-fp32 FFMA GEMMs) and the other BASELINE configs, compact
        if world == 1 and a.extras:
            del res
            torch.cuda.empty_cache()
            others = {}
            if a.gemm == "tf32" and a.config in ("c2", "c5"):
                try:
                    a2 = argparse.Namespace(**{**vars(a), "gemm": "fp32", "steps": max(3, a.steps // 4)})
                    r2 = run_config(a.config, a2, 1, 0, dev, dist, None)
                    line["value_fp32"] = {"value": r2["value"], "ms_per_step": r2["ms_per_step"], "e2e_value": r2["e2e_value"],
                                          "gemm": "fp32 (exact FFMA build of the same kernels)"}
                    del r2
                except Exception as e:
                    line["value_fp32"] = {"error": f"{type(e).__name__}: {e}"}
                torch.cuda.empty_cache()
            for other in (["c3", "c5"] if a.config == "c2" else []):
                try:
                    a3 = argparse.Namespace(**{**vars(a), "steps": 3 if other == "c5" else max(3, a.steps // 4), "env": "staged"})
                    r3 = run_config(other, a3, 1, 0, dev, dist, None)
                    rf = kernel_roofline(r3, a3, peaks, tf32_peak)
                    c3, _ = cpu_baseline(other, {"c3": 3, "c5": 2}[other]) if a.cpu_iters > 0 else (None, None)
                    ol = result_line(other, r3, a3, 1, rf, c3, None, {})
                    for k in ("clocks", "train_info_last", "vs_baseline", "higher_is_better", "data", "n_gpus"):
                        ol.pop(k, None)
                    others[other] = ol
                    del r3
                    torch.cuda.empty_cache()
                except Exception as e:                     # never lose the headline line to an extra
                    others[other] = {"error": f"{type(e).__name__}: {e}"}
            if others:
                line["other_configs"] = others
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed iterations (default 50; 5 for c4 and 10 for c5, ~0.1 - 0.5 s per iteration)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4", "c5"], help="BASELINE.json workload (default c2 = configs[1])")
    ap.add_argument("--gemm", default=os.environ.get("MAPPO_B200_GEMM", "tf32"), choices=["tf32", "fp32"],
                    help="GEMM engine of the update kernels (tf32 = tcgen05 tensor cores)")
    ap.add_argument("--no-prefetch", dest="no_prefetch", action="store_true", help="e2e: copy every step's inputs synchronously before its graph")
    ap.add_argument("--eager", action="store_true", help="no CUDA graph (for per-kernel profiling under ncu)")
    ap.add_argument("--env", default="staged", choices=["staged", "device"],
                    help="staged: synthetic env outputs uploaded per iteration (the BASELINE metric: the path only); "
                         "device: closed loop with the device-side simple_spread environment (c2 only)")
    ap.add_argument("--cpu-iters", type=int, default=100, help="oracle iterations for cpu_baseline (rank 0, N=1); 0 = skip")
    ap.add_argument("--no-extras", dest="extras", action="store_false", help="skip value_fp32 / other_configs")
    ap.add_argument("--no-breakdown", dest="breakdown", action="store_false")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after timing, write the outputs of one iteration from the seeded starting state as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps is None:
        a.steps = {"c4": 5, "c5": 10}.get(a.config, 50)
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_gpu(a)


if __name__ == "__main__":
    main()
