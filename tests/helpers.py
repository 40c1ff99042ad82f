"""Shared test helpers: golden fixture loading (tests/golden/*.npz, written by make_golden.py)."""
import ast
import os

import numpy as np
import torch

from oracle import mappo_oracle as O

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN_CASES = ["c1_mlp_discrete", "c3_gru_multidiscrete", "c4_gru_smac", "c5_mlp_switches", "naive_rnn_ptl",
                "c5_h512_hanabi", "c2_mlp_n128"]
# compact cases (make_golden.py `put`): initial weights = seed + checksums, big matrices = every 16th row + Frobenius norm
INFO_KEYS = ("value_loss", "policy_loss", "dist_entropy", "actor_grad_norm", "critic_grad_norm", "ratio")


class Golden:
    def __init__(self, name):
        self.name = name
        self.z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
        d = ast.literal_eval(str(self.z["cfg_json"]))
        d["act_dims"] = tuple(d["act_dims"])
        self.cfg = O.PathConfig(**d)
        self.iters = 1 + max(int(k[2:k.index("/")]) for k in self.z.files if k.startswith("it"))

    def init_params(self, which):
        """Initial state_dict of 'actor' / 'critic': stored in full, or (compact cases) regenerated from the seed with the
        engine's host-side initialiser, which draws exactly like the reference (test_host_logic.py pins that)."""
        if not self.has("init_seed"):
            return self.params(f"init/{which}/")
        if getattr(self, "_init", None) is None:
            from mappo_b200.core import reference_init_state_dict
            from argsutil import make_args
            cfg, seed = self.cfg, int(self.z["init_seed"])
            args = make_args(cfg)
            torch.set_num_threads(1)
            torch.manual_seed(seed)
            np.random.seed(seed)
            actor = reference_init_state_dict(args, cfg.obs_dim, list(cfg.act_dims), False, cfg.multi_discrete)
            critic = reference_init_state_dict(args, cfg.share_obs_dim, [1], True, False)
            self._init = dict(actor=actor, critic=critic)
            self.check_init("actor", actor)
            self.check_init("critic", critic)
        return self._init[which]

    def params(self, prefix):
        """{state_dict key: tensor} under e.g. 'init/actor/' or 'it0/critic/'."""
        return {k[len(prefix):]: torch.from_numpy(self.z[k].copy()) for k in self.z.files if k.startswith(prefix)}

    def feed(self, it):
        g = lambda n: self.z[f"it{it}/feed/{n}"].copy() if f"it{it}/feed/{n}" in self.z.files else None
        return O.SyntheticFeed(g("obs"), g("share_obs"), g("rewards"), g("dones"), g("active_masks"),
                               g("available_actions"))

    def get(self, key):
        return self.z[key]

    def cmp(self, key, value, rtol, atol, what=""):
        """assert_close against the stored tensor; compact matrices compare the stored rows and the Frobenius norm."""
        value = np.asarray(value)
        if key + "@rows" in self.z.files:
            idx = self.z[key + "@rows"]
            assert_close(value[idx], self.z[key], rtol, atol, what + " (every 16th row)")
            norm = float(np.sqrt((value.astype(np.float64) ** 2).sum()))
            assert_close(norm, float(self.z[key + "@norm"]), rtol, atol, what + " (Frobenius norm)")
        else:
            assert_close(value, self.z[key], rtol, atol, what)

    def check_init(self, net_name, state_dict):
        """compact cases: the nets were initialised from `init_seed`; compare with the reference's checksums."""
        for k, v in state_dict.items():
            a = v.detach().cpu().numpy().astype(np.float64)
            want = self.z[f"init_checksum/{net_name}/{k}"]
            assert_close(np.array([a.sum(), (a * a).sum()]), want, 1e-5, 1e-6, f"init {net_name} {k}")

    def has(self, key):
        return key in self.z.files


def assert_close(a, b, rtol, atol, what=""):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    err = np.abs(a - b)
    tol = atol + rtol * np.abs(b)
    if not np.all(err <= tol):
        i = np.unravel_index(np.argmax(err - tol), err.shape)
        raise AssertionError(f"{what}: max violation at {i}: got {a[i]!r} want {b[i]!r} "
                             f"(|err|={err[i]:.3e}, tol={tol[i]:.3e}); max|err|={err.max():.3e}")


def grad_agreement(got, want, key, smooth, tf32, report=None, l2_tol=None):
    """Agreement of one gradient tensor with the reference, as (ok, relative L2 error).

    Smooth (tanh) nets: every element within a |ref| + b max|ref| (fp32 build a 2e-3, b 1e-4; tcgen05 / tf32 build a = b = 5e-3;
    LayerNorm affine parameters b x 10-20: in the hidden >= 128 pipeline they are contractions of the folded weight gradients with
    the weights -- sums of H signed terms that largely cancel -- so they carry the weight gradients' absolute error at a smaller scale).

    ReLU nets: a unit whose pre-activation is within rounding distance of zero is on for one implementation and off for the other (the
    reference's own CPU and GPU runs differ the same way).  One such flip changes that unit's row of dW by its whole contribution of
    one sample, i.e. ~1/sqrt(active rows) of the row's scale -- 2-9 % here -- so the element-wise maximum is not a usable metric.
    Measured on the B200 (scripts/diag_big.py): every stored intermediate of the pipeline agrees with float64 algebra on ITS OWN inputs
    to 1e-6 (fp32 build) / 3e-4 (tf32), the flips are the entire difference.  Criterion: relative L2 error of the tensor
    (fp32 build 2e-2, tf32 5e-2; the callers add a bound on the whole gradient's L2 error and its cosine); the fraction of
    elements outside the smooth-net tolerance is reported."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    scale = np.abs(want).max() + 1e-300
    err = np.abs(got - want)
    ln = "feature_norm" in key or ".2." in key or "norm" in key
    if tf32:
        tol = 5e-3 * np.abs(want) + (5e-2 if ln else 5e-3) * scale
    else:
        tol = 2e-3 * np.abs(want) + (2e-3 if ln else 1e-4) * scale
    l2 = float(np.linalg.norm(got - want) / (np.linalg.norm(want) + 1e-300))
    outside = float((err > tol).mean())
    if smooth:
        ok = outside == 0.0
    else:
        ok = l2 <= (l2_tol if l2_tol is not None else (5e-2 if tf32 else 2e-2))
    if report is not None:
        report.append(f"{key}: max err / scale {err.max() / scale:.3e}, rel L2 {l2:.3e}, outside element tolerance {100 * outside:.2f} %"
                      + ("" if ok else "  <-- FAIL"))
    return ok, l2


def rollout_image_floats(in_dim, layer_n, use_fn, recurrent, head_total, hidden=64):
    """(warp-per-row image, 32-row tile image) sizes in floats of a hidden-64 net's rollout weights: the layouts of
    csrc/rollout_mlp.cuh make_fast_img (+ rollout_gru.cuh make_gru_fast_img) and csrc/common.cuh make_smem_w."""
    H = hidden
    k1 = (in_dim + 3) & ~3
    ap = (head_total + 3) & ~3
    fast = (2 * k1 if use_fn else 0) + k1 * H + 3 * H + layer_n * (H * H + 3 * H) + H * ap + ap
    if recurrent:
        fast += 2 * 3 * H * H + 2 * 3 * H + 2 * H
    ld1, ldh = in_dim | 1, H | 1
    tile = (2 * in_dim if use_fn else 0) + H * ld1 + 3 * H + layer_n * (H * ldh + 3 * H)
    if recurrent:
        tile += 2 * 3 * H * ldh + 2 * 3 * H + 2 * H
    tile += head_total * ldh + head_total
    return fast, (tile + 3) & ~3
