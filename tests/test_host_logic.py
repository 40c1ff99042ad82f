"""CPU-side tests: C-ABI exports, parameter layout, reference-identical initialisation, index arithmetic."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from oracle import mappo_oracle as O
from helpers import Golden, GOLDEN_CASES
from argsutil import make_args, make_spaces

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from mappo_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "mappo_b200.h")).read()
    declared = set(re.findall(r"\b(mappo_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"mappo_status"}
    lib = C.CDLL(_lib.lib_path())
    missing = [n for n in sorted(declared) if not hasattr(lib, n)]
    assert not missing, f"declared in mappo_b200.h but not exported: {missing}"
    assert declared == set(_lib.EXPORTS), (declared ^ set(_lib.EXPORTS))
    assert _lib.load().mappo_abi_version() == 5


def test_binding_arity_and_scalar_types_match_the_header():
    """ctypes does not check prototypes: every binding in mappo_b200/_lib.py must take exactly the parameters the header
    declares, with pointers, 32 / 64-bit integers and floats in the same positions."""
    from mappo_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "mappo_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", " ", hdr, flags=re.S)
    protos = dict(re.findall(r"\b(mappo_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", hdr, flags=re.S))
    kinds = {C.c_int32: "i32", C.c_int64: "i64", C.c_uint64: "i64", C.c_float: "f32", C.c_double: "f64"}

    def header_kind(param):
        param = " ".join(param.split())
        if "*" in param:
            return "ptr"
        for key, k in (("uint64_t", "i64"), ("int64_t", "i64"), ("int32_t", "i32"), ("float", "f32"), ("double", "f64")):
            if re.search(r"\b" + key + r"\b", param):
                return k
        raise AssertionError(f"unrecognised parameter type: {param!r}")

    def binding_kind(t):
        if t in kinds:
            return kinds[t]
        return "ptr"                                         # c_void_p, POINTER(...), arrays of pointers

    for name, (_, argtypes) in _lib._SIGS.items():
        assert name in protos, name
        params = [x for x in protos[name].split(",") if x.strip() and x.strip() != "void"]
        assert len(params) == len(argtypes), f"{name}: header has {len(params)} parameters, binding {len(argtypes)}"
        got = [binding_kind(t) for t in argtypes]
        want = [header_kind(x) for x in params]
        assert got == want, f"{name}: header {want} vs binding {got}"


def test_net_layout_matches_reference_param_count():
    from mappo_b200 import _lib
    lib = _lib.load()
    for name in GOLDEN_CASES:
        g = Golden(name)
        for which, in_dim, heads, crit in (("actor", g.cfg.obs_dim, list(g.cfg.act_dims), 0),
                                           ("critic", g.cfg.share_obs_dim, [1], 1)):
            d = _lib.NetDesc()
            d.in_dim, d.hidden, d.layer_n = in_dim, g.cfg.hidden_size, g.cfg.layer_N
            d.use_feature_norm, d.use_relu, d.recurrent = 1, int(g.cfg.use_ReLU), int(g.cfg.recurrent)
            d.n_heads = len(heads)
            for k, a in enumerate(heads):
                d.head_dim[k] = a
            d.is_critic = crit
            lay = _lib.NetLayout()
            assert lib.mappo_net_layout(C.byref(d), C.byref(lay)) == 0
            n_ref = sum(v.numel() for v in g.init_params(which).values())
            assert lay.total == n_ref, (name, which)


def test_tensor_core_build_selection_per_net_family():
    """MAPPO_GEMM_TF32 is built for hidden-64 MLP nets (layer_N 1, in_dim <= 63), hidden-64 GRU nets (same base) and the hidden
    >= 128 GEMM pipeline; the recurrent tcgen05 pipeline leaves the flat gradient in ONE slot and sizes its workspace (weight
    images, raw gradient slots, ten [position][64] planes in 128-position tiles) from the row count alone -- host-side queries, no
    GPU needed."""
    from mappo_b200 import _lib
    lib = _lib.load()

    def desc(in_dim, hidden, layer_n, recurrent, heads=(5,)):
        d = _lib.NetDesc()
        d.in_dim, d.hidden, d.layer_n = in_dim, hidden, layer_n
        d.use_feature_norm, d.use_relu, d.recurrent = 1, 0, recurrent
        d.n_heads = len(heads)
        for k, a in enumerate(heads):
            d.head_dim[k] = a
        d.is_critic = 0
        return d

    assert lib.mappo_tf32_supported(C.byref(desc(18, 64, 1, 0))) == 1
    assert lib.mappo_tf32_supported(C.byref(desc(21, 64, 1, 1, (5, 10)))) == 1          # c3: GRU, MultiDiscrete
    assert lib.mappo_tf32_supported(C.byref(desc(30, 64, 1, 1, (9,)))) == 1             # c4
    assert lib.mappo_tf32_supported(C.byref(desc(100, 64, 1, 1))) == 0                  # in_dim > 63: fp32 kernels only
    assert lib.mappo_tf32_supported(C.byref(desc(30, 64, 2, 1))) == 0                   # layer_N 2
    assert lib.mappo_tf32_supported(C.byref(desc(40, 512, 2, 0, (20,)))) == 1           # c5 widths: GEMM pipeline
    # rollout weight image of recurrent hidden-64 nets (rollout_gru.cuh): the feed-forward image + 2 x 3 gate matrices [k][lane][2] +
    # biases + rnn.norm; c3's actor: fn 2 x 24, fc1 24 x 64 + 3 x 64, fc2 64 x 64 + 3 x 64, heads 64 x 16 + 16 = 7104 floats
    assert lib.mappo_rollout_image_floats(C.byref(desc(21, 64, 1, 1, (5, 10)))) == 7104 + 2 * 3 * 64 * 64 + 2 * 192 + 2 * 64
    assert lib.mappo_rollout_image_floats(C.byref(desc(21, 64, 1, 0, (5, 10)))) == 7104
    gru = desc(30, 64, 1, 1, (9,))
    rows = 5120
    ws_fp32 = lib.mappo_update_workspace_floats(C.byref(gru), rows, _lib.GEMM_FP32)
    assert ws_fp32 == 8 * rows * 64
    # (the grid-dependent part of the tcgen05 workspace needs the device's SM count: only checked where a GPU is present)
    assert lib.mappo_update_slot_floats(C.byref(gru), _lib.GEMM_TF32) == lib.mappo_update_slot_floats(C.byref(gru), _lib.GEMM_FP32)


def test_bad_descriptor_is_rejected_with_message():
    from mappo_b200 import _lib
    lib = _lib.load()
    d = _lib.NetDesc()
    d.in_dim, d.hidden, d.layer_n, d.n_heads = 10, 64, 7, 1
    d.head_dim[0] = 3
    assert lib.mappo_net_layout(C.byref(d), C.byref(_lib.NetLayout())) == -3
    assert b"layer_N" in lib.mappo_last_error()


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_initialisation_is_seed_identical_to_reference(name):
    """torch.manual_seed(s) + the drop-in constructors' RNG consumption == the reference's initial weights."""
    from mappo_b200.core import reference_init_state_dict
    from tests_seeds import SEEDS
    g = Golden(name)
    args = make_args(g.cfg)
    torch.set_num_threads(1)          # train_mpe.py:96 (--n_training_threads 1); LAPACK QR is thread-count sensitive
    torch.manual_seed(SEEDS[name])
    np.random.seed(SEEDS[name])
    actor = reference_init_state_dict(args, g.cfg.obs_dim, list(g.cfg.act_dims), False, g.cfg.multi_discrete)
    critic = reference_init_state_dict(args, g.cfg.share_obs_dim, [1], True, False)
    if g.has("init_seed"):           # compact fixture: checksums of the reference's initial tensors
        g.check_init("actor", actor)
        g.check_init("critic", critic)
        return
    for k, v in g.params("init/actor/").items():
        assert torch.equal(actor[k], v), f"actor {k}"
    for k, v in g.params("init/critic/").items():
        assert torch.equal(critic[k], v), f"critic {k}"


def test_chunk_rows_oracle_straddles_like_reference():
    # T=25, L=10: chunk 2 = t 20..24 of lane 0 followed by t 0..4 of lane 1 (SURVEY App. B-3)
    T, N, M, L = 25, 2, 2, 10
    perm = np.arange(T * N * M // L)
    rows, first = O.chunk_minibatch_rows(perm, T, N, M, L, 1)[0]
    rows = rows.reshape(L, -1)
    E = N * M
    assert list(rows[:, 2]) == [t * E + 0 for t in range(20, 25)] + [t * E + 1 for t in range(0, 5)]
    assert first[2] == 20 * E


@pytest.mark.parametrize("recurrent", [0, 1])
def test_hidden64_dispatch_limits_at_widths_63_to_128(recurrent):
    """Which kernel family a hidden-64 net gets is decided by its input width: tf32 updates up to in_dim 63, the warp-per-row
    rollout image up to 64 and the 32-row tile image from 65 (csrc/rollout_mlp.cuh, rollout_gru.cuh, common.cuh)."""
    from mappo_b200 import _lib
    from helpers import rollout_image_floats
    lib = _lib.load()
    for in_dim in (63, 64, 65, 128):
        for layer_n, use_fn, heads in ((1, 1, (5,)), (2, 0, (5, 7)), (1, 1, (1,))):
            d = _lib.NetDesc()
            d.in_dim, d.hidden, d.layer_n, d.use_feature_norm, d.use_relu, d.recurrent = in_dim, 64, layer_n, use_fn, 1, recurrent
            d.n_heads = len(heads)
            for k, a in enumerate(heads):
                d.head_dim[k] = a
            d.is_critic = int(heads == (1,))
            want_tf32 = int(in_dim <= 63 and layer_n == 1)
            assert lib.mappo_tf32_supported(C.byref(d)) == want_tf32, (in_dim, layer_n)
            fast, tile = rollout_image_floats(in_dim, layer_n, use_fn, recurrent, sum(heads))
            assert fast != tile
            assert lib.mappo_rollout_image_floats(C.byref(d)) == (fast if in_dim <= 64 else tile), (in_dim, layer_n, heads)


def test_engine_takes_the_derived_share_obs_and_closed_loop_only_for_warp_per_row_nets():
    """mappo_rollout_persistent derives share_obs from obs, and mappo_rollout_closed_loop runs, only when both nets take the
    warp-per-row kernels; the engine mirrors that rule (a 4-agent simple_spread critic is 96 wide)."""
    from mappo_b200 import _lib
    from mappo_b200.engine import warp_per_row_rollout

    def desc(in_dim, hidden=64, heads=(5,)):
        d = _lib.NetDesc()
        d.in_dim, d.hidden, d.layer_n, d.n_heads = in_dim, hidden, 1, len(heads)
        for k, a in enumerate(heads):
            d.head_dim[k] = a
        return d

    assert warp_per_row_rollout(desc(18), desc(54, heads=(1,)))                   # 3-agent spread (c1 / c2)
    assert warp_per_row_rollout(desc(64), desc(64, heads=(1,)))
    assert not warp_per_row_rollout(desc(24), desc(96, heads=(1,)))               # 4-agent spread: the critic is 96 wide
    assert not warp_per_row_rollout(desc(65), desc(64, heads=(1,)))
    assert not warp_per_row_rollout(desc(18, hidden=128), desc(54, hidden=128, heads=(1,)))
    assert not warp_per_row_rollout(desc(18, heads=(20, 13)), desc(54, heads=(1,)))   # 33 head outputs
    assert warp_per_row_rollout(desc(18, heads=(20, 12)), desc(54, heads=(1,)))
