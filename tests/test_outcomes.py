"""Episode outcomes without a GPU: the fold restatements on hand-computed sequences, argument checks of the new C-ABI entries, the
SASS of the outcome kernels and folds, and the config defaults."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from tests import rl_games_outcome_oracle as oo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "bez_isaacgym_b200", "libbezk.so")
HEADER = os.path.join(ROOT, "include", "bezk.h")
NEW = ("bezk_outcome_classes", "bezk_post_physics_rollout_ep_outcome", "bezk_outcome_meter_update", "bezk_player_outcome_update")


# ------------------------------------------------------------------ fold restatements
def _random_partials(steps, k, w, seed, p_empty=0.2):
    rng = np.random.default_rng(seed)
    p = rng.integers(0, 4, size=(steps, k, w)).astype(np.int32)
    p[rng.random(steps) < p_empty] = 0                      # steps with no done env
    return p


def test_meter_recurrence_by_hand():
    p = np.zeros((3, 5, 2), np.int32)
    p[0, 3, 0] = 1                                            # one game, scored
    p[2, 0, 1], p[2, 4, 0] = 2, 1                             # (step 1 empty) 2 fell, 1 timeout
    mean, size = oo.meter(p, games_to_track=100)
    assert size == 4
    assert np.allclose(mean, [0.5, 0, 0, 0.25, 0.25]) and abs(mean.sum() - 1) < 1e-6
    mean, size = oo.meter(p, games_to_track=2)                # the window keeps the last step's 2 games only
    assert size == 2 and np.allclose(mean, [2 / 3, 0, 0, 0, 1 / 3])


def test_meter_chunking_invariance_and_size():
    p = _random_partials(40, 4, 7, 1)
    whole, size = oo.meter(p, 50)
    mean, sz = None, 0
    for t0 in range(0, 40, 7):
        mean, sz = oo.meter(p[t0:t0 + 7], 50, mean, sz)
    assert mean.tobytes() == whole.tobytes() and sz == size == 50


def test_player_fold_cutoff_mid_step_and_empty_steps():
    p = np.zeros((5, 5, 2), np.int32)
    p[0, 0, 0] = 1
    p[2, 3, 0], p[2, 4, 1], p[2, 1, 1] = 2, 1, 1              # step 2 crosses 3 games and is added whole
    p[3, 2, 0] = 7                                            # after the cutoff: nothing
    counts, per = oo.player_fold(p, games_num=3)
    assert counts.tolist() == [5.0, 1.0, 1.0, 0.0, 2.0, 1.0]
    assert per[:, :].sum(axis=1).tolist() == [1, 0, 4, 0, 0]


def test_player_fold_chunking_invariance():
    p = _random_partials(40, 5, 9, 2)
    whole, per = oo.player_fold(p, 333)
    assert whole[0] >= 333 and per[-1].sum() == 0
    for k in (1, 7, 32):
        counts, rows = None, []
        for t0 in range(0, 40, k):
            counts, ps = oo.player_fold(p[t0:t0 + k], 333, counts)
            rows.append(ps)
        assert counts.tobytes() == whole.tobytes() and np.concatenate(rows).tobytes() == per.tobytes()


# ------------------------------------------------------------------ C ABI
def _lib():
    from bez_isaacgym_b200 import _lib as L
    if not os.path.exists(L.LIB_PATH):
        pytest.skip("libbezk.so not built")
    return L, L.load()


def test_new_symbols_are_exported_and_match_the_header():
    L, lib = _lib()
    for name in NEW:
        assert name in L.SIGNATURES and getattr(lib, name) is not None
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    for name in NEW:
        m = re.search(r"\b" + name + r"\(([^)]*)\)", text)
        assert m, name
        params = [a for a in m.group(1).split(",") if a.strip() and a.strip() != "void"]
        assert len(params) == len(L.SIGNATURES[name][1]), name
        for a, t in zip(params, L.SIGNATURES[name][1]):
            a = a.strip()
            if "*" in a:
                assert t in (C.c_void_p,) or hasattr(t, "_type_"), (name, a)
            elif a.startswith(("int64_t", "uint64_t")):
                assert t in (C.c_int64, C.c_uint64), (name, a)
            elif a.startswith("float"):
                assert t is C.c_float, (name, a)
            else:
                assert t in (C.c_int, C.c_int32), (name, a)


def test_outcome_classes():
    _, lib = _lib()
    assert [lib.bezk_outcome_classes(t) for t in (0, 1, 2)] == [5, 4, 4]
    assert lib.bezk_outcome_classes(3) == 10001 and lib.bezk_outcome_classes(-1) == 10001
    from bez_isaacgym_b200.tasks import KickEnv, OrientEnv, WalkEnv
    assert KickEnv.OUTCOMES == ("fell", "strayed", "wide", "scored", "timeout")
    assert WalkEnv.OUTCOMES == OrientEnv.OUTCOMES == ("fell", "reached", "out", "timeout")


def _outcome_args(L, ep, outcome, task=0, norm=(None, None, None)):
    cfg = L.BezkTaskCfg()
    p = C.c_void_p(64)                                        # never dereferenced: the checks come first
    return [task] + [p] * 11 + [0, 0] + [p] * 4 + [C.byref(cfg), p, None, p, None, None, None, None, 0, 1024] + ep + \
        list(norm[:2]) + [1e-5, norm[2], outcome, None]


def test_outcome_entry_checks_come_before_device_access():
    L, lib = _lib()
    p = C.c_void_p(64)
    assert lib.bezk_post_physics_rollout_ep_outcome(*_outcome_args(L, [p, p, p], None)) == 10001
    assert b"outcome_partials NULL" in lib.bezk_last_error()
    for ep in ([None, None, None], [p, None, p], [p, p, None]):
        assert lib.bezk_post_physics_rollout_ep_outcome(*_outcome_args(L, ep, p)) == 10001
        assert b"episode accumulators" in lib.bezk_last_error()
    assert lib.bezk_post_physics_rollout_ep_outcome(*_outcome_args(L, [p, p, p], p, task=7)) == 10001
    assert b"unknown task" in lib.bezk_last_error()
    assert lib.bezk_post_physics_rollout_ep_outcome(*_outcome_args(L, [p, p, p], C.c_void_p(66))) == 10002
    assert b"outcome_partials must be 4-byte aligned" in lib.bezk_last_error()
    # the episode / normaliser checks of bezk_post_physics_rollout_ep_norm follow, with their codes
    assert lib.bezk_post_physics_rollout_ep_outcome(*_outcome_args(L, [p, p, C.c_void_p(68)], p)) == 10002
    assert lib.bezk_post_physics_rollout_ep_outcome(*_outcome_args(L, [p, p, p], p, norm=(p, None, p))) == 10001
    assert b"obs_mean, obs_var and obs_norm" in lib.bezk_last_error()


def test_fold_entries_check_their_arguments():
    _, lib = _lib()
    p = C.c_void_p(64)
    for fn, arg in ((lib.bezk_outcome_meter_update, "games_to_track"), (lib.bezk_player_outcome_update, "games_num")):
        assert fn(p, 2, 10, 0, 0, p, p, None) == 10001
        assert arg.encode() in lib.bezk_last_error()
        assert fn(p, 2, 10, 3, 5, p, p, None) == 10001
        assert b"unknown task" in lib.bezk_last_error()
        assert fn(p, -1, 10, 0, 5, p, p, None) == 10001
        assert fn(None, 2, 10, 0, 5, p, p, None) == 10001
        assert fn(p, 2, 10, 0, 5, None, p, None) == 10001
        assert fn(C.c_void_p(66), 2, 10, 0, 5, p, p, None) == 10002
        assert fn(None, 0, 10, 0, 5, None, None, None) == 0                  # empty input: no-op
        assert fn(None, 3, 0, 1, 5, None, None, None) == 0
    assert lib.bezk_outcome_meter_update(p, 2, 10, 0, 5, C.c_void_p(66), p, None) == 10002
    assert lib.bezk_outcome_meter_update(p, 2, 10, 0, 5, p, C.c_void_p(68), None) == 10002
    assert lib.bezk_player_outcome_update(p, 2, 10, 0, 5, C.c_void_p(68), None, None) == 10002
    assert lib.bezk_player_outcome_update(p, 2, 10, 0, 5, p, C.c_void_p(68), None) == 10002


def test_ops_wrappers_refuse_cpu_tensors():
    import torch
    from bez_isaacgym_b200 import ops
    from bez_isaacgym_b200._lib import BezkError
    _lib()
    w = 1
    with pytest.raises(BezkError, match="CUDA"):
        ops.outcome_meter_update(torch.zeros(2, 5, w, dtype=torch.int32), 32, "kick", 100, torch.zeros(5), torch.zeros(1, dtype=torch.long))
    with pytest.raises(BezkError, match="CUDA"):
        ops.player_outcome_update(torch.zeros(2, 4, w, dtype=torch.int32), 32, "walk", 100, torch.zeros(5, dtype=torch.float64))
    with pytest.raises(BezkError, match="CUDA"):
        ops.post_physics_rollout_ep_outcome("kick", None, None, None, None, None, None, None, torch.zeros(32, dtype=torch.long), None,
                                            ops.make_task_cfg(), None, None, torch.zeros(32), torch.zeros(32),
                                            torch.zeros(3, 1, dtype=torch.float64), torch.zeros(5, 1, dtype=torch.int32))


# ------------------------------------------------------------------ SASS
@pytest.fixture(scope="module")
def sass():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(LIB) or not os.path.exists(exe):
        pytest.skip("needs cuobjdump and a built libbezk.so")
    funcs, name = {}, None
    for line in subprocess.check_output([exe, "-sass", LIB], text=True).splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
        elif name is not None:
            funcs[name].append(line)
    return {k: "\n".join(v) for k, v in funcs.items()}


def test_outcome_kernels_keep_the_memory_path_of_their_base_kernel(sass):
    """24 kernels: outcome (EP base) and obsnorm_outcome (obsnorm base), plain and L2, three tasks, with and without cleats.  Each
    has its base kernel's bulk copies, gathers and loads, no CTA-wide barrier and no local memory; the only extra global stores
    are the outcome counts."""
    found = 0
    for task in ("Li0E", "Li1E", "Li2E"):
        for cleats in ("Lb0E", "Lb1E"):
            for new, base in (("task_tile_outcome_kernel", "task_tile_ep_kernel"), ("task_tile_outcome_l2_kernel", "task_tile_ep_l2_kernel"),
                              ("task_tile_obsnorm_outcome_kernel", "task_tile_obsnorm_kernel"),
                              ("task_tile_obsnorm_outcome_l2_kernel", "task_tile_obsnorm_l2_kernel")):
                tag = f"I{cleats}Li128E{task}"
                n = [k for k in sass if re.search(r"\d" + new + tag, k)]
                b = [k for k in sass if re.search(r"\d" + base + tag, k)]
                assert len(n) == 1 and len(b) == 1, (new, tag, n, b)
                body, ref = sass[n[0]], sass[b[0]]
                assert body.count("STL") <= ref.count("STL") and body.count("LDL") <= ref.count("LDL"), "no extra local memory"
                assert "BAR.SYNC" not in body, "no CTA-wide barrier"
                for op in ("UBLKCP.S.G", "UBLKCP.G.S", "LTC64B", "LTC128B", "LDG"):
                    assert body.count(op) == ref.count(op), (n[0], op)
                assert body.count("VOTE.ANY") > ref.count("VOTE.ANY"), "the class ballots"
                assert ref.count("STG") < body.count("STG") <= ref.count("STG") + 2, "the count stores"
                assert body.count("ATOM") == ref.count("ATOM") and body.count("RED.") == ref.count("RED."), "no atomics"
                found += 1
    assert found == 24


def test_fold_kernels_have_no_barrier_and_no_local_memory(sass):
    for name in ("outcome_meter_kernel", "player_outcome_kernel"):
        ks = [k for k in sass if name in k]
        assert len(ks) == 1, ks
        body = sass[ks[0]]
        assert "BAR.SYNC" not in body and "STL" not in body and "LDL" not in body


# ------------------------------------------------------------------ config
def test_config_defaults_and_the_existing_dicts():
    from bez_isaacgym_b200.learner import agent
    from bez_isaacgym_b200.utils import config
    assert agent.OUTCOME_DEFAULTS == dict(track_outcomes=False)
    assert "track_outcomes" not in agent.DEFAULT_CONFIG and "track_outcomes" not in agent.TRAIN_DEFAULTS
    assert "track_outcomes" not in config.AGENT_KEYS and "track_outcomes" not in config.TRAIN_LOOP_KEYS
    assert tuple(agent.TRAIN_DEFAULTS) == config.TRAIN_LOOP_KEYS
    assert config.train_loop_config({"params": {"config": dict(track_outcomes=True, max_epochs=3)}}) == dict(max_epochs=3)


def test_outcome_meter_refuses_unknown_class_lists():
    from bez_isaacgym_b200.learner import OutcomeMeter
    with pytest.raises(ValueError):
        OutcomeMeter(("a", "b"), 10, "cpu")
    with pytest.raises(ValueError):
        OutcomeMeter(("fell", "strayed", "wide", "scored", "timeout"), 0, "cpu")
    with pytest.raises(ValueError):
        OutcomeMeter(("a", "b", "c", "d"), 10, "cpu")            # four classes, but not an env's
    assert OutcomeMeter(("fell", "strayed", "wide", "scored", "timeout"), 10, "cpu").task == "kick"
    m = OutcomeMeter(("fell", "reached", "out", "timeout"), 10, "cpu")
    assert m.task == "walk"
    assert m.current_size == 0 and m.as_dict() == dict(fell=0.0, reached=0.0, out=0.0, timeout=0.0)
