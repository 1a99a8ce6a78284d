"""Reward terms without a GPU: the numpy restatements of the two summation orders on edge cases, argument checks of the new
C-ABI entries, the SASS and resource usage of the reward term kernels and fold, the env / meter / config surface."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from tests import reward_terms_oracle as ro

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "bez_isaacgym_b200", "libbezk.so")
HEADER = os.path.join(ROOT, "include", "bezk.h")
NEW = ("bezk_reward_terms", "bezk_post_physics_rollout_ep_terms", "bezk_reward_terms_update")


# ------------------------------------------------------------------ restatements
def test_shuffle_tree_order_by_hand():
    x = np.zeros(32)
    x[0], x[16], x[31] = 1.0, 1e16, -1e16
    # lane 0 = ((x0 + x16) + (x8 + x24)) + ... : 1 is absorbed by 1e16 before -1e16 (lane 31 -> 15 -> 7 -> 3 -> 1 -> 0) arrives
    assert ro.shuffle_tree(x) == 0.0
    assert ro.shuffle_tree(np.arange(32.0)) == float(sum(range(32)))
    w = ro.warp_sums(np.ones((2, 33), np.float32), 33)
    assert w.shape == (2, 2) and w.tolist() == [[32.0, 1.0], [32.0, 1.0]]


@pytest.mark.parametrize("w", [1, 5, 255, 256, 257, 1000])
def test_fold_of_constant_and_random_partials(w):
    t, k = 3, 6
    n = 32 * w - 3
    p = np.full((t, k, w), 0.5)
    assert np.array_equal(ro.fold(p, n), np.full(k, 0.5 * t * w / (t * n)))
    rng = np.random.default_rng(w)
    p = rng.normal(size=(t, k, w))
    assert np.allclose(ro.fold(p, n), p.sum(axis=(0, 2)) / (t * n), rtol=1e-12, atol=1e-15)


def test_fold_order_is_fixed_and_propagates_nan():
    p = np.zeros((2, 5, 300))
    p[0, 0, 0], p[0, 0, 256], p[1, 0, 0] = 1e16, 1.0, -1e16          # thread 0 adds slot 0 then slot 256: the 1 is absorbed
    assert ro.fold(p, 300 * 32)[0] == 0.0
    q = p.copy()
    q[0, 0, 0], q[0, 0, 256], q[0, 0, 1] = 1.0, 1.0, 1e16            # thread 0 holds 2 before the tree meets 1e16: it survives
    assert ro.fold(q, 300 * 32)[0] == 2.0 / (2 * 300 * 32)
    p[1, 3, 7] = np.nan
    m = ro.fold(p, 300 * 32)
    assert np.isnan(m[3]) and not np.isnan(m[[0, 1, 2, 4]]).any()


# ------------------------------------------------------------------ C ABI
def _lib():
    from bez_isaacgym_b200 import _lib as L
    if not os.path.exists(L.LIB_PATH):
        pytest.skip("libbezk.so not built")
    return L, L.load()


def test_new_symbols_are_exported_and_match_the_header():
    L, lib = _lib()
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    for name in NEW:
        assert name in L.SIGNATURES and getattr(lib, name) is not None
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


def test_reward_terms_match_the_envs():
    _, lib = _lib()
    from bez_isaacgym_b200 import ops
    from bez_isaacgym_b200.tasks import KickEnv, OrientEnv, WalkEnv
    for env in (KickEnv, WalkEnv, OrientEnv):
        assert lib.bezk_reward_terms({"kick": 0, "walk": 1, "orient": 2}[env.TASK]) == len(env.REWARD_TERMS)
        assert ops.reward_terms(env.TASK) == len(env.REWARD_TERMS) and env.REWARD_TERMS[-1] == "termination"
    assert KickEnv.REWARD_TERMS == ("ball_velocity", "approach", "height", "body_velocity", "posture", "termination")
    assert WalkEnv.REWARD_TERMS == ("goal_velocity", "uprightness", "body_velocity", "posture", "termination")
    assert OrientEnv.REWARD_TERMS == ("heading", "uprightness", "body_velocity", "posture", "termination")
    assert lib.bezk_reward_terms(3) == 10001 and lib.bezk_reward_terms(-1) == 10001


def _terms_args(L, ep, terms, outcome=None, task=0, norm=(None, None, None)):
    cfg = L.BezkTaskCfg()
    p = C.c_void_p(64)                                        # never dereferenced: the checks come first
    return [task] + [p] * 11 + [0, 0] + [p] * 4 + [C.byref(cfg), p, None, p, None, None, None, None, 0, 1024] + ep + \
        list(norm[:2]) + [1e-5, norm[2], outcome, terms, None]


def test_terms_entry_checks_come_before_device_access():
    L, lib = _lib()
    p = C.c_void_p(64)
    f = lib.bezk_post_physics_rollout_ep_terms
    assert f(*_terms_args(L, [p, p, p], None)) == 10001
    assert b"term_partials NULL" in lib.bezk_last_error()
    for ep in ([None, None, None], [p, None, p], [p, p, None]):
        assert f(*_terms_args(L, ep, p)) == 10001
        assert b"episode accumulators" in lib.bezk_last_error()
    assert f(*_terms_args(L, [p, p, p], p, task=7)) == 10001
    assert b"unknown task" in lib.bezk_last_error()
    for norm in ((p, p, p), (p, None, None), (None, None, p)):
        assert f(*_terms_args(L, [p, p, p], p, norm=norm)) == 10001
        assert b"observation normaliser" in lib.bezk_last_error()
    assert f(*_terms_args(L, [p, p, p], C.c_void_p(68))) == 10002
    assert b"term_partials must be 8-byte aligned" in lib.bezk_last_error()
    assert f(*_terms_args(L, [p, p, p], p, outcome=C.c_void_p(66))) == 10002
    assert b"outcome_partials must be 4-byte aligned" in lib.bezk_last_error()
    # the episode checks of the shared step follow, with their codes
    assert f(*_terms_args(L, [p, p, C.c_void_p(68)], p)) == 10002


def test_fold_entry_checks_its_arguments():
    _, lib = _lib()
    p = C.c_void_p(64)
    f = lib.bezk_reward_terms_update
    assert f(p, 2, 10, 3, p, None) == 10001 and b"unknown task" in lib.bezk_last_error()
    assert f(p, -1, 10, 0, p, None) == 10001
    assert f(p, 2, -1, 0, p, None) == 10001
    assert f(None, 2, 10, 0, p, None) == 10001
    assert f(p, 2, 10, 0, None, None) == 10001
    assert f(C.c_void_p(68), 2, 10, 0, p, None) == 10002
    assert f(p, 2, 10, 0, C.c_void_p(68), None) == 10002
    assert f(None, 0, 10, 0, None, None) == 0                 # empty input: no-op
    assert f(None, 3, 0, 1, None, None) == 0


def test_ops_wrappers_refuse_cpu_tensors():
    import torch
    from bez_isaacgym_b200 import ops
    from bez_isaacgym_b200._lib import BezkError
    _lib()
    with pytest.raises(BezkError, match="CUDA"):
        ops.reward_terms_update(torch.zeros(2, 6, 1, dtype=torch.float64), 32, "kick", torch.zeros(6, dtype=torch.float64))
    with pytest.raises(BezkError, match="steps x 5 x 1"):
        ops.reward_terms_update(torch.zeros(2, 6, 1, dtype=torch.float64), 32, "walk", torch.zeros(5, dtype=torch.float64), steps=2)
    with pytest.raises(BezkError, match="CUDA"):
        ops.post_physics_rollout_ep_terms("kick", None, None, None, None, None, None, None, torch.zeros(32, dtype=torch.long), None,
                                          ops.make_task_cfg(), None, None, torch.zeros(32), torch.zeros(32),
                                          torch.zeros(3, 1, dtype=torch.float64), torch.zeros(6, 1, dtype=torch.float64))


# ------------------------------------------------------------------ SASS
def _cuobjdump(flag):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(LIB) or not os.path.exists(exe):
        pytest.skip("needs cuobjdump and a built libbezk.so")
    return subprocess.check_output([exe, flag, LIB], text=True)


@pytest.fixture(scope="module")
def sass():
    funcs, name = {}, None
    for line in _cuobjdump("-sass").splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
        elif name is not None:
            funcs[name].append(line)
    return {k: "\n".join(v) for k, v in funcs.items()}


@pytest.fixture(scope="module")
def res_usage():
    out, name = {}, None
    for line in _cuobjdump("-res-usage").splitlines():
        m = re.search(r"Function (\S+):", line)
        if m:
            name = m.group(1)
        elif name is not None and "REG:" in line:
            out[name] = {k: int(v) for k, v in re.findall(r"(\w+):(\d+)", line)}
            name = None
    return out


NEW_KERNELS = (("task_tile_terms_kernel", "task_tile_ep_kernel"), ("task_tile_terms_l2_kernel", "task_tile_ep_l2_kernel"),
               ("task_tile_outcome_terms_kernel", "task_tile_outcome_kernel"),
               ("task_tile_outcome_terms_l2_kernel", "task_tile_outcome_l2_kernel"))


def test_term_kernels_keep_the_memory_path_and_resources_of_their_base_kernel(sass, res_usage):
    """24 kernels: terms (EP base) and outcome_terms (outcome base), plain and L2, three tasks, with and without cleats.  Each has
    its base kernel's bulk copies, gathers and loads, no CTA-wide barrier, no atomics, no local memory beyond the base kernel's
    stack frame, the same shared memory and at most 128 registers (__launch_bounds__(128, 4)); the only extra global stores are
    the K term sums."""
    found = 0
    for task, k in (("Li0E", 6), ("Li1E", 5), ("Li2E", 5)):
        for cleats in ("Lb0E", "Lb1E"):
            for new, base in NEW_KERNELS:
                tag = f"I{cleats}Li128E{task}"
                n = [x for x in sass if re.search(r"\d" + new + tag, x)]
                b = [x for x in sass if re.search(r"\d" + base + tag, x)]
                assert len(n) == 1 and len(b) == 1, (new, tag, n, b)
                body, ref = sass[n[0]], sass[b[0]]
                assert body.count("STL") <= ref.count("STL") and body.count("LDL") <= ref.count("LDL"), "no extra local memory"
                assert "BAR.SYNC" not in body, "no CTA-wide barrier"
                for op in ("UBLKCP.S.G", "UBLKCP.G.S", "LTC64B", "LTC128B", "LDG"):
                    assert body.count(op) == ref.count(op), (n[0], op)
                assert ref.count("STG") < body.count("STG") <= ref.count("STG") + 2 * k, "the term stores (the compiler may duplicate a store across paths)"
                assert body.count("ATOM") == ref.count("ATOM") and body.count("RED.") == ref.count("RED."), "no atomics"
                rn, rb = res_usage[n[0]], res_usage[b[0]]
                assert rn["REG"] <= 128 and rn["LOCAL"] == 0 and rn["STACK"] == rb["STACK"] == 32, (n[0], rn)
                assert rn["SHARED"] == rb["SHARED"], (n[0], rn, rb)
                found += 1
    assert found == 24


def test_fold_kernel_has_no_local_memory_and_no_atomics_on_the_sums(sass):
    ks = [k for k in sass if "reward_terms_kernel" in k]
    assert len(ks) == 1, ks
    body = sass[ks[0]]
    assert "STL" not in body and "LDL" not in body
    assert body.count("ATOM") == 1, "only the ticket"


# ------------------------------------------------------------------ env / meter / config
def test_config_defaults():
    from bez_isaacgym_b200.learner import agent
    from bez_isaacgym_b200.utils import config
    assert agent.REWARD_TERM_DEFAULTS == dict(track_reward_terms=False)
    for d in (agent.DEFAULT_CONFIG, agent.TRAIN_DEFAULTS, agent.OUTCOME_DEFAULTS):
        assert "track_reward_terms" not in d
    assert "track_reward_terms" not in config.AGENT_KEYS and "track_reward_terms" not in config.TRAIN_LOOP_KEYS
    assert config.train_loop_config({"params": {"config": dict(track_reward_terms=True, max_epochs=3)}}) == dict(max_epochs=3)


def test_reward_terms_meter_refuses_unknown_term_lists():
    from bez_isaacgym_b200.learner import RewardTerms
    from bez_isaacgym_b200.tasks import KickEnv, OrientEnv, WalkEnv
    with pytest.raises(ValueError):
        RewardTerms(("a", "b"), "cpu")
    with pytest.raises(ValueError):
        RewardTerms(KickEnv.REWARD_TERMS[:-1], "cpu")
    for env in (KickEnv, WalkEnv, OrientEnv):
        m = RewardTerms(env.REWARD_TERMS, "cpu")
        assert m.task == env.TASK and m.as_dict() == {k: 0.0 for k in env.REWARD_TERMS} and m.mean.dtype.is_floating_point
