"""Game term returns without a GPU: the numpy restatement of the two folds on edge cases (NaN, empty steps, the mid-step cutoff,
chunking), argument checks of the new C-ABI entries before any device access, the SASS and resource usage of the 72 step kernels
and both folds, the meter / config surface."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from tests import game_terms_oracle as go
from tests import reward_terms_oracle as ro
from tests.test_reward_terms import _cuobjdump, res_usage, sass  # noqa: F401  (module fixtures)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "bezk.h")
NEW = ("bezk_post_physics_rollout_ep_game_terms", "bezk_game_terms_meter_update", "bezk_player_game_terms_update")


def _partials(t, k, w, seed, p_done=0.3):
    """(T, 3, W) episode partials with integer done counts and (T, K, W) game term partials that are 0 where no env was done."""
    rng = np.random.default_rng(seed)
    cnt = (rng.random((t, w)) < p_done) * rng.integers(1, 33, size=(t, w))
    ep = np.zeros((t, 3, w))
    ep[:, 0] = cnt
    ep[:, 1] = rng.normal(size=(t, w)) * cnt
    ep[:, 2] = cnt * 50.0
    tp = rng.normal(size=(t, k, w)) * 10.0 * (cnt[:, None, :] > 0)
    return ep, tp


# ------------------------------------------------------------------ restatements
@pytest.mark.parametrize("w", [1, 5, 256, 257, 1000])
def test_step_sums_are_the_row_sums(w):
    ep, tp = _partials(4, 6, w, w)
    s = go.step_sums(ep, tp)
    assert s.shape == (4, 7)
    assert np.array_equal(s[:, 0], ep[:, 0].sum(axis=1)), "done counts are exact"
    assert np.allclose(s[:, 1:], tp.sum(axis=2), rtol=1e-12, atol=1e-9)


def test_step_sums_order_is_fixed():
    ep, tp = np.zeros((1, 3, 300)), np.zeros((1, 5, 300))
    tp[0, 0, 0], tp[0, 0, 256], tp[0, 0, 1] = 1e16, 1.0, -1e16          # thread 0 adds slot 0 then slot 256: the 1 is absorbed
    assert go.step_sums(ep, tp)[0, 1] == 0.0
    tp[0, 0, 0], tp[0, 0, 256], tp[0, 0, 1] = 1.0, 1.0, 1e16            # thread 0 holds 2 before the tree meets 1e16
    assert go.step_sums(ep, tp)[0, 1] == 1e16 + 2.0


def test_meter_is_rl_games_average_meter_over_per_game_rows():
    """Fed per step with the done envs' K-rows, rl_games' meter (fp32 torch.mean of the rows) and the fold agree when every step's
    rows average exactly; the size follows the done counts, capped at games_to_track."""
    from tests.rl_games_episode_oracle import AverageMeter
    import torch
    rows = [np.array([[1.0, -2.0, 0.5], [3.0, 0.0, 1.5]]), np.zeros((0, 3)), np.array([[4.0, 4.0, -4.0]])]
    ep, tp = np.zeros((3, 3, 1)), np.zeros((3, 3, 1))
    ref = AverageMeter(3, 2)
    for t, r in enumerate(rows):
        ep[t, 0, 0] = len(r)
        tp[t, :, 0] = r.sum(axis=0)
        ref.update(torch.tensor(r, dtype=torch.float32))
    mean, size = go.meter(ep, tp, 2)
    assert size == ref.current_size == 2
    assert np.array_equal(mean, ref.mean.numpy())


def test_meter_nan_and_empty_steps():
    ep, tp = np.zeros((3, 3, 2)), np.zeros((3, 5, 2))
    mean, size = go.meter(ep, tp, 100)                                   # no finished game: nothing changes
    assert size == 0 and np.array_equal(mean, np.zeros(5, np.float32))
    ep[1, 0, 1] = 2.0
    tp[1, :, 1] = [2.0, 4.0, np.nan, 6.0, np.inf]
    mean, size = go.meter(ep, tp, 100)
    assert size == 2 and mean[0] == 1.0 and mean[1] == 2.0 and np.isnan(mean[2]) and mean[3] == 3.0 and np.isinf(mean[4])


def test_player_fold_cutoff_and_chunking():
    ep, tp = _partials(40, 6, 9, 3, p_done=0.5)
    counts = go.step_sums(ep, tp)[:, 0]
    games_num = float(np.cumsum(counts)[20]) - 1.0                        # crossed inside step 20, which is added whole
    out, per = go.player_fold(ep, tp, games_num)
    assert out[0] == np.cumsum(counts)[20] and np.all(per[21:] == 0.0)
    from tests.rl_games_player_oracle import fold_partials
    tally, _ = fold_partials(ep, games_num)
    assert out[0] == tally[0], "games_counted equals the player tally's games_played"
    acc = None
    for a, b in ((0, 7), (7, 8), (8, 31), (31, 40)):                      # the same steps in chunks
        acc, _ = go.player_fold(ep[a:b], tp[a:b], games_num, acc)
    assert np.array_equal(acc, out)
    nan_tp = tp.copy()
    nan_tp[30, 2, 0] = np.nan                                             # after the cutoff: never added
    assert np.array_equal(go.player_fold(ep, nan_tp, games_num)[0], out)
    nan_tp[3, 2, 0] = np.nan
    got = go.player_fold(ep, nan_tp, games_num)[0]
    assert np.isnan(got[3]) and not np.isnan(np.delete(got, 3)).any()


def test_done_warp_sums_mask_live_envs():
    r = np.arange(2 * 40, dtype=np.float32).reshape(2, 40)
    r[1, 5] = np.nan                                                      # a live env's NaN is not summed
    done = np.zeros(40, bool)
    done[[0, 33]] = True
    got = go.done_warp_sums(r, done, 40)
    assert got.tolist() == [[0.0, 33.0], [40.0, 73.0]]
    assert np.array_equal(go.done_warp_sums(r, np.ones(40, bool), 40)[0], ro.warp_sums(r[:1], 40)[0])


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
    # the step takes every argument of bezk_post_physics_rollout_ep_terms, then the two game term pointers
    assert L.SIGNATURES[NEW[0]][1][:-3] == L.SIGNATURES["bezk_post_physics_rollout_ep_terms"][1][:-1]


def _game_args(L, ep, acc, part, outcome=None, terms=None, task=0, norm=(None, None, None)):
    cfg = L.BezkTaskCfg()
    p = C.c_void_p(64)                                        # never dereferenced: the checks come first
    return [task] + [p] * 11 + [0, 0] + [p] * 4 + [C.byref(cfg), p, None, p, None, None, None, None, 0, 1024] + ep + \
        list(norm[:2]) + [1e-5, norm[2], outcome, terms, acc, part, None]


def test_game_terms_entry_checks_come_before_device_access():
    L, lib = _lib()
    p = C.c_void_p(64)
    f = lib.bezk_post_physics_rollout_ep_game_terms
    for acc, part in ((None, None), (p, None), (None, p)):
        assert f(*_game_args(L, [p, p, p], acc, part)) == 10001
        assert b"game_term_returns / game_term_partials NULL" in lib.bezk_last_error()
    for ep in ([None, None, None], [p, None, p], [p, p, None]):
        assert f(*_game_args(L, ep, p, p)) == 10001
        assert b"episode accumulators" in lib.bezk_last_error()
    assert f(*_game_args(L, [p, p, p], p, p, task=7)) == 10001
    assert b"unknown task" in lib.bezk_last_error()
    for norm in ((p, p, p), (p, None, None), (None, None, p)):
        assert f(*_game_args(L, [p, p, p], p, p, terms=p, norm=norm)) == 10001
        assert b"observation normaliser" in lib.bezk_last_error()
    for norm in ((p, None, None), (None, p, p)):              # without term_partials the normaliser is all or nothing
        assert f(*_game_args(L, [p, p, p], p, p, norm=norm)) == 10001
        assert b"all NULL or all non-NULL" in lib.bezk_last_error()
    assert f(*_game_args(L, [p, p, p], C.c_void_p(66), p)) == 10002
    assert f(*_game_args(L, [p, p, p], p, C.c_void_p(68))) == 10002
    assert b"game_term_partials 8-byte aligned" in lib.bezk_last_error()
    assert f(*_game_args(L, [p, p, p], p, p, terms=C.c_void_p(68))) == 10002
    assert b"term_partials must be 8-byte aligned" in lib.bezk_last_error()
    assert f(*_game_args(L, [p, p, p], p, p, outcome=C.c_void_p(66))) == 10002
    assert b"outcome_partials must be 4-byte aligned" in lib.bezk_last_error()
    assert f(*_game_args(L, [p, p, C.c_void_p(68)], p, p)) == 10002     # the episode checks of the shared step follow
    assert f(*_game_args(L, [p, p, p], p, p, norm=(p, p, C.c_void_p(72)))) == 10002


@pytest.mark.parametrize("name", ["bezk_game_terms_meter_update", "bezk_player_game_terms_update"])
def test_fold_entries_check_their_arguments(name):
    _, lib = _lib()
    p, odd = C.c_void_p(64), C.c_void_p(68)
    f = getattr(lib, name)
    assert f(p, p, 2, 10, 3, 100, p, p, None) == 10001 and b"unknown task" in lib.bezk_last_error()
    assert f(p, p, -1, 10, 0, 100, p, p, None) == 10001
    assert f(p, p, 2, -1, 0, 100, p, p, None) == 10001
    assert f(p, p, 2, 10, 0, 0, p, p, None) == 10001                  # games_to_track / games_num must be positive
    assert f(None, p, 2, 10, 0, 100, p, p, None) == 10001
    assert f(p, None, 2, 10, 0, 100, p, p, None) == 10001
    assert f(odd, p, 2, 10, 0, 100, p, p, None) == 10002
    assert f(p, odd, 2, 10, 0, 100, p, p, None) == 10002
    assert f(None, None, 0, 10, 0, 100, None, None, None) == 0        # empty input: no-op
    assert f(None, None, 3, 0, 1, 100, None, None, None) == 0
    if name == "bezk_game_terms_meter_update":
        assert f(p, p, 2, 10, 0, 100, None, p, None) == 10001
        assert f(p, p, 2, 10, 0, 100, p, None, None) == 10001
        assert f(p, p, 2, 10, 0, 100, p, odd, None) == 10002          # size 8-byte aligned
    else:
        assert f(p, p, 2, 10, 0, 100, None, None, None) == 10001
        assert f(p, p, 2, 10, 0, 100, odd, None, None) == 10002
        assert f(p, p, 2, 10, 0, 100, p, odd, None) == 10002          # per_step 8-byte aligned


def test_ops_wrappers_refuse_cpu_tensors():
    import torch
    from bez_isaacgym_b200 import ops
    from bez_isaacgym_b200._lib import BezkError
    _lib()
    f64 = dict(dtype=torch.float64)
    with pytest.raises(BezkError, match="CUDA"):
        ops.game_terms_meter_update(torch.zeros(2, 3, 1, **f64), torch.zeros(2, 6, 1, **f64), 32, "kick", 100, torch.zeros(6),
                                    torch.zeros(1, dtype=torch.long))
    with pytest.raises(BezkError, match="CUDA"):
        ops.player_game_terms_update(torch.zeros(2, 3, 1, **f64), torch.zeros(2, 5, 1, **f64), 32, "walk", 100, torch.zeros(6, **f64))
    with pytest.raises(BezkError, match="term_partials must hold steps x 5 x 1"):
        ops.game_terms_meter_update(torch.zeros(2, 3, 1, **f64), torch.zeros(2, 6, 1, **f64), 32, "orient", 100, torch.zeros(5),
                                    torch.zeros(1, dtype=torch.long), steps=2)
    with pytest.raises(BezkError, match="ep_partials must hold steps x 3 x 1"):
        ops.player_game_terms_update(torch.zeros(1, 3, 1, **f64), torch.zeros(2, 6, 1, **f64), 32, "kick", 100, torch.zeros(7, **f64))
    with pytest.raises(BezkError, match="CUDA"):
        ops.post_physics_rollout_ep_game_terms("kick", None, None, None, None, None, None, None, torch.zeros(32, dtype=torch.long), None,
                                               ops.make_task_cfg(), None, None, torch.zeros(32), torch.zeros(32),
                                               torch.zeros(3, 1, **f64), torch.zeros(6, 32), torch.zeros(6, 1, **f64))


# ------------------------------------------------------------------ SASS
# each game pack and the kernel that runs the same pack without the game term returns
PACKS = (("NS_6EpArgsENS_12GameTermArgsEEE", "task_tile_ep"), ("NS_6EpArgsENS_8NormArgsENS_12GameTermArgsEEE", "task_tile_obsnorm"),
         ("NS_6EpArgsENS_7OutArgsENS_12GameTermArgsEEE", "task_tile_outcome"),
         ("NS_6EpArgsENS_8NormArgsENS_7OutArgsENS_12GameTermArgsEEE", "task_tile_obsnorm_outcome"),
         ("NS_6EpArgsENS_8TermArgsENS_12GameTermArgsEEE", "task_tile_terms"),
         ("NS_6EpArgsENS_7OutArgsENS_8TermArgsENS_12GameTermArgsEEE", "task_tile_outcome_terms"))


def test_game_kernels_keep_the_memory_path_and_resources_of_their_base_kernel(sass, res_usage):  # noqa: F811
    """72 kernels: six packs, plain and L2, three tasks, with and without cleats.  Each has its base kernel's bulk copies and
    gathers, exactly K more global loads (the accumulators), more global stores only for the K accumulators and the K partials
    (the compiler may duplicate a store across the fast path and the exact retry), no CTA-wide barrier, no atomics, no local
    memory beyond the base kernel's stack frame, the same shared memory and at most 128 registers (__launch_bounds__(128, 4))."""
    found = 0
    for task, k in (("Li0E", 6), ("Li1E", 5), ("Li2E", 5)):
        for cleats in ("Lb0E", "Lb1E"):
            for l2 in ("", "_l2"):
                for pack, base in PACKS:
                    tag = f"I{cleats}Li128E{task}"
                    n = [x for x in sass if re.search(r"\dtask_tile_game" + l2 + r"_kernel" + tag + "J" + pack, x)]
                    b = [x for x in sass if re.search(r"\d" + base + l2 + r"_kernel" + tag + "EEv", x)]
                    assert len(n) == 1 and len(b) == 1, (pack, base, l2, tag, n, b)
                    body, ref = sass[n[0]], sass[b[0]]
                    assert body.count("STL") <= ref.count("STL") and body.count("LDL") <= ref.count("LDL"), "no extra local memory"
                    assert "BAR.SYNC" not in body, "no CTA-wide barrier"
                    for op in ("UBLKCP.S.G", "UBLKCP.G.S", "LTC64B", "LTC128B"):
                        assert body.count(op) == ref.count(op), (n[0], op)
                    assert body.count("LDG") == ref.count("LDG") + k, (n[0], "the K accumulator loads")
                    assert ref.count("STG") + 2 * k <= body.count("STG") <= ref.count("STG") + 4 * k, (n[0], "the 2K stores")
                    assert body.count("ATOM") == ref.count("ATOM") == 0 and body.count("RED.") == ref.count("RED."), "no atomics"
                    rn, rb = res_usage[n[0]], res_usage[b[0]]
                    assert rn["REG"] <= 128 and rn["LOCAL"] == 0 and rn["STACK"] == rb["STACK"] == 32, (n[0], rn)
                    assert rn["SHARED"] == rb["SHARED"], (n[0], rn, rb)
                    found += 1
    assert found == 72
    assert len([x for x in sass if "task_tile_game" in x]) == 72, "no pack that nothing launches"


def test_fold_kernels_have_no_barrier_and_no_local_memory(sass, res_usage):  # noqa: F811
    for name in ("game_terms_meter_kernel", "player_game_terms_kernel"):
        ks = [k for k in sass if name in k]
        assert len(ks) == 1, ks
        body = sass[ks[0]]
        assert "BAR.SYNC" not in body and "STL" not in body and "LDL" not in body, name
        assert body.count("ATOM") == 2, "only the two tickets"
        assert res_usage[ks[0]]["LOCAL"] == 0 and res_usage[ks[0]]["STACK"] == 0


# ------------------------------------------------------------------ meter / config
def test_config_defaults():
    from bez_isaacgym_b200.learner import agent
    from bez_isaacgym_b200.utils import config
    assert agent.GAME_TERM_DEFAULTS == dict(track_game_reward_terms=False)
    for d in (agent.DEFAULT_CONFIG, agent.TRAIN_DEFAULTS, agent.OUTCOME_DEFAULTS, agent.REWARD_TERM_DEFAULTS):
        assert "track_game_reward_terms" not in d
    assert "track_game_reward_terms" not in config.AGENT_KEYS and "track_game_reward_terms" not in config.TRAIN_LOOP_KEYS
    assert config.train_loop_config({"params": {"config": dict(track_game_reward_terms=True, max_epochs=3)}}) == dict(max_epochs=3)
    import inspect
    from bez_isaacgym_b200.learner import PpoPlayerContinuous
    assert inspect.signature(PpoPlayerContinuous).parameters["track_reward_terms"].default is False


def test_game_term_meter_refuses_unknown_term_lists():
    from bez_isaacgym_b200.learner import GameTermMeter
    from bez_isaacgym_b200.tasks import KickEnv, OrientEnv, WalkEnv
    with pytest.raises(ValueError):
        GameTermMeter(("a", "b"), 100, "cpu")
    with pytest.raises(ValueError):
        GameTermMeter(KickEnv.REWARD_TERMS[:-1], 100, "cpu")
    with pytest.raises(ValueError):
        GameTermMeter(KickEnv.OUTCOMES, 100, "cpu")
    with pytest.raises(ValueError):
        GameTermMeter(KickEnv.REWARD_TERMS, 0, "cpu")
    for env in (KickEnv, WalkEnv, OrientEnv):
        m = GameTermMeter(env.REWARD_TERMS, 10, "cpu")
        assert m.task == env.TASK and m.current_size == 0 and m.as_dict() == {k: 0.0 for k in env.REWARD_TERMS}
        m._mean.fill_(1.0); m._size.fill_(3)
        m.clear()
        assert m.current_size == 0 and m.as_dict() == {k: 0.0 for k in env.REWARD_TERMS}
