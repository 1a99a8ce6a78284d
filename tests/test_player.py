"""The player without a GPU: the rl_games tally restatement on hand-computed sequences, argument checks of the two new C-ABI
entries, the SASS of the fused step with the observation normaliser and of the tally fold, and the player config extractor."""
import ctypes as C
import math
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from tests import rl_games_player_oracle as po

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "bez_isaacgym_b200", "libbezk.so")


# ------------------------------------------------------------------ tally restatement
def test_rl_games_tally_stops_after_the_step_that_reaches_the_cutoff():
    t = po.RlGamesTally(4, games_num=3)
    assert t.step(torch.tensor([1.0, 2.0, 3.0, 4.0]), torch.tensor([0, 1, 0, 0]))          # 1 game: return 2, length 1
    assert t.games_played == 1 and t.sum_rewards == 2.0 and t.sum_steps == 1.0
    assert t.step(torch.tensor([0.0, 0.0, 0.0, 0.0]), torch.tensor([0, 0, 0, 0]))          # an empty step changes nothing
    assert t.games_played == 1 and t.sum_rewards == 2.0
    # 3 more games: 4 >= 3, so rl_games stops after adding the whole step (overshoot)
    assert not t.step(torch.tensor([1.0, 1.0, 1.0, 1.0]), torch.tensor([1, 1, 0, 1]))
    # cr = [2, 1, 4, 5], steps = [3, 2, 3, 3] before the reset of envs 0, 1, 3
    assert t.games_played == 4 and t.sum_rewards == 2.0 + 8.0 and t.sum_steps == 1.0 + 8.0
    assert t.lines[-1] == (8.0 / 3, 8.0 / 3) and t.result()["av_reward"] == 10.0 / 4


def test_rl_games_tally_nan_return_and_game_lives():
    t = po.RlGamesTally(2, games_num=2, n_game_life=2)
    assert t.n_games == 4
    assert t.step(torch.tensor([float("nan"), 1.0]), torch.tensor([1, 0]))
    assert math.isnan(t.sum_rewards) and t.sum_steps == 1.0
    assert t.step(torch.tensor([0.0, 1.0]), torch.tensor([0, 1]))
    assert not t.step(torch.tensor([1.0, 1.0]), torch.tensor([1, 1]))
    r = t.result()
    assert r["games_played"] == 4 and r["sum_steps"] == 1 + 2 + 2 + 1 and r["av_steps"] == 6 / 4 * 2


def _partials(rows, w=2):
    """rows: per step, a list of (count, return sum, length sum) per slot."""
    p = np.zeros((len(rows), 3, w))
    for t, slots in enumerate(rows):
        for s, (c, r, l) in enumerate(slots):
            p[t, :, s] = (c, r, l)
    return p


def test_fold_cutoff_mid_step_with_overshoot_and_empty_steps():
    p = _partials([[(1, 5.0, 10)], [], [(2, 3.0, 7), (1, 1.0, 2)], [(1, 100.0, 1)], []])
    tally, per = po.fold_partials(p, games_num=3)
    assert tally.tolist() == [4.0, 9.0, 19.0, 3.0]                       # step 2 crosses 3 games and is added whole
    assert per.tolist() == [[1, 5, 10], [0, 0, 0], [3, 4, 9], [0, 0, 0], [0, 0, 0]]


def test_fold_does_not_depend_on_chunking():
    rng = np.random.default_rng(0)
    p = np.zeros((40, 3, 5))
    p[:, 0] = rng.integers(0, 3, size=(40, 5))
    p[:, 1] = p[:, 0] * rng.normal(size=(40, 5))
    p[:, 2] = p[:, 0] * rng.integers(1, 50, size=(40, 5))
    whole, per = po.fold_partials(p, games_num=37)
    for k in (1, 7, 32):
        tally, rows = None, []
        for t0 in range(0, 40, k):
            tally, ps = po.fold_partials(p[t0:t0 + k], games_num=37, tally=tally)
            rows.append(ps)
        assert tally.tobytes() == whole.tobytes() and np.concatenate(rows).tobytes() == per.tobytes()
    assert whole[0] >= 37 and whole[3] < 40


def test_fold_nan_return_and_fixed_order():
    p = _partials([[(1, float("nan"), 3)], [(1, 1.0, 1)]])
    tally, _ = po.fold_partials(p, games_num=10)
    assert math.isnan(tally[1]) and tally[2] == 4.0 and tally[0] == 2.0
    # 33 slots: lane 0 adds slot 0 then slot 32; the tree then folds lanes 16, 8, 4, 2, 1 into lane 0
    q = np.zeros((3, 33))
    q[1] = [1e16] + [1.0] * 31 + [-1e16]
    c, r, _ = po.step_sums(q)
    lane0 = (1e16 + -1e16)
    assert r == lane0 + 31.0 and c == 0.0


def test_player_restatement_against_the_fold_on_random_episodes():
    """rl_games' fp32 tally and the fp64 fold agree to rounding on the same episodes."""
    g = torch.Generator().manual_seed(3)
    n, steps = 64, 60
    rew = torch.randn(steps, n, generator=g)
    done = (torch.rand(steps, n, generator=g) < 0.1).long()
    ref = po.RlGamesTally(n, games_num=50)
    cr, ln = torch.zeros(n), torch.zeros(n)
    p = np.zeros((steps, 3, 2))
    for t in range(steps):
        if not ref.step(rew[t], done[t]):
            steps = t + 1
            break
    cr, ln = torch.zeros(n), torch.zeros(n)
    for t in range(steps):
        cr, ln = cr + rew[t], ln + 1
        d = done[t].bool()
        for s in range(2):
            m = d[s * 32:(s + 1) * 32]
            p[t, :, s] = (float(m.sum()), float(cr[s * 32:(s + 1) * 32][m].double().sum()), float(ln[s * 32:(s + 1) * 32][m].double().sum()))
        cr, ln = cr * (1.0 - d.float()), ln * (1.0 - d.float())
    tally, _ = po.fold_partials(p[:steps], games_num=50)
    assert tally[0] == ref.games_played and tally[2] == ref.sum_steps
    assert tally[1] == pytest.approx(ref.sum_rewards, rel=1e-5, abs=1e-4)


# ------------------------------------------------------------------ C ABI
def _lib():
    from bez_isaacgym_b200 import _lib as L
    if not os.path.exists(L.LIB_PATH):
        pytest.skip("libbezk.so not built")
    return L, L.load()


def _norm_args(L, ep, norm, eps=1e-5):
    cfg = L.BezkTaskCfg()
    p = C.c_void_p(64)                                     # never dereferenced: the checks come first
    return [0] + [p] * 11 + [0, 0] + [p] * 4 + [C.byref(cfg), p, None, p, None, None, None, None, 0, 1024] + ep + norm[:2] + [eps] + \
        norm[2:] + [None]


def test_norm_entry_rejects_partial_arming_before_touching_a_device():
    L, lib = _lib()
    p = C.c_void_p(64)
    for norm in ([p, None, None], [None, p, p], [p, p, None]):
        assert lib.bezk_post_physics_rollout_ep_norm(*_norm_args(L, [p, p, p], norm)) == 10001
        assert b"obs_mean, obs_var and obs_norm must be all NULL or all non-NULL" in lib.bezk_last_error()


def test_norm_entry_needs_the_episode_accumulators():
    L, lib = _lib()
    p = C.c_void_p(64)
    assert lib.bezk_post_physics_rollout_ep_norm(*_norm_args(L, [None, None, None], [p, p, p])) == 10001
    assert b"episode accumulators" in lib.bezk_last_error()
    # the episode checks come first, with bezk_post_physics_rollout_ep's codes
    assert lib.bezk_post_physics_rollout_ep_norm(*_norm_args(L, [p, None, None], [p, p, p])) == 10001
    assert b"ep_return, ep_length and ep_partials" in lib.bezk_last_error()


def test_norm_entry_alignment_and_eps():
    L, lib = _lib()
    p = C.c_void_p(64)
    assert lib.bezk_post_physics_rollout_ep_norm(*_norm_args(L, [p, p, p], [p, p, C.c_void_p(72)])) == 10002
    assert b"obs_norm must be 16-byte aligned" in lib.bezk_last_error()
    assert lib.bezk_post_physics_rollout_ep_norm(*_norm_args(L, [p, p, p], [C.c_void_p(68), p, p])) == 10002
    assert lib.bezk_post_physics_rollout_ep_norm(*_norm_args(L, [p, p, p], [p, p, p], eps=-1.0)) == 10001
    assert b"obs_eps" in lib.bezk_last_error()
    assert lib.bezk_post_physics_rollout_ep_norm(*_norm_args(L, [p, p, p], [p, p, p], eps=float("nan"))) == 10001


def test_tally_entry_checks_its_arguments():
    L, lib = _lib()
    p = C.c_void_p(64)
    assert lib.bezk_player_tally_update(p, 2, 10, 0, p, p, None) == 10001
    assert b"games_num" in lib.bezk_last_error()
    assert lib.bezk_player_tally_update(p, 2, 10, -5, p, None, None) == 10001
    assert lib.bezk_player_tally_update(p, -1, 10, 5, p, None, None) == 10001
    assert lib.bezk_player_tally_update(None, 2, 10, 5, p, None, None) == 10001
    assert lib.bezk_player_tally_update(C.c_void_p(68), 2, 10, 5, p, None, None) == 10002
    assert lib.bezk_player_tally_update(p, 2, 10, 5, C.c_void_p(68), None, None) == 10002
    assert lib.bezk_player_tally_update(p, 2, 10, 5, p, C.c_void_p(68), None) == 10002
    assert b"8-byte aligned" in lib.bezk_last_error()
    assert lib.bezk_player_tally_update(None, 0, 10, 5, None, None, None) == 0           # empty input: no-op
    assert lib.bezk_player_tally_update(None, 3, 0, 5, None, None, None) == 0


def test_ops_wrappers_refuse_cpu_tensors():
    from bez_isaacgym_b200 import ops
    from bez_isaacgym_b200._lib import BezkError
    _lib()
    with pytest.raises(BezkError, match="CUDA"):
        ops.player_tally_update(torch.zeros(2, 3, 1, dtype=torch.float64), 32, 100, torch.zeros(4, dtype=torch.float64))
    with pytest.raises(BezkError, match="CUDA"):
        ops.post_physics_rollout_ep_norm("kick", None, None, None, None, None, None, None, torch.zeros(32, dtype=torch.long), None,
                                         ops.make_task_cfg(), None, None, torch.zeros(32), torch.zeros(32),
                                         torch.zeros(3, 1, dtype=torch.float64), torch.zeros(54, dtype=torch.float64),
                                         torch.ones(54, dtype=torch.float64), torch.zeros(32, 54))


# ------------------------------------------------------------------ SASS of the new kernels
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


def test_obsnorm_kernels_keep_the_ep_kernels_memory_path(sass):
    """Every task x cleats x L2 policy has an obs-normaliser kernel: TMA bulk loads and (at least two) bulk stores, 64-byte
    gathers, no CTA-wide barrier, and no local memory beyond the EP kernel of the same instantiation."""
    found = 0
    for task in ("Li0E", "Li1E", "Li2E"):
        for cleats in ("Lb0E", "Lb1E"):
            for frag, ep_frag in ((f"task_tile_obsnorm_kernelI{cleats}Li128E{task}", f"task_tile_ep_kernelI{cleats}Li128E{task}"),
                                  (f"task_tile_obsnorm_l2_kernelI{cleats}Li128E{task}", f"task_tile_ep_l2_kernelI{cleats}Li128E{task}")):
                new = [k for k in sass if frag in k]
                ep = [k for k in sass if ep_frag in k]
                assert len(new) == 1 and len(ep) == 1, (frag, new, ep)
                body, ref = sass[new[0]], sass[ep[0]]
                assert body.count("UBLKCP.S.G") >= 2 and body.count("UBLKCP.G.S") >= 2, "bulk loads and bulk stores"
                assert "LTC64B" in body, "64-byte-granule gathers"
                assert "BAR.SYNC" not in body, "no CTA-wide barrier"
                assert body.count("STL") <= ref.count("STL") and body.count("LDL") <= ref.count("LDL"), "no extra local memory"
                found += 1
    assert found == 12


def test_tally_kernel_has_no_barrier_and_no_local_memory(sass):
    names = [k for k in sass if "player_tally_kernel" in k]
    assert len(names) == 1
    body = sass[names[0]]
    assert "BAR.SYNC" not in body and "STL" not in body and "LDL" not in body


# ------------------------------------------------------------------ config
def test_player_config_extractor():
    from bez_isaacgym_b200.utils import config
    from bez_isaacgym_b200.learner import agent
    assert config.player_config({"params": {"config": {"name": "Bez_Kick"}}}) == \
        dict(games_num=2000, deterministic=True, print_stats=True, n_game_life=1)
    train = {"params": {"config": dict(player=dict(games_num=100, determenistic=False, print_stats=False, n_game_life=3))}}
    assert config.player_config(train) == dict(games_num=100, deterministic=False, print_stats=False, n_game_life=3)
    train = {"params": {"config": dict(player=dict(deterministic=False, determenistic=True))}}
    assert config.player_config(train)["deterministic"] is False
    # the agent's key sets stay as they were
    assert "player" not in config.AGENT_KEYS and "player" not in config.TRAIN_LOOP_KEYS
    assert "games_num" not in agent.DEFAULT_CONFIG and "games_num" not in agent.TRAIN_DEFAULTS


def test_player_refuses_a_host_pipeline_and_bad_sync():
    from bez_isaacgym_b200.learner import PpoPlayerContinuous

    class HostEnv:
        host_staged = True

    with pytest.raises(NotImplementedError):
        PpoPlayerContinuous(HostEnv())
    with pytest.raises(ValueError):
        PpoPlayerContinuous(HostEnv(), sync_every=0)
