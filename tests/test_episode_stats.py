"""Episode statistics without a GPU: the rl_games AverageMeter restatement on hand-computed sequences, argument checks of the two
new C-ABI entries, the SASS of the fused step with episode accumulators, and the training-loop config extractor."""
import ctypes as C
import os
import re
import shutil
import subprocess

import pytest
import torch

from tests import rl_games_episode_oracle as eo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "bez_isaacgym_b200", "libbezk.so")


# ------------------------------------------------------------------ AverageMeter restatement
def test_meter_hand_computed_sequence():
    m = eo.AverageMeter(1, 4)
    m.update(torch.tensor([[1.0], [3.0]]))                 # mean 2, size 2
    assert m.current_size == 2 and float(m.mean) == 2.0
    m.update(torch.tensor([[6.0]]))                        # old_size = min(4 - 1, 2) = 2: (2 * 2 + 6) / 3
    assert m.current_size == 3 and float(m.mean) == pytest.approx(10.0 / 3.0)
    m.update(torch.tensor([[0.0], [0.0]]))                 # old_size = min(4 - 2, 3) = 2: (10/3 * 2 + 0) / 4
    assert m.current_size == 4 and float(m.mean) == pytest.approx(20.0 / 12.0)


def test_meter_clips_when_more_games_than_tracked_finish_in_one_step():
    m = eo.AverageMeter(1, 3)
    m.update(torch.tensor([[5.0]]))
    m.update(torch.arange(10, dtype=torch.float32).view(-1, 1))      # 10 games > max_size: size 3, old_size 0, mean of all 10
    assert m.current_size == 3 and float(m.mean) == 4.5


def test_meter_empty_update_is_a_no_op():
    m = eo.AverageMeter(1, 5)
    m.update(torch.tensor([[2.0]]))
    before = m.mean.clone()
    m.update(torch.empty(0, 1))
    assert m.current_size == 1 and torch.equal(m.mean, before)


def test_meter_converges_to_the_window():
    m = eo.AverageMeter(1, 10)
    for _ in range(200):
        m.update(torch.tensor([[7.0]]))
    assert m.current_size == 10 and float(m.mean) == pytest.approx(7.0, rel=1e-6)


def test_bookkeeping_restatement_multiplies_by_not_done():
    gr, gl = eo.AverageMeter(1, 100), eo.AverageMeter(1, 100)
    cr, cl = torch.zeros(3, 1), torch.zeros(3)
    cr, cl = eo.episode_bookkeeping(cr, cl, torch.tensor([1.0, float("nan"), 2.0]), torch.tensor([0, 0, 1]), gr, gl)
    assert cr[0, 0] == 1.0 and torch.isnan(cr[1, 0]) and cr[2, 0] == 0.0 and torch.equal(cl, torch.tensor([1.0, 1.0, 0.0]))
    assert gr.current_size == 1 and float(gr.mean) == 2.0 and float(gl.mean) == 1.0
    cr, cl = eo.episode_bookkeeping(cr, cl, torch.tensor([1.0, 1.0, 1.0]), torch.tensor([0, 1, 0]), gr, gl)
    assert torch.isnan(cr[1, 0]), "NaN * 0 stays NaN"
    assert torch.isnan(gr.mean).all() and float(gl.mean) == 1.5


# ------------------------------------------------------------------ C ABI
def _lib():
    from bez_isaacgym_b200 import _lib as L
    if not os.path.exists(L.LIB_PATH):
        pytest.skip("libbezk.so not built")
    return L, L.load()


def test_ep_entry_rejects_partial_arming_before_touching_a_device():
    L, lib = _lib()
    cfg = L.BezkTaskCfg()
    p = C.c_void_p(64)                                     # never dereferenced: the checks come first
    args = [0] + [p] * 11 + [0, 0] + [p] * 4 + [C.byref(cfg), p, None, p, None, None, None, None, 0, 1024]
    for ep in ([p, None, None], [None, p, p], [p, p, None]):
        rc = lib.bezk_post_physics_rollout_ep(*args, *ep, None)
        assert rc == 10001 and b"all NULL or all non-NULL" in lib.bezk_last_error()
    rc = lib.bezk_post_physics_rollout_ep(*args, C.c_void_p(66), p, p, None)
    assert rc == 10002
    rc = lib.bezk_post_physics_rollout_ep(9, *args[1:], p, p, p, None)
    assert rc == 10001 and b"unknown task" in lib.bezk_last_error()


def test_meter_entry_checks_its_arguments():
    L, lib = _lib()
    p = C.c_void_p(64)
    assert lib.bezk_episode_meter_update(p, -1, 10, 100, p, p, None) == 10001
    assert lib.bezk_episode_meter_update(p, 2, 10, 0, p, p, None) == 10001
    assert lib.bezk_episode_meter_update(None, 2, 10, 100, p, p, None) == 10001
    assert lib.bezk_episode_meter_update(C.c_void_p(68), 2, 10, 100, p, p, None) == 10002
    assert lib.bezk_episode_meter_update(None, 0, 10, 100, None, None, None) == 0          # empty input: no-op
    assert lib.bezk_episode_meter_update(None, 3, 0, 100, None, None, None) == 0


def test_ops_wrappers_refuse_cpu_tensors():
    from bez_isaacgym_b200 import ops
    from bez_isaacgym_b200._lib import BezkError
    _lib()
    with pytest.raises(BezkError, match="CUDA"):
        ops.episode_meter_update(torch.zeros(2, 3, 1, dtype=torch.float64), 32, 100, torch.zeros(2), torch.zeros(2, dtype=torch.long))
    with pytest.raises(BezkError, match="CUDA"):
        ops.post_physics_rollout_ep("kick", None, None, None, None, None, None, None, torch.zeros(32, dtype=torch.long), None,
                                    ops.make_task_cfg(), None, None, torch.zeros(32), torch.zeros(32),
                                    torch.zeros(3, 1, dtype=torch.float64))


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


def test_ep_kernels_keep_the_plain_kernels_memory_path(sass):
    """Every task x cleats x L2 policy has an EP kernel: TMA bulk copies, 64-byte gathers, no CTA-wide barrier, and no local
    memory beyond what the plain kernel of the same instantiation already has (the precise-fallback stack, no spills)."""
    found = 0
    for task in ("Li0E", "Li1E", "Li2E"):
        for cleats in ("Lb0E", "Lb1E"):
            for ep_frag, plain_frag in ((f"task_tile_ep_kernelI{cleats}Li128E{task}", f"task_tile_kernelILi7E{cleats}Li128E{task}"),
                                        (f"task_tile_ep_l2_kernelI{cleats}Li128E{task}", f"task_tile_l2_kernelILi7E{cleats}Li128E{task}")):
                ep = [k for k in sass if ep_frag in k]
                plain = [k for k in sass if plain_frag in k]
                assert len(ep) == 1 and len(plain) == 1, (ep_frag, ep, plain)
                body, ref = sass[ep[0]], sass[plain[0]]
                assert body.count("UBLKCP.S.G") >= 2 and "UBLKCP.G.S" in body and "SYNCS" in body
                assert "LTC64B" in body, "64-byte-granule gathers"
                assert "BAR.SYNC" not in body, "no CTA-wide barrier"
                assert body.count("STL") <= ref.count("STL") and body.count("LDL") <= ref.count("LDL"), "no extra local memory"
                found += 1
    assert found == 12


def test_meter_kernel_has_no_barrier_and_no_local_memory(sass):
    body = sass[[k for k in sass if "episode_meter_kernel" in k][0]]
    assert "BAR.SYNC" not in body and "STL" not in body and "LDL" not in body


# ------------------------------------------------------------------ config
def test_train_loop_config_extractor():
    from bez_isaacgym_b200.utils import config
    from bez_isaacgym_b200.learner import agent
    train = {"params": {"config": dict(name="Bez_Kick", score_to_win=20000, max_epochs=5000, save_best_after=50, save_frequency=100,
                                       games_to_track=100, gamma=0.99, horizon_length=32)}}
    got = config.train_loop_config(train)
    assert got == dict(name="Bez_Kick", score_to_win=20000, max_epochs=5000, save_best_after=50, save_frequency=100,
                       games_to_track=100)
    assert set(config.TRAIN_LOOP_KEYS) == set(agent.TRAIN_DEFAULTS)
    assert not set(config.TRAIN_LOOP_KEYS) & set(config.AGENT_KEYS)
    assert agent.TRAIN_DEFAULTS["games_to_track"] == 100
