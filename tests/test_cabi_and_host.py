"""CPU: the C-ABI library loads and exports every symbol include/bezk.h declares; host-side logic that needs no GPU."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    with open(os.path.join(ROOT, "include", "bezk.h")) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    return sorted(set(re.findall(r"\b(bezk_[a-z0-9_]+)\s*\(", text)))


def test_build_entry_produces_library():
    import __graft_entry__ as ge
    ge.build()
    assert os.path.isfile(ge.LIB)


def test_library_exports_every_declared_symbol():
    from bez_isaacgym_b200 import _lib
    lib = _lib.load()
    declared = _declared_symbols()
    assert len(declared) >= 18
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/bezk.h but not exported by libbezk.so"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature in bez_isaacgym_b200/_lib.py"
    assert sorted(_lib.SIGNATURES) == declared, "ctypes table and header disagree"
    assert lib.bezk_version() == 130


def test_struct_layout_matches_header():
    """BezkTaskCfg / BezkPpoCfg are passed by pointer from Python and by value into kernels: sizes must agree."""
    from bez_isaacgym_b200 import _lib
    assert ctypes.sizeof(_lib.BezkTaskCfg) == 6 * 4 + 5 * 4 + 2 * 4 + 4 * 4 + 3 * 18 * 4
    assert ctypes.sizeof(_lib.BezkPpoCfg) == 7 * 4


def test_argument_validation_without_gpu():
    """Entry points reject bad arguments before touching the device (error codes + bezk_last_error)."""
    from bez_isaacgym_b200 import _lib, ops
    lib = _lib.load()
    cfg = ops.make_task_cfg()
    assert lib.bezk_pre_physics(None, None, None, ctypes.byref(cfg), 4, None) == 10001
    assert b"NULL" in lib.bezk_last_error()
    assert lib.bezk_pre_physics(None, None, None, ctypes.byref(cfg), 0, None) == 0          # empty input is a no-op
    bad = ops.make_task_cfg()
    bad.imu_body = 99
    assert lib.bezk_pre_physics(None, None, None, ctypes.byref(bad), 4, None) == 10003
    assert lib.bezk_gae(None, None, None, None, None, 7, 0.99, 0.95, None, None, 32, 8, None) == 10001
    assert lib.bezk_gae(None, None, None, None, None, 0, 0.99, 0.95, None, None, 0, 8, None) == 0
    assert lib.bezk_post_physics(*([None] * 9), 0, 0, *([None] * 4), ctypes.byref(cfg), None, None, None, 0, 4, None) == 10001


def test_ops_refuse_cpu_tensors_no_fallback():
    from bez_isaacgym_b200 import ops
    cfg = ops.make_task_cfg()
    with pytest.raises(ops.BezkError, match="CUDA only"):
        ops.pre_physics(torch.zeros(4, 18), torch.zeros(4, 18), cfg)
    with pytest.raises(ops.BezkError, match="CUDA only"):
        ops.gae(torch.zeros(2, 4), torch.zeros(2, 4), torch.zeros(2, 4, dtype=torch.uint8), torch.zeros(4),
                torch.zeros(4, dtype=torch.uint8), 0.99, 0.95, torch.zeros(2, 4), torch.zeros(2, 4))


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from bez_isaacgym_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.BezkError, match="no CPU / torch fallback"):
        _lib.load()


def test_task_cfg_constants_follow_reference_semantics():
    from bez_isaacgym_b200 import ops
    c = ops.make_task_cfg()
    assert c.max_episode_length == int(15 / 0.01667 + 0.5) == 900
    assert c.reset_pos_span == pytest.approx(0.3) and c.reset_pos_lo == pytest.approx(-0.15)
    # (hi - lo) is formed in double and THEN rounded to fp32, as torch does for python scalars
    assert c.reset_pos_span == ctypes.c_float(0.15 - -0.15).value
    assert c.left_foot_body == 12 and c.right_foot_body == 20 and c.imu_body == 1 and c.num_bodies == 22
    cc = ops.make_task_cfg(num_bodies=30, cleats=True)
    assert cc.left_foot_body == 13 and cc.right_foot_body == 25 and cc.flags & 1
    swapped = ops.make_task_cfg(dof_lower=[1.0] * 18, dof_upper=[-1.0] * 18)     # kick_env.py:395-397
    assert swapped.dof_lower[3] == -1.0 and swapped.dof_upper[3] == 1.0


def test_model_constants_match_reference_urdf():
    from oracle import reference_loader as rl
    if not rl.reference_available():
        pytest.skip("/root/reference not present")
    import numpy as np
    from bez_isaacgym_b200 import bez_model as bm
    from oracle.urdf_layout import parse
    base = os.path.join(rl.REFERENCE_ROOT, "resources", "assets", "bez", "model")
    lay = parse(os.path.join(base, "soccerbot_stl.urdf"))
    assert lay.dof_names == list(bm.DOF_NAMES)
    assert np.array_equal(np.float32(lay.lower), np.float32(bm.DOF_LOWER))
    assert np.array_equal(np.float32(lay.upper), np.float32(bm.DOF_UPPER))
    assert len(lay.bodies) + 1 == bm.BODIES_NO_CLEATS
    assert lay.bodies[bm.IMU_BODY] == "imu_link" and lay.bodies[bm.LEFT_FOOT_BODY] == "left_foot"
    assert lay.bodies[bm.RIGHT_FOOT_BODY] == "right_foot"
    sens = parse(os.path.join(base, "soccerbot_stl_sensor.urdf"))
    assert len(sens.bodies) + 1 == bm.BODIES_CLEATS
    assert all("left_foot_cleat" in b for b in sens.bodies[bm.LEFT_CLEATS[0]:bm.LEFT_CLEATS[1]])
    assert all("right_foot_cleat" in b for b in sens.bodies[bm.RIGHT_CLEATS[0]:bm.RIGHT_CLEATS[1]])
    import yaml
    with open(os.path.join(rl.REFERENCE_ROOT, "bez_isaacgym", "cfg", "task", "bez_kick_test.yaml")) as f:
        ref_cfg = yaml.safe_load(f)
    mine = bm.default_task_cfg(1)
    for key in ("bezInitState", "ballInitState", "goalState", "readyJointAngles"):
        assert mine["env"][key] == ref_cfg["env"][key], key
    assert mine["env"]["clipActions"] == ref_cfg["env"]["clipActions"] and mine["sim"]["dt"] == ref_cfg["sim"]["dt"]
    assert mine["env"]["learn"]["episodeLength_s"] == ref_cfg["env"]["learn"]["episodeLength_s"]


# ----------------------------------------------------------------------------------------------- DR schedule / gate logic (CPU)
def _reference_dr_params(p, last_step):
    """The parameter arithmetic of the reference's apply_randomizations (tasks/base/vec_task.py:562-618), restated."""
    dist, op_type = p["distribution"], p["operation"]
    sched_type = p.get("schedule")
    sched_step = p.get("schedule_steps")
    if sched_type == "linear":
        s = 1.0 / sched_step * min(last_step, sched_step)
    elif sched_type == "constant":
        s = 0 if last_step < sched_step else 1
    else:
        s = 1
    if dist == "gaussian":
        mu, var = p["range"]
        mu_corr, var_corr = p.get("range_correlated", [0., 0.])
        if op_type == "additive":
            mu *= s; var *= s; mu_corr *= s; var_corr *= s
        elif op_type == "scaling":
            var = var * s
            mu = mu * s + 1.0 * (1.0 - s)
            var_corr = var_corr * s
            mu_corr = mu_corr * s + 1.0 * (1.0 - s)
        return {"mu": mu, "var": var, "mu_corr": mu_corr, "var_corr": var_corr}
    lo, hi = p["range"]
    lo_corr, hi_corr = p.get("range_correlated", [0., 0.])
    if op_type == "additive":
        lo *= s; hi *= s; lo_corr *= s; hi_corr *= s
    elif op_type == "scaling":
        lo = lo * s + 1.0 * (1.0 - s); hi = hi * s + 1.0 * (1.0 - s)
        lo_corr = lo_corr * s + 1.0 * (1.0 - s); hi_corr = hi_corr * s + 1.0 * (1.0 - s)
    return {"lo": lo, "hi": hi, "lo_corr": lo_corr, "hi_corr": hi_corr}


def test_apply_randomizations_gate_and_schedules_match_the_reference_logic():
    """Host logic of ``VecTask.apply_randomizations`` (frequency gate, first-call rule, linear / constant schedules, additive /
    scaling, gaussian / uniform) against the restated reference arithmetic -- no kernel runs (the lambdas are only built)."""
    import types
    import torch
    from bez_isaacgym_b200.tasks.base.vec_task import VecTask
    specs = {
        "observations": {"range": [0.1, .002], "range_correlated": [0.2, 0.03], "operation": "additive", "distribution": "gaussian",
                         "schedule": "linear", "schedule_steps": 40},
        "actions": {"range": [0.9, 1.2], "range_correlated": [0.95, 1.05], "operation": "scaling", "distribution": "uniform",
                    "schedule": "constant", "schedule_steps": 25},
    }
    fake = types.SimpleNamespace(sim=types.SimpleNamespace(frame=0), first_randomization=True, last_step=-1, last_rand_step=-1,
                                 randomize_buf=torch.zeros(8, dtype=torch.long), reset_buf=torch.ones(8, dtype=torch.long),
                                 dr_randomizations={}, _dr_seed=1, compute_device=torch.device("cpu"))
    params = dict(frequency=10, **specs)
    rebuilt = []
    last_rand = None
    for frame in (0, 3, 9, 10, 12, 24, 30, 55):
        fake.sim.frame = frame
        fake.randomize_buf += 4
        before = {k: dict(v) for k, v in fake.dr_randomizations.items()}
        VecTask.apply_randomizations(fake, params)
        expect_rebuild = last_rand is None or frame - last_rand >= 10
        if expect_rebuild:
            last_rand = frame
            rebuilt.append(frame)
            for name, spec in specs.items():
                want = _reference_dr_params(spec, frame)
                got = fake.dr_randomizations[name]
                for k, v in want.items():
                    assert got[k] == pytest.approx(v, rel=1e-12, abs=1e-15), (frame, name, k)
                assert callable(got["noise_lambda"]) and "corr" not in got          # the correlated draw is redrawn lazily
        else:
            assert {k: {kk: vv for kk, vv in v.items() if kk != "noise_lambda"} for k, v in fake.dr_randomizations.items()} == \
                   {k: {kk: vv for kk, vv in v.items() if kk != "noise_lambda"} for k, v in before.items()}
    assert rebuilt == [0, 10, 24, 55]
    assert fake.first_randomization is False
    with pytest.raises(NotImplementedError):
        VecTask.apply_randomizations(fake, {"sim_params": {"gravity": {}}})


def test_reference_task_yaml_loads_without_hydra():
    """``utils.config.load_task_config`` resolves the reference's own cfg/task/*.yaml (Hydra interpolations + the four custom
    resolvers of train.py:53-58) to what ``bez_model.default_task_cfg`` hard-codes.  Needs /root/reference."""
    from bez_isaacgym_b200 import bez_model as bm
    from bez_isaacgym_b200.utils import config as cfgmod
    root = os.environ.get("BEZ_REFERENCE_ROOT", "/root/reference")
    path = os.path.join(root, "bez_isaacgym", "cfg", "task", "bez_kick.yaml")
    if not os.path.isfile(path):
        pytest.skip("needs /root/reference (authoring container)")
    cfg = cfgmod.load_task_config(path, num_envs=512)
    want = bm.default_task_cfg(512)
    assert cfg["env"]["numEnvs"] == 512 and cfg["physics_engine"] == "physx"
    assert cfg["sim"]["use_gpu_pipeline"] is True and cfg["sim"]["physx"]["use_gpu"] is True
    assert cfg["sim"]["physx"]["num_threads"] == 4 and cfg["sim"]["physx"]["num_subscenes"] == 4
    for key in ("clipActions", "bezInitState", "ballInitState", "goalState", "readyJointAngles"):
        assert cfg["env"][key] == want["env"][key], key
    assert cfg["env"]["learn"]["episodeLength_s"] == want["env"]["learn"]["episodeLength_s"]
    assert cfg["env"]["asset"]["cleats"] == want["env"]["asset"]["cleats"] and cfg["sim"]["dt"] == want["sim"]["dt"]
    assert cfg["task"]["randomize"] is False and "observations" in cfg["task"]["randomization_params"]
    # defaults: numEnvs 4096 when num_envs is '' ; CPU pipeline flips both flags
    assert cfgmod.load_task_config(path)["env"]["numEnvs"] == 4096
    cpu = cfgmod.load_task_config(path, pipeline="cpu", sim_device="cpu")
    assert cpu["sim"]["use_gpu_pipeline"] is False and cpu["sim"]["physx"]["use_gpu"] is False
    for name, goal in (("bez_walk.yaml", [2.0, 0.0]), ("bez_orient.yaml", [2.0, 0.0])):
        c = cfgmod.load_task_config(os.path.join(root, "bez_isaacgym", "cfg", "task", name), num_envs=64)
        assert c["env"]["goalState"]["goal"] == goal and c["env"]["learn"]["episodeLength_s"] == 10
    with pytest.raises(KeyError):
        cfgmod.load_task_config(path, nonsense=1)
    # every key the env classes read (tasks/kick_env.py, tasks/base/vec_task.py) is present in the reference's own files
    for name in ("bez_kick.yaml", "bez_walk.yaml", "bez_orient.yaml"):
        c = cfgmod.load_task_config(os.path.join(root, "bez_isaacgym", "cfg", "task", name), num_envs=8)
        env = c["env"]
        for state in ("bezInitState",) + (("ballInitState",) if name == "bez_kick.yaml" else ()):
            assert all(len(env[state][k]) == n for k, n in (("pos", 3), ("rot", 4), ("vLinear", 3), ("vAngular", 3)))
        assert len(env["goalState"]["goal"]) == 2 and isinstance(env["asset"]["cleats"], bool)
        assert set(bm.DOF_NAMES) <= set(env["readyJointAngles"])
        assert env["control"]["stiffness"] > 0 and env["control"]["damping"] > 0 and env["learn"]["episodeLength_s"] > 0
        assert isinstance(c["task"]["randomize"], bool) and c["sim"]["dt"] > 0 and c["sim"]["up_axis"] == "z"
        assert isinstance(env["debug"]["rewards"], bool) and env["clipActions"] == 3.9 and "clipObservations" not in env
        if name == "bez_orient.yaml":
            assert env["goalState"]["goal_angle"] == pytest.approx(1.5708)


def test_reference_train_yaml_pins_the_agent_defaults():
    """``learner.agent.DEFAULT_CONFIG`` is what the reference's own cfg/train/bez_kickPPO.yaml says (:45-79), read through the
    Hydra-free loader (``${....task.env.numEnvs}``, ``${.name}``, ``${if:...}``, ``${resolve_default:...}``)."""
    from bez_isaacgym_b200.learner.agent import DEFAULT_CONFIG
    from bez_isaacgym_b200.utils import config as cfgmod
    root = os.environ.get("BEZ_REFERENCE_ROOT", "/root/reference")
    tpath = os.path.join(root, "bez_isaacgym", "cfg", "task", "bez_kick.yaml")
    ppath = os.path.join(root, "bez_isaacgym", "cfg", "train", "bez_kickPPO.yaml")
    if not os.path.isfile(ppath):
        pytest.skip("needs /root/reference (authoring container)")
    task = cfgmod.load_task_config(tpath, num_envs=2048)
    train = cfgmod.load_train_config(ppath, task, checkpoint="")
    p = train["params"]
    assert p["seed"] == 42 and p["load_checkpoint"] is False and p["load_path"] == ""
    assert p["config"]["num_actors"] == 2048 and p["config"]["name"] == "Bez_Kick_36" == p["config"]["full_experiment_name"]
    assert p["config"]["max_epochs"] == 100000
    assert p["network"]["mlp"]["units"] == [400, 200, 100] and p["network"]["space"]["continuous"]["fixed_sigma"] is True
    got = cfgmod.agent_config(train)
    for k, v in got.items():
        assert DEFAULT_CONFIG[k] == v, (k, DEFAULT_CONFIG[k], v)
    assert set(got) == set(cfgmod.AGENT_KEYS)
    assert cfgmod.load_train_config(ppath, task, checkpoint="runs/x.pth")["params"]["load_checkpoint"] is True


def test_ctypes_signatures_match_the_header_prototypes():
    """Argument COUNT and coarse kind (pointer / integer / floating) of every ctypes signature against the prototype in
    include/bezk.h -- an ABI drift between the two would corrupt arguments silently on the GPU box."""
    import ctypes as C
    import re
    from bez_isaacgym_b200 import _lib
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "bezk.h")).read()
    header = re.sub(r"/\*.*?\*/", " ", header, flags=re.S)
    protos = dict(re.findall(r"\b(?:int|int64_t|const char\*)\s+(bezk_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", header, flags=re.S))
    assert set(protos) == set(_lib.SIGNATURES)

    def kind_of_param(text):
        text = " ".join(text.split())
        if text in ("void", ""):
            return None
        if "*" in text:
            return "ptr"
        if re.search(r"\b(float|double)\b", text):
            return "fp"
        return "int"

    def kind_of_ctype(t):
        if t in (C.c_void_p, C.c_char_p) or hasattr(t, "contents") or getattr(t, "_type_", None) is not None and issubclass(t, C._Pointer):
            return "ptr"
        if t in (C.c_float, C.c_double):
            return "fp"
        return "int"

    for name, params in protos.items():
        want = [k for k in (kind_of_param(p) for p in params.split(",")) if k is not None]
        got = [kind_of_ctype(t) for t in _lib.SIGNATURES[name][1]]
        assert got == want, (name, got, want)
        # 64-bit integers must be declared 64-bit on the Python side too
        widths = [("64" in p) for p in params.split(",") if kind_of_param(p) == "int"]
        cw = [C.sizeof(t) == 8 for t in _lib.SIGNATURES[name][1] if kind_of_ctype(t) == "int"]
        assert widths == cw, (name, widths, cw)


def test_ctypes_structs_match_the_header_layout(tmp_path):
    """sizeof / offsetof of the three by-value config structs, as gcc lays them out from include/bezk.h (which must stay plain
    C), against the ctypes mirrors in bez_isaacgym_b200/_lib.py."""
    import ctypes as C
    import shutil
    import subprocess
    from bez_isaacgym_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    structs = {"BezkTaskCfg": _lib.BezkTaskCfg, "BezkPpoCfg": _lib.BezkPpoCfg, "BezkNoiseCfg": _lib.BezkNoiseCfg,
               "BezkRolloutCfg": _lib.BezkRolloutCfg}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "bezk.h"', 'int main(void) {']
    for sname, st in structs.items():
        lines.append(f'  printf("{sname} %zu\\n", sizeof({sname}));')
        for fname, _ in st._fields_:
            lines.append(f'  printf("{sname}.{fname} %zu\\n", offsetof({sname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)])
    out = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    for sname, st in structs.items():
        assert int(out[sname]) == C.sizeof(st), sname
        for fname, _ in st._fields_:
            assert int(out[f"{sname}.{fname}"]) == getattr(st, fname).offset, (sname, fname)


@pytest.mark.parametrize("task,cleats", [("kick", False), ("kick", True), ("walk", False), ("orient", False)])
def test_host_pack_gathers_the_sparse_rows(task, cleats):
    """``bezk_host_pack_begin`` / ``_wait`` (host worker threads, no CUDA call): every env's record holds, bit for bit, the
    IMU-link slice, the foot (cleat) force rows and the root-state subset of the Isaac Gym AoS tensors -- for ragged chunk sizes, a
    non-zero env0, more jobs in flight than the ring has slots, and an empty job."""
    import numpy as np
    from bez_isaacgym_b200 import _lib, ops
    lib = _lib.load()
    assert lib.bezk_host_pack_config(3, 50, -1) >= 3 and lib.bezk_host_pack_config(99, -1, -1) == -10001
    tid = ops._TASK_ID[task]
    nb = (30 if cleats else 22) - (0 if task == "kick" else 1)
    actors = 2 if task == "kick" else 1
    cfg = ops.make_task_cfg(num_bodies=nb, cleats=cleats)
    fw = 12 if cleats else 3
    nroot = 7 if task == "kick" else 3
    rs = lib.bezk_host_pack_record_floats(tid, ctypes.byref(cfg))
    assert rs == -(-(10 + 2 * fw + nroot + 1) // 4) * 4 and (rs, task, cleats) != (24, "kick", True)   # always >= 1 pad float
    if task == "kick" and not cleats:
        assert rs == 24                                          # 96 B per env
    n = 70_001
    rng = np.random.default_rng(5)
    rb = rng.standard_normal((n, nb, 13), dtype=np.float32)
    cf = rng.standard_normal((n, nb, 3), dtype=np.float32)
    root = rng.standard_normal((n, actors, 13), dtype=np.float32)
    cf[::7, cfg.left_foot_body] = np.nan                       # NaN forces travel unchanged
    rec = np.full((n, rs), -7.0, dtype=np.float32)
    dof = rng.standard_normal((n, 36), dtype=np.float32)
    P = lambda a, off=0: ctypes.c_void_p(a.ctypes.data + 4 * off)           # noqa: E731
    # 97 ragged jobs (> 64 ring slots) issued before any wait, covering [0, n) in order
    edges = sorted(set([0, n] + [int(x) for x in rng.integers(1, n, size=96)]))
    tickets = [lib.bezk_host_pack_begin(tid, P(rb), P(cf), P(root), None, None, ctypes.byref(cfg), P(rec, lo * rs), lo, hi - lo)
               for lo, hi in zip(edges[:-1], edges[1:])]
    assert all(t > 0 for t in tickets) and tickets == sorted(tickets)
    for t in reversed(tickets):
        assert lib.bezk_host_pack_wait(t) == 0
    assert lib.bezk_host_pack_wait(tickets[0]) == 0              # waiting twice is fine
    bits = lambda a: np.ascontiguousarray(a).view(np.uint32)     # noqa: E731
    assert np.array_equal(bits(rec[:, 0:10]), bits(rb[:, cfg.imu_body, 3:13]))
    k = fw // 3
    left = cf[:, cfg.left_foot_body:cfg.left_foot_body + k].reshape(n, -1)
    right = cf[:, cfg.right_foot_body:cfg.right_foot_body + k].reshape(n, -1)
    assert np.array_equal(bits(rec[:, 10:10 + fw]), bits(left))
    assert np.array_equal(bits(rec[:, 10 + fw:10 + 2 * fw]), bits(right))
    ro = 10 + 2 * fw
    flat = root.reshape(n, -1)
    want_root = flat[:, [0, 1, 2, 13, 14, 20, 21]] if task == "kick" else flat[:, 0:3]
    assert np.array_equal(bits(rec[:, ro:ro + nroot]), bits(want_root))
    assert (rec[:, ro + nroot:] == 0).all()
    # empty job, bad arguments
    # chunk layout with the dense dof_state rows copied along: dst = [k x 36 dof floats | k records]
    lo, k = 4099, 30_001
    buf = np.full(k * (36 + rs), -7.0, dtype=np.float32)
    vals = rng.standard_normal(n, dtype=np.float32)            # critic values ride in the record's last (pad) float
    assert lib.bezk_host_pack_wait(lib.bezk_host_pack_begin(tid, P(rb), P(cf), P(root), P(dof), P(vals), ctypes.byref(cfg), P(buf), lo,
                                                            k)) == 0
    assert np.array_equal(bits(buf[:k * 36].reshape(k, 36)), bits(dof[lo:lo + k]))
    got = buf[k * 36:].reshape(k, rs)
    assert np.array_equal(bits(got[:, :rs - 1]), bits(rec[lo:lo + k, :rs - 1])) and np.array_equal(bits(got[:, rs - 1]), bits(vals[lo:lo + k]))
    assert lib.bezk_host_pack_begin(tid, P(rb), P(cf), P(root), None, None, ctypes.byref(cfg), P(rec), 5, 0) == 0
    assert lib.bezk_host_pack_wait(0) == 0
    assert lib.bezk_host_pack_begin(tid, None, P(cf), P(root), None, None, ctypes.byref(cfg), P(rec), 0, 4) == -10001
    assert lib.bezk_host_pack_begin(9, P(rb), P(cf), P(root), None, None, ctypes.byref(cfg), P(rec), 0, 4) == -10001
    assert lib.bezk_host_pack_begin(tid, P(rb), P(cf), P(root), None, None, ctypes.byref(cfg), P(rec, 1), 0, 4) == -10002
    assert lib.bezk_host_pack_wait(1 << 40) == 10001
    assert lib.bezk_post_physics_packed(tid, *([None] * 10), 0, 0, *([None] * 4), ctypes.byref(cfg), None, None, None, 7, 4, 0, None, None,
                                        None, None, None, None, None) == 10001


def test_bench_arms_share_one_workload_config(monkeypatch):
    """The driver compares the ``config`` objects of ``bench.py`` and ``bench.py --impl reference``: both come from ONE function of
    the same arguments, name the BASELINE configs[3] shard size by default and carry no model keys."""
    import importlib
    import sys
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    bench = importlib.import_module("bench")
    a = bench.parse()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--gpus", "1", "--steps", "3", "--warmup", "1"])
    b = bench.parse()
    ca, cb = bench.workload_config(a), bench.workload_config(b)
    assert ca == cb and ca["envs_per_gpu"] == 262144 and ca["horizon"] == 32 and "workload" in ca and "model" not in ca
    assert a.gpus == 1 and a.warmup >= 3 and a.e2e_mode == "auto"
    assert bench.METRIC == "task+GAE env-steps/s" and bench.UNIT == "env-steps/s"


def test_bench_dump_outputs_is_a_fixed_sample_within_the_size_limit(monkeypatch, tmp_path):
    """``bench.py --dump-outputs DIR``: the env sample is the same on every run and fits the size limit; the files are float32
    (float64 stays float64); an oversized dump is refused before anything is written; ``--steps`` below 1 is refused."""
    import importlib
    import sys
    import numpy as np
    bench = importlib.import_module("bench")
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "7", "--dump-outputs", str(tmp_path / "d")])
    a = bench.parse()
    assert a.steps == 7 and a.dump_outputs == str(tmp_path / "d")
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        monkeypatch.setattr(sys, "argv", ["bench.py", *bad])
        with pytest.raises(SystemExit):
            bench.parse()
    idx = bench.sample_envs(262144, 241)
    assert torch.equal(idx, bench.sample_envs(262144, 241)) and bool((idx[1:] > idx[:-1]).all())
    assert 0 < 4 * 241 * len(idx) <= bench.DUMP_BYTES and int(idx[-1]) < 262144
    assert torch.equal(bench.sample_envs(100, 241), torch.arange(100))
    bench.write_outputs(str(tmp_path / "d"), {"obs": torch.ones(3, 2), "reset": torch.ones(3, dtype=torch.long),
                                              "stats": torch.ones(2, dtype=torch.float64)})
    got = {p.stem: np.load(p) for p in (tmp_path / "d").iterdir()}
    assert {k: v.dtype for k, v in got.items()} == {"obs": np.float32, "reset": np.float32, "stats": np.float64}
    with pytest.raises(ValueError, match="dump limit"):
        bench.write_outputs(str(tmp_path / "big"), {"x": torch.empty(bench.DUMP_BYTES // 4 + 1)})
    assert not (tmp_path / "big").exists()


def test_host_pack_pool_serves_several_issuing_threads():
    """The pool is process-wide: jobs issued and awaited from several Python threads at once (two envs stepping in two threads)
    all complete with the right bytes."""
    import threading
    import numpy as np
    from bez_isaacgym_b200 import _lib, ops
    lib = _lib.load()
    lib.bezk_host_pack_config(3, 50, -1)
    cfg = ops.make_task_cfg(num_bodies=22)
    rs = lib.bezk_host_pack_record_floats(0, ctypes.byref(cfg))
    n, errors = 20_000, []
    P = lambda a, off=0: ctypes.c_void_p(a.ctypes.data + 4 * off)           # noqa: E731

    def worker(seed):
        rng = np.random.default_rng(seed)
        rb = rng.standard_normal((n, 22, 13), dtype=np.float32)
        cf = rng.standard_normal((n, 22, 3), dtype=np.float32)
        root = rng.standard_normal((n, 2, 13), dtype=np.float32)
        rec = np.zeros((n, rs), np.float32)
        for it in range(40):
            cut = int(rng.integers(1, n))
            ts = [lib.bezk_host_pack_begin(0, P(rb), P(cf), P(root), None, None, ctypes.byref(cfg), P(rec, lo * rs), lo, hi - lo)
                  for lo, hi in ((0, cut), (cut, n))]
            if any(lib.bezk_host_pack_wait(t) for t in ts) or not np.array_equal(rec[:, :10], rb[:, cfg.imu_body, 3:13]) \
                    or not np.array_equal(rec[:, 16:19], root[:, 0, 0:3]):
                errors.append((seed, it))
                return
            rec[:] = 0

    threads = [threading.Thread(target=worker, args=(s,)) for s in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(120)
    assert not errors and not any(t.is_alive() for t in threads)
