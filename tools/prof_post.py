#!/usr/bin/env python
"""ncu target: a few fused post-physics launches at --envs through KickEnv (no graph), nothing else."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from bez_isaacgym_b200 import bez_model as bm, synthetic_gym as sg  # noqa: E402
from bez_isaacgym_b200.synthetic_sim import SyntheticGym  # noqa: E402
from bez_isaacgym_b200.tasks.kick_env import KickEnv  # noqa: E402


class Sim(SyntheticGym):
    owns_root_reset = True


ap = argparse.ArgumentParser()
ap.add_argument("--envs", type=int, default=262144)
ap.add_argument("--launches", type=int, default=8)
a = ap.parse_args()
n, dev = a.envs, torch.device("cuda:0")
cfg = bm.default_task_cfg(n)
cfg["env"]["imuPrevVelAliasing"] = False
env = KickEnv(cfg, "cuda:0", 0, True, sim=Sim(n, device="cuda:0"))
p, r = sg.make_bookkeeping(n, device=dev)
env.progress_buf.copy_(p); env.reset_buf.copy_(r)
vals = torch.randn(n, device=dev); sh = torch.empty(n, device=dev); dn = torch.empty(n, dtype=torch.uint8, device=dev)
env.set_rollout_targets(values=vals, shaped_rewards=sh, dones_u8=dn)
for _ in range(a.launches):
    env.post_physics_step()
torch.cuda.synchronize()
print("ok")
