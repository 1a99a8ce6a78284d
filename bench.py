#!/usr/bin/env python
"""BezKick hot-path benchmark: one rollout segment = horizon x (K0 + fused post-physics step with rl_games' reward shaping in
its epilogue) + one GAE scan, at 262 144 envs per GPU (BASELINE configs[3] shard size).

    python bench.py --gpus N --steps K --warmup W                    # this repo's CUDA path (one process per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference torch path on the host CPU, same config
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR # also write the last timed rollout's outputs (.npy) to DIR

Legs of the B200 arm (ONE JSON line, rank 0):
  value / roofline   the rollout with everything resident in HBM, replayed as one CUDA graph; the fused kernel's duration is read
                     from timing events recorded INSIDE the timed graph (external event nodes around 4 of its 32 launches) and,
                     next to it, from per-launch events of an eager timed pass (roofline.eager)
  e2e                the same rollout through ``KickEnv.step`` with HOST buffers (simulator tensors, actions, targets, results and
                     the critic values of every step in pinned host memory; copies inside the timed region), same envs per GPU,
                     the reward shaping / value bootstrap / uint8 dones written by the step's epilogue as in the device leg
  learner            BASELINE configs[2]/[3]: the PPO epoch math on a 4096 x 32 rollout per GPU -- GAE, advantage moments, value
                     RunningMeanStd x2, the obs RunningMeanStd's mini_epochs x minibatches updates planned once (moments of the
                     distinct minibatches -> one all-reduce -> one merge-sequence kernel), then mini_epochs x minibatches x
                     (normalise, fused PPO loss fwd+bwd, flat 124 237-float gradient bucket all-reduce), no MLP; with its own
                     roofline and the collectives' cost (with-collectives minus without)
  cpu_baseline       the reference torch ops (oracle port) on the host cores, bounded sample of the same workload (N=1 only)
  gpu_torch_baseline the same port with CUDA tensors on the same B200 (SURVEY 2.3: the torch-eager op sequence is the bar)
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree it runs from untouched (it may be read-only)

import torch  # noqa: E402

METRIC = "task+GAE env-steps/s"
UNIT = "env-steps/s"
K0_BYTES = 144                         # SURVEY 8(d): actions 72 R + targets 72 W
POST_BYTES = 536 + 9                   # fused post-physics (prev_lin_vel buffer mode) + epilogue: value 4 R, shaped reward 4 W, done 1 W
GAE_BYTES_PER_SAMPLE = 17
POLICY_PARAMS = 124237                 # 54-400-200-100 ELU MLP + mu(18) + value(1) + sigma(18), cfg/train/bez_kickPPO.yaml:10-32
DUMP_BYTES = 32 << 20                  # --dump-outputs writes at most this much (plus the .npy headers)


def sample_envs(n, floats_per_env, seed=0):
    """Sorted ids of a fixed, seeded sample of the n envs, as many as fit DUMP_BYTES at `floats_per_env` float32 values each."""
    k = min(n, DUMP_BYTES // (4 * floats_per_env))
    if k == n:
        return torch.arange(n)
    return torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:k].sort().values


def write_outputs(out_dir, arrays):
    """name -> tensor as out_dir/<name>.npy: float64 stays float64, everything else becomes float32."""
    import numpy as np
    arrays = {k: (t.double() if t.dtype == torch.float64 else t.float()).cpu().numpy() for k, t in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise ValueError(f"{total} bytes of outputs exceed the {DUMP_BYTES}-byte dump limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--envs-per-gpu", type=int, default=262144)
    p.add_argument("--horizon", type=int, default=32)
    p.add_argument("--e2e-mode", default="auto", choices=["auto", "zero_copy", "staged", "staged_ce", "staged_pack"])
    p.add_argument("--e2e-steps", type=int, default=0, help="rollouts of the e2e leg (0: min(--steps, 10))")
    p.add_argument("--cpu-rollouts", type=int, default=8, help="rollouts of the bounded CPU-baseline sample (~10-30 s)")
    p.add_argument("--learner-envs", type=int, default=4096, help="envs per GPU of the learner leg (configs[2]: 4096 x 32)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-gpu-torch-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-learner", action="store_true")
    p.add_argument("--fusion", default="fused", choices=["fused", "split"])
    p.add_argument("--no-graph", action="store_true", help="time eager launches instead of a CUDA-graph replay of the step")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write what the last timed rollout computed (rank 0, a fixed seeded sample of its envs) as DIR/<name>.npy")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        p.error("--dump-outputs writes the outputs of the b200 arm")
    return args


def workload_config(args):
    """The `config` object: IDENTICAL in both arms (the driver compares them)."""
    n, T = args.envs_per_gpu, args.horizon
    return {"workload": f"bez_kick {n} envs/GPU (BASELINE configs[3] shard size): {T} x (pre-physics K0 + post-physics step with "
                        f"reward shaping / value bootstrap) + 1 GAE scan per rollout",
            "envs_per_gpu": n, "horizon": T, "gamma": 0.99, "tau": 0.95, "reward_scale": 0.01, "value_bootstrap": True,
            "imu_prev_lin_vel": "buffer", "cleats": False}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.sm_max = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:                       # noqa: BLE001
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap", nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:                   # noqa: BLE001
                pass
            time.sleep(0.004)

    def summary(self):
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons),
                "samples": len(sm)}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------------------------- reference arm
def torch_port_rollouts(n, horizon, rollouts, device="cpu", threads=None, warmup=1):
    """The reference torch path (oracle port of the reference's own functions, op for op; rl_games' play_steps reward path
    and discount_values as restated) on `device`: `rollouts` x (horizon task steps with reward shaping + one GAE scan) at n
    envs.  Returns (env-steps/s, seconds, threads).  device="cpu": the reference arm / cpu_baseline; a CUDA device: the same
    torch-eager op sequence on the GPU (gpu_torch_baseline)."""
    from bez_isaacgym_b200 import synthetic_gym as sg
    from oracle import rl_games_oracle as rg
    from oracle import task_oracle as to
    on_cpu = torch.device(device).type == "cpu"
    if on_cpu:
        threads = threads or os.cpu_count()
        torch.set_num_threads(threads)
    st = sg.make_state(n, seed=1234, filler=False, device=device)
    goal, ball_init, default, lower, upper = sg.make_constants(n, device)
    orc = to.KickStepOracle(n, st.root_states, st.dof_state, st.rigid_body, st.net_contact, default, lower, upper,
                            goal, ball_init, torch.tensor([0.0, 0.0], device=device), st.root_states.clone(), alias_prev_lin_vel=False)
    orc.prev_lin_vel = torch.zeros(n, 3, device=device)      # a real simulator owns the root reset: rows are unchanged
    progress, reset = sg.make_bookkeeping(n, seed=99, device=device)
    orc.progress_buf[:] = progress
    orc.reset_buf[:] = reset
    actions = sg.make_actions(n, device=device)
    rewards, values, dones, last_values, _ = sg.make_rollout(n, horizon, seed=7, device=device)
    fdones = dones.float()

    def rollout():
        cur = fdones[0]
        for t in range(horizon):
            fdones[t] = cur
            orc.pre_physics_step(actions)
            _, rew, reset_buf, time_outs = orc.post_physics_step()
            rewards[t] = rg.shape_rewards(rew, values[t], time_outs, 0.99)
            cur = reset_buf.float()
        adv = rg.discount_values(cur, last_values, fdones, values, rewards, 0.99, 0.95)
        return adv + values

    for _ in range(warmup):
        rollout()
    if not on_cpu:
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(rollouts):
        rollout()
    if not on_cpu:
        torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return n * horizon * rollouts / dt, dt, threads


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n, T, K = args.envs_per_gpu, args.horizon, max(1, args.steps)
    rate, secs, threads = torch_port_rollouts(n, T, K, warmup=max(1, args.warmup))
    sample = (f"{K} rollouts of {T} task steps (reward shaping included) + GAE at {n} envs on the host CPU, after {max(1, args.warmup)} "
              f"warm-up rollouts; the oracle port of the reference's torch functions (/root/reference is absent on the GPU box), "
              f"torch.set_num_threads({threads})")
    out = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * secs / K, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args),
           "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
           "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


# ----------------------------------------------------------------------------------------------- B200 arm: helpers
def _barrier(world, dev):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize(dev)


def _max_over_ranks(x, world, dev):
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return x


def rollout_leg(args, world, rank, dev):
    """value + roofline: the HBM-resident rollout."""
    from bez_isaacgym_b200 import bez_model as bm, ops, synthetic_gym as sg
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym
    from bez_isaacgym_b200.tasks.kick_env import KickEnv

    n, T = args.envs_per_gpu, args.horizon
    cfg = bm.default_task_cfg(n, rl_device=str(dev))
    cfg["env"]["imuPrevVelAliasing"] = False                # the general (680 B/env-step) path with a prev_lin_vel buffer
    cfg["env"]["envBase"] = rank * n                        # global env ids: the Philox reset noise does not depend on sharding
    cfg["seed"] = 42

    class OwnedRootSim(SyntheticGym):
        owns_root_reset = True                              # as with Isaac Gym: the simulator restores root states

    sim = OwnedRootSim(n, device=str(dev), seed=1234 + rank, filler=True)
    env = KickEnv(cfg, str(dev), 0, True, sim=sim, fusion=args.fusion)
    progress, reset = sg.make_bookkeeping(n, seed=99 + rank, device=dev)
    env.progress_buf.copy_(progress); env.reset_buf.copy_(reset)
    actions = sg.make_actions(n, seed=4321 + rank, device=dev)
    rewards, values, _, last_values, _ = sg.make_rollout(n, T, seed=7 + rank, device=dev)
    dones = torch.zeros(T + 1, n, dtype=torch.uint8, device=dev)     # slot t = dones at the START of step t; slot T = after the last
    advs, rets = torch.empty_like(rewards), torch.empty_like(rewards)
    stream = torch.cuda.current_stream(dev)
    fused = args.fusion == "fused"
    launches_per_step = T * (2 if fused else 3) + 1
    ev_pairs = []                                           # (start, end) around single post-physics launches

    def bench_step(mark=(), external=False):
        dones[0].copy_(dones[T])                            # the dones carried over from the previous rollout (torch copy, N bytes)
        for t in range(T):
            env.pre_physics_step(actions)
            env.sim.simulate()
            if fused:                                       # a16: shaped reward -> rewards[t], uint8 done -> dones[t+1], in the epilogue
                env.set_rollout_targets(values=values[t], shaped_rewards=rewards[t], dones_u8=dones[t + 1], gamma=0.99,
                                        scale_value=0.01)
            if t in mark:
                cur = torch.cuda.current_stream(dev)        # the capture stream while a graph is being recorded
                e0 = torch.cuda.Event(enable_timing=True, external=external)
                e1 = torch.cuda.Event(enable_timing=True, external=external)
                e0.record(cur)
                env.post_physics_step()
                e1.record(cur)
                ev_pairs.append((e0, e1))
            else:
                env.post_physics_step()
        ops.gae(rewards, values, dones[:T], last_values, dones[T], 0.99, 0.95, advs, rets)

    W = max(3, args.warmup)
    for _ in range(W):
        bench_step()
    _barrier(world, dev)
    graph, in_graph_events = None, False
    marks = (T // 3, 2 * T // 3)                            # 2 of the 32 launches carry timing events inside the graph
    if not args.no_graph:
        # the step is 65 dependent launches of 7..45 us kernels: replaying it as ONE CUDA graph removes the CPU-side
        # launch cost and most of the inter-kernel gaps (the kernels, arguments and work are identical)
        try:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                bench_step(mark=marks, external=True)
            in_graph_events = True
        except Exception as exc:                            # noqa: BLE001  (external event nodes unsupported: plain capture)
            print(f"bench: in-graph timing events unavailable ({exc!r}); falling back", file=sys.stderr)
            del ev_pairs[:]
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                bench_step()
        stream = torch.cuda.current_stream(dev)
        graph.replay()
    _barrier(world, dev)
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    _barrier(world, dev)
    start.record(stream)
    for _ in range(args.steps):
        if graph is not None:
            graph.replay()
        else:
            bench_step(mark=range(T))
    end.record(stream)
    _barrier(world, dev)
    ms = start.elapsed_time(end)
    sampler.stop_flag = True
    sampler.join()
    outputs = None
    if args.dump_outputs and rank == 0:
        # the last timed rollout's results, taken before the passes below step the envs again: the PD targets of K0, what the
        # post-physics step hands back, the dof rows its masked reset wrote, the epilogue's rollout storage, the GAE scan's output
        idx = sample_envs(n, 18 + 54 + 4 + 36 + 2 * T + (2 * T + 1 if fused else 0))
        per_env = {"pd_targets": env.targets, "obs": env._observations_out(), "rew": env.rew_buf, "reset": env.reset_buf,
                   "time_outs": env.timeout_buf, "progress": env.progress_buf, "dof_state": env.dof_state.view(n, 36)}
        per_step = {"advantages": advs.view(T, n), "returns": rets.view(T, n)}
        if fused:
            per_step.update(shaped_rewards=rewards.view(T, n), dones=dones)
        outputs = {k: t[idx.to(t.device)].cpu() for k, t in per_env.items()}
        outputs.update({k: t[:, idx.to(t.device)].cpu() for k, t in per_step.items()})
    post_graph_ms = post_eager_ms = eager_step_ms = in_region_ms = None
    if graph is not None and in_graph_events:
        try:
            in_region_ms = sum(a.elapsed_time(b) for a, b in ev_pairs) / len(ev_pairs)     # the LAST replay of the timed region
        except Exception:                                   # noqa: BLE001
            in_region_ms = None
    if graph is not None:
        del ev_pairs[:]
        # eager timed pass: the same steps launched one by one, per-launch events around every post-physics launch
        ke = min(args.steps, 10)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        _barrier(world, dev)
        e0.record(stream)
        for _ in range(ke):
            bench_step(mark=range(T))
        e1.record(stream)
        _barrier(world, dev)
        eager_step_ms = e0.elapsed_time(e1) / ke
    post_eager_ms = sum(a.elapsed_time(b) for a, b in ev_pairs) / len(ev_pairs)
    if graph is not None:
        # back-to-back duration: a graph holding only the T post-physics launches of one rollout, replayed between two events
        # right after the timed region.  An event pair around ONE launch (in_region / eager) also times the launch latency the
        # event nodes expose (no programmatic-dependent-launch overlap across an event node): ~7 us on a 36 us kernel.
        pg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(pg):
            for _ in range(T):
                env.post_physics_step()
        pg.replay()
        _barrier(world, dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(10):
            pg.replay()
        e1.record(stream)
        _barrier(world, dev)
        post_graph_ms = e0.elapsed_time(e1) / (10 * T)
    reset_rate = float(env.reset_buf.float().mean())
    ms = _max_over_ranks(ms, world, dev)
    value = n * world * T * args.steps / (ms * 1e-3)

    peak, peak_src = peaks()
    post_ms = post_graph_ms if graph is not None else post_eager_ms
    achieved = POST_BYTES * n / (post_ms * 1e-3) / 1e9
    eager_gbs = POST_BYTES * n / (post_eager_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "bezk::task_tile_kernel<7> (fused post-physics + reward-shaping epilogue)" if fused
                else "bezk::task_tile_kernel<3>+<4>", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "algorithmic_bytes_per_env": POST_BYTES, "envs_per_launch": n,
                "avg_launch_ms": post_ms, "peak_source": peak_src,
                "timing": ("CUDA events around a replayed graph of one rollout's 32 post-physics launches (back to back, as in the timed "
                           "graph), taken right after the timed region; in_region / eager = event pairs around single launches")
                if graph is not None else "per-launch CUDA events inside the eager timed region",
                "in_region": None if in_region_ms is None else {
                    "avg_launch_ms": in_region_ms, "frac": POST_BYTES * n / (in_region_ms * 1e-3) / 1e9 / peak,
                    "timing": f"timing events recorded as external event nodes INSIDE the replayed graph of the timed region, around the "
                              f"post-physics launches of env steps {list(marks)}, read after the last timed replay (each pair also "
                              f"times the launch latency its event nodes expose)"},
                "eager": {"avg_launch_ms": post_eager_ms, "achieved": eager_gbs, "frac": eager_gbs / peak,
                          "timing": "per-launch CUDA events around every post-physics launch of an eager (no graph) timed pass"},
                "whole_step_gbs": ((K0_BYTES + POST_BYTES) * n * T + GAE_BYTES_PER_SAMPLE * n * T) * args.steps / (ms * 1e-3) / 1e9}
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file):
        with open(traffic_file) as f:
            roofline["traffic"] = json.load(f).get("post_physics_bytes_per_launch")
    run = {"launch": "cuda_graph_replay" if graph is not None else "eager", "fusion": args.fusion,
           "l2": "inputs larger than L2 (state footprint ~%.0f MB/GPU, 126 MB L2)" % (n * 4 * (26 + 36 + 16 * bm.BODIES_NO_CLEATS) / 1e6),
           "ms_per_step_eager_with_events": eager_step_ms, "reset_rate_per_step": reset_rate,
           "parallelism": f"env-sharded x{world}, no data-path collective (the exchanges are in the learner leg)"}
    out = dict(value=value, ms_per_step=ms / args.steps, warmup=W, roofline=roofline, run=run, clocks=sampler.summary(),
               gpu_launches=launches_per_step * args.steps, outputs=outputs)
    del env, sim, graph
    torch.cuda.empty_cache()
    return out


def e2e_leg(args, world, rank, dev):
    """The same rollout through the reference-facing call with HOST buffers."""
    from bez_isaacgym_b200 import bez_model as bm, ops, synthetic_gym as sg
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym
    from bez_isaacgym_b200.tasks.kick_env import KickEnv

    class OwnedRootSim(SyntheticGym):
        owns_root_reset = True

    n, T = args.envs_per_gpu, args.horizon
    steps = args.e2e_steps or min(args.steps, 10)
    mode = args.e2e_mode
    # "auto": KickEnv picks staged_pack when this rank has >= 8 host cores to gather with, else staged_ce (copy-engine pulls)
    hcfg = bm.default_task_cfg(n, use_gpu_pipeline=False, rl_device="cpu")
    hcfg["env"]["imuPrevVelAliasing"] = False
    hcfg["env"]["hostPipeline"] = mode
    hcfg["env"]["envBase"] = rank * n
    hsim = OwnedRootSim(n, device=str(dev), seed=1234 + rank, host=True, filler=True)
    henv = KickEnv(hcfg, str(dev), 0, True, sim=hsim, fusion=args.fusion)
    hact = sg.make_actions(n, seed=1).pin_memory()
    # host side of the rollout: the critic values of every step and the bootstrap values (the policy lives with the simulator on
    # the host); device side: the rollout storage the step's reward epilogue and the GAE scan work on
    _, hv, _, hlv, _ = [t.pin_memory() for t in sg.make_rollout(n, T, seed=3)]
    d_r, d_v, d_lv = (torch.empty_like(t, device=dev) for t in (hv, hv, hlv))
    d_d = torch.zeros(T + 1, n, dtype=torch.uint8, device=dev)       # slot t = dones at the START of step t
    d_adv, d_ret = torch.empty_like(d_r), torch.empty_like(d_r)
    h_adv, h_ret = torch.empty_like(hv).pin_memory(), torch.empty_like(hv).pin_memory()
    gae_h2d = sum(t.numel() * t.element_size() for t in (hv, hlv))
    gae_d2h = sum(t.numel() * t.element_size() for t in (h_adv, h_ret))
    vals_in_step = 0 if henv.host_pipeline == "staged_pack" else n * 4      # staged_pack: the values ride inside the records

    def e2e_step():
        d_d[0].copy_(d_d[T])
        for t in range(T):
            # a16 in the step's epilogue (shaped reward -> d_r[t], uint8 done -> d_d[t + 1]), values arriving from the host
            henv.set_rollout_targets(values=hv[t].view(-1), shaped_rewards=d_r[t].view(-1), dones_u8=d_d[t + 1], gamma=0.99,
                                     scale_value=0.01)
            henv.step(hact)
        d_v.copy_(hv, non_blocking=True); d_lv.copy_(hlv, non_blocking=True)
        ops.gae(d_r, d_v, d_d[:T], d_lv, d_d[T], 0.99, 0.95, d_adv, d_ret)
        h_adv.copy_(d_adv, non_blocking=True); h_ret.copy_(d_ret, non_blocking=True)
        torch.cuda.synchronize(dev)

    e2e_step()
    henv.reset_link_counters()
    _barrier(world, dev)
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_step()
    _barrier(world, dev)
    dt = _max_over_ranks(time.perf_counter() - t0, world, dev)
    link = henv.link_counters()
    out = {"value": n * world * T * steps / dt, "unit": UNIT,
           "h2d_bytes_per_step": link["h2d_bytes"] // steps + gae_h2d + T * vals_in_step,
           "d2h_bytes_per_step": link["d2h_bytes"] // steps + gae_d2h,
           "envs_per_gpu": n, "steps": steps, "ms_per_step": 1e3 * dt / steps, "host_pipeline": henv.host_pipeline,
           "host_pack_threads": getattr(henv, "host_pack_threads", None), "byte_count": link["how"],
           "note": "KickEnv.step with use_gpu_pipeline=False: simulator tensors, actions and PD targets in pinned HOST memory, "
                   "obs / rew / reset / time_outs handed back on the host every env step (one stream sync per step); the step's "
                   "critic values come from the host (inside the packed records, or one extra copy per step) and the reward "
                   "shaping / value bootstrap / uint8 dones are written by the step's epilogue into device rollout storage; "
                   "values + bootstrap values H2D and advantages / returns D2H per GAE scan; bytes per step = per rollout, this rank"}
    del henv, hsim
    torch.cuda.empty_cache()
    return out


def learner_leg(args, world, rank, dev):
    """BASELINE configs[2]/[3]: PPO epoch math on an (T x envs) rollout per GPU with the path's collectives, no MLP."""
    import torch.distributed as dist
    from bez_isaacgym_b200 import learner as L, ops, synthetic_gym as sg
    n, T, mbs, mini_epochs = args.learner_envs, args.horizon, 32768, 5
    M = n * T
    if M % mbs:
        mbs = M
    E = mbs // T
    nmb = M // mbs
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    rewards, values, dones, last_values, last_dones = sg.make_rollout(n, T, seed=21 + rank, device=dev)
    obses = torch.randn(T, n, 54, generator=g, device=dev) * 2 + 0.5
    mb = {k: v.to(dev) for k, v in sg.make_minibatch(M, seed=5 + rank).items()}
    tm = lambda x, w: x.view(T, n, w) if w > 1 else x.view(T, n)          # noqa: E731  (time-major rollout storage)
    actions, old_mu, old_sigma = tm(mb["actions"], 18), tm(mb["old_mu"], 18), tm(mb["old_sigma"], 18)
    old_neglogp = tm(mb["old_neglogp"], 1)
    mu_net, val_net, logstd = mb["mu"][:mbs].contiguous(), mb["values"].view(-1)[:mbs].contiguous(), mb["logstd"]
    advs, rets = torch.empty_like(rewards), torch.empty_like(rewards)
    adv_n = torch.empty(T, n, device=dev)
    vals_n, rets_n = torch.empty_like(values), torch.empty_like(values)
    norm_obs = torch.empty(nmb, mbs, 54, device=dev)                         # one mini-epoch of network inputs
    bucket = torch.randn(POLICY_PARAMS + 1, generator=g, device=dev)       # flat gradient bucket (+ the KL scalar for the shared LR)
    stats = torch.empty(8, dtype=torch.float64, device=dev)
    part = torch.empty(ops.ppo_scratch_doubles(), dtype=torch.float64, device=dev)
    kc = ops.make_ppo_cfg()
    gmu, gv, gls = torch.empty(mbs, 18, device=dev), torch.empty(mbs, device=dev), torch.empty(18, device=dev)
    stream = torch.cuda.current_stream(dev)

    def make_epoch(group):
        obs_rms = L.RunningMeanStd(54, process_group=group).to(dev)
        val_rms = L.RunningMeanStd(1, process_group=group).to(dev)
        counters = {"collectives": 0, "bytes": 0}

        def epoch():
            ops.gae(rewards, values, dones, last_values, last_dones, 0.99, 0.95, advs, rets)
            L.normalize_advantages(rets, values, process_group=group, out=adv_n.view(-1))       # moments -> all-reduce -> normalise
            val_rms(values, out=vals_n); val_rms(rets, out=rets_n)                               # two train-mode updates per epoch
            # the obs normaliser's 5 x 4 train-mode updates: the moments of the 4 distinct minibatches ONCE (+ one all-reduce of
            # all of them), one merge kernel for the whole sequence, then ONE normalise launch per mini-epoch (each minibatch
            # with the statistics after ITS update)
            views = [obses[:, i * E:(i + 1) * E] for i in range(nmb)]
            obs_rms.plan(views, list(range(nmb)) * mini_epochs)
            for me in range(mini_epochs):
                obs_rms.planned_group(me * nmb, views, out=norm_obs)
                for i in range(nmb):
                    sl = slice(i * E, (i + 1) * E)
                    ops.ppo_loss_slabs(actions[:, sl], mu_net, logstd, old_mu[:, sl], old_sigma[:, sl], val_net, vals_n[:, sl],
                                       rets_n[:, sl], old_neglogp[:, sl], adv_n[:, sl], kc, stats, part, grad_mu=gmu,
                                       grad_values=gv, grad_logstd=gls)
                    if group is not None:
                        dist.all_reduce(bucket, group=group)                                   # PPO gradients (+ KL), one flat bucket
        if group is not None:
            counters["collectives"] = 3 + 1 + mini_epochs * nmb
            counters["bytes"] = 8 * (3 + 2 * 3) + 8 * 109 * nmb + mini_epochs * nmb * 4 * (POLICY_PARAMS + 1)
        return epoch, counters

    def timed(epoch, iters):
        for _ in range(2):
            epoch()
        _barrier(world, dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(iters):
            epoch()
        b.record(stream)
        _barrier(world, dev)
        return _max_over_ranks(a.elapsed_time(b) / iters, world, dev)

    iters = max(3, min(args.steps, 20))
    local_epoch, _ = make_epoch(None)
    ms_local = timed(local_epoch, iters)
    ms_graph = None
    try:                                                    # the collective-free chain also as one CUDA graph (launch-bound sizes)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            local_epoch()
        ms_graph = timed(gr.replay, iters)
    except Exception:                                       # noqa: BLE001
        ms_graph = None
    ms_dist, counters = ms_local, {"collectives": 0, "bytes": 0}
    ms_dist_graph = None
    if world > 1:
        dist_epoch, counters = make_epoch(dist.group.WORLD)
        ms_dist = timed(dist_epoch, iters)
        # the same epoch, collectives included, replayed as ONE CUDA graph: eager launches expose every rank's Python jitter at each of
        # the 43 collectives (the slowest rank sets the pace); a graph leaves only the NCCL kernels' own latency
        gd, ok = None, 1
        try:
            gd = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gd, capture_error_mode="thread_local"):
                dist_epoch()
        except Exception as exc:                            # noqa: BLE001
            print(f"bench: NCCL graph capture of the learner epoch unavailable on rank {rank} ({exc!r})", file=sys.stderr)
            ok = 0
        # replay only if EVERY rank captured: a rank that skipped the replays would leave the others waiting in their all-reduces
        flag = torch.tensor([ok], device=dev, dtype=torch.int32)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 1:
            ms_dist_graph = timed(gd.replay, iters)
    graph_ms = ms_dist_graph if world > 1 else ms_graph
    best, best_how = (graph_ms, "cuda_graph_replay (NCCL collectives captured)" if world > 1 else "cuda_graph_replay") \
        if graph_ms is not None else (ms_dist, "eager")
    # per-kernel timings at the minibatch size (graph-replayed x20) for the leg's roofline: the kernel furthest below peak
    def ktime(fn, reps=20):
        for _ in range(3):
            fn()
        gk = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gk):
            for _ in range(reps):
                fn()
        gk.replay()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(5):
            gk.replay()
        b.record(stream)
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / (5 * reps)
    rms = L.RunningMeanStd(54).to(dev)
    sl = slice(0, E)
    k_rms = ktime(lambda: rms(obses[:, sl], out=norm_obs[0]))
    k_ppo = ktime(lambda: ops.ppo_loss_slabs(actions[:, sl], mu_net, logstd, old_mu[:, sl], old_sigma[:, sl], val_net, vals_n[:, sl],
                                             rets_n[:, sl], old_neglogp[:, sl], adv_n[:, sl], kc, stats, part, grad_mu=gmu,
                                             grad_values=gv, grad_logstd=gls))
    k_gae = ktime(lambda: ops.gae(rewards, values, dones, last_values, last_dones, 0.99, 0.95, advs, rets))
    peak, _ = peaks()
    kernels = {"rms_train_forward": {"ms": k_rms, "bytes": 432 * mbs}, "ppo_loss_fwd_bwd": {"ms": k_ppo, "bytes": 384 * mbs},
               "gae": {"ms": k_gae, "bytes": GAE_BYTES_PER_SAMPLE * M}}
    for k in kernels.values():
        k["gbs"] = k["bytes"] / (k["ms"] * 1e-3) / 1e9
        k["frac"] = k["gbs"] / peak
    worst = min(kernels, key=lambda k: kernels[k]["frac"])
    return {"workload": f"PPO epoch math per GPU on a {T} x {n} rollout: GAE, advantage moments + normalise, value RunningMeanStd x2, "
                        f"the {mini_epochs} x {nmb} train-mode updates of the obs RunningMeanStd planned once (moments of the {nmb} distinct "
                        f"minibatches on slab views, one all-reduce, one merge-sequence kernel), then {mini_epochs} x {nmb} minibatches of "
                        f"{mbs} x (normalise with the statistics of that update, fused PPO loss fwd+bwd, {POLICY_PARAMS}-float gradient "
                        f"bucket all-reduce); no MLP",
            "envs_per_gpu": n, "horizon": T, "minibatch": mbs, "mini_epochs": mini_epochs, "n_gpus": world,
            "ms_per_epoch": best, "launch": best_how,
            "ms_per_epoch_eager": ms_dist, "ms_per_epoch_eager_no_collectives": ms_local,
            "ms_per_epoch_graph": ms_dist_graph if world > 1 else ms_graph, "ms_per_epoch_graph_no_collectives": ms_graph,
            "collective_us_per_epoch_eager": (ms_dist - ms_local) * 1e3,
            "collective_us_per_epoch_graph": None if (ms_dist_graph is None or ms_graph is None) else (ms_dist_graph - ms_graph) * 1e3,
            "collectives_per_epoch": counters["collectives"],
            "collective_bytes_per_epoch": counters["bytes"], "samples_per_s": M * world / (best * 1e-3),
            "env_steps_per_s": M * world / (best * 1e-3),
            "timing": "CUDA events around `iters` epochs after 2 warm-up epochs, max over ranks; collective cost = with - without",
            "roofline": {"bound": "hbm (launch-latency-bound at this size)", "kernel": worst, "achieved": kernels[worst]["gbs"],
                         "peak": peak, "unit": "GB/s", "frac": kernels[worst]["frac"], "per_kernel": kernels,
                         "timing": "each kernel chain graph-replayed x20 between CUDA events, minibatch = 32768 samples"}}


def run_b200(args):
    import torch.distributed as dist
    import __graft_entry__ as ge
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # stdout carries the ONE JSON line: NCCL's own log lines (whatever NCCL_DEBUG level the caller chose -- it is NOT
        # touched here) go to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    ge.build()

    roll = rollout_leg(args, world, rank, dev)
    e2e = None if args.no_e2e else e2e_leg(args, world, rank, dev)
    learner = None if args.no_learner else learner_leg(args, world, rank, dev)

    cpu_baseline = gpu_torch = None
    n, T = args.envs_per_gpu, args.horizon
    if rank == 0 and world == 1 and not args.no_gpu_torch_baseline:
        rate, secs, _ = torch_port_rollouts(n, T, 2, device=str(dev))
        gpu_torch = {"value": rate, "unit": UNIT, "kind": "port", "device": torch.cuda.get_device_name(dev),
                     "sample": f"2 rollouts of {T} task steps + GAE at {n} envs ({secs:.2f} s): the reference's torch-eager op "
                               f"sequence (oracle port) with CUDA tensors on the same GPU"}
        torch.cuda.empty_cache()
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rate, secs, threads = torch_port_rollouts(n, T, args.cpu_rollouts)
        cpu_baseline = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": f"{args.cpu_rollouts} rollouts of {T} task steps + GAE at {n} envs ({secs:.1f} s), reference torch ops "
                                  f"(oracle port; /root/reference is absent on the GPU box) with torch.set_num_threads({threads})"}

    if rank == 0:
        out = {"metric": METRIC, "value": roll["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": roll["warmup"],
               "ms_per_step": roll["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
               "data": "synthetic", "config": workload_config(args), "run": roll["run"], "clocks": roll["clocks"],
               "gpu_launches": roll["gpu_launches"], "roofline": roll["roofline"], "e2e": e2e, "learner": learner,
               "cpu_baseline": cpu_baseline, "gpu_torch_baseline": gpu_torch}
        if args.dump_outputs:
            write_outputs(args.dump_outputs, roll["outputs"])
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
