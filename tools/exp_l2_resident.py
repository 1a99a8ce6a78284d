"""A/B of the L2 residency of the fused step's carried state (BEZK_L2_RESIDENT=0 / 1), in one GPU session.

Each arm runs in its own process (the knob is read once per process), the arms alternate, ``--repeats`` rounds:
  * the unmodified ``bench.py`` rollout leg (``--no-e2e --no-learner --no-cpu-baseline --no-gpu-torch-baseline``) at each
    ``--sizes`` env count: ``value`` and ``roofline.avg_launch_ms`` (the fused kernel back to back in a replayed graph);
  * the walk / orient fused steps at 262 144 envs (32 back-to-back launches replayed as a graph, median of 5 replays of 5).
Writes ``<out>/r03_l2_resident.jsonl`` (one line per run, plus a header line with the card, its power limit and clocks) and
prints a per-arm summary (median, spread = max - min)."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def sibling_child(n):
    import torch
    sys.path.insert(0, ROOT)
    from bez_isaacgym_b200 import bez_model as bm, synthetic_gym as sg, tasks as T
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym

    class Sim(SyntheticGym):
        owns_root_reset = True

    dev = torch.device("cuda:0")
    out = {}
    for task, cls in (("walk", T.WalkEnv), ("orient", T.OrientEnv)):
        cfg = bm.default_task_cfg(n, task=task)
        cfg["env"]["imuPrevVelAliasing"] = False
        env = cls(cfg, "cuda:0", 0, True, sim=Sim(n, device="cuda:0", task=task))
        p, r = sg.make_bookkeeping(n, device=dev, max_episode_length=600)
        env.progress_buf.copy_(p); env.reset_buf.copy_(r)
        for _ in range(5):
            env.post_physics_step()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(32):
                env.post_physics_step()
        g.replay(); torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(5):
                g.replay()
            b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) / 160 * 1e3)
        out[task + "_us"] = statistics.median(ts)
        env.close()
        del env, g
        torch.cuda.empty_cache()
    print(json.dumps(out))


def last_json(text):
    for line in reversed(text.splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError("no JSON line in:\n" + text[-2000:])


def run(cmd, arm, timeout):
    env = dict(os.environ, BEZK_L2_RESIDENT=str(arm))
    p = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=timeout)
    if p.returncode != 0:
        raise RuntimeError(f"{cmd} failed ({p.returncode}):\n{p.stderr[-3000:]}")
    return last_json(p.stdout)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as exc:
        return f"unavailable: {exc!r}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--child-siblings", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--sizes", default="65536,262144,1048576")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    if args.child_siblings:
        return sibling_child(args.child_siblings)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "r03_l2_resident.jsonl")
    rows = []
    with open(path, "w") as f:
        f.write(json.dumps({"gpu": gpu_info(), "sizes": args.sizes, "repeats": args.repeats, "steps": args.steps}) + "\n")
        for rep in range(args.repeats):
            for n in [int(x) for x in args.sizes.split(",")]:
                for arm in ((0, 1) if rep % 2 == 0 else (1, 0)):
                    r = run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(args.steps), "--envs-per-gpu", str(n),
                             "--no-e2e", "--no-learner", "--no-cpu-baseline", "--no-gpu-torch-baseline"], arm, 900)
                    row = {"kind": "bench", "envs": n, "l2_resident": arm, "rep": rep, "value": r["value"],
                           "avg_launch_ms": r["roofline"]["avg_launch_ms"], "ms_per_step": r.get("ms_per_step"),
                           "clocks": r.get("clocks")}
                    rows.append(row); f.write(json.dumps(row) + "\n"); f.flush()
                    print(json.dumps(row), flush=True)
            for arm in ((0, 1) if rep % 2 == 0 else (1, 0)):
                r = run([sys.executable, os.path.abspath(__file__), "--child-siblings", "262144"], arm, 600)
                row = {"kind": "siblings", "envs": 262144, "l2_resident": arm, "rep": rep, **r}
                rows.append(row); f.write(json.dumps(row) + "\n"); f.flush()
                print(json.dumps(row), flush=True)
        f.write(json.dumps({"gpu_after": gpu_info()}) + "\n")
    print("gpu:", gpu_info())
    keys = [("bench", n, k) for n in [int(x) for x in args.sizes.split(",")] for k in ("value", "avg_launch_ms")]
    keys += [("siblings", 262144, k) for k in ("walk_us", "orient_us")]
    for kind, n, k in keys:
        arms = {}
        for arm in (0, 1):
            v = [r[k] for r in rows if r["kind"] == kind and r["envs"] == n and r["l2_resident"] == arm]
            arms[arm] = (statistics.median(v), max(v) - min(v)) if v else (float("nan"), float("nan"))
        (m0, s0), (m1, s1) = arms[0], arms[1]
        print(f"{kind:8s} {n:8d} {k:14s} off {m0:.6g} (spread {s0:.3g})  on {m1:.6g} (spread {s1:.3g})  on/off {m1 / m0:.4f}")


if __name__ == "__main__":
    sys.exit(main())
