"""A/B of the fused step's episode accumulators (``bezk_post_physics_rollout_ep``) in one GPU session.

At each ``--sizes`` env count a KickEnv (GPU pipeline, synthetic state) steps with the rollout targets armed as
``A2CAgent.play_steps`` arms them (critic values, shaped rewards, uint8 dones), arm A without and arm B with the episode targets
(returns, lengths, per-step partials).  The arms alternate, ``--repeats`` rounds; each measurement is 32 back-to-back fused steps
replayed as a CUDA graph (median of 5 replays of 5).  The L2 policy picks its variant per size as in production (the hinted
kernel at 262 144 envs on B200, the plain one at 65 536 and 1 048 576).  It also times the meter fold
(``bezk_episode_meter_update``) over T = 32 steps of partials, eagerly and replayed in a CUDA graph.  Writes ``<out>/r04_episode_stats.jsonl`` (a header line with the
card, its power limit and clocks, then one line per measurement) and ``<out>/r04_episode_stats.md`` (the medians)."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as exc:
        return f"unavailable: {exc!r}"


def _graph_us(torch, fn, launches=32):
    for _ in range(3):
        fn()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(launches):
            fn()
    g.replay()
    torch.cuda.synchronize()
    ts = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(5):
            g.replay()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / (5 * launches) * 1e3)
    return statistics.median(ts)


def measure(n, repeats, horizon):
    import torch
    from bez_isaacgym_b200 import bez_model as bm, ops, synthetic_gym as sg
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym
    from bez_isaacgym_b200.tasks import KickEnv

    dev = torch.device("cuda:0")
    env = KickEnv(bm.default_task_cfg(n), "cuda:0", 0, True, sim=SyntheticGym(n, device="cuda:0"))
    p, r = sg.make_bookkeeping(n, device=dev)
    env.progress_buf.copy_(p)
    env.reset_buf.copy_(r)
    w = (n + 31) // 32
    values, shaped = torch.randn(n, device=dev), torch.empty(n, device=dev)
    dones = torch.empty(n, dtype=torch.uint8, device=dev)
    ret, length = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    part = torch.zeros(horizon, 3, w, dtype=torch.float64, device=dev)
    arms = {
        "rollout": dict(values=values, shaped_rewards=shaped, dones_u8=dones),
        "rollout+episode": dict(values=values, shaped_rewards=shaped, dones_u8=dones, episode_returns=ret, episode_lengths=length,
                                episode_partials=part[0]),
    }
    rows = []
    for rep in range(repeats):
        for arm in (list(arms) if rep % 2 == 0 else list(arms)[::-1]):
            env.set_rollout_targets(**arms[arm])
            rows.append({"kind": "step", "envs": n, "arm": arm, "rep": rep, "us": _graph_us(torch, env.post_physics_step)})
            print(json.dumps(rows[-1]), flush=True)
    env.set_rollout_targets()
    mean2, size2 = torch.zeros(2, device=dev), torch.zeros(2, dtype=torch.long, device=dev)
    for rep in range(repeats):
        ops.episode_meter_update(part, n, 100, mean2, size2)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(100):
            ops.episode_meter_update(part, n, 100, mean2, size2)
        b.record()
        torch.cuda.synchronize()
        rows.append({"kind": "fold", "envs": n, "steps": horizon, "rep": rep, "us": a.elapsed_time(b) / 100 * 1e3,
                     "graph_us": _graph_us(torch, lambda: ops.episode_meter_update(part, n, 100, mean2, size2))})
        print(json.dumps(rows[-1]), flush=True)
    env.close()
    del env
    torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="65536,262144,1048576")
    ap.add_argument("--repeats", type=int, default=4)
    ap.add_argument("--horizon", type=int, default=32)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("exp_episode_stats needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    sizes = [int(x) for x in args.sizes.split(",")]
    rows = []
    with open(os.path.join(args.out, "r04_episode_stats.jsonl"), "w") as f:
        f.write(json.dumps({"gpu": info, "device": torch.cuda.get_device_name(0), "sizes": sizes, "repeats": args.repeats,
                            "horizon": args.horizon}) + "\n")
        for n in sizes:
            for row in measure(n, args.repeats, args.horizon):
                rows.append(row)
                f.write(json.dumps(row) + "\n")
        f.write(json.dumps({"gpu_after": gpu_info()}) + "\n")
    lines = [f"# Episode accumulators in the fused step: A/B ({info})", "",
             f"Fused KickEnv step with the rollout targets armed, without / with the episode targets; 32 launches per CUDA-graph "
             f"replay, median over {args.repeats} alternated rounds (each the median of 5 x 5 replays). Fold: "
             f"`bezk_episode_meter_update` over T = {args.horizon} steps of partials: eager = mean of 100 back-to-back calls from "
             f"Python (host API time included), graph = the same call replayed in a CUDA graph (32 per replay); medians over rounds.",
             "", "| envs | step, rollout (us) | step, rollout + episode (us) | delta | spread A / B (us) | fold eager (us) | "
             "fold graph (us) |", "|---:|---:|---:|---:|---:|---:|---:|"]
    for n in sizes:
        a = [r["us"] for r in rows if r["kind"] == "step" and r["envs"] == n and r["arm"] == "rollout"]
        b = [r["us"] for r in rows if r["kind"] == "step" and r["envs"] == n and r["arm"] == "rollout+episode"]
        fo = [r["us"] for r in rows if r["kind"] == "fold" and r["envs"] == n]
        fg = [r["graph_us"] for r in rows if r["kind"] == "fold" and r["envs"] == n]
        ma, mb = statistics.median(a), statistics.median(b)
        lines.append(f"| {n} | {ma:.2f} | {mb:.2f} | {100 * (mb / ma - 1):+.1f} % | {max(a) - min(a):.2f} / {max(b) - min(b):.2f} | "
                     f"{statistics.median(fo):.2f} | {statistics.median(fg):.2f} |")
    text = "\n".join(lines) + "\n"
    with open(os.path.join(args.out, "r04_episode_stats.md"), "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    sys.exit(main())
