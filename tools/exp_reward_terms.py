"""A/B of the fused step's reward term sums (``bezk_post_physics_rollout_ep_terms``) in one GPU session.

For each ``--cases`` entry (task:envs) an env (GPU pipeline, synthetic state) steps with the rollout and episode targets armed as
``A2CAgent.play_steps`` arms them, in four arms: EP (episode accumulators), EP + reward terms, EP + outcome counts and EP + outcome
counts + reward terms.  The arms alternate (the order reverses every round), ``--repeats`` rounds; each measurement is 32
back-to-back fused steps replayed as a CUDA graph (median of 5 replays of 5).  The L2 policy picks its variant per size as in
production.  It also times the fold (``bezk_reward_terms_update``) over T = 32 steps of partials, replayed in a CUDA graph.  Writes
``<out>/r07_reward_terms.jsonl`` (a header line with the card, its power limit and clocks, then one line per measurement) and
``<out>/r07_reward_terms.md`` (the medians)."""
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


ARMS = ("ep", "ep+terms", "ep+outcome", "ep+outcome+terms")


def measure(task, n, repeats, horizon):
    import torch
    from bez_isaacgym_b200 import bez_model as bm, ops, synthetic_gym as sg
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym
    from bez_isaacgym_b200 import tasks

    dev = torch.device("cuda:0")
    cls = {"kick": tasks.KickEnv, "walk": tasks.WalkEnv, "orient": tasks.OrientEnv}[task]
    env = cls(bm.default_task_cfg(n, task=task), "cuda:0", 0, True, sim=SyntheticGym(n, device="cuda:0", task=task))
    p, r = sg.make_bookkeeping(n, device=dev)
    env.progress_buf.copy_(p)
    env.reset_buf.copy_(r)
    w, k, kt = (n + 31) // 32, len(env.OUTCOMES), len(env.REWARD_TERMS)
    values, shaped = torch.randn(n, device=dev), torch.empty(n, device=dev)
    dones = torch.empty(n, dtype=torch.uint8, device=dev)
    ret, length = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    part = torch.zeros(horizon, 3, w, dtype=torch.float64, device=dev)
    oc = torch.zeros(horizon, k, w, dtype=torch.int32, device=dev)
    tm = torch.zeros(horizon, kt, w, dtype=torch.float64, device=dev)
    base = dict(values=values, shaped_rewards=shaped, dones_u8=dones, episode_returns=ret, episode_lengths=length, episode_partials=part[0])
    arms = {"ep": base, "ep+terms": dict(base, reward_terms=tm[0]), "ep+outcome": dict(base, episode_outcomes=oc[0]),
            "ep+outcome+terms": dict(base, episode_outcomes=oc[0], reward_terms=tm[0])}
    rows = []
    for rep in range(repeats):
        for arm in (ARMS if rep % 2 == 0 else ARMS[::-1]):
            env.set_rollout_targets(**arms[arm])
            rows.append({"kind": "step", "task": task, "envs": n, "arm": arm, "rep": rep, "us": _graph_us(torch, env.post_physics_step)})
            print(json.dumps(rows[-1]), flush=True)
    # partials of real steps for the folds
    env.set_rollout_targets()
    for t in range(horizon):
        env.set_rollout_targets(**dict(base, episode_partials=part[t], reward_terms=tm[t]))
        env.post_physics_step()
    env.set_rollout_targets()
    mean = torch.zeros(kt, dtype=torch.float64, device=dev)
    for rep in range(repeats):
        rows.append({"kind": "fold", "task": task, "envs": n, "steps": horizon, "rep": rep,
                     "fold_graph_us": _graph_us(torch, lambda: ops.reward_terms_update(tm, n, task, mean))})
        print(json.dumps(rows[-1]), flush=True)
    env.close()
    del env
    torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="kick:65536,walk:65536,orient:65536,kick:262144,walk:262144,orient:262144,kick:1048576,walk:1048576,orient:1048576")
    ap.add_argument("--repeats", type=int, default=4)
    ap.add_argument("--horizon", type=int, default=32)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("exp_reward_terms needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    cases = [(c.split(":")[0], int(c.split(":")[1])) for c in args.cases.split(",")]
    rows = []
    with open(os.path.join(args.out, "r07_reward_terms.jsonl"), "w") as f:
        f.write(json.dumps({"gpu": info, "device": torch.cuda.get_device_name(0), "cases": args.cases, "repeats": args.repeats,
                            "horizon": args.horizon}) + "\n")
        for task, n in cases:
            for row in measure(task, n, args.repeats, args.horizon):
                rows.append(row)
                f.write(json.dumps(row) + "\n")
        f.write(json.dumps({"gpu_after": gpu_info()}) + "\n")
    lines = [f"# Reward terms in the fused step: A/B ({info})", "",
             f"Fused step with the rollout and episode targets armed (EP), without / with the reward term sums, and the same with the "
             f"outcome counts (OC); 32 launches per CUDA-graph replay, median over {args.repeats} alternated rounds (each the median "
             f"of 5 x 5 replays). Fold over T = {args.horizon} steps of term partials, replayed in a CUDA graph (32 per replay); "
             f"medians over rounds.", "",
             "| task | envs | EP (us) | EP + terms (us) | delta | EP+OC (us) | EP+OC + terms (us) | delta | spread, 4 arms (us) | "
             "fold (us) |", "|---|---:|---:|---:|---:|---:|---:|---:|---|---:|"]
    for task, n in cases:
        med, spread = {}, []
        for arm in ARMS:
            v = [r["us"] for r in rows if r["kind"] == "step" and r["task"] == task and r["envs"] == n and r["arm"] == arm]
            med[arm] = statistics.median(v)
            spread.append(f"{max(v) - min(v):.2f}")
        ff = statistics.median(r["fold_graph_us"] for r in rows if r["kind"] == "fold" and r["task"] == task and r["envs"] == n)
        lines.append(f"| {task} | {n} | {med['ep']:.2f} | {med['ep+terms']:.2f} | {100 * (med['ep+terms'] / med['ep'] - 1):+.1f} % | "
                     f"{med['ep+outcome']:.2f} | {med['ep+outcome+terms']:.2f} | "
                     f"{100 * (med['ep+outcome+terms'] / med['ep+outcome'] - 1):+.1f} % | {' / '.join(spread)} | {ff:.2f} |")
    text = "\n".join(lines) + "\n"
    with open(os.path.join(args.out, "r07_reward_terms.md"), "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    sys.exit(main())
