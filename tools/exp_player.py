"""A/B of one player step's observation normalisation in one GPU session: the fused normaliser
(``bezk_post_physics_rollout_ep_norm``) against the episode-accumulator step followed by a separate ``bezk_rms_normalize``.

At each ``--sizes`` env count a KickEnv (GPU pipeline, synthetic state, ``clip_obs`` finite so the clipped row is the one
normalised, as in the reference's config) steps with the episode targets armed, as ``learner.PpoPlayerContinuous`` arms them:
  * ``ep``       -- the EP step alone (``task_tile_ep_kernel``, no normalisation; the reference point);
  * ``ep+rms``   -- arm B: the EP step + ``bezk_rms_normalize`` of the returned rows (eval mode);
  * ``fused``    -- arm A: the step with ``obs_norm`` armed (``task_tile_obsnorm_kernel``).
The arms alternate, ``--repeats`` rounds; each measurement is 32 back-to-back steps replayed as a CUDA graph (median of 5
replays of 5), timed with CUDA events.  The L2 policy picks its variant per size as in production.  Writes
``<out>/r05_player.jsonl`` (a header line with the card, its power limit and clocks, then one line per measurement) and
``<out>/r05_player.md`` (the medians)."""
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


def measure(n, repeats):
    import torch
    from bez_isaacgym_b200 import bez_model as bm, ops, synthetic_gym as sg
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym
    from bez_isaacgym_b200.tasks import KickEnv

    dev = torch.device("cuda:0")
    cfg = bm.default_task_cfg(n)
    cfg["env"]["clipObservations"] = 5.0
    env = KickEnv(cfg, "cuda:0", 0, True, sim=SyntheticGym(n, device="cuda:0"))
    p, r = sg.make_bookkeeping(n, device=dev)
    env.progress_buf.copy_(p)
    env.reset_buf.copy_(r)
    w = (n + 31) // 32
    ret, length = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    part = torch.zeros(3, w, dtype=torch.float64, device=dev)
    mean = torch.randn(54, dtype=torch.float64, device=dev)
    var = torch.rand(54, dtype=torch.float64, device=dev) + 0.1
    norm, norm_b = torch.empty(n, 54, device=dev), torch.empty(n, 54, device=dev)
    ep = dict(episode_returns=ret, episode_lengths=length, episode_partials=part)

    def step_b():
        env.post_physics_step()
        ops.rms_normalize(env._observations_out(), mean, var, norm_b)

    arms = {"ep": (ep, env.post_physics_step), "ep+rms": (ep, step_b),
            "fused": (dict(ep, obs_norm=norm, obs_mean=mean, obs_var=var), env.post_physics_step)}
    rows = []
    for rep in range(repeats):
        for arm in (list(arms) if rep % 2 == 0 else list(arms)[::-1]):
            targets, fn = arms[arm]
            env.set_rollout_targets(**targets)
            rows.append({"envs": n, "arm": arm, "rep": rep, "us": _graph_us(torch, fn)})
            print(json.dumps(rows[-1]), flush=True)
    env.set_rollout_targets()
    env.close()
    del env
    torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="4096,65536,262144")
    ap.add_argument("--repeats", type=int, default=6)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("exp_player needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    sizes = [int(x) for x in args.sizes.split(",")]
    rows = []
    with open(os.path.join(args.out, "r05_player.jsonl"), "w") as f:
        f.write(json.dumps({"gpu": info, "device": torch.cuda.get_device_name(0), "sizes": sizes, "repeats": args.repeats}) + "\n")
        for n in sizes:
            for row in measure(n, args.repeats):
                rows.append(row)
                f.write(json.dumps(row) + "\n")
        f.write(json.dumps({"gpu_after": gpu_info()}) + "\n")
    lines = [f"# Player step: fused observation normaliser vs a separate pass ({info})", "",
             "KickEnv post-physics step (clip_obs = 5) with the episode targets armed; 32 launches per CUDA-graph replay, median "
             f"over {args.repeats} alternated rounds (each the median of 5 x 5 replays). ep = EP step alone; B = EP step + "
             "`bezk_rms_normalize`; A = step with `obs_norm` armed.", "",
             "| envs | ep (us) | B: ep + rms (us) | A: fused (us) | A vs B | A vs ep | spread ep / B / A (us) |",
             "|---:|---:|---:|---:|---:|---:|---:|"]
    for n in sizes:
        m = {a: [r["us"] for r in rows if r["envs"] == n and r["arm"] == a] for a in ("ep", "ep+rms", "fused")}
        e, b, a = (statistics.median(m[k]) for k in ("ep", "ep+rms", "fused"))
        spread = " / ".join(f"{max(v) - min(v):.2f}" for v in m.values())
        lines.append(f"| {n} | {e:.2f} | {b:.2f} | {a:.2f} | {100 * (a / b - 1):+.1f} % | {100 * (a / e - 1):+.1f} % | {spread} |")
    text = "\n".join(lines) + "\n"
    with open(os.path.join(args.out, "r05_player.md"), "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    sys.exit(main())
