"""A/B of the fused step's game term returns (``bezk_post_physics_rollout_ep_game_terms``) in one GPU session.

For each ``--cases`` entry (task:envs) an env (GPU pipeline, synthetic state) steps with the rollout and episode targets armed as
``A2CAgent.play_steps`` arms them, in four arms: EP (episode accumulators), EP + game term returns, EP + observation normaliser
(the player's step) and EP + normaliser + game term returns.  The arms alternate (the order reverses every round), ``--repeats``
rounds; each measurement is 32 back-to-back fused steps replayed as a CUDA graph (median of 5 replays of 5).  The L2 policy picks
its variant per size as in production.  It also times both folds (``bezk_game_terms_meter_update``,
``bezk_player_game_terms_update``) over T = 32 steps of partials, replayed in a CUDA graph.  Writes ``<out>/r08_game_terms.jsonl``
(a header line with the card, its power limit and clocks, then one line per measurement) and ``<out>/r08_game_terms.md`` (the
medians)."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from exp_reward_terms import _graph_us, gpu_info  # noqa: E402

ARMS = ("ep", "ep+game", "ep+norm", "ep+norm+game")


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
    w, kt = (n + 31) // 32, len(env.REWARD_TERMS)
    values, shaped = torch.randn(n, device=dev), torch.empty(n, device=dev)
    dones = torch.empty(n, dtype=torch.uint8, device=dev)
    ret, length = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    part = torch.zeros(horizon, 3, w, dtype=torch.float64, device=dev)
    acc = torch.zeros(kt, n, device=dev)
    gp = torch.zeros(horizon, kt, w, dtype=torch.float64, device=dev)
    norm = dict(obs_norm=torch.empty(n, env.num_obs, device=dev), obs_mean=torch.zeros(env.num_obs, dtype=torch.float64, device=dev),
                obs_var=torch.ones(env.num_obs, dtype=torch.float64, device=dev))
    base = dict(values=values, shaped_rewards=shaped, dones_u8=dones, episode_returns=ret, episode_lengths=length, episode_partials=part[0])
    game = dict(game_term_returns=acc, game_term_partials=gp[0])
    arms = {"ep": base, "ep+game": dict(base, **game), "ep+norm": dict(base, **norm), "ep+norm+game": dict(base, **norm, **game)}
    rows = []
    for rep in range(repeats):
        for arm in (ARMS if rep % 2 == 0 else ARMS[::-1]):
            env.set_rollout_targets(**arms[arm])
            rows.append({"kind": "step", "task": task, "envs": n, "arm": arm, "rep": rep, "us": _graph_us(torch, env.post_physics_step)})
            print(json.dumps(rows[-1]), flush=True)
    # partials of real steps for the folds
    env.set_rollout_targets()
    for t in range(horizon):
        env.set_rollout_targets(**dict(base, episode_partials=part[t], game_term_returns=acc, game_term_partials=gp[t]))
        env.post_physics_step()
    env.set_rollout_targets()
    mean = torch.zeros(kt, device=dev)
    size = torch.zeros(1, dtype=torch.int64, device=dev)
    sums = torch.zeros(1 + kt, dtype=torch.float64, device=dev)
    for rep in range(repeats):
        rows.append({"kind": "fold", "task": task, "envs": n, "steps": horizon, "rep": rep,
                     "meter_graph_us": _graph_us(torch, lambda: ops.game_terms_meter_update(part, gp, n, task, 100, mean, size)),
                     "player_graph_us": _graph_us(torch, lambda: ops.player_game_terms_update(part, gp, n, task, 10 ** 12, sums))})
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
        raise SystemExit("exp_game_terms needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    cases = [(c.split(":")[0], int(c.split(":")[1])) for c in args.cases.split(",")]
    rows = []
    with open(os.path.join(args.out, "r08_game_terms.jsonl"), "w") as f:
        f.write(json.dumps({"gpu": info, "device": torch.cuda.get_device_name(0), "cases": args.cases, "repeats": args.repeats,
                            "horizon": args.horizon}) + "\n")
        for task, n in cases:
            for row in measure(task, n, args.repeats, args.horizon):
                rows.append(row)
                f.write(json.dumps(row) + "\n")
        f.write(json.dumps({"gpu_after": gpu_info()}) + "\n")
    lines = [f"# Game term returns in the fused step: A/B ({info})", "",
             f"Fused step with the rollout and episode targets armed (EP), without / with the game term returns, and the same with the "
             f"observation normaliser (the player's step); 32 launches per CUDA-graph replay, median over {args.repeats} alternated "
             f"rounds (each the median of 5 x 5 replays). Folds over T = {args.horizon} steps of partials, replayed in a CUDA graph "
             f"(32 per replay); medians over rounds.", "",
             "| task | envs | EP (us) | EP + game (us) | delta | EP+norm (us) | EP+norm + game (us) | delta | spread, 4 arms (us) | "
             "meter fold (us) | player fold (us) |", "|---|---:|---:|---:|---:|---:|---:|---:|---|---:|---:|"]
    for task, n in cases:
        med, spread = {}, []
        for arm in ARMS:
            v = [r["us"] for r in rows if r["kind"] == "step" and r["task"] == task and r["envs"] == n and r["arm"] == arm]
            med[arm] = statistics.median(v)
            spread.append(f"{max(v) - min(v):.2f}")
        folds = [r for r in rows if r["kind"] == "fold" and r["task"] == task and r["envs"] == n]
        fm = statistics.median(r["meter_graph_us"] for r in folds)
        fp = statistics.median(r["player_graph_us"] for r in folds)
        lines.append(f"| {task} | {n} | {med['ep']:.2f} | {med['ep+game']:.2f} | {100 * (med['ep+game'] / med['ep'] - 1):+.1f} % | "
                     f"{med['ep+norm']:.2f} | {med['ep+norm+game']:.2f} | {100 * (med['ep+norm+game'] / med['ep+norm'] - 1):+.1f} % | "
                     f"{' / '.join(spread)} | {fm:.2f} | {fp:.2f} |")
    text = "\n".join(lines) + "\n"
    with open(os.path.join(args.out, "r08_game_terms.md"), "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    sys.exit(main())
