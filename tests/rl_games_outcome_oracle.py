"""numpy restatement of the two outcome folds (TEST INFRASTRUCTURE ONLY): rl_games' ``AverageMeter(K, games_to_track)`` fed with
one one-hot row per done env (torch_ext.AverageMeter, RECALLED, as in ``tests/rl_games_episode_oracle.py``) and the player's
per-outcome tally with ``BasePlayer.run``'s cutoff (as in ``tests/rl_games_player_oracle.py``).  ``bezk_outcome_meter_update`` and
``bezk_player_outcome_update`` are tested against it."""
import numpy as np


def step_counts(partials):
    """(steps, K, W) int32 outcome partials -> (steps, K) exact int64 class counts."""
    return np.asarray(partials, dtype=np.int64).sum(axis=2)


def meter(partials, games_to_track, mean=None, size=0):
    """AverageMeter(K, games_to_track).update(one_hot_rows) once per step, in order: new_mean = count_k / total (fp32 division of
    exact counts; torch.mean of 0/1 rows), size = total; a step with no done env is a no-op.  Returns (mean (K,) fp32, size)."""
    counts = step_counts(partials)
    k = counts.shape[1]
    mean = np.zeros(k, np.float32) if mean is None else np.asarray(mean, np.float32).copy()
    for row in counts:
        total = int(row.sum())
        if total == 0:
            continue
        s = min(total, games_to_track)
        old = min(games_to_track - s, size)
        size_sum = old + s
        size = size_sum
        new_mean = row.astype(np.float32) / np.float32(total)
        mean = (mean * np.float32(old) + new_mean * np.float32(s)) / np.float32(size_sum)
    return mean.astype(np.float32), size


def player_fold(partials, games_num, counts=None):
    """[games_counted, count_0..count_{K-1}] (fp64) and the (steps, K) per-step rows: a step that starts with games_counted >=
    games_num adds nothing, the step that reaches it is added whole."""
    c = step_counts(partials)
    k = c.shape[1]
    out = np.zeros(1 + k) if counts is None else np.asarray(counts, np.float64).copy()
    per = np.zeros((c.shape[0], k))
    for t, row in enumerate(c):
        if out[0] >= games_num:
            continue
        out[0] += float(row.sum())
        out[1:] += row
        per[t] = row
    return out, per
