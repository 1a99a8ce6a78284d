"""numpy restatement of the two game term folds (TEST INFRASTRUCTURE ONLY): rl_games' ``AverageMeter(K, games_to_track)`` fed with
one K-row of per-term episode returns per done env (torch_ext.AverageMeter, RECALLED, as in ``tests/rl_games_episode_oracle.py``)
and the player's per-term sums with ``BasePlayer.run``'s cutoff (as in ``tests/rl_games_player_oracle.py``), in the summation
order of ``csrc/bezk_rollout.cu``'s ``epm_step_sums``, so that ``bezk_game_terms_meter_update`` and
``bezk_player_game_terms_update`` can be compared bit for bit; and the fused step's per-warp sums of the done envs' returns."""
import numpy as np

from tests.reward_terms_oracle import FOLD_THREADS, shuffle_tree


def step_sums(ep_partials, term_partials):
    """(T, 3, W) episode partials and (T, K, W) game term partials -> (T, 1 + K) float64 [done count, sum_0 .. sum_{K-1}]: thread i
    of 256 adds slots i, i + 256, ... in order from 0.0, a shuffle tree per warp, the 8 warp sums in order from 0.0."""
    ep = np.asarray(ep_partials, dtype=np.float64)
    tp = np.asarray(term_partials, dtype=np.float64)
    rows = np.concatenate([ep[:, :1], tp], axis=1)
    t, r, w = rows.shape
    rounds = max(1, -(-w // FOLD_THREADS))
    x = np.zeros((t, r, rounds * FOLD_THREADS))
    x[..., :w] = rows
    x = x.reshape(t, r, rounds, FOLD_THREADS)
    acc = np.zeros((t, r, FOLD_THREADS))
    for j in range(rounds):
        acc = acc + x[:, :, j, :]
    ws = shuffle_tree(acc.reshape(t, r, FOLD_THREADS // 32, 32))
    out = np.zeros((t, r))
    for j in range(FOLD_THREADS // 32):
        out = out + ws[:, :, j]
    return out


def meter(ep_partials, term_partials, games_to_track, mean=None, size=0):
    """AverageMeter(K, games_to_track).update(rows) once per step, in order: new_mean = (float)(sum_k / count) in fp64, size =
    count; a step with no done env is a no-op.  Returns (mean (K,) fp32, size)."""
    s = step_sums(ep_partials, term_partials)
    k = s.shape[1] - 1
    mean = np.zeros(k, np.float32) if mean is None else np.asarray(mean, np.float32).copy()
    for row in s:
        cnt = row[0]
        if not cnt > 0.0:
            continue
        sz = min(int(cnt), games_to_track)
        old = min(games_to_track - sz, size)
        size_sum = old + sz
        size = size_sum
        new_mean = (row[1:] / cnt).astype(np.float32)
        mean = (mean * np.float32(old) + new_mean * np.float32(sz)) / np.float32(size_sum)
    return mean.astype(np.float32), size


def player_fold(ep_partials, term_partials, games_num, sums=None):
    """[games_counted, sum_0 .. sum_{K-1}] (fp64) and the (steps, K) per-step rows: a step that starts with games_counted >=
    games_num adds nothing, the step that reaches it is added whole."""
    s = step_sums(ep_partials, term_partials)
    k = s.shape[1] - 1
    out = np.zeros(1 + k) if sums is None else np.asarray(sums, np.float64).copy()
    per = np.zeros((s.shape[0], k))
    for t, row in enumerate(s):
        if out[0] >= games_num:
            continue
        per[t] = row[1:]
        if row[0] > 0.0:
            out[0] += row[0]
            out[1:] = out[1:] + row[1:]
    return out, per


def done_warp_sums(r, done, n):
    """(K, n) float32 per-term returns r_k and (n,) done mask -> (K, ceil(n/32)) float64: each warp's tree over its done envs."""
    r = np.asarray(r, dtype=np.float32)
    x = np.where(np.asarray(done, dtype=bool)[None, :], r.astype(np.float64), 0.0)
    k, w = r.shape[0], (n + 31) // 32
    y = np.zeros((k, w * 32))
    y[:, :n] = x
    return shuffle_tree(y.reshape(k, w, 32))
