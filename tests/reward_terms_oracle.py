"""numpy restatements of the reward term sums' two summation orders: the fused step's per-warp shuffle tree and
``bezk_reward_terms_update``'s fold (``csrc/bezk_rollout.cu``), so that device results can be compared bit for bit."""
import numpy as np

FOLD_THREADS = 256


def shuffle_tree(x):
    """A shuffle-down tree (16, 8, 4, 2, 1) over the last axis (32 lanes, float64): lane 0's result."""
    x = np.array(x, dtype=np.float64, copy=True)
    assert x.shape[-1] == 32
    for o in (16, 8, 4, 2, 1):
        x[..., :o] = x[..., :o] + x[..., o:2 * o]
    return x[..., 0]


def warp_sums(terms, n):
    """(K, n) float32 per-env terms -> (K, ceil(n/32)) float64: each warp's tree over its envs (0 past the last env)."""
    terms = np.asarray(terms, dtype=np.float32)
    k = terms.shape[0]
    w = (n + 31) // 32
    x = np.zeros((k, w * 32), dtype=np.float64)
    x[:, :n] = terms.astype(np.float64)
    return shuffle_tree(x.reshape(k, w, 32))


def fold(partials, n):
    """(T, K, W) float64 term partials of n envs -> (K,) float64 means per env-step, in the fold kernel's order: CTA (t, k) thread i
    adds slots i, i + 256, ... from 0.0, a shuffle tree per warp, the 8 warp sums in order from 0.0; then each term's step sums in
    step order from 0.0, divided by T * n."""
    p = np.asarray(partials, dtype=np.float64)
    t, k, w = p.shape
    rounds = max(1, -(-w // FOLD_THREADS))
    x = np.zeros((t, k, rounds * FOLD_THREADS))
    x[..., :w] = p
    x = x.reshape(t, k, rounds, FOLD_THREADS)
    acc = np.zeros((t, k, FOLD_THREADS))
    for r in range(rounds):
        acc = acc + x[:, :, r, :]
    ws = shuffle_tree(acc.reshape(t, k, FOLD_THREADS // 32, 32))
    step = np.zeros((t, k))
    for j in range(FOLD_THREADS // 32):
        step = step + ws[:, :, j]
    total = np.zeros(k)
    for s in range(t):
        total = total + step[s]
    return total / (float(t) * float(n))
