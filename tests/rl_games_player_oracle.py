"""torch-CPU restatement of rl_games' player tally (TEST INFRASTRUCTURE ONLY; RECALLED, not vendored, so parity is unpinned):
``rl_games/common/player.py`` ``BasePlayer.run`` (v1.1.x; the reference's fork is ``utils/player.py``).  The library's fold
(``bezk_player_tally_update``) and ``learner.PpoPlayerContinuous.run`` are tested against it.

Two forms:
  * ``RlGamesTally`` -- rl_games itself: fp32 ``cr`` / ``steps`` tensors, ``cr[done].sum().item()`` per step, Python-float sums;
  * ``fold_partials`` -- the same rule fed the kernel's per-step partials (3, W), with the fold's fixed summation order, in fp64:
    what the library must match bit for bit."""
import numpy as np
import torch


class RlGamesTally:
    """BasePlayer.run's bookkeeping around ``env_step``.  ``step(r, done)`` returns False once rl_games would stop."""

    def __init__(self, batch_size, games_num, n_game_life=1):
        self.n_games = games_num * n_game_life
        self.n_game_life = n_game_life
        self.games_played = 0
        self.sum_rewards = 0.0
        self.sum_steps = 0.0
        self.lines = []
        self.reset(batch_size)

    def reset(self, batch_size):
        """``env_reset``: fresh ``cr`` / ``steps``."""
        self.cr = torch.zeros(batch_size, dtype=torch.float32)
        self.steps = torch.zeros(batch_size, dtype=torch.float32)

    def step(self, r, done):
        self.cr += r
        self.steps += 1
        done_indices = done.nonzero(as_tuple=False)
        done_count = len(done_indices)
        self.games_played += done_count
        if done_count > 0:
            cur_rewards = self.cr[done_indices].sum().item()
            cur_steps = self.steps[done_indices].sum().item()
            self.cr = self.cr * (1.0 - done.float())
            self.steps = self.steps * (1.0 - done.float())
            self.sum_rewards += cur_rewards
            self.sum_steps += cur_steps
            self.lines.append((cur_rewards / done_count, cur_steps / done_count))
            if self.games_played >= self.n_games:
                return False
        return True

    def result(self):
        g = self.games_played
        return dict(games_played=g, sum_rewards=self.sum_rewards, sum_steps=self.sum_steps,
                    av_reward=self.sum_rewards / g * self.n_game_life, av_steps=self.sum_steps / g * self.n_game_life)


def step_sums(partials_step):
    """One step's [count, return sum, length sum] from its (3, W) partials in the fold's order: lane l (of 32) adds slots
    l, l + 32, ... in order, then the shuffle-down tree (16, 8, 4, 2, 1) -- a lane whose source is out of range adds itself."""
    p = np.asarray(partials_step, dtype=np.float64).reshape(3, -1)
    w = p.shape[1]
    out = []
    for k in range(3):
        acc = np.zeros(32, dtype=np.float64)
        for j in range(0, w, 32):
            chunk = p[k, j:j + 32]
            acc[:chunk.size] = acc[:chunk.size] + chunk
        for o in (16, 8, 4, 2, 1):
            src = np.concatenate([acc[o:], acc[32 - o:]])       # out-of-range lanes read their own value
            acc = acc + src
        out.append(acc[0])
    return out


def fold_partials(partials, games_num, tally=None):
    """The fold over (steps, 3, W) partials: returns (tally [games, sum_rewards, sum_steps, steps_folded], per_step (steps, 3))."""
    games, sr, sl, folded = (0.0, 0.0, 0.0, 0.0) if tally is None else tuple(float(x) for x in tally)
    partials = np.asarray(partials, dtype=np.float64)
    per_step = np.zeros((partials.shape[0], 3), dtype=np.float64)
    for t in range(partials.shape[0]):
        if games >= games_num:
            continue
        c, r, l = step_sums(partials[t])
        folded += 1.0
        per_step[t] = (c, r, l)
        if c > 0.0:
            games += c
            sr = sr + r
            sl = sl + l
    return np.array([games, sr, sl, folded]), per_step
