"""CPU: the fp64 references of ``tests/learner_reference.py`` against the rl_games restatement in ``oracle/rl_games_oracle.py``, so the
targets the learner kernels are held to are themselves checked without a GPU."""
import pytest
import torch

from oracle import rl_games_oracle as rg
from tests import learner_reference as R


def _obs(m, c, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(m, c, generator=g) * (torch.rand(c, generator=g) * 2 + 0.25) + torch.randn(c, generator=g) * 2
    if c > 2:
        x[:, 1] = 1000.0 + torch.randn(m, generator=g)        # |mean| / std = 1e3
        x[:, -1] = 0.175                                       # constant, like the ball_init columns
    return x


@pytest.mark.parametrize("m,c", [(1, 1), (2, 1), (297, 1), (1, 54), (3, 54), (4099, 54), (2049, 7)])
def test_ref_stats_match_the_oracle_update_in_float64(m, c):
    """The oracle's train-mode update fed float64 rows computes its batch moments in float64: it must agree with the two-pass
    reference to float64 rounding (NaN variance for a one-row batch in both)."""
    orc = rg.RunningMeanStd(c)
    mean, var, count = torch.zeros(c, dtype=torch.float64), torch.ones(c, dtype=torch.float64), 1.0
    for it in range(3):
        x = _obs(m, c, 10 * m + it)
        orc(x.double())
        mean, var, count = R.ref_stats(mean, var, count, [x])
        assert count == float(orc.count)
        torch.testing.assert_close(mean, orc.running_mean, rtol=1e-12, atol=1e-12, equal_nan=True)
        torch.testing.assert_close(var, orc.running_var, rtol=1e-12, atol=1e-12, equal_nan=True)


def test_ref_stats_of_several_batches_is_the_sequence_of_updates():
    x = [_obs(500 + k, 54, k) for k in range(3)]
    start = (torch.linspace(-1, 1, 54).double(), torch.full((54,), 2.0, dtype=torch.float64), 1000.0)
    one = R.ref_stats(*start, x)
    step = start
    for b in x:
        step = R.ref_stats(*step, [b])
    assert torch.equal(one[0], step[0]) and torch.equal(one[1], step[1]) and one[2] == step[2]


def test_replay_merges_agrees_with_ref_stats():
    """Pivoted sums replayed through the sequence kernel's arithmetic give the two-pass reference's statistics."""
    c = 54
    batches = [_obs(700 + 13 * k, c, 40 + k) for k in range(4)]
    pivot = torch.linspace(-1, 1, c).double()
    acc = torch.stack([torch.cat([torch.tensor([float(b.shape[0])], dtype=torch.float64), (b.double() - pivot).sum(0),
                                  ((b.double() - pivot) ** 2).sum(0)]) for b in batches])
    order = [0, 1, 2, 3, 2, 0]
    mean0, var0 = pivot.clone(), torch.full((c,), 2.0, dtype=torch.float64)
    seq, cnt = R.replay_merges(acc, order, pivot, mean0, var0, 1000.0)
    want = (mean0, var0, 1000.0)
    for u, b in enumerate(order):
        want = R.ref_stats(*want, [batches[b]])
        torch.testing.assert_close(seq[u, 0], want[0], rtol=1e-12, atol=1e-12)
        torch.testing.assert_close(seq[u, 1], want[1], rtol=1e-9, atol=1e-12)
    assert cnt == want[2]


@pytest.mark.parametrize("unnorm", [False, True])
def test_ref_normalize_is_the_oracle_expression_bit_for_bit(unnorm):
    c = 54
    x = _obs(3001, c, 5) * 1.5
    x[7, 3] = float("nan")
    orc = rg.RunningMeanStd(c)
    orc.training = False
    orc.running_mean = torch.randn(c, generator=torch.Generator().manual_seed(1)).double()
    orc.running_mean[1] = 1000.25
    orc.running_var = torch.rand(c, generator=torch.Generator().manual_seed(2)).double() + 1e-3
    orc.running_var[5] = float("nan")
    got = R.ref_normalize(x, orc.running_mean, orc.running_var, unnorm=unnorm)
    want = orc(x, unnorm=unnorm)
    # torch's vectorised CPU sqrt may miss the correctly rounded result by 1 ulp: bit for bit in every column where it does not
    s_cpu = torch.sqrt(orc.running_var.float() + 1e-5)
    exact = s_cpu == torch.sqrt((orc.running_var.float() + 1e-5).double()).float()
    exact |= torch.isnan(s_cpu)
    assert bool(R.bits_equal(got[:, exact], want[:, exact]).all())
    torch.testing.assert_close(got, want, rtol=2.0 ** -22, atol=0.0, equal_nan=True)
    assert bool(torch.isnan(got[:, 5]).all()) and bool(torch.isnan(got[7, 3]))


@pytest.mark.parametrize("m", [1, 2, 3, 297, 4099, 131075])
def test_ref_advantages_match_prepare_dataset(m):
    g = torch.Generator().manual_seed(m)
    r, v = torch.randn(m, 1, generator=g) * 2 + 0.3, torch.randn(m, 1, generator=g)
    want, _, _ = rg.prepare_dataset(r, v, rg.RunningMeanStd(1))
    y, ambiguous, cands = R.ref_advantages(r, v)
    assert ambiguous == (len(cands) > 1)
    assert any(bool(R.bits_equal(y, cnd).all()) for cnd in cands)
    # the oracle sums in fp32: within prepare_dataset's tolerance of the float64-statistics result
    torch.testing.assert_close(y, want, rtol=1e-5, atol=2e-6, equal_nan=True)
    if m == 1:
        assert bool(torch.isnan(y).all()), "torch.std of one sample is NaN, and so is the normalised advantage"
    # float64 end to end, for the exact statistics
    d = (r - v).double().view(-1)
    if m > 1:
        torch.testing.assert_close(y.double(), (d - d.mean()) / (d.std() + 1e-8), rtol=1e-6, atol=1e-6)


def test_ref_advantages_of_constant_advantages_are_zero():
    r, v = torch.full((4099, 1), 0.7), torch.full((4099, 1), 0.2)
    y, ambiguous, _ = R.ref_advantages(r, v)
    assert not ambiguous and torch.equal(y, torch.zeros(4099))


def test_ref_advantages_flags_a_rounding_tie():
    """A float64 mean half-way between two fp32 values is flagged, and y is offered for both of its roundings."""
    r = torch.tensor([1.0, 1.0 + 2.0 ** -23])               # both exact in fp32; the mean 1 + 2^-24 is a tie
    y, ambiguous, cands = R.ref_advantages(r, torch.zeros(2))
    assert ambiguous and len(cands) == 2
    assert any(bool(R.bits_equal(y, cnd).all()) for cnd in cands)
    assert not bool(R.bits_equal(cands[0], cands[1]).all())
