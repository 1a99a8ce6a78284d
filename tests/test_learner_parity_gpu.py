"""GPU parity of the rollout / learner CUDA kernels (through the C ABI) against ``oracle.rl_games_oracle``
(the restated rl_games==1.1.3 math -- parity unpinned beyond the checkpoint identities, see the oracle header).

fp32 results: rtol 1e-5 / atol 1e-6.  Statistics: the kernels accumulate in fp64 where torch's ``mean``/``var``
accumulate in fp32, so running stats are compared with rtol 2e-6 (the fp32 batch moments' own error)."""
import math

import pytest
import torch

from bez_isaacgym_b200 import synthetic_gym as sg
from tests import _util as U

pytestmark = pytest.mark.gpu


def _ops():
    from bez_isaacgym_b200 import ops
    return ops


# ----------------------------------------------------------------------------------------------- GAE
@pytest.mark.parametrize("n,horizon", [(1, 1), (31, 32), (64, 5), (4096, 32), (4099, 17), (70001, 32)])
@pytest.mark.parametrize("dones_dtype", [torch.uint8, torch.float32])
def test_gae_matches_discount_values(n, horizon, dones_dtype):
    from oracle import rl_games_oracle as rg
    ops = _ops()
    rewards, values, dones, last_values, last_dones = sg.make_rollout(n, horizon, seed=n + horizon, p_done=0.05)
    gamma, tau = 0.99, 0.95
    want_adv = rg.discount_values(last_dones.float(), last_values, dones.float(), values, rewards, gamma, tau)
    want_ret = want_adv + values
    d_dones, d_last = dones.to(dones_dtype).cuda(), last_dones.to(dones_dtype).cuda()
    advs = torch.full((horizon, n, 1), float("nan"), device="cuda")
    rets = torch.full((horizon, n, 1), float("nan"), device="cuda")
    ops.gae(rewards.cuda(), values.cuda(), d_dones, last_values.cuda(), d_last, gamma, tau, advs, rets)
    # the recurrence's terms are O(|v|) while advantages can cancel to ~0: condition-aware scale = |v| + |r|
    scale = values.abs() + rewards.abs() + 1.0
    U.assert_close(advs, want_adv, scale=scale, what="advantages")
    U.assert_close(rets, want_ret, scale=scale, what="returns")


def test_gae_all_done_and_none_done():
    from oracle import rl_games_oracle as rg
    ops = _ops()
    n, horizon = 257, 8
    rewards, values, dones, last_values, last_dones = sg.make_rollout(n, horizon, seed=3)
    for fill in (0, 1):
        dones.fill_(fill); last_dones.fill_(fill)
        want = rg.discount_values(last_dones.float(), last_values, dones.float(), values, rewards, 0.99, 0.95)
        advs = torch.empty(horizon, n, 1, device="cuda"); rets = torch.empty_like(advs)
        ops.gae(rewards.cuda(), values.cuda(), dones.cuda(), last_values.cuda(), last_dones.cuda(), 0.99, 0.95, advs, rets)
        U.assert_close(advs, want, scale=values.abs() + 1.0, what=f"advantages dones={fill}")
        if fill == 1:                                    # every step terminal: adv = r - v exactly
            assert torch.equal(advs.cpu(), rewards - values)


def test_gae_linearity_at_full_size():
    """Size-independent property at the BASELINE size (262144 envs x 32): GAE is linear in (rewards, values,
    last_values) for fixed dones, so gae(a*x + y) == a*gae(x) + gae(y) up to fp32 rounding."""
    ops = _ops()
    n, horizon = 262144, 32
    r1, v1, dones, lv1, ld = [t.cuda() for t in sg.make_rollout(n, horizon, seed=1)]
    r2, v2, _, lv2, _ = [t.cuda() for t in sg.make_rollout(n, horizon, seed=2)]
    def run(r, v, lv):
        a = torch.empty_like(r); ret = torch.empty_like(r)
        ops.gae(r, v, dones, lv, ld, 0.99, 0.95, a, ret)
        return a, ret
    a1, _ = run(r1, v1, lv1)
    a2, _ = run(r2, v2, lv2)
    a3, ret3 = run(2.0 * r1 + r2, 2.0 * v1 + v2, 2.0 * lv1 + lv2)
    assert torch.allclose(a3, 2.0 * a1 + a2, rtol=1e-4, atol=1e-4)
    assert torch.allclose(ret3, a3 + (2.0 * v1 + v2), rtol=0, atol=0)


# ----------------------------------------------------------------------------------------------- RunningMeanStd
def _rms_forward_gpu(x, mean, var, count, train=True, unnorm=False):
    ops = _ops()
    c = mean.numel()
    if train:
        acc = torch.empty(1 + 2 * c, dtype=torch.float64, device="cuda")
        partials = torch.empty(ops.rms_scratch_doubles(c), dtype=torch.float64, device="cuda")
        pivot = mean.clone()
        ops.rms_moments(x, pivot, acc, partials)
        ops.rms_merge(acc, pivot, mean, var, count)
    y = torch.empty_like(x)
    ops.rms_normalize(x, mean, var, y, unnorm=unnorm)
    return y


@pytest.mark.parametrize("m,c", [(2, 54), (37, 54), (1000, 54), (4096, 54), (4099, 54), (32768, 54), (100040, 54), (1000, 1),
                                 (131072, 1), (333, 7), (4096, 2), (512, 200), (64, 200)])
def test_running_mean_std_train_forward(m, c):
    from oracle import rl_games_oracle as rg
    g = torch.Generator().manual_seed(m + c)
    scale = torch.rand(c, generator=g) * 3 + 0.1
    shift = torch.randn(c, generator=g) * 2
    orc = rg.RunningMeanStd(c)
    mean = torch.zeros(c, dtype=torch.float64, device="cuda"); var = torch.ones(c, dtype=torch.float64, device="cuda")
    count = torch.ones((), dtype=torch.float64, device="cuda")
    for it in range(3):                                   # three successive updates exercise the merge
        x = torch.randn(m, c, generator=g) * scale + shift + it
        want = orc(x)
        got = _rms_forward_gpu(x.cuda(), mean, var, count)
        assert torch.allclose(mean.cpu(), orc.running_mean, rtol=2e-6, atol=1e-7), "running_mean"
        assert torch.allclose(var.cpu(), orc.running_var, rtol=2e-5, atol=1e-7), "running_var"
        assert count.item() == orc.count.item()
        # normalised output: compare against the oracle formula evaluated with the GPU's own stats, so the
        # check isolates the normalise kernel (the stats were compared above)
        ref = torch.clamp((x - mean.cpu().float()) / torch.sqrt(var.cpu().float() + 1e-5), -5.0, 5.0)
        U.assert_close(got, ref, what="normalised (own stats)")
        # and end to end against the oracle (stats differ by fp32-vs-fp64 accumulation only)
        assert torch.allclose(got.cpu(), want, rtol=1e-4, atol=1e-4)


def test_running_mean_std_eval_and_unnorm():
    from oracle import rl_games_oracle as rg
    c, m = 54, 5000
    g = torch.Generator().manual_seed(0)
    orc = rg.RunningMeanStd(c)
    orc.running_mean = torch.randn(c, generator=g).double(); orc.running_var = (torch.rand(c, generator=g) + 0.01).double()
    orc.training = False
    x = 4 * torch.randn(m, c, generator=g)
    mean, var = orc.running_mean.cuda(), orc.running_var.cuda()
    count = torch.ones((), dtype=torch.float64, device="cuda")
    U.assert_close(_rms_forward_gpu(x.cuda(), mean, var, count, train=False), orc(x), what="eval normalise")
    U.assert_close(_rms_forward_gpu(x.cuda(), mean, var, count, train=False, unnorm=True), orc(x, unnorm=True),
                   what="unnorm")
    assert torch.equal(mean.cpu(), orc.running_mean) and count.item() == 1.0      # eval mode leaves stats alone


def test_rms_moments_are_additive_across_shards():
    """Exact multi-GPU merge: pivoted sums of two shards add up to the sums of the union (what the single SUM
    all-reduce relies on) -- checked to fp64 round-off."""
    ops = _ops()
    c, m = 54, 8192
    x = (torch.randn(m, c, generator=torch.Generator().manual_seed(1)) * 2 + 1).cuda()
    pivot = torch.randn(c, dtype=torch.float64, device="cuda")
    scratch = torch.empty(ops.rms_scratch_doubles(c), dtype=torch.float64, device="cuda")
    def mom(t):
        acc = torch.empty(1 + 2 * c, dtype=torch.float64, device="cuda")
        return ops.rms_moments(t.contiguous(), pivot, acc, scratch).clone()
    whole, a, b = mom(x), mom(x[:3000]), mom(x[3000:])
    assert torch.allclose(a + b, whole, rtol=1e-12, atol=1e-9)
    want = torch.cat([torch.tensor([float(m)], dtype=torch.float64),
                      (x.double().cpu() - pivot.cpu()).sum(0), ((x.double().cpu() - pivot.cpu()) ** 2).sum(0)])
    assert torch.allclose(whole.cpu(), want, rtol=1e-12, atol=1e-9)
    # bit-wise run-to-run determinism (fixed reduction order)
    assert torch.equal(mom(x), whole)


# ----------------------------------------------------------------------------------------------- advantages
@pytest.mark.parametrize("m", [2, 1000, 131072, 131075])
def test_advantage_normalisation(m):
    from oracle import rl_games_oracle as rg
    ops = _ops()
    g = torch.Generator().manual_seed(m)
    returns = torch.randn(m, 1, generator=g) * 2 + 0.3
    values = torch.randn(m, 1, generator=g)
    want, _, _ = rg.prepare_dataset(returns, values, rg.RunningMeanStd(1))
    acc = torch.empty(3, dtype=torch.float64, device="cuda")
    scratch = torch.empty(ops.rms_scratch_doubles(1), dtype=torch.float64, device="cuda")
    r_d, v_d = returns.cuda(), values.cuda()
    ops.adv_moments(r_d, v_d, acc, scratch)
    out = torch.empty(m, device="cuda")
    ops.adv_normalize(r_d, v_d, acc, out)
    adv = (returns - values).squeeze(1)
    assert math.isclose(acc[1].item() / m, adv.double().mean().item(), rel_tol=1e-9, abs_tol=1e-12)
    assert torch.allclose(out.cpu(), want, rtol=1e-5, atol=2e-6)
    raw = torch.empty(m, device="cuda")
    ops.adv_normalize(r_d, v_d, None, raw, normalize=False)
    assert torch.equal(raw.cpu(), adv)


# ----------------------------------------------------------------------------------------------- PPO loss
# 75777: CTAs of the 592-CTA persistent grid take a second tile (mbarrier phase flip, grad_mu store drained first);
# 700001: CTA 140 takes 10 tiles -- a mid-loop fp32 -> fp64 flush after PPO_FLUSH = 8 and a ragged last tile
@pytest.mark.parametrize("m", [1, 127, 128, 4099, 32768, 75777, 700001])
@pytest.mark.parametrize("bound_form", ["v1.1.3", "outside"])
def test_ppo_loss_forward_backward(m, bound_form):
    from oracle import rl_games_oracle as rg
    ops = _ops()
    mb = sg.make_minibatch(m, seed=m)
    mb["mu"][: max(1, m // 8)] *= 4.0                     # push some means beyond the 1.1 soft bound
    mb["advantages"][:: 5] *= -1.0
    mu = mb["mu"].clone().requires_grad_(True)
    values = mb["values"].clone().requires_grad_(True)
    logstd = mb["logstd"].clone().requires_grad_(True)
    o = rg.ppo_loss(dict(mb, mu=mu, values=values, logstd=logstd), bound_form=bound_form)
    o["loss"].backward()

    cfg = ops.make_ppo_cfg(bound_form=bound_form)
    dev = {k: v.cuda().contiguous() for k, v in mb.items()}
    stats = torch.empty(8, dtype=torch.float64, device="cuda")
    partials = torch.empty(ops.ppo_scratch_doubles(), dtype=torch.float64, device="cuda")
    g_mu = torch.full((m, 18), float("nan"), device="cuda"); g_v = torch.full((m,), float("nan"), device="cuda")
    g_ls = torch.full((18,), float("nan"), device="cuda"); nlp = torch.empty(m, device="cuda")
    ops.ppo_loss(dev["actions"], dev["mu"], dev["logstd"], dev["old_mu"], dev["old_sigma"], dev["values"].view(-1),
                 dev["old_values"].view(-1), dev["returns"].view(-1), dev["old_neglogp"], dev["advantages"], cfg, stats,
                 partials, grad_mu=g_mu, grad_values=g_v, grad_logstd=g_ls, neglogp_out=nlp)
    s = stats.cpu()
    for idx, key in [(0, "loss"), (1, "a_loss"), (2, "c_loss"), (3, "entropy"), (4, "b_loss"), (5, "kl")]:
        assert math.isclose(s[idx].item(), o[key].item(), rel_tol=2e-5, abs_tol=2e-6), (key, s[idx].item(), o[key].item())
    assert torch.allclose(nlp.cpu(), o["neglogp"].detach(), rtol=1e-5, atol=1e-5)
    gscale = 1.0 / m
    assert torch.allclose(g_mu.cpu(), mu.grad, rtol=1e-4, atol=1e-5 * gscale), "d loss / d mu"
    assert torch.allclose(g_v.cpu(), values.grad.view(-1), rtol=1e-4, atol=1e-5 * gscale), "d loss / d value"
    assert torch.allclose(g_ls.cpu(), logstd.grad, rtol=1e-4, atol=1e-5), "d loss / d logstd"
