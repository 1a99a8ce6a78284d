"""fp64 references for the learner's statistics kernels (``csrc/bezk_learner.cu``, ``csrc/bezk_fused.cu``): RunningMeanStd's batch
moments and parallel-variance merge, its fp32 normalisation, and ``prepare_dataset``'s advantage normalisation.  Where a kernel
promises rl_games' fp32 expression (IEEE division and sqrt, no FMA contraction) its output can be compared with these bit for bit."""
import itertools

import torch

EPS_F32_1E8 = torch.tensor(1e-8, dtype=torch.float32)


def batch_moments(x):
    """Two-pass float64 mean and unbiased variance over the rows of fp32 ``x`` ((B, c) or (B,)); NaN variance for B == 1, like
    ``torch.var``."""
    x64 = x.double()
    b = x64.shape[0]
    mean = x64.sum(0) / b
    var = ((x64 - mean) ** 2).sum(0) / (b - 1) if b > 1 else torch.full_like(mean, float("nan"))
    return mean, var, b


def merge(mean, var, count, batch_mean, batch_var, batch_count):
    """rl_games ``RunningMeanStd._update_mean_var_count_from_moments`` in float64."""
    delta = batch_mean - mean
    tot = count + batch_count
    new_mean = mean + delta * batch_count / tot
    m2 = var * count + batch_var * batch_count + delta ** 2 * count * batch_count / tot
    return new_mean, m2 / tot, tot


def ref_stats(mean, var, count, batches):
    """Running statistics after train-mode updates with each of ``batches`` in turn: two-pass float64 moments of the fp32 rows, then
    rl_games' parallel-variance merge in float64.  ``mean`` / ``var``: (c,) float64, ``count``: a number; returns (mean, var, count)."""
    mean, var, count = mean.double().cpu(), var.double().cpu(), float(count)
    for x in batches:
        bm, bv, b = batch_moments(x.reshape(-1, mean.numel()).cpu())
        mean, var, count = merge(mean, var, count, bm, bv, float(b))
    return mean, var, count


def replay_merges(acc, order, pivot, mean, var, count):
    """``rms_merge_sequence_kernel``'s updates in float64, operation for operation: ``acc`` (n_batches, 1 + 2c) = [B, sum(x - p),
    sum((x - p)^2)] per batch, all with the pivot ``pivot``; update u merges batch ``order[u]``.  Returns ``seq`` (n_updates, 2, c) =
    [mean, var] after each update, and the final count."""
    acc, pivot = acc.double().cpu(), pivot.double().cpu()
    mean, var, cnt = mean.double().cpu().clone(), var.double().cpu().clone(), float(count)
    c = mean.numel()
    seq = torch.empty(len(order), 2, c, dtype=torch.float64)
    for u, b in enumerate(order):
        a = acc[b]
        bb = float(a[0])
        if bb > 0.0:
            tot = cnt + bb
            s, ss = a[1:1 + c], a[1 + c:1 + 2 * c]
            mean_b = pivot + s / bb
            var_b = (ss - s * s / bb) / (bb - 1.0)
            delta = mean_b - mean
            new_mean = mean + delta * bb / tot
            var = (var * cnt + var_b * bb + delta * delta * cnt * bb / tot) / tot
            mean = new_mean
            cnt = tot
        seq[u, 0], seq[u, 1] = mean, var
    return seq, cnt


def f32(t):
    """Round float64 to fp32.  One IEEE fp32 operation (+, -, *, /, sqrt) on fp32 operands, evaluated in float64 and rounded once,
    is the correctly rounded fp32 result (53 >= 2 * 24 + 2 bits: the double rounding is innocuous).  The references spell every fp32
    operation this way because torch's vectorised CPU ``sqrt`` is not always correctly rounded (Sleef's 0.5001-ulp routine)."""
    return t.float()


def ref_normalize(x, mean, var, eps=1e-5, unnorm=False):
    """rl_games' fp32 normalisation with the given float64 statistics: ``clamp((x - mean.float()) / sqrt(var.float() + eps), -5, 5)``
    (``unnorm``: ``sqrt(var.float() + eps) * clamp(x) + mean.float()``), every fp32 operation correctly rounded (see ``f32``), as
    IEEE fp32 arithmetic evaluates it.  Broadcasts, so (n, rows, c) inputs with (n, 1, c) statistics give n batches at once."""
    x = x.cpu().float().double()
    m = mean.cpu().float().double()
    s = f32(torch.sqrt(f32(var.cpu().float().double() + torch.tensor(eps, dtype=torch.float32).double()).double())).double()
    if unnorm:
        return f32(f32(s * torch.clamp(x, min=-5.0, max=5.0)).double() + m)
    return torch.clamp(f32(f32(x - m).double() / s), min=-5.0, max=5.0)


def _roundings(v, rel=1e-12):
    """The fp32 roundings of float64 ``v`` perturbed by +-``rel`` relative (one value where both agree, or v is NaN / 0)."""
    lo = torch.tensor(float(v) * (1.0 - rel), dtype=torch.float64).float()
    hi = torch.tensor(float(v) * (1.0 + rel), dtype=torch.float64).float()
    if bool(torch.isnan(lo)) or bool(lo == hi):
        return [torch.tensor(float(v), dtype=torch.float64).float()]
    return [lo, hi]


def ref_advantages(r, v):
    """``prepare_dataset``'s ``(adv - adv.mean()) / (adv.std() + 1e-8)`` with exact statistics: ``d = r - v`` in fp32, its mean and
    unbiased variance in float64 (two passes), ``mean_f = f32(mean)``, ``den_f = f32(sqrt(var)) + f32(1e-8)`` in fp32, then
    ``y = (d - mean_f) / den_f`` in fp32.  Returns (y, ambiguous, candidates): ``ambiguous`` is set when the fp32 rounding of the mean
    or of the standard deviation changes under a 1e-12 relative perturbation of its float64 value (a kernel that sums in another order
    may then round the other way); ``candidates`` holds ``y`` for every combination of the possible roundings (``[y]`` otherwise)."""
    d = r.reshape(-1).cpu().float() - v.reshape(-1).cpu().float()
    d64 = d.double()
    n = d64.numel()
    mean = d64.sum() / n
    var = ((d64 - mean) ** 2).sum() / (n - 1) if n > 1 else torch.tensor(float("nan"), dtype=torch.float64)
    std = torch.sqrt(var)

    def normalise(mf, sf):
        den = f32(sf.double() + EPS_F32_1E8.double())
        return f32(f32(d.double() - mf.double()).double() / den.double())

    y = normalise(mean.float(), std.float())
    cands = [normalise(mf, sf) for mf, sf in itertools.product(_roundings(mean), _roundings(std))]
    return y, len(cands) > 1, cands


def bits_equal(a, b):
    """Element-wise: the same fp32 bit pattern, or NaN in both (any payload)."""
    a, b = a.detach().cpu().float().contiguous(), b.detach().cpu().float().contiguous()
    assert a.shape == b.shape, (tuple(a.shape), tuple(b.shape))
    return (a.view(torch.int32) == b.view(torch.int32)) | (torch.isnan(a) & torch.isnan(b))
