"""GPU: the learner's statistics kernels on every branch training takes, against the float64 references of
``tests/learner_reference.py``.  Normalised outputs are compared BIT FOR BIT: the kernels evaluate rl_games' fp32 expressions with
IEEE division and sqrt and without FMA contraction (``Mth`` in ``bezk_common.cuh``, ``-fmad=false`` in the Makefile), so given the
statistics a kernel wrote back, ``y`` has exactly one right answer.  Every output buffer sits between guard bands (``_util.Guarded``).

Which case reaches which branch (thresholds from the launcher constants; line numbers in ``csrc/``):

  fused  = one cooperative kernel (``fused_stats_kernel``, bezk_fused.cu:80), taken by ``bezk_rms_train_forward`` for c == 1
           (bezk_api.cu:623) and by ``bezk_adv_normalize_fused`` (bezk_api.cu:659) when 2 <= m <= B, where
           B = min(SMs, FOLD_MAXB = 160) * FUSED_MAX_STAGE_BYTES / 4 = min(SMs, 160) * 40960 (bezk_fused.cu:25, 38, 223-230);
           6 062 080 on a 148-SM B200.  Each of the grid's CTAs holds ceil(m / grid) rows (even); its unrolled loop moves
           8 x 256 rows per iteration, so m = 2048 / 2049 is the edge of that loop, m = 297 a single CTA with a ragged loop.
  chain  = moments (``flat_partials_kernel`` for c == 1, else the kernels below) -> finalize -> merge + normalise: m == 1 or m > B
           for c == 1, every m for c > 1.
  TMA    = ``rms_partials_tma_kernel`` (bezk_learner.cu:170): 16-byte aligned x, 64-row tiles (RMS_TR) whose byte sizes are multiples
           of 16, m >= 4 * 64, 4 * 64 * c * 4 <= 220 KB -- c <= 220 (bezk_learner.cu:530-532).  Grid: min(tiles, 148 * per_sm)
           with per_sm = 4 for c = 52 / 54 (55 KB rings) -> 592 CTAs (bezk_learner.cu:541-546).  CTA k owns tiles k, k + 592, ...:
           the in-loop refill (bezk_learner.cu:217) needs >= 4 tiles (m >= 3 * 592 * 64 + 1 = 113 665), reusing a stage with the
           flipped parity (bezk_learner.cu:215) needs >= 5 (m >= 4 * 592 * 64 + 1 = 151 553).
  plain  = ``rms_partials_kernel<VEC>`` (bezk_learner.cu:101) for everything else up to RMS_MAX_C = 256; VEC = 2 for even c and
           8-byte aligned x, else 1.  c = 257 is refused.

  A  train forward, c=1    m = 1                          chain; variance NaN like torch.var
                           m = 2, 3, 297, 2048, 2049,     fused: single CTA, ragged last CTA, the 8 x 256-row loop's edge
                               131072
                           m = B - 1, B, B + 1            fused / chain boundary
                           m = 8 388 608                  chain at the full grid (the default 262144 envs x 32)
                           slab (32, n, 1)[:, e0:e0+E]    fused slab addressing (E = 1001); scalar chain (E = B / 32 + 1); odd e0
     c=54                  m = 32768                      TMA, <= 1 tile per CTA (the training minibatch)
                           m = 4099 / 255                 plain, VEC = 2 (ragged tail not 16-byte sized / below 4 tiles)
                           view offset by one float       plain, VEC = 1; scalar normalisation
                           m = 113 700, 151 600, 400 002  TMA ring: refill, one wrap, several wraps + partial last tile
                           slabs T=32, E=1024 / E=100     TMA slabs / plain slabs
     c=52                  m = 4099                       TMA with a ragged (3-row, 624-byte) tail, 208-byte rows
     c=7, 220, 221, 256    m = 4099                       VEC = 1; TMA at the shared-memory limit (220) / plain (221); RMS_MAX_C
  B  sharded merge         2 and 3 uneven shards           rms_moments_ext -> summed heads -> rms_merge_normalize; adv_moments ->
                                                           summed heads -> adv_normalize (the multi-GPU path on one GPU)
  C  advantages            m = 1 and m > B: chain; 2 <= m <= B: fused (``normalize_advantages`` -> bezk_adv_normalize_fused)
  D  planned obs update    nmb minibatches share the 592 CTAs (bezk_learner.cu:604): nmb = 256 -> 2 CTAs x 256 tiles each (ring
                           wraps); nmb = 2048 > RMS_MAX_BLOCKS = 1184 -> per-batch launches; E = 100 (not a multiple of 64) -> per
                           batch plain slabs
  E  PPO loss slabs        T = 32, E = 20480: 5120 tiles of 128 on 592 CTAs (bezk_learner.cu:1041) -> 8-9 tiles per CTA, the
                           mbarrier phase flip (:855) and the mid-loop fp32 -> fp64 flush after PPO_FLUSH = 8 tiles (:954)
"""
import math

import pytest
import torch

from tests import learner_reference as R
from tests._util import Guarded

pytestmark = pytest.mark.gpu

EPS = 1e-5
# Error bound of a float64 sum as the kernels form it (serial per-thread chains of at most a few hundred terms at these sizes,
# then fixed-order folds over <= 1184 partials): |error| <= K * eps64 * sum(|terms|) with K = 1024, i.e. 2^-43 ~ 1.1e-13.
K_EPS = 2.0 ** -43


def _fused_limit():
    """B: the largest m the cooperative kernel takes (``fused_geometry``: min(SMs, 160) CTAs of at most 40960 fp32 rows)."""
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    return min(sms, 160) * 40960


def _resolve(m):
    if isinstance(m, int):
        return m
    return eval(m, {"B": _fused_limit()})              # "B-1", "B", "B+1", "B//32+1"


def bits_ok(a, b, what):
    ok = R.bits_equal(a, b)
    if not bool(ok.all()):
        bad = (~ok).nonzero()
        i = tuple(bad[0].tolist())
        a, b = a.detach().cpu(), b.detach().cpu()
        raise AssertionError(f"{what}: {bad.shape[0]} of {ok.numel()} elements differ in their bits; first at {i}: "
                             f"got {a[i].item()!r} want {b[i].item()!r}")


# ----------------------------------------------------------------------------------------------------------- inputs
SHIFT_COL, NAN_COL = 1, 3


def _obs(m, c, seed, kind="obs"):
    """fp32 rows (m, c): random columns of assorted scale / offset, column 1 with |mean| / std = 1e3, the last column constant like
    the ball_init columns 52:54 of the observation.  c == 1: ``kind`` picks the one column ("shift" or "const")."""
    g = torch.Generator().manual_seed(seed)
    if c == 1:
        x = 1000.0 + torch.randn(m, 1, generator=g) if kind == "shift" else torch.full((m, 1), 0.175)
        return x
    x = torch.randn(m, c, generator=g) * (torch.rand(c, generator=g) * 2 + 0.25) + torch.randn(c, generator=g) * 2
    x[:, SHIFT_COL] = 1000.0 + torch.randn(m, generator=g)
    x[:, -1] = 0.175
    if kind == "nan":
        x[m // 2, NAN_COL] = float("nan")
    return x


def _warm_state(c, kind="obs"):
    """A running state after training has started: means near the data's, variance 2, count 1000."""
    mean = torch.zeros(c, dtype=torch.float64)
    if c > 1 or kind == "shift":
        mean[SHIFT_COL if c > 1 else 0] = 1000.25
    if c > 1 or kind == "const":
        mean[-1] = 0.2
    return mean, torch.full((c,), 2.0, dtype=torch.float64), 1000.0


COLD = "cold"                                           # rl_games' (0, 1, 1) start


def _start(c, start, kind):
    if start == COLD:
        return torch.zeros(c, dtype=torch.float64), torch.ones(c, dtype=torch.float64), 1.0
    return _warm_state(c, kind)


# ----------------------------------------------------------------------------------------------------------- statistics checks
def check_stats(mean, var, count, ref, prev, rows, what):
    """Kernel statistics after one update against ``ref`` = ref_stats(prev, [rows]).

    count: exact.  The kernels sum (x - p) and (x - p)^2 in float64 with p = the running mean before the update, so
      mean: |err| <= 1e-12 (|mean| + std) + K_EPS * sum|x - p| / tot
      var:  |err| <= 1e-9 |var| + 4 K_EPS * sum (x - p)^2 / (B - 1) * B / tot
    The second var term is the pivot's cancellation: var_b = (SS - S^2 / B) / (B - 1) loses (mean_b - p)^2 / var_b of its relative
    precision.  With p near the batch mean it is ~4e-13 of var and the 1e-9 term rules; from the (0, 1, 1) start the first update
    pivots at 0 and the |mean| / std = 1e3 column cancels 1e6-fold: its bound is then ~4.4e-7 relative.  NaN exactly where ``ref``
    has NaN (a NaN input poisons its own column and no other)."""
    rmean, rvar, rcount = ref
    assert float(count) == rcount, f"{what}: count {float(count)} != {rcount}"
    mean, var = mean.detach().double().cpu(), var.detach().double().cpu()
    c = rmean.numel()
    x = rows.reshape(-1, c).double()
    b = x.shape[0]
    p = prev[0]
    dev = x - p
    s_abs, ss = dev.abs().sum(0), (dev * dev).sum(0)
    std = torch.nan_to_num(rvar.clamp_min(0).sqrt(), nan=0.0)
    tol_m = 1e-12 * (rmean.abs() + std) + K_EPS * s_abs / rcount
    tol_v = 1e-9 * rvar.abs() + 4 * K_EPS * ss / max(b - 1, 1) * b / rcount
    for got, want, tol, name in ((mean, rmean, tol_m, "mean"), (var, rvar, tol_v, "var")):
        nan = torch.isnan(want)
        assert torch.equal(torch.isnan(got), nan), f"{what}: {name} NaN in columns {torch.isnan(got).nonzero().view(-1).tolist()}, " \
                                                  f"want {nan.nonzero().view(-1).tolist()}"
        err = (got - want).abs()
        bad = (err > tol) & ~nan
        if bool(bad.any()):
            j = int(bad.nonzero()[0])
            raise AssertionError(f"{what}: running {name}[{j}] = {got[j].item()!r}, want {want[j].item()!r} (err {err[j].item():.3e} "
                                 f"> tol {tol[j].item():.3e})")


# ----------------------------------------------------------------------------------------------------------- A: train forward
def _rows_of(x, c):
    """The batch rows a (possibly slab-view) device input stands for, on the CPU, in the kernels' row order (t-major in a slab)."""
    return x.detach().cpu().reshape(-1, c)


def _train_forward_runs(inputs, c, start, kind, via_module):
    """Three train-mode forwards from ``start``; returns [(y, mean, var, count)] per update, and the guard set."""
    from bez_isaacgym_b200 import ops
    from bez_isaacgym_b200.learner import RunningMeanStd
    g = Guarded()
    m0, v0, n0 = _start(c, start, kind)
    if via_module:
        mod = RunningMeanStd(c).cuda().train()
        mod.running_mean.copy_(m0); mod.running_var.copy_(v0); mod.count.fill_(n0)
        mean, var, count = mod.running_mean, mod.running_var, mod.count.view(1)
    else:
        mean = g.make((c,), torch.float64, fill=m0.cuda())
        var = g.make((c,), torch.float64, fill=v0.cuda())
        count = g.make((1,), torch.float64, fill=torch.tensor([n0], dtype=torch.float64, device="cuda"))
        scratch = g.make((ops.rms_scratch_doubles(c),), torch.float64)
    out = []
    for x in inputs:
        rows = x.shape[0] * x.shape[1] if not x.is_contiguous() else x.numel() // c
        y = g.make((rows, c))
        if via_module:
            mod(x, out=y)
        else:
            ops.rms_train_forward(x, mean, var, count, y, scratch, eps=EPS)
        out.append((y.cpu(), mean.cpu().clone(), var.cpu().clone(), count.cpu().clone()))
    g.check()
    return out


def _contiguous_inputs(m, c, seed, kind, offset=False):
    xs = []
    for it in range(3):
        x = _obs(m, c, seed + it, kind)
        if c == 1:
            x = x.view(m)
        if offset:                                      # 4-byte aligned only: VEC = 1 moments, scalar normalisation
            buf = torch.empty(m * c + 1, device="cuda")
            buf[1:].copy_(x.reshape(-1).cuda())
            xs.append(buf[1:].view(m, c))
        else:
            xs.append(x.cuda())
    return xs


def _slab_inputs(T, E, e0, c, seed, kind):
    n = e0 + E + 3
    xs = []
    for it in range(3):
        st = _obs(T * n, c, seed + it, kind).view(T, n, c).cuda()
        xs.append(st[:, e0:e0 + E])
    return xs


A_CASES = [
    # (c, m, kind, layout); layout: "rows", "offset", or ("slabs", T, E, e0)
    (1, 1, "shift", "rows"), (1, 2, "shift", "rows"), (1, 3, "shift", "rows"), (1, 297, "shift", "rows"),
    (1, 2048, "shift", "rows"), (1, 2049, "const", "rows"), (1, 131072, "shift", "rows"),
    (1, "B-1", "shift", "rows"), (1, "B", "const", "rows"), (1, "B+1", "shift", "rows"), (1, 8388608, "shift", "rows"),
    (1, None, "shift", ("slabs", 32, 1001, 3)), (1, None, "shift", ("slabs", 32, "B//32+1", 1)),
    (54, 32768, "obs", "rows"), (54, 4099, "nan", "rows"), (54, 255, "obs", "rows"), (54, 3001, "obs", "offset"),
    (52, 4099, "obs", "rows"), (54, 113700, "obs", "rows"), (54, 151600, "obs", "rows"), (54, 400002, "obs", "rows"),
    (54, None, "obs", ("slabs", 32, 1024, 64)), (54, None, "obs", ("slabs", 32, 100, 7)),
    (7, 4099, "obs", "rows"), (220, 4099, "obs", "rows"), (221, 4099, "obs", "rows"), (256, 4099, "obs", "rows"),
]


def _a_id(case):
    c, m, kind, layout = case
    lay = layout if isinstance(layout, str) else f"slabs{layout[1]}x{layout[2]}@{layout[3]}"
    return f"c{c}-m{m}-{kind}-{lay}"


@pytest.mark.parametrize("case", A_CASES, ids=[_a_id(k) for k in A_CASES])
@pytest.mark.parametrize("start", ["warm", COLD])
def test_train_forward_matches_reference(case, start):
    """``RunningMeanStd.forward`` in train mode (run 1) and ``ops.rms_train_forward`` (run 2, every buffer guarded), three updates
    each: exact count, statistics against ``ref_stats``, ``y`` against ``ref_normalize`` with the kernel's own statistics bit for
    bit, and the two runs bit-identical."""
    c, m, kind, layout = case
    seed = 1000 * c + (_resolve(m) % 997 if m is not None else 5)
    if layout == "rows" or layout == "offset":
        inputs = _contiguous_inputs(_resolve(m), c, seed, kind, offset=layout == "offset")
    else:
        _, T, E, e0 = layout
        inputs = _slab_inputs(T, _resolve(E), e0, c, seed, kind)
    runs = [_train_forward_runs(inputs, c, start, kind, via_module) for via_module in (True, False)]
    prev = _start(c, start, kind)
    for u, x in enumerate(inputs):
        rows = _rows_of(x, c)
        ref = R.ref_stats(prev[0], prev[1], prev[2], [rows])
        y, mean, var, count = runs[0][u]
        check_stats(mean, var, count, ref, prev, rows, f"update {u}")
        bits_ok(y.view(-1, c), R.ref_normalize(rows, mean, var, EPS), f"y of update {u}")
        bits_ok(runs[1][u][0], y, f"run 2 vs run 1: y of update {u}")
        for a, b, name in zip(runs[1][u][1:], runs[0][u][1:], ("mean", "var", "count")):
            assert bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all()), f"run 2 vs run 1: {name} of update {u}"
        prev = ref
    if kind == "nan":                                   # only the poisoned column goes NaN
        y, mean, var, _ = runs[0][0]
        assert bool(torch.isnan(mean[NAN_COL])) and int(torch.isnan(mean).sum()) == 1
        assert bool(torch.isnan(y.view(-1, c)[:, NAN_COL]).all())
        assert int(torch.isnan(y).sum()) == y.view(-1, c).shape[0]
    if m == 1:
        assert bool(torch.isnan(runs[0][0][2]).all()), "a one-row batch has NaN variance, like torch.var"


def test_train_forward_refuses_more_than_256_columns():
    from bez_isaacgym_b200 import ops
    from bez_isaacgym_b200._lib import BezkError
    c = 257
    x = torch.randn(4099, c, device="cuda")
    mean = torch.zeros(c, dtype=torch.float64, device="cuda"); var = torch.ones(c, dtype=torch.float64, device="cuda")
    count = torch.ones(1, dtype=torch.float64, device="cuda")
    with pytest.raises(BezkError):
        ops.rms_train_forward(x, mean, var, count, torch.empty_like(x),
                              torch.empty(ops.rms_scratch_doubles(c), dtype=torch.float64, device="cuda"))
    torch.cuda.synchronize()
    assert float(count) == 1.0 and bool((mean == 0).all())


# ----------------------------------------------------------------------------------------------------------- B: sharded merge
def _shards(layout, nshards, c, seed):
    """(union rows on the CPU, union as one contiguous device tensor, device shards)."""
    if layout == "rows":
        m = 50001
        x = _obs(m, c, seed, "shift" if c == 1 else "obs")
        cuts = [0, 17000, m] if nshards == 2 else [0, 9001, 31337, m]
        xd = x.cuda()
        shards = [xd[a:b] for a, b in zip(cuts[:-1], cuts[1:])]
        return x, xd, shards
    T, n = 16, 3002
    st = _obs(T * n, c, seed, "shift" if c == 1 else "obs").view(T, n, c).cuda()
    cuts = [0, 1024, n] if nshards == 2 else [0, 1024, 2001, n]
    shards = [st[:, a:b] for a, b in zip(cuts[:-1], cuts[1:])]
    return st.cpu().reshape(-1, c), st.reshape(-1, c), shards


@pytest.mark.parametrize("layout", ["rows", "slabs"])
@pytest.mark.parametrize("nshards", [2, 3])
@pytest.mark.parametrize("c", [1, 54])
def test_sharded_rms_merge_on_one_gpu(c, nshards, layout):
    """The multi-GPU train forward with the all-reduce done by hand: ``rms_moments_ext`` per shard, the shards' [:1 + 2c] heads
    summed and written back to every shard, ``rms_merge_normalize`` per shard.  Every shard ends with the same statistics bit for
    bit, equal to ``rms_train_forward`` on the union to 1e-12 and to ``ref_stats``; each shard's ``y`` is ``ref_normalize``'s."""
    from bez_isaacgym_b200 import ops
    kind = "shift" if c == 1 else "obs"
    union_cpu, union_dev, shards = _shards(layout, nshards, c, seed=77 + c + nshards)
    m0, v0, n0 = _warm_state(c, kind)
    g = Guarded()
    st = []
    for x in shards:
        rows = x.shape[0] * x.shape[1] if x.dim() == 3 else x.shape[0]
        st.append(dict(x=x, mean=g.make((c,), torch.float64, fill=m0.cuda()), var=g.make((c,), torch.float64, fill=v0.cuda()),
                       count=g.make((1,), torch.float64, fill=torch.tensor([n0], dtype=torch.float64, device="cuda")),
                       acc=g.make((2 + 4 * c,), torch.float64), scratch=g.make((ops.rms_scratch_doubles(c),), torch.float64),
                       y=g.make((rows, c))))
    for s in st:
        ops.rms_moments_ext(s["x"], s["mean"], s["var"], s["count"], s["acc"], s["scratch"])
    head = st[0]["acc"][:1 + 2 * c].clone()
    for s in st[1:]:
        head += s["acc"][:1 + 2 * c]
    for s in st:
        s["acc"][:1 + 2 * c].copy_(head)
    for s in st:
        ops.rms_merge_normalize(s["x"], s["acc"], s["mean"], s["var"], s["count"], s["y"], eps=EPS)
    g.check()
    for s in st[1:]:
        for k in ("mean", "var", "count"):
            assert torch.equal(s[k], st[0][k]), f"shards disagree on {k}"
    mean, var, count = st[0]["mean"].cpu(), st[0]["var"].cpu(), st[0]["count"].cpu()
    # the union in one call
    um, uv, uc = m0.cuda(), v0.cuda(), torch.tensor([n0], dtype=torch.float64, device="cuda")
    ops.rms_train_forward(union_dev if c > 1 else union_dev.view(-1), um, uv, uc, torch.empty_like(union_dev),
                          torch.empty(ops.rms_scratch_doubles(c), dtype=torch.float64, device="cuda"), eps=EPS)
    assert float(count) == float(uc) == n0 + union_cpu.shape[0]
    std = uv.cpu().clamp_min(0).sqrt()
    assert bool(((mean - um.cpu()).abs() <= 1e-12 * (um.cpu().abs() + std)).all()), "mean vs the union's train forward"
    assert bool(((var - uv.cpu()).abs() <= 1e-12 * uv.cpu().abs()).all()), "var vs the union's train forward"
    check_stats(mean, var, count, R.ref_stats(m0, v0, n0, [union_cpu]), (m0, v0, n0), union_cpu, "shards vs ref_stats")
    for k, s in enumerate(st):
        bits_ok(s["y"], R.ref_normalize(_rows_of(s["x"], c), mean, var, EPS), f"y of shard {k}")


def _adv_check(out, r, v, what):
    """``out`` against ``ref_advantages(r, v)``: bit for bit, or -- where the float64 statistics sit within 1e-12 of an fp32
    rounding boundary -- equal to one of the candidate roundings, element by element."""
    y, ambiguous, cands = R.ref_advantages(r, v)
    if not ambiguous:
        bits_ok(out, y, what)
        return
    ok = torch.zeros(y.shape, dtype=torch.bool)
    for cnd in cands:
        ok |= R.bits_equal(out, cnd)
    assert bool(ok.all()), f"{what}: {int((~ok).sum())} elements match none of the {len(cands)} candidate roundings"


@pytest.mark.parametrize("m", [4099, 1000003])
@pytest.mark.parametrize("nshards", [2, 3])
def test_sharded_advantages_on_one_gpu(m, nshards):
    """``adv_moments`` per shard, the [B, S, SS] heads summed and handed to every shard's ``adv_normalize``: the global
    normalisation ``normalize_advantages`` does with a process group, compared against ``ref_advantages`` on the union."""
    from bez_isaacgym_b200 import ops
    gen = torch.Generator().manual_seed(m + nshards)
    r, v = torch.randn(m, generator=gen) * 2 + 0.3, torch.randn(m, generator=gen)
    cuts = [0, m // 3 + 1, m] if nshards == 2 else [0, m // 5 + 3, m // 2 + 1, m]
    g = Guarded()
    rd, vd = r.cuda(), v.cuda()
    parts = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        parts.append(dict(r=rd[a:b], v=vd[a:b], acc=g.make((3,), torch.float64),
                          scratch=g.make((ops.rms_scratch_doubles(1),), torch.float64), out=g.make((b - a,))))
    for p in parts:
        ops.adv_moments(p["r"], p["v"], p["acc"], p["scratch"])
    head = parts[0]["acc"].clone()
    for p in parts[1:]:
        head += p["acc"]
    for p in parts:
        ops.adv_normalize(p["r"], p["v"], head, p["out"])
    g.check()
    assert float(head[0]) == m
    _adv_check(torch.cat([p["out"].cpu() for p in parts]), r, v, f"{nshards} shards")


# ----------------------------------------------------------------------------------------------------------- C: advantages
ADV_SHAPES = [(1, 1), (2, 1), (3, 1), (27, 11), (32, 4096), (5, 26215), (32, "B//32"), (1, "B+1"), (32, 262144)]


@pytest.mark.parametrize("T,n", ADV_SHAPES, ids=[f"{t}x{n}" for t, n in ADV_SHAPES])
def test_normalize_advantages_matches_reference(T, n):
    """``normalize_advantages`` on the (T, n, 1) tensors the agent passes, into a guarded ``out=``: ``r - v`` exactly without
    normalisation; with it, ``ref_advantages`` bit for bit and within ``prepare_dataset``'s tolerance; NaN for one sample like
    torch.std; exactly 0 for constant advantages."""
    from bez_isaacgym_b200.learner import a2c_common
    from oracle import rl_games_oracle as rg
    n = _resolve(n)
    m = T * n
    gen = torch.Generator().manual_seed(m)
    r, v = torch.randn(T, n, 1, generator=gen) * 2 + 0.3, torch.randn(T, n, 1, generator=gen)
    rd, vd = r.cuda(), v.cuda()
    g = Guarded()
    raw, out = g.make((m,)), g.make((m,))
    a2c_common.normalize_advantages(rd, vd, normalize=False, out=raw)
    a2c_common.normalize_advantages(rd, vd, normalize=True, out=out)
    g.check()
    bits_ok(raw, (r - v).view(-1), "normalize=False")
    _adv_check(out.cpu(), r, v, "normalize=True")
    want, _, _ = rg.prepare_dataset(r.view(-1, 1), v.view(-1, 1), rg.RunningMeanStd(1))
    torch.testing.assert_close(out.cpu(), want, rtol=1e-5, atol=2e-6, equal_nan=True)
    if m == 1:
        assert bool(torch.isnan(out).all()), "one sample: torch.std is NaN, so is the normalised advantage"
        return
    const = g.make((m,))
    a2c_common.normalize_advantages(torch.full_like(rd, 0.7), torch.full_like(vd, 0.2), out=const)
    g.check()
    assert torch.equal(const.cpu(), torch.zeros(m)), "constant advantages normalise to exactly 0"


# ----------------------------------------------------------------------------------------------------------- D: planned update
def _plan_cases():
    cases = []
    for c in (54, 52):
        for layout in ("rows", "slabs"):
            cases += [(c, nmb, 32, E, layout) for nmb in (1, 3, 4) for E in (64, 100, 1024)]
            cases += [(c, 256, 32, 64, layout), (c, 2048, 4, 64, layout)]
    return cases


PLAN_CASES = _plan_cases()


@pytest.mark.parametrize("c,nmb,T,E,layout", PLAN_CASES, ids=[f"c{c}-nmb{k}-T{t}-E{e}-{lay}" for c, k, t, e, lay in PLAN_CASES])
def test_planned_obs_update_at_training_geometry(c, nmb, T, E, layout):
    """``RunningMeanStd.plan`` over the epoch's minibatches (order ``range(nmb) * 5``) and ``planned_group`` per mini-epoch: every
    accumulator row equals that batch's ``rms_moments_slabs`` to 1e-13 and the float64 pivoted sums within their rounding bound,
    ``seq`` equals a float64 replay of the merges bit for bit, and each normalised minibatch is ``ref_normalize``'s with ``seq[u]``
    bit for bit."""
    from bez_isaacgym_b200 import ops
    from bez_isaacgym_b200.learner import RunningMeanStd
    mini_epochs = 5
    n = nmb * E
    obses = _obs(T * n, c, seed=c * 100003 + nmb * 101 + E).view(T, n, c).cuda()
    if layout == "slabs":
        batches = [obses[:, i * E:(i + 1) * E] for i in range(nmb)]
    else:                                               # equally spaced contiguous blocks of one tensor, same rows
        blocks = torch.stack([obses[:, i * E:(i + 1) * E].reshape(-1, c) for i in range(nmb)])
        batches = [blocks[i] for i in range(nmb)]
    order = list(range(nmb)) * mini_epochs
    mod = RunningMeanStd(c).cuda().train()
    m0, v0, n0 = _warm_state(c)
    mod.running_mean.copy_(m0); mod.running_var.copy_(v0); mod.count.fill_(n0)
    seq = mod.plan(batches, order).cpu()
    acc = mod._plan_acc.cpu()
    pivot = m0
    # accumulator rows: the same moments per batch, one launch each
    scratch = torch.empty(ops.rms_scratch_doubles(c), dtype=torch.float64, device="cuda")
    one = torch.empty(1 + 2 * c, dtype=torch.float64, device="cuda")
    rows = obses.cpu().view(T, nmb, E, c).transpose(0, 1).reshape(nmb, T * E, c).double()      # every batch's rows, t-major
    dev = rows - pivot
    s_abs, ss = dev.abs().sum(1), (dev * dev).sum(1)
    want = torch.cat([torch.full((nmb, 1), float(T * E), dtype=torch.float64), dev.sum(1), ss], 1)
    for i, b in enumerate(batches):
        ops.rms_moments_slabs(b, mod._pivot, one, scratch)
        per = one.cpu()
        assert float(acc[i, 0]) == float(per[0]) == T * E
        assert bool(((acc[i, 1:] - per[1:]).abs() <= 1e-13 * torch.cat([s_abs[i], ss[i]])).all()), f"acc row {i} vs its own launch"
    assert bool(((acc[:, 1:] - want[:, 1:]).abs() <= K_EPS * torch.cat([s_abs, ss], 1)).all()), "acc vs float64 pivoted sums"
    # the sequence of merges
    seq_ref, cnt = R.replay_merges(acc, order, pivot, m0, v0, n0)
    assert torch.equal(seq, seq_ref), "seq vs the float64 replay of the merges"
    assert float(mod.count) == cnt == n0 + mini_epochs * T * n
    assert torch.equal(mod.running_mean.cpu(), seq_ref[-1, 0]) and torch.equal(mod.running_var.cpu(), seq_ref[-1, 1])
    # one normalise launch per mini-epoch
    g = Guarded()
    y = g.make((nmb, T * E, c))
    x32 = rows.float()
    for me in range(mini_epochs):
        mod.planned_group(me * nmb, batches, out=y)
        g.check()
        u = slice(me * nmb, (me + 1) * nmb)
        bits_ok(y, R.ref_normalize(x32, seq[u, 0].unsqueeze(1), seq[u, 1].unsqueeze(1), EPS), f"mini-epoch {me}")


# ----------------------------------------------------------------------------------------------------------- E: PPO loss slabs
def test_ppo_loss_slabs_multi_tile_equals_the_flat_minibatch():
    """T = 32, E = 20480 read in place from (T, N) rollout storage: 8-9 tiles per CTA with the mid-loop flush.  Per-sample outputs,
    the gradients and the loss statistics equal ``ppo_loss`` on the same minibatch flattened, bit for bit (the same tiles in the same
    CTAs), and a second run repeats every bit."""
    from bez_isaacgym_b200 import ops
    import bez_isaacgym_b200.synthetic_gym as sg
    T, E, e0 = 32, 20480, 128
    n = E + 256
    m = T * E
    mb = {k: v.cuda() for k, v in sg.make_minibatch(m, seed=31).items()}
    mb["mu"][: m // 8] *= 4.0
    mb["advantages"][::5] *= -1.0
    store = {}
    for k in ("actions", "old_mu", "old_sigma"):
        s = torch.randn(T, n, 18, device="cuda").abs() + 0.5
        s[:, e0:e0 + E] = mb[k].view(T, E, 18)
        store[k] = s
    for k in ("old_values", "returns", "old_neglogp", "advantages"):
        s = torch.randn(T, n, device="cuda")
        s[:, e0:e0 + E] = mb[k].reshape(T, E)
        store[k] = s
    sl = {k: v[:, e0:e0 + E] for k, v in store.items()}
    flat = {k: v.contiguous().view(m, -1) if v.dim() == 3 else v.contiguous().view(m) for k, v in sl.items()}
    cfg = ops.make_ppo_cfg()
    g = Guarded()

    def run(fn, src):
        o = dict(stats=g.make((8,), torch.float64), part=g.make((ops.ppo_scratch_doubles(),), torch.float64),
                 grad_mu=g.make((m, 18)), grad_values=g.make((m,)), grad_logstd=g.make((18,)), neglogp_out=g.make((m,)))
        fn(src["actions"], mb["mu"], mb["logstd"], src["old_mu"], src["old_sigma"], mb["values"].view(-1), src["old_values"],
           src["returns"], src["old_neglogp"], src["advantages"], cfg, o["stats"], o["part"], grad_mu=o["grad_mu"],
           grad_values=o["grad_values"], grad_logstd=o["grad_logstd"], neglogp_out=o["neglogp_out"])
        g.check()
        return {k: v.cpu() for k, v in o.items() if k != "part"}

    a = run(ops.ppo_loss_slabs, sl)
    b = run(ops.ppo_loss, flat)
    a2 = run(ops.ppo_loss_slabs, sl)
    assert bool(torch.isfinite(a["stats"]).all())
    for k in a:
        assert torch.equal(a[k], b[k]), f"slabs vs flat: {k}"
        assert torch.equal(a2[k], a[k]), f"second run: {k}"
    assert math.isfinite(float(a["stats"][0]))
