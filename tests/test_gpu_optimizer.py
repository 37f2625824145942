"""The optimizer tail of the training step on the GPU (csrc/train.cu: dadd_sumsq, dadd_clip_coef, dadd_adamw_step(_dev),
dadd_minsnr_mse) against float64 references computed on the CPU from the same float32 inputs the kernels see: ragged sizes
(n % 4 != 0 tails, which thread 0 of block 0 handles), buffers longer than one grid-stride pass, non-finite gradients.  Then the
trainer's loss-scaled, skip-on-overflow step against torch.amp.GradScaler (Lightning "16-mixed" with gradient clipping), eager,
as a captured graph and across a checkpoint."""

import math
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
U = 2.0 ** -24                      # unit roundoff of fp32, round to nearest
INF, NAN = float("inf"), float("nan")


def _ops():
    from progressive_stable_diffusion_b200 import ops
    return ops


def f32(x: float) -> float:
    return float(np.float32(x))


def _bits(t: torch.Tensor) -> torch.Tensor:
    return t.detach().view(torch.int32).cpu()


# ------------------------------------------------------------------------------------------------ sum of squares + clip coefficient
SUMSQ_SIZES = [0, 1, 3, 4, 5, 4 * 296 * 256, 3_000_003]          # 3 000 003: 2.5 grid-stride passes at 296 x 256 threads


def _clip_checks(part: torch.Tensor, sumsq64: float, ctx) -> None:
    """dadd_clip_coef over ``part`` against clip_grad_norm_'s arithmetic in float64, for every grad_scale / max_norm regime."""
    ops = _ops()
    coef = torch.empty(2, device=DEV)
    for gs in (1.0, 2.0 ** -13, 0.5):
        norm = gs * math.sqrt(sumsq64)
        for max_norm in [0.0, 3.0 * norm + 1.0] + ([norm / 3.0] if norm > 0 else []):
            ops.clip_coef_(part, max_norm, gs, coef)
            c, got = coef.tolist()
            assert got == pytest.approx(norm, rel=1e-6, abs=0.0), (ctx, gs, max_norm)
            if max_norm == 0.0 or max_norm > norm:
                assert c == gs, (ctx, gs, max_norm, c)                # no clipping: exactly the grad scale
            else:
                assert c == pytest.approx(gs * max_norm / (norm + 1e-6), rel=1e-6), (ctx, gs, max_norm)


@pytest.mark.parametrize("partials", ["one", "all"])
@pytest.mark.parametrize("n", SUMSQ_SIZES)
def test_sumsq_and_clip_coef_match_float64(n, partials):
    ops = _ops()
    k = 1 if partials == "one" else ops.SUMSQ_PARTIALS
    gen = torch.Generator().manual_seed(n + k)
    host = torch.randn(n, generator=gen) * torch.rand(n, generator=gen).mul(6.0).exp2()     # magnitudes over 2^0 .. 2^6
    g = host.to(DEV)                                             # (n = 0: torch gives an empty tensor no address)
    part = torch.full((k,), NAN, device=DEV)                     # every partial must be written, empty blocks included
    ops.sumsq_(g, part)
    assert torch.isfinite(part).all()
    ss = float((host.double() ** 2).sum())
    assert part.double().sum().item() == pytest.approx(ss, rel=2e-6, abs=0.0)
    _clip_checks(part, ss, (n, k))


def test_clip_coef_over_the_partials_of_several_buffers():
    """The trainer's layout: one row of SUMSQ_PARTIALS partial sums per bucket, one clip over all of them."""
    ops = _ops()
    sizes = [5, 4 * 296 * 256, 3, 1027, 1]
    gen = torch.Generator().manual_seed(17)
    hosts = [torch.randn(n, generator=gen) * (i + 1) for i, n in enumerate(sizes)]
    part = torch.full((len(sizes), ops.SUMSQ_PARTIALS), NAN, device=DEV)
    bufs = [h.to(DEV) for h in hosts]
    for i, g in enumerate(bufs):
        ops.sumsq_(g, part[i])
    _clip_checks(part.view(-1), float(sum((h.double() ** 2).sum() for h in hosts)), sizes)


@pytest.mark.parametrize("where", ["first", "middle_lane", "last_tail"])
@pytest.mark.parametrize("partials", ["one", "all"])
@pytest.mark.parametrize("n", [4099, 3_000_003])
def test_non_finite_gradient_poisons_the_clip_coefficient(n, partials, where):
    """+inf at index 0, NaN in one lane of a float4 in the middle, inf in the last (scalar tail) element: coef[0] = NaN (the AdamW
    launches skip the step) and a non-finite norm, whatever the clip and grad-scale settings."""
    ops = _ops()
    assert n % 4 == 3
    k = 1 if partials == "one" else ops.SUMSQ_PARTIALS
    host = torch.randn(n, generator=torch.Generator().manual_seed(n))
    i, val = {"first": (0, INF), "middle_lane": ((n // 8) * 4 + 2, NAN), "last_tail": (n - 1, INF)}[where]
    host[i] = val
    part = torch.empty(k, device=DEV)
    ops.sumsq_(host.to(DEV), part)
    coef = torch.empty(2, device=DEV)
    for gs in (1.0, 2.0 ** -13):
        for max_norm in (0.0, 1.0):
            ops.clip_coef_(part, max_norm, gs, coef)
            c, norm = coef.tolist()
            assert math.isnan(c) and not math.isfinite(norm), (where, gs, max_norm, c, norm)


# ------------------------------------------------------------------------------------------------ AdamW
B1, B2, EPS = f32(0.9), f32(0.999), f32(1e-8)       # the kernels take float32 hyper-parameters: the reference uses the same values
ADAM_SIZES = [1, 3, 5, 4099, 3_000_003]              # 3 000 003: 2.5 grid-stride passes at 8 x 148 blocks


def _adamw64(p, g, m, v, c, lr, wd, t):
    """One torch.optim.AdamW step in float64 (documented update: decoupled decay, then the moments, then the bias-corrected step)
    on the kernel's float32 inputs, with a per-element bound on |fp32 result - exact| from the roundings the kernel performs:
    one per fp32 operation (2 for rsqrtf), 1 - powf(beta, t) within 4 ulp of beta^t, amplified by the cancellation."""
    gk = g * c
    m1 = B1 * m + (1 - B1) * gk
    v1 = B2 * v + (1 - B2) * gk * gk
    pd = p * (1 - lr * wd)
    bc1, bc2 = 1 - B1 ** t, 1 - B2 ** t
    s = v1.sqrt() / math.sqrt(bc2)
    den = s + EPS
    upd = (lr / bc1) * m1 / den
    p1 = pd - upd
    tm = U * m1.abs() + 2 * U * (1 - B1) * gk.abs()
    tv = U * v1 + 4 * U * (1 - B2) * gk * gk
    ebc1, ebc2 = U + 8 * U * B1 ** t / bc1, U + 8 * U * B2 ** t / bc2
    rel = 12 * U + ebc1 + ebc2 / 2 + (s / den) * torch.where(v1 > 0, tv / (2 * v1), torch.zeros_like(v1))
    tp = 4 * U * pd.abs() + upd.abs() * rel + (lr / bc1) / den * tm + U * p1.abs()
    bc_gap = upd.abs() * (ebc1 + ebc2 / 2 + 4 * U)          # how far two roundings of the bias corrections can move the update
    return (p1, m1, v1), (2 * tp, 2 * tm, 2 * tv), 2 * bc_gap      # (x2: second-order terms)


def _ulp(x: torch.Tensor) -> torch.Tensor:
    a = x.abs().cpu().numpy().astype(np.float32)
    return torch.from_numpy(np.spacing(a).astype(np.float64))


@pytest.mark.parametrize("wd", [0.0, 0.05])
@pytest.mark.parametrize("n", ADAM_SIZES)
def test_adamw_both_entry_points_match_float64(n, wd):
    """20 steps of dadd_adamw_step_dev (lr scale and t on the device) and dadd_adamw_step (bias corrections from the host) from
    the same fp32 state, each checked element by element against one float64 AdamW step; the lr scale follows the epoch
    schedule and coef is None, a constant and a per-step value in turn.  The two entry points agree: m and v bit for bit, p
    within 2 ulps plus what the two bias corrections' own errors can move the update (powf on the device, double on the host).
    A NaN coef leaves p, m and v bit-identical."""
    from progressive_stable_diffusion_b200.training import warmup_cosine_lr
    ops = _ops()
    gen = torch.Generator().manual_seed(n * 10 + int(wd * 100))
    lr, wd = f32(1e-2), f32(wd)
    p = (torch.rand(n, generator=gen) + 0.25) * torch.randn(n, generator=gen).sign()
    state = [p.to(DEV), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)]
    dev_state = torch.tensor([1.0, 0.0], device=DEV)
    const = torch.tensor([f32(0.37), 0.0], device=DEV)
    nan_coef = torch.tensor([NAN, 0.0], device=DEV)
    for t in range(1, 21):
        scale = f32(warmup_cosine_lr((t - 1) // 4, 1.0, 2, 6, 0.01, 0.0))            # warm-up, then cosine, per "epoch" of 4 steps
        g_host = torch.randn(n, generator=gen) * 10.0 ** (3.0 * torch.rand(1, generator=gen).item() - 2.0)
        coef = (None, const, torch.tensor([f32(0.5 ** (t % 5) * (0.2 + 0.8 * torch.rand(1, generator=gen).item())), 0.0], device=DEV))[t % 3]
        c = 1.0 if coef is None else coef[0].item()
        g = g_host.to(DEV)
        dev_state.copy_(torch.tensor([scale, float(t)]))
        lr_t = float(np.float32(lr) * np.float32(scale))                              # lr * dev_state[0] as the kernel rounds it
        a, b = [x.clone() for x in state], [x.clone() for x in state]
        ops.adamw_step_dev_(a[0], g, a[1], a[2], lr, B1, B2, EPS, wd, dev_state, coef)
        ops.adamw_step_(b[0], g, b[1], b[2], lr_t, B1, B2, EPS, wd, t, coef)
        p64, m64, v64 = (x.double().cpu() for x in state)
        want, tol, bc_gap = _adamw64(p64, g_host.double(), m64, v64, c, lr_t, wd, t)
        for name, w, tl, ga, gb in zip("pmv", want, tol, a, b):
            for variant, got in (("dev", ga), ("host", gb)):
                err = (got.double().cpu() - w).abs()
                bad = (err > tl).nonzero()
                assert bad.numel() == 0, (variant, name, t, n, bad[:4].flatten().tolist(), (err / tl).max().item())
        assert torch.equal(_bits(a[1]), _bits(b[1])) and torch.equal(_bits(a[2]), _bits(b[2])), t
        assert ((a[0] - b[0]).abs().double().cpu() <= 2 * _ulp(a[0]) + bc_gap).all(), t
        state = a
        if t in (1, 10):
            for call in (lambda s: ops.adamw_step_dev_(s[0], g, s[1], s[2], lr, B1, B2, EPS, wd, dev_state, nan_coef),
                         lambda s: ops.adamw_step_(s[0], g, s[1], s[2], lr_t, B1, B2, EPS, wd, t, nan_coef)):
                s = [x.clone() for x in state]
                call(s)
                assert all(torch.equal(_bits(x), _bits(y)) for x, y in zip(s, state)), t


# ------------------------------------------------------------------------------------------------ Min-SNR MSE loss
@pytest.mark.parametrize("upstream", [1.0, 8192.0])
@pytest.mark.parametrize("E", [4092, 4096, 16384, 65536, 262144, 360000])    # 262144: 64 slices; 360000: slice cap + grid stride
@pytest.mark.parametrize("B", [1, 3, 26])
def test_minsnr_mse_matches_float64(B, E, upstream):
    ops = _ops()
    gen = torch.Generator().manual_seed(B * 1000003 + E)
    pred, target = torch.randn(B, E, generator=gen), torch.randn(B, E, generator=gen) * 0.5
    w = torch.rand(B, generator=gen) + 0.05
    if B > 1:
        w[B // 2] = 0.0                                                   # Min-SNR weights can vanish
    loss, grad = ops.minsnr_mse(pred.to(DEV), target.to(DEV), w.to(DEV), need_grad=True, upstream=upstream)
    d = pred.double() - target.double()
    want = (w.double() * (d * d).mean(dim=1)).mean().item()
    assert loss.item() == pytest.approx(want, rel=1e-5)
    # grad = (2 w_b upstream / (B E)) * (pred - target): three fp32 roundings (the quotient, the difference, the product)
    gref = 2.0 * w.double()[:, None] * upstream / (B * E) * d
    err = (grad.double().cpu() - gref).abs()
    assert (err <= 3.0001 * U * gref.abs()).all(), (err / (gref.abs() * U + 1e-300)).max().item()
    loss2, none = ops.minsnr_mse(pred.to(DEV), target.to(DEV), w.to(DEV), need_grad=False, upstream=upstream)
    assert none is None and torch.equal(_bits(loss2.reshape(1)), _bits(loss.reshape(1)))


# ------------------------------------------------------------------------------------------------ the trainer's step
TRAINER_KW = dict(lr=1e-2, weight_decay=0.05, max_grad_norm=0.5, bucket_bytes=64, ema_decay=0.9, ema_update_every_n_steps=1,
                  ema_update_starting_at_step=0)


def _tiny_trainer(**kw):
    """The 6 -> 5 -> 4 MLP of the CPU tests on the fused CUDA optimizer, fp32, several gradient buckets."""
    from progressive_stable_diffusion_b200 import training as T
    from tests.test_training_cpu import _Tiny
    m = _Tiny().to(DEV)
    tr = T.DataParallelTrainer(m, **dict(TRAINER_KW, **kw))
    assert len(tr.buckets) > 2
    return m, tr


def _data():
    gen = torch.Generator().manual_seed(12)
    return torch.randn(16, 6, generator=gen).to(DEV), torch.randn(16, 4, generator=gen).to(DEV)


def _snapshot(tr):
    """Raw bits of p, m, v and the EMA of every bucket (moments not yet allocated read as zeros), and of {lr scale, t}."""
    zero = lambda bk: torch.zeros_like(bk.flat_p)
    out = {"dev_state": _bits(tr.dev_state)}
    for i, bk in enumerate(tr.buckets):
        out[f"p{i}"] = _bits(bk.flat_p)
        out[f"m{i}"] = _bits(zero(bk) if bk.m is None else bk.m)
        out[f"v{i}"] = _bits(zero(bk) if bk.v is None else bk.v)
        out[f"avg{i}"] = _bits(bk.avg)
    return out


def _differ(a, b, keys=None):
    return [k for k in (keys or a) if not torch.equal(a[k], b[k])]


def _pmv(snap):
    return [k for k in snap if k[0] in "pmv"]


def test_power_of_two_loss_scale_is_exact():
    """Scaling the loss by 2^13 scales every gradient exactly in fp32, and the clip folds 2^-13 back in exactly (sum of squares
    2^26 x, its square root 2^13 x, coef 2^-13 x, g * coef): p, m, v, the EMA and the gradient norm are bit-identical to
    loss_scale = 1."""
    x, y = _data()
    ma, ta = _tiny_trainer(loss_scale=1.0)
    mb, tb = _tiny_trainer(loss_scale=2.0 ** 13)
    for s in range(5):
        la = ta.step(lambda: ((ma(x) - y) ** 2).mean())
        lb = tb.step(lambda: ((mb(x) - y) ** 2).mean())
        assert torch.equal(la, lb)
        assert torch.equal(_bits(ta.grad_norm.reshape(1)), _bits(tb.grad_norm.reshape(1))), s
        assert (tb.coef[0] * 2.0 ** 13).item() == ta.coef[0].item()
        assert not _differ(_snapshot(ta), _snapshot(tb)), (s, _differ(_snapshot(ta), _snapshot(tb)))


@pytest.mark.parametrize("overflow_at,steps", [(1, 5), (3, 7)], ids=["first_of_5", "third_of_7"])
def test_loss_scaled_step_matches_grad_scaler(overflow_at, steps):
    """The fused step against Lightning's "16-mixed" step with gradient clipping: GradScaler(init_scale=2^13) scale -> backward ->
    unscale_ -> clip_grad_norm_ -> scaler.step(AdamW) -> update, with the loss of one step multiplied by a device inf.  The
    overflowed step leaves p, m, v bit for bit and AdamW's t (dev_state[1]) where they were; the trainer's caller halves the
    loss scale as the scaler does; the EMA still averages (the callback runs on every batch)."""
    from torch.optim.swa_utils import AveragedModel, get_ema_avg_fn
    from progressive_stable_diffusion_b200 import training as T
    from tests.test_training_cpu import _Tiny
    x, y = _data()
    scale = 2.0 ** 13
    m, tr = _tiny_trainer(loss_scale=scale)
    ref = _Tiny().to(DEV)
    ref.load_state_dict(m.state_dict())
    used = [p for n, p in ref.named_parameters() if n not in T.UNUSED_PARAMETERS]
    groups = [{"params": [p for p in g["params"] if any(p is q for q in used)], "lr": g["lr"]} for g in T.parameter_groups(ref, 1e-2)]
    opt = torch.optim.AdamW(groups, weight_decay=0.05)
    scaler = torch.amp.GradScaler("cuda", init_scale=scale, growth_interval=10 ** 9)
    avg = AveragedModel(ref, avg_fn=get_ema_avg_fn(0.9), use_buffers=True)
    flag = torch.ones((), device=DEV)
    applied = 0
    for s in range(1, steps + 1):
        flag.fill_(INF if s == overflow_at else 1.0)
        before = _snapshot(tr)
        tr.step(lambda: ((m(x) - y) ** 2).mean() * flag)
        opt.zero_grad()
        scaler.scale(((ref(x) - y) ** 2).mean() * flag).backward()
        scaler.unscale_(opt)
        norm = torch.nn.utils.clip_grad_norm_(used, 0.5)
        scaler.step(opt)
        scaler.update()
        avg.update_parameters(ref)
        over = tr.step_overflowed()
        assert over == (s == overflow_at), s
        if over:
            tr.loss_scale *= 0.5
            assert not _differ(before, _snapshot(tr), _pmv(before) + ["dev_state"]), s
        else:
            applied += 1
            assert tr.grad_norm.item() == pytest.approx(norm.item(), rel=1e-4), s
        assert tr.loss_scale == scaler.get_scale(), s
        assert tr.steps == s and tr.optimizer_steps == applied, (s, tr.optimizer_steps)
        if applied:
            assert int(opt.state[used[0]]["step"]) == applied
        for (n, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
            torch.testing.assert_close(p, q, rtol=1e-4, atol=1e-6, msg=f"step {s}: {n}")
        ema = tr.ema_state_dict()
        for n, v in avg.module.state_dict().items():
            torch.testing.assert_close(ema[n], v, rtol=1e-4, atol=1e-6, msg=f"EMA step {s}: {n}")


def test_captured_step_skips_an_overflowed_replay_like_the_eager_step():
    """capture() of the whole step with the overflow flag in a static tensor: a replay with the flag set is skipped exactly like
    the eager step, and every replay equals an eager trainer fed the same sequence bit for bit (same model, same kernels).  The
    loss scale is a constant of the graph: neither trainer changes it."""
    x, y = _data()
    ma, ta = _tiny_trainer(loss_scale=2.0 ** 10)
    mb, tb = _tiny_trainer(loss_scale=2.0 ** 10)
    fa, fb = torch.ones((), device=DEV), torch.ones((), device=DEV)
    loss_a = lambda: ((ma(x) - y) ** 2).mean() * fa
    replay = tb.capture(lambda: ((mb(x) - y) ** 2).mean() * fb, warmup=2)
    for _ in range(2):
        ta.step(loss_a)
    assert not _differ(_snapshot(ta), _snapshot(tb))
    for s, f in enumerate([1.0, INF, 1.0, 1.0]):
        before = _snapshot(tb)
        fa.fill_(f)
        fb.copy_(torch.tensor(f))
        la = ta.step(loss_a)
        lb = replay()
        torch.cuda.synchronize()
        assert torch.equal(la, lb), (s, la, lb)
        assert ta.step_overflowed() == tb.step_overflowed() == (f == INF), s
        after = _snapshot(tb)
        assert not _differ(_snapshot(ta), after), (s, _differ(_snapshot(ta), after))
        if f == INF:
            assert not _differ(before, after, _pmv(before) + ["dev_state"]), s
    assert tb.steps == 6 and tb.optimizer_steps == 5


def test_resume_after_a_skipped_step_is_bit_exact(tmp_path):
    """A checkpoint taken right after a skipped step carries AdamW's own step count (1) next to global_step (2); a fresh trainer
    loaded from it continues bit for bit with the uninterrupted run."""
    x, y = _data()
    ma, ta = _tiny_trainer()
    flag = torch.ones((), device=DEV)
    for f in (1.0, INF):
        flag.fill_(f)
        ta.step(lambda: ((ma(x) - y) ** 2).mean() * flag)
    flag.fill_(1.0)
    assert ta.step_overflowed() and ta.steps == 2 and ta.optimizer_steps == 1
    path = tmp_path / "skipped.ckpt"
    torch.save(ta.checkpoint(epoch=0), path)
    ck = torch.load(path, weights_only=False)
    assert ck["global_step"] == 2 and ck["optimizer_step"] == 1
    mb, tb = _tiny_trainer()
    tb.load_checkpoint(ck)
    assert tb.steps == 2 and tb.optimizer_steps == 1
    assert not _differ(_snapshot(ta), _snapshot(tb))
    for s in range(3):
        la = ta.step(lambda: ((ma(x) - y) ** 2).mean())
        lb = tb.step(lambda: ((mb(x) - y) ** 2).mean())
        assert torch.equal(la, lb), s
        assert not _differ(_snapshot(ta), _snapshot(tb)), (s, _differ(_snapshot(ta), _snapshot(tb)))
    assert tb.optimizer_steps == 4
