"""Host logic of the training step on CPU: LR schedule, parameter groups, the differentiable conditioning front end vs the
oracle, and the bucketed data-parallel trainer on two gloo ranks (reference: diffusion_module_ip.py:392-462,500-536;
training_pipeline_ip.py:103-123 DDP ``find_unused_parameters=False``)."""

import math
import os
import subprocess
import sys
import textwrap

import pytest
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import conditioning, weights  # noqa: E402
from progressive_stable_diffusion_b200 import training as T  # noqa: E402


def test_warmup_cosine_closed_form():
    # src/models/lr_scheduler.py:41-64: linear from warmup_start_lr over warmup_epochs, then half-cosine to eta_min
    base, start, eta, wu, mx = 1e-4, 1e-6, 1e-6, 5, 100
    assert T.warmup_cosine_lr(0, base, wu, mx, start, eta) == pytest.approx(start)
    assert T.warmup_cosine_lr(3, base, wu, mx, start, eta) == pytest.approx(start + (base - start) * 0.6)
    assert T.warmup_cosine_lr(5, base, wu, mx, start, eta) == pytest.approx(base)
    assert T.warmup_cosine_lr(52, base, wu, mx, start, eta) == pytest.approx(eta + (base - eta) * 0.5 * (1 + math.cos(math.pi * 47 / 95)))
    assert T.warmup_cosine_lr(100, base, wu, mx, start, eta) == pytest.approx(eta)
    assert T.warmup_cosine_lr(140, base, wu, mx, start, eta) == pytest.approx(eta)          # progress clamps at 1


class _Tiny(nn.Module):
    """Stand-in with the attribute names ``parameter_groups`` reads."""

    def __init__(self):
        super().__init__()
        torch.manual_seed(3)
        self.unet = nn.Sequential(nn.Linear(6, 5), nn.Tanh(), nn.Linear(5, 4))
        self.ordinal_embedder = nn.Module()
        self.ordinal_embedder.base = nn.Parameter(torch.randn(4))
        self.ordinal_embedder.norm = nn.LayerNorm(4)                      # never used in forward (SURVEY.md 7.3)
        self.ordinal_embedder.null_embedding = nn.Parameter(torch.zeros(1, 4))
        self.image_projection = nn.Linear(4, 4)
        self.feature_purifier = nn.Linear(4, 4)

    def forward(self, x):
        h = self.unet(x) + self.ordinal_embedder.base
        return self.feature_purifier(self.image_projection(h))


def test_parameter_groups_follow_the_reference():
    m = _Tiny()
    g = T.parameter_groups(m, 1e-4)
    assert [x["name"] for x in g] == ["unet", "ordinal_embedder", "image_projection", "feature_purifier"]
    assert [x["lr"] for x in g] == [1e-4, 1e-4, 2e-4, 2e-4]                # diffusion_module_ip.py:504-514
    tr = T.DataParallelTrainer(m, lr=1e-4, optimizer="torch", bucket_bytes=64)
    bucketed = {id(p) for bk in tr.buckets for p in bk.params}
    names = dict(m.named_parameters())
    for n in T.UNUSED_PARAMETERS:
        assert id(names[n]) not in bucketed, n
    assert len(bucketed) == len(names) - 3 and len(tr.buckets) > 2
    # parameters are views of their bucket: the module sees the optimizer's in-place update
    bk = tr.buckets[0]
    assert bk.params[0].data_ptr() == bk.flat_p.data_ptr() + bk.offsets[0] * 4


def test_trainer_matches_torch_adamw_and_detects_missing_gradients():
    torch.manual_seed(0)
    m, ref = _Tiny(), _Tiny()
    ref.load_state_dict(m.state_dict())
    tr = T.DataParallelTrainer(m, lr=1e-2, weight_decay=0.05, max_grad_norm=0.5, optimizer="torch", bucket_bytes=64)
    used = [p for n, p in ref.named_parameters() if n not in T.UNUSED_PARAMETERS]
    groups = [{"params": [p for p in g["params"] if any(p is q for q in used)], "lr": g["lr"]} for g in T.parameter_groups(ref, 1e-2)]
    opt = torch.optim.AdamW(groups, betas=(0.9, 0.999), weight_decay=0.05)
    x, y = torch.randn(16, 6), torch.randn(16, 4)
    for _ in range(4):
        loss = tr.step(lambda: ((m(x) - y) ** 2).mean())
        opt.zero_grad()
        lref = ((ref(x) - y) ** 2).mean()
        lref.backward()
        norm = torch.nn.utils.clip_grad_norm_(used, 0.5)
        opt.step()
        assert loss.item() == pytest.approx(lref.item(), rel=1e-5)
        assert tr.grad_norm.item() == pytest.approx(norm.item(), rel=1e-5)
    for (n, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
        torch.testing.assert_close(p, q, rtol=2e-5, atol=2e-6, msg=n)
    with pytest.raises(RuntimeError, match="received no gradient"):
        tr.step(lambda: (m.unet(x) ** 2).mean())                          # purifier / projection / AOE left out of the loss


def test_ema_weight_averaging_follows_the_reference_callback():
    """DataParallelTrainer's EMA against torch.optim.swa_utils.AveragedModel + get_ema_avg_fn - the machinery Lightning's
    WeightAveraging drives in the reference (src/callbacks/ema_callback.py:135-197,414-472) - on the callback's schedule:
    update after optimizer step s when (s - 1) >= update_starting_at_step and (s - 1) % update_every_n_steps == 0."""
    from torch.optim.swa_utils import AveragedModel, get_ema_avg_fn
    torch.manual_seed(1)
    m = _Tiny()
    decay, every, start = 0.9, 2, 1
    tr = T.DataParallelTrainer(m, lr=1e-2, weight_decay=0.05, max_grad_norm=0.5, optimizer="torch", bucket_bytes=64,
                               ema_decay=decay, ema_update_every_n_steps=every, ema_update_starting_at_step=start)
    avg = AveragedModel(m, avg_fn=get_ema_avg_fn(decay), use_buffers=True)
    x, y = torch.randn(16, 6), torch.randn(16, 4)
    updates = 0
    for s in range(1, 9):
        tr.step(lambda: ((m(x) - y) ** 2).mean())
        step_idx = s - 1
        if step_idx >= start and step_idx % every == 0:                   # EMAWeightAveraging.should_update
            avg.update_parameters(m)
            updates += 1
        assert tr.ema_updates == updates
        ema = tr.ema_state_dict()
        for n, v in avg.module.state_dict().items():
            torch.testing.assert_close(ema[n], v, rtol=1e-6, atol=1e-7, msg=f"step {s}: {n}")
    assert updates == 3
    before = {n: p.detach().clone() for n, p in m.named_parameters()}
    tr.swap_ema_weights()                                                 # validation runs on the averaged weights ...
    for n, p in m.named_parameters():
        torch.testing.assert_close(p, avg.module.state_dict()[n], rtol=1e-6, atol=1e-7, msg=n)
    tr.swap_ema_weights()                                                 # ... and training continues on the current ones
    for n, p in m.named_parameters():
        assert torch.equal(p, before[n]), n
    tr.copy_ema_to_model()                                                # end of fit
    for n, p in m.named_parameters():
        torch.testing.assert_close(p, avg.module.state_dict()[n], rtol=1e-6, atol=1e-7, msg=n)


def test_checkpoint_layout_and_resume(tmp_path):
    """The trainer writes the reference's checkpoint layout (ema_callback.py:291-330: averaged weights under ``state_dict``, the
    training weights under ``current_model_state``) and a resumed trainer continues bit for bit."""
    torch.manual_seed(2)
    x, y = torch.randn(16, 6), torch.randn(16, 4)
    kw = dict(lr=1e-2, weight_decay=0.05, max_grad_norm=0.5, optimizer="torch", bucket_bytes=64, ema_decay=0.9,
              ema_update_every_n_steps=1, ema_update_starting_at_step=0)
    m = _Tiny()
    tr = T.DataParallelTrainer(m, **kw)
    for _ in range(3):
        tr.step(lambda: ((m(x) - y) ** 2).mean())
    path = tmp_path / "last.ckpt"
    torch.save(tr.checkpoint(epoch=1), path)
    ck = torch.load(path, weights_only=False)
    assert set(ck) >= {"state_dict", "current_model_state", "averaging_state", "global_step", "epoch"}
    assert ck["global_step"] == 3 and int(ck["averaging_state"]["n_averaged"]) == 3
    assert set(ck["state_dict"]) == set(m.state_dict())
    ema = tr.ema_state_dict()
    assert all(torch.equal(ck["state_dict"][k], ema[k]) for k in ema)
    assert any(not torch.equal(ck["state_dict"][k], ck["current_model_state"][k]) for k in ema)
    # an inference-side loader reads state_dict (= averaged weights): the module API takes it as is
    m_inf = _Tiny()
    m_inf.load_state_dict(ck["state_dict"], strict=True)
    # resume: same next step as the uninterrupted run
    m2 = _Tiny()
    tr2 = T.DataParallelTrainer(m2, **kw)
    tr2.load_checkpoint(ck)
    l1 = tr.step(lambda: ((m(x) - y) ** 2).mean())
    l2 = tr2.step(lambda: ((m2(x) - y) ** 2).mean())
    assert torch.equal(l1, l2)
    for (n, p), (_, q) in zip(m.named_parameters(), m2.named_parameters()):
        assert torch.equal(p, q), n
    e1, e2 = tr.ema_state_dict(), tr2.ema_state_dict()
    assert all(torch.equal(e1[k], e2[k]) for k in e1)


def _optimizer_state(tr):
    """(p, m, v) of every bucket, cloned; moments not yet allocated read as zeros."""
    zero = lambda bk: torch.zeros_like(bk.flat_p)
    return [(bk.flat_p.clone(), zero(bk) if bk.m is None else bk.m.clone(), zero(bk) if bk.v is None else bk.v.clone())
            for bk in tr.buckets]


@pytest.mark.parametrize("overflow_at", [1, 3])
def test_torch_optimizer_skips_overflowed_steps_like_grad_scaler(overflow_at):
    """optimizer="torch" against Lightning's "16-mixed" step with gradient clipping (GradScaler: scale, backward, unscale_,
    clip_grad_norm_, step, update) when the loss of one step is inf: that step leaves parameters and moments untouched, AdamW's
    step count does not advance (GradScaler skips optimizer.step()), the caller halves the loss scale as the scaler does."""
    torch.manual_seed(4)
    m, ref = _Tiny(), _Tiny()
    ref.load_state_dict(m.state_dict())
    scale = 2.0 ** 13
    tr = T.DataParallelTrainer(m, lr=1e-2, weight_decay=0.05, max_grad_norm=0.5, optimizer="torch", bucket_bytes=64, loss_scale=scale)
    used = [p for n, p in ref.named_parameters() if n not in T.UNUSED_PARAMETERS]
    groups = [{"params": [p for p in g["params"] if any(p is q for q in used)], "lr": g["lr"]} for g in T.parameter_groups(ref, 1e-2)]
    opt = torch.optim.AdamW(groups, weight_decay=0.05)
    scaler = torch.amp.GradScaler("cpu", init_scale=scale, growth_interval=10 ** 9)
    x, y = torch.randn(16, 6), torch.randn(16, 4)
    for s in range(1, 6):
        flag = math.inf if s == overflow_at else 1.0
        before = _optimizer_state(tr)
        tr.step(lambda: ((m(x) - y) ** 2).mean() * flag)
        opt.zero_grad()
        scaler.scale(((ref(x) - y) ** 2).mean() * flag).backward()
        scaler.unscale_(opt)
        torch.nn.utils.clip_grad_norm_(used, 0.5)
        scaler.step(opt)
        scaler.update()
        assert tr.step_overflowed() == (s == overflow_at), s
        if tr.step_overflowed():
            tr.loss_scale *= 0.5
            for (p0, m0, v0), (p1, m1, v1) in zip(before, _optimizer_state(tr)):
                assert torch.equal(p0, p1) and torch.equal(m0, m1) and torch.equal(v0, v1), s
        assert tr.loss_scale == scaler.get_scale()
        assert tr.steps == s and tr.optimizer_steps == s - (s >= overflow_at)
        if s > overflow_at or overflow_at > 1:
            assert int(opt.state[used[0]]["step"]) == tr.optimizer_steps
        for (n, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
            torch.testing.assert_close(p, q, rtol=2e-5, atol=2e-6, msg=f"step {s}: {n}")


def test_skipped_step_is_not_counted_by_adamw_and_survives_resume(tmp_path):
    """global_step counts every step, AdamW's t the applied ones; the checkpoint keeps both, and a trainer resumed after a skipped
    step continues bit for bit.  A checkpoint without ``optimizer_step`` resumes t from global_step."""
    torch.manual_seed(5)
    x, y = torch.randn(16, 6), torch.randn(16, 4)
    kw = dict(lr=1e-2, weight_decay=0.05, max_grad_norm=0.5, optimizer="torch", bucket_bytes=64, ema_decay=0.9,
              ema_update_every_n_steps=1, ema_update_starting_at_step=0)
    m = _Tiny()
    tr = T.DataParallelTrainer(m, **kw)
    for flag in (1.0, math.inf):
        tr.step(lambda: ((m(x) - y) ** 2).mean() * flag)
    assert tr.step_overflowed() and tr.steps == 2 and tr.optimizer_steps == 1
    assert all(torch.isfinite(p).all() for p in m.parameters())
    path = tmp_path / "skipped.ckpt"
    torch.save(tr.checkpoint(epoch=0), path)
    ck = torch.load(path, weights_only=False)
    assert ck["global_step"] == 2 and ck["optimizer_step"] == 1
    m2 = _Tiny()
    tr2 = T.DataParallelTrainer(m2, **kw)
    tr2.load_checkpoint(ck)
    assert tr2.steps == 2 and tr2.optimizer_steps == 1
    for _ in range(3):
        l1 = tr.step(lambda: ((m(x) - y) ** 2).mean())
        l2 = tr2.step(lambda: ((m2(x) - y) ** 2).mean())
        assert torch.equal(l1, l2)
    assert tr2.optimizer_steps == tr.optimizer_steps == 4
    for (n, p), (_, q) in zip(m.named_parameters(), m2.named_parameters()):
        assert torch.equal(p, q), n
    e1, e2 = tr.ema_state_dict(), tr2.ema_state_dict()
    assert all(torch.equal(e1[k], e2[k]) for k in e1)
    legacy = {k: v for k, v in ck.items() if k != "optimizer_step"}
    tr3 = T.DataParallelTrainer(_Tiny(), **kw)
    tr3.load_checkpoint(legacy)
    assert tr3.optimizer_steps == 2


def test_conditioning_train_functions_match_oracle():
    """aoe_train / purifier_train are the autograd twins of the inference kernels: same numbers as the (reference-pinned) oracle."""
    from progressive_stable_diffusion_b200.feature_purifier import FeaturePurifier
    from progressive_stable_diffusion_b200.ordinal_embedder import AdditiveOrdinalEmbedder
    aw, pw = weights.make_aoe_state(), weights.make_purifier_state()
    aoe = AdditiveOrdinalEmbedder(4, 768, num_tokens=16)
    aoe.load_state_dict(aw)
    pur = FeaturePurifier(768, 8, 2)
    pur.load_state_dict(pw)
    labels = torch.tensor([0.0, 0.4, 1.0, 2.5, 3.0, 3.7, -1.0])
    got = T.aoe_train(aoe, labels, noise_std=0.0)
    torch.testing.assert_close(got, conditioning.aoe_forward(aw, labels), rtol=1e-5, atol=1e-5)
    g = torch.Generator().manual_seed(5)
    img = torch.randn(7, 16, 768, generator=g)
    torch.testing.assert_close(T.purifier_train(pur, img, got), conditioning.purifier_forward(pw, img, got), rtol=1e-4, atol=1e-4)
    # training-mode noise: N(0, 0.005^2) on the interpolated embedding before the projector (ordinal_embedder.py:172-175)
    noisy = T.aoe_train(aoe, labels, noise_std=0.005, generator=torch.Generator().manual_seed(1))
    assert 0 < (noisy - got).abs().max() < 1.0
    # gradients reach every AOE / purifier parameter that takes part in a forward
    loss = T.purifier_train(pur, img, T.aoe_train(aoe, labels, 0.0)).square().mean()
    loss.backward()
    missing = [n for n, p in list(aoe.named_parameters()) + list(pur.named_parameters()) if p.grad is None]
    assert sorted(missing) == ["norm.bias", "norm.weight", "null_embedding"], missing


WORKER = textwrap.dedent("""
    import sys, torch, torch.nn as nn
    sys.path.insert(0, %r)
    sys.path.insert(0, %r)
    from progressive_stable_diffusion_b200 import parallel, training as T
    from test_training_cpu import _Tiny
    rank, local, world = parallel.init_from_env(backend="gloo")
    m = _Tiny()
    tr = T.DataParallelTrainer(m, lr=1e-2, weight_decay=0.05, max_grad_norm=0.5, optimizer="torch", bucket_bytes=64)
    g = torch.Generator().manual_seed(7)
    X, Y = torch.randn(2, 8, 6, generator=g), torch.randn(2, 8, 4, generator=g)        # rank r trains on shard r
    for _ in range(3):
        tr.step(lambda: ((m(X[rank]) - Y[rank]) ** 2).mean())
    flat = torch.cat([p.detach().reshape(-1) for p in m.parameters()])
    both = [torch.empty_like(flat) for _ in range(world)]
    torch.distributed.all_gather(both, flat)
    assert torch.equal(both[0], both[1]), "ranks diverged"
    if rank == 0:
        # single process, same global batch: mean of the two shard losses = the gradient DDP averages
        ref = _Tiny()
        used = [p for n, p in ref.named_parameters() if n not in T.UNUSED_PARAMETERS]
        groups = [{"params": [p for p in gr["params"] if any(p is q for q in used)], "lr": gr["lr"]} for gr in T.parameter_groups(ref, 1e-2)]
        opt = torch.optim.AdamW(groups, weight_decay=0.05)
        for _ in range(3):
            opt.zero_grad()
            (0.5 * (((ref(X[0]) - Y[0]) ** 2).mean() + ((ref(X[1]) - Y[1]) ** 2).mean())).backward()
            torch.nn.utils.clip_grad_norm_(used, 0.5)
            opt.step()
        want = torch.cat([p.detach().reshape(-1) for p in ref.parameters()])
        torch.testing.assert_close(flat, want, rtol=5e-5, atol=5e-6)
        print("OK", len(tr.buckets))
    parallel.barrier()
""") % (ROOT, os.path.join(ROOT, "tests"))


def test_two_rank_gloo_bucketed_allreduce_equals_single_process(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29641", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r), LOCAL_RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert "OK" in outs[0], outs
