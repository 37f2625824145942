"""The pairwise-statistics kernel (RBF_SUM / KNN / COVER) against float64 references, its determinism, capture and memory, the
CMMD / precision-recall metrics and their backbones, and an evaluation sweep end to end."""

import math
from pathlib import Path

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SHAPES = [1, 5, 127, 128, 129, 1000, 4099]
PAIRS = [(1, 1), (1, 5), (5, 127), (127, 128), (128, 129), (129, 1000), (1000, 4099), (4099, 5)]
DIMS = [8, 768, 4096]
KINDS = ["unit", "relu", "dup"]


def _features(n: int, d: int, kind: str, seed: int) -> torch.Tensor:
    """unit-norm rows, non-negative post-ReLU-like rows, or unit rows of which every third repeats an earlier row exactly."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, d, generator=g)
    if kind == "relu":
        return torch.relu(x) * 3.0
    x = torch.nn.functional.normalize(x, dim=1)
    if kind == "dup":
        idx = torch.arange(2, max(n, 2), 3)
        x[idx] = x[idx - 2]
    return x.contiguous()


def _sq64(x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    from progressive_stable_diffusion_b200 import metrics
    return metrics._sqdist64(x, y)


def _d2_bound(x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """Bound on |d2_kernel - d2_exact| per pair, derived from the kernel's arithmetic (|a| = row norm):
    - the split x = hi + lo, hi = tf32(x) rounded to nearest, |lo| <= 2^-11 |x|: the dropped lo.lo term is <= 2^-22 |x_i||y_i|,
      and the tensor core's tf32 view of lo loses <= 2^-10 |lo| in each of the two lo terms: 1.25 * 2^-20 |x_i||y_i| per element;
    - fp32 accumulation in TMEM over S = 3 ceil(D / 8) MMAs, each rounding by <= 2^-23 of a partial sum <= sum |x_i||y_i|
      (truncating, the worst case): S * 2^-23;
    Cauchy-Schwarz turns sum |x_i||y_i| into |x||y|, so the Gram error is <= (1.25 * 2^-20 + S * 2^-23) |x||y|.  d2 =
    |x|^2 + |y|^2 - 2 g doubles it and adds the fp32 roundings of the norms and of the two-operation epilogue: 4 * 2^-24
    (|x|^2 + |y|^2)."""
    d = x.shape[1]
    s = 3 * math.ceil(d / 8)
    nx, ny = x.double().norm(dim=1), y.double().norm(dim=1)
    gram = (1.25 * 2.0 ** -20 + s * 2.0 ** -23) * nx[:, None] * ny[None, :]
    return 2.0 * gram + 4 * 2.0 ** -24 * (nx[:, None] ** 2 + ny[None, :] ** 2)


@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("m,n", PAIRS)
@pytest.mark.parametrize("kind", KINDS)
def test_rbf_sum_vs_float64(m, n, d, kind):
    from progressive_stable_diffusion_b200 import ops
    x, y = _features(m, d, kind, 1), _features(n, d, kind, 2)
    ref = _sq64(x, y)
    gamma = 1.0 / max(ref.mean().item(), 1e-3)
    want = torch.exp(-gamma * ref)
    # |exp(-g a) - exp(-g b)| <= g |a - b| exp(-g min(a, b)); plus expf's own error (2 ulp) per term
    bound = ((gamma * _d2_bound(x, y)).clamp_max(1.0) * torch.exp(-gamma * (ref - _d2_bound(x, y)).clamp_min(0)) + 2.4e-7 * want).sum()
    got = ops.pairwise_rbf_sum(x.to(DEV), y.to(DEV), gamma).item()
    err = abs(got - want.sum().item())
    print(f"rbf {kind} {m}x{n} D={d}: err {err:.3g} (bound {bound.item():.3g}, sum {want.sum().item():.6g})")
    assert err <= bound.item(), (err, bound.item())


@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("m", [s for s in SHAPES if s > 4])
@pytest.mark.parametrize("kind", KINDS)
def test_knn_radii_vs_float64(m, d, kind):
    from progressive_stable_diffusion_b200 import metrics, ops
    x = _features(m, d, kind, 3)
    k = 3
    want = metrics.knn_radii_reference(x, k)
    tol = _d2_bound(x, x).max(dim=1).values         # the k-th order statistic moves by at most the largest per-pair error
    got = ops.knn_radii(x.to(DEV), k).double().cpu()
    err = (got - want).abs()
    print(f"knn {kind} M={m} D={d}: max err {err.max().item():.3g}, max err / bound {(err / tol).max().item():.3g}")
    assert (err <= tol).all()
    if kind == "dup":                               # a duplicate's nearest other point is its copy: radius (k = 1) ~ 0
        assert (ops.knn_radii(x.to(DEV), 1).double().cpu()[2::3] <= tol[2::3]).all()


def _margin_radii(d2: torch.Tensor, tol: torch.Tensor) -> torch.Tensor:
    """Per column j, a radius in the middle of the widest gap between the sorted d2[:, j] whose every point clears the
    bound; -1 (no ball) where there is no such gap.  Every (i, j) then has |d2 - r_j| > tol[i, j]."""
    r = torch.full((d2.shape[1],), -1.0, dtype=torch.float64)
    for j in range(d2.shape[1]):
        v, order = d2[:, j].sort()
        if v.numel() == 1:
            r[j] = v[0] + 2 * tol[order[0], j] + 1e-3
            continue
        gaps = v[1:] - v[:-1]
        q = int(gaps.argmax())
        mid = 0.5 * (v[q] + v[q + 1])
        if ((d2[:, j] - mid).abs() > tol[:, j]).all():
            r[j] = mid
    return r.float().double()                           # an fp32 radius, exactly what the kernel compares with


@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("m,n", PAIRS)
@pytest.mark.parametrize("kind", KINDS)
def test_cover_vs_float64(m, n, d, kind):
    from progressive_stable_diffusion_b200 import metrics, ops
    q, ref = _features(m, d, kind, 4), _features(n, d, kind, 5)
    d2 = _sq64(q, ref)
    tol = _d2_bound(q, ref)
    # (1) radii of the reference set itself (k-NN, as the metric uses them) or, for tiny sets, the median distance
    radii = metrics.knn_radii_reference(ref, 3).float() if n > 4 else d2.median(dim=0).values.float()
    want = (d2 <= radii.double()[None]).any(1)
    got = ops.within_radii(q.to(DEV), ref.to(DEV), radii.to(DEV)).cpu()
    ambiguous = ((d2 - radii.double()[None]).abs() <= tol).any(1)
    assert torch.equal(got[~ambiguous], want[~ambiguous])
    print(f"cover {kind} {m}x{n} D={d}: {int(ambiguous.sum())} rows within the bound of a tie, {int((got != want).sum())} differ")
    # (2) radii with a guaranteed margin: exact agreement
    r2 = _margin_radii(d2, tol)
    want2 = (d2 <= r2[None]).any(1)
    got2 = ops.within_radii(q.to(DEV), ref.to(DEV), r2.float().to(DEV)).cpu()
    assert torch.equal(got2, want2)


def test_repeated_calls_are_bit_identical():
    from progressive_stable_diffusion_b200 import ops
    x = _features(4099, 768, "unit", 6).to(DEV)
    y = _features(1000, 768, "relu", 7).to(DEV)
    r = ops.knn_radii(y, 3)
    a = [ops.pairwise_rbf_sum(x, y, 0.01).item() for _ in range(3)]
    b = [ops.knn_radii(x, 5) for _ in range(3)]
    c = [ops.within_radii(x, y, r) for _ in range(3)]
    assert a[0] == a[1] == a[2]
    assert all(torch.equal(b[0], t) for t in b) and all(torch.equal(c[0], t) for t in c)


def test_graph_capture_replays_the_eager_call():
    from progressive_stable_diffusion_b200 import ops
    x = _features(1000, 768, "unit", 8).to(DEV)
    y = _features(129, 768, "unit", 9).to(DEV)
    r = ops.knn_radii(y, 3)
    eager = (ops.pairwise_rbf_sum(x, y, 0.005), ops.knn_radii(x, 3), ops.within_radii(x, y, r))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                          # warm-up on the capture stream
        ops.pairwise_rbf_sum(x, y, 0.005)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = (ops.pairwise_rbf_sum(x, y, 0.005), ops.knn_radii(x, 3), ops.within_radii(x, y, r))
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip(out, eager):
        assert torch.equal(a, b)


def test_fifty_thousand_points_without_a_distance_matrix():
    """M = N = 50 000 at D = 768: one fp32 distance matrix alone would be 10 GB.  Budget: the features (154 MB), the kernel's
    workspace (the tf32 hi / lo split, 307 MB, plus per-slice partials) and the outputs: under 1 GB of peak allocation."""
    from progressive_stable_diffusion_b200 import ops
    x = torch.nn.functional.normalize(torch.randn(50_000, 768, device=DEV, generator=torch.Generator(DEV).manual_seed(1)), dim=1)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    s = ops.pairwise_rbf_sum(x, None, 1.0 / 200.0)
    r = ops.knn_radii(x, 3)
    f = ops.within_radii(x[:2400].contiguous(), x, r)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    print(f"50k x 50k: peak {peak / 1e6:.0f} MB above the inputs, mean k = {s.item() / 50_000 ** 2:.6f}")
    assert peak < 1.0e9, peak
    assert math.isfinite(s.item()) and torch.isfinite(r).all() and bool(f.all())      # each point lies in its own ball


def test_metrics_match_float64_formulas():
    import progressive_stable_diffusion_b200 as P
    from progressive_stable_diffusion_b200 import metrics
    g = torch.Generator().manual_seed(10)
    real = torch.nn.functional.normalize(torch.randn(700, 768, generator=g), dim=1)
    fake = torch.nn.functional.normalize(torch.randn(500, 768, generator=g) + 0.3, dim=1)
    want = metrics.cmmd_reference(real, fake)
    got = P.cmmd(real.to(DEV), fake.to(DEV))
    print(f"cmmd {got:.6f} vs float64 {want:.6f}")
    assert abs(got - want) <= 2e-3 * abs(want) + 2e-3
    assert abs(P.cmmd(real.to(DEV), real.to(DEV))) < 1e-5
    vr, vf = torch.relu(torch.randn(600, 4096, generator=g)), torch.relu(torch.randn(400, 4096, generator=g) * 1.1)
    p, r = P.precision_recall(vr.to(DEV), vf.to(DEV), k=3)
    wp, wr = metrics.precision_recall_reference(vr, vf, k=3)
    print(f"precision / recall {p:.4f} {r:.4f} vs float64 {wp:.4f} {wr:.4f}")
    assert abs(p - wp) <= 2 / 400 and abs(r - wr) <= 2 / 600         # at most two points sit within the bound of a tie
    far = vf + 50.0
    assert P.precision_recall(vr.to(DEV), far.to(DEV), k=3) == (0.0, 0.0)
    assert P.precision_recall(vr.to(DEV), vr.clone().to(DEV), k=3) == (1.0, 1.0)


def test_clip_336_tower_matches_the_oracle():
    import progressive_stable_diffusion_b200 as P
    from oracle import image_front_end as fe, weights
    w = weights.make_clip_vision_state(seed=5, image=336)
    pixels = torch.randn(1, 3, 336, 336, generator=torch.Generator().manual_seed(11))
    with torch.no_grad():
        hidden_ref, embeds_ref = fe.clip_hidden_states(w, pixels, 16, 14)
    enc = P.ImageEncoder("openai/clip-vit-large-patch14-336")
    enc.image_encoder.load_state_dict(w, strict=True)
    enc.to(DEV)
    hidden, embeds = enc.get_hidden_states(pixels.to(DEV)), enc(pixels.to(DEV))
    assert hidden.shape == (1, 577, 1024)
    rel = lambda a, b: ((a.double().cpu() - b.double()).abs().max() / b.double().abs().max()).item()
    eh, ee = rel(hidden, hidden_ref), rel(embeds, embeds_ref)
    print(f"CLIP ViT-L/14-336 fp16: hidden rel err {eh:.4g}, embeds rel err {ee:.4g}")
    assert eh <= 5e-3 and ee <= 5e-3                   # the 224 tower's fp16 tolerance
    emb = P.ClipEmbedder()
    emb.load_state_dict(w, strict=True)
    e = emb.to(DEV)(torch.rand(3, 3, 256, 256, generator=torch.Generator().manual_seed(12)))
    assert e.shape == (3, 768) and torch.allclose(e.norm(dim=1), torch.ones(3, device=DEV), atol=1e-5)


def test_vgg_features_match_torchvision():
    """fp16 channels-last VGG16 up to fc2 vs torchvision's fp32 CPU forward on the same weights: 13 convolutions and two GEMMs
    with fp16 activations (11 bits) and fp32 accumulation; bound 1e-2 of the largest feature."""
    import torchvision
    import progressive_stable_diffusion_b200 as P
    from progressive_stable_diffusion_b200 import metrics
    torch.manual_seed(13)
    tv = torchvision.models.vgg16(weights=None).eval()
    v = P.VGGFeatures()
    v.load_state_dict(tv.state_dict(), strict=True)
    images = torch.rand(2, 3, 256, 256, generator=torch.Generator().manual_seed(14))
    x = torch.nn.functional.interpolate(images, size=(224, 224), mode="bilinear", align_corners=False)
    mean, std = torch.tensor(metrics.IMAGENET_MEAN).view(1, 3, 1, 1), torch.tensor(metrics.IMAGENET_STD).view(1, 3, 1, 1)
    with torch.no_grad():
        h = torch.flatten(tv.avgpool(tv.features((x - mean) / std)), 1)
        want = tv.classifier[:metrics.VGG_FC2_END](h)
    got = v.to(DEV)(images)
    e = ((got.double().cpu() - want.double()).abs().max() / want.double().abs().max()).item()
    print(f"VGG16 fc2 fp16: rel err {e:.4g}")
    assert got.shape == (2, 4096) and e <= 1e-2, e


def test_sweep_generate_group_evaluate():
    import progressive_stable_diffusion_b200 as P
    from oracle import weights
    from progressive_stable_diffusion_b200 import evaluation_pipeline as ev
    module = P.DiffusionModuleWithIP(P.default_config())
    module.load_state_dict(weights.make_module_state(seed=0), strict=True)
    module.to(DEV).eval()
    jobs = [ev.GenerationJob(Path(f"src{s}.png"), s, t) for s in range(4) for t in range(4) if t != s]
    jobs_sorted, sources = ev.sweep_order(jobs)
    tokens = torch.randn(len(sources), 16, 768, generator=torch.Generator().manual_seed(15))
    images = ev.generate_all(module, ev.as_index_jobs(jobs_sorted, sources), tokens, DEV, batch_size=6, sampling_steps=2)
    size = module.cfg.dataset.image_size
    fake = ev.group_by_target(images, jobs_sorted, size)
    assert all(fake[c].shape[0] == 3 for c in ev.ALL_MES_CLASSES)
    g = torch.Generator().manual_seed(16)
    real = {c: torch.rand(5, 3, size, size, generator=g) for c in ev.ALL_MES_CLASSES}
    clip = P.ClipEmbedder()
    clip.load_state_dict(weights.make_clip_vision_state(seed=5, image=336), strict=True)
    res = ev.evaluate_images(real, fake, clip.to(DEV), P.VGGFeatures().to(DEV), k=1)
    assert sorted(res, key=str) == sorted([*ev.ALL_MES_CLASSES, "all"], key=str)
    for key, r in res.items():
        print(key, r)
        assert set(r) == {"cmmd", "precision", "recall"} and all(math.isfinite(v) for v in r.values()), (key, r)
