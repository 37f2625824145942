"""The pairwise kernel's COUNT and RATIO_MAX modes and the cross-set k-NN radii against float64 references, their determinism,
capture and memory, and the density / coverage and realism metrics up to the evaluation pipeline."""

import math

import pytest
import torch

from tests.test_gpu_metrics import _d2_bound, _margin_radii
from tests.test_gpu_metrics import _features as _unit_relu_dup

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
EPS = 1e-5
# (M, N, D): single points, the 128-row and 256-column tile edges, several slices, and the metric's own size
SHAPES = [(1, 1, 8), (1, 5, 8), (5, 1, 768), (127, 255, 8), (128, 256, 768), (129, 257, 768), (129, 257, 4096),
          (1000, 4099, 768), (2400, 11264, 4096)]
KINDS = ["gauss", "relu", "unit", "dup"]


def _features(n: int, d: int, kind: str, seed: int) -> torch.Tensor:
    """Gaussian rows, or test_gpu_metrics' unit-norm / ReLU-Gaussian / duplicated-unit rows."""
    if kind == "gauss":
        return torch.randn(n, d, generator=torch.Generator().manual_seed(seed))
    return _unit_relu_dup(n, d, kind, seed)


def _pair(m: int, n: int, d: int, kind: str):
    """Query and reference sets on the device; with "dup", every fourth query row is a copy of a reference row (d2 = 0)."""
    q, ref = _features(m, d, kind, 20), _features(n, d, kind, 21)
    if kind == "dup":
        idx = torch.arange(0, m, 4)
        q[idx] = ref[idx % n]
    return q.to(DEV), ref.to(DEV)


def _radii(q: torch.Tensor, ref: torch.Tensor, d2: torch.Tensor) -> torch.Tensor:
    """fp32 radii as the metrics use them: the reference set's own k-NN radii, or the per-column median for tiny sets."""
    from progressive_stable_diffusion_b200 import metrics
    n = ref.shape[0]
    return (metrics.knn_radii_reference(ref, 3) if n > 4 else d2.median(dim=0).values).float()


@pytest.mark.parametrize("m,n,d", SHAPES)
@pytest.mark.parametrize("kind", KINDS)
def test_count_vs_float64(m, n, d, kind):
    from progressive_stable_diffusion_b200 import metrics, ops
    q, ref = _pair(m, n, d, kind)
    d2, tol = metrics._sqdist64(q, ref), _d2_bound(q, ref)
    radii = _radii(q, ref, d2)
    want = (d2 <= radii.double()[None]).sum(1)
    got = ops.count_within_radii(q, ref, radii).long()
    near = ((d2 - radii.double()[None]).abs() <= tol).sum(1)           # pairs within the bound of a tie
    err = (got - want).abs()
    print(f"count {kind} {m}x{n} D={d}: {int(near.sum())} pairs near a tie, {int((err > 0).sum())} rows differ, "
          f"max err {int(err.max())}")
    assert (err <= near).all()
    # radii with a guaranteed margin around every d2 of their column: exact
    r2 = _margin_radii(d2.cpu(), tol.cpu()).float().to(DEV)
    assert torch.equal(ops.count_within_radii(q, ref, r2).long(), (d2 <= r2.double()[None]).sum(1))


@pytest.mark.parametrize("m,n,d", SHAPES)
@pytest.mark.parametrize("kind", KINDS)
def test_ratio_max_vs_float64(m, n, d, kind):
    from progressive_stable_diffusion_b200 import metrics, ops
    q, ref = _pair(m, n, d, kind)
    d2, tol = metrics._sqdist64(q, ref), _d2_bound(q, ref)
    r = _radii(q, ref, d2).double()
    want = (r[None] / (d2 + EPS)).amax(1)
    # |r / (a + eps) - r / (d2 + eps)| <= r tol / ((max(d2 - tol, 0) + eps)(d2 + eps)) for the kernel's |a - d2| <= tol; the max
    # moves by at most the largest such change; plus the fp32 roundings of a + eps and of the division
    bound = (r[None] * tol / (((d2 - tol).clamp_min(0) + EPS) * (d2 + EPS))).amax(1) + 2.4e-7 * want
    got = ops.max_radius_ratio(q, ref, r.float(), EPS).double()
    err = (got - want).abs()
    print(f"ratio_max {kind} {m}x{n} D={d}: max err / bound {(err / bound).max().item():.3g}")
    assert (err <= bound).all()


@pytest.mark.parametrize("m,n,d", [(1, 4, 8), (129, 257, 768), (1000, 4099, 768), (2400, 11264, 4096)])
@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_cross_set_knn_radii_vs_float64(m, n, d, k, kind):
    from progressive_stable_diffusion_b200 import metrics, ops
    q, ref = _pair(m, n, d, kind)
    want = metrics._sqdist64(q, ref).kthvalue(k, dim=1).values            # nothing excluded across sets
    tol = _d2_bound(q, ref).max(dim=1).values
    got = ops.knn_radii(q, k, ref=ref).double()
    err = (got - want).abs()
    print(f"knn(ref) {kind} {m}x{n} D={d} k={k}: max err / bound {(err / tol).max().item():.3g}")
    assert (err <= tol).all()


def _real_fake(d: int, kind: str):
    """Generated rows correlated with the first real rows, so that density, coverage and realism are all informative."""
    g = torch.Generator().manual_seed(30)
    if kind == "relu":
        z = torch.randn(600, d, generator=g)
        return torch.relu(z).to(DEV), torch.relu(0.6 * z[:400] + 0.8 * torch.randn(400, d, generator=g)).to(DEV)
    real = torch.nn.functional.normalize(torch.randn(700, d, generator=g), dim=1)
    return real.to(DEV), torch.nn.functional.normalize(torch.randn(500, d, generator=g) + 0.3 * real[:500], dim=1).to(DEV)


@pytest.mark.parametrize("d,kind", [(4096, "relu"), (768, "unit")])
def test_density_coverage_match_float64(d, kind):
    import progressive_stable_diffusion_b200 as P
    from progressive_stable_diffusion_b200 import metrics
    real, fake = _real_fake(d, kind)
    k = 3
    dens, cov = P.density_coverage(real, fake, k)
    want_d, want_c = metrics.density_coverage_reference(real, fake, k)
    # the kernel's radii move by <= rtol, each d2 by <= tol, and r2 is compared one fp32 ulp below: a (fake, real) pair or a real
    # can only be judged differently when its d2 lies within that much of r2
    r = metrics.knn_radii_reference(real, k)
    rtol = _d2_bound(real, real).max(dim=1).values + r * 2.0 ** -22
    d2, tol = metrics._sqdist64(fake, real), _d2_bound(fake, real)
    near_pairs = int(((d2 - r[None]).abs() <= tol + rtol[None]).sum())
    near_reals = int(((d2.min(dim=0).values - r).abs() <= tol.max(dim=0).values + rtol).sum())
    print(f"density {dens:.6f} vs {want_d:.6f} ({near_pairs} pairs near a tie), coverage {cov:.6f} vs {want_c:.6f} "
          f"({near_reals} reals near a tie)")
    assert abs(dens - want_d) <= near_pairs / (k * fake.shape[0]) + 1e-12
    assert abs(cov - want_c) <= near_reals / real.shape[0] + 1e-12
    assert P.density_coverage(real, fake + 50.0, k) == (0.0, 0.0)


@pytest.mark.parametrize("d,kind", [(4096, "relu"), (768, "unit")])
def test_realism_scores_match_float64(d, kind):
    import progressive_stable_diffusion_b200 as P
    from progressive_stable_diffusion_b200 import metrics, ops
    real, fake = _real_fake(d, kind)
    k = 3
    r = metrics.knn_radii_reference(real, k)
    rtol = _d2_bound(real, real).max(dim=1).values
    # the pruning may only differ from float64 for a real whose radius lies within the bound of the percentile; the float64
    # formula below then uses the kernel's pruning
    keep, keep64 = metrics._realism_kept(ops.knn_radii(real, k)), metrics._realism_kept(r)
    cut = torch.quantile(r, metrics.REALISM_PRUNE_PERCENTILE / 100.0)
    assert ((r - cut).abs()[keep != keep64] <= 2 * rtol.max()).all()
    rk, tolk = r[keep], rtol[keep]
    d2, tol = metrics._sqdist64(fake, real[keep]), _d2_bound(fake, real[keep])
    got = P.realism_scores(real, fake, k).double()
    want = (rk[None] / (d2 + EPS)).amax(1).sqrt()
    if torch.equal(keep, keep64):
        assert torch.allclose(want, metrics.realism_scores_reference(real, fake, k), rtol=1e-12, atol=0)
    # squared score: |r' / (a + eps) - r / (d2 + eps)| <= rtol / (lo + eps) + r tol / ((lo + eps)(d2 + eps)), lo = max(d2 - tol, 0);
    # then |sqrt(u) - sqrt(v)| <= |u - v| / sqrt(v), plus the fp32 roundings (division, a + eps, sqrt)
    lo = (d2 - tol).clamp_min(0) + EPS
    sq = (tolk[None] / lo + rk[None] * tol / (lo * (d2 + EPS))).amax(1) + 2.4e-7 * want ** 2
    bound = sq / want + 1.2e-7 * want
    err = (got - want).abs()
    print(f"realism {kind} D={d}: {int((keep != keep64).sum())} reals pruned differently, max err / bound "
          f"{(err / bound).max().item():.3g}, scores {want.min().item():.3f}..{want.max().item():.3f}")
    assert got.shape == (fake.shape[0],) and got.dtype == torch.float64 and (err <= bound).all()
    assert P.realism_scores(real, fake, k).dtype == torch.float32


def test_repeated_calls_are_bit_identical():
    from progressive_stable_diffusion_b200 import ops
    x, y = _pair(4099, 1000, 768, "unit")
    r = ops.knn_radii(y, 3)
    a = [ops.count_within_radii(x, y, r) for _ in range(3)]
    b = [ops.max_radius_ratio(x, y, r, EPS) for _ in range(3)]
    c = [ops.knn_radii(x, 3, ref=y) for _ in range(3)]
    for outs in (a, b, c):
        assert all(torch.equal(outs[0], t) for t in outs)


def test_graph_capture_replays_the_eager_call():
    from progressive_stable_diffusion_b200 import ops
    x, y = _pair(1000, 129, 768, "relu")
    r = ops.knn_radii(y, 3)
    eager = (ops.count_within_radii(x, y, r), ops.max_radius_ratio(x, y, r, EPS), ops.knn_radii(x, 1, ref=y))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                          # warm-up on the capture stream
        ops.count_within_radii(x, y, r)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = (ops.count_within_radii(x, y, r), ops.max_radius_ratio(x, y, r, EPS), ops.knn_radii(x, 1, ref=y))
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip(out, eager):
        assert torch.equal(a, b)


def test_fifty_thousand_point_count_without_a_distance_matrix():
    """COUNT at M = N = 50 000, D = 768: a distance matrix alone would be 10 GB.  Budget: the kernel's workspace (the tf32
    hi / lo split of both sets, 614 MB, plus per-slice counts) and the output: under 1 GB of peak allocation."""
    from progressive_stable_diffusion_b200 import ops
    x = torch.nn.functional.normalize(torch.randn(50_000, 768, device=DEV, generator=torch.Generator(DEV).manual_seed(1)), dim=1)
    r = ops.knn_radii(x, 3)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    c = ops.count_within_radii(x, x, r)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    print(f"50k x 50k COUNT: peak {peak / 1e6:.0f} MB above the inputs, mean count {c.double().mean().item():.3f}")
    assert peak < 1.0e9, peak
    assert (c >= 1).all()                               # each point lies in its own ball


def _tiny_images(size: int = 64):
    g = torch.Generator().manual_seed(40)
    real = {c: torch.rand(5, 3, size, size, generator=g) for c in range(4)}
    fake = {c: torch.rand(3, 3, size, size, generator=g) for c in range(4)}
    return real, fake


def test_evaluate_images_with_density_coverage():
    import progressive_stable_diffusion_b200 as P
    from oracle import weights
    from progressive_stable_diffusion_b200 import evaluation_pipeline as ev
    real, fake = _tiny_images()
    clip = P.ClipEmbedder()
    clip.load_state_dict(weights.make_clip_vision_state(seed=5, image=336), strict=True)
    clip, vgg = clip.to(DEV), P.VGGFeatures().to(DEV)
    base = ev.evaluate_images(real, fake, clip, vgg, k=1)
    res = ev.evaluate_images(real, fake, clip, vgg, k=1, density_coverage=True)
    assert list(res) == list(base)
    for key, r in res.items():
        print(key, r)
        assert set(r) == {"cmmd", "precision", "recall", "density", "coverage"}
        assert all(r[m] == base[key][m] for m in ("cmmd", "precision", "recall")), (key, r, base[key])
        assert math.isfinite(r["density"]) and math.isfinite(r["coverage"]), (key, r)


def test_realism_by_class_scores_each_generated_image_in_order():
    import progressive_stable_diffusion_b200 as P
    from progressive_stable_diffusion_b200 import evaluation_pipeline as ev, metrics
    real, _ = _tiny_images()
    k = 2                                               # (k = 1 radii come in exactly tied mutual-neighbour pairs)
    real[3] = real[3][:k + 1]                           # k + 1 reals: left out
    vgg = P.VGGFeatures().to(DEV)
    fake = {}
    for c in (0, 2, 3):
        # a copy of the real with the smallest radius (always kept) among flat images far from every real
        r = metrics.knn_radii_reference(vgg(real[c]).double(), k) if real[c].shape[0] > k + 1 else torch.zeros(1)
        flat = [torch.full((3, 64, 64), v) for v in (0.0, 1.0, 0.5)]
        fake[c] = torch.stack([flat[0], real[c][int(r.argmin())], flat[1], flat[2]])
    fake[1] = torch.zeros(0, 3, 64, 64)                 # empty: left out
    got = ev.realism_by_class(real, fake, vgg, k=k)
    flipped = ev.realism_by_class(real, {c: f.flip(0) for c, f in fake.items()}, vgg, k=k)
    assert sorted(got) == [0, 2] and sorted(flipped) == [0, 2]
    for c, s in got.items():
        print(c, s.tolist())
        assert s.shape == (4,) and s.dtype == torch.float32 and s.device.type == "cpu"
        assert int(s.argmax()) == 1 and int(flipped[c].argmax()) == 2     # the copy scores highest, where it sits
        # each class against its own reals, image n at index n (the kernel's precision is tested above)
        assert torch.equal(s, metrics.realism_scores(vgg(real[c]), vgg(fake[c]), k).cpu())
        assert torch.equal(flipped[c], metrics.realism_scores(vgg(real[c]), vgg(fake[c].flip(0)), k).cpu())
