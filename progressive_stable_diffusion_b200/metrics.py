"""Image-quality metrics of the evaluation sweep: CMMD, improved precision / recall, density / coverage and realism scores.

Replaces the CMMD and precision / recall halves of ``evaluate_one_run`` (reference
``src/pipelines/evaluation/evaluation_pipeline.py:577-839,978-1179``), and adds their usual companions:

- ``cmmd``: google-research/cmmd's ``mmd`` over CLIP ViT-L/14-336 embeddings (``ClipEmbedder``);
- ``precision_recall``: Kynkaanniemi et al. 2019 over VGG16 ``fc2`` features (``VGGFeatures``);
- ``density_coverage``: Naeem et al. 2020 (clovaai/generative-evaluation-prdc) on the same features and real-set radii;
- ``realism_scores``: the per-image realism score of Kynkaanniemi et al. 2019 (section 5), for ranking generated images.

All reduce to statistics over all pairs of feature vectors, which ``ops.pairwise_rbf_sum`` / ``ops.knn_radii`` /
``ops.within_radii`` / ``ops.count_within_radii`` / ``ops.max_radius_ratio`` compute on one fused tcgen05 kernel without
materialising the M x N distance matrix.  The ``*_reference``
functions are the same formulas in float64 on whatever device their inputs are on (the tests' yardstick).  FID is not here:
its backbone is torch-fidelity's TF-ported InceptionV3, which this package cannot restate faithfully.
"""

from __future__ import annotations

from typing import Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops, wcache
from .attention_processor import compute_dtype
from .image_encoder import _ARCH, _CLIPVisionTower

CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)
CLIP_STD = (0.26862954, 0.26130258, 0.27577711)
IMAGENET_MEAN = (0.485, 0.456, 0.406)
IMAGENET_STD = (0.229, 0.224, 0.225)

# VGG16 feature layer: the output of ``classifier[:VGG_FC2_END]`` = fc2 before its ReLU, the layer the common PyTorch port of
# the improved precision / recall metric uses.  The original project's metric code is not available here, so its exact layer
# choice could not be checked against it.
VGG_FC2_END = 4

# Realism score (Kynkaanniemi et al. 2019, section 5): the real set is first pruned to the points whose k-NN radius is at most
# the REALISM_PRUNE_PERCENTILE-th percentile of all radii (linear interpolation, as np.percentile), which drops the half of the
# balls with the largest radii, so that outliers cannot dominate the max; REALISM_EPS (added to the squared distance) keeps the
# ratio finite when a generated point lands on a real one.  The original project's metric code is not available here, so these
# two values could not be checked against it.
REALISM_EPS = 1e-5
REALISM_PRUNE_PERCENTILE = 50.0


# --------------------------------------------------------------------------------------------- the metrics
def _feats(t: torch.Tensor) -> torch.Tensor:
    return t.detach().float().contiguous()


def cmmd(real_embeds: torch.Tensor, fake_embeds: torch.Tensor, sigma: float = 10.0, scale: float = 1000.0) -> float:
    """CMMD = scale * (mean k(x, x') + mean k(y, y') - 2 mean k(x, y)), k(a, b) = exp(-|a - b|^2 / (2 sigma^2)), every mean over
    all pairs including the diagonal (google-research/cmmd ``distance.mmd``).  Embeddings: (M, D), (N, D) CUDA tensors."""
    x, y = _feats(real_embeds), _feats(fake_embeds)
    gamma = 1.0 / (2.0 * sigma * sigma)
    m, n = x.shape[0], y.shape[0]
    k_xx = ops.pairwise_rbf_sum(x, None, gamma) / (m * m)
    k_yy = ops.pairwise_rbf_sum(y, None, gamma) / (n * n)
    k_xy = ops.pairwise_rbf_sum(x, y, gamma) / (m * n)
    return float(scale * (k_xx + k_yy - 2.0 * k_xy))


def precision_recall(real_feats: torch.Tensor, fake_feats: torch.Tensor, k: int = 3) -> Tuple[float, float]:
    """Improved precision and recall (Kynkaanniemi et al. 2019) on squared Euclidean distances: a set's manifold is the union
    of balls around its points with radius the distance to the k-th nearest OTHER point of the set; precision is the fraction
    of fake points inside the real manifold, recall the fraction of real points inside the fake one (``d2 <= r2``)."""
    x, y = _feats(real_feats), _feats(fake_feats)
    r_real, r_fake = ops.knn_radii(x, k), ops.knn_radii(y, k)
    precision = ops.within_radii(y, x, r_real).float().mean()
    recall = ops.within_radii(x, y, r_fake).float().mean()
    return float(precision), float(recall)


def density_coverage(real_feats: torch.Tensor, fake_feats: torch.Tensor, k: int = 3) -> Tuple[float, float]:
    """Density and coverage (Naeem et al. 2020) on squared Euclidean distances, with the real k-NN radii r2 of
    ``precision_recall`` and strict ``<`` as in clovaai/generative-evaluation-prdc:
    density = sum_j #{i : d2(y_j, x_i) < r2_i} / (k N), coverage = #{i : min_j d2(x_i, y_j) < r2_i} / M.  Needs M > k + 1 real
    and N >= 2 generated points."""
    x, y = _feats(real_feats), _feats(fake_feats)
    r_real = ops.knn_radii(x, k)
    below = torch.nextafter(r_real, torch.full_like(r_real, -float("inf")))      # d2 < r2  <=>  d2 <= the float below r2
    density = ops.count_within_radii(y, x, below).double().sum() / (k * y.shape[0])
    coverage = (ops.knn_radii(x, 1, ref=y) < r_real).double().mean()
    return float(density), float(coverage)


def _realism_kept(r_real: torch.Tensor) -> torch.Tensor:
    """The reals whose radius is at most the REALISM_PRUNE_PERCENTILE-th percentile of all radii."""
    r = r_real.double()
    return r <= torch.quantile(r, REALISM_PRUNE_PERCENTILE / 100.0)


def realism_scores(real_feats: torch.Tensor, fake_feats: torch.Tensor, k: int = 3) -> torch.Tensor:
    """(N,) float32 realism score of each generated point (Kynkaanniemi et al. 2019, section 5):
    R_j = sqrt(max over kept reals i of r2_i / (d2(y_j, x_i) + REALISM_EPS)), the ratio of Euclidean distances, where the
    kept reals are those with r2_i at most the REALISM_PRUNE_PERCENTILE-th percentile of the radii of the whole real set.
    R_j >= 1 roughly means y_j lies inside the pruned real manifold.  Needs M > k + 1 real points."""
    x, y = _feats(real_feats), _feats(fake_feats)
    r_real = ops.knn_radii(x, k)
    keep = _realism_kept(r_real)
    return ops.max_radius_ratio(y, x[keep].contiguous(), r_real[keep].contiguous(), REALISM_EPS).sqrt_()


def _sqdist64(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """float64 |a_i - b_j|^2 as |a_i|^2 + |b_j|^2 - 2 a_i . b_j (cancellation costs ~1e-16 |a||b|, far below fp32)."""
    a, b = a.double(), b.double()
    return ((a * a).sum(1)[:, None] + (b * b).sum(1)[None, :] - 2.0 * a @ b.T).clamp_min(0.0)


def cmmd_reference(real_embeds: torch.Tensor, fake_embeds: torch.Tensor, sigma: float = 10.0, scale: float = 1000.0) -> float:
    """``cmmd`` in float64 with the full distance matrices."""
    x, y = real_embeds, fake_embeds
    g = 1.0 / (2.0 * sigma * sigma)
    k = lambda a, b: torch.exp(-g * _sqdist64(a, b)).mean()
    return float(scale * (k(x, x) + k(y, y) - 2.0 * k(x, y)))


def knn_radii_reference(x: torch.Tensor, k: int) -> torch.Tensor:
    """float64 k-th smallest squared distance from each row to the OTHER rows (index j == i excluded)."""
    d = _sqdist64(x, x)
    d.fill_diagonal_(float("inf"))
    return d.kthvalue(k, dim=1).values


def within_radii_reference(q: torch.Tensor, ref: torch.Tensor, radii: torch.Tensor) -> torch.Tensor:
    return (_sqdist64(q, ref) <= radii.double()[None, :]).any(dim=1)


def precision_recall_reference(real_feats: torch.Tensor, fake_feats: torch.Tensor, k: int = 3) -> Tuple[float, float]:
    r_real, r_fake = knn_radii_reference(real_feats, k), knn_radii_reference(fake_feats, k)
    return (float(within_radii_reference(fake_feats, real_feats, r_real).double().mean()),
            float(within_radii_reference(real_feats, fake_feats, r_fake).double().mean()))


def density_coverage_reference(real_feats: torch.Tensor, fake_feats: torch.Tensor, k: int = 3) -> Tuple[float, float]:
    """``density_coverage`` in float64 with the full distance matrix."""
    r = knn_radii_reference(real_feats, k)
    inside = _sqdist64(fake_feats, real_feats) < r[None, :]                      # [fake j][real i]
    return float(inside.double().sum() / (k * fake_feats.shape[0])), float(inside.any(dim=0).double().mean())


def realism_scores_reference(real_feats: torch.Tensor, fake_feats: torch.Tensor, k: int = 3) -> torch.Tensor:
    """``realism_scores`` in float64 with the full distance matrix."""
    r = knn_radii_reference(real_feats, k)
    keep = _realism_kept(r)
    ratio = r[keep][None, :] / (_sqdist64(fake_feats, real_feats[keep]) + REALISM_EPS)
    return ratio.amax(dim=1).sqrt()


# --------------------------------------------------------------------------------------------- backbones
def _batches(images: torch.Tensor, batch_size: int, device: torch.device):
    for s in range(0, images.shape[0], batch_size):
        yield images[s:s + batch_size].to(device=device, dtype=torch.float32)


def _normalise(x: torch.Tensor, mean, std) -> torch.Tensor:
    m = torch.tensor(mean, device=x.device, dtype=x.dtype).view(1, 3, 1, 1)
    s = torch.tensor(std, device=x.device, dtype=x.dtype).view(1, 3, 1, 1)
    return (x - m) / s


class ClipEmbedder(_CLIPVisionTower):
    """CMMD's image embedding: CLIP ViT-L/14 at 336 pixels (openai/clip-vit-large-patch14-336) on this package's kernels.
    [0, 1] images (B, 3, H, W) -> bicubic resize to 336, CLIP mean / std normalisation, no crop (google-research/cmmd
    ``embedding.py``) -> projected ``image_embeds``, L2-normalised, fp32 (B, 768).  The state-dict keys are those of
    transformers' ``CLIPVisionModelWithProjection``: real weights load through ``load_state_dict``."""

    def __init__(self, batch_size: int = 32) -> None:
        super().__init__(*_ARCH["clip-vit-large-patch14-336"])
        self.batch_size = batch_size
        self.requires_grad_(False)
        self.eval()

    @torch.no_grad()
    def forward(self, images: torch.Tensor) -> torch.Tensor:
        size = self.config.image_size
        dev = self.visual_projection.weight.device
        out = []
        for x in _batches(images, self.batch_size, dev):
            x = F.interpolate(x, size=(size, size), mode="bicubic", align_corners=False)
            e = super().forward(_normalise(x, CLIP_MEAN, CLIP_STD)).image_embeds
            out.append(e / e.norm(dim=-1, keepdim=True))
        return torch.cat(out) if out else torch.zeros(0, self.config.projection_dim, device=dev)


class VGGFeatures(nn.Module):
    """Improved precision / recall features: torchvision VGG16's 4096-d fc2 output (``classifier[:VGG_FC2_END]``).  [0, 1]
    images (B, 3, H, W) -> bilinear resize to 224, ImageNet normalisation -> fp32 (B, 4096).  Runs in the package's compute
    dtype, channels-last, convolutions on cuDNN, the two GEMMs through ``ops.linear``.  Parameters keep torchvision's
    ``vgg16`` names and dtype: real weights load through ``load_state_dict``."""

    def __init__(self, batch_size: int = 64) -> None:
        super().__init__()
        import torchvision
        vgg = torchvision.models.vgg16(weights=None)
        self.features, self.avgpool, self.classifier = vgg.features, vgg.avgpool, vgg.classifier
        self.batch_size = batch_size
        self.requires_grad_(False)
        self.eval()

    def _forward16(self, x: torch.Tensor) -> torch.Tensor:
        dt = compute_dtype()
        x = _normalise(F.interpolate(x, size=(224, 224), mode="bilinear", align_corners=False), IMAGENET_MEAN, IMAGENET_STD)
        x = x.to(dt).contiguous(memory_format=torch.channels_last)
        for layer in self.features:
            if isinstance(layer, nn.Conv2d):
                x = F.conv2d(x, wcache.conv_filter(layer, "w", layer.weight, dt), wcache.cast(layer, "b", layer.bias, dt),
                             padding=layer.padding)
            elif isinstance(layer, nn.ReLU):
                x = F.relu_(x)
            else:
                x = layer(x)
        x = torch.flatten(self.avgpool(x), 1).contiguous()
        for layer in self.classifier[:VGG_FC2_END]:
            if isinstance(layer, nn.Linear):
                x = ops.linear(x, wcache.cast(layer, "w", layer.weight, dt), wcache.cast(layer, "b32", layer.bias, torch.float32),
                               bias_lp=wcache.cast(layer, "b", layer.bias, dt))
            elif isinstance(layer, nn.ReLU):
                x = F.relu_(x)
        return x.float()

    @torch.no_grad()
    def forward(self, images: torch.Tensor) -> torch.Tensor:
        dev = self.classifier[0].weight.device
        out = [self._forward16(x) for x in _batches(images, self.batch_size, dev)]
        return torch.cat(out) if out else torch.zeros(0, self.classifier[3].out_features, device=dev)
