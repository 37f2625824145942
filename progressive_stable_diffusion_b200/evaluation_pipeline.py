"""Batched evaluation sampling for B200: the sampling half of
``/root/reference/src/pipelines/evaluation/evaluation_pipeline.py`` (``_prepare_conditioning`` :406-461,
``_set_delta_scale`` :464-468, ``_ddim_sample_batched`` :471-564, ``_decode_latents`` :567-574, ``GenerationJob`` / ``_collect_jobs``
:83-89,843-864, the job order, batching and per-class grouping of ``generate_all`` :867-975) - and its scoring: ``evaluate_images`` computes CMMD and improved precision / recall per target class
(``evaluate_one_run`` :577-839,978-1179), optionally density / coverage, on ``metrics.py``; ``realism_by_class`` scores each
generated image.  A sweep runs ``generate_all`` -> ``group_by_target`` -> ``evaluate_images`` / ``realism_by_class``.  FID is not computed: its backbone, torch-fidelity's TF-ported InceptionV3, is not available here.
"""

from __future__ import annotations

from dataclasses import dataclass
from pathlib import Path
from typing import Dict, List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import metrics, parallel
from .inference_pipeline_ip import (_latents_to_images, _prepare_conditioning as _prep, _sample,
                                    _set_delta_scale_on_processors)


ALL_MES_CLASSES = [0, 1, 2, 3]                                                   # reference :79
IMAGE_EXTENSIONS = {".bmp", ".png", ".jpg", ".jpeg", ".tif", ".tiff"}            # reference :80


@dataclass
class GenerationJob:
    """One source image -> one target MES class (reference :83-89)."""

    source_path: Path
    source_label: int
    target_label: int


def _collect_jobs(data_roots: Sequence[Path], max_per_class: int = 0) -> List[GenerationJob]:
    """Every source image under ``<root>/<class>/`` produces one job for each of the three OTHER MES classes, roots and classes
    in order, files sorted, at most ``max_per_class`` files per class directory (reference :843-864)."""
    jobs: List[GenerationJob] = []
    for data_root in data_roots:
        for cls in ALL_MES_CLASSES:
            cls_dir = Path(data_root) / str(cls)
            if not cls_dir.is_dir():
                continue
            paths = sorted(q for q in cls_dir.iterdir() if q.suffix.lower() in IMAGE_EXTENSIONS)
            if max_per_class > 0:
                paths = paths[:max_per_class]
            for q in paths:
                jobs.extend(GenerationJob(q, cls, target) for target in ALL_MES_CLASSES if target != cls)
    return jobs


def sweep_order(jobs: Sequence[GenerationJob]) -> Tuple[List[GenerationJob], List[Path]]:
    """The order ``generate_all`` of the reference walks the jobs in (:897-903): sorted by (str(source path), target label), i.e.
    grouped by source image.  Returns the sorted jobs and the distinct source paths in first-appearance order (the structure
    images to load / encode ONCE each: the reference re-loads one per batch, :921-933)."""
    jobs_sorted = sorted(jobs, key=lambda j: (str(j.source_path), j.target_label))
    sources: List[Path] = []
    for j in jobs_sorted:
        if not sources or sources[-1] != j.source_path:
            sources.append(j.source_path)
    return jobs_sorted, sources


def as_index_jobs(jobs_sorted: Sequence[GenerationJob], sources: Sequence[Path]) -> List[Tuple[int, float, float]]:
    """``GenerationJob``s -> the (source index, source label, target label) triples ``generate_all`` below takes."""
    where = {q: i for i, q in enumerate(sources)}
    return [(where[j.source_path], float(j.source_label), float(j.target_label)) for j in jobs_sorted]


def group_by_target(images: Dict[int, Tensor], jobs_sorted: Sequence[GenerationJob], image_size: int) -> Dict[int, Tensor]:
    """Per-job images -> ``{target class: (N, 3, H, W)}`` in sweep order, empty classes as (0, 3, H, W): what the reference's
    ``generate_all`` returns (:955-975).  ``images``: job index -> (3, H, W) (this rank's share, or all ranks' merged)."""
    out: Dict[int, Tensor] = {}
    for cls in ALL_MES_CLASSES:
        picked = [images[i][None] for i, j in enumerate(jobs_sorted) if j.target_label == cls and i in images]
        out[cls] = torch.cat(picked, dim=0) if picked else torch.zeros(0, 3, image_size, image_size)
    return out


def _prepare_conditioning(module, target_labels: Tensor, source_labels: Tensor, structure_images: Tensor,
                          image_scale: float = 1.0, zero_aoe: bool = False) -> Tensor:
    return _prep(module, target_labels, source_labels, structure_images, image_scale=image_scale, zero_aoe=zero_aoe)


def _set_delta_scale(module, scale: float) -> None:
    _set_delta_scale_on_processors(module, scale)


@torch.no_grad()
def _ddim_sample_batched(module, target_labels: Tensor, source_labels: Tensor, structure_images: Tensor,
                         sampling_steps: int, device: torch.device, eta: float = 0.0, image_scale: float = 1.0,
                         steer_scale: float = 0.0, guidance_scale: float = 1.0, *, init_latents: Optional[Tensor] = None,
                         use_graph: bool = True) -> Tensor:
    """Like ``_ddim_sample_ip`` but every sample draws its own initial noise (reference :506)."""
    device = torch.device(device)
    routing = getattr(module.diff_cfg, "use_routing_gates", True)
    do_cfg = (not routing) and (guidance_scale != 1.0)
    b = target_labels.shape[0]
    h = module.cfg.dataset.image_size // 8
    if sampling_steps > module.diff_cfg.num_train_timesteps:
        raise ValueError(f"sampling_steps={sampling_steps} must be <= num_train_timesteps={module.diff_cfg.num_train_timesteps}")
    if init_latents is None:
        init_latents = torch.randn(b, module.cfg.model.latent_channels, h, h, device=device, dtype=torch.float32)
    return _sample(module, target_labels, source_labels, structure_images, init_latents.to(device), sampling_steps, device,
                   eta, image_scale, None, steer_scale, guidance_scale, do_cfg, use_graph)


@torch.no_grad()
def _decode_latents(module, latents: Tensor) -> Tensor:
    """latents -> [0,1] RGB (B,3,H,W) on the CPU (reference :567-574)."""
    return _latents_to_images(module, latents).float().cpu()


@torch.no_grad()
def generate_all(module, jobs: Sequence[Tuple[int, float, float]], image_tokens: Tensor, device: torch.device,
                 batch_size: int = 12, sampling_steps: int = 50, image_scale: float = 1.0, steer_scale: float = 0.0,
                 guidance_scale: float = 1.0, eta: float = 0.0, seed: int = 42, rank: int = 0, world_size: int = 1,
                 decode: bool = True) -> Dict[int, Tensor]:
    """Run this rank's share of an evaluation sweep.  ``jobs`` = (source index into ``image_tokens``, source label,
    target label), already in the reference's sorted order (:897-903).  The reference seeds once and draws noise batch by
    batch (:909,506); to keep a sharded run identical to the single-process one, ALL initial noise is drawn up front in
    job order from one seeded generator and each rank takes its slice (SURVEY.md 8e)."""
    device = torch.device(device)
    h = module.cfg.dataset.image_size // 8
    c = module.cfg.model.latent_channels
    gen = torch.Generator(device="cpu").manual_seed(seed)
    noise = torch.randn(len(jobs), c, h, h, generator=gen, dtype=torch.float32)
    mine = parallel.shard_indices(len(jobs), rank, world_size)
    out: Dict[int, Tensor] = {}
    for s in range(0, len(mine), batch_size):
        idx = mine[s:s + batch_size]
        if len(idx) < batch_size:                       # keep the captured batch shape: pad with repeats, drop after
            idx_run = idx + [idx[-1]] * (batch_size - len(idx))
        else:
            idx_run = idx
        src = torch.tensor([jobs[i][1] for i in idx_run], dtype=torch.float32, device=device)
        tgt = torch.tensor([jobs[i][2] for i in idx_run], dtype=torch.float32, device=device)
        tok = image_tokens[[jobs[i][0] for i in idx_run]].to(device)
        lat = _ddim_sample_batched(module, tgt, src, tok, sampling_steps, device, eta, image_scale, steer_scale,
                                   guidance_scale, init_latents=noise[idx_run].to(device))
        res = _decode_latents(module, lat) if decode else lat.cpu()
        for k, i in enumerate(idx):
            out[i] = res[k]
    return out


@torch.no_grad()
def evaluate_images(real_by_class: Dict[int, Tensor], fake_by_class: Dict[int, Tensor], clip: "metrics.ClipEmbedder",
                    vgg: "metrics.VGGFeatures", k: int = 3, density_coverage: bool = False) -> Dict[object, Dict[str, float]]:
    """CMMD and improved precision / recall of generated against real [0, 1] images, per target class and over all classes.
    ``real_by_class`` / ``fake_by_class``: ``{class: (N, 3, H, W)}`` as ``group_by_target`` returns them.  Returns
    ``{class: {"cmmd", "precision", "recall"}, ..., "all": {...}}``.  A class missing or empty on either side is left out;
    precision and recall are NaN where a side has k + 1 points or fewer (a k-NN radius needs k other points and more).
    ``density_coverage``: each group also gets ``"density"`` and ``"coverage"`` (Naeem et al. 2020, on the same VGG features
    and real radii), NaN under the same condition."""
    out: Dict[object, Dict[str, float]] = {}
    feats = {}
    for cls in ALL_MES_CLASSES:
        real, fake = real_by_class.get(cls), fake_by_class.get(cls)
        if real is None or fake is None or real.shape[0] == 0 or fake.shape[0] == 0:
            continue
        feats[cls] = (clip(real), clip(fake), vgg(real), vgg(fake))
    groups = list(feats.items())
    if feats:
        groups.append(("all", tuple(torch.cat([f[i] for f in feats.values()]) for i in range(4))))
    for key, (cr, cf, vr, vf) in groups:
        res = {"cmmd": metrics.cmmd(cr, cf), "precision": float("nan"), "recall": float("nan")}
        if density_coverage:
            res["density"] = res["coverage"] = float("nan")
        if min(vr.shape[0], vf.shape[0]) > k + 1:
            res["precision"], res["recall"] = metrics.precision_recall(vr, vf, k)
            if density_coverage:
                res["density"], res["coverage"] = metrics.density_coverage(vr, vf, k)
        out[key] = res
    return out


@torch.no_grad()
def realism_by_class(real_by_class: Dict[int, Tensor], fake_by_class: Dict[int, Tensor], vgg: "metrics.VGGFeatures",
                     k: int = 3) -> Dict[int, Tensor]:
    """Realism score (``metrics.realism_scores``) of every generated [0, 1] image against the real images of its own class:
    ``{class: (N_fake,) CPU float32}``, index n scoring the n-th image of ``fake_by_class[class]`` (``group_by_target``'s
    order), for ranking or filtering generated images.  A class is left out when either side is missing or empty, or when it
    has k + 1 real images or fewer."""
    out: Dict[int, Tensor] = {}
    for cls in ALL_MES_CLASSES:
        real, fake = real_by_class.get(cls), fake_by_class.get(cls)
        if real is None or fake is None or real.shape[0] <= k + 1 or fake.shape[0] == 0:
            continue
        out[cls] = metrics.realism_scores(vgg(real), vgg(fake), k).cpu()
    return out
