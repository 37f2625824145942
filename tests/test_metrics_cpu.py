"""CMMD / improved precision-recall without a GPU: the pairwise entry point's argument checks (they run before any CUDA call),
the 336-pixel CLIP tower's layout, the float64 reference formulas of metrics.py, and the pairwise kernel's sm_100a instructions."""

import math
import re
import shutil
import subprocess

import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__
    __graft_entry__.build()
    from progressive_stable_diffusion_b200 import _lib
    return _lib


def test_pairwise_rejects_bad_arguments_before_any_cuda_call(lib):
    l = lib.load()
    err = lambda: l.dadd_last_error().decode()
    RBF, KNN, COVER = 0, 1, 2
    big = 1 << 40

    def call(M=100, N=100, D=64, mode=RBF, k=3, same=0, radii=16, ws_bytes=big, x=16, y=32):
        return l.dadd_pairwise(x, y, M, N, D, mode, k, same, 0.5, radii, 16, 16, ws_bytes, None)

    assert call(D=12) != 0 and "dadd_pairwise" in err() and "D % 8" in err()
    assert l.dadd_pairwise_workspace_bytes(100, 100, 12, RBF, 0, 0) == -1 and "D % 8" in err()
    assert call(mode=KNN, k=0) != 0 and "dadd_pairwise" in err() and "1 <= k <= 16" in err()
    assert call(mode=KNN, k=17) != 0 and "1 <= k <= 16" in err()
    assert call(mode=KNN, k=3, N=3) != 0 and "dadd_pairwise" in err() and "more than k" in err()
    assert call(mode=KNN, k=3, M=4, N=4, same=1, y=None) != 0 and "more than k + 1" in err()
    assert l.dadd_pairwise_workspace_bytes(5, 5, 64, KNN, 3, 1) > 0                       # N = k + 2 with same_set is enough
    assert l.dadd_pairwise_workspace_bytes(4, 4, 64, KNN, 3, 0) > 0                       # N = k + 1 without
    assert call(mode=COVER, radii=None) != 0 and "dadd_pairwise" in err() and "radii" in err()
    need = l.dadd_pairwise_workspace_bytes(100, 100, 64, RBF, 0, 0)
    assert need > 0
    assert call(ws_bytes=need - 1) != 0 and "dadd_pairwise" in err() and "workspace" in err()
    assert call(mode=7) != 0 and "mode" in err()
    assert call(same=1, N=99, y=None) != 0 and "same_set" in err()
    assert call(x=None) != 0 and "dadd_pairwise" in err()


def test_pairwise_workspace_has_no_m_by_n_term(lib):
    """The workspace is the tf32 split of the rows plus per-slice partials: linear in M + N, never M x N."""
    l = lib.load()
    for mode, k in ((0, 0), (1, 16), (2, 0)):
        ws = l.dadd_pairwise_workspace_bytes(50_000, 50_000, 768, mode, k, 1 if mode != 2 else 0)
        split = (1 if mode != 2 else 2) * 50_000 * 768 * 8
        assert split <= ws < split + 50_000 * 4 * (2 + 16 * 40) + 4096, (mode, ws)
    assert l.dadd_pairwise_workspace_bytes(50_000, 50_000, 768, 0, 0, 1) < 50_000 * 50_000 * 4 / 20


def test_clip_336_tower_layout():
    import progressive_stable_diffusion_b200 as P
    from oracle import weights
    enc = P.ImageEncoder("openai/clip-vit-large-patch14-336")
    assert enc.image_encoder.vision_model.embeddings.position_embedding.num_embeddings == 577
    assert enc.hidden_size == 1024 and enc.projection_dim == 768
    state = weights.make_clip_vision_state(image=336)
    enc.image_encoder.load_state_dict(state, strict=True)
    emb = P.ClipEmbedder()
    emb.load_state_dict(state, strict=True)                  # the metric's embedder takes transformers' keys as they are


def test_vgg_features_take_torchvision_state_dicts():
    import torchvision
    import progressive_stable_diffusion_b200 as P
    from progressive_stable_diffusion_b200 import metrics
    v = P.VGGFeatures()
    v.load_state_dict(torchvision.models.vgg16(weights=None).state_dict(), strict=True)
    assert metrics.VGG_FC2_END == 4 and v.classifier[metrics.VGG_FC2_END - 1].out_features == 4096


def test_reference_formulas_on_hand_computed_cases():
    from progressive_stable_diffusion_b200 import metrics as m
    # two 1-D points at 0 and 3, one at 1: d2(x, x') in {0, 9}, d2(x, y) in {1, 4}
    x = torch.tensor([[0.0], [3.0]])
    y = torch.tensor([[1.0]])
    sigma = 2.0
    g = 1 / (2 * sigma ** 2)
    kxx = (2 + 2 * math.exp(-9 * g)) / 4
    kyy = 1.0
    kxy = (math.exp(-1 * g) + math.exp(-4 * g)) / 2
    assert m.cmmd_reference(x, y, sigma=sigma, scale=1.0) == pytest.approx(kxx + kyy - 2 * kxy, rel=1e-12)
    # radii on a line 0, 1, 3, 7: nearest other point (k = 1) and second nearest (k = 2), squared
    p = torch.tensor([[0.0], [1.0], [3.0], [7.0]])
    assert m.knn_radii_reference(p, 1).tolist() == [1.0, 1.0, 4.0, 16.0]
    assert m.knn_radii_reference(p, 2).tolist() == [9.0, 4.0, 9.0, 36.0]
    # the index, not the distance, excludes a point: a duplicate is a neighbour at distance 0
    assert m.knn_radii_reference(torch.tensor([[0.0], [0.0], [5.0]]), 1).tolist() == [0.0, 0.0, 25.0]
    # coverage is inclusive: 2 lies on the balls of radius^2 = 1 around 1 and 3, 7.5 on the one of 0.25 around 7, 10 in none
    q = torch.tensor([[2.0], [10.0], [7.5]])
    assert m.within_radii_reference(q, p, torch.tensor([0.5, 1.0, 1.0, 0.25])).tolist() == [True, False, True]
    assert m.within_radii_reference(q, p, torch.tensor([0.5, 0.5, 0.5, 0.24])).tolist() == [False, False, False]
    # real radii (k = 1) [1, 1, 4, 16]: fakes 2 (d2 1 to 1), 2.5 (0.25 to 3), 10 (9 to 7) are in, 11.5 (20.25 to 7) is out;
    # fake radii [0.25, 0.25, 2.25, 2.25]: of the reals only 3 (0.25 to 2.5) is in
    fake = torch.tensor([[2.0], [2.5], [10.0], [11.5]])
    assert m.precision_recall_reference(p, fake, k=1) == (0.75, 0.25)


def test_reference_closed_forms():
    from progressive_stable_diffusion_b200 import metrics as m
    g = torch.Generator().manual_seed(0)
    x = torch.nn.functional.normalize(torch.randn(40, 16, generator=g), dim=1)
    assert abs(m.cmmd_reference(x, x)) < 1e-9
    assert m.precision_recall_reference(x, x.clone(), k=3) == (1.0, 1.0)
    far = x + 100.0
    assert m.precision_recall_reference(x, far, k=3) == (0.0, 0.0)
    k_xx = torch.exp(-m._sqdist64(x, x) / 2).mean().item()           # sigma = 1; far away k(x, y) = 0 and k_yy = k_xx
    assert m.cmmd_reference(x, far, sigma=1.0, scale=1.0) == pytest.approx(2 * k_xx, rel=1e-6)


def test_ops_refuse_cpu_tensors(lib):
    from progressive_stable_diffusion_b200 import ops
    x = torch.zeros(10, 8)
    with pytest.raises(lib.DaddError):
        ops.pairwise_rbf_sum(x, None, 0.5)
    with pytest.raises(lib.DaddError):
        ops.knn_radii(x, 3)
    with pytest.raises(lib.DaddError):
        ops.within_radii(x, x, torch.zeros(10))


def test_pairwise_kernel_is_blackwell_native(lib):
    """Like the other tcgen05 kernels: tcgen05 MMAs, TMA tensor loads and TMEM loads in every mode's instance."""
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    lib.load()
    sass = subprocess.run(["cuobjdump", "-sass", lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    per, name = {}, None
    for line in sass.splitlines():
        f = re.search(r"Function : (\S+)", line)
        if f:
            name = f.group(1)
            per[name] = ""
            continue
        ins = re.search(r"(UTCHMMA|UTMALDG|LDTM)", line)
        if name and ins:
            per[name] += ins.group(1) + " "
    ks = [v for k, v in per.items() if "pairwise_kernel" in k]
    assert len(ks) == 3
    assert all("UTCHMMA" in v and "UTMALDG" in v and "LDTM" in v for v in ks)
