"""Density / coverage and realism scores without a GPU: the COUNT and RATIO_MAX modes' argument checks (they run before any
CUDA call) and workspace, the float64 reference formulas on a hand-computed case and closed forms, and the new ops' refusal
of CPU tensors."""

import math

import pytest
import torch

RBF, KNN, COVER, COUNT, RATIO_MAX = 0, 1, 2, 3, 4


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__
    __graft_entry__.build()
    from progressive_stable_diffusion_b200 import _lib
    return _lib


def test_count_and_ratio_max_reject_bad_arguments_before_any_cuda_call(lib):
    l = lib.load()
    err = lambda: l.dadd_last_error().decode()

    def call(mode, M=100, N=100, D=64, same=0, eps=1e-5, radii=16, y=32):
        return l.dadd_pairwise(16, y, M, N, D, mode, 0, same, eps, radii, 16, 16, 1 << 40, None)

    for mode in (COUNT, RATIO_MAX):
        assert call(mode, radii=None) != 0 and "dadd_pairwise" in err() and "radii" in err()
        assert call(mode, same=1, y=None) != 0 and "same_set" in err()
        assert l.dadd_pairwise_workspace_bytes(100, 100, 64, mode, 0, 1) == -1 and "same_set" in err()
        assert l.dadd_pairwise_workspace_bytes(100, 100, 64, mode, 0, 0) > 0
    for eps in (0.0, -1.0, math.nan, math.inf):
        assert call(RATIO_MAX, eps=eps) != 0 and "dadd_pairwise" in err() and "eps" in err(), eps
    for mode in (5, 7):
        assert call(mode) != 0 and "mode" in err(), mode
        assert l.dadd_pairwise_workspace_bytes(100, 100, 64, mode, 0, 0) == -1


def test_count_and_ratio_max_workspace_is_linear_in_m_plus_n(lib):
    """The tf32 split of both sets plus one int32 / float per (row, column slice): the same bytes as COVER, never M x N."""
    l = lib.load()
    split = 2 * 50_000 * 768 * 8
    ws = [l.dadd_pairwise_workspace_bytes(50_000, 50_000, 768, mode, 0, 0) for mode in (COVER, COUNT, RATIO_MAX)]
    assert ws[0] == ws[1] == ws[2]
    assert split <= ws[1] < split + 50_000 * 4 * (2 + 40) + 4096, ws


def test_reference_formulas_on_hand_computed_case():
    from progressive_stable_diffusion_b200 import metrics as m
    # reals 0, 1, 3, 7 on a line: r2 (k = 1) = [1, 1, 4, 16]
    real = torch.tensor([[0.0], [1.0], [3.0], [7.0]])
    fake = torch.tensor([[2.0], [2.5], [10.0], [11.5]])
    # density: 2 is strictly inside only the ball of 3 (d2 = 1 to real 1 is on that ball's edge), 2.5 only the ball of 3,
    # 10 the ball of 7, 11.5 none: 3 / (k N) = 0.75.  Coverage: of the reals only 3 (0.25 < 4) and 7 (9 < 16) have a fake
    # strictly inside their ball; real 1's nearest fake sits on its edge (1 < 1 is false).
    assert m.density_coverage_reference(real, fake, k=1) == (0.75, 0.5)
    # the 50th percentile of [1, 1, 4, 16] is 2.5: the kept reals are 0 and 1 (r2 = 1)
    assert m._realism_kept(m.knn_radii_reference(real, 1)).tolist() == [True, True, False, False]
    want = torch.tensor([1.0, 2.0 / 3.0, 1.0 / 9.0, 1.0 / 10.5], dtype=torch.float64)
    got = m.realism_scores_reference(real, fake, k=1)
    assert torch.allclose(got, want, rtol=1e-5, atol=0), got          # eps = 1e-5 moves 1 / sqrt(1 + eps) by 5e-6


def test_reference_closed_forms():
    from progressive_stable_diffusion_b200 import metrics as m
    g = torch.Generator().manual_seed(0)
    x = torch.nn.functional.normalize(torch.randn(40, 16, generator=g), dim=1)
    far = x + 100.0
    assert m.density_coverage_reference(x, far, k=3) == (0.0, 0.0)
    assert (m.realism_scores_reference(x, far, k=3) < 1e-2).all()         # r2 <= 4 against d2 ~ 1.6e5
    r = m.knn_radii_reference(x, 3)
    kept = m._realism_kept(r).nonzero().flatten()
    copy = x[kept[:3]]                                                     # generated copies of kept reals: d2 = 0
    floor = math.sqrt(r.min().item() / m.REALISM_EPS)
    assert (m.realism_scores_reference(x, copy, k=3) >= floor * (1 - 1e-9)).all()
    assert m.REALISM_EPS == 1e-5 and m.REALISM_PRUNE_PERCENTILE == 50.0


def test_new_ops_refuse_cpu_tensors(lib):
    from progressive_stable_diffusion_b200 import ops
    x = torch.zeros(10, 8)
    with pytest.raises(lib.DaddError):
        ops.count_within_radii(x, x, torch.zeros(10))
    with pytest.raises(lib.DaddError):
        ops.max_radius_ratio(x, x, torch.zeros(10), 1e-5)
    with pytest.raises(lib.DaddError):
        ops.knn_radii(x, 1, ref=x)
