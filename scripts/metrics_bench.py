"""Time the fused pairwise kernel (ops.knn_radii / within_radii / pairwise_rbf_sum / count_within_radii / max_radius_ratio)
against the torch fp32 path (cdist + topk / exp().mean() / a comparison or ratio reduced over the rows) on the evaluation
metrics' sizes: a LIMUC-sized real set of 11 264 images against itself (IPR radii, VGG16 fc2 width 4096), 2 400 generated
against it (IPR coverage, density counts), 2 400 generated against the kept half of it (realism scores), and CMMD's CLIP
width 768.

    python scripts/metrics_bench.py [--reps 10]

Times are CUDA events around whole calls (the tf32 split pre-pass, the GEMM with its epilogue, the merge pass and the
workspace allocation), after a warm-up call.  The 4096-wide sets (185 MB and 39 MB) exceed the 126 MB L2.  TFLOP/s counts the three tf32 passes, 3 * 2 * M * N * D, against the dense TF32 data-sheet peak of one B200.
"""

from __future__ import annotations

import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

TF32_PEAK = 1125e12          # dense TF32, one B200 at 1000 W (NVIDIA HGX B200 data sheet / 16)


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps * 1e-3, torch.cuda.max_memory_allocated() - base, out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    from progressive_stable_diffusion_b200 import metrics, ops
    assert torch.cuda.is_available(), "needs a CUDA device"
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:                                      # noqa: BLE001
        q = torch.cuda.get_device_name()
    print(f"device: {q}")
    g = torch.Generator(device="cuda").manual_seed(0)
    real = torch.relu(torch.randn(11264, 4096, device="cuda", generator=g))
    fake = torch.relu(torch.randn(2400, 4096, device="cuda", generator=g) * 1.05)
    creal = torch.nn.functional.normalize(torch.randn(11264, 768, device="cuda", generator=g), dim=1)
    cfake = torch.nn.functional.normalize(torch.randn(2400, 768, device="cuda", generator=g) + 0.02, dim=1)
    k, gamma = 3, 1.0 / 200.0
    r_real = ops.knn_radii(real, k)
    keep = metrics._realism_kept(r_real)
    kept, r_kept = real[keep].contiguous(), r_real[keep].contiguous()

    def torch_radii():
        d = torch.cdist(real, real).square_()
        d.fill_diagonal_(float("inf"))
        return torch.topk(d, k, dim=1, largest=False).values[:, -1]

    work = [
        ("radii 11264 x 11264, D 4096, k 3", 11264, 11264, 4096, lambda: ops.knn_radii(real, k), torch_radii,
         lambda a, b: f"max |diff| / max radius {((a - b).abs().max() / b.max()).item():.2e}"),
        ("coverage 2400 x 11264, D 4096", 2400, 11264, 4096, lambda: ops.within_radii(fake, real, r_real),
         lambda: (torch.cdist(fake, real).square_() <= r_real[None]).any(1),
         lambda a, b: f"{int((a != b).sum())} of {a.numel()} flags differ"),
        ("CMMD sum 11264 x 2400, D 768", 11264, 2400, 768, lambda: ops.pairwise_rbf_sum(creal, cfake, gamma),
         lambda: torch.exp(-gamma * torch.cdist(creal, cfake).square_()).sum(),
         lambda a, b: f"relative diff {abs(a.item() - b.item()) / b.item():.2e}"),
        ("density counts 2400 x 11264, D 4096", 2400, 11264, 4096, lambda: ops.count_within_radii(fake, real, r_real),
         lambda: (torch.cdist(fake, real).square_() <= r_real[None]).sum(1),
         lambda a, b: f"{int((a != b).sum())} of {a.numel()} counts differ, max |diff| {int((a - b).abs().max())}"),
        (f"realism 2400 x {kept.shape[0]} kept, D 4096", 2400, kept.shape[0], 4096,
         lambda: ops.max_radius_ratio(fake, kept, r_kept, metrics.REALISM_EPS),
         lambda: (r_kept[None] / (torch.cdist(fake, kept).square_() + metrics.REALISM_EPS)).amax(1),
         lambda a, b: f"max relative diff {((a - b).abs() / b).max().item():.2e}"),
    ]
    print(f"torch.backends.cuda.matmul.allow_tf32 = {torch.backends.cuda.matmul.allow_tf32} (cdist runs in fp32)")
    for name, m, n, d, ours, ref, agree in work:
        t0, m0, o0 = timed(ours, args.reps)
        t1, m1, o1 = timed(ref, args.reps)
        flops = 3 * 2.0 * m * n * d
        print(f"{name}: kernel {t0 * 1e3:.2f} ms ({flops / t0 / 1e12:.0f} TFLOP/s three-pass, {flops / t0 / TF32_PEAK * 100:.1f} % of "
              f"the tf32 peak), peak mem {m0 / 1e6:.0f} MB | torch fp32 {t1 * 1e3:.2f} ms, peak mem {m1 / 1e6:.0f} MB | "
              f"speed-up {t1 / t0:.2f}x | {agree(o0.double() if o0.is_floating_point() else o0.long(), o1.double() if o1.is_floating_point() else o1.long())}")


if __name__ == "__main__":
    main()
