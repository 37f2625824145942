"""Parity of each sm_100a kernel (called through the C ABI wrappers) against the CPU oracle / golden vectors."""

import math
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import conditioning, processors, sampler  # noqa: E402
from tests.golden import cases  # noqa: E402
from tests.golden.store import Golden  # noqa: E402

GOLD = Golden(os.path.join(os.path.dirname(__file__), "golden", "reference_modules.npz"))
DEV = "cuda:0"


def _ops():
    from progressive_stable_diffusion_b200 import ops
    return ops


def rel_err(a: torch.Tensor, ref: torch.Tensor) -> float:
    """max |a - ref| / max |ref| : the 'max relative error' of BASELINE.md section 4."""
    return ((a.double().cpu() - ref.double().cpu()).abs().max() / ref.double().abs().max().clamp_min(1e-30)).item()


# ------------------------------------------------------------------------------------------------ DDIM (bit-exact)
@pytest.mark.parametrize("eta", [0.0, 0.5])
@pytest.mark.parametrize("cfg", [False, True])
@pytest.mark.parametrize("eps_dtype", [torch.float32, torch.bfloat16])
def test_ddim_step_bit_exact_all_schedule_positions(eta, cfg, eps_dtype):
    ops = _ops()
    from progressive_stable_diffusion_b200.inference_pipeline_ip import ddim_schedule
    _, ac = sampler.build_noise_schedule()
    ts, table = ddim_schedule(ac, 1000, 50, eta)
    assert ts.tolist() == sampler.ddim_timesteps().tolist()
    g = torch.Generator().manual_seed(5)
    n = 13 * 4 * 32 * 32
    x = torch.randn(n, generator=g) * 3
    for i in range(50):
        ec = torch.randn(n, generator=g).to(eps_dtype)
        eu = torch.randn(n, generator=g).to(eps_dtype) if cfg else None
        noise = torch.randn(n, generator=g)
        eps_ref = sampler.cfg_combine(ec.float(), eu.float(), 2.5) if cfg else ec.float()
        t_prev = None if i == 49 else int(ts[i + 1])
        want = sampler.ddim_update(x, eps_ref, ac, int(ts[i]), t_prev, eta, noise)
        row = table[i].tolist()
        got = ops.ddim_step_(x.to(DEV).clone(), ec.to(DEV), None if eu is None else eu.to(DEV), 2.5, row[0], row[1], row[2],
                             row[3], row[4], noise.to(DEV) if eta else None, 4.0, bool(row[5]))
        assert torch.equal(got.cpu(), want), f"step {i}: max diff {(got.cpu() - want).abs().max()}"
        x = want if i < 49 else x


def test_ddim_step_table_matches_scalar_version():
    ops = _ops()
    from progressive_stable_diffusion_b200.inference_pipeline_ip import ddim_schedule
    _, ac = sampler.build_noise_schedule()
    ts, table = ddim_schedule(ac, 1000, 50, 0.0)
    g = torch.Generator().manual_seed(6)
    n = 4096 * 3 + 5
    x0 = torch.randn(n, generator=g)
    eps = torch.randn(50, n, generator=g)
    terms = torch.randn(50, 64, generator=g)
    xa = x0.to(DEV).clone()
    xb = x0.to(DEV).clone()
    state = torch.zeros(2, dtype=torch.int32, device=DEV)
    row_out = torch.zeros(1, 64, device=DEV)
    tab = table.to(DEV)
    for i in range(50):
        r = table[i].tolist()
        ops.ddim_step_(xa, eps[i].to(DEV), None, 1.0, r[0], r[1], r[2], r[3], r[4], None, 4.0, bool(r[5]))
        ops.step_begin_(state, terms.to(DEV), row_out)
        assert torch.equal(row_out.cpu()[0], terms[i])
        ops.ddim_step_table_(xb, eps[i].to(DEV), None, 1.0, tab, state, None, 4.0)
        assert torch.equal(xa, xb)
    assert state.tolist() == [49, 50]


# ------------------------------------------------------------------------------------------------ GroupNorm
GN_SHAPES = [(320, 32), (640, 32), (960, 32), (320, 16), (640, 16), (1280, 16), (1920, 16), (640, 8), (1280, 8), (1920, 8),
             (2560, 8), (1280, 4), (2560, 4), (128, 64), (512, 32)]


@pytest.mark.parametrize("c,hw", GN_SHAPES)
@pytest.mark.parametrize("layout", ["nhwc", "nchw"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
def test_groupnorm_silu_16bit(c, hw, layout, dtype):
    ops = _ops()
    g = torch.Generator().manual_seed(c + hw)
    b = 3
    x = (torch.randn(b, c, hw, hw, generator=g) * 1.5 + 0.7).to(dtype)
    gamma = 1 + 0.2 * torch.randn(c, generator=g)
    beta = 0.2 * torch.randn(c, generator=g)
    add = torch.randn(b, c, generator=g)
    for silu, use_add, eps in ((True, False, 1e-5), (True, True, 1e-5), (False, False, 1e-6)):
        xin = x.float() + (add[:, :, None, None] if use_add else 0)
        ref = F.group_norm(xin, 32, gamma, beta, eps)
        ref = F.silu(ref) if silu else ref
        xd = x.to(DEV)
        if layout == "nhwc":
            xd = xd.contiguous(memory_format=torch.channels_last)
        y = ops.group_norm(xd, gamma.to(DEV), beta.to(DEV), 32, eps, silu, add.to(DEV) if use_add else None)
        assert y.stride() == xd.stride()
        err = (y.float().cpu() - ref).abs().max().item()
        ulp = 2.0 ** -7 if dtype == torch.bfloat16 else 2.0 ** -10
        assert err <= ulp * max(1.0, ref.abs().max().item()), (c, hw, layout, silu, use_add, err)


@pytest.mark.parametrize("layout", ["nhwc", "nchw"])
def test_groupnorm_fp32_and_large_mean(layout):
    ops = _ops()
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 320, 16, 16, generator=g) * 0.1 + 30.0          # |mean| >> std: cancellation trap
    gamma, beta = torch.ones(320), torch.zeros(320)
    ref = F.group_norm(x.double(), 32, gamma.double(), beta.double(), 1e-5).float()
    xd = x.to(DEV).contiguous(memory_format=torch.channels_last) if layout == "nhwc" else x.to(DEV)
    y = ops.group_norm(xd, gamma.to(DEV), beta.to(DEV), 32, 1e-5, False)
    assert (y.cpu() - ref).abs().max().item() < 2e-3


def test_groupnorm_expanded_chan_add_row():
    ops = _ops()
    g = torch.Generator().manual_seed(4)
    x = torch.randn(4, 320, 8, 8, generator=g).to(torch.bfloat16)
    row = torch.randn(1, 640, generator=g)
    gamma, beta = torch.ones(320), torch.zeros(320)
    add = row[:, 320:].expand(4, -1)                                     # stride-0 rows, offset view
    ref = F.silu(F.group_norm(x.float() + add[:, :, None, None], 32, gamma, beta, 1e-5))
    y = ops.group_norm(x.to(DEV).contiguous(memory_format=torch.channels_last), gamma.to(DEV), beta.to(DEV), 32, 1e-5, True,
                       row.to(DEV)[:, 320:].expand(4, -1))
    assert (y.float().cpu() - ref).abs().max().item() < 0.04


# the 12 skip concatenations of the up path (C_hidden, C_skip, side) at 256x256, plus a 512x512 site (flat path -> not supported)
GN_CAT_SHAPES = [(1280, 1280, 4), (1280, 1280, 8), (1280, 640, 8), (1280, 640, 16), (640, 640, 16), (640, 320, 16),
                 (640, 320, 32), (320, 320, 32)]


@pytest.mark.parametrize("c1,c2,hw", GN_CAT_SHAPES)
@pytest.mark.parametrize("b", [3, 26])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
def test_groupnorm_cat_equals_groupnorm_of_concatenation(c1, c2, hw, b, dtype):
    """dadd_groupnorm_cat_fwd([x1 | x2]) must equal dadd_groupnorm_fwd(torch.cat) BIT FOR BIT (same kernel, same arithmetic,
    only the addressing differs) and match the fp32 reference."""
    ops = _ops()
    g = torch.Generator().manual_seed(c1 + c2 + hw + b)
    x1 = (torch.randn(b, c1, hw, hw, generator=g) * 1.5 + 0.7).to(dtype).to(DEV).contiguous(memory_format=torch.channels_last)
    x2 = (torch.randn(b, c2, hw, hw, generator=g) * 0.6 - 0.4).to(dtype).to(DEV).contiguous(memory_format=torch.channels_last)
    c = c1 + c2
    gamma, beta = (1 + 0.2 * torch.randn(c, generator=g)).to(DEV), (0.2 * torch.randn(c, generator=g)).to(DEV)
    add = torch.randn(b, c, generator=g).to(DEV)
    assert ops.group_norm_cat_supported(x1, x2, 32)
    cat = torch.cat([x1, x2], dim=1).contiguous(memory_format=torch.channels_last)
    for silu, use_add in ((True, False), (True, True), (False, False)):
        want = ops.group_norm(cat, gamma, beta, 32, 1e-5, silu, add if use_add else None)
        got = ops.group_norm_cat(x1, x2, gamma, beta, 32, 1e-5, silu, add if use_add else None)
        assert got.shape == want.shape and got.stride() == want.stride()
        assert torch.equal(got, want), (c1, c2, hw, silu, use_add, (got.float() - want.float()).abs().max().item())
    ref = F.group_norm(cat.float().cpu(), 32, gamma.cpu(), beta.cpu(), 1e-5)       # the last combination: no SiLU, no add
    ulp = 2.0 ** -7 if dtype == torch.bfloat16 else 2.0 ** -10
    assert (got.float().cpu() - ref).abs().max().item() <= ulp * max(1.0, ref.abs().max().item())


def test_groupnorm_cat_large_activations_take_the_flat_passes():
    """A 512x512-latent site (7.9 MB per sample) and a > 48 MB batch: the flat stats/apply kernels read both sources too, and
    equal the kernel on the materialised concatenation bit for bit."""
    ops = _ops()
    for b, c1, c2, hw in ((2, 640, 320, 64), (60, 320, 320, 32)):
        g = torch.Generator().manual_seed(b + hw)
        x1 = torch.randn(b, c1, hw, hw, generator=g).to(torch.bfloat16).to(DEV).contiguous(memory_format=torch.channels_last)
        x2 = (torch.randn(b, c2, hw, hw, generator=g) * 0.5 + 1).to(torch.bfloat16).to(DEV).contiguous(memory_format=torch.channels_last)
        gamma, beta = (1 + 0.2 * torch.randn(c1 + c2, generator=g)).to(DEV), (0.2 * torch.randn(c1 + c2, generator=g)).to(DEV)
        add = torch.randn(b, c1 + c2, generator=g).to(DEV)
        assert ops.group_norm_cat_supported(x1, x2, 32)
        cat = torch.cat([x1, x2], dim=1).contiguous(memory_format=torch.channels_last)
        want = ops.group_norm(cat, gamma, beta, 32, 1e-5, True, add)
        got = ops.group_norm_cat(x1, x2, gamma, beta, 32, 1e-5, True, add)
        assert torch.equal(got, want)
        ref = F.silu(F.group_norm(cat[:2].float().cpu() + add[:2].cpu()[:, :, None, None], 32, gamma.cpu(), beta.cpu(), 1e-5))
        assert (got[:2].float().cpu() - ref).abs().max().item() <= 2.0 ** -7 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("b,c,hw", [(26, 320, 32), (13, 128, 128), (5, 960, 32), (2, 2560, 4), (1, 64, 200)])
def test_groupnorm_nhwc_many_chunks_and_reproducible(b, c, hw):
    """Shapes whose samples split into many pixel chunks (incl. > 16: the separate finalise pass, and ragged last chunks);
    the two-pass kernels use no atomics, so two runs agree bit for bit."""
    ops = _ops()
    g = torch.Generator().manual_seed(b * c + hw)
    x = (torch.randn(b, c, hw, hw, generator=g) * 2 - 1.3).to(torch.bfloat16)
    gamma, beta = 1 + 0.2 * torch.randn(c, generator=g), 0.2 * torch.randn(c, generator=g)
    add = torch.randn(b, c, generator=g)
    ref = F.silu(F.group_norm(x.float() + add[:, :, None, None], 32, gamma, beta, 1e-5))
    xd = x.to(DEV).contiguous(memory_format=torch.channels_last)
    y1 = ops.group_norm(xd, gamma.to(DEV), beta.to(DEV), 32, 1e-5, True, add.to(DEV))
    y2 = ops.group_norm(xd, gamma.to(DEV), beta.to(DEV), 32, 1e-5, True, add.to(DEV))
    assert torch.equal(y1, y2)
    assert (y1.float().cpu() - ref).abs().max().item() <= 2.0 ** -7 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("b,c,hw,dtype", [(104, 320, 32, torch.float16), (30, 640, 16, torch.bfloat16), (150, 1280, 4, torch.float16),
                                          (7, 2560, 8, torch.float16), (2, 320, 64, torch.float16)])
def test_groupnorm_streaming_kernel_many_items_graph_replay(b, c, hw, dtype):
    """The one-launch streaming kernel (persistent CTAs, flag-published partial sums, device-side launch generation): many
    items per CTA, samples whose slabs straddle rounds, repeated launches and a captured graph replayed several times must all give
    the same bits, and match fp32 GroupNorm.  (Opt-in through dadd_groupnorm_select(1): the cluster kernel is still the faster one.)"""
    ops = _ops()
    from progressive_stable_diffusion_b200 import _lib
    prev = _lib.load().dadd_groupnorm_select(1)
    try:
        _streaming_case(ops, b, c, hw, dtype)
    finally:
        _lib.load().dadd_groupnorm_select(prev)


def _streaming_case(ops, b, c, hw, dtype):
    g = torch.Generator().manual_seed(b + c + hw)
    x = (torch.randn(b, c, hw, hw, generator=g) * 1.7 - 0.9).to(dtype).to(DEV).contiguous(memory_format=torch.channels_last)
    gamma, beta = (1 + 0.2 * torch.randn(c, generator=g)).to(DEV), (0.2 * torch.randn(c, generator=g)).to(DEV)
    add = torch.randn(b, c, generator=g).to(DEV)
    ys = [ops.group_norm(x, gamma, beta, 32, 1e-5, True, add) for _ in range(3)]
    assert torch.equal(ys[0], ys[1]) and torch.equal(ys[0], ys[2])
    out = torch.empty_like(x)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        ops.group_norm(x, gamma, beta, 32, 1e-5, True, add, out=out)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=st):
            ops.group_norm(x, gamma, beta, 32, 1e-5, True, add, out=out)
            ops.group_norm(x, gamma, beta, 32, 1e-5, True, add, out=out)
        for _ in range(3):
            out.zero_()
            graph.replay()
            torch.cuda.synchronize()
            assert torch.equal(out, ys[0])
    sel = slice(0, min(b, 4))
    ref = F.silu(F.group_norm(x[sel].float().cpu() + add[sel].cpu()[:, :, None, None], 32, gamma.cpu(), beta.cpu(), 1e-5))
    ulp = 2.0 ** -7 if dtype == torch.bfloat16 else 2.0 ** -10
    assert (ys[0][sel].float().cpu() - ref).abs().max().item() <= ulp * max(1.0, ref.abs().max().item())



@pytest.mark.parametrize("c1,c2,hw,b", [(1280, 640, 8, 9), (640, 320, 32, 26), (320, 320, 32, 3)])
def test_groupnorm_streaming_kernel_two_sources(c1, c2, hw, b):
    """Streaming kernel on [x1 | x2]: bit-equal to the same kernel on the materialised concatenation, and within an fp16 ulp of fp32."""
    ops = _ops()
    from progressive_stable_diffusion_b200 import _lib
    g = torch.Generator().manual_seed(c1 + c2 + hw)
    x1 = (torch.randn(b, c1, hw, hw, generator=g) * 1.5 + 0.7).half().to(DEV).contiguous(memory_format=torch.channels_last)
    x2 = (torch.randn(b, c2, hw, hw, generator=g) * 0.6 - 0.4).half().to(DEV).contiguous(memory_format=torch.channels_last)
    c = c1 + c2
    gamma, beta = (1 + 0.2 * torch.randn(c, generator=g)).to(DEV), (0.2 * torch.randn(c, generator=g)).to(DEV)
    add = torch.randn(b, c, generator=g).to(DEV)
    cat = torch.cat([x1, x2], dim=1).contiguous(memory_format=torch.channels_last)
    prev = _lib.load().dadd_groupnorm_select(1)
    try:
        want = ops.group_norm(cat, gamma, beta, 32, 1e-5, True, add)
        got = ops.group_norm_cat(x1, x2, gamma, beta, 32, 1e-5, True, add)
    finally:
        _lib.load().dadd_groupnorm_select(prev)
    assert torch.equal(got, want)
    ref = F.silu(F.group_norm(cat.float().cpu() + add.cpu()[:, :, None, None], 32, gamma.cpu(), beta.cpu(), 1e-5))
    assert (got.float().cpu() - ref).abs().max().item() <= 2.0 ** -10 * max(1.0, ref.abs().max().item())


# ------------------------------------------------------------------------------------------------ LayerNorm / GEGLU
@pytest.mark.parametrize("rows", [1, 7, 1024 * 3 + 5])
@pytest.mark.parametrize("c", [320, 640, 1280, 768, 2048, 8])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32])
def test_add_layernorm(rows, c, dtype):
    """Residual add fused with the LayerNorm that consumes it: the sum is rounded to the tensor dtype first (what the
    unfused graph feeds LayerNorm), ragged row counts exercise the rows-per-warp tail."""
    ops = _ops()
    g = torch.Generator().manual_seed(c + rows)
    x = (torch.randn(rows, c, generator=g) * 2 + 0.5).to(dtype)
    r = torch.randn(rows, c, generator=g).to(dtype)
    gamma, beta = 1 + 0.1 * torch.randn(c, generator=g), 0.1 * torch.randn(c, generator=g)
    s_ref = (x.float() + r.float()).to(dtype)
    ref = F.layer_norm(s_ref.float(), (c,), gamma, beta, 1e-5)
    s, y = ops.add_layer_norm(x.to(DEV), r.to(DEV), gamma.to(DEV), beta.to(DEV), 1e-5)
    assert torch.equal(s.cpu(), s_ref)
    tol = {torch.bfloat16: 2.0 ** -7 * ref.abs().max().item(), torch.float16: 2.0 ** -10 * ref.abs().max().item(),
           torch.float32: 3e-5}[dtype]
    assert (y.float().cpu() - ref).abs().max().item() <= tol
    _, y2 = ops.add_layer_norm(x.to(DEV), r.to(DEV), gamma.to(DEV), beta.to(DEV), 1e-5, want_sum=False)
    assert torch.equal(y, y2)
    # sum_bias rides on the stored sum only: LayerNorm output unchanged, stored sum = x + r + bias rounded ONCE
    bias = torch.randn(c, generator=g)
    s3, y3 = ops.add_layer_norm(x.to(DEV), r.to(DEV), gamma.to(DEV), beta.to(DEV), 1e-5, sum_bias=bias.to(DEV))
    assert torch.equal(y3, y)
    assert torch.equal(s3.cpu(), ((x.float() + r.float()) + bias).to(dtype))


@pytest.mark.parametrize("shape", [(3, 320, 32, 32), (2, 1280, 4, 4), (26, 64, 640), (1, 1, 8), (5, 1031, 24)])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32])
def test_bias_residual(shape, dtype):
    ops = _ops()
    g = torch.Generator().manual_seed(sum(shape))
    a = torch.randn(*shape, generator=g).to(dtype)
    r = torch.randn(*shape, generator=g).to(dtype)
    c = shape[1] if len(shape) == 4 else shape[-1]
    bias = torch.randn(c, generator=g)
    bview = bias.view(1, -1, 1, 1) if len(shape) == 4 else bias
    ad, rd = a.to(DEV), r.to(DEV)
    if len(shape) == 4:
        ad, rd = ad.contiguous(memory_format=torch.channels_last), rd.contiguous(memory_format=torch.channels_last)
    for use_r, use_b in ((True, True), (True, False), (False, True)):
        ref = (a.float() + (r.float() if use_r else 0) + (bview if use_b else 0)).to(dtype)
        y = ops.bias_residual(ad, rd if use_r else None, bias.to(DEV) if use_b else None)
        assert y.stride() == ad.stride()
        assert torch.equal(y.cpu(), ref), (use_r, use_b)
    y = ops.bias_residual(ad.clone(), rd, bias.to(DEV), out=None)
    inplace = ad.clone()
    ops.bias_residual(inplace, rd, bias.to(DEV), out=inplace)
    assert torch.equal(inplace, y)


@pytest.mark.parametrize("c", [320, 640, 1280, 768])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32])
def test_layernorm(c, dtype):
    ops = _ops()
    g = torch.Generator().manual_seed(c)
    x = (torch.randn(3, 77, c, generator=g) * 2 + 0.5).to(dtype)
    gamma, beta = 1 + 0.1 * torch.randn(c, generator=g), 0.1 * torch.randn(c, generator=g)
    ref = F.layer_norm(x.float(), (c,), gamma, beta, 1e-5)
    y = ops.layer_norm(x.to(DEV), gamma.to(DEV), beta.to(DEV), 1e-5)
    tol = {torch.bfloat16: 2.0 ** -7 * ref.abs().max().item(), torch.float16: 2.0 ** -10 * ref.abs().max().item(),
           torch.float32: 2e-5}[dtype]
    assert (y.float().cpu() - ref).abs().max().item() <= tol


@pytest.mark.parametrize("inner", [1280, 2560, 5120])
def test_geglu(inner):
    ops = _ops()
    g = torch.Generator().manual_seed(inner)
    x = (torch.randn(2, 50, 2 * inner, generator=g) * 2).to(torch.bfloat16)
    a, gate = x.float().chunk(2, dim=-1)
    ref = a * F.gelu(gate)
    y = ops.geglu(x.to(DEV))
    assert (y.float().cpu() - ref).abs().max().item() <= 2.0 ** -7 * ref.abs().max().item()


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("m,k,inner", [(1024 * 3, 320, 1280), (256 * 5, 640, 2560), (64 * 7 + 5, 1280, 5120), (16, 1280, 5120),
                                        (1024 * 40, 320, 1280), (300, 72, 128)])
def test_ff_geglu_gemm_vs_fp32(m, k, inner, dtype):
    """Fused projection + GEGLU vs fp32 `h * gelu_erf(g)` on the same 16-bit operands (ragged M, K not a multiple of 64,
    many tiles per persistent CTA), and vs the unfused library GEMM + dadd_geglu_fwd path it replaces."""
    ops = _ops()
    g = torch.Generator().manual_seed(m + k + inner)
    x = torch.randn(m, k, generator=g).to(dtype)
    w = (torch.randn(2 * inner, k, generator=g) * (1.5 / math.sqrt(k))).to(dtype)
    bias = 0.3 * torch.randn(2 * inner, generator=g)
    rows = slice(0, m) if m <= 4096 else slice(m - 2048, m)            # the fp32 reference of the big case: its last rows
    proj = F.linear(x[rows].float(), w.float(), bias)
    ref = proj[:, :inner] * F.gelu(proj[:, inner:])
    got = ops.ff_geglu(x.to(DEV), w.to(DEV), bias.to(DEV))
    assert got.shape == (m, inner) and got.dtype == dtype
    tol = 6e-3 if dtype == torch.bfloat16 else 1e-3
    assert rel_err(got[rows], ref) <= tol, rel_err(got[rows], ref)
    unfused = ops.geglu(F.linear(x.to(DEV), w.to(DEV), bias.to(DEV).to(dtype)))
    assert rel_err(got, unfused.float()) <= 2 * tol


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("m,n,k", [(1024 * 3, 320, 320), (256 * 5, 640, 640), (64 * 7 + 5, 1280, 1280), (16, 1280, 1280),
                                    (1024 * 40, 960, 320), (2048, 320, 1280), (300, 192, 72), (500, 64, 136), (1664, 3840, 1280), (777, 1920, 640),
                                    (129, 512, 512)])
def test_linear_gemm_bias_residual_vs_fp32(m, n, k, dtype):
    """dadd_linear_fwd (both tile widths, ragged M, K not a multiple of 64, many tiles per CTA) with every bias / residual
    combination vs fp32 on the same 16-bit operands; the residual may alias the output."""
    ops = _ops()
    g = torch.Generator().manual_seed(m + n + k)
    x = torch.randn(m, k, generator=g).to(dtype)
    w = (torch.randn(n, k, generator=g) * (1.5 / math.sqrt(k))).to(dtype)
    bias = 0.3 * torch.randn(n, generator=g)
    res = torch.randn(m, n, generator=g).to(dtype)
    rows = slice(0, m) if m <= 4096 else slice(m - 2048, m)
    base = F.linear(x[rows].float(), w.float())
    xd, wd, bd, rd = x.to(DEV), w.to(DEV), bias.to(DEV), res.to(DEV)
    tol = 6e-3 if dtype == torch.bfloat16 else 1e-3
    for use_bias, use_res in ((False, False), (True, False), (False, True), (True, True)):
        ref = base + (bias if use_bias else 0) + (res[rows].float() if use_res else 0)
        got = ops.linear(xd, wd, bd if use_bias else None, rd if use_res else None, impl="tc")
        assert got.shape == (m, n) and got.dtype == dtype
        lib = ops.linear(xd, wd, bd if use_bias else None, rd if use_res else None, impl="lib")
        assert rel_err(lib[rows], ref) <= tol
        assert rel_err(got[rows], ref) <= tol, (use_bias, use_res, rel_err(got[rows], ref))
    inplace = rd.clone()
    ops.linear(xd, wd, bd, inplace, out=inplace, impl="tc")
    assert torch.equal(inplace, got)


def test_linear_library_path_for_other_widths():
    ops = _ops()
    g = torch.Generator().manual_seed(9)
    x, w = torch.randn(100, 64, generator=g).to(torch.bfloat16), torch.randn(24, 64, generator=g).to(torch.bfloat16)
    bias, res = torch.randn(24, generator=g), torch.randn(100, 24, generator=g).to(torch.bfloat16)
    got = ops.linear(x.to(DEV), w.to(DEV), bias.to(DEV), res.to(DEV))
    ref = F.linear(x.float(), w.float(), bias) + res.float()
    assert rel_err(got, ref) <= 1e-2
    from progressive_stable_diffusion_b200._lib import DaddError
    with pytest.raises(DaddError):
        ops.linear(x.to(DEV), w.to(DEV), bias.to(DEV), res.to(DEV), impl="tc")


# ------------------------------------------------------------------------------------------------ attention cores
SELF_SHAPES = [(1024, 40, 2), (256, 80, 2), (64, 160, 3), (16, 160, 2), (100, 40, 1), (4096, 40, 1), (200, 64, 1),
               (130, 128, 1), (256, 160, 2), (1024, 80, 1), (128, 40, 3), (384, 72, 1),
               # ragged key / query tiles (900, 1000, 300), d % 64 == 0 (no spare column for the tensor-core row sums), d = 96 / 120
               (512, 40, 3), (512, 80, 2), (900, 40, 2), (1000, 64, 1), (2048, 40, 1), (300, 128, 1), (200, 96, 2), (640, 120, 1)]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("impl", ["mma", "tc"])
@pytest.mark.parametrize("n,d,b", SELF_SHAPES)
def test_self_attention_core(n, d, b, impl, dtype):
    """Both self-attention kernels (warp-level mma.sync; tcgen05/TMEM/TMA) against fp32 SDPA on the same 16-bit inputs."""
    ops = _ops()
    if impl == "tc" and n < 128:
        pytest.skip("the tcgen05 kernel takes N >= 128 (shorter sequences are one mma.sync tile)")
    h = 8
    g = torch.Generator().manual_seed(n + d)
    qkv = (torch.randn(b, n, 3 * h * d, generator=g) * 1.2).to(dtype)
    c = h * d
    q, k, v = (qkv[..., i * c:(i + 1) * c].float().view(b, n, h, d).transpose(1, 2) for i in range(3))
    ref = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(b, n, c)
    qd = qkv.to(DEV)
    o = ops.self_attention(qd[..., :c], qd[..., c:2 * c], qd[..., 2 * c:], h, impl=impl)
    torch.cuda.synchronize()
    tol = 1.5e-2 if dtype == torch.bfloat16 else 3e-3
    assert rel_err(o, ref) <= tol, rel_err(o, ref)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("n,d,h,b", [(1024, 512, 1, 2), (1000, 512, 1, 1), (77, 512, 1, 3), (256, 256, 2, 2), (4096, 512, 1, 1)])
def test_self_attention_wide_heads(n, d, h, b, dtype):
    """d = 256 / 512 (the VAE mid block's single head): the column-split mma.sync kernel against fp32 SDPA, ragged N included,
    q / k / v as strided views of one fused buffer and growing row maxima along the keys."""
    ops = _ops()
    g = torch.Generator().manual_seed(n + d)
    c = h * d
    qkv = (torch.randn(b, n, 3 * c, generator=g) * 0.35).to(dtype)
    qkv[..., c:2 * c] *= torch.linspace(0.5, 2.0, n)[None, :, None].to(dtype)       # later keys score higher: rescales on most tiles
    q, k, v = (qkv[..., i * c:(i + 1) * c].float().view(b, n, h, d).transpose(1, 2) for i in range(3))
    ref = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(b, n, c)
    qd = qkv.to(DEV)
    o = ops.self_attention(qd[..., :c], qd[..., c:2 * c], qd[..., 2 * c:], h)
    torch.cuda.synchronize()
    tol = 1.5e-2 if dtype == torch.bfloat16 else 3e-3
    assert rel_err(o, ref) <= tol, rel_err(o, ref)


@pytest.mark.parametrize("n,d,b", [(1024, 40, 26), (640, 80, 20), (256, 64, 40), (256, 80, 40), (256, 160, 24), (128, 40, 60)])
def test_self_attention_persistent_many_items_and_growing_maxima(n, d, b):
    """More work items than SMs (every persistent CTA walks several), and scores whose row maxima keep growing along the
    key axis by far more than 2^8 so the lazy O-rescale path runs on most key tiles."""
    ops = _ops()
    h = 8
    c = h * d
    g = torch.Generator().manual_seed(n * d + b)
    qkv = torch.randn(b, n, 3 * c, generator=g)
    ramp = torch.linspace(0.0, 6.0, n)[None, :, None]                  # |k| grows with the key index
    qkv[..., c:2 * c] *= (0.3 + ramp)
    qkv[..., :c] *= 1.5
    qkv = qkv.to(torch.bfloat16)
    q, k, v = (qkv[..., i * c:(i + 1) * c].float().view(b, n, h, d).transpose(1, 2) for i in range(3))
    ref = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(b, n, c)
    qd = qkv.to(DEV)
    o = ops.self_attention(qd[..., :c], qd[..., c:2 * c], qd[..., 2 * c:], h, impl="tc")
    torch.cuda.synchronize()
    assert rel_err(o, ref) <= 1.5e-2, rel_err(o, ref)


def test_self_attention_dispatch_uses_both_kernels():
    ops = _ops()
    from progressive_stable_diffusion_b200 import _lib
    g = torch.Generator().manual_seed(0)
    for n in (64, 256):
        qkv = torch.randn(1, n, 3 * 320, generator=g).to(torch.bfloat16).to(DEV)
        a = ops.self_attention(qkv[..., :320], qkv[..., 320:640], qkv[..., 640:], 8)
        b = ops.self_attention(qkv[..., :320], qkv[..., 320:640], qkv[..., 640:], 8, impl="mma")
        assert rel_err(a, b.float()) < 1e-2
    assert _lib.launch_count() > 0


@pytest.fixture(params=[torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
def compute(request):
    import progressive_stable_diffusion_b200 as P
    P.set_compute_dtype(request.param)
    yield request.param
    P.set_compute_dtype(P.DEFAULT_COMPUTE_DTYPE)


@pytest.mark.parametrize("case", cases.PROCESSOR_CASES, ids=lambda c: c["name"])
def test_cross_attention_processors_vs_reference_golden(case, compute):
    """Product processor (fused kernel, 16-bit operands) vs the VERBATIM reference processor's fp32 output."""
    import progressive_stable_diffusion_b200 as P
    from progressive_stable_diffusion_b200.unet2d import Attention
    w, x, ehs = cases.processor_inputs(case)
    c = case["c"]
    attn = Attention(c, 768, 8, c // 8)
    if case["kind"] == "split":
        proc = P.SplitInjectionAttentionProcessor(c, 768, 16, 16, 16, "both", case["gates"][0], case["gates"][1],
                                                  case["delta_scale"])
    else:
        proc = P.OrdinalIPAttnProcessor2_0(c, 768, 16, 16, case["mode"])
    attn.set_processor(proc)
    attn.load_state_dict(w)
    attn.to(DEV)
    with torch.no_grad():
        out = attn(x.to(DEV), encoder_hidden_states=ehs.to(DEV))
    assert out.dtype == torch.float32
    got, ref = GOLD.pair("processor_" + case["name"], out)
    assert rel_err(got, ref) <= (2e-2 if compute == torch.bfloat16 else 4e-3), rel_err(got, ref)


def _cross_ref(q, k, v, gates, heads, seg, nseg):
    """fp32: sum_s gates[s] softmax(q k_s^T / sqrt d) v_s on the 16-bit operands the kernels see."""
    b, n, c = q.shape
    d = c // heads
    qh = q.float().view(b, n, heads, d).transpose(1, 2)
    out = torch.zeros(b, heads, n, d)
    for s in range(nseg):
        ks, vs = k.float()[:, :, s * seg:(s + 1) * seg], v.float()[:, :, s * seg:(s + 1) * seg]
        out += gates[s] * torch.softmax(qh @ ks.transpose(-1, -2) * d ** -0.5, dim=-1) @ vs
    return out.transpose(1, 2).reshape(b, n, c)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("seg,nseg", [(16, 3), (16, 2), (32, 1)])
@pytest.mark.parametrize("n,d,b", [(1024, 40, 3), (256, 80, 5), (128, 64, 2), (200, 40, 2), (4096, 40, 1), (333, 128, 1), (1024, 40, 40),
                                   (1024, 40, 80), (640, 64, 90)])      # >= 2 (sample, head) groups per CTA: the group-walk order
def test_cross_attention_core_tcgen05_vs_mma_vs_fp32(n, d, b, seg, nseg, dtype):
    """The tcgen05 kernel (N >= 128), the mma.sync kernel and the fp32 reference on the same 16-bit operands; q is a strided
    view (row stride 2C) as when it aliases a fused projection, and b = 40 gives every persistent CTA several items."""
    ops = _ops()
    heads, c = 8, 8 * d
    g = torch.Generator().manual_seed(n + d + b + seg * nseg)
    q = (1.5 * torch.randn(b, n, 2 * c, generator=g)).to(dtype)[:, :, c // 8: c // 8 + c]
    k = (1.2 * torch.randn(b, heads, seg * nseg, d, generator=g)).to(dtype)
    v = torch.randn(b, heads, seg * nseg, d, generator=g).to(dtype)
    gates = torch.tensor([0.9, 0.1, 3.0][:nseg])
    ref = _cross_ref(q, k, v, gates, heads, seg, nseg)
    qd = torch.empty(b, n, 2 * c, dtype=dtype, device=DEV)[:, :, c // 8: c // 8 + c]
    qd.copy_(q)
    assert not qd.is_contiguous()
    tc = ops.cross_attention(qd, k.to(DEV), v.to(DEV), gates.to(DEV), heads, seg, nseg, impl="tc")
    mma = ops.cross_attention(qd, k.to(DEV), v.to(DEV), gates.to(DEV), heads, seg, nseg, impl="mma")
    auto = ops.cross_attention(qd, k.to(DEV), v.to(DEV), gates.to(DEV), heads, seg, nseg)
    tol = 1.2e-2 if dtype == torch.bfloat16 else 2e-3
    assert rel_err(tc, ref) <= tol, rel_err(tc, ref)
    assert rel_err(mma, ref) <= tol, rel_err(mma, ref)
    assert torch.equal(auto, tc)                         # N >= 128, d <= 128 dispatches to the tcgen05 kernel, deterministically


def test_cross_attention_tcgen05_rejects_unsupported_shapes():
    ops = _ops()
    from progressive_stable_diffusion_b200._lib import DaddError
    q = torch.zeros(1, 64, 320, dtype=torch.bfloat16, device=DEV)
    kv = torch.zeros(1, 8, 48, 40, dtype=torch.bfloat16, device=DEV)
    with pytest.raises(DaddError):
        ops.cross_attention(q, kv, kv, torch.ones(3, device=DEV), 8, 16, 3, impl="tc")      # N < 128


def test_cross_attention_delta_zero_skips_pathway():
    """I2: delta_scale == 0 must equal a 2-segment launch regardless of what the delta tokens hold (even NaN)."""
    import progressive_stable_diffusion_b200 as P
    from progressive_stable_diffusion_b200.unet2d import Attention
    case = cases.PROCESSOR_CASES[1]
    w, x, ehs = cases.processor_inputs(case)
    attn = Attention(320, 768, 8, 40)
    proc = P.SplitInjectionAttentionProcessor(320, 768, delta_scale=0.0, anat_gate_init=0.1, dis_gate_init=0.9)
    attn.set_processor(proc)
    attn.load_state_dict(w)
    attn.to(DEV)
    ehs_nan = ehs.clone()
    ehs_nan[:, -16:] = float("nan")
    with torch.no_grad():
        a = attn(x.to(DEV), encoder_hidden_states=ehs.to(DEV))
        b = attn(x.to(DEV), encoder_hidden_states=ehs_nan.to(DEV))
    assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ conditioning front end
def test_purifier_matches_reference_golden():
    import progressive_stable_diffusion_b200 as P
    w, img, aoe = cases.purifier_inputs()
    pur = P.FeaturePurifier(768, 8, 2)
    pur.load_state_dict(w)
    pur.to(DEV)
    with torch.no_grad():
        out = pur(img.to(DEV), aoe.to(DEV))
    torch.testing.assert_close(*GOLD.pair("purifier", out), atol=2e-4, rtol=1e-4)


def test_aoe_matches_reference_golden():
    import progressive_stable_diffusion_b200 as P
    w, labels, src = cases.aoe_inputs()
    emb = P.AdditiveOrdinalEmbedder(4, 768, delta_scale=0.05, num_tokens=16)
    emb.load_state_dict(w)
    emb.to(DEV)
    with torch.no_grad():
        torch.testing.assert_close(*GOLD.pair("aoe_forward", emb(labels.to(DEV))), atol=2e-5, rtol=1e-4)
        torch.testing.assert_close(*GOLD.pair("aoe_negative", emb.get_negative_embedding(labels.to(DEV))), atol=2e-5, rtol=1e-4)
        torch.testing.assert_close(*GOLD.pair("aoe_delta", emb.get_ordinal_delta_embedding(src.to(DEV), labels.to(DEV))),
                                   atol=4e-5, rtol=1e-4)
        same = emb.get_ordinal_delta_embedding(labels.to(DEV), labels.to(DEV))
        assert same.abs().max().item() == 0.0                                           # invariant I1
        # interpolation itself: table + gather + lerp, vs the oracle restatement
        interp = emb._interp(labels.to(DEV)).cpu()
        torch.testing.assert_close(interp, conditioning.aoe_interp(w, labels), atol=1e-7, rtol=1e-6)


@pytest.mark.parametrize("shape", [(3, 1280, 4, 4), (2, 640, 16, 16), (5, 128, 7, 9), (1, 8, 1, 1)])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32])
def test_upsample_nearest2x_bit_exact(shape, dtype):
    ops = _ops()
    x = torch.randn(*shape, generator=torch.Generator().manual_seed(sum(shape))).to(dtype)
    want = F.interpolate(x.float(), scale_factor=2.0, mode="nearest").to(dtype)
    got = ops.upsample_nearest2x(x.to(DEV).contiguous(memory_format=torch.channels_last))
    assert got.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(got.cpu(), want)


# ------------------------------------------------------------------------------------------------ CLIP + resampler front end
FE = Golden(os.path.join(os.path.dirname(__file__), "golden", "front_end.npz"))


def test_quick_gelu():
    ops = _ops()
    x = torch.randn(3, 257, 4096, generator=torch.Generator().manual_seed(2)) * 3
    for dtype, tol in ((torch.float32, 2e-6), (torch.bfloat16, 2.0 ** -7), (torch.float16, 2.0 ** -10)):
        xd = x.to(dtype)
        ref = xd.float() * torch.sigmoid(1.702 * xd.float())
        got = ops.quick_gelu_(xd.to(DEV).clone())
        assert (got.float().cpu() - ref).abs().max().item() <= tol * max(1.0, ref.abs().max().item())


def test_clip_tower_vs_transformers_golden(compute):
    """ImageEncoder (ViT-L/14, B200 kernels, 16-bit) vs the REAL transformers CLIPVisionModelWithProjection (fp32) on the
    same seeded weights and pixels: last hidden states (what the resampler consumes) and the projected embedding."""
    import progressive_stable_diffusion_b200 as P
    d, w, pixels = cases.clip_inputs("l14")
    enc = P.ImageEncoder("openai/clip-vit-large-patch14")
    enc.image_encoder.load_state_dict(w, strict=True)
    enc.to(DEV)
    hidden = enc.get_hidden_states(pixels.to(DEV))
    embeds = enc(pixels.to(DEV))
    assert hidden.shape == (2, 257, 1024) and embeds.shape == (2, 768)
    eh, ee = rel_err(*FE.pair("clip_l14_hidden", hidden)), rel_err(embeds, torch.from_numpy(FE["clip_l14_embeds"]))
    print(f"CLIP ViT-L/14 {compute}: hidden rel err {eh:.4g}, embeds rel err {ee:.4g}")
    tol = 3e-2 if compute == torch.bfloat16 else 5e-3
    assert eh <= tol and ee <= tol, (eh, ee)


def test_image_projections_vs_reference_golden():
    import progressive_stable_diffusion_b200 as P
    plus = P.ImageProjectionPlus(clip_hidden_dim=1024, cross_attention_dim=768, num_tokens=16, num_heads=8, depth=2)
    plus.load_state_dict(cases.projection_plus_inputs(), strict=True)
    plus.to(DEV)
    with torch.no_grad():
        got = plus(cases.clip_l14_hidden().to(DEV))
    torch.testing.assert_close(*FE.pair("projection_plus", got), atol=2e-3, rtol=1e-3)
    bw, emb = cases.projection_basic_inputs()
    basic = P.ImageProjection(clip_embedding_dim=768, cross_attention_dim=768, num_tokens=4)
    basic.load_state_dict(bw, strict=True)
    basic.to(DEV)
    with torch.no_grad():
        torch.testing.assert_close(*FE.pair("projection_basic", basic(emb.to(DEV))), atol=2e-3, rtol=1e-3)


def test_module_front_end_from_pixels(compute):
    """_get_image_embeds on CLIP-preprocessed pixels (the reference's call, diffusion_module_ip.py:315-332) vs golden tokens."""
    import progressive_stable_diffusion_b200 as P
    _, w, pixels = cases.clip_inputs("l14")
    module = P.DiffusionModuleWithIP(P.default_config(), build_vae=False, build_image_encoder=True)
    module.image_encoder.image_encoder.load_state_dict(w, strict=True)
    module.image_projection.load_state_dict(cases.projection_plus_inputs(), strict=True)
    assert any(k.startswith("image_encoder.image_encoder.vision_model.encoder.layers.23.mlp.fc2") for k in module.state_dict())
    module.to(DEV).eval()
    with torch.no_grad():
        tokens = module._get_image_embeds(pixels.to(DEV))
        assert torch.equal(module._get_image_embeds(tokens), tokens)          # projected tokens pass through
    e = rel_err(*FE.pair("projection_plus", tokens))
    print(f"front end pixels -> tokens {compute}: rel err {e:.4g}")
    assert e <= (3e-2 if compute == torch.bfloat16 else 5e-3), e
    bare = P.DiffusionModuleWithIP(P.default_config(), build_vae=False)
    with pytest.raises(RuntimeError):
        bare._get_image_embeds(pixels)


def test_image_post():
    ops = _ops()
    x = torch.linspace(-2, 2, 1001)
    ref = ((x.clamp(-1, 1) + 1) / 2).clamp(0, 1)
    assert torch.equal(ops.image_post(x.to(DEV)).cpu(), ref)


def test_cpu_tensors_are_rejected():
    ops = _ops()
    from progressive_stable_diffusion_b200._lib import DaddError
    with pytest.raises(DaddError):
        ops.layer_norm(torch.zeros(2, 320), torch.ones(320), torch.zeros(320))
