"""Tensor-level wrappers over the C ABI (``include/dadd_b200.h``).

PyTorch is used for device memory and streams only: every function below hands raw ``data_ptr()``s and the current
CUDA stream to ``libdadd_b200.so``.  All of them are CUDA-graph capturable (nothing synchronises) and none has a CPU or
eager fallback: CPU tensors raise.
"""

from __future__ import annotations

from typing import Optional

import torch

from . import _lib

F32, BF16, F16 = 0, 1, 2
NCHW, NHWC = 0, 1


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    if t.dtype == torch.float16:
        return F16
    raise TypeError(f"dadd kernels take float32, bfloat16 or float16 tensors, got {t.dtype}")


def _cuda(*ts: Optional[torch.Tensor]) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.DaddError("dadd kernels run on CUDA tensors only (there is no CPU fallback)")


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


# --------------------------------------------------------------------------------------------- DDIM
def ddim_step_(x: torch.Tensor, eps_cond: torch.Tensor, eps_uncond: Optional[torch.Tensor], guidance: float,
               sqrt_ab_t: float, sqrt_1mab_t: float, sqrt_ab_prev: float, eps_coef: float, sigma: float = 0.0,
               noise: Optional[torch.Tensor] = None, clamp: float = 4.0, is_last: bool = False) -> torch.Tensor:
    """In-place fused CFG + x0 + clamp + DDIM update (inference_pipeline_ip.py:427-468)."""
    _cuda(x, eps_cond, eps_uncond, noise)
    assert x.dtype == torch.float32 and x.is_contiguous() and eps_cond.is_contiguous()
    assert eps_cond.numel() == x.numel() and (eps_uncond is None or (eps_uncond.is_contiguous() and eps_uncond.dtype == eps_cond.dtype))
    assert noise is None or (noise.dtype == torch.float32 and noise.is_contiguous() and noise.numel() == x.numel())
    _lib.check(_lib.load().dadd_ddim_step(x.data_ptr(), eps_cond.data_ptr(), _ptr(eps_uncond), _dt(eps_cond), guidance,
                                          sqrt_ab_t, sqrt_1mab_t, sqrt_ab_prev, eps_coef, sigma, _ptr(noise), clamp,
                                          int(is_last), x.numel(), _stream()), "dadd_ddim_step")
    return x


def ddim_step_table_(x: torch.Tensor, eps_cond: torch.Tensor, eps_uncond: Optional[torch.Tensor], guidance: float,
                     coef_table: torch.Tensor, step_state: torch.Tensor, noise: Optional[torch.Tensor] = None,
                     clamp: float = 4.0) -> torch.Tensor:
    _cuda(x, eps_cond, eps_uncond, coef_table, step_state, noise)
    assert x.dtype == torch.float32 and x.is_contiguous() and eps_cond.is_contiguous()
    assert coef_table.dtype == torch.float32 and coef_table.dim() == 2 and coef_table.shape[-1] == 8 and coef_table.is_contiguous()
    assert step_state.dtype == torch.int32 and step_state.numel() == 2
    assert eps_cond.numel() == x.numel() and (eps_uncond is None or (eps_uncond.is_contiguous() and eps_uncond.dtype == eps_cond.dtype
                                                                     and eps_uncond.numel() == x.numel()))
    n_steps = coef_table.shape[0]
    assert noise is None or (noise.dtype == torch.float32 and noise.is_contiguous() and noise.numel() == n_steps * x.numel())
    _lib.check(_lib.load().dadd_ddim_step_table(x.data_ptr(), eps_cond.data_ptr(), _ptr(eps_uncond), _dt(eps_cond),
                                                guidance, coef_table.data_ptr(), step_state.data_ptr(), n_steps, _ptr(noise),
                                                clamp, x.numel(), _stream()), "dadd_ddim_step_table")
    return x


def step_begin_(step_state: torch.Tensor, table: Optional[torch.Tensor] = None, row_out: Optional[torch.Tensor] = None,
                n_steps: Optional[int] = None) -> None:
    """Advance the device-side step counter and stage row ``step`` of ``table`` (n_steps, row) into ``row_out``."""
    _cuda(step_state, table, row_out)
    row_bytes = 0
    if table is not None:
        assert table.dim() == 2 and table.is_contiguous() and row_out.is_contiguous() and table.dtype == row_out.dtype
        row_bytes = row_out.numel() * row_out.element_size()
        assert table[0].numel() == row_out.numel()
        assert n_steps is None or n_steps == table.shape[0]
        n_steps = table.shape[0]
    _lib.check(_lib.load().dadd_step_begin(step_state.data_ptr(), _ptr(table), _ptr(row_out), row_bytes,
                                           1 if n_steps is None else int(n_steps), _stream()), "dadd_step_begin")


# --------------------------------------------------------------------------------------------- norms
def group_norm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, num_groups: int, eps: float, silu: bool,
               chan_add: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GroupNorm(+SiLU) of a 4-D ``(B, C, H, W)`` tensor, either contiguous (NCHW) or channels_last (NHWC) in memory.
    ``chan_add`` (B, C) fp32 is added to x before the statistics (the resnet time-embedding term)."""
    _cuda(x, gamma, beta, chan_add)
    assert x.dim() == 4
    b, c, h, w = x.shape
    if x.is_contiguous():            # (when C == 1 or H*W == 1 both layouts describe the same bytes)
        layout = NCHW
    elif x.is_contiguous(memory_format=torch.channels_last):
        layout = NHWC
    else:
        raise ValueError("group_norm needs a contiguous or channels_last tensor")
    assert gamma.dtype == torch.float32 and beta.dtype == torch.float32
    if chan_add is not None:
        assert chan_add.dtype == torch.float32 and chan_add.shape == (b, c) and chan_add.stride(1) == 1
    y = torch.empty_like(x) if out is None else out
    assert y.stride() == x.stride()
    lib = _lib.load()
    ws, ws_bytes = None, 0
    if layout == NHWC:      # the two-pass NHWC kernels keep their chunk partials in a caller-owned scratch buffer
        ws_bytes = int(lib.dadd_groupnorm_workspace_bytes(b, c, h * w, num_groups, layout))
        ws = torch.empty(max(ws_bytes, 8), dtype=torch.uint8, device=x.device)
    _lib.check(lib.dadd_groupnorm_fwd(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), _ptr(chan_add),
                                      0 if chan_add is None else chan_add.stride(0), y.data_ptr(), b, c, h * w, num_groups, eps,
                                      int(silu), layout, _dt(x), _ptr(ws), ws_bytes, _stream()), "dadd_groupnorm_fwd")
    return y


def group_norm_cat_supported(x1: torch.Tensor, x2: torch.Tensor, num_groups: int) -> bool:
    b, c1, h, w = x1.shape
    return (x1.dtype in (torch.bfloat16, torch.float16) and x1.is_contiguous(memory_format=torch.channels_last)
            and x2.is_contiguous(memory_format=torch.channels_last)
            and bool(_lib.load().dadd_groupnorm_cat_supported(b, c1, x2.shape[1], h * w, num_groups, _dt(x1))))


def group_norm_cat(x1: torch.Tensor, x2: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, num_groups: int, eps: float,
                   silu: bool, chan_add: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GroupNorm(+SiLU) of ``torch.cat([x1, x2], dim=1)`` without materialising the concatenation (channels_last, 16-bit)."""
    _cuda(x1, x2, gamma, beta, chan_add)
    b, c1, h, w = x1.shape
    c2 = x2.shape[1]
    assert x2.shape == (b, c2, h, w) and x1.dtype == x2.dtype
    assert x1.is_contiguous(memory_format=torch.channels_last) and x2.is_contiguous(memory_format=torch.channels_last)
    assert gamma.dtype == torch.float32 and beta.dtype == torch.float32 and gamma.numel() == c1 + c2
    if chan_add is not None:
        assert chan_add.dtype == torch.float32 and chan_add.shape == (b, c1 + c2) and chan_add.stride(1) == 1
    y = torch.empty((b, c1 + c2, h, w), dtype=x1.dtype, device=x1.device, memory_format=torch.channels_last)
    lib = _lib.load()
    ws_bytes = int(lib.dadd_groupnorm_workspace_bytes(b, c1 + c2, h * w, num_groups, NHWC))
    ws = torch.empty(max(ws_bytes, 8), dtype=torch.uint8, device=x1.device)
    _lib.check(lib.dadd_groupnorm_cat_fwd(x1.data_ptr(), c1, x2.data_ptr(), c2, gamma.data_ptr(), beta.data_ptr(),
                                          _ptr(chan_add), 0 if chan_add is None else chan_add.stride(0), y.data_ptr(),
                                          b, h * w, num_groups, eps, int(silu), _dt(x1), ws.data_ptr(), ws_bytes, _stream()),
               "dadd_groupnorm_cat_fwd")
    return y


def upsample_nearest2x(x: torch.Tensor) -> torch.Tensor:
    """``F.interpolate(x, scale_factor=2.0, mode="nearest")`` for a channels_last ``(B, C, H, W)`` tensor."""
    _cuda(x)
    b, c, h, w = x.shape
    assert x.is_contiguous(memory_format=torch.channels_last)
    y = torch.empty((b, c, 2 * h, 2 * w), dtype=x.dtype, device=x.device, memory_format=torch.channels_last)
    _lib.check(_lib.load().dadd_upsample_nearest2x_fwd(x.data_ptr(), y.data_ptr(), b, h, w, c, _dt(x), _stream()),
               "dadd_upsample_nearest2x_fwd")
    return y


def layer_norm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    _cuda(x, gamma, beta)
    assert x.is_contiguous() and gamma.dtype == torch.float32 and beta.dtype == torch.float32
    c = x.shape[-1]
    y = torch.empty_like(x)
    _lib.check(_lib.load().dadd_layernorm_fwd(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(),
                                              x.numel() // c, c, eps, _dt(x), _stream()), "dadd_layernorm_fwd")
    return y


def add_layer_norm(x: torch.Tensor, r: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5,
                   want_sum: bool = True, sum_bias: Optional[torch.Tensor] = None):
    """``s = x + r`` (rounded to the tensor dtype) and ``LayerNorm(s)`` in one pass; returns ``(s or None, norm)``.
    ``sum_bias`` (C,) fp32 is added to the RETURNED sum only (LayerNorm sees ``x + r``): the bias of the output projection of
    the next residual branch, so that branch's ``proj(...) + s`` is one accumulating GEMM."""
    _cuda(x, r, gamma, beta, sum_bias)
    assert x.is_contiguous() and r.is_contiguous() and x.shape == r.shape and x.dtype == r.dtype
    assert gamma.dtype == torch.float32 and beta.dtype == torch.float32
    c = x.shape[-1]
    assert sum_bias is None or (want_sum and sum_bias.dtype == torch.float32 and sum_bias.numel() == c and sum_bias.is_contiguous())
    s = torch.empty_like(x) if want_sum else None
    y = torch.empty_like(x)
    _lib.check(_lib.load().dadd_add_layernorm_fwd(x.data_ptr(), r.data_ptr(), _ptr(s), _ptr(sum_bias), gamma.data_ptr(),
                                                  beta.data_ptr(), y.data_ptr(), x.numel() // c, c, eps, _dt(x), _stream()),
               "dadd_add_layernorm_fwd")
    return s, y


def bias_residual(a: torch.Tensor, res: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``a (+ res) (+ bias[c])`` with the channel dimension innermost in memory: ``a`` is either a channels_last 4-D
    activation ``(B, C, H, W)`` or a contiguous ``(..., C)`` token matrix; ``res`` must share its layout; bias is fp32."""
    _cuda(a, res, bias)
    assert res is not None or bias is not None
    if a.dim() == 4 and not a.is_contiguous():
        assert a.is_contiguous(memory_format=torch.channels_last)
        c = a.shape[1]
    else:
        assert a.is_contiguous()
        c = a.shape[-1] if a.dim() != 4 else a.shape[1] * a.shape[2] * a.shape[3] // max(1, a.shape[2] * a.shape[3])
        if a.dim() == 4:        # contiguous NCHW only describes channel-innermost memory when H*W == 1
            assert a.shape[2] * a.shape[3] == 1 or bias is None
    if res is not None:
        assert res.shape == a.shape and res.stride() == a.stride() and res.dtype == a.dtype
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == c and bias.is_contiguous()
    y = torch.empty_like(a) if out is None else out
    assert y.stride() == a.stride() and y.dtype == a.dtype
    _lib.check(_lib.load().dadd_bias_residual_fwd(a.data_ptr(), _ptr(res), _ptr(bias), y.data_ptr(), a.numel() // c, c,
                                                  _dt(a), _stream()), "dadd_bias_residual_fwd")
    return y


def geglu(x: torch.Tensor) -> torch.Tensor:
    """``a * gelu(gate)`` with ``[a | gate] = x.chunk(2, -1)`` (diffusers GEGLU, SURVEY.md A.5)."""
    _cuda(x)
    assert x.is_contiguous() and x.shape[-1] % 16 == 0
    inner = x.shape[-1] // 2
    y = torch.empty(*x.shape[:-1], inner, device=x.device, dtype=x.dtype)
    _lib.check(_lib.load().dadd_geglu_fwd(x.data_ptr(), y.data_ptr(), x.numel() // x.shape[-1], inner, _dt(x), _stream()),
               "dadd_geglu_fwd")
    return y


# Which GEMM ``linear(..., impl="auto")`` runs: "lib" = cuBLAS (+ one fused bias / residual pass), "tc" = dadd_linear_fwd where
# the shape qualifies.  Measured on B200: round 1's one-CTA kernel lost 10-25 % to cuBLAS (profiles/r01_linear_gemm.txt); round 2's
# CTA-pair (cta_group::2) kernel with a TMA-store epilogue is 4-17 % behind on the UNet's shapes and far behind at M < 2000
# (profiles/r02_linear_gemm.txt), so the default is still "lib".
LINEAR_IMPL = "lib"


def quick_gelu_(x: torch.Tensor) -> torch.Tensor:
    """In place ``x * sigmoid(1.702 x)`` (CLIP's activation)."""
    _cuda(x)
    assert x.is_contiguous() and x.numel() % 8 == 0
    _lib.check(_lib.load().dadd_quick_gelu_fwd(x.data_ptr(), x.data_ptr(), x.numel(), _dt(x), _stream()), "dadd_quick_gelu_fwd")
    return x


def linear(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
           out: Optional[torch.Tensor] = None, impl: str = "auto", bias_lp: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``F.linear(x, w, bias) (+ residual)``: x (..., K) 16-bit, w (N, K) same dtype, bias (N,) fp32, residual (..., N).
    ``impl``: "tc" = the tcgen05 GEMM with bias / residual in its epilogue (``dadd_linear_fwd``; K % 8 == 0, N % 64 == 0,
    dense operands), "lib" = library GEMM followed by the fused bias / residual pass, "auto" = ``LINEAR_IMPL``.
    ``bias_lp``: the same bias in x's dtype for the library GEMM's own epilogue (callers keep it in ``wcache``; cast on the
    fly when absent)."""
    _cuda(x, w, bias, residual)
    k, n = x.shape[-1], w.shape[0]
    m = x.numel() // k
    assert w.shape == (n, k) and w.dtype == x.dtype and x.dtype in (torch.bfloat16, torch.float16)
    assert bias is None or (bias.dtype == torch.float32 and bias.numel() == n)
    shape = (*x.shape[:-1], n)
    lib = _lib.load()
    impl = LINEAR_IMPL if impl == "auto" else impl
    tc_ok = bool(lib.dadd_linear_supported(m, n, k)) and x.is_contiguous() and w.is_contiguous() and (residual is None or residual.is_contiguous())
    if impl == "tc" and not tc_ok:
        raise _lib.DaddError(f"dadd_linear_fwd does not take M={m} N={n} K={k} (or an operand is not dense)")
    if impl == "tc":
        y = torch.empty(shape, dtype=x.dtype, device=x.device) if out is None else out
        assert y.is_contiguous() and y.shape == shape and (residual is None or residual.shape == shape)
        _lib.check(lib.dadd_linear_fwd(x.data_ptr(), w.data_ptr(), _ptr(bias), _ptr(residual), y.data_ptr(), m, n, k, _dt(x),
                                       _stream()), "dadd_linear_fwd")
        return y
    if residual is None:                               # bias in the library GEMM's own epilogue
        y = torch.nn.functional.linear(x, w, None if bias is None else (bias_lp if bias_lp is not None else bias.to(x.dtype)))
        if out is not None:
            out.copy_(y)
            y = out
        return y
    if bias is None:                                   # residual only: the library GEMM accumulates onto it (beta = 1)
        y = torch.empty(shape, dtype=x.dtype, device=x.device) if out is None else out
        return torch.addmm(residual.reshape(m, n), x.reshape(m, k), w.t(), out=y.view(m, n)).view(shape)
    y = torch.nn.functional.linear(x, w)
    return bias_residual(y, residual, bias, out=y if out is None else out)


def ff_geglu(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """``h, g = F.linear(x, w, bias).chunk(2, -1); h * gelu(g)`` as one tcgen05 GEMM with the gate in its epilogue.
    x (..., K) 16-bit contiguous, w (2*inner, K) same dtype, bias (2*inner,) fp32 -> (..., inner)."""
    _cuda(x, w, bias)
    k = x.shape[-1]
    inner = w.shape[0] // 2
    assert x.is_contiguous() and w.is_contiguous() and w.shape == (2 * inner, k) and w.dtype == x.dtype
    assert x.dtype in (torch.bfloat16, torch.float16) and bias.dtype == torch.float32 and bias.numel() == 2 * inner
    y = torch.empty(*x.shape[:-1], inner, dtype=x.dtype, device=x.device)
    _lib.check(_lib.load().dadd_ff_geglu_fwd(x.data_ptr(), w.data_ptr(), bias.data_ptr(), y.data_ptr(), x.numel() // k, k, inner,
                                             _dt(x), _stream()), "dadd_ff_geglu_fwd")
    return y


# --------------------------------------------------------------------------------------------- attention
def _rows(t: torch.Tensor) -> int:
    """Row stride (elements) of a (B, N, *) view whose last dim is dense and whose batch stride is N * row stride."""
    assert t.dim() == 3 and t.stride(2) == 1, "attention operands must be (B, N, C) with unit inner stride"
    assert t.shape[0] == 1 or t.stride(0) == t.shape[1] * t.stride(1), "batch stride must equal N * row stride"
    return t.stride(1)


def cross_attention(q: torch.Tensor, k_cat: torch.Tensor, v_cat: torch.Tensor, gates: torch.Tensor, heads: int,
                    seg_len: int, n_seg: int, scale: Optional[float] = None, impl: str = "auto") -> torch.Tensor:
    """sum_s gates[s] softmax(q k_s^T scale) v_s; q (B,N,H*d) bf16 (may be a strided view), k_cat/v_cat (B,H,L,d).
    ``impl``: "auto" (tcgen05 kernel for N >= 128, d <= 128), "mma" or "tc"."""
    _cuda(q, k_cat, v_cat, gates)
    b, n, c = q.shape
    d = c // heads
    assert q.dtype in (torch.bfloat16, torch.float16) and k_cat.dtype == q.dtype and v_cat.dtype == q.dtype
    assert k_cat.is_contiguous() and v_cat.is_contiguous() and k_cat.shape == (b, heads, seg_len * n_seg, d) == v_cat.shape
    assert gates.dtype == torch.float32 and gates.numel() >= n_seg
    o = torch.empty(b, n, c, device=q.device, dtype=q.dtype)
    _lib.check(_lib.load().dadd_cross_attn_fwd(q.data_ptr(), _rows(q), k_cat.data_ptr(), v_cat.data_ptr(), o.data_ptr(), c,
                                               b, heads, n, d, seg_len, n_seg, gates.data_ptr(),
                                               float(d ** -0.5 if scale is None else scale), _dt(q),
                                               {"auto": 0, "mma": 1, "tc": 2}[impl], _stream()),
               "dadd_cross_attn_fwd")
    return o


def self_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int, scale: Optional[float] = None,
                   impl: str = "auto") -> torch.Tensor:
    """softmax(q k^T scale) v per head; q,k,v (B,N,H*d) bf16/fp16, possibly strided views of one fused QKV buffer.
    ``impl``: "auto" (N >= 128 -> tcgen05 kernel, else mma.sync kernel), "mma" or "tc"."""
    _cuda(q, k, v)
    b, n, c = q.shape
    d = c // heads
    assert q.dtype == k.dtype == v.dtype and q.dtype in (torch.bfloat16, torch.float16) and k.shape == q.shape == v.shape
    o = torch.empty(b, n, c, device=q.device, dtype=q.dtype)
    _lib.check(_lib.load().dadd_self_attn_fwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), _rows(q), _rows(k), _rows(v),
                                              o.data_ptr(), c, b, heads, n, d,
                                              float(d ** -0.5 if scale is None else scale), _dt(q),
                                              {"auto": 0, "mma": 1, "tc": 2}[impl], _stream()),
               "dadd_self_attn_fwd")
    return o


# --------------------------------------------------------------------------------------------- conditioning front end
def purifier_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int) -> torch.Tensor:
    _cuda(q, k, v)
    assert q.dtype == k.dtype == v.dtype == torch.float32 and q.is_contiguous() and k.is_contiguous() and v.is_contiguous()
    b, lq, dm = q.shape
    o = torch.empty_like(q)
    _lib.check(_lib.load().dadd_purifier_attn_fwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), b, lq, k.shape[1],
                                                  dm, heads, _stream()), "dadd_purifier_attn_fwd")
    return o


def purifier_gate_ln(img: torch.Tensor, gate_logits: torch.Tensor, disease: torch.Tensor, gamma: torch.Tensor,
                     beta: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    _cuda(img, gate_logits, disease, gamma, beta)
    for t in (img, gate_logits, disease, gamma, beta):
        assert t.dtype == torch.float32 and t.is_contiguous()
    dm = img.shape[-1]
    y = torch.empty_like(img)
    _lib.check(_lib.load().dadd_purifier_gate_ln_fwd(img.data_ptr(), gate_logits.data_ptr(), disease.data_ptr(),
                                                     gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), img.numel() // dm, dm,
                                                     eps, _stream()), "dadd_purifier_gate_ln_fwd")
    return y


def aoe_interp(base: torch.Tensor, deltas: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
    _cuda(base, deltas, labels)
    for t in (base, deltas, labels):
        assert t.dtype == torch.float32 and t.is_contiguous()
    k, dm = deltas.shape[0] + 1, base.shape[0]
    out = torch.empty(labels.shape[0], dm, device=base.device, dtype=torch.float32)
    _lib.check(_lib.load().dadd_aoe_interp_fwd(base.data_ptr(), deltas.data_ptr(), labels.data_ptr(), out.data_ptr(),
                                               labels.shape[0], k, dm, _stream()), "dadd_aoe_interp_fwd")
    return out


def image_post(x: torch.Tensor) -> torch.Tensor:
    """clamp(-1,1) -> (x+1)/2 -> clamp(0,1) (inference_pipeline_ip.py:483-485); returns fp32 with x's strides."""
    _cuda(x)
    y = torch.empty_like(x, dtype=torch.float32)
    assert y.stride() == x.stride()
    _lib.check(_lib.load().dadd_image_post_fwd(x.data_ptr(), y.data_ptr(), x.numel(), _dt(x), _stream()), "dadd_image_post_fwd")
    return y


# --------------------------------------------------------------------------------------------- training step (backward, loss, optimizer)
def layer_norm_bwd(x: torch.Tensor, dy: torch.Tensor, gamma: torch.Tensor, eps: float):
    """Backward of ``layer_norm``: (dx like x, dgamma (C,) fp32, dbeta (C,) fp32); statistics recomputed from ``x``."""
    _cuda(x, dy, gamma)
    c = x.shape[-1]
    assert x.is_contiguous() and dy.is_contiguous() and x.shape == dy.shape and x.dtype == dy.dtype
    assert gamma.dtype == torch.float32 and gamma.numel() == c
    rows = x.numel() // c
    lib = _lib.load()
    dx = torch.empty_like(x)
    dgb = torch.empty(2, c, dtype=torch.float32, device=x.device)
    ws = torch.empty(max(int(lib.dadd_layernorm_bwd_workspace_bytes(c)), 8), dtype=torch.uint8, device=x.device)
    _lib.check(lib.dadd_layernorm_bwd(x.data_ptr(), dy.data_ptr(), gamma.data_ptr(), dx.data_ptr(), dgb[0].data_ptr(),
                                      dgb[1].data_ptr(), ws.data_ptr(), rows, c, eps, _dt(x), _stream()), "dadd_layernorm_bwd")
    return dx, dgb[0], dgb[1]


def geglu_bwd(proj: torch.Tensor, dy: torch.Tensor) -> torch.Tensor:
    """Backward of ``geglu``: ``proj`` (..., 2I) = [value | gate], ``dy`` (..., I) -> dproj like proj."""
    _cuda(proj, dy)
    inner = dy.shape[-1]
    assert proj.is_contiguous() and dy.is_contiguous() and proj.shape[-1] == 2 * inner and proj.dtype == dy.dtype
    dproj = torch.empty_like(proj)
    _lib.check(_lib.load().dadd_geglu_bwd(proj.data_ptr(), dy.data_ptr(), dproj.data_ptr(), dy.numel() // inner, inner, _dt(proj),
                                          _stream()), "dadd_geglu_bwd")
    return dproj


def group_norm_bwd(x: torch.Tensor, dy: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, num_groups: int, eps: float,
                   silu: bool, chan_add: Optional[torch.Tensor] = None, need_dchan_add: bool = False):
    """Backward of ``group_norm`` on channels_last tensors: (dx, dgamma, dbeta, dchan_add or None)."""
    _cuda(x, dy, gamma, beta, chan_add)
    assert x.dim() == 4 and x.is_contiguous(memory_format=torch.channels_last) and dy.shape == x.shape and dy.dtype == x.dtype
    if not dy.is_contiguous(memory_format=torch.channels_last):
        dy = dy.contiguous(memory_format=torch.channels_last)
    b, c, h, w = x.shape
    if chan_add is not None:
        assert chan_add.dtype == torch.float32 and chan_add.shape == (b, c)
        chan_add = chan_add.contiguous()
    lib = _lib.load()
    dx = torch.empty_like(x)
    dgamma = torch.empty(c, dtype=torch.float32, device=x.device)
    dbeta = torch.empty(c, dtype=torch.float32, device=x.device)
    dadd = torch.empty(b, c, dtype=torch.float32, device=x.device) if (need_dchan_add and chan_add is not None) else None
    ws = torch.empty(max(int(lib.dadd_groupnorm_bwd_workspace_bytes(b, c, h * w, num_groups)), 8), dtype=torch.uint8, device=x.device)
    _lib.check(lib.dadd_groupnorm_bwd(x.data_ptr(), _ptr(chan_add), dy.data_ptr(), gamma.data_ptr(), beta.data_ptr(), dx.data_ptr(),
                                      dgamma.data_ptr(), dbeta.data_ptr(), _ptr(dadd), ws.data_ptr(), b, h * w, c, num_groups, eps,
                                      int(silu), _dt(x), _stream()), "dadd_groupnorm_bwd")
    return dx, dgamma, dbeta, dadd


def cross_attention_bwd(q: torch.Tensor, k_cat: torch.Tensor, v_cat: torch.Tensor, gates: torch.Tensor, dout: torch.Tensor,
                        heads: int, seg_len: int, n_seg: int):
    """Backward of ``cross_attention``: (dq like q, dk_cat fp32, dv_cat fp32)."""
    _cuda(q, k_cat, v_cat, gates, dout)
    b, n, c = q.shape
    d = c // heads
    l = n_seg * seg_len
    assert q.stride(-1) == 1 and dout.stride(-1) == 1 and dout.shape == q.shape and dout.dtype == q.dtype
    assert k_cat.is_contiguous() and v_cat.is_contiguous() and k_cat.shape == (b, heads, l, d) == v_cat.shape and k_cat.dtype == q.dtype
    assert gates.dtype == torch.float32 and gates.numel() >= n_seg
    lib = _lib.load()
    dq = torch.empty(b, n, c, dtype=q.dtype, device=q.device)
    dk = torch.empty(b, heads, l, d, dtype=torch.float32, device=q.device)
    dv = torch.empty_like(dk)
    ws = torch.empty(max(int(lib.dadd_cross_attn_bwd_workspace_bytes(b, heads, n, d, l)), 8), dtype=torch.uint8, device=q.device)
    _lib.check(lib.dadd_cross_attn_bwd(q.data_ptr(), q.stride(-2), k_cat.data_ptr(), v_cat.data_ptr(), gates.data_ptr(), dout.data_ptr(),
                                       dout.stride(-2), dq.data_ptr(), c, dk.data_ptr(), dv.data_ptr(), ws.data_ptr(), b, heads, n, d, l,
                                       seg_len, float(d ** -0.5), _dt(q), _stream()), "dadd_cross_attn_bwd")
    return dq, dk, dv


def minsnr_mse(pred: torch.Tensor, target: torch.Tensor, weight: torch.Tensor, need_grad: bool = True, upstream: float = 1.0):
    """loss = mean_b weight[b] * mean(pred[b] - target[b])^2 and (optionally) dloss/dpred * upstream, one pass."""
    _cuda(pred, target, weight)
    assert pred.dtype == torch.float32 and target.dtype == torch.float32 and weight.dtype == torch.float32
    assert pred.is_contiguous() and target.is_contiguous() and pred.shape == target.shape and weight.numel() == pred.shape[0]
    b = pred.shape[0]
    e = pred.numel() // b
    lib = _lib.load()
    loss = torch.empty(1, dtype=torch.float32, device=pred.device)
    grad = torch.empty_like(pred) if need_grad else None
    ws = torch.empty(int(lib.dadd_minsnr_mse_workspace_bytes(b)), dtype=torch.uint8, device=pred.device)
    _lib.check(lib.dadd_minsnr_mse(pred.data_ptr(), target.data_ptr(), weight.data_ptr(), loss.data_ptr(), _ptr(grad), ws.data_ptr(),
                                   b, e, upstream, _stream()), "dadd_minsnr_mse")
    return loss[0], grad


SUMSQ_PARTIALS = 296      # partial sums per flat buffer (2 x 148 SMs)


def sumsq_(g: torch.Tensor, partials: torch.Tensor) -> None:
    """partials[:] = SUMSQ_PARTIALS partial sums of g^2 (flat fp32)."""
    _cuda(g, partials)
    assert g.dtype == torch.float32 and g.is_contiguous() and partials.dtype == torch.float32 and partials.is_contiguous()
    _lib.check(_lib.load().dadd_sumsq(g.data_ptr(), g.numel(), partials.data_ptr(), partials.numel(), _stream()), "dadd_sumsq")


def clip_coef_(partials: torch.Tensor, max_norm: float, grad_scale: float, coef_and_norm: torch.Tensor) -> None:
    _cuda(partials, coef_and_norm)
    assert partials.dtype == torch.float32 and partials.is_contiguous() and coef_and_norm.numel() >= 2
    _lib.check(_lib.load().dadd_clip_coef(partials.data_ptr(), partials.numel(), max_norm, grad_scale, coef_and_norm.data_ptr(),
                                          _stream()), "dadd_clip_coef")


def adamw_step_dev_(p: torch.Tensor, g: torch.Tensor, m: torch.Tensor, v: torch.Tensor, lr: float, beta1: float, beta2: float,
                    eps: float, weight_decay: float, dev_state: torch.Tensor, coef: Optional[torch.Tensor] = None) -> None:
    """``adamw_step_`` with the learning-rate scale and the step number read from ``dev_state`` = [scale, step] on the device
    (graph-capturable: no host-side argument depends on the step)."""
    _cuda(p, g, m, v, dev_state, coef)
    for t in (p, g, m, v):
        assert t.dtype == torch.float32 and t.is_contiguous() and t.numel() == p.numel()
    assert dev_state.dtype == torch.float32 and dev_state.numel() >= 2
    _lib.check(_lib.load().dadd_adamw_step_dev(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), lr, beta1, beta2, eps,
                                               weight_decay, dev_state.data_ptr(), _ptr(coef), _stream()), "dadd_adamw_step_dev")


def ema_update_(avg: torch.Tensor, p: torch.Tensor, decay: float, first: bool = False) -> None:
    """``avg += (p - avg) * (1 - decay)`` on flat fp32 buffers (``first``: ``avg = p``): torch.optim.swa_utils.get_ema_avg_fn."""
    _cuda(avg, p)
    assert avg.dtype == p.dtype == torch.float32 and avg.is_contiguous() and p.is_contiguous() and avg.numel() == p.numel()
    _lib.check(_lib.load().dadd_ema_update(avg.data_ptr(), p.data_ptr(), p.numel(), float(decay), int(first), _stream()), "dadd_ema_update")


def adamw_step_(p: torch.Tensor, g: torch.Tensor, m: torch.Tensor, v: torch.Tensor, lr: float, beta1: float, beta2: float,
                eps: float, weight_decay: float, step: int, coef: Optional[torch.Tensor] = None) -> None:
    """torch.optim.AdamW's update on flat fp32 buffers, in place; ``g`` is scaled by ``coef[0]`` (device scalar) on the fly."""
    _cuda(p, g, m, v, coef)
    for t in (p, g, m, v):
        assert t.dtype == torch.float32 and t.is_contiguous() and t.numel() == p.numel()
    _lib.check(_lib.load().dadd_adamw_step(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), lr, beta1, beta2, eps,
                                           weight_decay, 1.0 - beta1 ** step, 1.0 - beta2 ** step, _ptr(coef), _stream()),
               "dadd_adamw_step")


# --------------------------------------------------------------------------------------------- evaluation metrics
RBF_SUM, KNN, COVER, COUNT, RATIO_MAX = 0, 1, 2, 3, 4


def _features(*ts: torch.Tensor) -> None:
    _cuda(*ts)
    for t in ts:
        if t.dtype != torch.float32 or t.dim() != 2 or not t.is_contiguous():
            raise _lib.DaddError(f"pairwise statistics take contiguous 2-D float32 feature matrices, got {t.dtype} {tuple(t.shape)}")


def _pairwise(x: torch.Tensor, y: Optional[torch.Tensor], mode: int, out: torch.Tensor, k: int = 0, gamma: float = 0.0,
              radii: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = _lib.load()
    m, d = x.shape
    n = m if y is None else y.shape[0]
    if y is not None and y.shape[1] != d:
        raise _lib.DaddError(f"feature widths differ: {d} vs {y.shape[1]}")
    same = int(y is None)
    ws_bytes = int(lib.dadd_pairwise_workspace_bytes(m, n, d, mode, k, same))
    if ws_bytes < 0:
        _lib.check(1, "dadd_pairwise_workspace_bytes")
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
    _lib.check(lib.dadd_pairwise(x.data_ptr(), _ptr(y), m, n, d, mode, k, same, float(gamma), _ptr(radii), out.data_ptr(),
                                 ws.data_ptr(), ws_bytes, _stream()), "dadd_pairwise")
    return out


def pairwise_rbf_sum(x: torch.Tensor, y: Optional[torch.Tensor], gamma: float) -> torch.Tensor:
    """sum over all (i, j) of exp(-gamma |x_i - y_j|^2) as a float64 device scalar; ``y=None``: y is x.  x: (M, D), y: (N, D)
    float32, D % 8 == 0 (the kernel sums of google-research/cmmd's ``mmd``)."""
    _features(x, *(() if y is None else (y,)))
    return _pairwise(x, y, RBF_SUM, torch.empty((), dtype=torch.float64, device=x.device), gamma=gamma)


def knn_radii(x: torch.Tensor, k: int, ref: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(M,) float32: the squared distance from each row of x to its k-th nearest OTHER row (1 <= k <= 16, M > k + 1): the
    manifold radii of improved precision / recall (Kynkaanniemi et al. 2019).  With ``ref`` (N, D): the k-th smallest squared
    distance from each row of x to the rows of ref (N > k), nothing excluded (k = 1: the nearest-neighbour distance)."""
    _features(x, *(() if ref is None else (ref,)))
    return _pairwise(x, ref, KNN, torch.empty(x.shape[0], dtype=torch.float32, device=x.device), k=k)


def _radii(q: torch.Tensor, ref: torch.Tensor, radii: torch.Tensor) -> None:
    _features(q, ref)
    _cuda(radii)
    if radii.dtype != torch.float32 or radii.shape != (ref.shape[0],) or not radii.is_contiguous():
        raise _lib.DaddError(f"radii must be a contiguous float32 ({ref.shape[0]},) tensor")


def within_radii(q: torch.Tensor, ref: torch.Tensor, radii: torch.Tensor) -> torch.Tensor:
    """(M,) bool: whether each row of q lies in at least one ball |q_i - ref_j|^2 <= radii[j] (improved precision / recall)."""
    _radii(q, ref, radii)
    return _pairwise(q, ref, COVER, torch.empty(q.shape[0], dtype=torch.bool, device=q.device), radii=radii)


def count_within_radii(q: torch.Tensor, ref: torch.Tensor, radii: torch.Tensor) -> torch.Tensor:
    """(M,) int32: for each row of q, the number of balls |q_i - ref_j|^2 <= radii[j] it lies in (density, Naeem et al. 2020)."""
    _radii(q, ref, radii)
    return _pairwise(q, ref, COUNT, torch.empty(q.shape[0], dtype=torch.int32, device=q.device), radii=radii)


def max_radius_ratio(q: torch.Tensor, ref: torch.Tensor, radii: torch.Tensor, eps: float) -> torch.Tensor:
    """(M,) float32: max over j of radii[j] / (|q_i - ref_j|^2 + eps), eps finite and > 0, 0 when no ratio is positive (the
    squared realism score of Kynkaanniemi et al. 2019)."""
    _radii(q, ref, radii)
    return _pairwise(q, ref, RATIO_MAX, torch.empty(q.shape[0], dtype=torch.float32, device=q.device), gamma=eps, radii=radii)
