"""DADD training step on B200 (SURVEY.md 8f row f1, BASELINE config 3).

What the reference does through Lightning (``/root/reference/src/models/diffusion_module_ip.py:392-462`` training_step,
``:334-381`` _prepare_conditioning(is_training=True), ``:299-313`` _q_sample / _min_snr_weight, ``:500-536`` AdamW groups;
``src/pipelines/training/training_pipeline_ip.py:103-123`` precision "16-mixed", gradient_clip_val, DDP
``find_unused_parameters=False``) is restated here as a plain PyTorch-autograd program over the SAME module tree
(``DiffusionModuleWithIP``: fp32 master parameters, diffusers key names), with

* 16-bit (bf16 by default) channels-last activations, weights cast per step (the autocast policy of "16-mixed");
* the memory-bound norm / gate layers and both attention cores on this package's CUDA kernels in forward, and hand-written
  backward kernels for GroupNorm(+temb)(+SiLU), LayerNorm, GEGLU and the triple-pathway cross-attention core
  (``csrc/train.cu``); the self-attention core recomputes its backward through the library flash-attention backward - marked
  below; convolutions and GEMMs are cuDNN / cuBLAS in both directions (off-path by the north-star);
* the Min-SNR-weighted MSE loss and its gradient in one kernel;
* data parallelism as one process per GPU: gradients live in flat fp32 buckets that are all-reduced (NCCL over NVLink) as soon
  as the backward pass has filled them, overlapped with the rest of backward; the three parameters the reference never uses in
  any forward (``ordinal_embedder.norm.{weight,bias}``, ``ordinal_embedder.null_embedding``; SURVEY.md 7.3) stay outside the
  buckets - the ``find_unused_parameters=False`` contract;
* gradient-norm clipping and AdamW (the reference's four parameter groups, lr x2 for the projection and the purifier) as one
  kernel launch per bucket over flat fp32 parameter / moment buffers, with the clip coefficient kept on the device.

There is no CPU fallback: CPU tensors raise in the kernels' wrappers.
"""

from __future__ import annotations

import math
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist
import torch.nn as nn
import torch.nn.functional as F

from . import ops, wcache
from .attention_processor_routing_gates import SplitInjectionAttentionProcessor
from .unet2d import (BasicTransformerBlock, ResnetBlock2D, Transformer2DModel, UNet2DConditionModel)

CL = torch.channels_last
UNUSED_PARAMETERS = ("ordinal_embedder.norm.weight", "ordinal_embedder.norm.bias", "ordinal_embedder.null_embedding")


# ================================================================================================ autograd nodes on our kernels
class _GroupNorm(torch.autograd.Function):
    """GroupNorm (+ per-(sample, channel) additive term) (+ SiLU): dadd_groupnorm_fwd / dadd_groupnorm_bwd."""

    @staticmethod
    def forward(ctx, x, gamma, beta, chan_add, groups: int, eps: float, silu: bool):
        g32, b32 = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
        add = None if chan_add is None else chan_add.detach().float().contiguous()
        ctx.save_for_backward(x, g32, b32, add)
        ctx.cfg = (groups, eps, silu, chan_add is not None and chan_add.requires_grad, gamma.dtype)
        return ops.group_norm(x, g32, b32, groups, eps, silu, add)

    @staticmethod
    def backward(ctx, dy):
        x, g32, b32, add = ctx.saved_tensors
        groups, eps, silu, need_dadd, pdt = ctx.cfg
        dx, dg, db, dadd = ops.group_norm_bwd(x, dy, g32, b32, groups, eps, silu, add, need_dchan_add=need_dadd)
        return dx, dg.to(pdt), db.to(pdt), dadd, None, None, None


class _LayerNorm(torch.autograd.Function):
    """LayerNorm over the last dimension of 16-bit tokens: dadd_layernorm_fwd / dadd_layernorm_bwd."""

    @staticmethod
    def forward(ctx, x, gamma, beta, eps: float):
        g32, b32 = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
        x = x.contiguous()
        ctx.save_for_backward(x, g32)
        ctx.cfg = (eps, gamma.dtype)
        return ops.layer_norm(x, g32, b32, eps)

    @staticmethod
    def backward(ctx, dy):
        x, g32 = ctx.saved_tensors
        eps, pdt = ctx.cfg
        dx, dg, db = ops.layer_norm_bwd(x, dy.contiguous(), g32, eps)
        return dx, dg.to(pdt), db.to(pdt), None


class _GEGLU(torch.autograd.Function):
    """value * gelu(gate) of a (M, 2I) projection: dadd_geglu_fwd / dadd_geglu_bwd."""

    @staticmethod
    def forward(ctx, proj):
        proj = proj.contiguous()
        ctx.save_for_backward(proj)
        return ops.geglu(proj)

    @staticmethod
    def backward(ctx, dy):
        (proj,) = ctx.saved_tensors
        return ops.geglu_bwd(proj, dy.contiguous())


class _SelfAttention(torch.autograd.Function):
    """Forward: the tcgen05 flash kernel (dadd_self_attn_fwd) on the fused QKV projection in place.  Backward: recomputed through
    the LIBRARY flash-attention backward (F.scaled_dot_product_attention under autograd) - no hand-written kernel yet."""

    @staticmethod
    def forward(ctx, q, k, v, heads: int):
        ctx.save_for_backward(q, k, v)
        ctx.heads = heads
        return ops.self_attention(q, k, v, heads)

    @staticmethod
    def backward(ctx, do):
        q, k, v = ctx.saved_tensors
        h = ctx.heads
        b, n, c = q.shape
        with torch.enable_grad():
            qq, kk, vv = (t.detach().reshape(b, n, h, c // h).transpose(1, 2).requires_grad_(True) for t in (q, k, v))
            o = F.scaled_dot_product_attention(qq, kk, vv).transpose(1, 2).reshape(b, n, c)
            dq, dk, dv = torch.autograd.grad(o, (qq, kk, vv), do)
        back = lambda t: t.transpose(1, 2).reshape(b, n, c)
        return back(dq), back(dk), back(dv), None


class _CrossAttention(torch.autograd.Function):
    """The fused triple-pathway core (per-segment softmax over the 16-token segments, gate-weighted merge):
    dadd_cross_attn_fwd / dadd_cross_attn_bwd."""

    @staticmethod
    def forward(ctx, q, k_cat, v_cat, gates, heads: int, seg_len: int, n_seg: int):
        ctx.save_for_backward(q, k_cat, v_cat, gates)
        ctx.cfg = (heads, seg_len, n_seg)
        return ops.cross_attention(q, k_cat, v_cat, gates, heads, seg_len, n_seg)

    @staticmethod
    def backward(ctx, do):
        q, k_cat, v_cat, gates = ctx.saved_tensors
        heads, seg_len, n_seg = ctx.cfg
        dq, dk, dv = ops.cross_attention_bwd(q, k_cat, v_cat, gates, do.contiguous(), heads, seg_len, n_seg)
        return dq, dk.to(k_cat.dtype), dv.to(v_cat.dtype), None, None, None, None


# ================================================================================================ differentiable forward
def _w(p: torch.Tensor, dt: torch.dtype) -> torch.Tensor:
    return p.to(dt)


def _lin(mod: nn.Linear, x: torch.Tensor) -> torch.Tensor:
    return F.linear(x, _w(mod.weight, x.dtype), None if mod.bias is None else _w(mod.bias, x.dtype))


def _conv(mod: nn.Conv2d, x: torch.Tensor) -> torch.Tensor:
    w = _w(mod.weight, x.dtype).contiguous(memory_format=CL)
    return F.conv2d(x, w, None if mod.bias is None else _w(mod.bias, x.dtype), mod.stride, mod.padding)


def _gn(mod: nn.GroupNorm, x: torch.Tensor, silu: bool, chan_add: Optional[torch.Tensor] = None) -> torch.Tensor:
    return _GroupNorm.apply(x.contiguous(memory_format=CL), mod.weight, mod.bias, chan_add, mod.num_groups, mod.eps, silu)


def _ln(mod: nn.LayerNorm, x: torch.Tensor) -> torch.Tensor:
    return _LayerNorm.apply(x, mod.weight, mod.bias, mod.eps)


def _resnet(res: ResnetBlock2D, x: torch.Tensor, emb_act: torch.Tensor) -> torch.Tensor:
    """diffusers ResnetBlock2D (SURVEY.md A.3); the time-embedding term enters norm2 as the GN kernel's additive input."""
    h = _conv(res.conv1, _gn(res.norm1, x, True))
    temb = F.linear(emb_act, res.time_emb_proj.weight.float(), res.time_emb_proj.bias.float())      # fp32 (B, cout)
    h = _conv(res.conv2, _gn(res.norm2, h, True, temb))
    if res.conv_shortcut is not None:
        x = _conv(res.conv_shortcut, x)
    return x + h


def _cross_kv(proc: SplitInjectionAttentionProcessor, attn, ehs: torch.Tensor, dt: torch.dtype):
    """K_cat / V_cat (B, H, n_seg * 16, d) in token order dis | anat (| delta), projected under autograd (to_k / to_v for the
    anatomy tokens, to_k_dis / to_v_dis for the AOE tokens; attention_processor_routing_gates.py:129-137,161-162)."""
    n = proc.num_aoe_tokens
    with_delta = proc.delta_scale != 0.0
    e = ehs.to(dt)
    dis, anat = e[:, :n], e[:, n:n + proc.num_image_tokens]

    def project(wa: torch.Tensor, wd: torch.Tensor) -> torch.Tensor:
        parts = [F.linear(dis, _w(wd, dt)), F.linear(anat, _w(wa, dt))]
        if with_delta:
            parts.append(F.linear(e[:, -proc.num_delta_tokens:], _w(wd, dt)))
        cat = torch.cat(parts, dim=1)
        b, l, c = cat.shape
        return cat.view(b, l, attn.heads, c // attn.heads).permute(0, 2, 1, 3).contiguous()

    return project(attn.to_k.weight, proc.to_k_dis.weight), project(attn.to_v.weight, proc.to_v_dis.weight), (3 if with_delta else 2)


def _block(blk: BasicTransformerBlock, t: torch.Tensor, ehs: torch.Tensor) -> torch.Tensor:
    """diffusers BasicTransformerBlock (SURVEY.md A.5) with the split-injection processor on attn2."""
    a1, a2 = blk.attn1, blk.attn2
    c = t.shape[-1]
    wqkv = torch.cat([a1.to_q.weight, a1.to_k.weight, a1.to_v.weight], dim=0)
    qkv = F.linear(_ln(blk.norm1, t), _w(wqkv, t.dtype))
    o = _SelfAttention.apply(qkv[..., :c], qkv[..., c:2 * c], qkv[..., 2 * c:], a1.heads)
    t = t + _lin(a1.to_out[0], o)
    proc = a2.processor
    if not isinstance(proc, SplitInjectionAttentionProcessor):
        raise NotImplementedError("the training step covers the shipped configuration (use_routing_gates=True)")
    q = _lin(a2.to_q, _ln(blk.norm2, t))
    k_cat, v_cat, n_seg = _cross_kv(proc, a2, ehs, t.dtype)
    z = _CrossAttention.apply(q.contiguous(), k_cat, v_cat, proc.gate_vector(), a2.heads, proc.num_aoe_tokens, n_seg)
    t = t + _lin(a2.to_out[0], z)
    g = _GEGLU.apply(_lin(blk.ff.net[0].proj, _ln(blk.norm3, t)))
    return t + _lin(blk.ff.net[2], g)


def _transformer(tr: Transformer2DModel, x: torch.Tensor, ehs: torch.Tensor) -> torch.Tensor:
    b, c, h, w = x.shape
    t = _conv(tr.proj_in, _gn(tr.norm, x, False))
    t = t.permute(0, 2, 3, 1).reshape(b, h * w, c)                   # free view (channels-last)
    for blk in tr.transformer_blocks:
        t = _block(blk, t, ehs)
    return _conv(tr.proj_out, t.view(b, h, w, c).permute(0, 3, 1, 2)) + x


def unet_forward_train(unet: UNet2DConditionModel, sample: torch.Tensor, timesteps: torch.Tensor, ehs: torch.Tensor,
                       compute_dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """eps = UNet(sample, t, cond) under autograd (same graph as ``UNet2DConditionModel.forward`` / SURVEY.md Appendix A)."""
    half = unet.config.block_out_channels[0] // 2
    freqs = torch.exp(-math.log(10000.0) * torch.arange(half, dtype=torch.float32, device=sample.device) / half)
    args = timesteps.to(torch.float32)[:, None] * freqs[None, :]
    te = unet.time_embedding
    emb = F.linear(torch.cat([torch.cos(args), torch.sin(args)], dim=-1), te.linear_1.weight.float(), te.linear_1.bias.float())
    emb_act = F.silu(F.linear(F.silu(emb), te.linear_2.weight.float(), te.linear_2.bias.float()))
    x = _conv(unet.conv_in, sample.to(compute_dtype).contiguous(memory_format=CL))
    skips = [x]
    for blk in unet.down_blocks:
        for j, res in enumerate(blk.resnets):
            x = _resnet(res, x, emb_act)
            if len(blk.attentions) > 0:
                x = _transformer(blk.attentions[j], x, ehs)
            skips.append(x)
        if blk.downsamplers is not None:
            x = _conv(blk.downsamplers[0].conv, x)
            skips.append(x)
    mb = unet.mid_block
    x = _resnet(mb.resnets[0], x, emb_act)
    x = _transformer(mb.attentions[0], x, ehs)
    x = _resnet(mb.resnets[1], x, emb_act)
    for blk in unet.up_blocks:
        for j, res in enumerate(blk.resnets):
            x = _resnet(res, torch.cat([x, skips.pop()], dim=1).contiguous(memory_format=CL), emb_act)
            if len(blk.attentions) > 0:
                x = _transformer(blk.attentions[j], x, ehs)
        if blk.upsamplers is not None:
            x = _conv(blk.upsamplers[0].conv, F.interpolate(x, scale_factor=2.0, mode="nearest"))
    return _conv(unet.conv_out, _gn(unet.conv_norm_out, x, True)).float().contiguous()


# ---- conditioning front end under autograd (fp32, (B, 16, 768) tokens: once per step, library GEMMs) ----
def _mha(mha: nn.MultiheadAttention, q_in: torch.Tensor, kv_in: torch.Tensor) -> torch.Tensor:
    d, h = mha.embed_dim, mha.num_heads
    wi, bi = mha.in_proj_weight, mha.in_proj_bias
    q = F.linear(q_in, wi[:d], bi[:d])
    k = F.linear(kv_in, wi[d:2 * d], bi[d:2 * d])
    v = F.linear(kv_in, wi[2 * d:], bi[2 * d:])
    split = lambda t: t.view(t.shape[0], t.shape[1], h, d // h).transpose(1, 2)
    o = F.scaled_dot_product_attention(split(q), split(k), split(v)).transpose(1, 2).reshape(q.shape)
    return F.linear(o, mha.out_proj.weight, mha.out_proj.bias)


def aoe_train(emb_mod, labels: torch.Tensor, noise_std: float = 0.005, generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """``AdditiveOrdinalEmbedder.forward(labels, is_training=True)`` (ordinal_embedder.py:129-180) under autograd."""
    k = emb_mod.num_classes
    table = torch.cat([emb_mod.base[None], emb_mod.base[None] + torch.cumsum(emb_mod.deltas, dim=0)], dim=0)      # (K, D)
    y = labels.to(table.device, torch.float32).reshape(-1).clamp(0.0, float(k - 1))
    lo = torch.floor(y).long()
    hi = torch.clamp(lo + 1, max=k - 1)
    a = (y - lo.float())[:, None]
    emb = table[lo] * (1.0 - a) + table[hi] * a
    if noise_std > 0:
        emb = emb + torch.randn(emb.shape, device=emb.device, dtype=emb.dtype, generator=generator) * noise_std
    p0, p2 = emb_mod.projector[0], emb_mod.projector[2]
    out = F.linear(F.gelu(F.linear(emb, p0.weight, p0.bias)), p2.weight, p2.bias)
    return out.view(-1, emb_mod.num_tokens, emb_mod.embedding_dim)


def purifier_train(pur, image_embeds: torch.Tensor, source_aoe: torch.Tensor) -> torch.Tensor:
    """``FeaturePurifier.forward`` (feature_purifier.py:64-95) under autograd."""
    ln = lambda m, x: F.layer_norm(x, (x.shape[-1],), m.weight, m.bias, m.eps)
    img_n, aoe_n = ln(pur.norm_img, image_embeds), ln(pur.norm_aoe, source_aoe)
    disease = _mha(pur.cross_attn, img_n, aoe_n)
    gate = torch.sigmoid(F.linear(F.gelu(F.linear(torch.cat([disease, img_n], dim=-1), pur.gate[0].weight, pur.gate[0].bias)),
                                  pur.gate[2].weight, pur.gate[2].bias))
    return ln(pur.norm_out, image_embeds - gate * disease)


def projection_plus_train(proj, hidden_states: torch.Tensor) -> torch.Tensor:
    """``ImageProjectionPlus.forward`` (image_encoder.py:193-228) under autograd."""
    ln = lambda m, x: F.layer_norm(x, (x.shape[-1],), m.weight, m.bias, m.eps)
    hs = hidden_states.float()
    if isinstance(proj.proj_in, nn.Linear):
        hs = F.linear(hs, proj.proj_in.weight, proj.proj_in.bias)
    lat = proj.latents.expand(hs.shape[0], -1, -1)
    for layer in proj.layers:
        lat = lat + _mha(layer["cross_attn"], ln(layer["norm1"], lat), hs)
        ff = layer["ff"]
        lat = lat + F.linear(F.gelu(F.linear(ln(layer["norm2"], lat), ff[0].weight, ff[0].bias)), ff[2].weight, ff[2].bias)
    return ln(proj.norm_out, lat)


# ================================================================================================ the step
def sample_timesteps(module, batch_size: int, device, generator: Optional[torch.Generator] = None) -> torch.Tensor:
    return torch.randint(0, module.diff_cfg.num_train_timesteps, (batch_size,), device=device, dtype=torch.long, generator=generator)


def q_sample(module, x0: torch.Tensor, t: torch.Tensor, noise: torch.Tensor) -> torch.Tensor:
    ac = module.alphas_cumprod.to(x0.device)[t]
    return torch.sqrt(ac).view(-1, 1, 1, 1) * x0 + torch.sqrt(1.0 - ac).view(-1, 1, 1, 1) * noise


def min_snr_weight(module, t: torch.Tensor) -> torch.Tensor:
    if not module.cfg.training.use_min_snr_weighting:
        return torch.ones_like(t, dtype=torch.float32)
    snr = module.snr_values.to(t.device)[t]
    return torch.clamp(snr, max=float(module.diff_cfg.min_snr_gamma)) / (snr + 1e-8)      # min(snr, gamma), no host tensor (graph capture)


class _MinSnrMse(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target, weight):
        loss, grad = ops.minsnr_mse(pred.contiguous(), target.contiguous(), weight.contiguous().float(), need_grad=True)
        ctx.save_for_backward(grad)
        return loss

    @staticmethod
    def backward(ctx, dloss):
        (grad,) = ctx.saved_tensors
        return grad * dloss, None, None


def training_loss(module, latents: torch.Tensor, labels: torch.Tensor, image_tokens: torch.Tensor, *,
                  generator: Optional[torch.Generator] = None, compute_dtype: torch.dtype = torch.bfloat16,
                  noise: Optional[torch.Tensor] = None, timesteps: Optional[torch.Tensor] = None, aoe_noise_std: float = 0.005,
                  drop_mask: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, Dict[str, torch.Tensor]]:
    """The body of ``training_step`` (diffusion_module_ip.py:404-452) from the scaled latents on.

    ``image_tokens``: raw projected image tokens (B, 16, 768) - ``ImageProjection(Plus)`` output - or CLIP hidden states
    (B, 257, 1024) that go through the module's trainable ``image_projection`` first.  ``noise`` / ``timesteps`` /
    ``drop_mask`` inject the step's random draws (tests); by default they come from ``generator``."""
    dev = latents.device
    b = latents.shape[0]
    if noise is None:
        noise = torch.randn(latents.shape, device=dev, dtype=latents.dtype, generator=generator)
    t = sample_timesteps(module, b, dev, generator) if timesteps is None else timesteps.to(dev)
    noisy = q_sample(module, latents, t, noise)
    # _prepare_conditioning(labels, structure_images, is_training=True): source == target -> delta = 0
    aoe = aoe_train(module.ordinal_embedder, labels, aoe_noise_std, generator)
    img = image_tokens.to(dev).float()
    if img.shape[-1] != aoe.shape[-1] or img.shape[1] != module.diff_cfg.num_image_tokens:
        img = projection_plus_train(module.image_projection, img)
    if module.feature_purifier is not None:
        img = purifier_train(module.feature_purifier, img, aoe)
    p_drop = float(getattr(module.cfg.model, "cfg_drop_prob", 0.1))
    if drop_mask is None:
        drop_mask = torch.rand(b, device=dev, generator=generator) < p_drop
    img = torch.where(drop_mask.view(-1, 1, 1), torch.zeros_like(img), img)
    cond = torch.cat([aoe, img, torch.zeros_like(aoe)], dim=1)      # [Source_AOE | E_clean | Delta_AOE = 0]
    pred = unet_forward_train(module.unet.unet, noisy, t, cond, compute_dtype)
    loss = _MinSnrMse.apply(pred, noise.float(), min_snr_weight(module, t))
    return loss, {"cfg_drop_rate": drop_mask.float().mean(), "timesteps": t}


def training_step(module, batch, batch_idx: int = 0, *, generator: Optional[torch.Generator] = None,
                  compute_dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """``DiffusionModuleWithIP.training_step(batch, batch_idx)``: batch = (images (B,3,H,W) in [-1,1], labels (B,),
    structure_images (B,3,224,224) CLIP-preprocessed).  The VAE and the CLIP tower are frozen (no_grad)."""
    images, labels, structure_images = batch
    with torch.no_grad():
        dist_ = module.vae.encode(images).latent_dist
        latents = dist_.sample(generator) * module.diff_cfg.latent_scale
        hidden = module.image_encoder.get_hidden_states(structure_images) if structure_images.dim() == 4 else structure_images
    loss, _ = training_loss(module, latents.float(), labels, hidden, generator=generator, compute_dtype=compute_dtype)
    return loss


# ================================================================================================ optimizer + data parallelism
def parameter_groups(module, lr: float) -> List[Dict]:
    """The reference's AdamW groups (diffusion_module_ip.py:504-514): UNet and AOE at lr, projection and purifier at 2 lr."""
    groups = [{"name": "unet", "params": list(module.unet.parameters()), "lr": lr},
              {"name": "ordinal_embedder", "params": list(module.ordinal_embedder.parameters()), "lr": lr}]
    if getattr(module, "image_projection", None) is not None:
        groups.append({"name": "image_projection", "params": list(module.image_projection.parameters()), "lr": lr * 2})
    if module.feature_purifier is not None:
        groups.append({"name": "feature_purifier", "params": list(module.feature_purifier.parameters()), "lr": lr * 2})
    return groups


def warmup_cosine_lr(epoch: int, base_lr: float, warmup_epochs: int, max_epochs: int, warmup_start_lr: float, eta_min: float) -> float:
    """LinearWarmupCosineAnnealingLR.get_lr of the reference (src/models/lr_scheduler.py:41-64), closed form per epoch."""
    warmup_epochs, max_epochs = max(0, int(warmup_epochs)), max(1, int(max_epochs))
    if warmup_epochs > 0 and epoch < warmup_epochs:
        return warmup_start_lr + (base_lr - warmup_start_lr) * (epoch / float(warmup_epochs))
    progress = min((epoch - warmup_epochs) / float(max(1, max_epochs - warmup_epochs)), 1.0)
    return eta_min + (base_lr - eta_min) * 0.5 * (1.0 + math.cos(math.pi * progress))


class _Bucket:
    def __init__(self, params: List[nn.Parameter], group: int, lr: float, device, dtype=torch.float32) -> None:
        self.params, self.group, self.lr = params, group, lr
        self.offsets, n = [], 0
        for p in params:
            self.offsets.append(n)
            n += (p.numel() + 3) // 4 * 4                                    # 16-byte aligned slots
        self.numel = n
        self.flat_p = torch.zeros(n, device=device, dtype=dtype)
        self.flat_g = torch.zeros(n, device=device, dtype=dtype)
        self.m = self.v = None
        with torch.no_grad():
            for p, off in zip(params, self.offsets):
                self.flat_p[off:off + p.numel()].copy_(p.detach().reshape(-1))
                p.data = self.flat_p[off:off + p.numel()].view_as(p)          # the module's parameter IS a view of the bucket
                p.grad = self.flat_g[off:off + p.numel()].view_as(p)
        self.pending = len(params)
        self.work = None


class DataParallelTrainer:
    """One process per GPU.  ``step(loss_fn)``: zero the gradient buckets, run forward + backward (each bucket is all-reduced
    as soon as its last gradient has been accumulated - on NCCL's stream, under the rest of backward), clip by the global norm,
    AdamW - one kernel per bucket, no host synchronisation.  Works unchanged with world size 1 (no process group).

    ``process_group``: default group when torch.distributed is initialised.  With the gloo backend (CPU tests) only the bucket
    logic runs - the fused optimizer kernels need CUDA tensors; pass ``optimizer="torch"`` there."""

    def __init__(self, module, lr: float = 1e-4, betas: Tuple[float, float] = (0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 0.01, max_grad_norm: float = 1.0, bucket_bytes: int = 64 << 20,
                 param_groups: Optional[List[Dict]] = None, process_group=None, optimizer: str = "fused",
                 loss_scale: float = 1.0, ema_decay: Optional[float] = None, ema_update_every_n_steps: int = 1,
                 ema_update_starting_at_step: Optional[int] = None) -> None:
        self.module = module
        # EMA weight averaging = the reference's EMAWeightAveraging callback (src/callbacks/ema_callback.py:414-472 on Lightning's
        # WeightAveraging, :168-197; training_pipeline_ip.py:88-92: decay 0.999, from step 100, every 4th step): after optimizer
        # step number s (1-based) the average is updated when should_update(step_idx = s - 1); the first update copies the
        # parameters (AveragedModel.n_averaged == 0), later ones are avg += (p - avg) * (1 - decay), one kernel per bucket.
        self.ema_decay = ema_decay
        self.ema_every, self.ema_start = int(ema_update_every_n_steps), ema_update_starting_at_step
        self.ema_updates = 0
        self._ema_latest_step = 0
        # fp16 compute needs a loss scale (Lightning "16-mixed" runs a GradScaler): the backward pass sees loss * loss_scale, the
        # clip coefficient folds 1 / loss_scale back in, and a step whose scaled gradients overflowed is skipped on the device
        # (``step_overflowed`` reads the flag; halve ``loss_scale`` then).  bf16 (the default compute dtype) runs at 1.
        # Like GradScaler.step, a skipped step leaves parameters and moments alone and does not advance AdamW's step count t
        # (``optimizer_steps``); ``steps`` counts every step, as Lightning's global_step does, and keys the EMA schedule.
        self.loss_scale = float(loss_scale)
        self.betas, self.eps, self.weight_decay, self.max_grad_norm = betas, eps, weight_decay, max_grad_norm
        self.world = dist.get_world_size(process_group) if dist.is_initialized() else 1
        self.pg = process_group
        self.optimizer = optimizer
        self.base_lr = lr
        groups = parameter_groups(module, lr) if param_groups is None else param_groups
        names = {id(p): n for n, p in module.named_parameters()}
        self.unused = [names.get(id(p), "?") for g in groups for p in g["params"] if names.get(id(p)) in UNUSED_PARAMETERS]
        self.buckets: List[_Bucket] = []
        seen = set()
        for gi, g in enumerate(groups):
            # reverse registration order ~ the order gradients become ready in backward
            ps = [p for p in reversed(g["params"]) if p.requires_grad and names.get(id(p)) not in UNUSED_PARAMETERS and id(p) not in seen]
            seen.update(id(p) for p in ps)
            cur, cur_bytes = [], 0
            for p in ps:
                cur.append(p)
                cur_bytes += p.numel() * 4
                if cur_bytes >= bucket_bytes:
                    self.buckets.append(_Bucket(cur, gi, g["lr"], p.device))
                    cur, cur_bytes = [], 0
            if cur:
                self.buckets.append(_Bucket(cur, gi, g["lr"], cur[0].device))
        self._bucket_of = {}
        for bk in self.buckets:
            for p, off in zip(bk.params, bk.offsets):
                self._bucket_of[id(p)] = (bk, off)
                p.register_post_accumulate_grad_hook(self._on_grad)
        self.steps = 0
        if self.ema_decay is not None:       # AveragedModel(pl_module) at setup: a copy of the initial weights (ema_callback.py:135-166)
            for bk in self.buckets:
                bk.avg = bk.flat_p.clone()
        dev = self.buckets[0].flat_p.device
        self.coef = torch.ones(2, device=dev, dtype=torch.float32)
        self.partials = torch.zeros(len(self.buckets), ops.SUMSQ_PARTIALS, device=dev, dtype=torch.float32)
        self.lr_scale = 1.0
        self._torch_steps = 0                    # AdamW's t on the optimizer="torch" path
        # {lr scale, step number} as the fused AdamW reads them: on the device, advanced in stream order, so that a captured graph
        # of the whole step (``capture``) replays with the right schedule and bias corrections
        self.dev_state = torch.tensor([1.0, 0.0], device=dev, dtype=torch.float32) if dev.type == "cuda" else None
        self._graph = None
        self._reduce_after_backward = False      # capture() with world > 1: the graph holds forward + backward, the all-reduces follow it
        self._skip_allreduce = False             # measurement aid (bench: exposed share of the collective)
        self._capture_events = None              # [(bucket, external event)] in completion order, filled while capturing
        self.overlap_reduce = True               # captured data-parallel step: all-reduce buckets behind their events (else after the graph)
        self._reduce_stream = None

    # ------------------------------------------------------------------ backward-time hooks
    def _on_grad(self, p: nn.Parameter) -> None:
        bk, off = self._bucket_of[id(p)]
        slot_ptr = bk.flat_g.data_ptr() + off * bk.flat_g.element_size()
        if p.grad is not None and p.grad.data_ptr() != slot_ptr:      # autograd replaced the tensor: copy it back into its slot
            slot = bk.flat_g[off:off + p.numel()].view_as(p)
            slot.copy_(p.grad.reshape(slot.shape))
            p.grad = slot
        bk.pending -= 1
        if bk.pending == 0 and self.world > 1:
            if not self._reduce_after_backward:
                bk.work = dist.all_reduce(bk.flat_g, op=dist.ReduceOp.SUM, group=self.pg, async_op=True)
            elif self._capture_events is not None:
                # capturing forward + backward: mark "this bucket is complete" with an EXTERNAL event-record node; after every
                # replay a side stream waits for it and starts the bucket's all-reduce while the graph is still in backward
                ev = torch.cuda.Event(external=True)
                ev.record()
                self._capture_events.append((bk, ev))

    def zero_grad(self) -> None:
        for bk in self.buckets:
            bk.flat_g.zero_()
            bk.pending = len(bk.params)
            bk.work = None
            for p, off in zip(bk.params, bk.offsets):
                if p.grad is None or p.grad.data_ptr() != bk.flat_g.data_ptr() + off * bk.flat_g.element_size():
                    p.grad = bk.flat_g[off:off + p.numel()].view_as(p)

    def finish_reduce(self) -> None:
        """Wait for the bucket all-reduces; a bucket whose gradients did not all arrive breaks the ``find_unused_parameters=False``
        contract (the reference would hang or raise in DDP)."""
        late = [bk for bk in self.buckets if bk.pending != 0]
        if late:
            names = {id(p): n for n, p in self.module.named_parameters()}
            missing = [names.get(id(p), "?") for bk in late for p in bk.params][:5]
            raise RuntimeError(f"{sum(bk.pending for bk in late)} bucketed parameter(s) received no gradient (e.g. {missing}): "
                               "every trainable parameter outside UNUSED_PARAMETERS must take part in the loss")
        for bk in self.buckets:
            if bk.work is not None:
                bk.work.wait()
                bk.work = None

    # ------------------------------------------------------------------ optimizer
    def optimizer_step(self) -> None:
        self.steps += 1
        b1, b2 = self.betas
        inv_world = 1.0 / (self.world * self.loss_scale)
        if self.optimizer == "fused":
            for i, bk in enumerate(self.buckets):
                ops.sumsq_(bk.flat_g, self.partials[i])
            ops.clip_coef_(self.partials.view(-1), self.max_grad_norm, inv_world, self.coef)
            # the step number, in stream order (captured with the step): advanced only when the update will be applied
            self.dev_state[1:2].add_(torch.isfinite(self.coef[:1]))
            for bk in self.buckets:
                if bk.m is None:
                    bk.m, bk.v = torch.zeros_like(bk.flat_p), torch.zeros_like(bk.flat_p)
                ops.adamw_step_dev_(bk.flat_p, bk.flat_g, bk.m, bk.v, bk.lr, b1, b2, self.eps, self.weight_decay, self.dev_state,
                                    self.coef)
        else:       # reference arithmetic with stock PyTorch (CPU / gloo tests of the bucket logic)
            total = torch.sqrt(sum((bk.flat_g * inv_world).pow(2).sum() for bk in self.buckets))
            applied = bool(torch.isfinite(total))         # the fused path's rule: a non-finite norm skips the step
            coef = inv_world * (torch.clamp(self.max_grad_norm / (total + 1e-6), max=1.0) if self.max_grad_norm > 0 else 1.0)
            self.coef = torch.stack([torch.as_tensor(coef if applied else math.nan, dtype=torch.float32, device=total.device),
                                     total.float()])
            for bk in self.buckets:
                if bk.m is None:
                    bk.m, bk.v = torch.zeros_like(bk.flat_p), torch.zeros_like(bk.flat_p)
            if applied:
                self._torch_steps += 1
                t = self._torch_steps
                for bk in self.buckets:
                    g = bk.flat_g * coef
                    lr = bk.lr * self.lr_scale
                    bk.flat_p.mul_(1.0 - lr * self.weight_decay)
                    bk.m.mul_(b1).add_(g, alpha=1.0 - b1)
                    bk.v.mul_(b2).addcmul_(g, g, value=1.0 - b2)
                    denom = (bk.v.sqrt() / math.sqrt(1.0 - b2 ** t)).add_(self.eps)
                    bk.flat_p.addcdiv_(bk.m, denom, value=-lr / (1.0 - b1 ** t))
        wcache.clear()        # inference-time derived weights (16-bit / fused copies) are stale after an in-place update
        if self.ema_decay is not None and self.ema_should_update(self.steps - 1):
            self.ema_update()

    # ------------------------------------------------------------------ EMA weight averaging
    def ema_should_update(self, step_idx: int) -> bool:
        """EMAWeightAveraging.should_update(step_idx=...) (ema_callback.py:438-472), step conditions only."""
        meets_start = self.ema_start is None or step_idx >= self.ema_start
        meets_frequency = self.ema_every > 0 and step_idx % self.ema_every == 0
        return meets_start and meets_frequency

    def ema_update(self) -> None:
        first = self.ema_updates == 0
        for bk in self.buckets:
            if self.optimizer == "fused":
                ops.ema_update_(bk.avg, bk.flat_p, self.ema_decay, first)
            elif first:
                bk.avg.copy_(bk.flat_p)
            else:
                bk.avg.lerp_(bk.flat_p, 1.0 - self.ema_decay)              # torch.optim.swa_utils.get_ema_avg_fn
        self.ema_updates += 1
        self._ema_latest_step = self.steps

    def ema_state_dict(self) -> Dict[str, torch.Tensor]:
        """The module's state dict with every trained parameter replaced by its average: what the callback writes as
        ``checkpoint["state_dict"]`` (ema_callback.py:316-323).  Frozen / never-used parameters and buffers are constants of the
        run, so their average is their value.  Before the first update the average model holds the initial weights (:135-166)."""
        assert self.ema_decay is not None, "the trainer was built without ema_decay"
        sd = {k: v.detach().clone() for k, v in self.module.state_dict().items()}
        names = {id(p): n for n, p in self.module.named_parameters()}
        for bk in self.buckets:
            for p, off in zip(bk.params, bk.offsets):
                sd[names[id(p)]] = bk.avg[off:off + p.numel()].view_as(p).clone()
        return sd

    def swap_ema_weights(self) -> None:
        """Exchange the parameters with their averages in place (the callback's ``_swap_models`` around validation,
        ema_callback.py:235-265,379-395); call again to swap back."""
        assert self.ema_decay is not None, "the trainer was built without ema_decay"
        for bk in self.buckets:
            tmp = bk.flat_p.clone()
            bk.flat_p.copy_(bk.avg)
            bk.avg.copy_(tmp)
        wcache.clear()

    def copy_ema_to_model(self) -> None:
        """End of training: the module takes the averaged weights (``_copy_average_to_current``, ema_callback.py:219-233,397-411)."""
        assert self.ema_decay is not None, "the trainer was built without ema_decay"
        for bk in self.buckets:
            bk.flat_p.copy_(bk.avg)
        wcache.clear()

    # ------------------------------------------------------------------ checkpoints in the reference's layout
    def checkpoint(self, epoch: int = 0) -> Dict:
        """The dictionary Lightning + the EMA callback write (ema_callback.py:291-330): ``state_dict`` = averaged weights (what
        ``load_from_checkpoint`` and the inference / evaluation pipelines read), ``current_model_state`` = the weights training
        continues from, ``averaging_state`` = AveragedModel's own entries (``n_averaged``), the callback's ``latest_update_step``
        and the optimizer moments per bucket (bucket order: resume with the same ``bucket_bytes`` / parameter groups) with AdamW's
        step count (``optimizer_step``: below ``global_step`` once a step has been skipped).  Without EMA: ``state_dict`` = the
        current weights."""
        cur = {k: v.detach().clone() for k, v in self.module.state_dict().items()}
        ck = {"epoch": int(epoch), "global_step": int(self.steps), "state_dict": cur,
              "optimizer_moments": [None if bk.m is None else (bk.m.clone(), bk.v.clone()) for bk in self.buckets],
              "optimizer_step": self.optimizer_steps}
        if self.ema_decay is not None:
            ck["state_dict"] = self.ema_state_dict()
            ck["current_model_state"] = cur
            ck["averaging_state"] = {"n_averaged": torch.tensor(self.ema_updates, dtype=torch.long)}
            ck["callbacks"] = {"EMAWeightAveraging": {"latest_update_step": int(self._ema_latest_step)}}
        return ck

    def load_checkpoint(self, ck: Dict) -> None:
        """Resume: the module takes ``current_model_state`` and the averages come from ``state_dict`` (on_load_checkpoint,
        ema_callback.py:332-378); a checkpoint written without EMA initialises both from ``state_dict``.  A checkpoint without
        ``optimizer_step`` (written before skipped steps were told apart) resumes AdamW's step count from ``global_step``."""
        names = {id(p): n for n, p in self.module.named_parameters()}
        self.module.load_state_dict(ck.get("current_model_state", ck["state_dict"]), strict=False)     # copies into the bucket views
        self.steps = int(ck.get("global_step", 0))
        self._torch_steps = int(ck.get("optimizer_step", self.steps))
        if self.dev_state is not None:
            self.dev_state[1:2].fill_(float(self._torch_steps))
        if self.ema_decay is not None:
            for bk in self.buckets:
                for p, off in zip(bk.params, bk.offsets):
                    bk.avg[off:off + p.numel()].copy_(ck["state_dict"][names[id(p)]].reshape(-1))
            self.ema_updates = int(ck["averaging_state"]["n_averaged"]) if "averaging_state" in ck else 0
            self._ema_latest_step = int(ck.get("callbacks", {}).get("EMAWeightAveraging", {}).get("latest_update_step", 0))
        for bk, mom in zip(self.buckets, ck.get("optimizer_moments", [])):
            if mom is not None:
                bk.m, bk.v = mom[0].to(bk.flat_p.device).clone(), mom[1].to(bk.flat_p.device).clone()
        wcache.clear()

    def set_epoch_lr(self, epoch: int, warmup_epochs: int, max_epochs: int, min_lr: float) -> None:
        """Per-epoch LinearWarmupCosineAnnealingLR (diffusion_module_ip.py:521-527), applied as a scale on every group's lr."""
        lr = warmup_cosine_lr(epoch, self.base_lr, warmup_epochs, max_epochs, self.base_lr * 0.01, min_lr)
        self.lr_scale = lr / self.base_lr
        if self.dev_state is not None:
            self.dev_state[0:1].fill_(self.lr_scale)

    def step(self, loss_fn) -> torch.Tensor:
        self.zero_grad()
        loss = loss_fn()
        (loss if self.loss_scale == 1.0 else loss * self.loss_scale).backward()
        self.finish_reduce()
        self.optimizer_step()
        return loss.detach()

    def capture(self, loss_fn, generators=(), warmup: int = 2):
        """Capture the step as a CUDA graph and return ``replay() -> loss``.  At batch 8 per GPU the eager step is bound by the host
        (5 700 launches behind Python autograd; the kernels add up to half of its wall time); a replay is one launch.
          * one process (world size 1): ONE graph holds gradient-bucket zeroing, forward, backward, clip and AdamW;
          * data parallel: the graph holds zeroing + forward + backward; ``replay`` then all-reduces the buckets (NCCL, eager: a
            capture that includes the hook-launched all-reduces deadlocked against ProcessGroupNCCL's watchdog on this stack,
            torch 2.11 / NCCL 2.28) and runs the fused clip + AdamW kernels.  The hooks leave an external event-record node
            behind every completed bucket; ``replay`` makes a side stream wait for each event and start that bucket's all-reduce,
            so the collectives still run under the rest of the captured backward (``overlap_reduce = False``: after the graph).
        ``loss_fn`` must read its inputs from tensors that keep their address (copy each batch into them before ``replay()``) and
        draw its random numbers from the default CUDA generator or from ``generators`` (registered with the graph).  ``warmup``
        eager steps run first (they are real optimizer steps): cuDNN / cuBLAS plans, the allocator, NCCL.  The step number and the
        learning-rate scale live on the device (``dadd_adamw_step_dev``); EMA updates are issued by ``replay`` on the reference
        callback's schedule.  All ranks must capture and replay together.  The tensor ``replay`` returns is the graph's own loss
        buffer: the next replay overwrites it (``.item()`` / ``.clone()`` it to keep a value)."""
        assert self.optimizer == "fused" and self.dev_state is not None, "graph capture needs the fused CUDA optimizer"
        dev = self.buckets[0].flat_p.device
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self.step(loss_fn)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        for bk in self.buckets:                      # (moments exist before the capture: no allocation inside the graph's optimizer)
            if bk.m is None:
                bk.m, bk.v = torch.zeros_like(bk.flat_p), torch.zeros_like(bk.flat_p)
        graph = torch.cuda.CUDAGraph()
        for gen in generators:
            graph.register_generator_state(gen)
        whole = self.world == 1
        ema_decay, self.ema_decay = self.ema_decay, None      # the host-side EMA decision stays out of the captured step
        steps_before = self.steps
        self._reduce_after_backward = not whole
        self._capture_events = [] if not whole else None
        if not whole:                                 # no collective in flight while capturing (ProcessGroupNCCL's watchdog polls events)
            dist.barrier(group=self.pg)
            torch.cuda.synchronize(dev)
        try:
            with torch.cuda.graph(graph, capture_error_mode="global" if whole else "thread_local"):
                if whole:
                    loss = self.step(loss_fn)
                else:
                    self.zero_grad()
                    loss = loss_fn()
                    (loss if self.loss_scale == 1.0 else loss * self.loss_scale).backward()
                    loss = loss.detach()
        finally:
            self.ema_decay = ema_decay
            self.steps = steps_before                 # capturing executes nothing: the step is counted when it is replayed
            self._reduce_after_backward = False       # (hooks do not run on replay; an eager step() after this reduces as before)
        self._graph, self._graph_loss = graph, loss
        events, self._capture_events = self._capture_events, None
        if not whole:
            assert len(events) == len(self.buckets), "a gradient bucket never completed during the captured backward"
            self._reduce_stream = torch.cuda.Stream(device=dev)

        self._replays = 0

        def replay() -> torch.Tensor:
            graph.replay()
            if whole:
                self.steps += 1
                wcache.clear()
                if self.ema_decay is not None and self.ema_should_update(self.steps - 1):
                    self.ema_update()
            else:
                if not self._skip_allreduce:
                    works = []
                    # (the first replay reduces after the graph: its event nodes have never been recorded before this launch)
                    if self.overlap_reduce and self._replays > 0:
                        for bk, ev in events:         # completion order of the captured backward
                            self._reduce_stream.wait_event(ev)
                            with torch.cuda.stream(self._reduce_stream):
                                works.append(dist.all_reduce(bk.flat_g, op=dist.ReduceOp.SUM, group=self.pg, async_op=True))
                    else:
                        works = [dist.all_reduce(bk.flat_g, op=dist.ReduceOp.SUM, group=self.pg, async_op=True) for bk in self.buckets]
                    for w in works:
                        w.wait()
                self.optimizer_step()                 # (eager: ~90 launches; counts the step, clears caches, EMA)
            self._replays += 1
            return self._graph_loss

        return replay

    @property
    def grad_norm(self) -> torch.Tensor:
        return self.coef[1]

    @property
    def optimizer_steps(self) -> int:
        """AdamW's step count t (``state["step"]`` of torch.optim.AdamW): the updates applied, skipped steps excluded.  The fused
        optimizer keeps it on the device: reading it synchronises."""
        return int(self.dev_state[1].item()) if self.optimizer == "fused" else self._torch_steps

    def step_overflowed(self) -> bool:
        """True when the last step was skipped because its (loss-scaled) gradients were not finite.  Synchronises."""
        return not bool(torch.isfinite(self.coef[0]).item())
