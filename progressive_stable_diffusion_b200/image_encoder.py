"""Conditioning front end for B200: CLIP vision tower -> ``ImageProjection`` / ``ImageProjectionPlus`` -> anatomy tokens.

Mirrors ``/root/reference/src/models/image_encoder.py`` (``ImageEncoder`` :17-88, ``ImageProjection`` :91-133,
``ImageProjectionPlus`` :136-228; SURVEY.md 8f row f3): same class names, constructor arguments, parameter names and
state-dict keys (``image_encoder.vision_model.*`` / ``image_encoder.visual_projection.weight`` are the keys of transformers'
``CLIPVisionModelWithProjection``, so a Lightning checkpoint of the reference loads as is).  There is no network here, so
``ImageEncoder`` builds the architecture named by ``pretrained_path`` (ViT-L/14 or ViT-B/16) with random weights instead of
downloading them; real weights arrive through ``load_state_dict``.

Execution: 16-bit activations; LayerNorm, residual-add + LayerNorm, the self-attention core (``dadd_self_attn_fwd``: N = 257,
d = 64 runs the tcgen05 kernel), ``quick_gelu`` and the resampler's attention core are this package's kernels; the GEMMs go
through ``ops.linear``; the one patch-embedding convolution is cuDNN.  The front end runs once per sampling call.
"""

from __future__ import annotations

from types import SimpleNamespace
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops, wcache
from .attention_processor import compute_dtype

_ARCH = {   # pretrained_path suffix -> (hidden, intermediate, layers, heads, image, patch, projection)
    "clip-vit-large-patch14": (1024, 4096, 24, 16, 224, 14, 768),
    "clip-vit-large-patch14-336": (1024, 4096, 24, 16, 336, 14, 768),      # CMMD's embedding (metrics.ClipEmbedder)
    "clip-vit-base-patch16": (768, 3072, 12, 12, 224, 16, 512),
    "clip-vit-base-patch32": (768, 3072, 12, 12, 224, 32, 512),
}


def _f32(mod, tag: str, p: torch.Tensor) -> torch.Tensor:
    return wcache.cast(mod, tag, p, torch.float32)


def _w16(mod: nn.Linear) -> torch.Tensor:
    return wcache.cast(mod, "w", mod.weight, compute_dtype())


def _lin16(mod: nn.Linear, x: torch.Tensor, residual: Optional[torch.Tensor] = None) -> torch.Tensor:
    bias = None if mod.bias is None else _f32(mod, "b32", mod.bias)
    bias_lp = None if mod.bias is None else wcache.cast(mod, "b", mod.bias, compute_dtype())
    return ops.linear(x, _w16(mod), bias, residual, bias_lp=bias_lp)


def _ln16(mod: nn.LayerNorm, x: torch.Tensor) -> torch.Tensor:
    return ops.layer_norm(x, _f32(mod, "w", mod.weight), _f32(mod, "b", mod.bias), mod.eps)


class _Container(nn.Module):
    """Attribute bag that registers sub-modules / parameters under the names transformers uses."""


class _CLIPVisionTower(nn.Module):
    """Parameter layout of transformers' ``CLIPVisionModelWithProjection`` with a B200 forward."""

    def __init__(self, hidden: int, inter: int, layers: int, heads: int, image: int, patch: int, proj: int) -> None:
        super().__init__()
        self.config = SimpleNamespace(hidden_size=hidden, intermediate_size=inter, num_hidden_layers=layers,
                                      num_attention_heads=heads, image_size=image, patch_size=patch, projection_dim=proj,
                                      hidden_act="quick_gelu", layer_norm_eps=1e-5)
        vm = _Container()
        emb = _Container()
        emb.class_embedding = nn.Parameter(torch.randn(hidden))
        emb.patch_embedding = nn.Conv2d(3, hidden, patch, stride=patch, bias=False)
        emb.position_embedding = nn.Embedding((image // patch) ** 2 + 1, hidden)
        vm.embeddings = emb
        vm.pre_layrnorm = nn.LayerNorm(hidden, eps=1e-5)            # (sic: transformers' spelling, part of the checkpoint keys)
        enc = _Container()
        enc.layers = nn.ModuleList()
        for _ in range(layers):
            lyr = _Container()
            attn = _Container()
            for name in ("k_proj", "v_proj", "q_proj", "out_proj"):
                setattr(attn, name, nn.Linear(hidden, hidden))
            lyr.self_attn = attn
            lyr.layer_norm1 = nn.LayerNorm(hidden, eps=1e-5)
            mlp = _Container()
            mlp.fc1 = nn.Linear(hidden, inter)
            mlp.fc2 = nn.Linear(inter, hidden)
            lyr.mlp = mlp
            lyr.layer_norm2 = nn.LayerNorm(hidden, eps=1e-5)
            enc.layers.append(lyr)
        vm.encoder = enc
        vm.post_layernorm = nn.LayerNorm(hidden, eps=1e-5)
        self.vision_model = vm
        self.visual_projection = nn.Linear(hidden, proj, bias=False)

    def _qkv(self, attn) -> tuple:
        srcw = (attn.q_proj.weight, attn.k_proj.weight, attn.v_proj.weight)
        srcb = (attn.q_proj.bias, attn.k_proj.bias, attn.v_proj.bias)
        w = wcache.get(attn, "wqkv", srcw, lambda: torch.cat([p.detach() for p in srcw], 0).to(compute_dtype()).contiguous())
        b32 = wcache.get(attn, "bqkv32", srcb, lambda: torch.cat([p.detach() for p in srcb], 0).float().contiguous())
        blp = wcache.get(attn, "bqkv", srcb, lambda: torch.cat([p.detach() for p in srcb], 0).to(compute_dtype()).contiguous())
        return w, b32, blp

    @torch.no_grad()
    def forward(self, pixel_values: torch.Tensor, output_hidden_states: bool = True):
        """-> namespace(image_embeds (B, proj) fp32, last_hidden (B, 1 + patches, hidden) fp32 = ``hidden_states[-1]``)."""
        cfg, vm = self.config, self.vision_model
        dt = compute_dtype()
        emb = vm.embeddings
        w = wcache.conv_filter(emb.patch_embedding, "w", emb.patch_embedding.weight, dt)
        x = F.conv2d(pixel_values.to(dt).contiguous(memory_format=torch.channels_last), w, None, stride=cfg.patch_size)
        b, c = x.shape[:2]
        x = x.permute(0, 2, 3, 1).reshape(b, -1, c)                  # channels-last conv output: a free view
        x = torch.cat([emb.class_embedding.detach().to(dt).expand(b, 1, c), x], dim=1)
        x = (x.float() + emb.position_embedding.weight.detach().float()[None]).to(dt).contiguous()
        x = _ln16(vm.pre_layrnorm, x)
        heads = cfg.num_attention_heads
        h = _ln16(vm.encoder.layers[0].layer_norm1, x)
        for i, lyr in enumerate(vm.encoder.layers):
            wqkv, b32, blp = self._qkv(lyr.self_attn)
            qkv = ops.linear(h, wqkv, b32, bias_lp=blp)
            o = ops.self_attention(qkv[..., :c], qkv[..., c:2 * c], qkv[..., 2 * c:], heads)
            # x += out_proj(o); h = LN2(x) in one pass
            x, h = ops.add_layer_norm(x, _lin16(lyr.self_attn.out_proj, o), _f32(lyr.layer_norm2, "w", lyr.layer_norm2.weight),
                                      _f32(lyr.layer_norm2, "b", lyr.layer_norm2.bias), lyr.layer_norm2.eps)
            x = _lin16(lyr.mlp.fc2, ops.quick_gelu_(_lin16(lyr.mlp.fc1, h)), residual=x)
            if i + 1 < len(vm.encoder.layers):
                h = _ln16(vm.encoder.layers[i + 1].layer_norm1, x)
        pooled = F.layer_norm(x[:, 0].float(), (c,), vm.post_layernorm.weight.float(), vm.post_layernorm.bias.float(), 1e-5)
        embeds = F.linear(pooled, self.visual_projection.weight.float())
        return SimpleNamespace(image_embeds=embeds, last_hidden=x.float(), hidden_states=(x.float(),))


class ImageEncoder(nn.Module):
    """Frozen CLIP vision encoder (reference :17-88)."""

    def __init__(self, pretrained_path: str = "openai/clip-vit-base-patch16", torch_dtype: torch.dtype = torch.float32,
                 local_files_only: bool = False) -> None:
        super().__init__()
        key = pretrained_path.rstrip("/").split("/")[-1]
        if key not in _ARCH:
            raise ValueError(f"unknown CLIP vision architecture {pretrained_path!r}: known are {sorted(_ARCH)}")
        self.image_encoder = _CLIPVisionTower(*_ARCH[key]).to(torch_dtype)
        self.image_processor = None      # CLIPImageProcessor is host-side preprocessing: callers pass preprocessed pixels
        self.image_encoder.requires_grad_(False)
        self.image_encoder.eval()
        self.hidden_size = self.image_encoder.config.hidden_size
        self.projection_dim = self.image_encoder.config.projection_dim

    @torch.no_grad()
    def forward(self, clip_images: torch.Tensor) -> torch.Tensor:
        """(B, 3, 224, 224) CLIP-preprocessed pixels -> projected image embedding (B, projection_dim) (reference :53-68)."""
        return self.image_encoder(pixel_values=clip_images, output_hidden_states=True).image_embeds

    @torch.no_grad()
    def get_hidden_states(self, clip_images: torch.Tensor) -> torch.Tensor:
        """-> (B, 257, hidden): the last encoder layer's output, CLS + patches (reference :70-87)."""
        return self.image_encoder(pixel_values=clip_images, output_hidden_states=True).hidden_states[-1]


class ImageProjection(nn.Module):
    """CLIP embedding -> ``num_tokens`` cross-attention tokens (reference :91-133)."""

    def __init__(self, clip_embedding_dim: int = 512, cross_attention_dim: int = 768, num_tokens: int = 4) -> None:
        super().__init__()
        self.num_tokens = num_tokens
        self.cross_attention_dim = cross_attention_dim
        self.projection = nn.Linear(clip_embedding_dim, cross_attention_dim * num_tokens)
        self.norm = nn.LayerNorm(cross_attention_dim)

    def forward(self, image_embeds: torch.Tensor) -> torch.Tensor:
        e = F.linear(image_embeds.float(), _f32(self.projection, "w", self.projection.weight), _f32(self.projection, "b", self.projection.bias))
        e = e.reshape(-1, self.num_tokens, self.cross_attention_dim).contiguous()
        return ops.layer_norm(e, _f32(self.norm, "w", self.norm.weight), _f32(self.norm, "b", self.norm.bias), self.norm.eps)


class ImageProjectionPlus(nn.Module):
    """Perceiver resampler over the CLIP patch tokens (reference :136-228), fp32 (16 query tokens per image)."""

    def __init__(self, clip_hidden_dim: int = 768, cross_attention_dim: int = 768, num_tokens: int = 16, num_heads: int = 8,
                 depth: int = 2) -> None:
        super().__init__()
        self.num_tokens = num_tokens
        self.cross_attention_dim = cross_attention_dim
        self.num_heads = num_heads
        self.latents = nn.Parameter(torch.randn(1, num_tokens, cross_attention_dim) * 0.02)
        self.proj_in = nn.Linear(clip_hidden_dim, cross_attention_dim) if clip_hidden_dim != cross_attention_dim else nn.Identity()
        self.layers = nn.ModuleList([
            nn.ModuleDict({
                "cross_attn": nn.MultiheadAttention(cross_attention_dim, num_heads, batch_first=True),
                "ff": nn.Sequential(nn.Linear(cross_attention_dim, cross_attention_dim * 4), nn.GELU(),
                                    nn.Linear(cross_attention_dim * 4, cross_attention_dim)),
                "norm1": nn.LayerNorm(cross_attention_dim),
                "norm2": nn.LayerNorm(cross_attention_dim),
            }) for _ in range(depth)])
        self.norm_out = nn.LayerNorm(cross_attention_dim)

    def _ln(self, mod: nn.LayerNorm, x: torch.Tensor) -> torch.Tensor:
        return ops.layer_norm(x.contiguous(), _f32(mod, "w", mod.weight), _f32(mod, "b", mod.bias), mod.eps)

    def forward(self, hidden_states: torch.Tensor) -> torch.Tensor:
        b = hidden_states.shape[0]
        d = self.cross_attention_dim
        hs = hidden_states.float()
        if isinstance(self.proj_in, nn.Linear):
            hs = F.linear(hs, _f32(self.proj_in, "w", self.proj_in.weight), _f32(self.proj_in, "b", self.proj_in.bias))
        lat = self.latents.detach().float().expand(b, -1, -1).contiguous()
        for layer in self.layers:
            mha = layer["cross_attn"]
            wi, bi = _f32(mha, "wi", mha.in_proj_weight), _f32(mha, "bi", mha.in_proj_bias)
            q = F.linear(self._ln(layer["norm1"], lat), wi[:d], bi[:d])
            kv = F.linear(hs, wi[d:], bi[d:])                       # K and V of the patches in one GEMM
            core = ops.purifier_attention(q.contiguous(), kv[..., :d].contiguous(), kv[..., d:].contiguous(), self.num_heads)
            lat = lat + F.linear(core, _f32(mha.out_proj, "w", mha.out_proj.weight), _f32(mha.out_proj, "b", mha.out_proj.bias))
            ff0, ff2 = layer["ff"][0], layer["ff"][2]
            x = F.gelu(F.linear(self._ln(layer["norm2"], lat), _f32(ff0, "w", ff0.weight), _f32(ff0, "b", ff0.bias)))
            lat = lat + F.linear(x, _f32(ff2, "w", ff2.weight), _f32(ff2, "b", ff2.bias))
        return self._ln(self.norm_out, lat)
