"""Seeded inputs shared by ``make_golden.py`` (which runs the verbatim reference on them) and the tests."""

from __future__ import annotations

import torch

from oracle import weights

PROCESSOR_CASES = [
    dict(name="split_d40_l3", kind="split", c=320, n=64, b=2, gates=(0.1, 0.9), delta_scale=3.0, seed=11),
    dict(name="split_d40_l0", kind="split", c=320, n=64, b=2, gates=(0.1, 0.9), delta_scale=0.0, seed=12),
    dict(name="split_d80_l1", kind="split", c=640, n=48, b=1, gates=(0.9, 0.1), delta_scale=1.0, seed=13),
    dict(name="split_d160_l3", kind="split", c=1280, n=16, b=2, gates=(0.5, 0.5), delta_scale=3.0, seed=14),
    dict(name="base_d40_both", kind="base", c=320, n=64, b=2, mode="both", seed=15),
    dict(name="base_d80_img", kind="base", c=640, n=32, b=1, mode="image_dominant", seed=16),
    dict(name="base_d160_aoe", kind="base", c=1280, n=16, b=1, mode="aoe_dominant", seed=17),
    # N >= 128: the tcgen05 cross-attention kernel (full tiles, a ragged last tile, 2 / 3 segments, one 32-token segment)
    dict(name="split_d40_n256_l3", kind="split", c=320, n=256, b=1, gates=(0.1, 0.9), delta_scale=3.0, seed=18),
    dict(name="split_d80_n136_l3", kind="split", c=640, n=136, b=1, gates=(0.9, 0.1), delta_scale=2.0, seed=19),
    dict(name="split_d40_n128_l0", kind="split", c=320, n=128, b=1, gates=(0.3, 0.7), delta_scale=0.0, seed=20),
    dict(name="base_d40_n192_both", kind="base", c=320, n=192, b=1, mode="both", seed=21),
]


def processor_inputs(case):
    g = torch.Generator().manual_seed(case["seed"])
    it = weights._Init(case["seed"] + 1000, 1.7, 0.0)     # gain > 1 so the softmaxes are not flat
    c = case["c"]
    it.linear("to_q", c, c, bias=False)
    it.linear("to_k", 768, c, bias=False)
    it.linear("to_v", 768, c, bias=False)
    it.linear("to_out.0", c, c)
    if case["kind"] == "split":
        it.linear("processor.to_k_dis", 768, c, bias=False)
        it.linear("processor.to_v_dis", 768, c, bias=False)
        it.sd["processor.anat_gate"] = torch.tensor(float(case["gates"][0]))
        it.sd["processor.dis_gate"] = torch.tensor(float(case["gates"][1]))
    x = 2.0 * torch.randn(case["b"], case["n"], c, generator=g)
    tokens = 48 if case["kind"] == "split" else 32
    ehs = 2.0 * torch.randn(case["b"], tokens, 768, generator=g)
    return it.sd, x, ehs


def cross_attention_processor_names():
    return [f"{p}.transformer_blocks.0.attn2.processor" for p, _ in weights.attention_sites()]


def purifier_inputs():
    g = torch.Generator().manual_seed(21)
    w = weights.make_purifier_state(seed=22)
    return w, torch.randn(3, 16, 768, generator=g), torch.randn(3, 16, 768, generator=g)


def aoe_inputs():
    w = weights.make_aoe_state(seed=23)
    labels = torch.cat([torch.linspace(0, 3, 13), torch.tensor([-0.5, 3.7, 2.999, 1.0])])
    src = torch.full_like(labels, 2.0)
    return w, labels, src


# ---- conditioning front end (CLIP vision tower + resamplers), SURVEY.md 8f row f3 --------------------------------------
def clip_inputs(kind: str):
    """(dims, seeded CLIPVisionModelWithProjection state dict, seeded pixels): ``tiny`` is CPU-sized, ``l14`` is ViT-L/14."""
    from oracle import image_front_end as fe
    dims = fe.CLIP_TINY if kind == "tiny" else fe.CLIP_L14
    w = weights.make_clip_vision_state(seed=5 if kind == "l14" else 7, **dims)
    g = torch.Generator().manual_seed(31 if kind == "l14" else 32)
    pixels = torch.randn(2, 3, dims["image"], dims["image"], generator=g)            # CLIP-normalised pixels are ~N(0, 1)
    return dims, w, pixels


def clip_l14_hidden():
    """The resamplers' input: ViT-L/14 last hidden states on ``clip_inputs("l14")``, from the oracle tower.  The golden file
    keeps only a sample of the transformers tower's states, which this reproduces to ~1e-6 relative."""
    from oracle import image_front_end as fe
    dims, w, pixels = clip_inputs("l14")
    with torch.no_grad():
        return fe.clip_hidden_states(w, pixels, dims["heads"], dims["patch"])[0]


def projection_plus_inputs():
    return weights.make_projection_plus_state(seed=6)


def projection_basic_inputs():
    it = weights._Init(8, 1.0, 0.1)
    it.linear("projection", 768, 768 * 4)
    it.norm("norm", 768)
    g = torch.Generator().manual_seed(33)
    return it.sd, torch.randn(3, 768, generator=g)
