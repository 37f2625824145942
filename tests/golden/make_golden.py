"""Generate golden vectors by running the VERBATIM reference modules of the original project.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py <checkout of umutdundar99/progressive-stable-diffusion>

Imports ``src.models.{feature_purifier,ordinal_embedder,attention_processor_routing_gates,attention_processor_base}``
from that checkout (a 3-line ``sys.modules`` shim stands in for the absent ``diffusers`` import, which those files use
only to name ``AttnProcessor2_0``), loads the seeded weights of ``oracle/weights.py`` into them, runs them on the seeded
inputs of ``tests/golden/cases.py`` and stores the OUTPUTS as fp32 ``.npz`` next to this file, in the sampled format of
``tests/golden/store.py``.  The tests only read the committed ``.npz`` files.
"""

from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "src", "models")):
    sys.exit(__doc__)
sys.path.insert(0, os.path.abspath(sys.argv[1]))
sys.dont_write_bytecode = True

# shim: the processor files do ``from diffusers.models.attention_processor import AttnProcessor2_0``
_d = types.ModuleType("diffusers")
_dm = types.ModuleType("diffusers.models")
_da = types.ModuleType("diffusers.models.attention_processor")
_da.AttnProcessor2_0 = type("AttnProcessor2_0", (), {})
sys.modules.update({"diffusers": _d, "diffusers.models": _dm, "diffusers.models.attention_processor": _da})

from src.models.attention_processor_base import OrdinalIPAttnProcessor2_0, get_frequency_mode_for_block  # noqa: E402
from src.models.attention_processor_routing_gates import SplitInjectionAttentionProcessor, get_block_type  # noqa: E402
from src.models.feature_purifier import FeaturePurifier  # noqa: E402
from src.models.ordinal_embedder import AdditiveOrdinalEmbedder  # noqa: E402

from tests.golden import cases  # noqa: E402
from tests.golden.store import pack  # noqa: E402


class _StubAttn(torch.nn.Module):
    """The fields of diffusers' ``Attention`` the processors read (SURVEY.md section 8b)."""

    def __init__(self, w, c, heads=8):
        super().__init__()
        self.heads = heads
        self.spatial_norm = None
        self.group_norm = None
        self.norm_cross = None
        self.residual_connection = False
        self.rescale_output_factor = 1.0
        self.to_q = torch.nn.Linear(c, c, bias=False)
        self.to_k = torch.nn.Linear(768, c, bias=False)
        self.to_v = torch.nn.Linear(768, c, bias=False)
        self.to_out = torch.nn.ModuleList([torch.nn.Linear(c, c), torch.nn.Dropout(0.0)])
        with torch.no_grad():
            self.to_q.weight.copy_(w["to_q.weight"])
            self.to_k.weight.copy_(w["to_k.weight"])
            self.to_v.weight.copy_(w["to_v.weight"])
            self.to_out[0].weight.copy_(w["to_out.0.weight"])
            self.to_out[0].bias.copy_(w["to_out.0.bias"])


@torch.no_grad()
def main() -> None:
    out = {}
    # ---- routing processor -------------------------------------------------------------------------------
    for case in cases.PROCESSOR_CASES:
        w, x, ehs = cases.processor_inputs(case)
        attn = _StubAttn(w, case["c"])
        if case["kind"] == "split":
            proc = SplitInjectionAttentionProcessor(case["c"], 768, 16, 16, 16, "both",
                                                    case["gates"][0], case["gates"][1], case["delta_scale"])
            proc.to_k_dis.weight.copy_(w["processor.to_k_dis.weight"])
            proc.to_v_dis.weight.copy_(w["processor.to_v_dis.weight"])
        else:
            proc = OrdinalIPAttnProcessor2_0(case["c"], 768, 16, 16, case["mode"])
        out["processor_" + case["name"]] = proc(attn, x, ehs).numpy()
    # ---- role maps ---------------------------------------------------------------------------------------
    names = cases.cross_attention_processor_names()
    out["roles"] = np.array([get_block_type(n) for n in names])
    out["freq_modes"] = np.array([get_frequency_mode_for_block(n) for n in names])
    # ---- purifier ----------------------------------------------------------------------------------------
    pw, img, aoe = cases.purifier_inputs()
    pur = FeaturePurifier(768, 8, 2)
    pur.load_state_dict(pw)
    out["purifier"] = pur(img, aoe).numpy()
    # ---- AOE ---------------------------------------------------------------------------------------------
    aw, labels, src = cases.aoe_inputs()
    emb = AdditiveOrdinalEmbedder(4, 768, delta_scale=0.05, num_tokens=16)
    emb.load_state_dict(aw)
    out["aoe_forward"] = emb(labels, is_training=False).numpy()
    out["aoe_negative"] = emb.get_negative_embedding(labels).numpy()
    out["aoe_delta"] = emb.get_ordinal_delta_embedding(src, labels).numpy()
    out["aoe_delta_same"] = emb.get_ordinal_delta_embedding(labels, labels).numpy()
    out["aoe_table"] = emb._compute_class_table().numpy()
    np.savez_compressed(os.path.join(HERE, "reference_modules.npz"), **pack(out))
    for k, v in out.items():
        print(k, v.shape, v.dtype)
    # ---- conditioning front end: the REAL transformers CLIP tower + the verbatim reference resamplers -----------
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection
    from src.models.image_encoder import ImageProjection, ImageProjectionPlus
    fe = {}
    for kind in ("tiny", "l14"):
        d, w, pixels = cases.clip_inputs(kind)
        clip = CLIPVisionModelWithProjection(CLIPVisionConfig(
            hidden_size=d["hidden"], intermediate_size=d["inter"], num_hidden_layers=d["layers"], num_attention_heads=d["heads"],
            image_size=d["image"], patch_size=d["patch"], projection_dim=d["proj"])).eval()
        missing, unexpected = clip.load_state_dict(w, strict=False)
        assert not unexpected and all("position_ids" in k for k in missing), (missing, unexpected)
        o = clip(pixel_values=pixels, output_hidden_states=True)
        fe[f"clip_{kind}_hidden"] = o.hidden_states[-1].numpy()        # what ImageEncoder.get_hidden_states returns (:82-87)
        fe[f"clip_{kind}_embeds"] = o.image_embeds.numpy()             # what ImageEncoder.forward returns (:63-68)
    plus = ImageProjectionPlus(clip_hidden_dim=1024, cross_attention_dim=768, num_tokens=16, num_heads=8, depth=2)
    plus.load_state_dict(cases.projection_plus_inputs())
    fe["projection_plus"] = plus(torch.from_numpy(fe["clip_l14_hidden"])).numpy()
    bw, emb_in = cases.projection_basic_inputs()
    basic = ImageProjection(clip_embedding_dim=768, cross_attention_dim=768, num_tokens=4)
    basic.load_state_dict(bw)
    fe["projection_basic"] = basic(emb_in).numpy()
    np.savez_compressed(os.path.join(HERE, "front_end.npz"), **pack(fe))
    for k, v in fe.items():
        print(k, v.shape, v.dtype)


if __name__ == "__main__":
    main()
