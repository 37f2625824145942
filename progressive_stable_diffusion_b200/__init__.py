"""B200-native implementation of DADD's UNet-denoising hot path (umutdundar99/progressive-stable-diffusion).

Host side: Python/PyTorch modules with the reference's names and call surfaces.  Device side: hand-written sm_100a
kernels in ``libdadd_b200.so`` reached through the C ABI of ``include/dadd_b200.h`` (no Triton, no CPU fallback).
"""

from . import _lib  # noqa: F401
from .attention_processor import AttnProcessor2_0, DEFAULT_COMPUTE_DTYPE, compute_dtype, set_compute_dtype  # noqa: F401
from .attention_processor_base import (OrdinalIPAttnProcessor2_0, get_frequency_mode_for_block,  # noqa: F401
                                       set_ordinal_ip_attention_processors)
from .attention_processor_routing_gates import (SplitInjectionAttentionProcessor, get_block_type,  # noqa: F401
                                                set_split_injection_processors)
from .diffusion_module_ip import DiffusionIPConfig, DiffusionModuleWithIP, default_config, load_config  # noqa: F401
from .feature_purifier import FeaturePurifier  # noqa: F401
from .image_encoder import ImageEncoder, ImageProjection, ImageProjectionPlus  # noqa: F401
from .metrics import ClipEmbedder, VGGFeatures, cmmd, density_coverage, precision_recall, realism_scores  # noqa: F401
from .ordinal_embedder import AdditiveOrdinalEmbedder  # noqa: F401
from .unet import OrdinalUNet, UNetConfig  # noqa: F401
from .vae import SDVAE  # noqa: F401

__all__ = [
    "AttnProcessor2_0", "DEFAULT_COMPUTE_DTYPE", "compute_dtype", "set_compute_dtype", "OrdinalIPAttnProcessor2_0", "SplitInjectionAttentionProcessor", "get_block_type",
    "get_frequency_mode_for_block", "set_ordinal_ip_attention_processors", "set_split_injection_processors",
    "DiffusionIPConfig", "DiffusionModuleWithIP", "default_config", "load_config", "FeaturePurifier",
    "AdditiveOrdinalEmbedder", "OrdinalUNet", "UNetConfig", "SDVAE", "ImageEncoder", "ImageProjection", "ImageProjectionPlus",
    "ClipEmbedder", "VGGFeatures", "cmmd", "precision_recall", "density_coverage", "realism_scores",
]
