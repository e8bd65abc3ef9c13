"""make_vq_module / Identity (reference: vector_quantizer/__init__.py:5-32) and install(), which swaps the
B200 VectorQuantizer into an importable copy of the reference so its unmodified models use it."""
import copy
import sys

from torch import nn

from .rvq import ResidualVectorQuantizer
from .vq_img import VectorQuantizer


def _get(cfg, key):
    return cfg[key] if isinstance(cfg, dict) else getattr(cfg, key)


def make_vq_module(vq_cfg, encoder_channels, depth):
    """vq_cfg: dict / EasyDict with the reference's keys (num_embeddings int or list, distance,
    kmeans_init, ... every VectorQuantizer kwarg).  Unknown keys raise TypeError like the reference.
    Extension: a `num_quantizers` key builds a ResidualVectorQuantizer with that many layers at every
    non-Identity level instead of a VectorQuantizer."""
    cls, extra = VectorQuantizer, {}
    if "num_quantizers" in vq_cfg:
        vq_cfg = copy.deepcopy(vq_cfg)
        cls, extra = ResidualVectorQuantizer, {"num_quantizers": vq_cfg.pop("num_quantizers")}
    num_embeddings = _get(vq_cfg, "num_embeddings")
    if isinstance(num_embeddings, int):
        codebook = nn.ModuleList([cls(**vq_cfg, **extra, dim=encoder_channels[i + 1]) for i in range(depth)])
    elif isinstance(num_embeddings, list):
        assert depth == len(num_embeddings), "depth and length of vq_cfg.num_embeddings must to be same number"
        lst = []
        vq_cfg = copy.deepcopy(vq_cfg)
        for i, num_embed in enumerate(num_embeddings):
            vq_cfg["num_embeddings"] = num_embed
            if num_embed == 0:
                lst.append(Identity())
            elif num_embed > 0:
                lst.append(cls(**vq_cfg, **extra, dim=encoder_channels[i + 1]))
            else:
                raise ValueError(f"{num_embed} is not available number of embeddings")
        codebook = nn.ModuleList(lst)
    else:
        raise TypeError(f"{type(num_embeddings)} is not available type")
    return codebook


class Identity(nn.Module):
    def __init__(self):
        super().__init__()
        self.embedding = nn.Identity()

    def forward(self, x):
        return self.embedding(x), None, None, None


# module globals of the reference that bind the class by name (SURVEY.md §8b)
_PATCH_POINTS = ["vector_quantizer", "vector_quantizer.vq_img", "models.networks.unet.net",
                 "models.networks.vqvaev2.net"]
# SURVEY.md §8f-3: the segmentation head class and the three other copies of `kmeans` (same signature as
# vq_img.py:29; prototype.py:36, segmentation_head.py:42, vq_segmentation_head.py:29)
_SEGHEAD_PATCH_POINTS = ["models.modules.vq_segmentation_head", "models.networks.vqseghead.net"]
_KMEANS_PATCH_POINTS = ["vector_quantizer.vq_img", "models.modules.prototype", "models.modules.segmentation_head",
                        "models.modules.vq_segmentation_head"]


def install(verbose=False, seghead=True, kmeans=False):
    """Monkeypatch every already-imported reference module that binds `VectorQuantizer` by name, so
    `make_model(cfg)` of the unmodified reference builds B200 codebooks.  `seghead` also swaps the VQ segmentation
    head class; `kmeans=True` replaces the reference's four copies of `kmeans` (prototype / segmentation-head
    initialisation) with the B200 one -- GPU tensors only from then on.  Returns the patched names."""
    done = []
    for name in _PATCH_POINTS:
        mod = sys.modules.get(name)
        if mod is not None and hasattr(mod, "VectorQuantizer"):
            setattr(mod, "VectorQuantizer", VectorQuantizer)
            done.append(name)
    if seghead:
        from .vq_segmentation_head import VQSegmentationHead
        for name in _SEGHEAD_PATCH_POINTS:
            mod = sys.modules.get(name)
            if mod is not None and hasattr(mod, "VQSegmentationHead"):
                setattr(mod, "VQSegmentationHead", VQSegmentationHead)
                done.append(name + ":VQSegmentationHead")
    if kmeans:
        from .vq_img import kmeans as b200_kmeans
        for name in _KMEANS_PATCH_POINTS:
            mod = sys.modules.get(name)
            if mod is not None and hasattr(mod, "kmeans"):
                setattr(mod, "kmeans", b200_kmeans)
                done.append(name + ":kmeans")
    if verbose:
        print("vq_seg_b200.install: patched", done)
    return done
