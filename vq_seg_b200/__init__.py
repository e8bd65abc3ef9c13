"""vq_seg_b200: the vector-quantisation bottleneck of chaeyeongyun/VQ_SEG on B200 (sm_100a).

Drop-in for the reference's `vector_quantizer` package: VectorQuantizer, make_vq_module, Identity, and for
its VQ segmentation head (models/modules/vq_segmentation_head.py): VQSegmentationHead.
The kernels live in libvqseg.so (C ABI: include/vqseg.h); importing this package does not load it,
the first op call does -- and raises if it is missing (no CPU fallback)."""
from .vq_img import (VectorQuantizer, EuclideanCodebook, CosinesimCodebook, kmeans, sample_vectors,  # noqa: F401
                     batched_sample_vectors, batched_bincount, l2norm)
from .rvq import ResidualVectorQuantizer  # noqa: F401
from .vq_segmentation_head import VQSegmentationHead, EuclideanSegHead, CosinesimSegHead  # noqa: F401
from .factory import make_vq_module, Identity, install  # noqa: F401
from . import ops  # noqa: F401


def stack_code_usage(usages):
    """One device tensor from the per-layer code-usage scalars (None entries of Identity levels skipped): the callers'
    `code_usage.detach().cpu()` per layer per forward (modified_vqunet/net.py:233) serialises the stream three times a
    step; `stack_code_usage(lst).cpu()` synchronises once (SURVEY.md 8f-4)."""
    import torch
    vals = [u.detach().reshape(()) for u in usages if u is not None]
    return torch.stack(vals) if vals else torch.empty(0)

__version__ = "0.1.0"
