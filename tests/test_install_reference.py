"""Drop-in evidence against the UNMODIFIED reference models (needs a checkout of the original repository: VQSEG_REF).
`vq_seg_b200.install()` swaps the class into the reference's modules; `make_model` of the reference then builds
the north-star network (VQRePTUnet1x1v2, config/vqreptunet1x1v2.json) with B200 codebooks, and its state_dict
keys are the reference's.  Construction only: the forward needs a GPU (covered by test_gpu_parity.py)."""
import collections
import json
import os
import sys
import types

import pytest

from oracle.ref_loader import reference_root

REF = reference_root()


@pytest.mark.skipif(REF is None, reason="needs a reference checkout (VQSEG_REF)")
def test_reference_model_builds_with_b200_codebooks():
    # packages the reference imports that are not installed here (SURVEY 8b): easydict, pretrainedmodels
    class EasyDict(dict):
        def __init__(self, d=None, **kw):
            super().__init__()
            for k, v in dict(d or {}, **kw).items():
                self[k] = EasyDict(v) if isinstance(v, dict) else v

        def __getattr__(self, k):
            try:
                return self[k]
            except KeyError:
                raise AttributeError(k)

        __setattr__ = dict.__setitem__
    stubs = {}
    ed = types.ModuleType("easydict"); ed.EasyDict = EasyDict; stubs["easydict"] = ed
    pm = types.ModuleType("pretrainedmodels"); pmm = types.ModuleType("pretrainedmodels.models")
    pmt = types.ModuleType("pretrainedmodels.models.torchvision_models")
    pmt.pretrained_settings = collections.defaultdict(lambda: collections.defaultdict(dict))
    pm.models = pmm; pmm.torchvision_models = pmt
    stubs.update({"pretrainedmodels": pm, "pretrainedmodels.models": pmm, "pretrainedmodels.models.torchvision_models": pmt})
    saved = {k: sys.modules.get(k) for k in stubs}
    sys.modules.update(stubs)
    sys.path.insert(0, REF)
    added = set()
    before = set(sys.modules)
    try:
        import vector_quantizer                      # the reference package
        import models.networks as ref_networks
        import vq_seg_b200 as V
        patched = V.install()
        assert "vector_quantizer" in patched and "models.networks.unet.net" in patched
        cfg = json.load(open(os.path.join(REF, "config", "vqreptunet1x1v2.json")))
        params = EasyDict(cfg["model"]["params"])
        params["encoder_weights"] = None             # no network for the swsl weights
        model = ref_networks.network_dict[cfg["model"]["name"]](**params)
        kinds = [type(m).__module__ + "." + type(m).__name__ for m in model.codebook]
        assert kinds[:2] == ["vector_quantizer.Identity"] * 2
        assert kinds[2:] == ["vq_seg_b200.vq_img.VectorQuantizer"] * 3
        assert [tuple(m.codebook.embedding.weight.shape) for m in model.codebook[2:]] == [(512, 512), (512, 1024), (512, 2048)]
        keys = [k for k in model.state_dict() if k.startswith("codebook.")]
        assert keys == [f"codebook.{i}.codebook.embedding.weight" for i in (2, 3, 4)]
        assert all(m.codebook.kmeans_init and not m.codebook.initted for m in model.codebook[2:])
        # another family that binds the class by name (unet/net.py:10)
        v2 = ref_networks.network_dict["vqunet_v2"](encoder_name="resnet50", num_classes=3,
                                                    vq_cfg=EasyDict(num_embeddings=[0, 0, 512, 512, 512], distance="euclidean",
                                                                    kmeans_init=True), encoder_weights=None)
        assert sum(isinstance(m, V.VectorQuantizer) for m in v2.codebook) == 3
        # SURVEY 8f-3: the VQ segmentation head and the other copies of kmeans
        import models.modules.prototype as ref_proto
        import models.modules.segmentation_head as ref_sh
        import models.modules.vq_segmentation_head as ref_vsh
        patched = V.install(kmeans=True)
        assert "models.modules.vq_segmentation_head:VQSegmentationHead" in patched
        assert "models.networks.vqseghead.net:VQSegmentationHead" in patched
        assert ref_proto.kmeans is V.kmeans and ref_sh.kmeans is V.kmeans and ref_vsh.kmeans is V.kmeans
        net = ref_networks.network_dict["vqsegheadnet"](encoder_name="resnet50", num_classes=3, encoder_weights=None,
                                                        vq_cfg=EasyDict(num_embeddings=[0, 0, 512, 512, 512],
                                                                        distance="euclidean", kmeans_init=True))
        assert isinstance(net.segmentation_head, V.VQSegmentationHead)
        assert tuple(net.segmentation_head.codebook.embedding.weight.shape) == (3, 32)
        assert [k for k in net.state_dict() if k.startswith("segmentation_head.")] == ["segmentation_head.codebook.embedding.weight"]
    finally:
        added = set(sys.modules) - before
        for k in added:
            if k.split(".")[0] in ("vector_quantizer", "models", "loss", "utils", "data"):
                sys.modules.pop(k, None)
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
        sys.path.remove(REF)
