"""Loads the LIVE reference hot path (vector_quantizer/vq_img.py) by file path -- TEST INFRASTRUCTURE.

Only usable where the environment variable VQSEG_REF names a checkout of the original chaeyeongyun/VQ_SEG
repository; without one, reference_root() is None and the tests that need the live reference skip.  It is used to
pin the restated oracle (tests/test_oracle.py) and to generate tests/golden/*.pt (tests/golden/make_golden.py): the
stored goldens are the pin everywhere else, and nothing on the product path may depend on this module.
`import vector_quantizer` (the package) needs easydict, but vq_img.py itself needs only torch + einops
(SURVEY.md §8c).
"""
import importlib.util
import os


def reference_root():
    root = os.environ.get("VQSEG_REF", "")
    if root and os.path.isfile(os.path.join(root, "vector_quantizer", "vq_img.py")):
        return root
    return None


def load_reference_vq_img():
    root = reference_root()
    if root is None:
        return None
    path = os.path.join(root, "vector_quantizer", "vq_img.py")
    spec = importlib.util.spec_from_file_location("ref_vq_img", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load_reference_seghead():
    """models/modules/vq_segmentation_head.py of the live reference (needs only torch + einops)."""
    root = reference_root()
    if root is None:
        return None
    path = os.path.join(root, "models", "modules", "vq_segmentation_head.py")
    if not os.path.isfile(path):
        return None
    spec = importlib.util.spec_from_file_location("ref_vq_segmentation_head", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod
