"""CPU-side checks of the segmentation-head entry points for any class count and width: exported symbols, ctypes
signatures, and the backward workspace sizes (16 bytes per pixel for the tiled kernels, none for the per-pixel ones)."""
import pytest


@pytest.fixture(scope="module")
def lib():
    from vq_seg_b200 import build, _native
    build.build()
    return _native.lib()


def test_seghead_symbols_are_exported(lib):
    from vq_seg_b200 import _native
    for name in ("vqseg_seghead_map_f32", "vqseg_seghead_map_bwd_f32", "vqseg_seghead_map_bwd_workspace_bytes"):
        assert name in _native.SIGNATURES and hasattr(lib, name)


def test_seghead_bwd_workspace_sizes(lib):
    from vq_seg_b200 import ops
    ws = lib.vqseg_seghead_map_bwd_workspace_bytes
    assert ws(1000, 64, 3, ops.SEGHEAD_AUTO) == 0              # per-pixel kernels (the reference's 3-class head)
    assert ws(1000, 382, 32, ops.SEGHEAD_AUTO) == 0
    assert ws(1000, 383, 3, ops.SEGHEAD_AUTO) == 1000 * 16     # wider than the per-pixel kernels: tiled
    assert ws(1000, 64, 33, ops.SEGHEAD_AUTO) == 1000 * 16
    assert ws(1000, 64, 3, ops.SEGHEAD_TILED) == 1000 * 16     # forced
    assert ws(1000, 2048, 1000, ops.SEGHEAD_PIXEL) == 0
    assert ws(0, 64, 150, ops.SEGHEAD_AUTO) == 0
