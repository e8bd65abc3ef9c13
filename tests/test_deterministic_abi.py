"""CPU-side checks of the deterministic segmentation-head backward (VQSEG_SEGHEAD_DETERMINISTIC): the workspace it
asks for (the slices' partial sums on top of the tiled kernels' 16 bytes per pixel, never more than 32 MiB of
partials) and the forward map refusing the bit."""
import ctypes

import pytest

MIB = 1 << 20


@pytest.fixture(scope="module")
def lib():
    from vq_seg_b200 import build, _native
    build.build()
    return _native.lib()


def test_deterministic_bit_matches_the_header(lib):
    import os
    from vq_seg_b200 import ops
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "include", "vqseg.h")) as fh:
        assert f"#define VQSEG_SEGHEAD_DETERMINISTIC 0x{ops.SEGHEAD_DETERMINISTIC:x}" in fh.read()


@pytest.mark.parametrize("algo", ["AUTO", "PIXEL"])
def test_per_pixel_shapes_get_a_partials_workspace(lib, algo):
    from vq_seg_b200 import ops
    a = getattr(ops, "SEGHEAD_" + algo) | ops.SEGHEAD_DETERMINISTIC
    ws = lib.vqseg_seghead_map_bwd_workspace_bytes
    for n, d, k in ((1000, 64, 3), (1 << 18, 32, 3), (1 << 18, 382, 32), (5000, 100, 7)):
        b = ws(n, d, k, a)
        assert b > 0 and b % (4 * k * d) == 0, (n, d, k, b)
        assert b <= 32 * MIB
    assert ws(128, 64, 3, a) == 0                 # one 128-pixel tile: the kernel stores gE itself
    assert ws(0, 64, 3, a) == 0


def test_tiled_shapes_add_the_partials_to_the_scalars(lib):
    from vq_seg_b200 import ops
    ws = lib.vqseg_seghead_map_bwd_workspace_bytes
    for n, d, k, algo in ((1000, 383, 3, ops.SEGHEAD_AUTO), (1000, 64, 33, ops.SEGHEAD_AUTO),
                          (1000, 64, 3, ops.SEGHEAD_TILED), (1 << 18, 256, 150, ops.SEGHEAD_AUTO),
                          (1 << 18, 64, 1000, ops.SEGHEAD_AUTO), (1 << 18, 2048, 1000, ops.SEGHEAD_AUTO),
                          (1 << 18, 8192, 1024, ops.SEGHEAD_AUTO)):
        b = ws(n, d, k, algo | ops.SEGHEAD_DETERMINISTIC)
        assert b >= 16 * n and (b - 16 * n) % (4 * k * d) == 0 and b - 16 * n <= 32 * MIB, (n, d, k, b)
    # partials larger than 32 MiB for a single split: one split, written straight into gE
    assert ws(1 << 18, 8192, 1024, ops.SEGHEAD_DETERMINISTIC) == 16 << 18


@pytest.mark.parametrize("k,d", [(1000, 2048), (32, 382)])
def test_workspace_bound_at_a_quarter_million_pixels(lib, k, d):
    from vq_seg_b200 import ops
    n = 1 << 18
    b = lib.vqseg_seghead_map_bwd_workspace_bytes(n, d, k, ops.SEGHEAD_AUTO | ops.SEGHEAD_DETERMINISTIC)
    assert 0 < b <= 16 * n + 32 * MIB


def test_default_sizes_are_unchanged(lib):
    from vq_seg_b200 import ops
    ws = lib.vqseg_seghead_map_bwd_workspace_bytes
    assert ws(1 << 18, 32, 3, ops.SEGHEAD_AUTO) == 0
    assert ws(1 << 18, 256, 150, ops.SEGHEAD_AUTO) == 16 << 18


def test_forward_map_rejects_the_bit(lib):
    from vq_seg_b200 import ops
    buf = (ctypes.c_float * 64)()
    idx = (ctypes.c_int64 * 8)()
    p = ctypes.addressof(buf)
    for algo in (ops.SEGHEAD_AUTO, ops.SEGHEAD_TILED):
        rc = lib.vqseg_seghead_map_f32(p, 1, 4, 4, 16, 4, 1, p, 2, 0, p, 8, 1, 4, ctypes.addressof(idx), None, None,
                                       algo | ops.SEGHEAD_DETERMINISTIC, None)
        assert rc == -1                           # VQSEG_EINVAL, before any device work
