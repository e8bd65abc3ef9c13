"""A catalogue of the memory layouts a model hands the quantiser through `x.reshape(b, c, h * w).permute(0, 2, 1)`.

Every layout is built from one seeded storage tensor by torch views only, so the (B, P, D) view the ops receive is
a view of that storage (asserted: a silent copy would test the packed layout under another name), and the CPU and
the GPU copies of a case have identical strides.  Each layout reaches other branches of the kernels' layout tests:

  nchw               contiguous NCHW map: sP == 1, sD = H*W (what the rest of the suite feeds)
  nhwc               channels-last map: packed rows, sD == 1, sP == C
  nchw_ch_slice      channel slice [:, 4:4+C] of an NCHW map with 8 more channels: sB != C*H*W, base offset
  nchw_ch_slice_odd  channel slice [:, 1:1+C] of an NCHW map with 3 more channels (H*W odd: misaligned base)
  nhwc_ch_slice      channel slice of a channels-last map: rows padded to C+8 floats (sP > D), aligned
  nhwc_ch_slice_odd  channel slice of a channels-last map: rows padded to C+3 floats, misaligned base
  nchw_batch_step    every other image of an NCHW map: sB = 2*C*H*W
  nhwc_batch_step    every other image of a channels-last map: sD == 1 but the rows are not one flat range
  cnhw               permute(1, 0, 2, 3) of a (C, B, H, W) tensor: sB = H*W < sD = B*H*W
  map_1x1            an NCHW map of 1 x 1 pixels: P == 1, sP == sD == 1
  expand             one image expanded over the batch: sB == 0 (inputs of read-only ops only)
  rows_offset        packed rows starting one float into their storage: sD == 1, misaligned base
"""
import torch

LAYOUTS = ("nchw", "nhwc", "nchw_ch_slice", "nchw_ch_slice_odd", "nhwc_ch_slice", "nhwc_ch_slice_odd",
           "nchw_batch_step", "nhwc_batch_step", "cnhw", "map_1x1", "expand", "rows_offset")
WRITABLE = tuple(name for name in LAYOUTS if name != "expand")     # layouts without overlapping elements

# (B, C, H, W) and the codebook size used with it:
#   P = 63, not a multiple of 4 or of a 128-row tile;  an aligned map;  a codebook too large to stay resident
#   (streaming kernels only);  1 x 1 maps with enough rows and codes for AUTO to take a tensor-core filter
SHAPES = {"odd": ((3, 96, 7, 9), 300), "aligned": ((2, 96, 16, 16), 300), "stream": ((4, 200, 5, 5), 700),
          "px1": ((96, 64, 1, 1), 300)}


def cases(layouts=LAYOUTS, shapes=tuple(SHAPES)):
    """(layout, shape name) pairs: map_1x1 goes with the 1 x 1 shape only, the 1 x 1 shape with the layouts that
    differ from map_1x1 at H = W = 1"""
    out = []
    for s in shapes:
        one = SHAPES[s][0][2:] == (1, 1)
        for lay in layouts:
            if lay == "map_1x1" and not one:
                continue
            if one and lay in ("nchw", "nchw_ch_slice", "nchw_batch_step"):
                continue                                   # the same strides as map_1x1 up to sB
            if lay == "nchw_ch_slice" and (SHAPES[s][0][2] * SHAPES[s][0][3]) % 4:
                continue                                   # its base is 16-byte aligned only when H*W % 4 == 0
            if lay == "nchw_ch_slice_odd" and (SHAPES[s][0][2] * SHAPES[s][0][3]) % 2 == 0:
                continue                                   # its base is misaligned only when H*W is odd
            out.append((lay, s))
    return out


def case_id(case):
    return f"{case[0]}-{case[1]}"


def expected_strides(layout, shape):
    """(sB, sP, sD) of bpd(x) for a layout"""
    b, c, h, w = shape
    p = h * w
    return {"nchw": (c * p, 1, p), "nhwc": (p * c, c, 1),
            "nchw_ch_slice": ((c + 8) * p, 1, p), "nchw_ch_slice_odd": ((c + 3) * p, 1, p),
            "nhwc_ch_slice": (p * (c + 8), c + 8, 1), "nhwc_ch_slice_odd": (p * (c + 3), c + 3, 1),
            "nchw_batch_step": (2 * c * p, 1, p), "nhwc_batch_step": (2 * p * c, c, 1),
            "cnhw": (p, 1, b * p), "map_1x1": (c, 1, 1), "expand": (0, 1, p), "rows_offset": (p * c, c, 1)}[layout]


def make(layout, shape, seed, device="cpu"):
    """(full, x): `full` the seeded storage (built on the CPU, then moved to `device`), x the (B, C, H, W) view of it
    in the named layout"""
    b, c, h, w = shape
    g = torch.Generator().manual_seed(seed)
    rnd = lambda *s: torch.randn(*s, generator=g).to(device)  # noqa: E731
    if layout == "nchw":
        full = rnd(b, c, h, w)
        x = full
    elif layout == "nhwc":
        full = rnd(b, h, w, c)
        x = full.permute(0, 3, 1, 2)
    elif layout == "nchw_ch_slice":
        full = rnd(b, c + 8, h, w)
        x = full[:, 4:4 + c]
    elif layout == "nchw_ch_slice_odd":
        full = rnd(b, c + 3, h, w)
        x = full[:, 1:1 + c]
    elif layout == "nhwc_ch_slice":
        full = rnd(b, h, w, c + 8)
        x = full.permute(0, 3, 1, 2)[:, 4:4 + c]
    elif layout == "nhwc_ch_slice_odd":
        full = rnd(b, h, w, c + 3)
        x = full.permute(0, 3, 1, 2)[:, 1:1 + c]
    elif layout == "nchw_batch_step":
        full = rnd(2 * b, c, h, w)
        x = full[::2]
    elif layout == "nhwc_batch_step":
        full = rnd(2 * b, h, w, c)
        x = full.permute(0, 3, 1, 2)[::2]
    elif layout == "cnhw":
        full = rnd(c, b, h, w)
        x = full.permute(1, 0, 2, 3)
    elif layout == "map_1x1":
        assert (h, w) == (1, 1), "map_1x1 needs H = W = 1"
        full = rnd(b, c, 1, 1)
        x = full
    elif layout == "expand":
        full = rnd(1, c, h, w)
        x = full.expand(b, c, h, w)
    elif layout == "rows_offset":
        full = rnd(b * h * w * c + 1)
        x = full[1:].view(b, h, w, c).permute(0, 3, 1, 2)
    else:
        raise KeyError(layout)
    assert x.shape == shape
    bpd(x, full, layout)
    return full, x


def bpd(x, full=None, layout=None):
    """x.reshape(b, c, h*w).permute(0, 2, 1), asserted to be a view of `full` with the layout's strides"""
    b, c, h, w = x.shape
    v = x.reshape(b, c, h * w).permute(0, 2, 1)
    if full is not None:
        assert v.untyped_storage().data_ptr() == full.untyped_storage().data_ptr(), f"{layout}: the view is a copy"
        lo = full.data_ptr()
        assert lo <= v.data_ptr() < lo + full.numel() * full.element_size(), f"{layout}: outside the storage"
    if layout is not None:
        assert v.stride() == expected_strides(layout, x.shape), (layout, v.stride())
    return v


def seq_chain_normalize(v):
    """F.normalize over the last dim with the norm as one sequential fp32 chain acc = fl(acc + fl(v * v)) in element
    order, sqrt and division IEEE (numpy float32 arithmetic, independent of ATen)"""
    import numpy as np
    rows = v.detach().cpu().reshape(-1, v.shape[-1]).numpy().astype(np.float32)
    acc = np.zeros(rows.shape[0], np.float32)
    for d in range(rows.shape[1]):
        acc = (acc + (rows[:, d] * rows[:, d]).astype(np.float32)).astype(np.float32)
    nrm = np.maximum(np.sqrt(acc).astype(np.float32), np.float32(1e-12))
    return torch.from_numpy((rows / nrm[:, None]).astype(np.float32)).reshape(v.shape)
