"""The restated equations of the EMA dead-code expiry, for the tests of vqseg_ema_update_expire_f32.

Opt-in extension without a reference counterpart (parity unpinned): threshold_ema_dead_code of
lucidrains/vector-quantize-pytorch (expire_codes_ / replace).  tests/test_ema_expire.py checks this restatement against
a literal transcription of lucidrains's boolean-mask `replace`."""
from typing import Optional

import torch


def ema_expire(cluster_size: torch.Tensor, embed_avg: torch.Tensor, weight: torch.Tensor, cand: torch.Tensor,
               threshold: float, reset: Optional[float] = None):
    """`cluster_size`, `embed_avg`, `weight` are the results of the EMA update (oracle.vq_oracle.ema_update); `cand`
    the (K, D) candidate rows (sample_vectors of the batch).  expired = cluster_size < threshold in fp32; the r-th
    expired code in ascending k takes cand[r]: weight = cand[r], embed_avg = cand[r] * reset, cluster_size = reset
    (reset defaults to the threshold).  Returns (cluster_size, embed_avg, weight, number of expired codes)."""
    thr = torch.tensor(threshold, dtype=torch.float32, device=cluster_size.device)
    rst = thr if reset is None else torch.tensor(reset, dtype=torch.float32, device=cluster_size.device)
    expired = cluster_size < thr
    slot = torch.cumsum(expired.to(torch.int64), 0) - 1                  # exclusive prefix of the mask
    rows = cand[slot.clamp(min=0)]
    col = expired.unsqueeze(1)
    return (torch.where(expired, rst, cluster_size), torch.where(col, rows * rst, embed_avg),
            torch.where(col, rows, weight), int(expired.sum()))
