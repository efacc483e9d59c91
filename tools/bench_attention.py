"""Micro-benchmark of warp_attention at the three stage shapes of the 512^2 generator (GPU box), on the schedule this
process selects: the library reads IPER_ATT_WIDE once per process, so compare schedules with one run per setting:

    python tools/bench_attention.py; for w in 0 1 2; do IPER_ATT_WIDE=$w python tools/bench_attention.py; done
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch

from ipercore_b200 import ops
from ipercore_b200.ops import Planes

wide = os.environ.get("IPER_ATT_WIDE")      # the library's rule: unset or 3 -> chunked, 1 / 2 -> that schedule, else 0
w = 3 if wide is None else (int(wide) if wide.strip().isdigit() else 0)
print("schedule: %s (IPER_ATT_WIDE=%s)" % ("chunked" if w == 3 else "pixel-per-warp WIDE=%d" % (w if w in (1, 2) else 0), wide))
dev = "cuda:0"
B, ns = 50, 2
g = torch.Generator().manual_seed(0)
for C, h in ((256, 64), (128, 128), (64, 256)):
    kv = torch.rand((ns, h, h, 2 * C + 64), generator=g).to(dev)
    bv = torch.rand((C,), generator=g).to(dev)
    x = Planes.from_nchw(torch.rand((B, C, h, h), generator=g).to(dev), 2)
    # smooth flow: identity grid + a small seeded perturbation (neighbouring pixels sample neighbouring source pixels)
    ys, xs = torch.meshgrid(torch.linspace(-1, 1, h), torch.linspace(-1, 1, h), indexing="ij")
    T = torch.stack([xs, ys], -1)[None, None].repeat(B, ns, 1, 1, 1) * 0.9 + (torch.rand((B, ns, 1, 1, 2), generator=g) - 0.5) * 0.2
    T = T.contiguous().to(dev)
    out = Planes.empty(2, B, h, h, C, dev)
    for _ in range(3):
        ops.warp_attention(x, kv, bv, T, out)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        ops.warp_attention(x, kv, bv, T, out)
    e1.record(); torch.cuda.synchronize()
    print("C=%d h=%d  %.3f ms" % (C, h, e0.elapsed_time(e1) / 10))
