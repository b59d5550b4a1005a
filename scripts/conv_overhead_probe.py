#!/usr/bin/env python
"""Fixed per-launch cost of the trunk convolution: time rz_net_conv3x3_tc2 at several batch sizes (multiples of
the 74 CTA pairs) and fit t = a * tiles_per_pair + b.  b = prologue (barriers, TMEM, 147 KB of weights per CTA),
pipeline fill and drain; a = steady-state time per 256-position tile."""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rlzero_b200 import _lib as L  # noqa: E402


def main():
    lib = L.load()
    torch.manual_seed(0)
    w = (torch.randn(9, 128, 128, device='cuda') * 0.03).to(torch.bfloat16).contiguous()
    b = torch.zeros(128, device='cuda')
    flags = 4 if 'noepilogue' in sys.argv else 0
    pts = []
    for rounds in (4, 8, 16, 32, 64, 110):
        B = 74 * rounds
        x = (torch.randn(B * 256, 128, device='cuda') * 0.5).to(torch.bfloat16).contiguous()
        y = torch.empty_like(x)
        r = torch.empty_like(x).copy_(x)
        for res in (None, r):
            def run():
                L.check(lib.rz_net_conv3x3_tc2(L.ptr(x), L.ptr(w), L.ptr(b), L.ptr(res) if res is not None else None,
                                               L.ptr(y), B, 15, 15, 128, 1, 2, flags, 0, L.stream_ptr()))
            for _ in range(5):
                run()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(40):
                run()
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) / 40 * 1e3
            pts.append((rounds, res is not None, us))
            print(json.dumps({'boards': B, 'tiles_per_pair': rounds, 'residual': res is not None, 'us': us}), flush=True)
    for flag in (False, True):
        xs = np.array([p[0] for p in pts if p[1] == flag], dtype=np.float64)
        ys = np.array([p[2] for p in pts if p[1] == flag], dtype=np.float64)
        a, c = np.polyfit(xs, ys, 1)
        print(json.dumps({'fit': 'us = a * tiles_per_pair + b', 'residual': flag, 'a_us_per_tile': a, 'b_us_fixed': c,
                          'fixed_share_at_111_tiles': c / (a * 110.7 + c)}))


if __name__ == '__main__':
    main()
