"""Times the trunk + heads of NativeForward (ResNet-10, 15x15) on the batched one-launch route (rz_net_trunk_tc2.cu)
against one launch per layer, over batch sizes (the routing threshold) and chunk sizes (the chunk constant).

    python scripts/trunk_batched_probe.py > out.jsonl

Each point: CUDA events around `reps` forwards of the trunk and heads (the stem's output already in place), the two
routes alternating in `rounds` rounds after a warm-up; prints the median ms per forward of each, one JSON line per point.
"""
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({'card': smi}), flush=True)
    torch.manual_seed(0)
    net = ResNetPolicyValueNet(15, n_blocks=10).cuda().eval()
    nmax = 8192
    x = (torch.rand(nmax, 4, 15, 15) < 0.2).float().numpy()
    nf = NativeForward(net, max_batch=nmax)
    nf.forward_planes(x)

    def timed(n, batched, chunk, reps):
        nf.batched_trunk_min = 1 if batched else 1 << 30
        if batched and chunk != nf.trunk_chunk:
            nf.trunk_chunk, nf.scratch = chunk, None
            nf._alloc(n)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            nf._trunk_and_heads(n, nf.logp, nf.value)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / reps

    def point(n, chunk, reps, rounds=5):
        for _ in range(3):
            timed(n, True, chunk, reps)
            timed(n, False, chunk, reps)
        a, b = [], []
        for r in range(rounds):
            a.append(timed(n, True, chunk, reps))
            b.append(timed(n, False, chunk, reps))
        a.sort()
        b.sort()
        print(json.dumps({'n': n, 'chunk': chunk, 'batched_ms': round(a[rounds // 2], 4),
                          'per_layer_ms': round(b[rounds // 2], 4), 'gain_pct': round(100 * (b[rounds // 2] - a[rounds // 2]) / b[rounds // 2], 2),
                          'batched_all': [round(v, 4) for v in a], 'per_layer_all': [round(v, 4) for v in b]}), flush=True)

    # warm the card up to its power limit
    for _ in range(300):
        nf._trunk_and_heads(nmax, nf.logp, nf.value)
    for chunk in (4, 6, 8, 10, 12, 16):
        point(nmax, chunk, 40)
    for n in (300, 512, 768, 1024, 1536, 2048, 4096):
        point(n, 8, max(40, 40 * 8192 // n // 4))


if __name__ == '__main__':
    main()
