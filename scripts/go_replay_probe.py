#!/usr/bin/env python
"""The compact Go replay buffer (GoReplayBuffer) against the host route, on real 19x19 self-play records.

Self-play: BatchedSelfPlay on 19x19 Go with a ResNet-1 (17 planes, 362 actions), a few playouts per move and a move cap,
from the empty board, until at least ``--records`` plies have finished; the sizes go into the JSON.  Then, with CUDA
events (or a host clock around work that ends in a device synchronise):

  extend        GoReplayBuffer.extend of every drained record (rz_go_records_pack), per record
  sample        GoReplayBuffer.sample(batch): torch.randperm over the 8 * len (record, symmetry) pairs + the expansion
  expand        GoReplayBuffer.expand of the same batch of pairs (the slot arithmetic + rz_go_records_expand), and
                the kernel alone (20 back-to-back launches per timed window)
  host route    the same positions through BatchedSelfPlay._go_states in numpy (each with its 7 predecessors, without
                symmetries) + the copy of the float32 planes, pi and z to the device; the copy of the records to the
                host that the route starts with (BatchedSelfPlay.drain) is timed on its own

The buffer holds every record (several hundred MB at 19x19, more than the 126 MB of L2), so sampled records come from
HBM.  The card's name and power limit are read in the same run and stored with the numbers.

    python scripts/go_replay_probe.py [--records 200000] [--out profiles/go_replay.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rlzero_b200 import _lib as L  # noqa: E402
from rlzero_b200.games.gomoku.policy_value_net import ResNetPolicyValueNet  # noqa: E402
from rlzero_b200.selfplay import BatchedSelfPlay  # noqa: E402
from rlzero_b200.train_pipeline import GoReplayBuffer  # noqa: E402


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout.strip().splitlines()
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit=q[0] if q else None)


def event_ms(fn, reps):
    """Median over ``reps`` of the CUDA-event time of one call (after two warm-up calls)."""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--records', type=int, default=200000)
    ap.add_argument('--games', type=int, default=4096)
    ap.add_argument('--playouts', type=int, default=4)
    ap.add_argument('--max-moves', type=int, default=64)
    ap.add_argument('--batch', type=int, default=1024)
    ap.add_argument('--reps', type=int, default=50)
    ap.add_argument('--out', default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'profiles',
                                                  'go_replay.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('go_replay_probe.py measures on a CUDA device; none is visible')
    c = card()
    print('card:', c['torch_name'], '|', c['nvidia_smi_name_power_limit'], flush=True)
    H, A, B = 19, 19 * 19 + 1, args.batch

    # ---- real records
    torch.manual_seed(0)
    net = ResNetPolicyValueNet(H, n_blocks=1, n_actions=A, in_planes=17).cuda().eval()
    ring = 1 << max(17, int(np.ceil(np.log2(2 * args.records))))
    sp = BatchedSelfPlay(args.games, H, 1, net=net, n_playout=args.playouts, add_noise=True, seed=7, game_type=L.GAME_GO,
                         komi=7.5, max_moves=args.max_moves, ring_capacity=ring)
    t0 = time.time()
    moves = 0
    while sp.stats()['plies_done'] < args.records:
        sp.play(8)
        moves += 8
    torch.cuda.synchronize()
    selfplay_s = time.time() - t0
    sp.forest.raise_faults()
    st = sp.stats()
    rec = sp.forest.drain_trajectories_device()
    assert rec['dropped'] == 0
    N = int(rec['info'].shape[0])
    print('self-play: %d games, %d moves, %d records, %d episodes, %.1f s' % (args.games, moves, N, st['games_done'],
                                                                               selfplay_s), flush=True)

    # ---- extend: rz_go_records_pack of every record
    buf = GoReplayBuffer(N, H)

    def extend():
        buf.start, buf.size = 0, 0
        buf.extend(rec['rows'], rec['info'], rec['pi'])
    ext_ms, ext_all = event_ms(extend, max(5, args.reps // 5))
    assert len(buf) == N

    # ---- sample(B) and the expansion alone
    g = torch.Generator(device='cuda').manual_seed(1)
    smp_ms, smp_all = event_ms(lambda: buf.sample(B, generator=g), args.reps)
    k = torch.randperm(8 * N, generator=g, device='cuda')[:B]
    ridx, sym = k // 8, k % 8
    exp_ms, exp_all = event_ms(lambda: buf.expand(ridx, sym), args.reps)
    # the kernel alone: 20 back-to-back launches on precomputed slots per timed window
    slots = (ridx + buf.start) % buf.capacity
    o_s = torch.empty(B, 17, H, H, device='cuda')
    o_p, o_z = torch.empty(B, A, device='cuda'), torch.empty(B, device='cuda')

    def kernel20():
        for _ in range(20):
            L.check(buf.lib.rz_go_records_expand(C.byref(buf.gdesc), L.ptr(buf.planes), L.ptr(buf.mover),
                                                 L.ptr(buf.pis), L.ptr(buf.zs), buf.capacity, L.ptr(slots), L.ptr(sym),
                                                 B, L.ptr(o_s), L.ptr(o_p), L.ptr(o_z), L.stream_ptr()),
                    'rz_go_records_expand')
    k20_ms, k20_all = event_ms(kernel20, args.reps)
    kern_ms = k20_ms / 20

    # ---- the host route for the same B positions (no symmetries)
    rows_h = rec['rows'].cpu().numpy().view(np.uint32)
    info_h = rec['info'].cpu().numpy()
    pi_h = rec['pi'].cpu().numpy()[:, :A]
    pos = np.maximum(ridx.cpu().numpy(), 7)
    win = (pos[:, None] + np.arange(-7, 1)[None, :]).reshape(-1)

    def host_route():
        states = sp._go_states(rows_h[win], info_h[win])[7::8]
        s = torch.from_numpy(np.ascontiguousarray(states)).cuda()
        p = torch.from_numpy(np.ascontiguousarray(pi_h[pos])).cuda()
        z = torch.from_numpy(info_h[pos, 2].astype(np.float32)).cuda()
        torch.cuda.synchronize()
        return s, p, z
    host_route()
    host_all = []
    for _ in range(max(5, args.reps // 5)):
        t = time.perf_counter()
        s_h, _, _ = host_route()
        host_all.append((time.perf_counter() - t) * 1e3)
    host_ms = float(np.median(host_all))
    # both routes give the same planes for these positions at the identity symmetry
    s_d = buf.expand(torch.from_numpy(pos).cuda(), torch.full((B,), 6, dtype=torch.int64, device='cuda'))[0]
    same = bool(torch.equal(s_d, s_h))

    def drain_copy():
        for t in (rec['rows'], rec['info'], rec['pi']):
            t.cpu()
    t = time.perf_counter()
    drain_copy()
    torch.cuda.synchronize()
    d2h_ms = (time.perf_counter() - t) * 1e3

    bpp = buf.bytes_per_position()
    fl8 = 8 * (17 * H * H + A + 1) * 4
    out_bytes = B * (17 * H * H + A + 1) * 4
    res = {
        'card': c,
        'selfplay': {'board': H, 'network': 'ResNet-1, 17 planes, 362 actions', 'games': args.games,
                     'playouts_per_move': args.playouts, 'max_moves': args.max_moves, 'moves_played': moves,
                     'episodes_finished': st['games_done'], 'records': N, 'seconds': selfplay_s,
                     'start': 'empty board'},
        'bytes_per_position': {'go_replay_buffer': bpp, 'eight_augmented_float32_samples': fl8, 'ratio': fl8 / bpp,
                               'buffer_bytes_total': bpp * N},
        'extend': {'records': N, 'ms': ext_ms, 'ns_per_record': ext_ms * 1e6 / N, 'ms_all': ext_all,
                   'write_GB_per_s': bpp * N / ext_ms / 1e6},
        'sample': {'batch': B, 'pairs_drawn_from': 8 * N, 'ms': smp_ms, 'ms_all': smp_all,
                   'includes': 'torch.randperm(8 * len) on the device, the index arithmetic and rz_go_records_expand'},
        'expand': {'batch': B, 'ms': exp_ms, 'ms_all': exp_all, 'output_bytes': out_bytes,
                   'kernel_ms': kern_ms, 'kernel_ms_all_per_20': k20_all,
                   'kernel_write_GB_per_s': out_bytes / kern_ms / 1e6},
        'host_route': {'batch': B, 'ms': host_ms, 'ms_all': host_all,
                       'includes': 'BatchedSelfPlay._go_states in numpy on the B positions and their 7 predecessors (no '
                                   'symmetries) + host-to-device copy of planes, pi, z, ended by a synchronise',
                       'same_planes_as_expand_at_identity': same,
                       'drain_copy_to_host_ms_all_records': d2h_ms},
        'sample_speedup_vs_host_route': host_ms / smp_ms,
    }
    print(json.dumps({k: v for k, v in res.items() if k not in ('extend', 'sample', 'expand', 'host_route')}))
    print('extend %.3f ms for %d records (%.1f ns/record) | sample(%d) %.3f ms | expand %.3f ms (kernel %.4f ms) | '
          'host route %.2f ms (same planes: %s) | drain copy %.1f ms' % (ext_ms, N, ext_ms * 1e6 / N, B, smp_ms, exp_ms,
                                                                        kern_ms, host_ms, same, d2h_ms), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
