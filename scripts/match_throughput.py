#!/usr/bin/env python
"""Evaluation-match throughput: ``TrainPipeline.policy_evaluate`` played one game after another through
``GameControl.start_play`` against the same games as one ``BatchedMatch``.

The setting is the reference's evaluation (tools/train_alphazero.py:139-163): the trained net (``AlphaZeroPlayer``,
400 playouts) against pure MCTS (``RolloutPlayer``, 1000 playouts), on 6x6 four in a row with ``AlphaZeroAgent(6)``
and on 15x15 five in a row with ``AlphaZeroAgent(15)`` -- the stock PolicyValueNet, untrained.  Every time is host
wall time of the call, ending in a device synchronise; a batched time includes the graph captures of its fresh
forests, not their allocation.  One warm-up match per board runs first.  The last line is one JSON object with the
card's name and power limit.

    python scripts/match_throughput.py [--boards 6,15] [--games 10,100,1000] [--sequential 10]
                                       [--mixed-first 100]

``--mixed-first G`` also plays G games with alternating first movers, where both seats search every ply (the cost of
the waiting games' stale leaves in the net's batch).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rlzero_b200.match import BatchedMatch  # noqa: E402
from rlzero_b200.mcts import AlphaZeroPlayer, RolloutPlayer  # noqa: E402
from rlzero_b200.train_pipeline import TrainPipeline  # noqa: E402

BOARDS = {6: 4, 15: 5}


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout.strip().splitlines()
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q[0] if q else None)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.time()
    out = fn()
    torch.cuda.synchronize()
    return time.time() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--boards', default='6,15')
    ap.add_argument('--games', default='10,100,1000')
    ap.add_argument('--sequential', type=int, default=10, help='games of the sequential policy_evaluate (0: skip)')
    ap.add_argument('--mixed-first', type=int, default=0)
    ap.add_argument('--n-playout', type=int, default=400)
    ap.add_argument('--pure-playout', type=int, default=1000)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('match_throughput.py measures the GPU: no CUDA device')
    np.random.seed(0)
    torch.manual_seed(0)
    results = []
    for size in [int(s) for s in a.boards.split(',')]:
        k = BOARDS[size]
        pipe = TrainPipeline(board_size=size, n_in_row=k, n_playout=a.n_playout, pure_mcts_playout_num=a.pure_playout)
        pipe.alphazero_agent.policy_value_net.eval()

        def players():
            return (AlphaZeroPlayer(pipe.alphazero_agent.policy_value_fn, n_playout=a.n_playout, c_puct=pipe.c_puct),
                    RolloutPlayer(n_playout=a.pure_playout, c_puct=5))

        BatchedMatch(*players(), 2, size, k).play(seed=1)          # warm-up: module loads, first captures
        if a.sequential:
            dt, ratio = timed(lambda: pipe.policy_evaluate(n_games=a.sequential))
            results.append(dict(board=size, path='sequential policy_evaluate', games=a.sequential, seconds=dt,
                                games_per_s=a.sequential / dt, win_ratio=ratio))
            print(json.dumps(results[-1]), flush=True)
        runs = [(int(g), None) for g in a.games.split(',') if g]
        if a.mixed_first:
            runs.append((a.mixed_first, 'alternating'))
        for G, mixed in runs:
            m = BatchedMatch(*players(), G, size, k)
            first = (np.arange(G) % 2) if mixed else None
            dt, out = timed(lambda: m.play(first=first, seed=7))
            wc = out['win_cnt']
            results.append(dict(board=size, path='BatchedMatch', first=mixed or 'zeros', games=G, seconds=dt,
                                games_per_s=G / dt, mean_plies=float(out['plies'].mean()),
                                win_ratio=(wc[1] + 0.5 * wc[-1]) / G if not mixed else None))
            print(json.dumps(results[-1]), flush=True)
            del m
            torch.cuda.empty_cache()
    print(json.dumps(dict(card=card(), n_playout=a.n_playout, pure_playout=a.pure_playout, results=results)))


if __name__ == '__main__':
    main()
