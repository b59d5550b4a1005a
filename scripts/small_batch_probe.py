#!/usr/bin/env python
"""Small-batch wave latency: G games of Gomoku 15x15 on ResNet-10 (24 launches per wave), the graph-replayed wave timed
with CUDA events; with RZ_EAGER=1 a few eager waves at G = RZ_G for an ncu launch list."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rlzero_b200.games.gomoku.policy_value_net import ResNetPolicyValueNet  # noqa: E402
from rlzero_b200.selfplay import BatchedSelfPlay  # noqa: E402

torch.manual_seed(0)
net = ResNetPolicyValueNet(15, n_blocks=10).cuda().eval()
if os.environ.get('RZ_EAGER'):
    sp = BatchedSelfPlay(int(os.environ.get('RZ_G', '1')), 15, 5, net=net, n_playout=800, add_noise=True, seed=1)
    sp.set_random_start_positions()
    for _ in range(12):
        sp._wave()
    torch.cuda.synchronize()
    sys.exit(0)
for G in [int(g) for g in os.environ.get('RZ_GS', '1,8,64,512').split(',')]:
    sp = BatchedSelfPlay(G, 15, 5, net=net, n_playout=800, add_noise=True, seed=1)
    sp.set_random_start_positions()
    sp.warm_up()
    for _ in range(50):
        sp.step_wave()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(400):
        sp.step_wave()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1000 / 400
    print(json.dumps({'games': G, 'us_per_wave': us, 'sims_per_s': G / us * 1e6, 'pdl': os.environ.get('RZ_PDL', '1')}),
          flush=True)
