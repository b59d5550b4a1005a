#!/usr/bin/env python
"""Training-step time of Go networks: ``AlphaZeroAgent.learn`` on the hand-written tensor-core step
(``trainer='native'``) next to PyTorch autograd, with the arms and the FLOP formula of bench.py's ``train`` block.

Arms:
  native                  ResNetTrainer (bf16 tensor-core trunk; 19x19 runs the 20-stride layout) + the re-pack of the
                          inference weights
  autograd                PyTorch autograd, fp32 tensors with TF32 convolutions (PyTorch's default)
  autograd_fp32_strict    the same with cudnn.allow_tf32 = False
  autograd_bf16_autocast  torch.autocast(bf16), channels_last, fused Adam; no inference re-pack

Workloads: config 4's network (19x19 ResNet-20, 17 input planes, 362 actions) at batch 512 and 1024, and Go 9x9
ResNet-6 at batch 1024.  Every arm of a workload is warmed up first; then ``--rounds`` rounds time ``--steps`` steps of
each arm in turn (the arms alternate, so drift in the card's clock hits all of them), with CUDA events.  FLOPs per step
= 3 x flops_per_eval x batch (forward, data gradient, weight gradient).  The card's name and power limit are printed
with the numbers and go into the JSON log.

    python scripts/train_step_go.py [--rounds 3] [--steps 5] [--out profiles/train_step_go.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rlzero_b200.games.gomoku.alphazero_agent import AlphaZeroAgent  # noqa: E402
from rlzero_b200.games.gomoku.policy_value_net import ResNetPolicyValueNet  # noqa: E402

WORKLOADS = (('Go 19x19 ResNet-20 (config 4), batch 512', 19, 20, 512),
             ('Go 19x19 ResNet-20 (config 4), batch 1024', 19, 20, 1024),
             ('Go 9x9 ResNet-6, batch 1024', 9, 6, 1024))
ARMS = ('native', 'autograd', 'autograd_fp32_strict', 'autograd_bf16_autocast')


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout.strip().splitlines()
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q[0] if q else None)


def make_net(H, blocks):
    return ResNetPolicyValueNet(H, n_blocks=blocks, n_actions=H * H + 1, in_planes=17)


def batch(H, B, rs):
    x = (rs.rand(B, 17, H, H) < 0.2).astype(np.float32)
    x[:, 16] = (rs.rand(B, 1, 1) < 0.5)
    pi = rs.dirichlet(0.3 * np.ones(H * H + 1), size=B).astype(np.float32)
    z = rs.choice([-1.0, 0.0, 1.0], size=B).astype(np.float32)
    return (torch.from_numpy(t).cuda() for t in (x, pi, z))


def make_arm(kind, H, blocks, x, pi, z):
    """-> (step function returning the loss, the path description)."""
    torch.manual_seed(0)
    if kind != 'autograd_bf16_autocast':
        strict = kind == 'autograd_fp32_strict'
        agent = AlphaZeroAgent(H, net=make_net(H, blocks), trainer='native' if kind == 'native' else 'autograd')
        assert (agent.trainer is not None) == (kind == 'native')

        def step():
            torch.backends.cudnn.allow_tf32 = not strict
            torch.backends.cuda.matmul.allow_tf32 = False
            return agent.learn(x, pi, z)[0]
        path = ('hand-written kernels (%s)' % type(agent.trainer).__name__ if kind == 'native' else
                'PyTorch autograd, true fp32 convolutions' if strict else 'PyTorch autograd, TF32 convolutions')
        return step, path
    net = make_net(H, blocks).cuda().to(memory_format=torch.channels_last)
    opt = torch.optim.Adam(net.parameters(), lr=1e-3, weight_decay=1e-4, fused=True)
    xc = x.contiguous(memory_format=torch.channels_last)

    def step():
        torch.backends.cudnn.allow_tf32 = True
        net.train()
        with torch.autocast('cuda', dtype=torch.bfloat16):
            lp, v = net(xc)
        loss = F.mse_loss(v.float().view(-1), z) - torch.mean(torch.sum(pi * lp.float(), dim=1))
        opt.zero_grad()
        loss.backward()
        opt.step()
        return loss.detach()
    return step, 'PyTorch autograd, torch.autocast(bf16), channels_last, fused Adam; no inference re-pack'


def run_workload(name, H, blocks, B, rounds, steps, log):
    rs = np.random.RandomState(0)
    x, pi, z = batch(H, B, rs)
    flops = make_net(H, blocks).flops_per_eval()
    arms = {k: make_arm(k, H, blocks, x, pi, z) for k in ARMS}
    for k, (step, _) in arms.items():               # warm-up: module loads, algorithm selection, allocations
        for _ in range(2):
            step()
    torch.cuda.synchronize()
    times = {k: [] for k in ARMS}
    loss = {}
    for _ in range(rounds):
        for k, (step, _) in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                out = step()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / steps)
            loss[k] = float(out)
    entry = {'step': 'AlphaZeroAgent.learn, ' + name, 'board': H, 'blocks': blocks, 'batch': B,
             'flops_per_eval': flops}
    for k in ARMS:
        ms = float(np.median(times[k]))
        entry[k] = {'ms_per_step': ms, 'ms_per_round': times[k], 'samples_per_s': B * 1e3 / ms,
                    'tflops': 3.0 * flops * B / ms / 1e9, 'loss_after': loss[k], 'path': arms[k][1]}
    nat = entry['native']['ms_per_step']
    for k in ARMS[1:]:
        entry['speedup_vs_' + k] = entry[k]['ms_per_step'] / nat
    log('%-45s ' % name + '  '.join('%s %.2f ms (%.0f TFLOP/s)' % (k, entry[k]['ms_per_step'], entry[k]['tflops'])
                                    for k in ARMS))
    del arms
    torch.cuda.empty_cache()
    return entry


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--out', default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'profiles',
                                                  'train_step_go.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('train_step_go.py measures on a CUDA device; none is visible')
    c = card()
    print('card:', c['torch_name'], '|', c['nvidia_smi'], flush=True)
    res = {'card': c, 'rounds': args.rounds, 'steps_per_round': args.steps,
           'includes': 'native / autograd / autograd_fp32_strict: forward, loss, backward, Adam and the re-pack of the '
                       'inference weights (AlphaZeroAgent.learn); autograd_bf16_autocast: forward, loss, backward, Adam',
           'workloads': [run_workload(n, H, b, B, args.rounds, args.steps, lambda s: print(s, flush=True))
                         for n, H, b, B in WORKLOADS]}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
