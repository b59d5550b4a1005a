#!/usr/bin/env python
"""The multi-GPU generation loop on real GPUs (SURVEY 8 e1 / north star: NCCL only off the search path):

    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 scripts/generation_loop.py [generations] [--go]

Every rank plays its shard of the games (global ids rank*G ..), the finished plies are all-gathered as compact device
records, rank 0 augments them and runs the native training step, the weights are broadcast, every rank re-packs them and
its captured wave graph is re-captured.  Prints one JSON line per generation from rank 0; asserts that all ranks hold
bit-identical weights after every broadcast and that the search really runs on the new weights.

``--go``: 9x9 Go with a 17-plane ResNet on the tensor-core training step (trainer='native'), games capped at 60 moves
and started from the empty board (a set-up start would lack its history planes), 30 moves per generation; rank 0
trains on the 17 planes and 8 symmetries of a GoReplayBuffer."""
import json
import os
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rlzero_b200 import _lib as L  # noqa: E402
from rlzero_b200 import parallel  # noqa: E402
from rlzero_b200.games.gomoku.alphazero_agent import AlphaZeroAgent  # noqa: E402
from rlzero_b200.games.gomoku.policy_value_net import ResNetPolicyValueNet  # noqa: E402
from rlzero_b200.selfplay import BatchedSelfPlay  # noqa: E402


def main():
    pos = [a for a in sys.argv[1:] if not a.startswith('--')]
    gens = int(pos[0]) if pos else 4
    go = '--go' in sys.argv[1:]
    rank, world, local = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1)), int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    H, G, P = 9, 1024, 32
    torch.manual_seed(0)                                   # the same initial weights on every rank
    if go:
        agent = AlphaZeroAgent(H, net=ResNetPolicyValueNet(H, n_blocks=3, n_actions=H * H + 1, in_planes=17),
                               learning_rate=2e-3, trainer='native')
        sp = BatchedSelfPlay(G, H, 1, evaluator=agent.native, n_playout=P, add_noise=True, global_offset=rank * G, seed=3,
                             ring_capacity=1 << 17, game_type=L.GAME_GO, komi=7.5, max_moves=60)
    else:
        agent = AlphaZeroAgent(H, net=ResNetPolicyValueNet(H, n_blocks=3), learning_rate=2e-3)
        sp = BatchedSelfPlay(G, H, 5, evaluator=agent.native, n_playout=P, add_noise=True, global_offset=rank * G, seed=3,
                             ring_capacity=1 << 17)
        sp.set_random_start_positions(max_random_moves=40)
    for gen in range(gens):
        t0 = time.time()
        version = agent.native.weights_version
        out = parallel.generation_step(sp, agent, n_moves=30 if go else 12, batch_size=1024, epochs=4, learner=0)
        torch.cuda.synchronize()
        # every rank holds the learner's weights, bit for bit
        flat = torch.cat([p.detach().reshape(-1).double() for p in agent.policy_value_net.parameters()])
        h = torch.stack([flat.sum(), (flat * torch.arange(flat.numel(), device=flat.device, dtype=torch.float64)).sum()])
        hs = [torch.empty_like(h) for _ in range(world)]
        dist.all_gather(hs, h)
        assert all(torch.equal(hs[0], x) for x in hs), 'weights differ between ranks after the broadcast'
        assert agent.native.weights_version > version
        sp.step_wave()                                     # re-captures the wave graph with the new weights
        assert sp._graph_version == agent.native.weights_version
        if rank == 0:
            print(json.dumps({'game': 'go' if go else 'gomoku', 'generation': gen, 'records_gathered': out['records'],
                              'per_rank': out['per_rank'], 'loss': out['loss'], 'weight_bytes': out['weight_bytes'], 'seconds': time.time() - t0,
                              'games_done_rank0': sp.stats()['games_done']}), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
