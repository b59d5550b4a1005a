"""Multi-GPU plumbing around the self-play path (one process per GPU, ``torch.distributed``).

Self-play games are independent (the reference plays them one after another,
tools/train_alphazero.py:81-90), so they shard over ranks with NO collective on the search path:
rank r owns global game ids ``[r*G, (r+1)*G)`` and every per-game random stream is keyed by the
global id, which makes results independent of the shard count (SURVEY.md 8e).

The only exchanges are off the hot path, once per generation / training step:

* ``gather_records_device`` -- the finished plies of every rank as COMPACT device records (the
  trajectory ring's own format: two row-bitboards, 6 info words, pi -- 1.2 KB per ply at 15x15
  against 4.5 KB for float32 planes + pi), one NCCL all-gather on device tensors, no host hop for
  the payload; the 8-fold augmentation (``rz_augment_equi``; Go: ``GoReplayBuffer``) then expands them on the
  receiving GPU;
* ``broadcast_weights``     -- after ``AlphaZeroAgent.learn`` on the learner rank the parameters and
  buffers of the policy-value module go to every rank in one flat buffer per dtype, which then
  re-packs them for the kernels (``refresh_weights``; the captured wave graph is re-captured);
* ``generation_step``       -- the loop body: drain -> gather -> augment -> learn -> broadcast.

``gather_trajectories`` is the host-array variant (numpy in, numpy out) for callers that hold
``BatchedSelfPlay.drain()`` output.  Backend: NCCL over NVLink on the GPUs; the same code runs on
``gloo`` with CPU tensors in the tests.
"""
import numpy as np
import torch
import torch.distributed as dist


def shard_range(n_global_games, rank=None, world=None):
    """[lo, hi) global game ids of this rank: contiguous blocks, remainder to the low ranks."""
    rank = dist.get_rank() if rank is None else rank
    world = dist.get_world_size() if world is None else world
    base, rem = divmod(int(n_global_games), world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def _device_for_backend():
    if dist.get_backend() == 'nccl':
        return torch.device('cuda', torch.cuda.current_device())
    return torch.device('cpu')


def _counts(n, group):
    world = dist.get_world_size(group)
    dev = _device_for_backend()
    mine = torch.tensor([int(n)], dtype=torch.int64, device=dev)
    every = torch.empty(world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(every, mine, group=group)
    return every.cpu().tolist()


def pack_records(rows, info, pi):
    """rows int32 [n,2,H], info int32 [n,6], pi float32 [n,AS]  ->  one int32 tensor [n, 2H + 6 + AS]
    (pi bit-cast), the unit of the trajectory exchange."""
    n = int(info.shape[0])
    w_rows, w_info, w_pi = int(rows.shape[1] * rows.shape[2]), int(info.shape[1]), int(pi.shape[1])
    return torch.cat([rows.reshape(n, w_rows).to(torch.int32), info.reshape(n, w_info).to(torch.int32),
                      pi.reshape(n, w_pi).contiguous().view(torch.int32)], dim=1).contiguous()


def unpack_records(packed, board_size, info_words=6):
    H = int(board_size)
    n = int(packed.shape[0])
    rows = packed[:, :2 * H].reshape(n, 2, H).contiguous()
    info = packed[:, 2 * H:2 * H + info_words].contiguous()
    pi = packed[:, 2 * H + info_words:].contiguous().view(torch.float32)
    return rows, info, pi


def gather_records_device(rows, info, pi, global_offset=0, group=None):
    """All-gather ragged per-rank trajectory records that stay on the device.

    ``rows/info/pi``: this rank's drained plies (``SearchForest.drain_trajectories_device``).  Column 3 of ``info``
    (the LOCAL game slot) is rewritten to the GLOBAL game id ``global_offset + slot`` before it travels.  Returns
    ``(rows, info, pi, counts)``: the concatenation over ranks in rank order (device tensors) and the per-rank
    record counts.  One collective for the payload, one 8-byte collective for the counts."""
    world = dist.get_world_size(group)
    dev = _device_for_backend()
    H = int(rows.shape[-1])
    info = info.clone()
    if info.shape[0]:
        info[:, 3] += int(global_offset)
    packed = pack_records(rows.to(dev), info.to(dev), pi.to(dev))
    counts = _counts(packed.shape[0], group)
    n_max, width = max(counts), int(packed.shape[1])
    if n_max == 0:
        return rows, info, pi, counts
    send = torch.zeros(n_max, width, dtype=torch.int32, device=dev)
    send[:packed.shape[0]] = packed
    recv = torch.empty(world * n_max, width, dtype=torch.int32, device=dev)
    dist.all_gather_into_tensor(recv, send, group=group)
    keep = torch.cat([torch.arange(r * n_max, r * n_max + c, device=dev) for r, c in enumerate(counts)])
    out = recv[keep]
    r, i, p = unpack_records(out, H, info.shape[1])
    return r, i, p, counts


def gather_trajectories(states, pis, zs, info=None, group=None):
    """All-gather ragged per-rank trajectory records held as host arrays.

    states float32 [n,4,H,W], pis float32 [n,A], zs float32 [n], info int32 [n,6] (optional; column
    3 is the LOCAL slot, column 4 the episode, column 5 the ply -- see include/rlzero_b200.h
    ``ring_info``).  Every rank returns the concatenation over ranks in rank order.
    """
    world = dist.get_world_size(group)
    dev = _device_for_backend()
    n = int(len(zs))
    counts = _counts(n, group)
    n_max = max(counts) if counts else 0
    out = []
    for arr in (states, pis, zs, info):
        if arr is None:
            out.append(None)
            continue
        t = torch.as_tensor(np.ascontiguousarray(arr))
        pad = torch.zeros((n_max,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
        pad[:n] = t.to(dev)
        bufs = [torch.empty_like(pad) for _ in range(world)]
        dist.all_gather(bufs, pad, group=group)
        out.append(torch.cat([b[:c] for b, c in zip(bufs, counts)]).cpu().numpy())
    return tuple(out) + (counts,)


def broadcast_weights(module, src=0, group=None):
    """Broadcast parameters and buffers of ``module`` from rank ``src`` (flattened: one collective
    per dtype, sized for launch latency, not link count).  Returns the bytes moved."""
    dev = _device_for_backend()
    tensors = [p.data for p in module.parameters()] + [b.data for b in module.buffers()]
    by_dtype = {}
    for t in tensors:
        by_dtype.setdefault(t.dtype, []).append(t)
    moved = 0
    for dtype, ts in by_dtype.items():
        flat = torch.cat([t.reshape(-1).to(dev) for t in ts])
        dist.broadcast(flat, src=src, group=group)
        moved += flat.numel() * flat.element_size()
        off = 0
        for t in ts:
            k = t.numel()
            t.copy_(flat[off:off + k].reshape(t.shape).to(t.device))
            off += k
    return moved


def generation_step(selfplay, agent, n_moves=1, batch_size=512, epochs=1, learner=0, group=None, augment=True):
    """One generation of the multi-GPU loop: every rank plays ``n_moves`` moves of its games, the finished plies
    are all-gathered as compact device records, the learner rank augments them (8 symmetries, rz_augment_equi) and
    runs ``epochs`` ``AlphaZeroAgent.learn`` steps on mini-batches of them, the new weights are broadcast and every
    rank re-packs them (its captured wave graph is re-captured on the next wave).  Returns a dict of counters.

    Go: the learner packs the records into a ``GoReplayBuffer`` of this generation (17 planes, the history rebuilt
    from the preceding plies of each episode) and every epoch expands ``batch_size`` distinct (record, symmetry)
    pairs of the 8n.  The gathered records keep each rank's drain order, and column 3 of ``info`` holds global game
    ids, so an episode's plies stay contiguous and distinct from other ranks' episodes: the history is rebuilt across
    ranks as on one."""
    from .train_pipeline import GoReplayBuffer, augment_equi_device
    f = selfplay.forest
    selfplay.play(n_moves)
    rec = f.drain_trajectories_device()
    rows, info, pi, counts = gather_records_device(rec['rows'], rec['info'], rec['pi'],
                                                   global_offset=int(f.desc.global_offset), group=group)
    loss = None
    n = int(info.shape[0])
    if dist.get_rank(group) == learner and n > 0 and f.is_go:
        buf = GoReplayBuffer(n, f.H, device=rows.device)
        buf.extend(rows, info, pi)
        g = torch.Generator(device='cpu')
        g.manual_seed(n)
        for _ in range(epochs):
            k = torch.randperm(8 * n, generator=g)[:batch_size].to(rows.device)
            loss, _ = agent.learn(*buf.expand(k // 8, k % 8))
    elif dist.get_rank(group) == learner and n > 0:
        if augment:
            states, pis, zs = augment_equi_device(f.gdesc, rows, info, pi)
        else:
            raise NotImplementedError('generation_step trains on the augmented records')
        g = torch.Generator(device='cpu')
        g.manual_seed(n)
        for _ in range(epochs):
            idx = torch.randperm(states.shape[0], generator=g)[:batch_size].to(states.device)
            loss, _ = agent.learn(states[idx], pis[idx], zs[idx])
    moved = broadcast_weights(agent.policy_value_net, src=learner, group=group)
    if getattr(agent, 'trainer', None) is not None:
        agent.trainer.weights_changed()        # the trainer's own packed copies (non-learner ranks may train later)
    agent.native.refresh_weights()
    return dict(records=n, per_rank=counts, loss=loss, weight_bytes=moved)
