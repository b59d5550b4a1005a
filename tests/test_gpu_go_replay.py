"""GPU tests of the compact Go replay buffer (GoReplayBuffer: rz_go_records_pack / rz_go_records_expand): the expanded
17 planes, pi and z equal the host route (BatchedSelfPlay._go_states) bit for bit and GoEnv.observe of the oracle, the 8
symmetries are the numpy maps on planes and policy alike, the ring keeps the newest records with the history they were
packed with, and parallel.generation_step trains a Go network from them."""
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _go_net(n, blocks, seed=0):
    from rlzero_b200.games.gomoku.policy_value_net import ResNetPolicyValueNet
    torch.manual_seed(seed)
    return ResNetPolicyValueNet(n, n_blocks=blocks, n_actions=n * n + 1, in_planes=17).cuda().eval()


def _selfplay(n, G=4, max_moves=12, ring_capacity=4096, seed=5, random_start=False, moves=40):
    from rlzero_b200 import _lib as L
    from rlzero_b200.selfplay import BatchedSelfPlay
    sp = BatchedSelfPlay(G, n, 1, net=_go_net(n, 1, seed=seed), n_playout=8, temperature=1.0, add_noise=True, seed=seed,
                         game_type=L.GAME_GO, komi=0.5, max_moves=max_moves, ring_capacity=ring_capacity)
    if random_start:
        sp.set_random_start_positions(max_random_moves=5)
    sp.play(moves)
    torch.cuda.synchronize()
    sp.forest.raise_faults()
    return sp


def _host_states(H, rows, info):
    """BatchedSelfPlay._go_states on host arrays (it only needs the board's geometry)."""
    from rlzero_b200.selfplay import BatchedSelfPlay
    fake = types.SimpleNamespace(forest=types.SimpleNamespace(H=H, W=H))
    return BatchedSelfPlay._go_states(fake, np.asarray(rows).view(np.uint32), np.asarray(info))


def _host(rec):
    return rec['rows'].cpu().numpy().view(np.uint32), rec['info'].cpu().numpy(), rec['pi'].cpu().numpy()


def _expand_all(buf, sym=6):
    n = len(buf)
    return [t.cpu().numpy() for t in buf.expand(np.arange(n), np.full(n, sym))]


@pytest.mark.parametrize('n,case', [(5, 'plain'), (9, 'plain'), (5, 'overflow'), (9, 'random_start')])
def test_expansion_equals_the_host_route_bit_for_bit(n, case):
    """drain_trajectories_device -> GoReplayBuffer.extend -> expand(i, 6) == _go_states, pi[:, :A], info[:, 2].
    'overflow': the ring is smaller than what was played, so the first episode of the drain is partial; 'random_start':
    games set up with set_random_start_positions (both routes lack the set-up's history alike)."""
    from rlzero_b200.train_pipeline import GoReplayBuffer
    sp = _selfplay(n, ring_capacity=30 if case == 'overflow' else 4096, random_start=case == 'random_start')
    rec = sp.forest.drain_trajectories_device()
    if case == 'overflow':
        assert rec['dropped'] > 0
        cut = 1 if int(rec['info'][0, 5]) == 0 else 0         # start inside an episode even if the ring cut at one
        rec = {k: rec[k][cut:] for k in ('rows', 'info', 'pi')}
    rows, info, pi = _host(rec)
    N, A = len(info), n * n + 1
    assert N > 0 and sp.stats()['games_done'] >= 2 * sp.G
    if case == 'overflow':
        assert info[0, 5] > 0
    else:
        assert len(set(map(tuple, info[:, 3:5]))) >= 2 * sp.G
    buf = GoReplayBuffer(N, n)
    buf.extend(rec['rows'], rec['info'], rec['pi'])
    s, p, z = _expand_all(buf)
    want = sp._go_states(rows, info)
    assert s.shape == (N, 17, n, n) and s.dtype == np.float32
    assert np.array_equal(s.view(np.uint32), want.view(np.uint32))
    assert np.array_equal(p.view(np.uint32), pi[:, :A].view(np.uint32))
    assert np.array_equal(z, info[:, 2].astype(np.float32))
    assert s[:, 2:16].any()                                   # the history planes are not all empty


def test_expansion_equals_the_oracle_observation():
    """Episodes from the empty board replayed on GoEnvOracle: every expanded position is GoEnv.observe."""
    from oracle.go_oracle import GoEnvOracle
    from rlzero_b200.train_pipeline import GoReplayBuffer
    n = 5
    sp = _selfplay(n, max_moves=30, moves=64, seed=4)
    rec = sp.forest.drain_trajectories_device()
    info = rec['info'].cpu().numpy()
    buf = GoReplayBuffer(len(info), n)
    buf.extend(rec['rows'], rec['info'], rec['pi'])
    states = _expand_all(buf)[0]
    checked = 0
    for slot, ep in sorted(set((int(a), int(b)) for a, b in info[:, 3:5])):
        sel = np.nonzero((info[:, 3] == slot) & (info[:, 4] == ep))[0]
        assert list(info[sel, 5]) == list(range(len(sel)))
        env = GoEnvOracle(n, 0.5)
        env.reset()
        for j, i in enumerate(sel):
            want = env.observe(env.agent_selection)['observation'].transpose(2, 0, 1).astype(np.float32)
            assert np.array_equal(states[i], want), (slot, ep, j)
            if j + 1 < len(sel):
                env.step(int(info[sel[j + 1], 1]))
            checked += 1
    assert checked == len(info) > 0


def _np_sym(x, s):
    """Symmetry s on the last two axes: np.rot90 (s // 2 + 1) times, then np.fliplr when s is odd."""
    y = np.rot90(x, s // 2 + 1, axes=(-2, -1))
    return np.flip(y, axis=-1) if s & 1 else y


def _random_records(H, N, seed, slot=0, episode=0, ply0=0):
    """One synthetic episode of N plies: random boards (any bits; the kernels only move data), alternating movers."""
    rs = np.random.RandomState(seed)
    A = H * H + 1
    AS = (A + 31) // 32 * 32
    rows = rs.randint(0, 1 << H, size=(N, 2, H)).astype(np.int32)
    info = np.zeros((N, 6), dtype=np.int32)
    info[:, 5] = ply0 + np.arange(N)
    info[:, 0] = info[:, 5] % 2
    info[:, 1] = rs.randint(0, A, size=N)
    info[:, 2] = rs.choice([-1, 1], size=N)
    info[:, 3], info[:, 4] = slot, episode
    pi = np.zeros((N, AS), dtype=np.float32)
    pi[:, :A] = rs.dirichlet(np.ones(A), size=N)
    return rows, info, pi


def _dev(*arrays):
    return [torch.from_numpy(a).cuda() for a in arrays]


@pytest.mark.parametrize('H', [5, 9, 19])
def test_symmetries_are_the_numpy_maps_on_planes_and_policy(H):
    from rlzero_b200.train_pipeline import GoReplayBuffer
    rows, info, pi = _random_records(H, 12, seed=H)
    buf = GoReplayBuffer(12, H)
    buf.extend(*_dev(rows, info, pi))
    HW = H * H
    for i in (1, 5, 11):                                      # (record 0, at ply 0, has empty planes)
        s6, p6, z6 = [t.cpu().numpy() for t in buf.expand([i], [6])]
        outs = []
        for s in range(8):
            st, p, z = [t.cpu().numpy() for t in buf.expand([i], [s])]
            assert np.array_equal(st[0], _np_sym(s6[0], s)), (i, s)
            assert np.array_equal(p[0, :HW], _np_sym(p6[0, :HW].reshape(H, H), s).reshape(-1)), (i, s)
            assert p[0, HW] == p6[0, HW] and z[0] == z6[0]
            outs.append(st[0].tobytes())
        assert len(set(outs)) == 8                            # an asymmetric position has 8 distinct images
    # one black stone off every axis of symmetry, pi one-hot on its square: stone and mass stay together
    r, c = (0, 1) if H == 5 else (2, 5)
    rows = np.zeros((1, 2, H), dtype=np.int32)
    rows[0, 0, r] = 1 << c
    info = np.array([[1, r * H + c, 1, 0, 0, 1]], dtype=np.int32)
    pi = np.zeros((1, (HW + 1 + 31) // 32 * 32), dtype=np.float32)
    pi[0, r * H + c] = 1.0
    buf = GoReplayBuffer(1, H)
    buf.extend(*_dev(rows, info, pi))
    squares = set()
    for s in range(8):
        st, p, _ = [t.cpu().numpy() for t in buf.expand([0], [s])]
        stone = np.argwhere(st[0, 0] == 1.0)
        assert len(stone) == 1 and st[0, 1:16].sum() == 0 and st[0, 16].min() == 1.0
        assert int(np.argmax(p[0])) == stone[0][0] * H + stone[0][1] and p[0].max() == 1.0
        squares.add(tuple(stone[0]))
    assert len(squares) == 8


def test_ring_keeps_the_newest_records_with_their_history():
    from rlzero_b200.train_pipeline import GoReplayBuffer
    H = 9
    A = H * H + 1
    a = _random_records(H, 8, seed=1, slot=0, episode=0)
    b = _random_records(H, 5, seed=2, slot=1, episode=0)
    # wrap-around: 8 then 5 records into 10 slots keep a[3:] + b, and a[3:] keep the history of the evicted a[:3]
    buf = GoReplayBuffer(10, H)
    buf.extend(*_dev(*a))
    buf.extend(*_dev(*b))
    assert len(buf) == 10
    want = np.concatenate([_host_states(H, a[0], a[1])[3:], _host_states(H, b[0], b[1])])
    s, p, z = _expand_all(buf)
    assert np.array_equal(s, want) and s[0, 2:8].any()
    assert np.array_equal(p, np.concatenate([a[2][3:, :A], b[2][:, :A]]))
    assert np.array_equal(z, np.concatenate([a[1][3:, 2], b[1][:, 2]]).astype(np.float32))
    # the history survives later wraps: 4 more records evict a[3:7]; a[7] still carries a[0..6]
    c = _random_records(H, 4, seed=3, slot=2, episode=0)
    buf.extend(*_dev(*c))
    s = _expand_all(buf)[0]
    assert np.array_equal(s[0], _host_states(H, a[0], a[1])[7]) and s[0, 12:14].any()     # entry 6 = a[1]
    assert np.array_equal(s[-4:], _host_states(H, c[0], c[1]))
    # one extend larger than the ring: the newest 10 of 25, with the history of the inputs that were not kept
    d = _random_records(H, 25, seed=4, slot=3, episode=7, ply0=2)
    buf = GoReplayBuffer(10, H)
    buf.extend(*_dev(*_random_records(H, 3, seed=5)))
    buf.extend(*_dev(*d))
    assert len(buf) == 10
    s, p, z = _expand_all(buf)
    assert np.array_equal(s, _host_states(H, d[0], d[1])[-10:]) and s[0, 14:16].any()
    assert np.array_equal(p, d[2][-10:, :A]) and np.array_equal(z, d[1][-10:, 2].astype(np.float32))


def test_sample_draws_distinct_pairs_reproducibly():
    from rlzero_b200.train_pipeline import GoReplayBuffer
    H = 9
    buf = GoReplayBuffer(16, H)
    buf.extend(*_dev(*_random_records(H, 6, seed=9)))
    total = 8 * len(buf)
    gen = lambda: torch.Generator(device='cuda').manual_seed(123)
    s1, p1, z1 = buf.sample(total, generator=gen())
    s2, p2, z2 = buf.sample(total, generator=gen())
    assert torch.equal(s1, s2) and torch.equal(p1, p2) and torch.equal(z1, z2)
    assert s1.shape == (total, 17, H, H) and p1.shape == (total, H * H + 1) and z1.shape == (total,)
    # every one of the 8 * len pairs exactly once
    k = torch.randperm(total, generator=gen(), device='cuda')
    se, pe, ze = buf.expand(k // 8, k % 8)
    assert torch.equal(s1, se) and torch.equal(p1, pe) and torch.equal(z1, ze)
    assert sorted(k.tolist()) == list(range(total))
    flat = np.concatenate([s1.reshape(total, -1).cpu().numpy(), p1.cpu().numpy()], axis=1)
    assert len({row.tobytes() for row in flat}) == total
    s3 = buf.sample(7, generator=gen())[0]
    assert torch.equal(s3, s1[:7])
    with pytest.raises(ValueError):
        buf.sample(total + 1)


def test_generation_step_trains_go_from_the_compact_buffer(tmp_path):
    """A one-process NCCL world: two generation_step calls on 9x9 Go self-play with a trainer='native' agent count the
    records, return a finite loss, advance weights_version and re-capture the wave graph; then learn() on
    GoReplayBuffer.sample batches lowers the loss."""
    import torch.distributed as dist
    from rlzero_b200 import _lib as L
    from rlzero_b200 import parallel
    from rlzero_b200.games.gomoku.alphazero_agent import AlphaZeroAgent
    from rlzero_b200.learn import ResNetTrainer
    from rlzero_b200.selfplay import BatchedSelfPlay
    from rlzero_b200.train_pipeline import GoReplayBuffer
    H = 9
    torch.cuda.set_device(0)
    dist.init_process_group('nccl', store=dist.FileStore(str(tmp_path / 'store'), 1), rank=0, world_size=1,
                            device_id=torch.device('cuda', 0))
    try:
        agent = AlphaZeroAgent(H, net=_go_net(H, 2, seed=1), learning_rate=2e-3, trainer='native')
        assert isinstance(agent.trainer, ResNetTrainer)
        sp = BatchedSelfPlay(32, H, 1, evaluator=agent.native, n_playout=8, add_noise=True, seed=3, game_type=L.GAME_GO,
                             komi=7.5, max_moves=16, ring_capacity=1 << 14)
        total = 0
        for _ in range(2):
            version = agent.native.weights_version
            out = parallel.generation_step(sp, agent, n_moves=20, batch_size=256, epochs=2)
            torch.cuda.synchronize()
            assert out['records'] > 0 and out['per_rank'] == [out['records']]
            assert out['loss'] is not None and np.isfinite(out['loss'])
            assert agent.native.weights_version > version
            sp.step_wave()                                    # re-captures the wave graph on the new weights
            assert sp._graph is not None and sp._graph_version == agent.native.weights_version
            total += out['records']
        assert total <= sp.stats()['plies_done']
    finally:
        dist.destroy_process_group()
    sp.play(40)
    rec = sp.forest.drain_trajectories_device()
    buf = GoReplayBuffer(1 << 14, H)
    buf.extend(rec['rows'], rec['info'], rec['pi'])
    g = torch.Generator(device='cuda').manual_seed(0)
    losses = [agent.learn(*buf.sample(256, generator=g))[0] for _ in range(40)]
    print('loss', ['%.3f' % u for u in losses])
    assert np.all(np.isfinite(losses)) and np.mean(losses[-5:]) < np.mean(losses[:5]) - 0.2
