"""The Philox-4x32-10 restatement (oracle/philox.py) and the playout restatements built on it
(oracle/rollout_oracle.py, rzo_go_rollout_dm in oracle/c/rz_go_oracle.c), on the CPU.

The restatements are what tests/test_gpu_rollout_parity.py holds the device's random playouts and child-order
keys to, bit for bit; here they are pinned to the published Random123 known-answer vectors, to each other, and
(with the draw forced to the first / last candidate) to the fixtures the live reference produced."""
import copy
import ctypes as C
import json
import os

import numpy as np
import pytest

from oracle import dm_oracle, go_oracle, philox, pyoracle, rollout_oracle

HERE = os.path.dirname(os.path.abspath(__file__))

# Random123 kat_vectors, philox4x32_10: (counter, key) -> output
KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


def _seed(key):
    return key[0] | (key[1] << 32)          # rz_philox4: k[0] = low word of the seed, k[1] = high word


@pytest.mark.parametrize('ctr,key,want', KAT)
def test_known_answer_vectors(ctr, key, want):
    assert philox.philox4(*ctr, _seed(key)) == want
    got = philox.philox4_np(*[np.array([c]) for c in ctr], _seed(key))
    assert tuple(int(x) for x in got[:, 0]) == want


def test_scalar_and_vectorised_forms_agree():
    rs = np.random.RandomState(7)
    n = 2000
    ctr = [rs.randint(0, 2 ** 32, size=n, dtype=np.uint64).astype(np.int64) for _ in range(4)]
    ctr[1][:10] = 0
    ctr[3][10:20] = 0xffffffff
    seed = 0x517cc1b727220a95 ^ 12345
    got = philox.philox4_np(*ctr, seed)
    for i in range(0, n, 7):
        assert tuple(int(x) for x in got[:, i]) == philox.philox4(*(int(c[i]) for c in ctr), seed)
    # a per-counter seed array, and the high seed word reaching k1
    seeds = rs.randint(0, 2 ** 63, size=n, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    got = philox.philox4_np(*ctr, seeds)
    for i in range(0, n, 13):
        assert tuple(int(x) for x in got[:, i]) == philox.philox4(*(int(c[i]) for c in ctr), int(seeds[i]))


def test_c_restatement_agrees():
    """rzo_philox4 (oracle/c/rz_go_oracle.c) draws the Go playouts: the same words as the Python form."""
    from oracle import build_oracle
    lib = build_oracle.load()
    out = (C.c_uint32 * 4)()
    for ctr, key, want in KAT:
        lib.rzo_philox4(*ctr, _seed(key), out)
        assert tuple(out) == want
    rs = np.random.RandomState(3)
    for _ in range(200):
        ctr = [int(x) for x in rs.randint(0, 2 ** 32, size=4, dtype=np.uint64)]
        seed = int(rs.randint(0, 2 ** 63, dtype=np.uint64)) * 2 + 1
        lib.rzo_philox4(*ctr, seed, out)
        assert tuple(out) == philox.philox4(*ctr, seed)


def test_uniform_conversions():
    assert philox.u01_53(0, 0) == 0.5 / 2 ** 53
    assert philox.u01_53(0xffffffff, 0xffffffff) == 1.0 - 0.5 / 2 ** 53
    assert philox.u01_53(0x80000000, 0) == 0.5 + 0.5 / 2 ** 53
    assert philox.u01_24(0) == np.float32(0.5 / 2 ** 24)
    assert philox.u01_24(0xffffffff) == np.float32(1.0 - 0.5 / 2 ** 24)
    assert philox.u01_24(0xff) == philox.u01_24(0)          # the low 8 bits are dropped
    assert philox.pick(0, 7) == 0 and philox.pick(0xffffffff, 7) == 6 and philox.pick(0x80000000, 7) == 3


# ------------------------------------------------------------------ the playout restatements
CASES = json.load(open(os.path.join(HERE, 'golden', 'rollout.json')))['cases']


@pytest.mark.parametrize('case', CASES, ids=lambda c: '%dx%d_%s_%d' % (c['size'], c['size'], c['mode'], c['n_playout']))
def test_forced_az_rollout_matches_the_reference_fixtures(case):
    """With the draw forced to r = 0 / n - 1, the restated kernel playout inside RolloutSearch reproduces what the
    live reference's RolloutMCTS produced with its lowest / highest-move rollout policy: this pins the candidate
    order (ascending action), the loop bound and the value rule of the restatement."""
    b = pyoracle.Board(case['size'], case['k'])
    b.reset()
    for m in case['pre']:
        b.step(m)
    s = pyoracle.RolloutSearch(case['n_playout'], 5, rollout=rollout_oracle.AZRollout(0, 0, force=case['mode']))
    move = s.simulate(b)
    assert move == case['move']
    assert s.root_visits(case['size'] ** 2).tolist() == case['visits']
    assert s.root.n == case['root_N'] and s.root.w == case['root_W']


def _random_line_position(rs, board, max_stones):
    while True:
        board.reset()
        ok = True
        for _ in range(rs.randint(0, max_stones + 1)):
            legal = board.leagel_actions()
            board.step(legal[rs.randint(len(legal))])
            if board.game_end_winner()[0]:
                ok = False
                break
        if ok:
            return board


def test_az_rollout_loop_bound_and_value_rule():
    """A playout whose last allowed move ends the game is a tie (the status is tested before each move only); the
    same playout with one more move allowed is a decisive -1."""
    rs = np.random.RandomState(11)
    seen = 0
    for _ in range(400):
        b = _random_line_position(rs, pyoracle.Board(3, 3), 8)
        pos = rollout_oracle.LinePos.of(b)
        full = rollout_oracle.az_rollout(pos, 5, 3, pos.stones, 99, 1000)
        # plies the unlimited playout took: replay it ply by ply
        for n in range(0, 10):
            v = rollout_oracle.az_rollout(pos, 5, 3, pos.stones, 99, n)
            if v != 0:
                assert v == -1.0 and v == full
                assert rollout_oracle.az_rollout(pos, 5, 3, pos.stones, 99, n - 1) == 0
                seen += 1
                break
    assert seen > 50


def _py_go_rollouts(pos, g, visit, seed, n_limit, n_rollouts):
    """rz_eval_rollout_dm_kernel<rz_go_game> once more, over go_oracle.Position (independent of the C port)."""
    n = pos.N
    s0 = s1 = 0
    for r in range(n_rollouts):
        p = pos
        for i in range(n_limit + 1):
            if p.is_game_over() or i == n_limit:
                break
            cand = [int(a) for a in np.nonzero(p.all_legal_moves()[:n * n])[0]] + [n * n]
            a = cand[philox.pick(philox.philox4(g, visit, (r << 16) | i, 0xd311, seed)[0], len(cand))]
            p = p.play_move(go_oracle.from_flat(n, a))
        if p.is_game_over():
            r0 = 1 if p.result() == 1 else -1
            s0 += r0
            s1 -= r0
    return [s0 / n_rollouts, s1 / n_rollouts]


def test_go_rollouts_c_and_python_agree():
    rs = np.random.RandomState(5)
    for trial in range(6):
        n = 4 if trial < 3 else 5
        b = go_oracle.GoSearchBoard(n, 0.5)
        for _ in range(rs.randint(0, 12)):
            legal = b.leagel_actions()
            b.step(legal[rs.randint(len(legal))])
            if b.game_end_winner()[0]:
                b.reset()
        for n_limit in (0, 3, 60):
            want = _py_go_rollouts(b.pos, 7 + trial, trial, 1234 + trial, n_limit, 3)
            got, legal = rollout_oracle.go_dm_rollout(b.pos, 7 + trial, trial, 1234 + trial, n_limit, 3)
            assert got == want
            assert legal.tolist() == b.pos.all_legal_moves().tolist()


def test_dm_rollout_counts_a_game_ended_by_the_last_allowed_move():
    """rz_eval_rollout_dm tests the status once more after n_limit moves: one empty square left, n_limit = 1, the
    move completes a line -> a decided playout; the AlphaZero evaluator calls the same one-move playout a tie."""
    rs = np.random.RandomState(2)
    found = 0
    while found < 5:
        b = pyoracle.DMBoard(3, 3, zero_sum=True)
        b.reset()
        order = [int(a) for a in rs.permutation(9)]
        for a in order[:8]:
            b.step(a)
            if b.game_end_winner()[0]:
                break
        if b.game_end_winner()[0]:
            continue
        after = copy.deepcopy(b)
        after.step(order[8])
        end, winner = after.game_end_winner()
        if winner < 0:
            continue
        found += 1
        pos = rollout_oracle.LinePos.of(b)
        want = [1.0, -1.0] if winner == 0 else [-1.0, 1.0]
        assert rollout_oracle.dm_rollout(pos, 0, 0, 0, 1, 4, 0, rollout_oracle.RETURNS_ZERO_SUM) == want
        assert rollout_oracle.dm_rollout(pos, 0, 0, 0, 0, 4, 0, rollout_oracle.RETURNS_ZERO_SUM) == [0.0, 0.0]
        ref = [1.0, -1.0] if winner == 1 else [0.0, 0.0]            # GomokuEnv.returns: winner == 1 only
        assert rollout_oracle.dm_rollout(pos, 0, 0, 0, 1, 4, 0, rollout_oracle.RETURNS_REFERENCE) == ref
        assert rollout_oracle.az_rollout(pos, 0, 0, pos.stones, 0, 1) == 0.0
        assert rollout_oracle.az_rollout(pos, 0, 0, pos.stones, 0, 2) == -1.0


def test_shuffle_rank_orders_every_new_node():
    """ShuffleRank inside DMSearch: every node's children are a permutation of its legal actions, sorted by the
    restated key; the node indices are the device's allocation order (0 = the root, one per evaluated leaf)."""
    b = pyoracle.DMBoard(4, 3, zero_sum=True)
    b.reset()
    ev = rollout_oracle.DMRollout(0, 9, n_rollouts=2, returns_mode=rollout_oracle.RETURNS_ZERO_SUM)
    sh = rollout_oracle.ShuffleRank(0, 0, 0, 9)
    s = dm_oracle.DMSearch(ev, 60, 2, 'uct', solve=True, shuffle_fn=sh)
    ev.search = sh.search = s
    root = s.search(b)
    assert root.index == 0 and s.n_nodes > 1
    stack, seen = [root], set()
    while stack:
        nd = stack.pop()
        if nd.children:
            acts = [c.action for c in nd.children]
            keys = [(rollout_oracle.shuffle_rank(0, 0, 0, nd.index, a, 9), a) for a in acts]
            assert keys == sorted(keys) and len(set(acts)) == len(acts)
            stack.extend(nd.children)
        if nd.index >= 0:
            assert nd.index not in seen
            seen.add(nd.index)
    assert seen == set(range(s.n_nodes))

