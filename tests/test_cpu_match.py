"""CPU side of the evaluation match: rz_match_commit's argument checks (host-side, no launch), the restated match
(oracle/match_oracle.py) against the single-game restatement, and the restated root-policy draw on hand-worked
cases."""
import ctypes as C

import numpy as np
import pytest

from oracle import match_oracle as mo
from oracle import pyoracle
from oracle.evaluators import EVAL_HASH, EVAL_KAT, make_policy_value_fn


@pytest.fixture(scope='module')
def lib():
    from rlzero_b200 import build
    build.build()
    from rlzero_b200 import _lib
    return _lib.load()


def _desc(H=6, W=6, k=4, G=4, game_type=0):
    """A descriptor that passes rz_check_tree: fake non-null pointers, nothing is launched."""
    from rlzero_b200 import _lib as L
    A = W if game_type == L.GAME_CONNECT4 else H * W + int(game_type == L.GAME_GO)
    t = L.TreeDesc()
    t.game = L.GameDesc(H, k, A, (A + 31) // 32 * 32, W, game_type)
    t.n_trees, t.max_nodes, t.max_depth, t.rule, t.ln_table_len, t.store_priors = G, 16, H * W + 1, 0, 64, 1
    for i, (name, _) in enumerate(L.TreeDesc._fields_):
        if name in ('edge_N', 'edge_W', 'edge_P', 'edge_child', 'node_parent', 'node_paction', 'n_nodes', 'root_N',
                    'root_W', 'root_rows', 'root_meta', 'path_node', 'path_action', 'depth', 'leaf_rows',
                    'leaf_meta', 'ln_table'):
            setattr(t, name, 0x1000 * (i + 1))
    return t


def _commit(lib, t0, t1, log=0x8000, max_plies=36):
    return lib.rz_match_commit(C.byref(t0), C.byref(t1), None, None, log, max_plies, None)


def test_commit_accepts_the_reference_configuration(lib):
    # n_trees = 0: every check runs, nothing is launched
    assert _commit(lib, _desc(G=0), _desc(G=0)) == 0, lib.rz_last_error()


def _reject(lib, t0, t1, what, **kw):
    assert _commit(lib, t0, t1, **kw) != 0
    assert what in lib.rz_last_error(), lib.rz_last_error()


def test_commit_rejects_mismatched_seats(lib):
    _reject(lib, _desc(), _desc(k=5), b'game descriptors differ')
    _reject(lib, _desc(), _desc(H=5, W=5), b'game descriptors differ')
    _reject(lib, _desc(G=4), _desc(G=5), b'n_trees')


def test_commit_rejects_unsupported_searches(lib):
    from rlzero_b200 import _lib as L
    go0, go1 = _desc(H=5, W=5, k=1, game_type=L.GAME_GO), _desc(H=5, W=5, k=1, game_type=L.GAME_GO)
    for t in (go0, go1):
        t.root_hist, t.leaf_hist = 0x100000, 0x200000
    _reject(lib, go0, go1, b'Go', max_plies=25)
    dm = _desc()
    dm.flavour, dm.edge_O, dm.root_O = L.FLAVOUR_DEEPMIND, 0x100000, 0x200000
    _reject(lib, _desc(), dm, b'DeepMindMCTS')
    lp = _desc()
    lp.leaves_per_tree, lp.vl_saved_W = 4, 0x100000
    _reject(lib, lp, _desc(), b'leaves_per_tree')


def test_commit_rejects_bad_move_log(lib):
    from rlzero_b200 import _lib as L
    _reject(lib, _desc(), _desc(), b'move_log', log=None)
    _reject(lib, _desc(), _desc(), b'max_plies', max_plies=35)
    c4 = [_desc(H=6, W=7, k=4, game_type=L.GAME_CONNECT4) for _ in range(2)]
    _reject(lib, c4[0], c4[1], b'max_plies', max_plies=41)
    assert _commit(lib, *[_desc(H=6, W=7, k=4, G=0, game_type=L.GAME_CONNECT4) for _ in range(2)], max_plies=42) == 0


def test_match_rejects_unsupported_players():
    """Seats are checked before any device memory is touched."""
    from rlzero_b200 import _lib as L
    from rlzero_b200.match import BatchedMatch
    from rlzero_b200.mcts import AlphaZeroPlayer, RolloutPlayer
    pure = RolloutPlayer(n_playout=10, seed=1)
    with pytest.raises(ValueError, match='device evaluator'):
        BatchedMatch(AlphaZeroPlayer(make_policy_value_fn(EVAL_KAT), n_playout=10), pure, 4, 6, 4)

    class Fn(object):
        device_evaluator = object()

    with pytest.raises(ValueError, match='leaves_per_wave'):
        BatchedMatch(AlphaZeroPlayer(Fn(), n_playout=10, leaves_per_wave=4), pure, 4, 6, 4)
    with pytest.raises(ValueError, match='is_selfplay=False'):
        BatchedMatch(AlphaZeroPlayer(Fn(), n_playout=10, is_selfplay=True), pure, 4, 6, 4)
    with pytest.raises(ValueError, match='Go'):
        BatchedMatch(pure, pure, 4, 5, 1, game_type=L.GAME_GO)
    with pytest.raises(TypeError):
        BatchedMatch(object(), pure, 4, 6, 4)


# ---------------------------------------------------------------------------------------------- the restatement
@pytest.mark.parametrize('make,n_games', [(lambda: pyoracle.Board(3, 3), 24), (lambda: pyoracle.Board(4, 3), 6),
                                          (lambda: pyoracle.ConnectFourBoard(4, 5, 3), 12)])
def test_oracle_match_equals_single_games(make, n_games):
    """With every game started by player 0, the restated match is ``play_match`` (GameControl.start_play) of the
    same seats, game by game: the IDLE hand-over changes nothing but who searches."""
    az = mo.AZSeat(make_policy_value_fn(EVAL_HASH), 12, 5)
    roll = mo.RolloutSeat(seed=2 ** 64 - 3, n_playout=10)
    seed = 77
    winners, plies, moves = mo.play_match(make, az, roll, n_games, seed=seed, global_offset=2 ** 32 - 2)
    assert len(set(winners)) > 1
    for g in range(n_games):
        for s in (az, roll):
            s.gid, s.seed = 2 ** 32 - 2 + g, seed
        log = []

        class Logged(object):
            def __init__(self, seat):
                self.seat = seat

            def get_action(self, board):
                log.append(self.seat.get_action(board))
                return log[-1]

        assert pyoracle.play_match(make(), Logged(az), Logged(roll)) == winners[g]
        assert log == moves[g] and len(log) == plies[g]


def test_oracle_first_mover():
    roll0, roll1 = mo.RolloutSeat(seed=5, n_playout=6), mo.RolloutSeat(seed=6, n_playout=6)
    _, plies, moves = mo.play_match(lambda: pyoracle.Board(3, 3), roll0, roll1, 4, first=[0, 1, 1, 0])
    for g, f in enumerate([0, 1, 1, 0]):
        b = pyoracle.Board(3, 3)
        b.reset(start_player_idx=f)
        b.step(moves[g][0])
        assert b.states[moves[g][0]] == f


# ---------------------------------------------------------------------------------------------- the draws
def test_root_policy_draw_tie_split():
    visits = [(2, 7), (5, 7)]
    pi = mo.root_pi(visits)
    assert pi == [0.5, 0.5]
    assert mo.draw([2, 5], pi, 0.25) == 2
    assert mo.draw([2, 5], pi, 0.5) == 5            # the cumulative sum must EXCEED u
    assert mo.draw([2, 5], pi, 0.75) == 5


def test_root_policy_draw_one_hot():
    visits = [(0, 1), (3, 50), (4, 2), (8, 0)]
    pi = mo.root_pi(visits)
    assert pi == [0.0, 1.0, 0.0, 0.0]               # exp(1000 * log(1 / 50)) underflows
    for u in (1e-300, 0.5, 1.0 - 2 ** -53):
        assert mo.draw([0, 3, 4, 8], pi, u) == 3


def test_root_policy_draw_beyond_the_rounded_total():
    acts = list(range(3, 13))
    pi = mo.root_pi([(a, 4) for a in acts])
    assert pi == [0.1] * 10
    total = 0.0
    for p in pi:
        total += p
    assert total < 1.0                              # ten times 0.1 rounds to 1 - 2**-53
    assert mo.draw(acts, pi, total) == 12           # not exceeded anywhere: the last action
    assert mo.draw(acts, pi, 0.95) == 12
    assert mo.draw(acts, pi, 0.05) == 3


def test_root_policy_uniform_and_greedy():
    from oracle.philox import philox4, u01_53
    r = philox4(7, 0, 5, 0x5eed, (3 << 10) | 5)
    assert mo.policy_uniform(2 ** 32 + 7, 0, 5, (3 << 10) | 5) == u01_53(r[0], r[1])
    assert 0.0 < mo.policy_uniform(0, 0, 0, 0) < 1.0
    assert mo.greedy_move([(1, 5), (3, 7), (4, 7), (6, 2)]) == 3
    assert mo.greedy_move([(4, 0)]) == 4


def test_oracle_az_seat_is_the_restated_draw():
    """The AZ seat's move is the draw on the visit counts of a fresh restated search."""
    fn = make_policy_value_fn(EVAL_HASH)
    b = pyoracle.Board(4, 3)
    b.reset()
    b.step(5)
    seat = mo.AZSeat(fn, 20, 5)
    seat.gid, seat.seed = 9, 4
    s = pyoracle.Search(fn, 20, 5)
    s.simulate(b)
    visits = sorted((a, ch.n) for a, ch in s.root.children.items())
    assert seat.get_action(b) == mo.root_policy_move(visits, 9, 1, (4 << 10) | 1)
    assert len(b.states) == 1                       # the seat searched copies
    assert np.isclose(sum(mo.root_pi(visits)), 1.0)
