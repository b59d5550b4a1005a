"""``BatchedMatch`` on the device against its restatement (oracle/match_oracle.py), the single-game path and a G = 1
search, with exact equality only."""
import numpy as np
import pytest
import torch

from oracle import match_oracle as mo
from oracle import pyoracle
from oracle.evaluators import EVAL_HASH, make_policy_value_fn

pytestmark = pytest.mark.gpu

ROLL_SEED = 2 ** 64 - 9          # evaluator seed: seed + search counter wraps past 2^64 on the device
FORCE = {'first': 'first', 'last': 'last', 'random': None}


class _ClosedForm(object):
    """A policy_value_fn whose device side is the closed-form evaluator (rz_eval_closed_form)."""

    def __init__(self, eval_id):
        from rlzero_b200.engine import ClosedFormEvaluator
        self.device_evaluator = ClosedFormEvaluator(eval_id)


def _first(kind, G, rs):
    return {'zeros': np.zeros(G, np.int32), 'ones': np.ones(G, np.int32),
            'alternating': np.arange(G, dtype=np.int32) % 2,
            'random': rs.randint(0, 2, size=G).astype(np.int32)}[kind]


def _seats(spec, n_az, n_roll, rule):
    """(device player1, device player2, oracle seat0, oracle seat1) for 'az-<mode>' or 'roll-roll'."""
    from rlzero_b200 import _lib as L
    from rlzero_b200.mcts import AlphaZeroPlayer, RolloutPlayer
    if spec == 'roll-roll':
        return (RolloutPlayer(n_roll, 5, rollout='random', seed=ROLL_SEED),
                RolloutPlayer(n_roll + 3, 5, rollout='random', seed=11),
                mo.RolloutSeat(ROLL_SEED, n_roll, 5), mo.RolloutSeat(11, n_roll + 3, 5))
    mode = spec.split('-')[1]
    dev_rule = L.RULE_PUCT if rule == 'puct' else L.RULE_UCT
    ora_rule = pyoracle.RULE_PUCT if rule == 'puct' else pyoracle.RULE_UCT
    return (AlphaZeroPlayer(_ClosedForm(EVAL_HASH), n_playout=n_az, c_puct=5, rule=dev_rule),
            RolloutPlayer(n_roll, 5, rollout=mode, seed=ROLL_SEED),
            mo.AZSeat(make_policy_value_fn(EVAL_HASH), n_az, 5, ora_rule),
            mo.RolloutSeat(ROLL_SEED, n_roll, 5, force=FORCE[mode]))


# board (kind, H, W, k), seats, rule, first, G, playouts (az, rollout), global_offset
CASES = [
    (('gomoku', 3, 3, 3), 'az-first', 'uct', 'zeros', 256, (10, 8), 0),
    (('gomoku', 3, 3, 3), 'roll-roll', 'uct', 'random', 256, (6, 6), 2 ** 32 - 100),
    (('gomoku', 5, 5, 4), 'az-last', 'uct', 'alternating', 7, (16, 12), 3),
    (('gomoku', 5, 5, 4), 'az-random', 'puct', 'random', 7, (16, 12), 0),
    (('gomoku', 6, 6, 4), 'az-random', 'uct', 'ones', 7, (12, 10), 2 ** 32 - 3),
    (('gomoku', 6, 6, 4), 'az-first', 'uct', 'zeros', 1, (24, 16), 0),
    (('gomoku', 8, 8, 5), 'roll-roll', 'uct', 'alternating', 7, (6, 6), 0),
    (('gomoku', 8, 8, 5), 'az-last', 'puct', 'ones', 1, (12, 8), 5),
    (('c4', 6, 7, 4), 'az-random', 'uct', 'random', 7, (16, 12), 0),
    (('c4', 6, 7, 4), 'roll-roll', 'uct', 'zeros', 1, (10, 10), 1),
]


@pytest.mark.parametrize('board,seats,rule,first,G,playouts,offset', CASES, ids=lambda v: str(v))
def test_match_equals_the_restatement(board, seats, rule, first, G, playouts, offset):
    from rlzero_b200 import _lib as L
    from rlzero_b200.match import BatchedMatch
    kind, H, W, k = board
    p1, p2, o1, o2 = _seats(seats, playouts[0], playouts[1], rule)
    gt = L.GAME_CONNECT4 if kind == 'c4' else L.GAME_GOMOKU
    m = BatchedMatch(p1, p2, G, H, k, board_width=W, game_type=gt, global_offset=offset)
    make = (lambda: pyoracle.ConnectFourBoard(H, W, k)) if kind == 'c4' else (lambda: pyoracle.Board(H, k))
    rs = np.random.RandomState(G + H)
    for seed in (3, 2 ** 40 + 1):                      # two consecutive matches on the same forests
        fst = _first(first, G, rs)
        out = m.play(first=fst, seed=seed)
        winners, plies, moves = mo.play_match(make, o1, o2, G, first=fst, seed=seed, global_offset=offset)
        assert out['plies'].tolist() == plies
        for g in range(G):
            assert out['moves'][g, :plies[g]].tolist() == moves[g], (seed, g)
            assert (out['moves'][g, plies[g]:] == -1).all()
        assert out['winner'].tolist() == winners
        assert dict(out['win_cnt']) == {w: winners.count(w) for w in set(winners)}


def test_match_equals_start_play():
    """Two deterministic rollout players through GameControl.start_play play game 0 of their match."""
    from rlzero_b200.games.gomoku import GameControl, GomokuEnv
    from rlzero_b200.match import BatchedMatch
    from rlzero_b200.mcts import RolloutPlayer
    p1 = RolloutPlayer(40, 5, rollout='first', seed=1)
    p2 = RolloutPlayer(30, 5, rollout='first', seed=2)
    env = GomokuEnv(6, 4)
    game = GameControl(env)
    played = []
    step = env.step

    def logged(a):
        played.append(int(a))
        return step(a)

    env.step = logged
    winner = game.start_play(p1, p2, start_player=0, is_shown=False)
    out = BatchedMatch(p1, p2, 5, 6, 4).play(seed=9)
    assert out['moves'][0, :out['plies'][0]].tolist() == played
    assert int(out['winner'][0]) == winner
    assert (out['moves'] == out['moves'][0]).all()     # deterministic players: every game is the same game


def _record_policies(match):
    """Wrap the AZ seat's root_policy: (counter, visits [G,AS], status [G]) of every ply it moved."""
    from rlzero_b200 import _lib as L
    seat = match.seats[0]
    f = seat.forest
    rec = []
    orig = f.root_policy

    def root_policy(*a, **kw):
        orig(*a, **kw)
        rec.append((kw['seed'], f.visits.cpu().numpy().copy(), f.root_meta[:, L.META_STATUS].cpu().numpy().copy()))

    f.root_policy = root_policy
    return rec


def _g1_visits(evaluator, H, k, n_playout, first, moves, counter):
    from rlzero_b200 import _lib as L
    from rlzero_b200.engine import SearchForest
    f = SearchForest(1, H, k, n_playout=n_playout, c_puct=5, max_carry=0)
    f.reset_games()
    f.root_meta[:, L.META_PLAYER] = int(first)
    for a in moves:
        f.play_moves([a])
    f.search(evaluator, n_playout, seed=counter)
    f.root_policy(1e-3, want_move=False)
    return f.visits.cpu().numpy()[0]


@pytest.mark.parametrize('net,G,checked', [('resnet', 7, 7), ('stock', 7, 7), ('resnet', 160, 4)])
def test_real_net_moves_are_g1_searches(net, G, checked):
    """Every move of the net's seat: the root visits equal a G = 1 search of that position with the same evaluator
    (the forward is batch-invariant), and the logged move is the restated draw on them."""
    from rlzero_b200 import _lib as L
    from rlzero_b200.games.gomoku.alphazero_agent import AlphaZeroAgent
    from rlzero_b200.games.gomoku.policy_value_net import ResNetPolicyValueNet
    from rlzero_b200.match import BatchedMatch
    from rlzero_b200.mcts import AlphaZeroPlayer, RolloutPlayer
    torch.manual_seed(0)
    H, k, n_az = 6, 4, 24
    agent = AlphaZeroAgent(H, net=ResNetPolicyValueNet(H, n_blocks=2)) if net == 'resnet' else AlphaZeroAgent(H)
    agent.policy_value_net.eval()
    m = BatchedMatch(AlphaZeroPlayer(agent.policy_value_fn, n_playout=n_az, c_puct=5),
                     RolloutPlayer(20, 5, seed=4), G, H, k)
    rec = _record_policies(m)
    first = np.random.RandomState(1).randint(0, 2, size=G)
    out = m.play(first=first, seed=21)
    n_checked = 0
    for counter, visits, status in rec:
        ply = counter & 1023
        for g in range(checked):
            if status[g] != L.ACTIVE:
                continue
            hist = out['moves'][g, :ply].tolist()
            want = _g1_visits(agent.native, H, k, n_az, first[g], hist, counter)
            assert visits[g].tolist() == want.tolist(), (g, ply)
            acts = [(a, int(visits[g][a])) for a in range(H * H) if a not in hist]
            assert out['moves'][g, ply] == mo.root_policy_move(acts, g, ply, counter), (g, ply)
            n_checked += 1
    assert n_checked >= checked * 3


def test_idle_and_finished_roots_take_no_visits():
    """After every search, the roots that wait or whose game is over hold no visits and no tree; games of different
    lengths end independently."""
    from rlzero_b200 import _lib as L
    from rlzero_b200.match import BatchedMatch
    from rlzero_b200.mcts import AlphaZeroPlayer, RolloutPlayer
    G = 64
    m = BatchedMatch(AlphaZeroPlayer(_ClosedForm(EVAL_HASH), n_playout=12, c_puct=5),
                     RolloutPlayer(10, 5, seed=3), G, 5, 4)
    checks = []
    for seat in m.seats:
        f = seat.forest
        orig = f.search

        def search(*a, f=f, orig=orig, **kw):
            orig(*a, **kw)
            st = f.root_meta[:, L.META_STATUS].cpu().numpy()
            n = f.root_N.cpu().numpy()
            nn = f.n_nodes.cpu().numpy()
            active = st == L.ACTIVE
            assert (n[~active] == 0).all() and (nn[~active] == 0).all()
            assert (n[active] == kw.get('n_playout', a[1])).all()
            checks.append(int((~active).sum()))

        f.search = search
    first = np.arange(G) % 2
    out = m.play(first=first, seed=5)
    assert len(set(out['plies'].tolist())) > 2
    assert min(checks) >= G // 2 and max(checks) > G // 2     # waiting games, then finished ones too
    for g in range(G):
        p = int(out['plies'][g])
        assert (out['moves'][g, :p] >= 0).all() and (out['moves'][g, p:] == -1).all()
    for seat in m.seats:
        meta = seat.forest.root_meta.cpu().numpy()
        assert np.isin(meta[:, L.META_STATUS], (L.ENDED_WIN, L.ENDED_TIE)).all()
        assert meta[:, L.META_FAULT].tolist() == [0] * G


def test_pipeline_batched_evaluation(monkeypatch):
    from rlzero_b200 import match as match_mod
    from rlzero_b200.train_pipeline import TrainPipeline
    seen = []
    orig = match_mod.BatchedMatch.play

    def play(self, *a, **kw):
        out = orig(self, *a, **kw)
        seen.append(out)
        return out

    monkeypatch.setattr(match_mod.BatchedMatch, 'play', play)
    np.random.seed(0)
    pipe = TrainPipeline(board_size=6, n_in_row=4, n_playout=16, pure_mcts_playout_num=20, batched_evaluation=True)
    ratio = pipe.policy_evaluate(n_games=12)
    assert len(seen) == 1
    wc = seen[0]['win_cnt']
    assert sum(wc.values()) == 12
    assert ratio == 1.0 * (wc[1] + 0.5 * wc[-1]) / 12
    assert (seen[0]['plies'] > 0).all()
