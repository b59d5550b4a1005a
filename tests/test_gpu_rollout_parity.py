"""The device's random playouts and child-order keys against their restatement (oracle/rollout_oracle.py on
oracle/philox.py), bit for bit:

* ``rz_eval_rollout`` (RolloutMCTS / RolloutPlayer) and ``rz_eval_rollout_dm`` (DeepMindMCTS's
  RandomRolloutEvaluator) on single positions: priors and values;
* whole searches -- ``RolloutMCTS(rollout='random')`` against the restated ``RolloutSearch``, ``DeepMindMCTS`` with
  ``RandomRolloutEvaluator`` (and the random child shuffle) against the restated ``DMSearch`` -- over consecutive
  searches, in the captured-graph, unfused and eager wave loops;
* one evaluator shared by two forests.

Every comparison is exact: the draws are integer arithmetic and the statistics are the fp64 sums the tree
restatements already reproduce."""
import copy

import numpy as np
import pytest
import torch

from oracle import dm_oracle, go_oracle, pyoracle, rollout_oracle as ro

pytestmark = pytest.mark.gpu

BIG_SEED = 2 ** 64 - 5           # evaluator seed: seed + search counter wraps past 2^64 on the device
SEED_DEV = 9


class GoDM(go_oracle.GoSearchBoard):
    """GoSearchBoard with the methods DMSearch calls (returns [1, -1] iff black wins, go_env.py:142-143)."""

    def legal_actions(self, player=None):
        return self.leagel_actions()

    def is_terminal(self):
        return self.game_end_winner()[0]

    def returns(self):
        end, w = self.game_end_winner()
        return [0, 0] if not end else ([1, -1] if w == 0 else [-1, 1])


def _line_board(kind, H, W, k, returns_mode=0):
    if kind == 'c4':
        return pyoracle.ConnectFourBoard(H, W, k)
    return pyoracle.DMBoard(H, k, zero_sum=bool(returns_mode))


def _random_positions(rs, make, G, max_moves):
    """G non-terminal positions reached by random legal moves: (boards, move lists)."""
    boards, lists = [], []
    for _ in range(G):
        while True:
            b = make()
            b.reset()
            mv, ok = [], True
            for _ in range(rs.randint(0, max_moves + 1)):
                legal = list(b.leagel_actions())
                a = int(legal[rs.randint(len(legal))])
                b.step(a)
                mv.append(a)
                if b.game_end_winner()[0]:
                    ok = False
                    break
            if ok:
                break
        boards.append(b)
        lists.append(mv)
    return boards, lists


def _forest(G, kind, H, W, k, **kw):
    from rlzero_b200 import _lib as L
    from rlzero_b200.engine import SearchForest
    gt = {'gomoku': L.GAME_GOMOKU, 'c4': L.GAME_CONNECT4, 'go': L.GAME_GO}[kind]
    return SearchForest(G, H, k, n_playout=1, board_width=W, game_type=gt, **kw)


# ---------------------------------------------------------------------------------- 1. evaluator level
# kind, H, W, k, G, max random moves, games compared at n_rollouts = 33
BOARDS = [
    ('gomoku', 3, 3, 3, 2048, 7, 512),
    ('gomoku', 6, 6, 4, 512, 24, 96),
    ('gomoku', 9, 9, 5, 96, 50, 24),
    ('gomoku', 15, 15, 5, 24, 120, 4),
    ('c4', 6, 7, 4, 256, 30, 64),
    ('go', 5, 5, 1, 64, 16, 64),
    ('go', 9, 9, 1, 12, 40, 6),
    ('go', 19, 19, 1, 3, 60, 0),
]


@pytest.mark.parametrize('kind,H,W,k,G,max_moves,n33', BOARDS, ids=lambda v: str(v))
@pytest.mark.parametrize('returns_mode', [0, 1])
def test_evaluators_match_the_restatement(kind, H, W, k, G, max_moves, n33, returns_mode):
    from rlzero_b200.engine import RolloutEvaluator
    from rlzero_b200.mcts import RandomRolloutEvaluator
    rs = np.random.RandomState(H * 100 + W + returns_mode)
    if kind == 'go':
        boards, lists = _random_positions(rs, lambda: GoDM(H, 0.5), G, max_moves)
        f = _forest(G, kind, H, W, k, komi=0.5, global_offset=2 ** 32 - 3, returns_mode=returns_mode)
    else:
        boards, lists = _random_positions(rs, lambda: _line_board(kind, H, W, k, returns_mode), G, max_moves)
        f = _forest(G, kind, H, W, k, global_offset=2 ** 32 - 3, returns_mode=returns_mode)
    f.set_positions(lists)
    f.select()
    assert (f.depth.cpu().numpy() == 0).all()
    visits = rs.randint(0, 5000, size=G).astype(np.int32)
    f.root_N.copy_(torch.from_numpy(visits))
    f.seed_dev.fill_(SEED_DEV)
    seed = BIG_SEED + SEED_DEV
    gids = [(2 ** 32 - 3 + g) & 0xffffffff for g in range(G)]           # global_offset + g wraps to 0, 1, ...

    # priors: float32 1/n_legal over the legal slots, both evaluators
    if kind == 'go':
        legal = [np.asarray(b.pos.all_legal_moves(), dtype=bool) for b in boards]
    else:
        legal = []
        for b in boards:
            m = np.zeros(f.A, dtype=bool)
            m[list(b.leagel_actions())] = True
            legal.append(m)
    want_p = np.zeros((G, f.AS), dtype=np.float32)
    for g in range(G):
        want_p[g, :f.A][legal[g]] = ro.uniform_prior(int(legal[g].sum()))

    if kind != 'go':
        pos = [ro.LinePos.of(b) for b in boards]
        for n_limit in (0, 1, 7, 1000):
            if returns_mode:
                break                      # rz_eval_rollout has no returns convention: once per board
            f.prior.zero_()
            RolloutEvaluator(n_limit=n_limit, seed=BIG_SEED)(f)
            got = f.value.cpu().numpy()
            assert np.array_equal(f.prior.cpu().numpy(), want_p)
            want = np.array([ro.az_rollout(pos[g], gids[g], int(visits[g]), pos[g].stones, seed, n_limit)
                             for g in range(G)], dtype=np.float32)
            assert np.array_equal(got, want), (n_limit, np.nonzero(got != want)[0][:8])

    for n_rollouts, n_limit, n_cmp in ((1, 1000, G), (8, 1000, max(n33, min(G, 16))), (33, 1000, n33),
                                       (8, 0, G), (8, 1, G), (8, 5, min(G, 64))):
        if n_cmp == 0:
            continue
        ev = RandomRolloutEvaluator(n_rollouts=n_rollouts, n_limit=n_limit, seed=BIG_SEED)
        f.prior.zero_()
        ev(f)
        assert np.array_equal(f.prior.cpu().numpy(), want_p)
        got = ev.value64.cpu().numpy()
        for g in range(n_cmp):
            if kind == 'go':
                want = ro.go_dm_rollout(boards[g].pos, gids[g], int(visits[g]), seed, n_limit, n_rollouts)[0]
            else:
                want = ro.dm_rollout(pos[g], gids[g], int(visits[g]), seed, n_limit, n_rollouts,
                                     1 if kind == 'c4' else 0, returns_mode)
            assert got[g].tolist() == want, (n_rollouts, n_limit, g)


@pytest.mark.parametrize('returns_mode', [0, 1])
def test_evaluators_at_the_forced_end(returns_mode):
    """Every position has exactly ``F`` empty squares, so ``n_limit = F`` is the last move of every playout: a win by
    that move is a tie for rz_eval_rollout (status tested before each move) and counts for rz_eval_rollout_dm
    (tested once more at i == n_limit)."""
    from rlzero_b200.engine import RolloutEvaluator
    from rlzero_b200.mcts import RandomRolloutEvaluator
    rs = np.random.RandomState(4 + returns_mode)
    G, F = 1500, 3
    boards, lists = [], []
    while len(boards) < G:
        b = pyoracle.DMBoard(3, 3, zero_sum=bool(returns_mode))
        b.reset()
        mv = [int(a) for a in rs.permutation(9)[:9 - F]]
        ok = True
        for a in mv:
            b.step(a)
            if b.game_end_winner()[0]:
                ok = False
                break
        if ok:
            boards.append(b)
            lists.append(mv)
    f = _forest(G, 'gomoku', 3, 3, 3, global_offset=77, returns_mode=returns_mode)
    f.set_positions(lists)
    f.select()
    f.seed_dev.fill_(SEED_DEV)
    pos = [ro.LinePos.of(b) for b in boards]
    at_edge = None
    for n_limit in (F - 1, F, F + 1):
        RolloutEvaluator(n_limit=n_limit, seed=3)(f)
        want = np.array([ro.az_rollout(pos[g], 77 + g, 0, 9 - F, 3 + SEED_DEV, n_limit) for g in range(G)],
                        dtype=np.float32)
        assert np.array_equal(f.value.cpu().numpy(), want)
        ev = RandomRolloutEvaluator(n_rollouts=8, n_limit=n_limit, seed=3)
        ev(f)
        got = ev.value64.cpu().numpy()
        for g in range(G):
            assert got[g].tolist() == ro.dm_rollout(pos[g], 77 + g, 0, 3 + SEED_DEV, n_limit, 8, 0, returns_mode)
        if n_limit == F:
            # games whose AlphaZero playout is a tie while some DM playout of the same length is decided
            at_edge = int(((want == 0) & (np.abs(got).sum(1) > 0)).sum())
    assert at_edge > 20


# ---------------------------------------------------------------------------------- 2. RolloutMCTS
@pytest.mark.parametrize('size,k,n_playout,seed', [(3, 3, 40, 5), (6, 4, 120, 2 ** 40 + 1), (9, 5, 64, 0)])
def test_rollout_mcts_matches_the_restated_search(size, k, n_playout, seed):
    """RolloutMCTS(rollout='random', seed=s) over consecutive moves (update_with_move(-1) after each, as
    RolloutPlayer does): the search counter moves the stream; root visits, W, root N / W and the move are exact."""
    from rlzero_b200.games.gomoku import GomokuEnv
    from rlzero_b200.mcts import RolloutMCTS
    env = GomokuEnv(size, k)
    env.reset()
    b = pyoracle.Board(size, k)
    b.reset()
    for a in ([4] if size == 3 else [size * size // 2, 0]):
        env.step(a)
        b.step(a)
    mcts = RolloutMCTS(n_playout=n_playout, c_puct=5, rollout='random', seed=seed)
    for search in range(1, 4):
        move = mcts.simulate(env)
        visits, w, has, root_n, root_w = mcts._forest.root_stats()
        ev = ro.AZRollout(0, seed + search)
        ev.root_stones = len(b.states)
        s = pyoracle.RolloutSearch(n_playout, 5, rollout=ev)
        want_move = s.simulate(copy.deepcopy(b))
        A = size * size
        assert visits[0].tolist() == s.root_visits(A).tolist()
        want_w = [0.0] * A
        for a, ch in s.root.children.items():
            want_w[a] = float(ch.w)
        assert w[0].tolist() == want_w
        assert int(root_n[0]) == s.root.n and float(root_w[0]) == s.root.w
        assert move == want_move
        assert any(ch.w != 0 for ch in s.root.children.values())      # the playouts decide something
        env.step(move)
        b.step(move)
        mcts.update_with_move(-1)
        if b.game_end_winner()[0]:
            break


# ---------------------------------------------------------------------------------- 3. DeepMindMCTS
def _dm_case(game, rs):
    """(device env, oracle board) of a random non-terminal position."""
    if game == 'go':
        from rlzero_b200.games.go import GoEnv
        env = GoEnv(board_size=5, komi=0.5)
        b = GoDM(5, 0.5)
        n_moves = 6
    else:
        from rlzero_b200.games.gomoku import GomokuEnv
        env = GomokuEnv(4, 3)
        b = pyoracle.DMBoard(4, 3, zero_sum=True)
        n_moves = 3
    env.reset()
    b.reset()
    for _ in range(n_moves):
        legal = list(b.legal_actions())
        a = int(legal[rs.randint(len(legal))])
        env.step(a)
        b.step(a)
        assert not b.is_terminal()
    return env, b


def _dm_run(game, method, solve, shuffle, how, monkeypatch):
    """Two consecutive searches of one DeepMindMCTS bot (a move played in between) with a fresh
    RandomRolloutEvaluator; ``how`` picks the wave loop.  Returns the comparable digests and the roots' meta."""
    from rlzero_b200 import _lib as L
    from rlzero_b200.mcts import DeepMindMCTS, RandomRolloutEvaluator
    monkeypatch.setenv('RZ_FUSE_SELECT', '0' if how == 'unfused' else '1')
    rs = np.random.RandomState(17)
    env, b = _dm_case(game, rs)
    ev = RandomRolloutEvaluator(n_rollouts=4, n_limit=1000, seed=BIG_SEED)
    if how == 'eager':
        ev.graph_capturable = False            # run_waves then launches every wave from the host
    rmode = L.RETURNS_ZERO_SUM
    bot = DeepMindMCTS(env, uct_c=2, max_simulations=48, evaluator=ev, child_selection_method=method, solve=solve,
                       returns_mode=rmode, child_shuffle=shuffle, seed=0)
    out = []
    for search in range(2):
        root = bot.mcts_search(env)
        meta = bot._forest.root_meta[0].cpu().numpy()
        best, _ = bot._forest.best_child()
        out.append(dict(root_n=root.explore_count, root_w=root.total_reward, root_outcome=root.outcome,
                        children=[(c.action, c.explore_count, c.total_reward, c.outcome) for c in root.children],
                        best=int(best[0]), episode=int(meta[L.META_EPISODE]), ply=int(meta[L.META_PLY])))
        a = int(best[0])
        env.step(a)
        b.step(a)
        if b.is_terminal():
            break
    return out


def _dm_oracle(game, method, solve, shuffle, device_runs):
    rs = np.random.RandomState(17)
    _, b = _dm_case(game, rs)
    out = []
    for search, dev in enumerate(device_runs):
        counter = search + 1                   # DeepMindMCTS's search counter (seed=0, bumped per search)
        ev = ro.DMRollout(0, BIG_SEED + counter, n_limit=1000, n_rollouts=4, returns_mode=ro.RETURNS_ZERO_SUM)
        sh = ro.ShuffleRank(0, dev['episode'], dev['ply'], counter) if shuffle else None
        s = dm_oracle.DMSearch(ev, 48, 2, method, solve=solve, shuffle_fn=sh)
        ev.search = s
        if sh is not None:
            sh.search = s
        root = s.search(copy.deepcopy(b))
        kids = [(c.action, c.n, c.w, c.outcome) for c in root.children]
        if not shuffle:
            kids.sort()
        best = root.best_child().action
        out.append(dict(root_n=root.n, root_w=root.w, root_outcome=root.outcome, children=kids, best=best,
                        episode=dev['episode'], ply=dev['ply']))
        b.step(best)
    return out


@pytest.mark.parametrize('game', ['gomoku', 'go'])
@pytest.mark.parametrize('method', ['uct', 'puct'])
@pytest.mark.parametrize('solve', [False, True])
@pytest.mark.parametrize('shuffle', [False, True])
def test_deepmind_mcts_with_random_rollouts_matches_the_restatement(game, method, solve, shuffle, monkeypatch):
    """DeepMindMCTS(evaluator=RandomRolloutEvaluator()) -- the reference's own Go configuration -- over two
    consecutive searches of one bot: children (action, N, W, outcome), root N / W / outcome and best_child equal
    the restated search, in the captured-graph wave loop, with the backup unfused and with eager waves."""
    runs = {how: _dm_run(game, method, solve, shuffle, how, monkeypatch) for how in ('graph', 'unfused', 'eager')}
    want = _dm_oracle(game, method, solve, shuffle, runs['graph'])
    for how, got in runs.items():
        assert len(got) == len(want) == 2, how
        for search, (g, w) in enumerate(zip(got, want)):
            assert g == w, (how, search)
    # the rollouts reach the statistics: some child holds a value sum no terminal outcome explains
    assert any(c[2] != 0 and c[3] is None for r in want for c in r['children'])


# ---------------------------------------------------------------------------------- 4. one evaluator, two forests
def test_one_evaluator_shared_by_two_forests():
    """A RandomRolloutEvaluator re-allocates its returns buffer for a forest of another size: interleaved searches of
    two forests through one evaluator must equal the same searches each with an evaluator of its own."""
    from rlzero_b200 import _lib as L
    from rlzero_b200.engine import SearchForest
    from rlzero_b200.mcts import RandomRolloutEvaluator
    rs = np.random.RandomState(8)
    sizes = (5, 37)
    lists = {G: _random_positions(rs, lambda: pyoracle.DMBoard(4, 3, zero_sum=True), G, 5)[1] for G in sizes}

    def forest(G):
        f = SearchForest(G, 4, 3, n_playout=24, c_puct=2.0, rule=L.RULE_UCT, flavour=L.FLAVOUR_DEEPMIND, solve=True,
                         returns_mode=L.RETURNS_ZERO_SUM, max_carry=0)
        f.set_positions(lists[G])
        return f

    def stats(f):
        """Every tree's used edge blocks, root N / W.  The pool beyond n_nodes, and W of an edge never visited, are
        uninitialised."""
        nn = f.n_nodes.cpu().numpy()
        N = f.edge_N.cpu().numpy().reshape(f.G, -1)
        W = np.where(N > 0, f.edge_W.cpu().numpy().reshape(f.G, -1), 0.0)
        return ([N[g, :nn[g] * f.AS].tolist() for g in range(f.G)], [W[g, :nn[g] * f.AS].tolist() for g in range(f.G)],
                f.root_N.cpu().numpy().tolist(), f.root_W.cpu().numpy().tolist())

    shared = RandomRolloutEvaluator(n_rollouts=3, seed=21)
    own = {G: RandomRolloutEvaluator(n_rollouts=3, seed=21) for G in sizes}
    fs = {G: forest(G) for G in sizes}
    fo = {G: forest(G) for G in sizes}
    for search in range(1, 4):
        for G in sizes:
            for f, ev in ((fs[G], shared), (fo[G], own[G])):
                f.reset_trees()
                f.run_waves(24, ev, seed=search)
                f.raise_faults()
            a, b = stats(fs[G]), stats(fo[G])
            assert a == b, (search, G)
            assert any(w != 0 for w in a[3])
