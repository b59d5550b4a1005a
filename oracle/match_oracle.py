"""TEST INFRASTRUCTURE ONLY -- ``rlzero_b200.match.BatchedMatch`` restated game by game.

Each game is played with ``pyoracle`` searches per seat, keyed the way the device keys them at ply p of a match
started with ``seed`` (the search counter ``(seed << 10) | p``, see ``BatchedMatch``):

* an AlphaZero seat runs ``pyoracle.Search`` (a fresh tree, no noise) and draws its move with the restated
  ``rz_tree_root_policy`` draw (``root_policy_move``, rz_tree.cu:613-690);
* a rollout seat runs ``pyoracle.RolloutSearch`` whose leaf values are the device's playouts
  (``rollout_oracle.AZRollout`` with seed = the evaluator's seed + the counter and ``root_stones`` of the position)
  and plays the first most-visited child (``greedy_move``);
* the seats hand the position over as ``rz_match_commit`` does: the mover's root turns IDLE, the other ACTIVE.
"""
import copy
import math

from . import pyoracle
from . import rollout_oracle as ro
from .philox import MASK32, philox4, u01_53

ACTIVE, ENDED_WIN, ENDED_TIE, IDLE = range(4)


def root_pi(visits, temperature=1e-3):
    """``pi = softmax(log(N + 1e-10) / T)`` over the root's children, ``visits`` = [(action, N)] in ascending action
    order, as the kernel forms it: ``(1 / T) * log(N + 1e-10)``, the maximum subtracted, ``exp``, divided by the
    sum.  Agrees with the device to the last bits of ``log`` / ``exp`` and of the sum's order."""
    x = [(1.0 / temperature) * math.log(n + 1e-10) for _, n in visits]
    mx = max(x)
    e = [math.exp(v - mx) for v in x]
    s = sum(e)
    return [v / s for v in e]


def policy_uniform(gid, episode, stones, seed):
    """The uniform of the root-policy draw: ``u01_53(philox4(gid, episode, stones, 0x5eed, seed))``."""
    r = philox4(gid & MASK32, episode, stones, 0x5eed, seed)
    return u01_53(r[0], r[1])


def draw(actions, pi, u):
    """The first action whose cumulative ``pi`` (ascending action order) exceeds ``u``; the last one when ``u`` lies
    beyond the rounded total."""
    c = 0.0
    for a, p in zip(actions, pi):
        c += p
        if c > u:
            return a
    return actions[-1]


def root_policy_move(visits, gid, stones, seed, episode=0, temperature=1e-3):
    acts = [a for a, _ in visits]
    return draw(acts, root_pi(visits, temperature), policy_uniform(gid, episode, stones, seed))


def greedy_move(visits):
    """The first most-visited child (``max`` over ascending actions keeps the first maximum)."""
    return max(visits, key=lambda an: an[1])[0]


def _visits(root):
    return sorted((a, ch.n) for a, ch in root.children.items())


class AZSeat(object):
    """``AlphaZeroPlayer(policy_value_fn, n_playout, c_puct, rule)`` as a match seat."""

    def __init__(self, policy_value_fn, n_playout, c_puct=5, rule=pyoracle.RULE_UCT):
        self.fn, self.n_playout, self.c_puct, self.rule = policy_value_fn, n_playout, c_puct, rule
        self.gid, self.seed = 0, 0          # set per game by play_game

    def get_action(self, board):
        s = pyoracle.Search(self.fn, self.n_playout, self.c_puct, rule=self.rule)
        s.simulate(board)                   # copies the board per playout
        ply = len(board.states)
        return root_policy_move(_visits(s.root), self.gid, ply, (self.seed << 10) | ply)


class RolloutSeat(object):
    """``RolloutPlayer`` with ``RolloutEvaluator(n_limit, seed, mode)`` as a match seat (``force`` = None / 'first' /
    'last' for the modes 'random' / 'first' / 'last')."""

    def __init__(self, seed, n_playout, c_puct=5, n_limit=1000, force=None):
        self.ev_seed, self.n_playout, self.c_puct, self.n_limit, self.force = seed, n_playout, c_puct, n_limit, force
        self.gid, self.seed = 0, 0

    def get_action(self, board):
        ply = len(board.states)
        ev = ro.AZRollout(self.gid, self.ev_seed + ((self.seed << 10) | ply), self.n_limit, self.force)
        ev.root_stones = ply
        s = pyoracle.RolloutSearch(self.n_playout, self.c_puct, self.n_limit, rollout=ev)
        s.simulate(copy.deepcopy(board))
        return greedy_move(_visits(s.root))


def play_game(board, seats, first, gid, seed):
    """One game of the match: (winner, moves).  ``board`` is a fresh ``pyoracle.Board`` / ``ConnectFourBoard``,
    ``seats[s]`` plays env id s, ``first`` moves first.  Line games only, so the ply is the stone count."""
    for s in seats:
        s.gid, s.seed = gid, seed
    board.reset(start_player_idx=first)
    status = [ACTIVE if s == first else IDLE for s in (0, 1)]
    moves = []
    while True:
        mover = status.index(ACTIVE)
        m = seats[mover].get_action(board)
        board.step(m)
        moves.append(m)
        end, winner = board.game_end_winner()
        if end:
            return winner, moves
        status[mover], status[mover ^ 1] = IDLE, ACTIVE


def play_match(make_board, seat0, seat1, n_games, first=None, seed=0, global_offset=0):
    """``BatchedMatch.play`` restated: (winner [G], plies [G], moves [G] lists)."""
    first = [0] * n_games if first is None else [int(f) for f in first]
    winners, plies, moves = [], [], []
    for g in range(n_games):
        w, mv = play_game(make_board(), (seat0, seat1), first[g], global_offset + g, seed)
        winners.append(w)
        plies.append(len(mv))
        moves.append(mv)
    return winners, plies, moves
