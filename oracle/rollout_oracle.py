"""TEST INFRASTRUCTURE ONLY -- the device's random playouts and child-order keys, restated draw for draw.

Three pieces of device code decide with Philox-4x32-10 (``oracle/philox.py``) what a search backs up:

* ``rz_eval_rollout_kernel`` mode 0 (``rlzero_b200/csrc/rz_game.cu:247-311``): the leaf value of
  ``RolloutMCTS`` -- ``az_rollout``;
* ``rz_eval_rollout_dm_kernel`` (``rz_game.cu:319-390``): ``RandomRolloutEvaluator`` of ``DeepMindMCTS`` --
  ``dm_rollout`` (line games here, Go in ``oracle/c/rz_go_oracle.c`` through ``go_dm_rollout``);
* the child-order key of ``shuffle_mode == 1`` (``rz_tree.cu:384-395``) -- ``shuffle_rank``.

The semantics are the kernels', not the reference's (which draws from numpy's global stream and agrees
with the device in distribution only).  Positions are ``LinePos`` (Gomoku / Connect Four) built from the
oracle boards of ``oracle/pyoracle.py``.  ``RolloutSearch`` / ``DMSearch`` plug them in through
``AZRollout`` / ``DMRollout`` / ``ShuffleRank`` below.
"""
import numpy as np

from .philox import MASK32, philox4, pick

ACTIVE, ENDED_WIN, ENDED_TIE = 0, 1, 2
RETURNS_REFERENCE, RETURNS_ZERO_SUM = 0, 1
U64 = (1 << 64) - 1


class LinePos(object):
    """A k-in-a-row position as the device board holds it (rz_board.cuh): ``cells[r*W + c]`` is -1 / 0 / 1,
    ``player`` to move, ``stones`` moves played.  Connect Four (``gravity``) counts rows from the bottom,
    as ``pyoracle.ConnectFourBoard`` does, and its actions are the columns."""

    __slots__ = ('H', 'W', 'k', 'gravity', 'cells', 'player', 'stones', 'won')

    def __init__(self, H, W, k, gravity, cells, player, stones):
        self.H, self.W, self.k, self.gravity = H, W, k, bool(gravity)
        self.cells = list(cells)
        self.player = player
        self.stones = stones
        self.won = self._scan()          # winner of the whole board (-1 none), rz_board_status's line test

    @classmethod
    def of(cls, board):
        """From ``pyoracle.Board`` / ``DMBoard`` / ``ConnectFourBoard``."""
        W = getattr(board, 'board_width', board.board_size)
        cells = [-1] * (board.board_size * W)
        for m, p in board.states.items():
            cells[m] = p
        return cls(board.board_size, W, board.n_in_row, hasattr(board, 'heights'), cells,
                   board.current_player(), len(board.states))

    def copy(self):
        c = LinePos.__new__(LinePos)
        c.H, c.W, c.k, c.gravity = self.H, self.W, self.k, self.gravity
        c.cells, c.player, c.stones, c.won = list(self.cells), self.player, self.stones, self.won
        return c

    def _line_through(self, m):
        p = self.cells[m]
        r0, c0 = divmod(m, self.W)
        for dr, dc in ((0, 1), (1, 0), (1, 1), (1, -1)):
            n = 1
            for s in (1, -1):
                r, c = r0 + s * dr, c0 + s * dc
                while 0 <= r < self.H and 0 <= c < self.W and self.cells[r * self.W + c] == p:
                    n += 1
                    r += s * dr
                    c += s * dc
            if n >= self.k:
                return True
        return False

    def _scan(self):
        owners = [p for p in (0, 1) if any(self.cells[m] == p and self._line_through(m)
                                           for m in range(self.H * self.W))]
        return -1 if not owners else owners[0]          # rz_board_status: w0 ? 0 : 1

    def status(self):
        """(status, winner) of rz_board_status (rz_board.cuh:80-92), early-out at 2k - 1 stones included."""
        if self.stones >= 2 * self.k - 1 and self.won >= 0:
            return ENDED_WIN, self.won
        if self.stones >= self.H * self.W:
            return ENDED_TIE, -1
        return ACTIVE, -1

    def candidates(self):
        """move_candidates (rz_board.cuh:153-160) in the order the kernels count them: the empty squares in
        row-major order, or (gravity) the columns whose top square is empty, ascending."""
        if self.gravity:
            top = (self.H - 1) * self.W
            return [c for c in range(self.W) if self.cells[top + c] < 0]
        return [m for m, v in enumerate(self.cells) if v < 0]

    def play(self, a):
        """rz_board_play; the line test looks at the new stone only (the position before had no line)."""
        m = a
        if self.gravity:
            while self.cells[m] >= 0:
                m += self.W
        self.cells[m] = self.player
        if self.won < 0 and self._line_through(m):
            self.won = self.player
        self.player ^= 1
        self.stones += 1


def uniform_prior(n_legal):
    """float32 1/n_legal of the evaluators (``__fdiv_rn(1.0f, (float)n)``), 0 without a legal move."""
    return np.float32(1.0) / np.float32(n_legal) if n_legal > 0 else np.float32(0.0)


def game_returns(game_type, mode, status, winner):
    """rz_game_returns (rz_common.cuh:206-212)."""
    if status != ENDED_WIN:
        return 0, 0
    if game_type == 2:                                   # Go
        r0 = 1 if winner == 0 else -1
        return r0, -r0
    if mode == RETURNS_REFERENCE:
        return (1, -1) if winner == 1 else (0, 0)
    r0 = 1 if winner == 0 else -1
    return r0, -r0


def az_rollout(pos, g, visit, root_stones, seed, n_limit, force=None):
    """rz_eval_rollout_kernel mode 0 (rz_game.cu:269-310) from ``pos`` (not modified): the float32 value.

    ``g`` = global_offset + tree, ``visit`` = root_N at evaluation time, ``root_stones`` = the root's
    RZ_META_STONES, ``seed`` = the evaluator's seed plus the search counter (rz_tree_desc.seed_dev).
    ``force`` = 'first' / 'last' replaces the draw by r = 0 / n - 1 (the kernel's modes 1 / 2)."""
    b = pos.copy()
    c3 = (0x7011 + (root_stones << 16)) & MASK32
    seed &= U64
    winner = -1
    for i in range(n_limit):
        st, winner = b.status()          # tested before each move: a win by the n_limit-th move is a tie
        if st != ACTIVE:
            break
        cand = b.candidates()
        if force == 'first':
            r = 0
        elif force == 'last':
            r = len(cand) - 1
        else:
            r = pick(philox4(g, visit, i, c3, seed)[0], len(cand))
        b.play(cand[r])
    if winner == -1:
        return np.float32(0.0)
    return np.float32(1.0 if winner == b.player else -1.0)


def dm_rollout(pos, g, visit, seed, n_limit, n_rollouts, game_type, returns_mode):
    """rz_eval_rollout_dm_kernel for a line game (rz_game.cu:342-389): the float64 returns vector."""
    seed &= U64
    s0 = s1 = 0
    for r in range(n_rollouts):
        b = pos.copy()
        st, winner = ACTIVE, -1
        for i in range(n_limit + 1):
            st, winner = b.status()
            if st != ACTIVE or i == n_limit:
                break
            cand = b.candidates()
            b.play(cand[pick(philox4(g, visit, (r << 16) | i, 0xd311, seed)[0], len(cand))])
        r0, r1 = game_returns(game_type, returns_mode, st, winner)
        s0 += r0
        s1 += r1
    return [s0 / n_rollouts, s1 / n_rollouts]          # int / int: the correctly rounded float64 quotient


def go_dm_rollout(pos, g, visit, seed, n_limit, n_rollouts, max_moves=0):
    """rz_eval_rollout_dm_kernel<rz_go_game> for a ``go_oracle.Position``: (returns [2] float64, legal
    mask [N*N + 1] int8).  The playouts run in ``oracle/c/rz_go_oracle.c`` (``rzo_go_rollout_dm``)."""
    import ctypes as C
    from . import build_oracle
    lib = build_oracle.load()
    n = pos.N
    cells = np.ascontiguousarray(pos.board, dtype=np.int8).reshape(-1)
    out = np.zeros(2, dtype=np.float64)
    legal = np.zeros(n * n + 1, dtype=np.int8)
    rec = pos.recent
    pass1 = int(len(rec) >= 1 and rec[-1][1] is None)
    pass2 = int(len(rec) >= 2 and rec[-2][1] is None)
    rc = lib.rzo_go_rollout_dm(n, float(pos.komi), int(max_moves), cells.ctypes.data_as(C.POINTER(C.c_int8)),
                               -1 if pos.ko is None else pos.ko[0] * n + pos.ko[1], int(pos.to_play), int(pos.n),
                               pass1, pass2, int(n_rollouts), int(n_limit), int(g) & MASK32, int(visit) & MASK32,
                               int(seed) & U64, out.ctypes.data_as(C.POINTER(C.c_double)),
                               legal.ctypes.data_as(C.POINTER(C.c_int8)))
    if rc != 0:
        raise RuntimeError('rzo_go_rollout_dm: %d' % rc)
    return [float(out[0]), float(out[1])], legal


def shuffle_rank(g, episode, ply, node, action, seed):
    """Child-order key of shuffle_mode 1 (rz_tree.cu:384-395): child ``action`` of the node the device
    allocated as ``node`` (its expansion index in the tree), under a root with RZ_META_EPISODE / RZ_META_PLY
    ``episode`` / ``ply``.  ``seed`` = the expansion's seed (the search counter in a DeepMindMCTS search)."""
    w = philox4(g, (episode & 0xfffff) | (action << 20), (ply << 16) | node, 0xffff,
                (seed & U64) ^ 0x517cc1b727220a95)
    return w[0] >> 1


# ---- adapters for the oracle searches --------------------------------------------------------------------
class AZRollout(object):
    """``pyoracle.RolloutSearch(rollout=AZRollout(...))``: the device's leaf value for tree ``g``."""

    def __init__(self, g, seed, n_limit=1000, force=None):
        self.g, self.seed, self.n_limit, self.force = g, seed, n_limit, force
        self.root_stones = 0

    def __call__(self, board, root_n):
        return az_rollout(LinePos.of(board), self.g, root_n, self.root_stones, self.seed, self.n_limit, self.force)


class DMRollout(object):
    """Evaluator (deepmind_mcts.py:14-28) for ``dm_oracle.DMSearch``: the device's ``RandomRolloutEvaluator``.
    It reads the root's visit count from the search it is attached to (``search.root``)."""

    def __init__(self, g, seed, n_limit=1000, n_rollouts=20, returns_mode=RETURNS_REFERENCE):
        self.g, self.seed, self.n_limit, self.n_rollouts = g, seed, n_limit, n_rollouts
        self.returns_mode = returns_mode
        self.search = None

    def evaluate(self, env):
        visit = self.search.root.n
        if hasattr(env, 'pos'):                                   # go_oracle.GoSearchBoard
            return go_dm_rollout(env.pos, self.g, visit, self.seed, self.n_limit, self.n_rollouts,
                                 env.max_moves)[0]
        game_type = 1 if hasattr(env, 'heights') else 0
        return dm_rollout(LinePos.of(env), self.g, visit, self.seed, self.n_limit, self.n_rollouts, game_type,
                          self.returns_mode)

    def prior(self, env):
        legal = [int(a) for a in env.legal_actions()]
        return [(a, float(uniform_prior(len(legal)))) for a in legal]


class ShuffleRank(object):
    """``shuffle_fn`` of ``dm_oracle.DMSearch``: orders a new node's (action, prior) list by the device key,
    ties by action.  The node is ``search.expanding`` and carries the device's allocation index."""

    def __init__(self, g, episode, ply, seed):
        self.g, self.episode, self.ply, self.seed = g, episode, ply, seed
        self.search = None

    def __call__(self, pairs):
        node = self.search.expanding.index
        pairs.sort(key=lambda ap: (shuffle_rank(self.g, self.episode, self.ply, node, ap[0], self.seed), ap[0]))
