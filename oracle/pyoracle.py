"""TEST INFRASTRUCTURE ONLY -- pure-Python restatement of the reference hot path.

Restates, without sharing code, the algorithm of

* ``rlzero/games/gomoku/gomoku_env.py``  (``Board`` below)
* ``rlzero/mcts/node.py``                (``Node``)
* ``rlzero/mcts/alphazero_mcts.py``      (``Search``, ``SearchPlayer``)
* ``rlzero/games/gomoku/game.py``        (``self_play_episode``, ``play_match``)

so that parity tests and the CPU baseline can run where ``/root/reference``
does not exist (the GPU box).  It is pinned against the live reference by
``tests/test_oracle_vs_reference.py`` (authoring container) and against the
fixtures that run generated, ``tests/golden/*.json`` (everywhere).

Cost model on purpose mirrors the reference (one object per child, one board
copy per playout, win scan over all stones) so that timing it is a fair
stand-in for timing the reference's CPU path.
"""
import copy
import math

import numpy as np

RULE_UCT = 0   # reference behaviour: UCB1, +inf for unvisited (node.py:75-88)
RULE_PUCT = 1  # optional rule, formula of deepmind_mcts.py:149-151


class Board(object):
    """k-in-a-row on an N x N board (gomoku_env.py:11-285).

    cells[m] is -1 (empty) / 0 / 1; ``legal`` is the ascending list of empty
    squares from which played moves are removed (gomoku_env.py:31,56), which
    is what fixes the child order of every tree node.
    """

    def __init__(self, board_size=8, n_in_row=5, start_player_idx=0):
        self.board_size = board_size
        self.n_in_row = n_in_row
        self.players = [0, 1]
        self.start_player_idx = start_player_idx
        self._to_move = self.players[start_player_idx]
        self.legal = list(range(board_size * board_size))

    # -- gomoku_env.py:33-47
    def reset(self, start_player_idx=0):
        if self.board_size < self.n_in_row:
            raise ValueError('board_size < n_in_row')
        if start_player_idx not in (0, 1):
            raise ValueError('start_player_idx must be 0 or 1')
        self.start_player_idx = start_player_idx
        self._to_move = self.players[start_player_idx]
        self.legal = list(range(self.board_size * self.board_size))
        self.states = {}
        self.last_move = -1
        self.info = {}
        return self.current_state()

    # -- gomoku_env.py:49-70
    def step(self, action):
        if action not in self.legal:
            raise AssertionError('illegal action %r' % (action,))
        mover = self._to_move
        self.states[action] = mover
        self.legal.remove(action)
        self.last_move = action
        win, winner = self.has_a_winner()
        reward = 0
        if win:
            reward = 1 if winner == mover else -1
        self._to_move = 1 - mover
        return self.current_state(), reward, win, self.info

    def leagel_actions(self):  # [sic] gomoku_env.py:72-73
        return self.legal

    def legal_actions(self, player=None):  # gomoku_env.py:274-275
        return self.legal

    def current_player(self):
        return self._to_move

    # -- gomoku_env.py:95-114
    def current_state(self):
        n = self.board_size
        planes = np.zeros((4, n, n))
        for m, p in self.states.items():
            planes[0 if p == self._to_move else 1, m // n, m % n] = 1.0
        if self.states:
            planes[2, self.last_move // n, self.last_move % n] = 1.0
        if len(self.states) % 2 == 0:
            planes[3, :, :] = 1.0
        return planes

    # -- gomoku_env.py:116-170
    def has_a_winner(self):
        n, k = self.board_size, self.n_in_row
        st = self.states
        if len(st) < 2 * k - 1:
            return False, -1
        # The reference walks the stones in set order; with alternating legal
        # play at most one colour can own a line, so the order is immaterial.
        for m in sorted(st):
            h, w = divmod(m, n)
            p = st[m]
            room_r = w <= n - k
            room_u = h <= n - k
            room_l = w >= k - 1
            if room_r and all(st.get(m + i, -1) == p for i in range(k)):
                return True, p
            if room_u and all(st.get(m + i * n, -1) == p for i in range(k)):
                return True, p
            if room_r and room_u and all(
                    st.get(m + i * (n + 1), -1) == p for i in range(k)):
                return True, p
            if room_l and room_u and all(
                    st.get(m + i * (n - 1), -1) == p for i in range(k)):
                return True, p
        return False, -1

    # -- gomoku_env.py:196-208
    def game_end_winner(self):
        win, winner = self.has_a_winner()
        if win:
            return True, winner
        if not self.legal:
            return True, -1
        return False, -1

    def is_terminal(self):
        return self.game_end_winner()[0]

    # -- gomoku_env.py:210-225 (players are 0/1 but the test is ==1 / ==2)
    def returns(self):
        _, winner = self.has_a_winner()
        if winner == 1:
            return [1, -1]
        if winner == 2:
            return [-1, 1]
        return [0, 0]

    def move_to_location(self, move):
        return [move // self.board_size, move % self.board_size]

    def location_to_move(self, location):
        if len(location) != 2:
            return -1
        move = location[0] * self.board_size + location[1]
        if move not in range(self.board_size * self.board_size):
            return -1
        return move

    def max_utility(self):
        return 1


class Node(object):
    """Tree node (node.py:7-154): children keyed by action in insertion order."""
    __slots__ = ('parent', 'children', 'n', 'w', 'prior')

    def __init__(self, parent=None, prior=1.0):
        self.parent = parent
        self.children = {}
        self.n = 0
        self.w = 0
        self.prior = prior

    def score(self, c, rule):
        if rule == RULE_PUCT:  # deepmind_mcts.py:149-151
            return (self.n and self.w / self.n) + c * self.prior * math.sqrt(
                self.parent.n) / (self.n + 1)
        # node.py:75-88
        if self.parent.n == 0 or self.n == 0:
            return float('inf')
        return self.w / self.n + c * math.sqrt(math.log(self.parent.n) / self.n)

    def select(self, c, rule):  # node.py:32-42: first maximum wins
        if not self.children:
            raise ValueError('Node has no children.')
        best_a, best_node, best_s = None, None, None
        for a, ch in self.children.items():
            s = ch.score(c, rule)
            if best_s is None or s > best_s:
                best_a, best_node, best_s = a, ch, s
        return best_a, best_node

    def expand(self, action_priors, add_noise=False, rng=None):  # node.py:44-73
        action_priors = list(action_priors)
        if add_noise:
            noise = (rng or np.random).dirichlet(0.3 * np.ones(len(action_priors)))
            for i, (a, p) in enumerate(action_priors):
                if a not in self.children:
                    self.children[a] = Node(self, 0.75 * p + 0.25 * noise[i])
        else:
            for a, p in action_priors:
                if a not in self.children:
                    self.children[a] = Node(self, p)

    def backup(self, value):  # node.py:119-144 (iterative form of the recursion)
        node = self
        while node is not None:
            node.n += 1
            node.w += value
            value = -value
            node = node.parent


def softmax(x):  # alphazero_mcts.py:10-14
    e = np.exp(x - np.max(x))
    return e / np.sum(e)


class Search(object):
    """AlphaZeroMCTS restated (alphazero_mcts.py:17-103)."""

    def __init__(self, policy_value_fn, n_playout=1000, c_puct=5,
                 add_noise=False, rule=RULE_UCT, rng=None, leaves_per_wave=1, virtual_loss=1.0):
        # leaves_per_wave > 1: the product's opt-in leaf-parallel mode (rz_tree_desc.leaves_per_tree).  The
        # reference has no such mode -- PARITY UNPINNED for it: `wave` below restates the product's own
        # definition (include/rlzero_b200.h) so that the kernels can be checked bit for bit; with
        # leaves_per_wave == 1 this class is the reference's sequential search.
        self.leaves_per_wave = leaves_per_wave
        self.virtual_loss = virtual_loss
        self.root = Node(None, 1.0)
        self.policy_value_fn = policy_value_fn
        self.n_playout = n_playout
        self.c_puct = c_puct
        self.add_noise = add_noise
        self.rule = rule
        self.rng = rng

    def playout(self, board):  # alphazero_mcts.py:42-71
        node = self.root
        while node.children:
            a, node = node.select(self.c_puct, self.rule)
            board.step(a)
        priors, v = self.policy_value_fn(board)  # also on terminal leaves (:59)
        end, winner = board.game_end_winner()
        if not end:
            node.expand(priors, self.add_noise, self.rng)
        elif winner == -1:
            v = 0.0
        else:
            v = 1.0 if winner == board.current_player() else -1.0
        node.backup(-v)

    def wave(self, board, budget):
        """`budget` playouts that share one evaluation batch: descend, put a virtual visit and a virtual loss on the
        path, descend again ...; then take the virtual statistics off in reverse order (restoring the saved sums)
        and expand / back up the leaves in order; a leaf reached twice is expanded once and backed up twice."""
        leaves, undo = [], []
        for _ in range(budget):
            b = copy.deepcopy(board)
            node, path = self.root, []
            while node.children:
                a, node = node.select(self.c_puct, self.rule)
                b.step(a)
                path.append(node)
            leaves.append((b, node))
            for nd in path:
                undo.append((nd, nd.w))
                nd.w = (nd.w - self.virtual_loss) if nd.n > 0 else -self.virtual_loss
                nd.n += 1
            self.root.n += 1
        for nd, w in reversed(undo):
            nd.w = w
            nd.n -= 1
        self.root.n -= budget
        for b, node in leaves:
            priors, v = self.policy_value_fn(b)
            end, winner = b.game_end_winner()
            if not end:
                if not node.children:
                    node.expand(priors, self.add_noise, self.rng)
            elif winner == -1:
                v = 0.0
            else:
                v = 1.0 if winner == b.current_player() else -1.0
            node.backup(-v)

    def simulate(self, board, temperature=1e-3):  # alphazero_mcts.py:73-94
        if self.leaves_per_wave > 1:
            target = self.root.n + self.n_playout
            while self.root.n < target:
                budget = min(self.leaves_per_wave, target - self.root.n)
                self.wave(board, budget if self.root.children else 1)
        else:
            for _ in range(self.n_playout):
                self.playout(copy.deepcopy(board))
        acts = tuple(self.root.children.keys())
        visits = np.array([ch.n for ch in self.root.children.values()])
        return acts, softmax(1.0 / temperature * np.log(visits + 1e-10))

    def update_with_move(self, last_move):  # alphazero_mcts.py:96-103
        if last_move in self.root.children:
            self.root = self.root.children[last_move]
            self.root.parent = None
        else:
            self.root = Node(None, 1.0)

    # helpers for tests ----------------------------------------------------
    def root_visits(self, n_actions):
        out = np.zeros(n_actions, dtype=np.int32)
        for a, ch in self.root.children.items():
            out[a] = ch.n
        return out

    def root_values(self, n_actions):
        out = np.zeros(n_actions, dtype=np.float64)
        for a, ch in self.root.children.items():
            out[a] = ch.w
        return out


class SearchPlayer(object):
    """AlphaZeroPlayer restated (alphazero_mcts.py:109-165); uses the global
    ``np.random`` stream exactly like the reference unless ``rng`` is given."""

    def __init__(self, policy_value_fn, n_playout=1000, c_puct=5,
                 is_selfplay=False, rule=RULE_UCT, rng=None):
        self.is_selfplay = is_selfplay
        self.rng = rng
        self.mcts = Search(policy_value_fn, n_playout, c_puct,
                           add_noise=is_selfplay, rule=rule, rng=rng)

    def reset_player(self):
        self.mcts.update_with_move(-1)

    def get_action(self, board, temperature=1e-3, return_prob=False):
        rng = self.rng or np.random
        pi = np.zeros(board.board_size * board.board_size)
        if len(board.leagel_actions()) == 0:
            print('WARNING: the board is full')
            return None
        acts, probs = self.mcts.simulate(board, temperature)
        pi[list(acts)] = probs
        move = rng.choice(acts, p=probs)
        if self.is_selfplay:
            self.mcts.update_with_move(move)
        else:
            move = rng.choice(acts, p=probs)  # sampled twice (:157)
            self.mcts.update_with_move(-1)
        return (move, pi) if return_prob else move


def self_play_episode(board, player, temperature=1e-3):
    """GameControl.start_self_play restated (game.py:96-134)."""
    board.reset()
    states, pis, movers = [], [], []
    while True:
        move, pi = player.get_action(board, temperature=temperature,
                                     return_prob=True)
        states.append(board.current_state())
        pis.append(pi)
        movers.append(board.current_player())
        board.step(move)
        end, winner = board.game_end_winner()
        if end:
            z = np.zeros(len(movers))
            if winner != -1:
                z[np.array(movers) == winner] = 1.0
                z[np.array(movers) != winner] = -1.0
            player.reset_player()
            return winner, list(zip(states, pis, z))


def play_match(board, player0, player1):
    """GameControl.start_play restated (game.py:61-94): player 0 always moves
    first because the env is reset() without arguments."""
    board.reset()
    seats = {0: player0, 1: player1}
    while True:
        move = seats[board.current_player()].get_action(board)
        board.step(move)
        end, winner = board.game_end_winner()
        if end:
            return winner


class RolloutSearch(object):
    """RolloutMCTS restated (rollout_mcts.py:10-108): uniform priors, leaf value from a random
    playout.  ``rollout`` selects the rollout policy: 'random' draws ``np.random.rand(len(legal))``
    per ply and plays the argmax exactly like the reference (:96-100, :63-65); 'first' / 'last' play
    the lowest / highest legal move (deterministic stand-ins for device parity tests); a callable
    ``rollout(board, root_n)`` returns the leaf value itself (``rollout_oracle.AZRollout``: the device's
    counter-based playouts, draw for draw).

    Quirk kept on purpose: the winner is compared with ``current_player()`` AFTER the playout
    (:69-72), and the env flips the player after every move (gomoku_env.py:67-68), so every
    decisive playout yields -1 and only ties yield 0."""

    def __init__(self, n_playout=1000, c_puct=5.0, n_limit=1000, rollout='random', rng=None):
        self.root = Node(None, 1.0)
        self.n_playout = n_playout
        self.c_puct = c_puct
        self.n_limit = n_limit
        self.rollout = rollout
        self.rng = rng

    def policy_value_fn(self, board):  # :102-108
        legal = board.leagel_actions()
        return zip(legal, np.ones(len(legal)) / len(legal))

    def rollout_policy(self, board):  # :96-100
        legal = board.leagel_actions()
        if self.rollout == 'random':
            probs = (self.rng or np.random).rand(len(legal))
        elif self.rollout == 'first':
            probs = -np.arange(len(legal), dtype=np.float64)
        else:
            probs = np.arange(len(legal), dtype=np.float64)
        return zip(legal, probs)

    def evaluate(self, board):  # :49-74
        if callable(self.rollout):
            # a restatement of the device's playout (oracle/rollout_oracle.AZRollout), keyed by the root's
            # visit count at this evaluation
            return self.rollout(board, self.root.n)
        winner = -1
        for _ in range(self.n_limit):
            end, winner = board.game_end_winner()
            if end:
                break
            best = max(self.rollout_policy(board), key=lambda ap: ap[1])[0]
            board.step(best)
        if winner == -1:
            return 0
        return 1.0 if winner == board.current_player() else -1.0

    def playout(self, board):  # :23-47
        node = self.root
        while node.children:
            action, node = node.select(self.c_puct, RULE_UCT)
            board.step(action)
        priors = self.policy_value_fn(board)
        end, _ = board.game_end_winner()
        if not end:
            node.expand(priors)
        node.backup(-self.evaluate(board))

    def simulate(self, board, temperature=1e-3):  # :76-81
        for _ in range(self.n_playout):
            self.playout(copy.deepcopy(board))
        return max(self.root.children.items(), key=lambda an: an[1].n)[0]

    def update_with_move(self, last_move):  # :83-94
        if last_move in self.root.children:
            self.root = self.root.children[last_move]
            self.root.parent = None
        else:
            self.root = Node(None, 1.0)

    def root_visits(self, n_actions):
        out = np.zeros(n_actions, dtype=np.int32)
        for a, ch in self.root.children.items():
            out[a] = ch.n
        return out


class RolloutSearchPlayer(object):
    """RolloutPlayer restated (rollout_mcts.py:114-140)."""

    def __init__(self, n_playout=1000, c_puct=5, rollout='random', rng=None):
        self.mcts = RolloutSearch(n_playout, c_puct, rollout=rollout, rng=rng)

    def reset_player(self):
        self.mcts.update_with_move(-1)

    def get_action(self, board, **kwargs):
        if len(board.leagel_actions()) > 0:
            move = self.mcts.simulate(board)
            self.mcts.update_with_move(-1)
            return move
        print('WARNING: the board is full')


class ConnectFourBoard(object):
    """Connect Four (k-in-a-row with gravity on a rows x cols board) behind the duck-typed env API
    of the reference's search (SURVEY.md 8 b1).  The reference has no such env; this is the CPU
    definition the device kernels (RZ_GAME_CONNECT4) are checked against, written independently of
    ``Board`` (explicit direction scan instead of the reference's window test).  Actions are
    columns; ``states`` / ``last_move`` use the square index r*cols + c, row 0 at the bottom."""

    def __init__(self, rows=6, cols=7, n_in_row=4):
        self.board_size = rows          # the attribute the reference's player reads
        self.board_width = cols
        self.n_actions = cols
        self.n_in_row = n_in_row
        self.players = [0, 1]
        self._to_move = 0
        self.legal = list(range(cols))

    def reset(self, start_player_idx=0):
        self._to_move = self.players[start_player_idx]
        self.legal = list(range(self.board_width))
        self.heights = [0] * self.board_width
        self.states = {}
        self.last_move = -1
        self.info = {}
        return self.current_state()

    def step(self, action):
        if action not in self.legal:
            raise AssertionError('illegal action %r' % (action,))
        mover = self._to_move
        cell = self.heights[action] * self.board_width + action
        self.heights[action] += 1
        self.states[cell] = mover
        if self.heights[action] == self.board_size:
            self.legal.remove(action)
        self.last_move = cell
        win, winner = self.has_a_winner()
        reward = (1 if winner == mover else -1) if win else 0
        self._to_move = 1 - mover
        return self.current_state(), reward, win, self.info

    def leagel_actions(self):
        return self.legal

    def legal_actions(self, player=None):
        return self.legal

    def current_player(self):
        return self._to_move

    def current_state(self):
        h, w = self.board_size, self.board_width
        planes = np.zeros((4, h, w))
        for m, p in self.states.items():
            planes[0 if p == self._to_move else 1, m // w, m % w] = 1.0
        if self.states:
            planes[2, self.last_move // w, self.last_move % w] = 1.0
        if len(self.states) % 2 == 0:
            planes[3, :, :] = 1.0
        return planes

    def has_a_winner(self):
        h, w, k = self.board_size, self.board_width, self.n_in_row
        if len(self.states) < 2 * k - 1:
            return False, -1
        for m, p in self.states.items():
            r, c = divmod(m, w)
            for dr, dc in ((0, 1), (1, 0), (1, 1), (1, -1)):
                rr, cc, n = r, c, 0
                while 0 <= rr < h and 0 <= cc < w and self.states.get(rr * w + cc, -1) == p:
                    n += 1
                    rr += dr
                    cc += dc
                if n >= k:
                    return True, p
        return False, -1

    def game_end_winner(self):
        win, winner = self.has_a_winner()
        if win:
            return True, winner
        if not self.legal:
            return True, -1
        return False, -1

    def is_terminal(self):
        return self.game_end_winner()[0]


class DMBoard(Board):
    """``Board`` with the extra methods ``DeepMindMCTS`` calls (deepmind_mcts.py:497-506,595-597):
    ``legal_actions()`` without argument and a ``zero_sum`` switch for ``returns`` (the reference's
    ``GomokuEnv.returns`` tests winner == 1 / == 2 although players are 0 / 1, gomoku_env.py:216-219;
    ``zero_sum=True`` is the evident intent, RZ_RETURNS_ZERO_SUM on the device)."""

    def __init__(self, board_size=8, n_in_row=5, zero_sum=False):
        Board.__init__(self, board_size, n_in_row)
        self.zero_sum = zero_sum

    def returns(self):
        if not self.zero_sum:
            return Board.returns(self)
        win, winner = self.has_a_winner()
        if not win:
            return [0, 0]
        return [1, -1] if winner == 0 else [-1, 1]
