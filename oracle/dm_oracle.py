"""TEST INFRASTRUCTURE ONLY -- pure-Python restatement of the reference's second search driver,
``DeepMindMCTS`` (``rlzero/mcts/deepmind_mcts.py:65-175,384-646``; a port of OpenSpiel's MCTS bot).

Restated without sharing code: ``SearchNode`` (child score with the outcome shortcut :106-151,
``sort_key``/``best_child`` :153-175), ``_apply_tree_policy`` (:477-528, lazy expansion on the second
visit, root-only Dirichlet noise, first-maximum selection), ``mcts_search`` (:554-646, returns vector
indexed by the player who moved, terminal outcomes, MCTS-Solver backup, early stop on a proven root)
and ``step_with_policy`` (:447-472).

Pinned against the LIVE reference in the authoring container by
``tests/test_oracle_vs_reference.py::test_dm_*`` (the unmodified ``DeepMindMCTS`` runs on a two-line
adapter subclass of the reference ``GomokuEnv`` that gives ``legal_actions`` its default argument,
deepmind_mcts.py:497 calls it without one) and by the fixtures that run generated
(``tests/golden/dm_mcts.json``, ``scripts/make_golden_dm.py``).

Determinism: the reference shuffles a new node's children with its private ``RandomState``
(:508) -- a tie-break randomisation; parity runs replace ``_random_state`` by an object whose
``shuffle`` is a no-op (instance attribute injection, the class is untouched), so ties go to the
lowest action on both sides.  The env duck-type it needs: ``legal_actions()``, ``step(a)``,
``is_terminal()``, ``returns()``, ``current_player()``, ``max_utility()``, deep-copyable.
"""
import copy
import math

import numpy as np


class Node(object):
    __slots__ = ('action', 'player', 'prior', 'n', 'w', 'outcome', 'children', 'index')

    def __init__(self, action, player, prior):
        self.index = -1                  # the device's allocation index (set at the node's evaluation)
        self.action = action
        self.player = player
        self.prior = prior
        self.n = 0
        self.w = 0.0
        self.outcome = None
        self.children = []

    def uct(self, parent_n, c):          # deepmind_mcts.py:106-129
        if self.outcome is not None:
            return self.outcome[self.player]
        if self.n == 0:
            return float('inf')
        return self.w / self.n + c * math.sqrt(math.log(parent_n) / self.n)

    def puct(self, parent_n, c):         # deepmind_mcts.py:131-151
        if self.outcome is not None:
            return self.outcome[self.player]
        return (self.n and self.w / self.n) + c * self.prior * math.sqrt(parent_n) / (self.n + 1)

    def sort_key(self):                  # deepmind_mcts.py:153-171
        return (0 if self.outcome is None else self.outcome[self.player], self.n, self.w)

    def best_child(self):                # deepmind_mcts.py:173-175
        best = None
        for ch in self.children:
            if best is None or ch.sort_key() > best.sort_key():
                best = ch
        return best


class DMSearch(object):

    def __init__(self, evaluator, max_simulations=2000, uct_c=2, child_selection_method='puct',
                 add_exploration_noise=False, dirichlet_noise_epsilon=0.25, solve=True, max_utility=1,
                 noise_fn=None, shuffle_fn=None):
        self.evaluator = evaluator
        self.max_simulations = max_simulations
        self.uct_c = uct_c
        self.rule = child_selection_method
        self.add_noise = add_exploration_noise
        self.eps = dirichlet_noise_epsilon
        self.alpha = dirichlet_noise_epsilon    # sic: deepmind_mcts.py:439 stores epsilon as alpha
        self.solve = solve
        self.max_utility = max_utility
        self.noise_fn = noise_fn or (lambda k: np.random.dirichlet([self.alpha] * k))
        self.shuffle_fn = shuffle_fn          # in-place list shuffle (deepmind_mcts.py:508); None = keep the order
        # what an evaluator / shuffle_fn restating the device's random draws reads: the root of the running search
        # and the node whose children are being created (Node.index numbers nodes in the order the device
        # allocates them: at their first evaluation, where the reference creates children at the second visit)
        self.root = None
        self.expanding = None
        self.n_nodes = 0

    def _score(self, ch, parent_n):
        return ch.puct(parent_n, self.uct_c) if self.rule == 'puct' else ch.uct(parent_n, self.uct_c)

    def _descend(self, root, env):       # deepmind_mcts.py:477-528
        path = [root]
        work = copy.deepcopy(env)
        node = root
        while not work.is_terminal() and node.n > 0:
            if not node.children:
                pri = list(self.evaluator.prior(work))
                if node is root and self.add_noise:
                    noise = self.noise_fn(len(pri))
                    pri = [(a, self.eps * z + (1 - self.eps) * p) for (a, p), z in zip(pri, noise)]
                if self.shuffle_fn is not None:
                    self.expanding = node
                    self.shuffle_fn(pri)                  # "Reduce bias from move generation order" (:508)
                mover = work.current_player()
                node.children = [Node(a, mover, p) for a, p in pri]
            best, best_s = None, None
            for ch in node.children:                      # max(): first maximum
                s = self._score(ch, node.n)
                if best is None or s > best_s:
                    best, best_s = ch, s
            work.step(best.action)
            node = best
            path.append(node)
        return path, work

    def search(self, env):               # deepmind_mcts.py:554-646
        root = Node(None, env.current_player(), 1)
        self.root, self.n_nodes = root, 0
        for _ in range(self.max_simulations):
            path, work = self._descend(root, env)
            if work.is_terminal():
                returns = work.returns()
                path[-1].outcome = returns
                solved = self.solve
            else:
                returns = self.evaluator.evaluate(work)
                solved = False
                path[-1].index = self.n_nodes
                self.n_nodes += 1
            while path:
                node = path.pop()
                node.w += returns[node.player]
                node.n += 1
                if solved and node.children:
                    player = node.children[0].player
                    best, all_solved = None, True
                    for ch in node.children:
                        if ch.outcome is None:
                            all_solved = False
                        elif best is None or ch.outcome[player] > best.outcome[player]:
                            best = ch
                    if best is not None and (all_solved or best.outcome[player] == self.max_utility):
                        node.outcome = best.outcome
                    else:
                        solved = False
            if root.outcome is not None:
                break
        return root

    def step_with_policy(self, env):     # deepmind_mcts.py:447-472
        root = self.search(env)
        action = root.best_child().action
        return [(a, 1.0 if a == action else 0.0) for a in env.legal_actions()], action, root


class ClosedFormEvaluator(object):
    """Evaluator (deepmind_mcts.py:14-28) from a closed-form evaluator id of oracle/evaluators.py:
    evaluate -> [v, -v] in player order for the player to move, prior -> [(action, p)]."""

    def __init__(self, eval_id):
        from . import evaluators
        self.ev = evaluators
        self.eval_id = eval_id

    def evaluate(self, env):
        v = self.ev.value_of(self.eval_id, env.states, env.last_move)
        p = env.current_player()
        out = [0.0, 0.0]
        out[p] = v
        out[1 - p] = -v
        return out

    def prior(self, env):
        legal = [int(a) for a in env.legal_actions()]
        pri = self.ev.priors_of(self.eval_id, env.states, env.last_move, legal)
        return [(a, float(x)) for a, x in zip(legal, pri)]


class NoShuffle(object):
    """Replacement for DeepMindMCTS._random_state in parity runs: no child shuffle; the Dirichlet
    draw (root noise) comes from the wrapped RandomState, or is uniform when none is given."""

    def __init__(self, rs=None):
        self.rs = rs

    def shuffle(self, x):
        pass

    def dirichlet(self, alpha):
        if self.rs is None:
            return np.ones(len(alpha)) / len(alpha)
        return self.rs.dirichlet(alpha)


def tree_summary(root):
    """Comparable digest of a finished search: per root child (action, N, W, outcome), root N/W/outcome."""
    return dict(root_n=root.n, root_w=root.w, root_outcome=root.outcome,
                children=[(ch.action, ch.n, ch.w, ch.outcome) for ch in root.children])
