"""``DeepMindMCTS`` / ``MCTSBot`` / ``SearchNode`` / ``RandomRolloutEvaluator`` with the reference's
API (rlzero/mcts/deepmind_mcts.py:14-175,384-691 -- its port of OpenSpiel's MCTS bot), searching
on the GPU.

The search is the ``RZ_FLAVOUR_DEEPMIND`` mode of the tree kernels (csrc/rz_tree.cu): returns vector
indexed by the player who moved, the outcome shortcut in the child score, terminal outcomes, the
MCTS-Solver backup (``solve``), root-only Dirichlet noise, early stop once the root is proven, and
``best_child`` by ``(outcome, explore_count, total_reward)``.  Evaluation goes

* through the device for a native evaluator -- ``RandomRolloutEvaluator`` below (random playouts in
  ``rz_eval_rollout_dm``) or any object carrying a ``device_evaluator`` (the tensor-core network), or
* through ``evaluator.evaluate(env)`` / ``evaluator.prior(env)`` themselves (the reference's
  ``Evaluator`` contract, :14-28) per leaf on the host -- slow, but it accepts any user evaluator.

Randomness.  The reference owns a private ``np.random.RandomState`` (:444) that shuffles every new
node's ``children`` list (:508 -- ``max()`` takes the first maximum, so the list order is the tie-break
of the descent and of ``best_child``) and draws the root's Dirichlet noise (:539).  Three modes:

* ``random_state=np.random.RandomState(seed)`` -- the seeded parity path: the host walks the search one
  simulation at a time, draws noise and shuffle from that very stream in the reference's order (at a
  node's SECOND visit, when the reference creates its children) and hands the kernels the resulting
  float64 priors and child order: visit counts, value sums and the move equal the reference's for the
  same seed, bit for bit (``tests/golden/dm_mcts_shuffle.json``).  One tree, three small device-host
  copies per simulation: a checker, not the fast path;
* ``child_shuffle=True`` (default, like the reference) without a ``random_state`` -- counter-based random
  child order and root noise on the device, inside the captured wave graph (same distribution as the
  reference; the child order and the device playouts are pinned draw for draw to
  ``oracle/rollout_oracle.py``);
* ``child_shuffle=False`` -- no shuffle, ties to the lowest action (the deterministic fixtures).

The reference's quirks that change results are kept: the noise
concentration is ``dirichlet_noise_epsilon`` (:439 stores epsilon as alpha), and ``returns`` of a
finished Gomoku game follow ``GomokuEnv.returns`` literally unless ``returns_mode`` says otherwise.
"""
import ctypes as C
import time

import numpy as np
import torch

from .. import _lib as L
from ..engine import SearchForest
from .player import Player


class Evaluator(object):
    """Abstract evaluation function for a game (deepmind_mcts.py:14-28)."""

    def evaluate(self, game_env):
        """Returns evaluation on given state, one value per player."""
        raise NotImplementedError

    def prior(self, game_env):
        """Returns a probability for each legal action in the given state."""
        raise NotImplementedError


class RandomRolloutEvaluator(Evaluator):
    """Average outcome of ``n_rollouts`` uniformly random playouts (deepmind_mcts.py:31-62), played on
    the device for every leaf of the wave at once."""
    graph_capturable = True
    prior_is_log = False

    def __init__(self, n_rollouts=20, random_state=None, n_limit=1000, seed=0):
        self.n_rollouts = int(n_rollouts)
        self._random_state = random_state or np.random.RandomState()
        self.n_limit = int(n_limit)
        self.seed = int(seed)
        self.value64 = None         # float64 [G][2] returns vector handed to rz_tree_expand_backup_dm
        self.device_evaluator = self

    def __call__(self, forest):
        if self.value64 is None or self.value64.shape[0] != forest.G:
            self.value64 = torch.zeros(forest.G, 2, dtype=torch.float64, device=forest.device)
        L.check(forest.lib.rz_eval_rollout_dm(C.byref(forest.desc), self.n_rollouts, self.seed, self.n_limit,
                                              L.ptr(forest.prior), L.ptr(self.value64), forest._s()),
                'rz_eval_rollout_dm')

    # the reference's host-side methods, for callers that use the evaluator on its own
    def evaluate(self, game_env):
        import copy
        result = None
        for _ in range(self.n_rollouts):
            working_env = copy.deepcopy(game_env)
            while not working_env.is_terminal():
                legal_actions = working_env.legal_actions(game_env.current_player())
                working_env.step(self._random_state.choice(legal_actions))
            returns = np.array(working_env.returns())
            result = returns if result is None else result + returns
        return result / self.n_rollouts

    def prior(self, game_env):
        legal_actions = game_env.legal_actions(game_env.current_player())
        return [(action, 1.0 / len(legal_actions)) for action in legal_actions]


class _HostEvaluator(object):
    """Slow path: ``evaluator.prior(env)`` / ``evaluator.evaluate(env)`` per leaf on the host."""
    graph_capturable = False
    prior_is_log = False

    def __init__(self, evaluator, env_factory):
        self.evaluator = evaluator
        self.env_factory = env_factory
        self.value64 = None
        self.prior64 = None       # float64 priors for a forest that keeps them (the seeded parity path)

    def __call__(self, forest):
        rows, meta, depth = forest.leaf_boards()
        hist = forest.leaf_hist.cpu().numpy() if forest.is_go else None
        prior = np.zeros((forest.G, forest.AS), dtype=np.float64)
        if self.prior64 is None and forest.edge_P64 is not None:
            self.prior64 = torch.zeros(forest.G, forest.AS, dtype=torch.float64, device=forest.device)
        ret = np.zeros((forest.G, 2), dtype=np.float64)
        if self.value64 is None:
            self.value64 = torch.zeros(forest.G, 2, dtype=torch.float64, device=forest.device)
        for g in range(forest.G):
            if depth[g] < 0 or meta[g][L.META_STATUS] != L.ACTIVE:
                continue          # terminal leaves take env.returns() on the device (:597-600)
            env = self.env_factory(rows[g], meta[g], None if hist is None else hist[g])
            ret[g] = np.asarray(self.evaluator.evaluate(env), dtype=np.float64)[:2]
            for a, p in self.evaluator.prior(env):
                prior[g, int(a)] = p
        forest.prior.copy_(torch.from_numpy(prior.astype(np.float32)))
        if self.prior64 is not None:
            self.prior64.copy_(torch.from_numpy(prior))
        self.value64.copy_(torch.from_numpy(ret))


class SearchNode(object):
    """A node of the finished search (deepmind_mcts.py:65-226): host view of the device tree with the
    reference's attributes ``action, player, prior, explore_count, total_reward, outcome, children``."""
    __slots__ = ['action', 'player', 'prior', 'explore_count', 'total_reward', 'outcome', '_snap', '_node',
                 '_kids']

    def __init__(self, action, player, prior, explore_count=0, total_reward=0.0, outcome=None, _snap=None,
                 _node=-1):
        self.action = action
        self.player = player
        self.prior = prior
        self.explore_count = explore_count
        self.total_reward = total_reward
        self.outcome = outcome
        self._snap = _snap
        self._node = _node
        self._kids = None

    @staticmethod
    def _decode(code):
        return None if code == 0 else [(code & 3) - 1, ((code >> 2) & 3) - 1]

    @classmethod
    def from_snapshot(cls, snap, root_player):
        return cls(None, root_player, 1, snap['root_N'], snap['root_W'] if snap['root_N'] else 0.0,
                   cls._decode(snap.get('root_O', 0)), _snap=snap, _node=0 if snap['n_nodes'] > 0 else -1)

    @property
    def children(self):
        if self._kids is None:
            kids = []
            if self._snap is not None and self._node >= 0:
                s, i = self._snap, self._node
                mover = self.player if self.action is None else 1 - self.player   # who moves at this node
                for a in range(s['N'].shape[1]):
                    n = int(s['N'][i, a])
                    if n < 0:
                        continue
                    ch = int(s['child'][i, a]) if n >= 1 else -1
                    kids.append(SearchNode(a, mover, float(s['P'][i, a]), n, float(s['W'][i, a]) if n >= 1 else 0.0,
                                           self._decode(int(s['O'][i, a])) if 'O' in s else None, _snap=s,
                                           _node=ch if ch >= 0 else -1))
                if 'R' in s:      # the shuffled list order (deepmind_mcts.py:508), which max() breaks ties in
                    kids.sort(key=lambda c: (int(s['R'][i, c.action]), c.action))
            self._kids = kids
        return self._kids

    def uct_value(self, parent_explore_count, uct_c):
        import math
        if self.outcome is not None:
            return self.outcome[self.player]
        if self.explore_count == 0:
            return float('inf')
        return self.total_reward / self.explore_count + uct_c * math.sqrt(
            math.log(parent_explore_count) / self.explore_count)

    def puct_value(self, parent_explore_count, uct_c):
        import math
        if self.outcome is not None:
            return self.outcome[self.player]
        return (self.explore_count and self.total_reward / self.explore_count) + \
            uct_c * self.prior * math.sqrt(parent_explore_count) / (self.explore_count + 1)

    def sort_key(self):
        return (0 if self.outcome is None else self.outcome[self.player], self.explore_count, self.total_reward)

    def best_child(self):
        return max(self.children, key=SearchNode.sort_key)

    def children_str(self, game_env=None):
        return '\n'.join([c.to_str(game_env) for c in reversed(sorted(self.children, key=SearchNode.sort_key))])

    def to_str(self, game_env=None):
        return ('action:{}, player: {}, prior: {:5.3f}, value: {:6.3f}, sims: {:5d}, outcome: {}, {:3d} children'
                ).format(str(self.action), self.player, self.prior,
                         self.explore_count and self.total_reward / self.explore_count, self.explore_count,
                         ('{:4.1f}'.format(self.outcome[self.player]) if self.outcome else 'none'),
                         len(self.children))

    def __str__(self):
        return self.to_str(None)


class DeepMindMCTS(object):
    """Bot that uses Monte-Carlo Tree Search algorithm (deepmind_mcts.py:384-646), trees on the GPU."""

    def __init__(self, game_env, uct_c=2, max_simulations=2000, evaluator=None, child_selection_method='puct',
                 add_exploration_noise=False, dirichlet_noise_alpha=1.0, dirichlet_noise_epsilon=0.25, solve=True,
                 verbose=False, returns_mode=L.RETURNS_REFERENCE, device='cuda', seed=0, child_shuffle=True,
                 random_state=None):
        self.game_env = game_env
        self.uct_c = uct_c
        self.max_simulations = max_simulations
        self.evaluator = evaluator if evaluator is not None else RandomRolloutEvaluator()
        if child_selection_method not in ('puct', 'uct'):
            raise ValueError("child_selection_method must be 'puct' or 'uct'")
        self.child_selection_method = child_selection_method
        self.max_utility = game_env.max_utility()
        if add_exploration_noise:
            assert dirichlet_noise_alpha is not None
            assert dirichlet_noise_epsilon is not None
        self.add_exploration_noise = add_exploration_noise
        self.dirichlet_noide_alpha = dirichlet_noise_epsilon      # [sic] deepmind_mcts.py:439
        self.dirichlet_noise_epsilon = dirichlet_noise_epsilon
        self.verbose = verbose
        self.solve = solve
        self.returns_mode = int(returns_mode)
        self.device = device
        self._seed = int(seed)
        self.child_shuffle = bool(child_shuffle)
        self._random_state = random_state        # np.random.RandomState: the seeded parity path
        self._forest = None
        self._dev_eval = None

    # ---------------------------------------------------------------- plumbing
    @staticmethod
    def _geometry(env):
        """(H, k, W, game_type, komi) of a GomokuEnv-like or GoEnv-like env."""
        if hasattr(env, '_N'):                                   # GoEnv (go_env.py:47)
            return env._N, 1, env._N, L.GAME_GO, float(getattr(env, '_komi', 7.5))
        return (env.board_size, env.n_in_row, getattr(env, 'board_width', env.board_size),
                getattr(env, 'game_type', L.GAME_GOMOKU), 0.0)

    def _ensure_forest(self, env):
        H, k, W, game_type, komi = self._geometry(env)
        f = self._forest
        if (f is not None and (f.H, f.k, f.W, f.game_type) == (H, k, W, game_type) and f.komi == (komi if f.is_go else 0.0)
                and self.max_simulations <= f.n_playout and f.c_puct == float(self.uct_c)):
            return f
        rule = L.RULE_PUCT if self.child_selection_method == 'puct' else L.RULE_UCT
        seeded = self._random_state is not None
        shuffle = None if not self.child_shuffle else ('host' if seeded else 'random')
        self._forest = SearchForest(1, H, k, n_playout=self.max_simulations, c_puct=self.uct_c, rule=rule,
                                    max_carry=0, device=self.device, board_width=W, game_type=game_type,
                                    komi=komi, flavour=L.FLAVOUR_DEEPMIND, solve=self.solve,
                                    returns_mode=self.returns_mode, noise_root_only=True,
                                    child_shuffle=shuffle, prior_f64=seeded)
        native = getattr(self.evaluator, 'device_evaluator', None)
        if native is not None:
            self._dev_eval = native
        else:
            if game_type == L.GAME_GO:
                raise NotImplementedError('host evaluators on Go leaves: use RandomRolloutEvaluator or a network')
            from ..games.gomoku.gomoku_env import LeafEnvView
            self._dev_eval = _HostEvaluator(
                self.evaluator, lambda rows, meta, hist: LeafEnvView(rows, meta, H, k, W, game_type))
        return self._forest

    def _upload(self, env):
        f = self._forest
        state = env.device_state()
        if f.is_go:
            rows, hist, meta = state
            f.root_hist.copy_(hist.to(f.device))
        else:
            rows, meta = state
        f.root_rows.copy_(rows.to(f.device))
        f.root_meta.copy_(meta.to(f.device))
        f.root_meta[:, L.META_FAULT] = 0
        f.reset_trees()

    # ------------------------------------------------------------ reference API
    def mcts_search(self, game_env):
        """A vanilla Monte-Carlo Tree Search from ``game_env``'s position (deepmind_mcts.py:554-646);
        returns the root ``SearchNode``."""
        f = self._ensure_forest(game_env)
        self._upload(game_env)
        self._seed += 1
        if self._random_state is not None:
            self._search_seeded(f)
        else:
            eps = float(self.dirichlet_noise_epsilon) if self.add_exploration_noise else 0.0
            f.run_waves(self.max_simulations, self._dev_eval, noise_eps=eps,
                        noise_alpha=float(self.dirichlet_noide_alpha), seed=self._seed)
        f.raise_faults()
        return SearchNode.from_snapshot(f.dump_tree(0), int(game_env.current_player()))

    def _search_seeded(self, f):
        """The search with noise and child order drawn from ``self._random_state`` exactly when and how the
        reference draws them (deepmind_mcts.py:499-513): at the second visit of a node -- the kernels created its
        edge block at the first visit, with the evaluator's priors in action order -- the root's priors are mixed
        with Dirichlet noise (:484-485,530-552; float64, ``eps * noise + (1 - eps) * p``), then the (action,
        prior) list is shuffled, and the descent is repeated with that order as the tie-break."""
        rs = self._random_state
        ev = self._dev_eval
        prior_is_log = bool(getattr(ev, 'prior_is_log', False))
        AS, A = f.AS, f.A
        ordered = set()                   # edge blocks whose children the reference has created
        eps = float(self.dirichlet_noise_epsilon)
        for _ in range(self.max_simulations):
            f.select()
            depth = int(f.depth[0].item())
            if depth < 0:
                break                      # proven root (:643-644) or a finished game
            if depth > 0:
                node = int(f.path_node[0, depth - 1].item())
                if node not in ordered:
                    base = node * AS
                    legal = np.nonzero(f.edge_N[base:base + A].cpu().numpy() >= 0)[0]
                    pri = f.edge_P64[base:base + A].cpu().numpy()
                    pairs = [(int(a), float(pri[a])) for a in legal]
                    if node == 0 and self.add_exploration_noise:
                        noise = rs.dirichlet([self.dirichlet_noide_alpha] * len(pairs))
                        pairs = [(a, eps * z + (1 - eps) * p) for (a, p), z in zip(pairs, noise)]
                        new = np.zeros(AS, dtype=np.float64)
                        for a, p in pairs:
                            new[a] = p
                        f.edge_P64[base:base + AS] = torch.from_numpy(new).to(f.device)
                        f.edge_P[base:base + AS] = torch.from_numpy(new.astype(np.float32)).to(f.device)
                    if self.child_shuffle:
                        rs.shuffle(pairs)
                        f.set_child_order(0, node, [a for a, _ in pairs])
                    ordered.add(node)
                    f.select()             # the same descent, ties now broken in list order
            ev(f)
            f.expand_backup(prior_is_log, 0.0, 1.0, 0, value64=getattr(ev, 'value64', None),
                            prior64=getattr(ev, 'prior64', None))

    def step_with_policy(self, game_env):
        """Returns bot's policy and action at given state (deepmind_mcts.py:447-472)."""
        t1 = time.time()
        root = self.mcts_search(game_env)
        best, _ = self._forest.best_child()
        mcts_action = int(best[0])
        if self.verbose:
            seconds = time.time() - t1
            print('Finished {} sims in {:.3f} secs, {:.1f} sims/s'.format(
                root.explore_count, seconds, root.explore_count / seconds))
            print('Root:')
            print(root.to_str(game_env))
            print('Children:')
            print(root.children_str(game_env))
        legal_actions = game_env.legal_actions(game_env.current_player())
        policy = [(action, (1.0 if action == mcts_action else 0.0)) for action in legal_actions]
        return policy, mcts_action

    def step(self, game_env):
        return self.step_with_policy(game_env)[1]


class MCTSBot(Player):
    """deepmind_mcts.py:649-691: PUCT, 20 random rollouts per leaf, root noise, no solver."""

    def __init__(self, game_env, max_simulations=1000, player_id=0, player_name=''):
        super().__init__(player_id, player_name)
        evaluator = RandomRolloutEvaluator(n_rollouts=20)
        self.mcts = DeepMindMCTS(game_env, uct_c=2, max_simulations=max_simulations, evaluator=evaluator,
                                 child_selection_method='puct', add_exploration_noise=True,
                                 dirichlet_noise_alpha=1.0, dirichlet_noise_epsilon=0.25, solve=False,
                                 verbose=False)

    def get_action(self, game_env, **kwargs):
        sensible_moves = game_env.leagel_actions()
        if len(sensible_moves) > 0:
            return self.mcts.step(game_env)
        print('WARNING: the board is full')

    def __str__(self):
        return 'DeepMindMCTSBot, id: {}, name: {}.'.format(self.get_player_id(), self.get_player_name())
