"""``RolloutMCTS`` / ``RolloutPlayer`` with the reference's API (rlzero/mcts/rollout_mcts.py:10-140):
pure Monte-Carlo tree search (uniform priors, random playouts), the opponent
``TrainPipeline.policy_evaluate`` measures the trained policy against
(tools/train_alphazero.py:139-163).

Search, expansion and backup are the kernels of ``AlphaZeroMCTS``; the leaf evaluator is
``rz_eval_rollout`` (random playouts on the device, one warp per game).  The playouts draw from a
counter-based Philox stream instead of the global ``np.random`` stream of the reference (:96-100), so
moves agree with the reference in distribution, not draw by draw.  The device playouts themselves are
pinned draw for draw to a restatement (``oracle/rollout_oracle.py``): for the same ``seed`` visit
counts, value sums and the move are bit-identical to it (tests/test_gpu_rollout_parity.py).  With the
deterministic rollout modes ('first' / 'last') visit counts match the reference algorithm bit for bit.
"""
import numpy as np

from ..engine import RolloutEvaluator
from .alphazero_mcts import AlphaZeroMCTS
from .player import Player


class RolloutMCTS(AlphaZeroMCTS):

    def __init__(self, n_playout=1000, c_puct=5.0, n_limit=1000, rollout='random', seed=None, device='cuda'):
        super().__init__(self.policy_value_fn, n_playout=n_playout, c_puct=c_puct, add_noise=False,
                         device=device)
        self.n_limit = n_limit
        if seed is None:
            seed = int(np.random.randint(0, 2 ** 31 - 1))   # follows np.random.seed like the reference's playouts
        self._native_evaluator = RolloutEvaluator(n_limit=n_limit, seed=seed, mode=rollout)

    def simulate(self, game_env, temperature=1e-3):
        """``n_playout`` playouts, then the most visited root action (first maximum, :76-81)."""
        self._ensure_forest(game_env)
        self._upload(game_env)
        self._waves(self.n_playout)
        visits, _, has, _, _ = self._forest.root_stats()
        acts = np.nonzero(has[0])[0]
        if len(acts) == 0:
            raise ValueError('max() arg is an empty sequence')   # :80 on a terminal root
        return int(acts[int(np.argmax(visits[0][acts]))])

    def rollout_policy(self, game_env):
        """(:96-100) kept for API compatibility; the device playouts do not call it."""
        action_probs = np.random.rand(len(game_env.leagel_actions()))
        return zip(game_env.leagel_actions(), action_probs)

    def policy_value_fn(self, game_env):
        """uniform probabilities for pure MCTS (:102-108)."""
        legal = game_env.leagel_actions()
        return zip(legal, np.ones(len(legal)) / len(legal))

    def __str__(self):
        return 'RolloutMCTS'


class RolloutPlayer(Player):

    def __init__(self, n_playout=1000, c_puct=5, player_id=0, player_name='', rollout='random', seed=None,
                 device='cuda'):
        super().__init__(player_id, player_name)
        self.mcts = RolloutMCTS(n_playout, c_puct, rollout=rollout, seed=seed, device=device)

    def reset_player(self):
        self.mcts.update_with_move(-1)

    def get_action(self, game_env, **kwargs):
        sensible_moves = game_env.leagel_actions()
        if len(sensible_moves) > 0:
            move = self.mcts.simulate(game_env)
            self.mcts.update_with_move(-1)
            return move
        print('WARNING: the board is full')

    def __str__(self):
        return 'RolloutPlayer, id: {}, name: {}.'.format(self.get_player_id(), self.get_player_name())
