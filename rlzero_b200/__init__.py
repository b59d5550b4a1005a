"""rlzero_b200 -- B200-native batched self-play MCTS behind the RLZero API.

Product code.  The CUDA library (``librlzero_b200.so``, built by ``rlzero_b200.build``) is
mandatory: there is no CPU fallback, and nothing here imports ``oracle``.

Reference-facing modules mirror the reference's layout:
  rlzero_b200.mcts.alphazero_mcts   <-> rlzero/mcts/alphazero_mcts.py
  rlzero_b200.mcts.node             <-> rlzero/mcts/node.py
  rlzero_b200.mcts.player           <-> rlzero/mcts/player.py
  rlzero_b200.games.gomoku          <-> rlzero/games/gomoku/{gomoku_env,game}.py
Batched engine (the fast path): rlzero_b200.engine.SearchForest, rlzero_b200.selfplay, rlzero_b200.match.
"""
__version__ = '0.1.0'

from .match import BatchedMatch  # noqa: E402

__all__ = ['BatchedMatch']
