"""``BatchedMatch``: evaluation games between two search players, many at once on the GPU.

``GameControl.start_play`` (rlzero/games/gomoku/game.py:61-94) plays one game, one move at a time, each move a search
of one tree -- the fourth stage of ``TrainPipeline`` (tools/train_alphazero.py:139-163) runs that way.  Here each seat
owns a ``SearchForest`` of ``n_games`` trees, tree g of both forests is game g, and a ply is one batched search per
seat followed by one ``rz_match_commit`` launch that plays every running game's move.
"""
import ctypes as C
from collections import defaultdict

import numpy as np
import torch

from . import _lib as L
from .engine import SearchForest
from .mcts.alphazero_mcts import AlphaZeroPlayer
from .mcts.rollout_mcts import RolloutPlayer


class _Seat(object):

    def __init__(self, player, G, board_size, n_in_row, board_width, game_type, device, global_offset):
        if not isinstance(player, (RolloutPlayer, AlphaZeroPlayer)):
            raise TypeError('BatchedMatch seats are AlphaZeroPlayer or RolloutPlayer, not %r' % type(player).__name__)
        mcts = player.mcts
        if isinstance(player, RolloutPlayer):
            self.evaluator = mcts._native_evaluator
            self.sampled = False
        else:
            if player.is_selfplay:
                raise ValueError('a match seat plays evaluation moves: use AlphaZeroPlayer(is_selfplay=False)')
            self.evaluator = getattr(mcts.policy_value_fn, 'device_evaluator', None)
            if self.evaluator is None:
                raise ValueError('BatchedMatch needs a device evaluator (policy_value_fn.device_evaluator); a Python '
                                 'policy_value_fn plays through GameControl.start_play')
            if mcts.leaves_per_wave > 1:
                raise ValueError('BatchedMatch runs one leaf per tree and wave (leaves_per_wave=1)')
            self.sampled = True
        self.n_playout = int(mcts.n_playout)
        if self.n_playout < 1:
            raise ValueError('n_playout must be at least 1')
        # every move starts from a fresh tree and a playout expands at most one node: n_playout nodes suffice
        self.forest = SearchForest(G, board_size, n_in_row, n_playout=self.n_playout, c_puct=mcts._c_puct,
                                   rule=mcts.rule, max_carry=0, device=device, global_offset=global_offset,
                                   board_width=board_width, game_type=game_type)


class BatchedMatch(object):
    """``n_games`` games of ``player1`` (env player id 0) against ``player2`` (id 1), as ``start_play`` seats them.

    Seats, as the single-game classes play them:

    * ``AlphaZeroPlayer`` (not self-play; its ``policy_value_fn`` must carry a ``device_evaluator``): a fresh tree
      every move, no noise, the player's ``n_playout``, ``c_puct`` and rule, one leaf per wave.  The move is drawn
      from ``softmax(log(N + 1e-10) / 1e-3)`` by ``rz_tree_root_policy``.  The reference draws twice and plays the
      second draw (alphazero_mcts.py:157); both draws come from the same distribution, so the moves agree with it in
      distribution.
    * ``RolloutPlayer``: a fresh tree every move, the player's ``RolloutEvaluator`` (seed, ``n_limit``, mode); the
      move is the first most-visited root child (``RolloutMCTS.simulate``, rollout_mcts.py:76-81).

    Search counter and draw keys of ``play(first, seed)`` at ply p (p = 0 for the first move of every game):

    * each seat that has a mover in some game at this ply runs ``forest.search(evaluator, n_playout,
      seed=(seed << 10) | p)``: the counter ``(seed << 10) | p`` is ``rz_tree_desc.seed_dev``, so the rollout
      playouts of game g draw with the evaluator's seed plus that counter, the global id ``global_offset + g``, the
      root's visit count and the root's stone count (``rz_eval_rollout``);
    * an AlphaZero seat then runs ``root_policy(1e-3, seed=(seed << 10) | p)``: the uniform of game g is
      ``u01_53(philox4(global_offset + g, RZ_META_EPISODE (0), RZ_META_STONES, 0x5eed, (seed << 10) | p))`` and the
      move is the first action whose cumulative ``pi`` exceeds it (the last legal action if none does);
    * one ``rz_match_commit`` plays the moves, and one host read of the running-game count ends the loop.

    A game's slot never moves, so these keys depend on the game's global id only.  The network of an AlphaZero seat
    evaluates all ``n_games`` leaf slots in every wave, the waiting and finished games' stale leaves included: with
    every game started by the same seat the other seat's search is skipped for the whole ply, with mixed ``first``
    both seats search every ply.
    """

    def __init__(self, player1, player2, n_games, board_size, n_in_row, board_width=None, game_type=L.GAME_GOMOKU,
                 device='cuda', global_offset=0):
        if int(game_type) == L.GAME_GO:
            raise ValueError('BatchedMatch plays Gomoku / TicTacToe and Connect Four, not Go')
        self.G = int(n_games)
        if self.G < 1:
            raise ValueError('n_games must be at least 1')
        self.seats = [_Seat(p, self.G, board_size, n_in_row, board_width, game_type, device, global_offset)
                      for p in (player1, player2)]
        f0 = self.seats[0].forest
        self.device = f0.device
        self.lib = f0.lib
        self.max_plies = f0.cells           # a line game ends when the board is full

    def play(self, first=None, seed=0):
        """Play every game to its end.  ``first[g]`` is the env id that moves first in game g (default all 0: the
        reference's ``start_play`` always lets id 0 move first).  Returns a dict: ``winner`` [G] (env id, -1 tie),
        ``plies`` [G], ``moves`` [G, max_plies] (-1 after the game's end) numpy arrays, and ``win_cnt``, a
        ``defaultdict(int)`` keyed by winner id as ``policy_evaluate`` counts it."""
        G = self.G
        first = np.zeros(G, dtype=np.int32) if first is None else np.asarray(first, dtype=np.int32).reshape(-1)
        if first.shape != (G,) or not np.isin(first, (0, 1)).all():
            raise ValueError('first must hold n_games values, each 0 or 1')
        seed = int(seed)
        if not 0 <= seed < 2 ** 53:
            raise ValueError('seed must be in [0, 2**53)')
        fd = torch.from_numpy(first).to(self.device)
        for s, seat in enumerate(self.seats):
            f = seat.forest
            f.reset_games()
            f.root_meta[:, L.META_PLAYER] = fd
            f.root_meta[:, L.META_STATUS] = torch.where(fd == s, L.ACTIVE, L.IDLE).to(torch.int32)
        # seats with a mover at even / odd plies
        by_parity = [sorted(set((first ^ p).tolist())) for p in (0, 1)]
        move_log = torch.full((G, self.max_plies), -1, dtype=torch.int32, device=self.device)
        m0, m1 = self.seats[0].forest.root_meta, self.seats[1].forest.root_meta
        for ply in range(self.max_plies):
            counter = (seed << 10) | ply
            for s in by_parity[ply & 1]:
                seat = self.seats[s]
                seat.forest.search(seat.evaluator, seat.n_playout, seed=counter)
                if seat.sampled:
                    seat.forest.root_policy(1e-3, seed=counter)
            mv = [seat.forest.move if seat.sampled else None for seat in self.seats]
            L.check(self.lib.rz_match_commit(C.byref(self.seats[0].forest.desc), C.byref(self.seats[1].forest.desc),
                                             L.ptr(mv[0]), L.ptr(mv[1]), L.ptr(move_log), self.max_plies,
                                             L.stream_ptr()), 'rz_match_commit')
            running = ((m0[:, L.META_STATUS] == L.ACTIVE) | (m1[:, L.META_STATUS] == L.ACTIVE)).sum()
            faulty = ((m0[:, L.META_FAULT] | m1[:, L.META_FAULT]) != 0).sum()
            running, faulty = torch.stack([running, faulty]).tolist()
            if faulty:
                for seat in self.seats:
                    seat.forest.raise_faults()
            if running == 0:
                break
        else:
            raise RuntimeError('games still running after %d plies' % self.max_plies)
        meta = m0.cpu().numpy()
        winner = meta[:, L.META_WINNER].copy()
        win_cnt = defaultdict(int)
        for w in winner.tolist():
            win_cnt[w] += 1
        return dict(winner=winner, plies=meta[:, L.META_PLY].copy(), moves=move_log.cpu().numpy(), win_cnt=win_cnt)
