"""Batched self-play: G games searched and played concurrently on one GPU.

This is ``GameControl.start_self_play`` + ``AlphaZeroPlayer.get_action`` + ``AlphaZeroMCTS``
(rlzero/games/gomoku/game.py:96-134, rlzero/mcts/alphazero_mcts.py:73-165) for thousands of
games at once, entirely on the device:

    per wave  : rz_tree_select -> rz_net_stem_tc (encoder + first conv) -> 20 x rz_net_conv3x3_tc2 (the last
                with the heads' 1x1 convolutions) -> rz_net_heads_tc -> rz_tree_expand_backup
                                                                  (one CUDA graph, replayed)
    per move  : rz_tree_root_policy (pi, sampled move) -> rz_tree_advance (record ply, play the
                move, re-root with the kept subtree, finish episode -> z -> ring, restart slot)

Games are independent, so a multi-GPU job is one ``BatchedSelfPlay`` per rank with
``global_offset = rank * n_games`` and no communication on this path; per-game random streams
are keyed by the global game id, so results do not depend on how games are sharded.
"""
import numpy as np
import torch

from . import _lib as L
from .engine import SearchForest, capture_graph
from .games.gomoku.policy_value_net import NativeForward


class BatchedSelfPlay(object):

    def __init__(self, n_games, board_size=15, n_in_row=5, net=None, n_playout=800, c_puct=5.0,
                 rule=L.RULE_UCT, temperature=1.0, add_noise=True, noise_eps=0.25, noise_alpha=0.3,
                 device='cuda', global_offset=0, seed=0, evaluator=None, ring_capacity=None,
                 store_priors=True, n_ctas=0, board_width=None, game_type=L.GAME_GOMOKU, komi=7.5, max_moves=0,
                 leaves_per_tree=1, virtual_loss=1.0, net_mode=None):
        """``leaves_per_tree = K > 1``: leaf-parallel waves with virtual loss (``SearchForest``): a move is
        ``1 + ceil((n_playout - 1) / K)`` waves of up to K playouts per game and the network sees G*K leaves per
        wave -- for batches too small to fill the GPU.  Not the reference's sequential search order; 1 = parity mode.

        ``game_type = L.GAME_GO``: ``n_in_row`` is ignored, actions are the squares + the pass,
        ``komi`` as GoEnv's, ``max_moves`` > 0 ends and scores a game after that many moves (the
        reference has no cap; AlphaGo Zero used 2 * 19 * 19)."""
        self.G = int(n_games)
        self.n_playout = int(n_playout)
        self.temperature = float(temperature)
        self.noise_eps = float(noise_eps) if add_noise else 0.0
        self.noise_alpha = float(noise_alpha)
        self.seed = int(seed)
        self.forest = SearchForest(self.G, board_size, n_in_row, n_playout=n_playout, c_puct=c_puct,
                                   rule=rule, device=device, global_offset=global_offset,
                                   with_trajectories=True, ring_capacity=ring_capacity,
                                   store_priors=store_priors, board_width=board_width, game_type=game_type,
                                   komi=komi, max_moves=max_moves, leaves_per_tree=leaves_per_tree,
                                   virtual_loss=virtual_loss)
        self.K = self.forest.K
        self.waves_per_move = self.n_playout if self.K == 1 else 1 + (max(self.n_playout - 1, 0) + self.K - 1) // self.K
        if evaluator is None:
            if net is None:
                raise ValueError('BatchedSelfPlay needs a policy-value module (net=) or an evaluator')
            # net_mode: NativeForward's mode ('tc' runs the stock PolicyValueNet zero-padded on the tensor cores)
            evaluator = NativeForward(net, max_batch=self.forest.n_leaves, device=device, n_ctas=n_ctas,
                                      game_type=game_type, mode=net_mode)
        self.evaluator = evaluator
        self._arm_budget()
        self.waves_in_move = 0
        self.moves_played = 0
        self._graph = None
        self._graph8 = None           # eight waves per launch (small batches: a wave is shorter than a graph launch)
        self._graph_version = getattr(evaluator, 'weights_version', 0)
        self._pinned = None

    def _arm_budget(self):
        """Leaf-parallel mode: every tree takes exactly n_playout more playouts (rz_tree_desc.target_N)."""
        if self.K > 1:
            torch.add(self.forest.root_N, self.n_playout, out=self.forest.target_N)

    # ------------------------------------------------------------------ set-up
    def set_random_start_positions(self, global_ids=None, max_random_moves=31):
        """Game g starts after k_g = (1000+g) mod 31 uniformly random moves drawn with
        RandomState(1000+g) (SURVEY.md 8d); positions that happen to be over restart empty."""
        f = self.forest
        ids = np.arange(self.G) + int(f.desc.global_offset) if global_ids is None else np.asarray(global_ids)
        if f.is_go:
            return self._set_random_go_positions(ids, max_random_moves)
        lists = []
        for gid in ids:
            rs = np.random.RandomState(1000 + int(gid))
            k = (1000 + int(gid)) % max_random_moves
            if f.game_type == L.GAME_CONNECT4:
                # k random drops; a column is used at most H times
                seq = np.repeat(np.arange(f.W), f.H)
                lists.append(rs.permutation(seq)[:min(k, f.cells - 1)].tolist())
            else:
                lists.append(rs.permutation(f.A)[:k].tolist())
        f.set_positions(lists)
        import ctypes as C
        L.check(f.lib.rz_gomoku_reset(C.byref(f.gdesc), L.ptr(f.root_rows), L.ptr(f.root_meta), f.G, 1,
                                      L.stream_ptr()), 'rz_gomoku_reset')
        f.root_meta[:, L.META_EPISODE] = 0
        self.waves_in_move = 0
        self._arm_budget()

    def _set_random_go_positions(self, ids, max_random_moves):
        """Go: the same recipe, but a random square may be illegal (suicide / ko), so the moves are
        played ply by ply against the device's legal mask: game g plays, k_g times, the first legal
        square of its RandomState(1000+g) permutation that it has not tried yet."""
        import ctypes as C
        f = self.forest
        f.reset_games()
        perms = [np.random.RandomState(1000 + int(gid)).permutation(f.cells) for gid in ids]
        ks = [(1000 + int(gid)) % max_random_moves for gid in ids]
        ptr = np.zeros(f.G, dtype=np.int64)
        mask = torch.zeros(f.G, f.A, dtype=torch.uint8, device=f.device)
        for t in range(max(ks, default=0)):
            L.check(f.lib.rz_go_legal_mask(C.byref(f.gdesc), L.ptr(f.root_rows), L.ptr(f.root_meta), L.ptr(mask),
                                           f.G, L.stream_ptr()), 'rz_go_legal_mask')
            m = mask.cpu().numpy()
            acts = np.full(f.G, -1, dtype=np.int32)
            for g in range(f.G):
                if ks[g] <= t:
                    continue
                while ptr[g] < f.cells and not m[g, perms[g][ptr[g]]]:
                    ptr[g] += 1
                if ptr[g] < f.cells:
                    acts[g] = perms[g][ptr[g]]
                    ptr[g] += 1
            f.play_moves(acts)
        f.root_meta[:, L.META_PLY] = 0
        f.root_meta[:, L.META_EPISODE] = 0
        f.raise_faults()
        self.waves_in_move = 0
        self._arm_budget()

    # -------------------------------------------------------------------- waves
    def _wave(self):
        f = self.forest
        f.select()
        self.evaluator(f)
        f.expand_backup(bool(getattr(self.evaluator, 'prior_is_log', False)), self.noise_eps,
                        self.noise_alpha, self.seed)

    def kernels_per_wave(self):
        # select + evaluator kernels + expand/backup
        kpf = getattr(self.evaluator, 'kernels_per_forward', None)
        if kpf is None:
            return 3
        try:
            return 1 + kpf(self.forest.n_leaves) + 1
        except TypeError:
            return 1 + kpf() + 1

    def warm_up(self):
        """One eager wave (lazy attribute set-up) and capture of the wave graph."""
        if self._graph is not None:
            return
        self._wave()
        torch.cuda.synchronize()
        if getattr(self.evaluator, 'graph_capturable', False):
            g = torch.cuda.CUDAGraph()
            with capture_graph(g):
                self._wave()
            self._graph = g
        self.waves_in_move += 1

    def _check_weights(self):
        """A captured wave holds the weight pointers by value: re-capture after refresh_weights()."""
        v = getattr(self.evaluator, 'weights_version', 0)
        if self._graph is not None and v != self._graph_version:
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with capture_graph(g):
                self._wave()
            self._graph = g
            self._graph8 = None
        self._graph_version = v

    def step_wave(self):
        """One playout for every game; commits the move when ``n_playout`` waves are done."""
        self._check_weights()
        if self._graph is not None:
            self._graph.replay()
        else:
            self._wave()
        self.waves_in_move += 1
        if self.waves_in_move >= self.waves_per_move:
            self.commit_move()

    def step_waves(self, n):
        """``n`` waves; with a captured graph, eight waves share a launch while they do not cross a move commit.  For a
        handful of games a wave (40 .. 130 us of GPU time) is about as long as the host needs for one graph launch."""
        n = int(n)
        while n > 0:
            k = min(n, self.waves_per_move - self.waves_in_move)
            if self._graph is None or k < 8 or self.forest.n_leaves > 512:      # (long waves: nothing to gain)
                self.step_wave()
                n -= 1
                continue
            self._check_weights()
            if self._graph8 is None:
                torch.cuda.synchronize()
                g8 = torch.cuda.CUDAGraph()
                with capture_graph(g8):
                    for _ in range(8):
                        self._wave()
                self._graph8 = g8
            for _ in range(k // 8):
                self._graph8.replay()
            done = (k // 8) * 8
            self.waves_in_move += done
            n -= done
            if self.waves_in_move >= self.waves_per_move:
                self.commit_move()

    def commit_move(self):
        """pi + sampled move on the device, play it, re-root, record, refill finished games."""
        f = self.forest
        f.root_policy(self.temperature, seed=self.seed + 0x9E37)
        f.advance(keep_subtree=True, record=True, auto_reset=True)
        self.waves_in_move = 0
        self.moves_played += 1
        self._arm_budget()

    def play(self, n_moves):
        self.warm_up()
        self.step_waves(n_moves * self.waves_per_move)

    # ------------------------------------------------- host-buffer API (end to end)
    def get_actions(self, rows_host, meta_host, temperature=None, hist_host=None):
        """Batched ``AlphaZeroPlayer.get_action(env, temperature, return_prob=True)`` with HOST
        buffers: positions come from pinned host memory, the search runs ``n_playout`` playouts
        per game from fresh trees, and (moves [G], pi [G,A], visits [G,A]) come back to the host.
        ``rows_host``: uint32/int32 [G,2,H]; ``meta_host``: int32 [G,RZ_META_STRIDE]; Go also takes
        ``hist_host`` [G,14,H], the history planes (include/rlzero_b200.h)."""
        f = self.forest
        if self._pinned is None:
            self._pinned = dict(
                rows=torch.empty(f.G, 2, f.H, dtype=torch.int32).pin_memory(),
                meta=torch.empty(f.G, L.META_STRIDE, dtype=torch.int32).pin_memory(),
                move=torch.empty(f.G, dtype=torch.int32).pin_memory(),
                pi=torch.empty(f.G, f.AS, dtype=torch.float32).pin_memory(),
                visits=torch.empty(f.G, f.AS, dtype=torch.int32).pin_memory())
        p = self._pinned
        if f.is_go:
            if hist_host is None:
                raise ValueError('Go positions need their history planes (hist_host=)')
            if 'hist' not in p:
                p['hist'] = torch.empty(f.G, L.GO_HIST, f.H, dtype=torch.int32).pin_memory()
            p['hist'].copy_(torch.as_tensor(np.asarray(hist_host).view(np.int32)))
            f.root_hist.copy_(p['hist'], non_blocking=True)
        p['rows'].copy_(torch.as_tensor(np.asarray(rows_host).view(np.int32)))
        p['meta'].copy_(torch.as_tensor(np.asarray(meta_host)))
        f.root_rows.copy_(p['rows'], non_blocking=True)
        f.root_meta.copy_(p['meta'], non_blocking=True)
        f.reset_trees()
        self.warm_up_for_api()
        self._check_weights()
        self._arm_budget()
        for _ in range(self.waves_per_move):
            if self._graph is not None:
                self._graph.replay()
            else:
                self._wave()
        f.root_policy(self.temperature if temperature is None else temperature, seed=self.seed + 0x9E37)
        p['move'].copy_(f.move, non_blocking=True)
        p['pi'].copy_(f.pi, non_blocking=True)
        p['visits'].copy_(f.visits, non_blocking=True)
        torch.cuda.synchronize()
        f.raise_faults()
        A = f.A
        return p['move'].numpy().copy(), p['pi'].numpy()[:, :A].copy(), p['visits'].numpy()[:, :A].copy()

    def warm_up_for_api(self):
        if self._graph is None and getattr(self.evaluator, 'graph_capturable', False):
            # capture without disturbing the trees: run the eager warm-up wave, then reset
            f = self.forest
            self._wave()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with capture_graph(g):
                self._wave()
            self._graph = g
            f.reset_trees()

    def api_bytes(self):
        f = self.forest
        h2d = f.G * ((2 + (L.GO_HIST if f.is_go else 0)) * f.H * 4 + L.META_STRIDE * 4)
        d2h = f.G * (4 + f.AS * 4 + f.AS * 4)
        return h2d, d2h

    # ------------------------------------------------------------------- output
    def stats(self):
        t = self.forest.traj
        return dict(games_done=int(t['games_done'].item()), plies_done=int(t['plies_done'].item()),
                    moves_played=self.moves_played)

    def drain(self):
        """Finished episodes as training tuples in the reference's format (game.py:113-134):
        states float32 [n,4,H,W] (current_state planes), pis float32 [n,A], z float32 [n]."""
        f = self.forest
        out = f.drain_trajectories()
        rows, info = out['rows'], out['info']
        n, H, W = len(info), f.H, f.W
        if f.is_go:
            return self._go_states(rows, info), out['pi'], info[:, 2].astype(np.float32), info
        states = np.zeros((n, 4, H, W), dtype=np.float32)
        if n:
            bits = ((rows[:, :, :, None] >> np.arange(W, dtype=np.uint32)[None, None, None, :]) & 1).astype(np.float32)
            mover = info[:, 0]
            idx = np.arange(n)
            states[:, 0] = bits[idx, mover]
            states[:, 1] = bits[idx, 1 - mover]
            last = info[:, 1]
            has_last = last >= 0
            states[idx[has_last], 2, last[has_last] // W, last[has_last] % W] = 1.0
            stones = bits.sum(axis=(1, 2, 3)).astype(np.int64)
            states[stones % 2 == 0, 3] = 1.0
        return states, out['pi'], info[:, 2].astype(np.float32), info

    def _go_states(self, rows, info):
        """GoEnv.observe planes [n,17,H,W] (go_env.py:156-178) of the drained plies.  The trajectory
        keeps (black, white) per ply; the 8-position history is rebuilt from the preceding plies of the
        same episode, which the ring stores consecutively: entry e of ply j is the position before ply
        j-e as (stones of its last mover, stones of the player to move), zero for j-e < 1.  Exact for
        episodes recorded from the empty board (self-play); an episode that started from a set-up
        position, or whose first plies were overwritten in the ring, lacks the older entries."""
        f = self.forest
        n, H, W = len(info), f.H, f.W
        states = np.zeros((n, 17, H, W), dtype=np.float32)
        if n == 0:
            return states
        bits = ((rows[:, :, :, None] >> np.arange(W, dtype=np.uint32)[None, None, None, :]) & 1).astype(np.float32)
        mover, slot, episode, ply = info[:, 0], info[:, 3], info[:, 4], info[:, 5]
        idx = np.arange(n)
        for e in range(8):
            src = idx - e
            ok = (src >= 0)
            srcc = np.where(ok, src, 0)
            ok &= (slot[srcc] == slot) & (episode[srcc] == episode) & (ply[srcc] == ply - e) & (ply[srcc] >= 1)
            t = idx[ok]
            s_ = srcc[ok]
            states[t, 2 * e] = bits[s_, 1 - mover[s_]]
            states[t, 2 * e + 1] = bits[s_, mover[s_]]
        states[mover == 1, 16] = 1.0
        return states
