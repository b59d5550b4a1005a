"""Host side of the batched search: structure-of-arrays node pools in HBM + the wave loop.

``SearchForest`` owns G search trees (one per game) as flat torch CUDA tensors and drives
the C-ABI kernels of ``include/rlzero_b200.h``.  One *wave* = one playout for every tree:

    rz_tree_select  ->  evaluator (net forward / closed form / host callback)
                    ->  rz_tree_expand_backup

which is exactly ``AlphaZeroMCTS._playout`` (rlzero/mcts/alphazero_mcts.py:42-71) for every
game at once; ``n_playout`` waves are ``AlphaZeroMCTS.simulate`` (:73-94).  Because each tree
advances by one playout per wave, the per-tree order of updates is the reference's, and visit
counts / value sums are bit-identical to it.

PyTorch is used for device memory, streams and CUDA graphs only.
"""
import ctypes as C
import math
import os

import numpy as np
import torch

from . import _lib as L


class capture_graph:
    """``with capture_graph(g): ...`` = ``torch.cuda.graph(g)`` made safe against Python's garbage collector: a dead
    object that owns a ``CUDAGraph`` (an earlier forest and its closures form reference cycles) must not be destroyed
    WHILE a capture is under way -- freeing a graph is an operation the capturing stream does not permit, and it
    invalidates the capture.  This torch version no longer collects garbage when a capture starts, so: collect first,
    keep the collector off until the capture has ended."""

    def __init__(self, g, **kw):
        self.ctx = torch.cuda.graph(g, **kw)

    def __enter__(self):
        import gc
        gc.collect()
        self.gc_was_on = gc.isenabled()
        gc.disable()
        try:
            return self.ctx.__enter__()
        except BaseException:
            if self.gc_was_on:
                gc.enable()
            raise

    def __exit__(self, *exc):
        import gc
        try:
            return self.ctx.__exit__(*exc)
        finally:
            if self.gc_was_on:
                gc.enable()


def _round_up(x, m):
    return (x + m - 1) // m * m


_LN_CACHE = {}


def ln_table(n):
    """ln_table[k] = math.log(k): CPython's libm log, the function node.py:84 calls.  numpy's
    vectorised log may differ in the last bit, so the table is built with math.log."""
    if n not in _LN_CACHE:
        t = np.zeros(n, dtype=np.float64)
        for k in range(1, n):
            t[k] = math.log(k)
        _LN_CACHE[n] = t
    return _LN_CACHE[n]


class SearchForest(object):
    """G independent search trees + their root positions, resident in HBM."""

    def __init__(self, n_trees, board_size, n_in_row, n_playout=800, c_puct=5.0,
                 rule=L.RULE_UCT, max_carry=None, max_nodes=None, store_priors=True,
                 device='cuda', global_offset=0, ln_table_len=None, with_trajectories=False,
                 ring_capacity=None, board_width=None, game_type=L.GAME_GOMOKU, komi=7.5, max_moves=0,
                 flavour=L.FLAVOUR_ALPHAZERO, solve=False, returns_mode=L.RETURNS_REFERENCE,
                 noise_root_only=False, leaves_per_tree=1, virtual_loss=1.0, prior_f64=False,
                 child_shuffle=None):
        """``leaves_per_tree = K > 1`` switches to leaf-parallel waves with virtual loss (opt-in; not the
        reference's sequential order, see ``rz_tree_desc.leaves_per_tree``): every wave runs up to K playouts per
        tree and the evaluator sees ``n_leaves = G*K`` positions -- for a handful of games (the single-game API)
        this is what fills the network batch.  ``K = 1`` is the parity mode.

        ``prior_f64``: keep the priors in float64 as well (``rz_tree_desc.edge_P64``): ``TreeNode.prior`` is a Python
        float, and with Dirichlet noise the reference forms it in float64 (node.py:66-69), so the PUCT rule is only
        bit-exact under noise with this pool.  ``child_shuffle`` (DeepMindMCTS flavour): ``'random'`` = the children of
        every new node in a counter-based random order, ``'host'`` = the host writes numpy's permutation
        (``set_child_order``), ``None`` = unshuffled, ties to the lowest action (deepmind_mcts.py:508).

        ``flavour = L.FLAVOUR_DEEPMIND`` runs the reference's second search driver, DeepMindMCTS
        (rlzero/mcts/deepmind_mcts.py:384-646): returns vectors, outcome shortcut, terminal outcomes,
        ``solve`` (MCTS-Solver), root-only noise, early stop on a proven root."""
        if not torch.cuda.is_available():
            raise L.NativeLibraryError('rlzero_b200 needs a CUDA device (no CPU fallback)')
        self.lib = L.load()
        self.device = torch.device(device)
        self.G = int(n_trees)
        self.K = max(1, int(leaves_per_tree))
        self.n_leaves = self.G * self.K
        self.virtual_loss = float(virtual_loss)
        if self.K > 1 and int(flavour) != L.FLAVOUR_ALPHAZERO:
            raise ValueError('leaf-parallel waves (leaves_per_tree > 1) need the AlphaZero flavour')
        self.H = int(board_size)
        self.W = self.H if board_width is None else int(board_width)
        self.k = int(n_in_row)
        self.game_type = int(game_type)
        if not (1 <= self.H <= L.MAX_BOARD and 1 <= self.W <= L.MAX_BOARD):
            raise ValueError('board_size must be in [1, %d]' % L.MAX_BOARD)
        if max(self.H, self.W) < self.k:
            raise ValueError('Board board_size can not less than %d' % self.k)  # gomoku_env.py:35
        self.cells = self.H * self.W
        self.is_go = self.game_type == L.GAME_GO
        self.komi = float(komi) if self.is_go else 0.0
        self.max_moves = int(max_moves) if self.is_go else 0
        if self.is_go and self.W != self.H:
            raise ValueError('Go needs a square board')
        # actions: squares; the columns for Connect Four; squares + the pass for Go (go_env.py:74-77)
        self.A = self.W if self.game_type == L.GAME_CONNECT4 else self.cells + int(self.is_go)
        self.AS = _round_up(self.A, 32)
        self.n_playout = int(n_playout)
        self.c_puct = float(c_puct)
        self.rule = int(rule)
        if max_carry is None:
            # nodes of the chosen child's subtree that update_with_move keeps (alphazero_mcts.py:96-103).  Under
            # UCB1 with c = 5 the visits of a 15x15 search are spread almost evenly, so the kept subtree is a handful
            # of nodes and 64 bounds the pool (20 B x AS per node x thousands of games); small boards concentrate
            # them (a 4x4 / 400-playout search carries 70 nodes), and their blocks are small: carry everything
            max_carry = self.n_playout if (rule != L.RULE_UCT or self.AS <= 64) else 64
        self.max_carry = int(max_carry)
        self.max_nodes = int(max_nodes) if max_nodes else self.n_playout + self.max_carry
        if self.max_nodes > 6144:
            raise ValueError('max_nodes %d > 6144 (re-root bitmap lives in shared memory)' % self.max_nodes)
        # a path holds at most one edge per stone (line games) / per expanded node (Go: captures free squares)
        self.max_depth = self.max_nodes + 1 if self.is_go else self.cells + 1
        self.store_priors = bool(store_priors) or rule == L.RULE_PUCT
        G, AS, H, dev = self.G, self.AS, self.H, self.device
        i32, f64, f32 = torch.int32, torch.float64, torch.float32
        n_edges = G * self.max_nodes * AS
        self.edge_N = torch.empty(n_edges, dtype=i32, device=dev)
        self.edge_W = torch.empty(n_edges, dtype=f64, device=dev)
        self.edge_child = torch.empty(n_edges, dtype=i32, device=dev)
        self.edge_P = torch.empty(n_edges, dtype=f32, device=dev) if self.store_priors else None
        self.edge_P64 = torch.empty(n_edges, dtype=f64, device=dev) if (prior_f64 and self.store_priors) else None
        # search counter the captured wave graph reads (rz_tree_desc.seed_dev): bumped per search instead of
        # re-capturing the graph with a new by-value seed
        self.seed_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self.carry_dropped = 0       # re-roots whose kept subtree exceeded max_carry (tree restarted instead)
        self.node_parent = torch.empty(G * self.max_nodes, dtype=i32, device=dev)
        self.node_paction = torch.empty(G * self.max_nodes, dtype=i32, device=dev)
        self.n_nodes = torch.zeros(G, dtype=i32, device=dev)
        self.root_N = torch.zeros(G, dtype=i32, device=dev)
        self.root_W = torch.zeros(G, dtype=f64, device=dev)
        self.root_rows = torch.zeros(G, 2, H, dtype=i32, device=dev)
        self.root_meta = torch.zeros(G, L.META_STRIDE, dtype=i32, device=dev)
        NL = self.n_leaves      # wave slots: one per tree, or K per tree in leaf-parallel mode
        self.path_node = torch.zeros(NL, self.max_depth, dtype=i32, device=dev)
        self.path_action = torch.zeros(NL, self.max_depth, dtype=i32, device=dev)
        self.depth = torch.full((NL,), -1, dtype=i32, device=dev)
        self.leaf_rows = torch.zeros(NL, 2, H, dtype=i32, device=dev)
        self.leaf_meta = torch.zeros(NL, L.META_STRIDE, dtype=i32, device=dev)
        self.vl_saved_W = torch.zeros(NL * self.max_depth, dtype=f64, device=dev) if self.K > 1 else None
        self.target_N = torch.full((G,), 2 ** 31 - 1, dtype=i32, device=dev) if self.K > 1 else None
        # Go: board_history planes 2..15 of every root / leaf position (go_env.py:174-178)
        self.root_hist = torch.zeros(G, L.GO_HIST, H, dtype=i32, device=dev) if self.is_go else None
        self.leaf_hist = torch.zeros(NL, L.GO_HIST, H, dtype=i32, device=dev) if self.is_go else None
        self.flavour = int(flavour)
        self.is_dm = self.flavour == L.FLAVOUR_DEEPMIND
        self.edge_O = torch.zeros(n_edges, dtype=i32, device=dev) if self.is_dm else None
        self.root_O = torch.zeros(G, dtype=i32, device=dev) if self.is_dm else None
        self.best = torch.full((G,), -1, dtype=i32, device=dev) if self.is_dm else None
        if child_shuffle not in (None, 'random', 'host'):
            raise ValueError("child_shuffle must be None, 'random' or 'host'")
        if child_shuffle and not self.is_dm:
            raise ValueError('the child shuffle belongs to the DeepMindMCTS flavour')
        self.child_shuffle = child_shuffle
        self.edge_R = torch.zeros(n_edges, dtype=i32, device=dev) if child_shuffle else None
        n_ln = int(ln_table_len) if ln_table_len else max(1 << 16, 4 * self.n_playout + 2)
        self.ln_table = torch.from_numpy(ln_table(n_ln)).to(dev)
        # evaluator outputs for one wave
        self.prior = torch.zeros(NL, AS, dtype=f32, device=dev)
        self.value = torch.zeros(NL, dtype=f32, device=dev)
        # root policy outputs
        self.visits = torch.zeros(G, AS, dtype=i32, device=dev)
        self.pi = torch.zeros(G, AS, dtype=f32, device=dev)
        self.move = torch.full((G,), -1, dtype=i32, device=dev)

        self.gdesc = L.GameDesc(self.H, self.k, self.A, self.AS, self.W, self.game_type, self.komi, self.max_moves)
        d = L.TreeDesc()
        d.game = self.gdesc
        d.n_trees, d.max_nodes, d.max_depth = G, self.max_nodes, self.max_depth
        d.rule, d.ln_table_len, d.store_priors = self.rule, n_ln, int(self.store_priors)
        d.c_puct = self.c_puct
        d.global_offset = int(global_offset)
        for name in ('edge_N', 'edge_W', 'edge_child', 'node_parent', 'node_paction', 'n_nodes',
                     'root_N', 'root_W', 'root_rows', 'root_meta', 'path_node', 'path_action',
                     'depth', 'leaf_rows', 'leaf_meta', 'ln_table'):
            setattr(d, name, getattr(self, name).data_ptr())
        d.edge_P = self.edge_P.data_ptr() if self.edge_P is not None else None
        d.root_hist = self.root_hist.data_ptr() if self.is_go else None
        d.leaf_hist = self.leaf_hist.data_ptr() if self.is_go else None
        d.flavour, d.solve, d.returns_mode = self.flavour, int(bool(solve)), int(returns_mode)
        d.noise_root_only = int(bool(noise_root_only))
        d.edge_O = self.edge_O.data_ptr() if self.is_dm else None
        d.root_O = self.root_O.data_ptr() if self.is_dm else None
        d.leaves_per_tree = self.K
        d.target_N = self.target_N.data_ptr() if self.K > 1 else None
        d.vl_saved_W = self.vl_saved_W.data_ptr() if self.K > 1 else None
        d.virtual_loss = self.virtual_loss
        d.edge_P64 = self.edge_P64.data_ptr() if self.edge_P64 is not None else None
        d.seed_dev = self.seed_dev.data_ptr()
        d.edge_R = self.edge_R.data_ptr() if self.edge_R is not None else None
        d.shuffle_mode = 1 if child_shuffle == 'random' else 0
        self.desc = d
        self.traj = None
        self.tdesc = None
        if with_trajectories:
            self._alloc_trajectories(ring_capacity)
        self.reset_games()

    # ------------------------------------------------------------------ memory
    def _alloc_trajectories(self, ring_capacity):
        G, H, AS, dev = self.G, self.H, self.AS, self.device
        # plies one episode can hold: a line game fills the board; Go is capped by max_moves (or 2 * squares)
        P = (self.max_moves or 2 * self.cells) if self.is_go else self.cells
        cap = int(ring_capacity) if ring_capacity else max(4 * P, 2 * G * 16)
        cap = max(cap, P)
        i32, f32 = torch.int32, torch.float32
        self.traj = dict(
            stage_rows=torch.zeros(G, P, 2, H, dtype=i32, device=dev),
            stage_info=torch.zeros(G, P, 4, dtype=i32, device=dev),
            stage_pi=torch.zeros(G, P, AS, dtype=f32, device=dev),
            ring_rows=torch.zeros(cap, 2, H, dtype=i32, device=dev),
            ring_info=torch.zeros(cap, 6, dtype=i32, device=dev),
            ring_pi=torch.zeros(cap, AS, dtype=f32, device=dev),
            ring_cursor=torch.zeros(1, dtype=torch.int64, device=dev),
            games_done=torch.zeros(1, dtype=torch.int64, device=dev),
            plies_done=torch.zeros(1, dtype=torch.int64, device=dev))
        td = L.TrajDesc()
        td.max_plies, td.ring_capacity = P, cap
        for k, v in self.traj.items():
            setattr(td, k, v.data_ptr())
        self.tdesc = td
        self.ring_capacity = cap
        self._ring_read = 0

    def hbm_bytes(self):
        tot = 0
        for v in vars(self).values():
            if isinstance(v, torch.Tensor):
                tot += v.numel() * v.element_size()
        if self.traj:
            tot += sum(v.numel() * v.element_size() for v in self.traj.values())
        return tot

    # --------------------------------------------------------------- positions
    def _s(self):
        return L.stream_ptr()

    def reset_games(self):
        """GomokuEnv.reset() for every game + fresh trees (gomoku_env.py:33-47)."""
        if self.is_go:
            L.check(self.lib.rz_go_reset(C.byref(self.gdesc), L.ptr(self.root_rows), L.ptr(self.root_hist),
                                         L.ptr(self.root_meta), self.G, 0, self._s()), 'rz_go_reset')
        else:
            L.check(self.lib.rz_gomoku_reset(C.byref(self.gdesc), L.ptr(self.root_rows),
                                             L.ptr(self.root_meta), self.G, 0, self._s()), 'rz_gomoku_reset')
        self.reset_trees()

    def reset_trees(self, mask=None):
        m = None
        if mask is not None:
            m = torch.as_tensor(mask, dtype=torch.uint8, device=self.device).contiguous()
        L.check(self.lib.rz_tree_reset(C.byref(self.desc), L.ptr(m), self._s()), 'rz_tree_reset')

    def play_moves(self, actions):
        """env.step for every game (actions[g] < 0 skips); roots only, trees untouched."""
        a = torch.as_tensor(actions, dtype=torch.int32, device=self.device).contiguous()
        if self.is_go:
            L.check(self.lib.rz_go_step(C.byref(self.gdesc), L.ptr(self.root_rows), L.ptr(self.root_hist),
                                        L.ptr(self.root_meta), L.ptr(a), None, None, self.G, self._s()), 'rz_go_step')
            return
        L.check(self.lib.rz_gomoku_step(C.byref(self.gdesc), L.ptr(self.root_rows), L.ptr(self.root_meta),
                                        L.ptr(a), None, None, self.G, self._s()), 'rz_gomoku_step')

    def set_positions(self, move_lists):
        """Start every game from the position reached by its move list (legal, non-terminal)."""
        self.reset_games()
        longest = max((len(m) for m in move_lists), default=0)
        for t in range(longest):
            self.play_moves([m[t] if t < len(m) else -1 for m in move_lists])
        self.root_meta[:, L.META_PLY] = 0
        self.raise_faults()

    # -------------------------------------------------------------------- wave
    def select(self):
        L.check(self.lib.rz_tree_select(C.byref(self.desc), self._s()), 'rz_tree_select')

    def expand_backup(self, prior_is_log=False, noise_eps=0.0, noise_alpha=0.3, seed=0,
                      prior=None, value=None, value64=None, noise64=None, prior64=None):
        """``noise64`` / ``prior64`` (float64 [n_leaves][AS] device tensors): host-supplied Dirichlet noise / finished
        float64 priors of the new nodes (rz_tree_expand_backup_ex), the seeded-parity inputs."""
        prior = self.prior if prior is None else prior
        value = self.value if value is None else value
        if noise64 is not None or prior64 is not None:
            L.check(self.lib.rz_tree_expand_backup_ex(C.byref(self.desc), L.ptr(prior), int(prior_is_log),
                                                      L.ptr(value), L.ptr(value64), float(noise_eps),
                                                      float(noise_alpha), int(seed), L.ptr(noise64), L.ptr(prior64),
                                                      self._s()), 'rz_tree_expand_backup_ex')
            return
        if self.is_dm:      # value64 is then the evaluator's returns vector, float64 [G][2]
            L.check(self.lib.rz_tree_expand_backup_dm(C.byref(self.desc), L.ptr(prior), int(prior_is_log),
                                                      L.ptr(value), L.ptr(value64), float(noise_eps),
                                                      float(noise_alpha), int(seed), self._s()),
                    'rz_tree_expand_backup_dm')
            return
        L.check(self.lib.rz_tree_expand_backup(C.byref(self.desc), L.ptr(prior), int(prior_is_log),
                                               L.ptr(value), L.ptr(value64), float(noise_eps),
                                               float(noise_alpha), int(seed), self._s()),
                'rz_tree_expand_backup')

    def expand_backup_select(self, prior_is_log=False, noise_eps=0.0, noise_alpha=0.3, seed=0, value64=None):
        """expand_backup of this wave and select of the next one in one launch (one leaf per tree and wave)."""
        L.check(self.lib.rz_tree_expand_backup_select(C.byref(self.desc), L.ptr(self.prior), int(prior_is_log),
                                                      L.ptr(self.value), L.ptr(value64), float(noise_eps),
                                                      float(noise_alpha), int(seed), self._s()),
                'rz_tree_expand_backup_select')

    def eval_closed_form(self, eval_id):
        L.check(self.lib.rz_eval_closed_form(C.byref(self.desc), int(eval_id), L.ptr(self.prior),
                                             L.ptr(self.value), self._s()), 'rz_eval_closed_form')

    def root_policy(self, temperature=1e-3, u01=None, seed=0, want_move=True):
        u = None
        if u01 is not None:
            u = torch.as_tensor(u01, dtype=torch.float64, device=self.device).contiguous()
        L.check(self.lib.rz_tree_root_policy(C.byref(self.desc), float(temperature), L.ptr(self.visits),
                                             L.ptr(self.pi), L.ptr(self.move) if want_move else None,
                                             L.ptr(u), int(seed), self._s()), 'rz_tree_root_policy')

    def best_child(self):
        """SearchNode.best_child of every root (deepmind_mcts.py:153-175) -> (action [G], root outcome
        code [G]) host arrays; DeepMindMCTS flavour only."""
        if not self.is_dm:
            raise RuntimeError('best_child() belongs to the DeepMindMCTS flavour')
        oc = torch.zeros(self.G, dtype=torch.int32, device=self.device)
        L.check(self.lib.rz_tree_best_child(C.byref(self.desc), L.ptr(self.best), L.ptr(oc), self._s()),
                'rz_tree_best_child')
        return self.best.cpu().numpy(), oc.cpu().numpy()

    def advance(self, moves=None, keep_subtree=True, record=False, auto_reset=False):
        """env.step(move) on the roots + update_with_move (alphazero_mcts.py:96-103)."""
        mv = self.move if moves is None else torch.as_tensor(
            moves, dtype=torch.int32, device=self.device).contiguous()
        td = C.byref(self.tdesc) if (record and self.tdesc is not None) else None
        L.check(self.lib.rz_tree_advance(C.byref(self.desc), L.ptr(mv), int(keep_subtree),
                                         self.max_carry, td, L.ptr(self.pi) if record else None,
                                         int(auto_reset), self._s()), 'rz_tree_advance')

    # ------------------------------------------------------------------ search
    def run_waves(self, n_waves, evaluator, noise_eps=0.0, noise_alpha=0.3, seed=0, use_graph=True):
        """``n_waves`` playouts for every tree.  ``evaluator(forest)`` must fill ``forest.prior``
        / ``forest.value`` for the leaves of the wave on the current stream."""
        prior_is_log = bool(getattr(evaluator, 'prior_is_log', False))
        capturable = bool(getattr(evaluator, 'graph_capturable', False))

        # the per-search seed travels through the device word the kernels add to their by-value seed
        # (rz_tree_desc.seed_dev), so one captured graph serves every search
        self.seed_dev.fill_(int(seed))

        def wave():
            self.select()
            evaluator(self)
            self.expand_backup(prior_is_log, noise_eps, noise_alpha, 0,
                               value64=getattr(evaluator, 'value64', None),
                               prior64=getattr(evaluator, 'prior64', None))

        if not (use_graph and capturable) or n_waves < 4:
            for _ in range(n_waves):
                wave()
            return
        # one leaf per tree and wave, no host-supplied priors: the backup of wave w and the selection of wave w + 1 share a
        # launch (rz_tree_expand_backup_select).  A search of n waves is  select | (n - 1) x [evaluate, backup + select] |
        # [evaluate, backup]  -- two captured graphs instead of one
        fuse = (self.K == 1 and getattr(evaluator, 'prior64', None) is None
                and os.environ.get('RZ_FUSE_SELECT', '1') != '0')

        # value64 / prior64 are read after the evaluator has run: an evaluator may allocate them in its first call
        # (RandomRolloutEvaluator) or re-allocate them for a forest of another size
        def mid():
            evaluator(self)
            self.expand_backup_select(prior_is_log, noise_eps, noise_alpha, 0,
                                      value64=getattr(evaluator, 'value64', None))

        def last():
            evaluator(self)
            self.expand_backup(prior_is_log, noise_eps, noise_alpha, 0, value64=getattr(evaluator, 'value64', None),
                               prior64=getattr(evaluator, 'prior64', None))

        def buffers():
            # the evaluator's host-visible output buffers as a captured graph holds them: address and shape
            return tuple(None if t is None else (t.data_ptr(), tuple(t.shape))
                         for t in (getattr(evaluator, 'value64', None), getattr(evaluator, 'prior64', None)))

        # weights_version: a captured graph holds the weight pointers (and the fused head's filter taps) and the
        # evaluator's activation buffers by value, so repacked weights or re-allocated buffers need a new capture
        # (NativeForward bumps it in both cases); value64 / prior64 enter the key themselves.  The cache entry keeps
        # the evaluator alive: its id() is the key
        def cache_key():
            return (id(evaluator), getattr(evaluator, 'weights_version', 0), prior_is_log, float(noise_eps),
                    float(noise_alpha), fuse, buffers())

        key = cache_key()
        graphs = self.__dict__.setdefault('_graphs', {})
        if key not in graphs and len(graphs) >= 8:
            graphs.clear()                                              # bounded cache
        if key not in graphs:
            # warm-up outside capture (lazy module loads etc.), then capture
            if fuse:
                self.select()
                mid()                       # wave 1; leaves the leaves of wave 2 selected
                n_waves -= 1
                torch.cuda.synchronize()
                key = cache_key()           # the buffers the warm-up call left are the ones the graphs capture
                g_mid, g_last, g_mid8 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
                with capture_graph(g_mid):
                    mid()
                with capture_graph(g_last):
                    last()
                # eight waves per launch: for one game a wave is ~40 us of GPU time, about what the host needs to launch
                # a graph -- the search of a single game was bound by cudaGraphLaunch calls
                with capture_graph(g_mid8):
                    for _ in range(8):
                        mid()
                graphs[key] = (g_mid, evaluator, g_last, g_mid8)
                self._replay_fused(graphs[key], n_waves - 1)
                return
            wave()
            n_waves -= 1
            torch.cuda.synchronize()
            key = cache_key()
            g = torch.cuda.CUDAGraph()
            with capture_graph(g):
                wave()
            graphs[key] = (g, evaluator, None, None)
            # the capture itself did not run the wave
        g, _, g_last, _ = graphs[key]
        if g_last is not None:
            self.select()
            self._replay_fused(graphs[key], n_waves - 1)
            return
        for _ in range(n_waves):
            g.replay()

    @staticmethod
    def _replay_fused(entry, n_mid):
        """``n_mid`` x [evaluate, backup + select] (eight per graph launch while they last), then [evaluate, backup]."""
        g_mid, _, g_last, g_mid8 = entry
        for _ in range(n_mid // 8):
            g_mid8.replay()
        for _ in range(n_mid % 8):
            g_mid.replay()
        g_last.replay()

    def search(self, evaluator, n_playout=None, **kw):
        """``n_playout`` playouts for every tree (``AlphaZeroMCTS.simulate``, alphazero_mcts.py:83-85).  In
        leaf-parallel mode each tree stops at exactly ``n_playout`` more root visits: the first wave of a fresh
        tree only expands the root, the last wave may be partial."""
        n = self.n_playout if n_playout is None else int(n_playout)
        if self.K == 1:
            self.run_waves(n, evaluator, **kw)
            return
        torch.add(self.root_N, n, out=self.target_N)
        self.run_waves(1 + (max(n - 1, 0) + self.K - 1) // self.K, evaluator, **kw)
        self.target_N.fill_(2 ** 31 - 1)

    # ---------------------------------------------------------------- readback
    def faults(self):
        return self.root_meta[:, L.META_FAULT].cpu().numpy()

    def raise_faults(self):
        """Turn device fault bits into the reference's exceptions."""
        f = self.faults()
        if not f.any():
            return
        self.root_meta[:, L.META_FAULT] = 0
        # a kept subtree larger than max_carry is not an error of the caller: the tree restarted from a fresh root
        # (what update_with_move does for an unknown move, alphazero_mcts.py:102-103); count it
        dropped = (f & L.FAULT_CARRY_DROPPED) != 0
        self.carry_dropped += int(dropped.sum())
        f = f & ~np.int32(L.FAULT_CARRY_DROPPED)
        if not f.any():
            return
        g = int(np.nonzero(f)[0][0])
        bits = int(f[g])
        if bits & L.FAULT_ILLEGAL_MOVE:
            raise AssertionError('You input illegal action (game %d)' % g)  # gomoku_env.py:51
        if bits & L.FAULT_NO_CHILDREN:
            raise ValueError('Node has no children.')  # node.py:39
        raise RuntimeError('search fault bits 0x%x in game %d' % (bits, g))

    def root_stats(self):
        """(visits[G,A] int32, W[G,A] float64, has_child[G,A] bool, root_N[G], root_W[G]) on host."""
        G, A, AS = self.G, self.A, self.AS
        stride = self.max_nodes * AS
        idx = (torch.arange(G, device=self.device, dtype=torch.int64) * stride)[:, None] + \
            torch.arange(AS, device=self.device, dtype=torch.int64)[None, :]
        n = self.edge_N[idx][:, :A].cpu().numpy()
        w = self.edge_W[idx][:, :A].cpu().numpy()
        expanded = (self.n_nodes.cpu().numpy() > 0)[:, None]
        has = (n >= 0) & expanded
        visits = np.where(has, n, 0).astype(np.int32)
        wv = np.where(has & (n > 0), w, 0.0)
        return visits, wv, has, self.root_N.cpu().numpy(), self.root_W.cpu().numpy()

    def dump_tree(self, g):
        """Host copy of tree g as nested dicts (for the TreeNode view / debugging)."""
        nn = int(self.n_nodes[g])
        AS, A = self.AS, self.A
        base = g * self.max_nodes * AS
        sl = slice(base, base + max(nn, 1) * AS)
        N = self.edge_N[sl].cpu().numpy().reshape(-1, AS)[:, :A]
        W = self.edge_W[sl].cpu().numpy().reshape(-1, AS)[:, :A]
        Cc = self.edge_child[sl].cpu().numpy().reshape(-1, AS)[:, :A]
        P = (self.edge_P[sl].cpu().numpy().reshape(-1, AS)[:, :A] if self.edge_P is not None
             else np.ones_like(W, dtype=np.float32))
        if self.edge_P64 is not None:
            P = self.edge_P64[sl].cpu().numpy().reshape(-1, AS)[:, :A]
        out = dict(n_nodes=nn, N=N, W=W, child=Cc, P=P, root_N=int(self.root_N[g]),
                   root_W=float(self.root_W[g]))
        if self.edge_R is not None:
            out['R'] = self.edge_R[sl].cpu().numpy().reshape(-1, AS)[:, :A]
        if self.is_dm:
            out['O'] = self.edge_O[sl].cpu().numpy().reshape(-1, AS)[:, :A]
            out['root_O'] = int(self.root_O[g])
        return out

    def set_child_order(self, g, node, order):
        """DeepMindMCTS child shuffle, host mode: ``order`` = the legal actions of ``node`` of tree ``g`` in the
        order of the reference's shuffled ``children`` list (deepmind_mcts.py:508-513)."""
        base = (g * self.max_nodes + int(node)) * self.AS
        rank = torch.full((self.AS,), 2 ** 31 - 1, dtype=torch.int32)
        rank[torch.as_tensor(list(order), dtype=torch.int64)] = torch.arange(len(order), dtype=torch.int32)
        self.edge_R[base:base + self.AS] = rank.to(self.device)

    def boards(self):
        """Root positions as (rows[G,2,H] uint32, meta[G,8] int32) numpy arrays."""
        return (self.root_rows.cpu().numpy().view(np.uint32), self.root_meta.cpu().numpy())

    def leaf_boards(self):
        return (self.leaf_rows.cpu().numpy().view(np.uint32), self.leaf_meta.cpu().numpy(),
                self.depth.cpu().numpy())

    # ------------------------------------------------------------ trajectories
    def drain_trajectories_device(self):
        """Like ``drain_trajectories`` but the records stay on the device: dict of CUDA tensors
        rows int32 [n,2,H], info int32 [n,6], pi float32 [n,AS] (training-side kernels consume them)."""
        if self.traj is None:
            raise RuntimeError('forest was built without trajectories')
        cur = int(self.traj['ring_cursor'].item())
        lo = max(self._ring_read, cur - self.ring_capacity)
        dropped = lo - self._ring_read
        self._ring_read = cur
        ti = (torch.arange(lo, cur, device=self.device, dtype=torch.int64) % self.ring_capacity)
        return dict(rows=self.traj['ring_rows'][ti].contiguous(), info=self.traj['ring_info'][ti].contiguous(),
                    pi=self.traj['ring_pi'][ti].contiguous(), dropped=int(dropped))

    def drain_trajectories(self):
        """Finished-episode plies written since the last drain: dict of host arrays
        rows[n,2,H] uint32, info[n,6] (mover,last_move,z,slot,episode,ply), pi[n,A] float32."""
        if self.traj is None:
            raise RuntimeError('forest was built without trajectories')
        cur = int(self.traj['ring_cursor'].item())
        lo = max(self._ring_read, cur - self.ring_capacity)
        dropped = lo - self._ring_read  # overwritten before they were drained
        idx = (np.arange(lo, cur) % self.ring_capacity).astype(np.int64)
        self._ring_read = cur
        ti = torch.from_numpy(idx).to(self.device)
        return dict(rows=self.traj['ring_rows'][ti].cpu().numpy().view(np.uint32),
                    info=self.traj['ring_info'][ti].cpu().numpy(),
                    pi=self.traj['ring_pi'][ti][:, :self.A].cpu().numpy(),
                    dropped=int(dropped))


class ClosedFormEvaluator(object):
    """Device-side closed-form evaluator (parity tests, tree-only benchmarks)."""
    graph_capturable = True
    prior_is_log = False

    def __init__(self, eval_id):
        self.eval_id = int(eval_id)

    def __call__(self, forest):
        forest.eval_closed_form(self.eval_id)


class RolloutEvaluator(object):
    """Device-side random-playout evaluator of the pure-MCTS opponent
    (rlzero/mcts/rollout_mcts.py:49-74,96-108)."""
    graph_capturable = True
    prior_is_log = False
    MODES = {'random': 0, 'first': 1, 'last': 2}

    def __init__(self, n_limit=1000, seed=0, mode='random'):
        self.n_limit = int(n_limit)
        self.seed = int(seed)
        self.mode = self.MODES[mode]

    def __call__(self, forest):
        L.check(forest.lib.rz_eval_rollout(C.byref(forest.desc), self.mode, self.seed, self.n_limit,
                                           L.ptr(forest.prior), L.ptr(forest.value), forest._s()),
                'rz_eval_rollout')


class HostCallbackEvaluator(object):
    """Slow path honouring a user-supplied ``policy_value_fn(env)`` (alphazero_mcts.py:27-31):
    leaf positions are copied to the host, rebuilt as env objects, evaluated one by one, and
    the priors/values copied back.  Not graph-capturable; used by the single-game API shim
    and by record/replay parity tests."""
    graph_capturable = False
    prior_is_log = False

    def __init__(self, policy_value_fn, env_factory):
        self.fn = policy_value_fn
        self.env_factory = env_factory
        self.value64 = None
        self.prior64 = None     # float64 priors for forests that keep them (SearchForest(prior_f64=True))

    def _mix(self, act_probs, meta):
        """[(action, prior)] of the node to create; subclasses add the noise."""
        return act_probs

    def __call__(self, forest):
        rows, meta, depth = forest.leaf_boards()
        prior = np.zeros((forest.n_leaves, forest.AS), dtype=np.float64)
        value = np.zeros(forest.n_leaves, dtype=np.float64)
        if self.value64 is None:
            self.value64 = torch.zeros(forest.n_leaves, dtype=torch.float64, device=forest.device)
        if self.prior64 is None and forest.edge_P64 is not None:
            self.prior64 = torch.zeros(forest.n_leaves, forest.AS, dtype=torch.float64, device=forest.device)
        for g in range(forest.n_leaves):
            if depth[g] < 0:
                continue
            env = self.env_factory(rows[g], meta[g])
            act_probs, v = self.fn(env)
            value[g] = v
            if meta[g][L.META_STATUS] != L.ACTIVE:
                continue  # terminal leaf: evaluated (alphazero_mcts.py:59) but never expanded (:61-62)
            for a, p in self._mix(act_probs, meta[g]):
                prior[g, int(a)] = p
        forest.prior.copy_(torch.from_numpy(prior.astype(np.float32)))
        if self.prior64 is not None:
            self.prior64.copy_(torch.from_numpy(prior))   # TreeNode.prior is a Python float: keep every bit
        self.value64.copy_(torch.from_numpy(value))  # python floats are fp64: keep them exact
