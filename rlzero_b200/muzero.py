"""MuZero on a board game: representation / dynamics / prediction networks and a batched MCTS in
latent space (BASELINE.json config 5).

The reference has no MuZero code at all (SURVEY.md 8 c2), so this follows the pseudocode published
with the MuZero paper (``MuZeroConfig``, ``run_mcts``, ``select_child``, ``ucb_score``, ``expand_node``,
``backpropagate``, ``add_exploration_noise``, ``MinMaxStats``, ``select_action``) in the two-player
board-game setting: reward 0, discount 1, values negated between plies.  PARITY UNPINNED.

* ``MuZeroNet``      torch parameter container + fp32 checker:  h = stem conv3x3 + R residual blocks
                     (the AlphaZero trunk);  g = conv3x3 + D residual blocks on the hidden state whose
                     last channel is replaced by the one-hot plane of the action;  f = the reference's
                     policy / value heads (rlzero/games/gomoku/policy_value_net.py:19-25,41-51).
* ``MuZeroNative``   the same three functions on the tensor cores through the C ABI
                     (rz_net_stem_tc, rz_net_conv3x3_tc2/3, rz_net_heads_tc, rz_mz_gather).
* ``MuZeroSearch``   G latent-space trees in HBM + the per-move loop
                     h -> f -> rz_mz_root -> 50 x (rz_mz_select -> rz_mz_gather -> g -> f -> rz_mz_expand_backup),
                     captured as one CUDA graph.  Hidden states live node-major (pool[node][tree]) so the
                     dynamics network writes each simulation's new nodes as one contiguous tensor.
* ``BatchedMuZeroSelfPlay``  real games (device Gomoku / Connect Four rules) driven by that search.
"""
import ctypes as C
import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib as L
from .engine import capture_graph
from .games.gomoku.policy_value_net import NativeForward, _ResBlock


class MuZeroConfig(object):
    """The search-related fields of the paper's ``MuZeroConfig`` (board-game values)."""

    def __init__(self, num_simulations=50, discount=1.0, pb_c_base=19652, pb_c_init=1.25,
                 root_dirichlet_alpha=0.3, root_exploration_fraction=0.25, known_bounds=None):
        self.num_simulations = int(num_simulations)
        self.discount = float(discount)
        self.pb_c_base = pb_c_base
        self.pb_c_init = pb_c_init
        self.root_dirichlet_alpha = float(root_dirichlet_alpha)
        self.root_exploration_fraction = float(root_exploration_fraction)
        self.known_bounds = known_bounds        # (min, max) or None


class MuZeroNet(nn.Module):
    """h / g / f with a 128-channel hidden state of the board's shape."""

    def __init__(self, board_size, repr_blocks=4, dyn_blocks=2, in_planes=4, board_width=None, n_actions=None):
        super().__init__()
        self.board_size = board_size
        self.board_width = board_size if board_width is None else board_width
        hw = self.board_size * self.board_width
        self.n_actions = hw if n_actions is None else n_actions
        self.in_planes = in_planes
        c = 128
        self.repr_stem = nn.Conv2d(in_planes, c, 3, padding=1)
        self.repr_blocks = nn.ModuleList([_ResBlock(c) for _ in range(repr_blocks)])
        self.dyn_in = nn.Conv2d(c, c, 3, padding=1)
        self.dyn_blocks = nn.ModuleList([_ResBlock(c) for _ in range(dyn_blocks)])
        self.act_conv1 = nn.Conv2d(c, 4, kernel_size=1)
        self.act_fc1 = nn.Linear(4 * hw, self.n_actions)
        self.val_conv1 = nn.Conv2d(c, 2, kernel_size=1)
        self.val_fc1 = nn.Linear(2 * hw, 64)
        self.val_fc2 = nn.Linear(64, 1)

    # -- h
    def representation(self, obs):
        x = F.relu(self.repr_stem(obs))
        for blk in self.repr_blocks:
            x = blk(x)
        return x

    # -- g: the action enters as the last channel of the hidden state
    def dynamics(self, state, action):
        n, _, h, w = state.shape
        x = state.clone()
        plane = torch.zeros(n, h * w, dtype=state.dtype, device=state.device)
        a = torch.as_tensor(action, device=state.device).long()
        on_board = a < h * w
        plane[torch.nonzero(on_board).flatten(), a[on_board]] = 1.0
        x[:, 127] = plane.view(n, h, w)
        x = F.relu(self.dyn_in(x))
        for blk in self.dyn_blocks:
            x = blk(x)
        return x

    # -- f
    def prediction(self, state):
        hw = self.board_size * self.board_width
        a = F.relu(self.act_conv1(state)).reshape(-1, 4 * hw)
        logp = F.log_softmax(self.act_fc1(a), dim=1)
        v = F.relu(self.val_conv1(state)).reshape(-1, 2 * hw)
        v = torch.tanh(self.val_fc2(F.relu(self.val_fc1(v))))
        return logp, v

    def initial_inference(self, obs):
        s = self.representation(obs)
        return (s,) + tuple(self.prediction(s))

    def recurrent_inference(self, state, action):
        s = self.dynamics(state, action)
        return (s,) + tuple(self.prediction(s))

    def flops(self, which):
        hw, c = self.board_size * self.board_width, 128
        conv = 2 * hw * c * c * 9
        heads = 2 * hw * c * 6 + 2 * (4 * hw) * self.n_actions + 2 * (2 * hw) * 64 + 2 * 64
        if which == 'initial':
            return 2 * hw * self.in_planes * c * 9 + len(self.repr_blocks) * 2 * conv + heads
        return conv + len(self.dyn_blocks) * 2 * conv + heads


class _TrunkView(object):
    """What NativeForward needs to pack one conv stack + the heads of a MuZeroNet."""

    def __init__(self, net, first, blocks):
        self.board_size, self.board_width, self.n_actions = net.board_size, net.board_width, net.n_actions
        self._first, self._blocks = first, blocks
        for name in ('act_conv1', 'act_fc1', 'val_conv1', 'val_fc1', 'val_fc2'):
            setattr(self, name, getattr(net, name))

    def trunk_layers(self):
        layers = [(self._first, None, None, True)]
        for blk in self._blocks:
            skip = len(layers) - 1
            layers.append((blk.conv1, blk.bn1, None, True))
            layers.append((blk.conv2, blk.bn2, skip, True))
        return layers


class MuZeroNative(object):
    """h, g, f of a ``MuZeroNet`` on the tensor cores; hidden states in a node-major pool."""

    def __init__(self, net, n_trees, n_slots, game_type=L.GAME_GOMOKU, n_in_row=5, device='cuda', n_ctas=0):
        if not torch.cuda.is_available():
            raise L.NativeLibraryError('MuZeroNative needs a CUDA device (no CPU fallback)')
        self.lib = L.load()
        self.net = net
        self.G = int(n_trees)
        self.device = torch.device(device)
        self.game_type = int(game_type)
        # weight packing (BatchNorm folded, bf16 [tap][cout][cin]) through the AlphaZero packer
        self.h = NativeForward(_TrunkView(net, net.repr_stem, net.repr_blocks), mode='tc', max_batch=1,
                               device=device, n_ctas=n_ctas, game_type=game_type)
        self.g = NativeForward(_TrunkView(net, net.dyn_in, net.dyn_blocks), mode='tc', max_batch=1,
                               device=device, n_ctas=n_ctas, game_type=game_type)
        if self.h.stem is None:
            raise ValueError('the representation stem must take the 4 observation planes (fused encoder + stem)')
        self.H, self.W, self.S, self.P = self.h.H, self.h.W, self.h.S, self.h.P
        self.A, self.AS = self.h.A, self.h.AS
        self.k = int(n_in_row)
        self.slot_rows = (self.G * self.P + 255) // 256 * 256
        bf = torch.bfloat16
        self.pool = torch.zeros(int(n_slots), self.slot_rows, 128, dtype=bf, device=self.device)
        self.bufs = [torch.zeros(self.slot_rows, 128, dtype=bf, device=self.device) for _ in range(2)]
        # head features [G][6][P] (rz_net_head_features -> rz_net_heads_tc: the FCs of f on the tensor cores)
        self.feat = torch.zeros(self.G, 6, self.P, dtype=torch.float32, device=self.device)
        self.logp = torch.zeros(self.G, self.AS, dtype=torch.float32, device=self.device)
        self.value = torch.zeros(self.G, dtype=torch.float32, device=self.device)
        self.weights_version = 0

    def refresh_weights(self):
        self.h.refresh_weights()
        self.g.refresh_weights()
        self.weights_version += 1

    def hbm_bytes(self):
        return sum(t.numel() * t.element_size() for t in [self.pool] + self.bufs)

    def _blocks(self, nf, x, other, final_out):
        """Residual blocks nf.layers[1:] on the activation in ``x`` (``other`` = scratch); the last conv
        writes ``final_out``.  Returns nothing; with no blocks the caller wrote final_out already."""
        layers = nf.layers
        n_blocks = (len(layers) - 1) // 2
        for b in range(n_blocks):
            c1, c2 = layers[1 + 2 * b], layers[2 + 2 * b]
            nf._conv(c1, x, None, other, self.G)
            last = b == n_blocks - 1
            nf._conv(c2, other, x, final_out if last else x, self.G)      # residual may alias the output

    def representation(self, rows, meta, slot=0):
        """h(observation of the device positions) -> pool[slot]."""
        nf = self.h
        g = nf._gdesc(self.k)
        n_blocks = (len(nf.layers) - 1) // 2
        first_out = self.pool[slot] if n_blocks == 0 else self.bufs[0]
        st = nf.stem
        L.check(self.lib.rz_net_stem_tc(C.byref(g), L.ptr(rows), L.ptr(meta), L.ptr(st['w']), L.ptr(st['b']),
                                        L.ptr(first_out), self.G, int(st['relu']), 0, L.stream_ptr()),
                'rz_net_stem_tc')
        self._blocks(nf, self.bufs[0], self.bufs[1], self.pool[slot])

    def dynamics(self, parent, action, slot):
        """g(pool[parent[g]][g], action[g]) -> pool[slot] for every tree g."""
        L.check(self.lib.rz_mz_gather(L.ptr(self.pool), L.ptr(parent), L.ptr(action), L.ptr(self.bufs[0]), self.G,
                                      self.H, self.W, self.S, self.slot_rows, L.stream_ptr()), 'rz_mz_gather')
        nf = self.g
        n_blocks = (len(nf.layers) - 1) // 2
        first_out = self.pool[slot] if n_blocks == 0 else self.bufs[1]
        nf._conv(nf.layers[0], self.bufs[0], None, first_out, self.G)
        self._blocks(nf, self.bufs[1], self.bufs[0], self.pool[slot])

    def prediction(self, slot, logp=None, value=None):
        """f(pool[slot]) -> (log-probabilities [G][AS], value [G])."""
        logp = self.logp if logp is None else logp
        value = self.value if value is None else value
        L.check(self.lib.rz_net_head_features(C.byref(self.h.hdesc), L.ptr(self.pool[slot]), L.ptr(self.feat),
                                              self.G, L.stream_ptr()), 'rz_net_head_features')
        L.check(self.lib.rz_net_heads_tc(C.byref(self.h.hdesc), L.ptr(self.feat), L.ptr(logp), L.ptr(value),
                                         self.G, L.stream_ptr()), 'rz_net_heads_tc')
        return logp, value

    def unroll(self, rows, meta, actions):
        """Batched K-step unroll (BASELINE config 5; the MuZero paper's training / reanalysis unroll, forward
        side): s0 = h(position g), s_k = g(s_{k-1}, actions[g][k-1]), (p_k, v_k) = f(s_k) for every position of the
        batch at once.  ``actions``: int [G][K] (device or host).  Returns (logp [K+1][G][AS], value [K+1][G]) float32
        device tensors; hidden state k stays in pool slot k (needs K + 1 <= n_slots).  Positions are independent, so
        across GPUs the batch is simply sharded (no collective)."""
        a = torch.as_tensor(actions, dtype=torch.int32, device=self.device).contiguous()
        if a.dim() != 2 or a.shape[0] != self.G:
            raise ValueError('actions must be [G][K] with G = %d' % self.G)
        K = int(a.shape[1])
        if K + 1 > self.pool.shape[0]:
            raise ValueError('unroll of %d steps needs %d hidden-state slots, the pool has %d' % (K, K + 1, self.pool.shape[0]))
        logp = torch.zeros(K + 1, self.G, self.AS, dtype=torch.float32, device=self.device)
        value = torch.zeros(K + 1, self.G, dtype=torch.float32, device=self.device)
        at = a.t().contiguous()                       # [K][G]: one contiguous action vector per step
        self.representation(rows, meta, 0)
        self.prediction(0, logp[0], value[0])
        for k in range(K):
            parent = torch.full((self.G,), k, dtype=torch.int32, device=self.device)
            self.dynamics(parent, at[k], k + 1)
            self.prediction(k + 1, logp[k + 1], value[k + 1])
        return logp, value

    def kernels_per_simulation(self):
        return 1 + len(self.g.layers) + 2      # gather + convolutions + head features + FC heads

    def hidden_state(self, slot):
        """pool[slot] as float32 [G, 128, H, W] (tests)."""
        t = self.pool[slot][:self.G * self.P].view(self.G, self.S, self.S, 128)[:, :self.H, :self.W]
        return t.permute(0, 3, 1, 2).float()


def pbc_table(n, pb_c_base, pb_c_init):
    """pbc_table[N] = math.log((N + pb_c_base + 1) / pb_c_base) + pb_c_init with CPython's libm log."""
    t = np.zeros(n, dtype=np.float64)
    for k in range(n):
        t[k] = math.log((k + pb_c_base + 1) / pb_c_base) + pb_c_init
    return t


class MuZeroSearch(object):
    """G latent-space search trees + the networks, resident in HBM."""

    def __init__(self, n_trees, net, config=None, game_type=L.GAME_GOMOKU, n_in_row=5, device='cuda',
                 global_offset=0, seed=0, n_ctas=0):
        self.cfg = config or MuZeroConfig()
        self.G = int(n_trees)
        self.device = torch.device(device)
        self.seed = int(seed)
        S = self.cfg.num_simulations
        self.native = MuZeroNative(net, self.G, S + 1, game_type=game_type, n_in_row=n_in_row, device=device,
                                   n_ctas=n_ctas)
        self.lib = self.native.lib
        self.A, self.AS = self.native.A, self.native.AS
        self.max_nodes = S + 1
        G, AS, dev = self.G, self.AS, self.device
        i32, f64, f32 = torch.int32, torch.float64, torch.float32
        n_edges = G * self.max_nodes * AS
        self.edge_N = torch.zeros(n_edges, dtype=i32, device=dev)
        self.edge_W = torch.zeros(n_edges, dtype=f64, device=dev)
        self.edge_P = torch.zeros(n_edges, dtype=f32, device=dev)
        self.edge_child = torch.zeros(n_edges, dtype=i32, device=dev)
        for name in ('n_nodes', 'root_N', 'depth', 'leaf_parent', 'leaf_action', 'fault'):
            setattr(self, name, torch.zeros(G, dtype=i32, device=dev))
        for name in ('root_W', 'mm_min', 'mm_max'):
            setattr(self, name, torch.zeros(G, dtype=f64, device=dev))
        self.path_node = torch.zeros(G, self.max_nodes, dtype=i32, device=dev)
        self.path_action = torch.zeros(G, self.max_nodes, dtype=i32, device=dev)
        self.pbc = torch.from_numpy(pbc_table(S + 2, self.cfg.pb_c_base, self.cfg.pb_c_init)).to(dev)
        d = L.MzDesc()
        d.n_trees, d.n_actions, d.action_stride = G, self.A, AS
        d.max_nodes, d.max_depth, d.pbc_table_len = self.max_nodes, self.max_nodes, S + 2
        d.discount = self.cfg.discount
        kb = self.cfg.known_bounds
        d.known_min, d.known_max = (float('inf'), float('-inf')) if kb is None else (float(kb[0]), float(kb[1]))
        d.global_offset = int(global_offset)
        for name in ('edge_N', 'edge_W', 'edge_P', 'edge_child', 'n_nodes', 'root_N', 'root_W', 'mm_min', 'mm_max',
                     'path_node', 'path_action', 'depth', 'leaf_parent', 'leaf_action', 'fault'):
            setattr(d, name, getattr(self, name).data_ptr())
        d.pbc_table = self.pbc.data_ptr()
        self.desc = d
        self._graph = None
        self._graph_key = None
        self.moves_searched = 0

    def hbm_bytes(self):
        tot = self.native.hbm_bytes()
        for v in vars(self).values():
            if isinstance(v, torch.Tensor):
                tot += v.numel() * v.element_size()
        return tot

    # ------------------------------------------------------------------ pieces
    def _s(self):
        return L.stream_ptr()

    def root(self, rows, meta, legal=None, add_noise=True, move_id=0, move_ids=None):
        """initial_inference + expand_node(root, legal_actions) + add_exploration_noise.  ``move_ids``
        (int32 [G] on the device) keys the noise per game and move; it is read at run time, so a
        captured graph draws fresh noise on every replay."""
        nat = self.native
        nat.representation(rows, meta, 0)
        nat.prediction(0)
        eps = self.cfg.root_exploration_fraction if add_noise else 0.0
        L.check(self.lib.rz_mz_root(C.byref(self.desc), L.ptr(nat.logp), L.ptr(legal), float(eps),
                                    self.cfg.root_dirichlet_alpha, self.seed, int(move_id) & 0xffffffff,
                                    L.ptr(move_ids), self._s()),
                'rz_mz_root')

    def simulate(self, i):
        """Simulation i (0-based): creates node i + 1 of every tree."""
        nat = self.native
        L.check(self.lib.rz_mz_select(C.byref(self.desc), self._s()), 'rz_mz_select')
        nat.dynamics(self.leaf_parent, self.leaf_action, i + 1)
        nat.prediction(i + 1)
        L.check(self.lib.rz_mz_expand_backup(C.byref(self.desc), L.ptr(nat.logp), L.ptr(nat.value), self._s()),
                'rz_mz_expand_backup')

    def kernels_per_move(self):
        nat = self.native
        return (len(nat.h.layers) + 3) + self.cfg.num_simulations * (2 + nat.kernels_per_simulation())

    # ------------------------------------------------------------------- search
    def run(self, rows, meta, legal=None, add_noise=True, use_graph=True, move_ids=None):
        """run_mcts for every tree from the device positions (rows [G,2,H], meta [G,12]); ``legal``
        uint8 [G,A] restricts the root's children (None = the whole action space)."""
        S = self.cfg.num_simulations
        key = (rows.data_ptr(), meta.data_ptr(), None if legal is None else legal.data_ptr(), bool(add_noise),
               self.native.weights_version, None if move_ids is None else move_ids.data_ptr())
        if not use_graph:
            self.root(rows, meta, legal, add_noise, self.moves_searched, move_ids)
            for i in range(S):
                self.simulate(i)
        else:
            if self._graph is None or self._graph_key != key:
                # a launch-parameter counter would be frozen into the graph: per-move noise needs move_ids
                self.root(rows, meta, legal, add_noise, 0, move_ids)
                self.simulate(0)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with capture_graph(g):
                    self.root(rows, meta, legal, add_noise, 0, move_ids)
                    for i in range(S):
                        self.simulate(i)
                self._graph, self._graph_key = g, key
            self._graph.replay()
        self.moves_searched += 1

    def raise_faults(self):
        f = self.fault.cpu().numpy()
        if f.any():
            self.fault.zero_()
            raise RuntimeError('MuZero search fault bits 0x%x in tree %d' % (int(f[f != 0][0]), int(np.nonzero(f)[0][0])))

    # ----------------------------------------------------------------- readback
    def root_visits(self):
        """int32 [G, A] visit counts of the root's children (0 where there is no child)."""
        v = self.edge_N.view(self.G, self.max_nodes, self.AS)[:, 0, :self.A]
        return v.clamp(min=0)

    def select_action(self, temperature=1.0):
        """select_action of the pseudocode: sample a move from visit_count ** (1 / T) (argmax at T = 0)."""
        v = self.root_visits().double()
        if temperature == 0:
            return v.argmax(dim=1).int()
        w = v.pow(1.0 / temperature)
        return torch.multinomial(w / w.sum(dim=1, keepdim=True), 1).flatten().int()

    def dump_tree(self, g):
        nn_ = int(self.n_nodes[g])
        AS, A = self.AS, self.A
        sl = slice(g * self.max_nodes * AS, (g * self.max_nodes + max(nn_, 1)) * AS)
        return dict(n_nodes=nn_, N=self.edge_N[sl].cpu().numpy().reshape(-1, AS)[:, :A],
                    W=self.edge_W[sl].cpu().numpy().reshape(-1, AS)[:, :A],
                    P=self.edge_P[sl].cpu().numpy().reshape(-1, AS)[:, :A],
                    child=self.edge_child[sl].cpu().numpy().reshape(-1, AS)[:, :A],
                    root_N=int(self.root_N[g]), root_W=float(self.root_W[g]), mm_min=float(self.mm_min[g]),
                    mm_max=float(self.mm_max[g]))


class BatchedMuZeroSelfPlay(object):
    """G real games (device rules of rz_game.cu) whose moves come from MuZero searches: per move
    h(observation) -> 50 latent simulations -> sample from the visit counts -> env.step."""

    def __init__(self, n_games, board_size=15, n_in_row=5, net=None, config=None, temperature=1.0, device='cuda',
                 global_offset=0, seed=0, board_width=None, game_type=L.GAME_GOMOKU):
        if game_type == L.GAME_GO:
            raise NotImplementedError('MuZero self-play drives Gomoku / Connect Four boards')
        self.G = int(n_games)
        self.H = int(board_size)
        self.W = self.H if board_width is None else int(board_width)
        self.temperature = float(temperature)
        self.search = MuZeroSearch(self.G, net, config, game_type=game_type, n_in_row=n_in_row, device=device,
                                   global_offset=global_offset, seed=seed)
        self.lib = self.search.lib
        A = self.search.A
        self.gdesc = L.GameDesc(self.H, int(n_in_row), A, self.search.AS, self.W, int(game_type))
        dev = self.search.device
        self.rows = torch.zeros(self.G, 2, self.H, dtype=torch.int32, device=dev)
        self.meta = torch.zeros(self.G, L.META_STRIDE, dtype=torch.int32, device=dev)
        self.legal = torch.zeros(self.G, A, dtype=torch.uint8, device=dev)
        self.win = torch.zeros(self.G, dtype=torch.int32, device=dev)
        self.move_ids = torch.zeros(self.G, dtype=torch.int32, device=dev)     # noise counter per game
        self.games_done = 0
        self.moves_played = 0
        self._reset(False)

    def _reset(self, only_ended):
        L.check(self.lib.rz_gomoku_reset(C.byref(self.gdesc), L.ptr(self.rows), L.ptr(self.meta), self.G,
                                         int(only_ended), L.stream_ptr()), 'rz_gomoku_reset')

    def play_move(self, add_noise=True):
        s = L.stream_ptr()
        L.check(self.lib.rz_gomoku_legal_mask(C.byref(self.gdesc), L.ptr(self.rows), L.ptr(self.legal), self.G, s),
                'rz_gomoku_legal_mask')
        self.search.run(self.rows, self.meta, self.legal, add_noise=add_noise, move_ids=self.move_ids)
        self.move_ids += 1
        move = self.search.select_action(self.temperature)
        L.check(self.lib.rz_gomoku_step(C.byref(self.gdesc), L.ptr(self.rows), L.ptr(self.meta), L.ptr(move), None,
                                        L.ptr(self.win), self.G, s), 'rz_gomoku_step')
        ended = (self.meta[:, L.META_STATUS] != L.ACTIVE)
        self.games_done += int(ended.sum().item())
        self._reset(True)                           # finished games restart from the empty board
        self.moves_played += 1
        return move
