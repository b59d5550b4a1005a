"""``TrainPipeline`` with the reference's structure (tools/train_alphazero.py:16-195): self-play ->
8-fold augmentation -> replay buffer -> Adam updates with KL early stopping -> periodic evaluation
against pure MCTS -> checkpoints.

Two collection modes behind the same attributes and methods:

* ``n_parallel_games == 1`` (default): exactly the reference's loop -- one game at a time through
  ``GameControl.start_self_play`` and the host-side ``get_equi_data`` (numpy, same code path);
* ``n_parallel_games > 1``: ``BatchedSelfPlay`` plays that many games concurrently on the GPU;
  finished plies are augmented on the device (``rz_augment_equi``) and appended to a device replay
  buffer (``DeviceReplayBuffer``), mini-batches are gathered on the device (``rz_gather_rows``):
  trajectories never leave HBM between self-play and ``AlphaZeroAgent.learn``.

The training step itself is ``AlphaZeroAgent.learn`` (PyTorch autograd, like the reference).
"""
import ctypes as C
import random
from collections import defaultdict, deque

import numpy as np
import torch

from . import _lib as L
from .games.gomoku import GameControl, GomokuEnv
from .games.gomoku.alphazero_agent import AlphaZeroAgent
from .mcts import AlphaZeroPlayer, RolloutPlayer


class DeviceReplayBuffer(object):
    """``deque(maxlen=buffer_size)`` of (state, pi, z) samples (tools/train_alphazero.py:34) as three
    device rings.  Logical index 0 is the oldest sample, like the deque; ``sample`` draws the indices
    with ``random.sample(range(len), k)``, which consumes the ``random`` stream exactly as the
    reference's ``random.sample(self.data_buffer, k)`` does."""

    def __init__(self, capacity, board_size, device='cuda'):
        self.capacity = int(capacity)
        self.H = int(board_size)
        self.A = self.H * self.H
        self.device = torch.device(device)
        self.states = torch.zeros(self.capacity, 4 * self.A, dtype=torch.float32, device=self.device)
        self.pis = torch.zeros(self.capacity, self.A, dtype=torch.float32, device=self.device)
        self.zs = torch.zeros(self.capacity, 1, dtype=torch.float32, device=self.device)
        self.start = 0      # physical slot of logical index 0
        self.size = 0
        self.lib = L.load()

    def __len__(self):
        return self.size

    def extend(self, states, pis, zs):
        """Append n samples (device tensors [n,4,H,W] / [n,A] / [n]); the oldest fall out."""
        n = int(zs.shape[0])
        if n == 0:
            return
        states = states.reshape(n, 4 * self.A)
        zs = zs.reshape(n, 1)
        if n >= self.capacity:                       # only the newest `capacity` samples survive
            states, pis, zs = states[-self.capacity:], pis[-self.capacity:], zs[-self.capacity:]
            n = self.capacity
            self.start, self.size = 0, 0
        end = (self.start + self.size) % self.capacity
        first = min(n, self.capacity - end)
        for dst, src in ((self.states, states), (self.pis, pis), (self.zs, zs)):
            dst[end:end + first] = src[:first]
            if n > first:
                dst[:n - first] = src[first:]
        overflow = max(0, self.size + n - self.capacity)
        self.start = (self.start + overflow) % self.capacity
        self.size = min(self.capacity, self.size + n)

    def sample(self, batch_size):
        idx = random.sample(range(self.size), batch_size)
        return self.gather(idx)

    def gather(self, logical_indices):
        n = len(logical_indices)
        phys = torch.as_tensor([(self.start + i) % self.capacity for i in logical_indices], dtype=torch.int64,
                               device=self.device)
        out_s = torch.empty(n, 4 * self.A, dtype=torch.float32, device=self.device)
        out_p = torch.empty(n, self.A, dtype=torch.float32, device=self.device)
        out_z = torch.empty(n, 1, dtype=torch.float32, device=self.device)
        s = L.stream_ptr()
        for src, dst, width in ((self.states, out_s, 4 * self.A), (self.pis, out_p, self.A), (self.zs, out_z, 1)):
            L.check(self.lib.rz_gather_rows(L.ptr(src), L.ptr(phys), L.ptr(dst), n, width, s), 'rz_gather_rows')
        return out_s.reshape(n, 4, self.H, self.H), out_p, out_z.reshape(n)


class GoReplayBuffer(object):
    """Replay buffer of Go self-play positions on the device, kept compact: per position the first 16 GoEnv.observe
    planes as row bitmasks (the history is rebuilt from the trajectory ring's records when they are packed, as
    ``BatchedSelfPlay._go_states`` does on the host), the mover, pi [A] and z -- 2672 bytes at 19x19 against 208 000
    for the 8 augmented float32 copies ``DeviceReplayBuffer`` would hold.  The 8 board symmetries are applied when a
    mini-batch is expanded (``rz_go_records_expand``).  Logical index 0 is the oldest record."""

    def __init__(self, capacity, board_size, device='cuda'):
        if not torch.cuda.is_available():
            raise L.NativeLibraryError('GoReplayBuffer needs a CUDA device (no CPU fallback)')
        self.lib = L.load()
        self.capacity = int(capacity)
        if self.capacity < 1:
            raise ValueError('capacity must be at least 1')
        self.H = int(board_size)
        self.A = self.H * self.H + 1
        self.gdesc = L.GameDesc(self.H, 1, self.A, (self.A + 31) // 32 * 32, self.H, L.GAME_GO, 0.0, 0)
        self.device = torch.device(device)
        self.planes = torch.zeros(self.capacity, 16, self.H, dtype=torch.int32, device=self.device)
        self.mover = torch.zeros(self.capacity, dtype=torch.int32, device=self.device)
        self.pis = torch.zeros(self.capacity, self.A, dtype=torch.float32, device=self.device)
        self.zs = torch.zeros(self.capacity, dtype=torch.float32, device=self.device)
        self.start = 0      # physical slot of logical index 0
        self.size = 0

    def __len__(self):
        return self.size

    def bytes_per_position(self):
        return 16 * self.H * 4 + 4 + self.A * 4 + 4

    def extend(self, rows, info, pi):
        """Append n trajectory-ring records in drain order (``SearchForest.drain_trajectories_device`` or
        ``parallel.gather_records_device``: rows int32 [n,2,H], info int32 [n,6], pi float32 [n,AS]); the oldest
        records fall out.  The history of a record comes from the records of this call only, so pass whole drains."""
        n = int(info.shape[0])
        if n == 0:
            return
        if tuple(rows.shape[1:]) != (2, self.H) or int(pi.shape[1]) != self.gdesc.action_stride:
            raise ValueError('ring records of a %dx%d Go board expected (rows [n,2,%d], pi [n,%d])' % (
                self.H, self.H, self.H, self.gdesc.action_stride))
        rows, info, pi = rows.contiguous(), info.contiguous(), pi.contiguous()
        end = (self.start + self.size) % self.capacity
        L.check(self.lib.rz_go_records_pack(C.byref(self.gdesc), L.ptr(rows), L.ptr(info), int(info.shape[1]),
                                            L.ptr(pi), n, L.ptr(self.planes), L.ptr(self.mover), L.ptr(self.pis),
                                            L.ptr(self.zs), self.capacity, end, L.stream_ptr()), 'rz_go_records_pack')
        size = min(self.capacity, self.size + n)
        self.start = (self.start + self.size + n - size) % self.capacity
        self.size = size

    def expand(self, logical_idx, sym):
        """Records ``logical_idx`` (in [0, len)) under symmetries ``sym`` (in [0, 8); device or host integer sequences
        of one length) -> (states [B,17,H,H], pis [B,A], zs [B]) float32 device tensors.  Symmetry s: ``np.rot90`` (s // 2 + 1) times,
        then ``np.fliplr`` when s is odd (6 is the identity), on the planes and on the H*H square probabilities."""
        idx = torch.as_tensor(logical_idx, dtype=torch.int64, device=self.device).reshape(-1)
        sym = torch.as_tensor(sym, dtype=torch.int64, device=self.device).reshape(-1)
        if idx.shape != sym.shape:
            raise ValueError('logical_idx and sym differ in length')
        B = int(idx.shape[0])
        slots = (idx + self.start) % self.capacity
        out_s = torch.empty(B, 17, self.H, self.H, dtype=torch.float32, device=self.device)
        out_p = torch.empty(B, self.A, dtype=torch.float32, device=self.device)
        out_z = torch.empty(B, dtype=torch.float32, device=self.device)
        L.check(self.lib.rz_go_records_expand(C.byref(self.gdesc), L.ptr(self.planes), L.ptr(self.mover),
                                              L.ptr(self.pis), L.ptr(self.zs), self.capacity, L.ptr(slots), L.ptr(sym),
                                              B, L.ptr(out_s), L.ptr(out_p), L.ptr(out_z), L.stream_ptr()),
                'rz_go_records_expand')
        return out_s, out_p, out_z

    def sample(self, batch_size, generator=None):
        """``batch_size`` distinct (record, symmetry) pairs out of the 8 * len: ``random.sample`` over the 8-fold
        augmented buffer, drawn with ``torch.randperm`` on the device (``generator``: a CUDA generator, or None)."""
        batch_size = int(batch_size)
        total = 8 * self.size
        if batch_size < 0 or batch_size > total:
            raise ValueError('sample larger than population or is negative')
        k = torch.randperm(total, generator=generator, device=self.device)[:batch_size]
        return self.expand(k // 8, k % 8)


def augment_equi_device(forest_or_desc, rows, info, pi):
    """Device ``get_equi_data`` (tools/train_alphazero.py:59-79) for n trajectory records:
    rows int32 [n,2,H], info int32 [n,6] (mover, last_move, z, ...), pi float32 [n,AS] ->
    (states [8n,4,H,W], pis [8n,A], zs [8n]) float32 device tensors, reference order."""
    gd = forest_or_desc
    H, A = gd.board_size, gd.n_actions
    n = int(info.shape[0])
    dev = rows.device
    out_s = torch.empty(8 * n, 4, H, H, dtype=torch.float32, device=dev)
    out_p = torch.empty(8 * n, A, dtype=torch.float32, device=dev)
    out_z = torch.empty(8 * n, dtype=torch.float32, device=dev)
    L.check(L.load().rz_augment_equi(C.byref(gd), L.ptr(rows), L.ptr(info), int(info.shape[1]), L.ptr(pi),
                                     L.ptr(out_s), L.ptr(out_p), L.ptr(out_z), n, L.stream_ptr()),
            'rz_augment_equi')
    return out_s, out_p, out_z


class TrainPipeline(object):

    def __init__(self, board_size=6, n_in_row=4, n_playout=400, n_parallel_games=1, device='cuda', net=None,
                 game_batch_num=64, check_freq=50, pure_mcts_playout_num=100, leaves_per_wave=1,
                 batched_evaluation=False):
        # leaves_per_wave > 1: leaf-parallel self-play search of the single-game path (an extension; the default is
        # the reference's sequential search)
        # batched_evaluation: policy_evaluate plays its games at once on the device (BatchedMatch) instead of one after
        # another through GameControl.start_play.  The two paths draw from different random streams, so their results
        # agree in distribution, not game for game
        self.batched_evaluation = bool(batched_evaluation)
        # params of the board and the game (tools/train_alphazero.py:19-26)
        self.board_size = board_size
        self.n_in_row = n_in_row
        self.board = GomokuEnv(board_size=self.board_size, n_in_row=self.n_in_row)
        self.game = GameControl(self.board)
        # training params (:27-45)
        self.learn_rate = 2e-3
        self.lr_multiplier = 1.0
        self.temperature = 1.0
        self.n_playout = n_playout
        self.c_puct = 5
        self.buffer_size = 1000
        self.batch_size = 32
        self.data_buffer = deque(maxlen=self.buffer_size)
        self.play_batch_size = 1
        self.epochs = 5
        self.kl_targ = 0.02
        self.check_freq = check_freq
        self.game_batch_num = game_batch_num
        self.best_win_ratio = 0.0
        self.device = torch.device(device)
        self.pure_mcts_playout_num = pure_mcts_playout_num
        self.alphazero_agent = AlphaZeroAgent(self.board_size, device=self.device, net=net)
        self.mcts_player = AlphaZeroPlayer(self.alphazero_agent.policy_value_fn, n_playout=self.n_playout,
                                           c_puct=self.c_puct, is_selfplay=True, leaves_per_wave=leaves_per_wave)
        # batched collection
        self.n_parallel_games = int(n_parallel_games)
        self.selfplay = None
        self.device_buffer = None
        self.episode_len = 0

    # ------------------------------------------------------------------ data
    def get_equi_data(self, play_data):
        """augment the data set by rotation and flipping (:59-79); host version, reference order."""
        extend_data = []
        for state, mcts_porb, winner in play_data:
            for i in [1, 2, 3, 4]:
                equi_state = np.array([np.rot90(s, i) for s in state])
                equi_mcts_prob = np.rot90(np.flipud(mcts_porb.reshape(self.board_size, self.board_size)), i)
                extend_data.append((equi_state, np.flipud(equi_mcts_prob).flatten(), winner))
                equi_state = np.array([np.fliplr(s) for s in equi_state])
                equi_mcts_prob = np.fliplr(equi_mcts_prob)
                extend_data.append((equi_state, np.flipud(equi_mcts_prob).flatten(), winner))
        return extend_data

    def _ensure_batched(self):
        if self.selfplay is None:
            from .selfplay import BatchedSelfPlay
            self.selfplay = BatchedSelfPlay(self.n_parallel_games, self.board_size, self.n_in_row,
                                            evaluator=self.alphazero_agent.native, n_playout=self.n_playout,
                                            c_puct=self.c_puct, temperature=self.temperature, add_noise=True,
                                            device=self.device)
            self.device_buffer = DeviceReplayBuffer(self.buffer_size, self.board_size, self.device)

    def collect_selfplay_data(self, n_games=1):
        """collect self-play data for training (:81-90)."""
        if self.n_parallel_games <= 1:
            for _ in range(n_games):
                winner, play_data = self.game.start_self_play(self.mcts_player, temperature=self.temperature)
                play_data = list(play_data)[:]
                self.episode_len = len(play_data)
                play_data = self.get_equi_data(play_data)
                self.data_buffer.extend(play_data)
            return
        # batched: advance every game by moves until at least n_games episodes have finished
        self._ensure_batched()
        sp, f = self.selfplay, self.selfplay.forest
        done0 = sp.stats()['games_done']
        while sp.stats()['games_done'] - done0 < n_games:
            sp.play(1)
        out = f.drain_trajectories_device()
        n = int(out['info'].shape[0])
        if n:
            states, pis, zs = augment_equi_device(f.gdesc, out['rows'], out['info'], out['pi'])
            self.device_buffer.extend(states, pis, zs)
            self.episode_len = n // max(1, sp.stats()['games_done'] - done0)

    def _buffer_len(self):
        return len(self.device_buffer) if self.n_parallel_games > 1 and self.device_buffer is not None \
            else len(self.data_buffer)

    # ---------------------------------------------------------------- update
    def policy_update(self):
        """update the policy-value net (:92-137)."""
        if self.n_parallel_games > 1:
            return self._policy_update_device()
        else:
            mini_batch = random.sample(self.data_buffer, self.batch_size)
            state_batch = [data[0] for data in mini_batch]
            mcts_probs_batch = [data[1] for data in mini_batch]
            winner_batch = [data[2] for data in mini_batch]
        old_probs, old_v = self.alphazero_agent.policy_value(state_batch)
        for i in range(self.epochs):
            loss, entropy = self.alphazero_agent.learn(state_batch, mcts_probs_batch, winner_batch)
            new_probs, new_v = self.alphazero_agent.policy_value(state_batch)
            kl = np.mean(np.sum(old_probs * (np.log(old_probs + 1e-10) - np.log(new_probs + 1e-10)), axis=1))
            if kl > self.kl_targ * 4:  # early stopping if D_KL diverges badly
                break
        # adaptively adjust the learning rate (computed but, as in the reference, never applied)
        if kl > self.kl_targ * 2 and self.lr_multiplier > 0.1:
            self.lr_multiplier /= 1.5
        elif kl < self.kl_targ / 2 and self.lr_multiplier < 10:
            self.lr_multiplier *= 1.5
        wb = np.array(winner_batch)
        explained_var_old = 1 - np.var(wb - old_v.flatten()) / np.var(wb)
        explained_var_new = 1 - np.var(wb - new_v.flatten()) / np.var(wb)
        print(('kl:{:.5f},lr_multiplier:{:.3f},loss:{},entropy:{},explained_var_old:{:.3f},'
               'explained_var_new:{:.3f}').format(kl, self.lr_multiplier, loss, entropy, explained_var_old,
                                                  explained_var_new))
        self.last_kl = float(kl)
        return loss, entropy

    def _policy_update_device(self):
        """The same update (:92-137) on a mini-batch gathered from the device replay buffer: states, targets, the
        KL early-stop test and the explained variances stay in HBM; only the printed scalars reach the host."""
        agent = self.alphazero_agent
        state_batch, mcts_probs_batch, winner_batch = self.device_buffer.sample(self.batch_size)
        old_probs, old_v = agent.policy_value_device(state_batch)
        for i in range(self.epochs):
            loss, entropy = agent.learn(state_batch, mcts_probs_batch, winner_batch)
            new_probs, new_v = agent.policy_value_device(state_batch)
            kl = float(torch.mean(torch.sum(old_probs * (torch.log(old_probs + 1e-10) - torch.log(new_probs + 1e-10)),
                                            dim=1)).item())
            if kl > self.kl_targ * 4:  # early stopping if D_KL diverges badly
                break
        if kl > self.kl_targ * 2 and self.lr_multiplier > 0.1:
            self.lr_multiplier /= 1.5
        elif kl < self.kl_targ / 2 and self.lr_multiplier < 10:
            self.lr_multiplier *= 1.5
        var_z = torch.var(winner_batch, unbiased=False)      # np.var is the population variance
        explained_var_old = float((1 - torch.var(winner_batch - old_v.flatten(), unbiased=False) / var_z).item())
        explained_var_new = float((1 - torch.var(winner_batch - new_v.flatten(), unbiased=False) / var_z).item())
        print(('kl:{:.5f},lr_multiplier:{:.3f},loss:{},entropy:{},explained_var_old:{:.3f},'
               'explained_var_new:{:.3f}').format(kl, self.lr_multiplier, loss, entropy, explained_var_old,
                                                  explained_var_new))
        self.last_kl = kl
        return loss, entropy

    def policy_evaluate(self, n_games=10):
        """Evaluate the trained policy against the pure MCTS player (:139-163).  With ``batched_evaluation`` the
        games run as one ``BatchedMatch`` whose draws follow ``np.random.seed`` through its ``seed``."""
        current_mcts_player = AlphaZeroPlayer(self.alphazero_agent.policy_value_fn, n_playout=self.n_playout,
                                              c_puct=self.c_puct)
        pure_mcts_player = RolloutPlayer(n_playout=self.pure_mcts_playout_num, c_puct=5)
        if self.batched_evaluation:
            # every game starts with player1 (id 0), as start_play does whatever start_player says
            from .match import BatchedMatch
            match = BatchedMatch(current_mcts_player, pure_mcts_player, n_games, self.board_size, self.n_in_row,
                                 device=self.device)
            win_cnt = match.play(seed=int(np.random.randint(0, 2 ** 31 - 1)))['win_cnt']
        else:
            win_cnt = defaultdict(int)
            for i in range(n_games):
                winner = self.game.start_play(current_mcts_player, pure_mcts_player, start_player=i % 2, is_shown=0)
                win_cnt[winner] += 1
        win_ratio = 1.0 * (win_cnt[1] + 0.5 * win_cnt[-1]) / n_games
        print('num_playouts:{}, win: {}, lose: {}, tie:{}'.format(self.pure_mcts_playout_num, win_cnt[1],
                                                                  win_cnt[2], win_cnt[-1]))
        return win_ratio

    def run(self):
        """run the training pipeline (:165-190)."""
        try:
            for i in range(self.game_batch_num):
                self.collect_selfplay_data(self.play_batch_size)
                print('batch i:{}, episode_len:{}'.format(i + 1, self.episode_len))
                if self._buffer_len() > self.batch_size:
                    self.policy_update()
                if (i + 1) % self.check_freq == 0:
                    print('current self-play batch: {}'.format(i + 1))
                    win_ratio = self.policy_evaluate()
                    self.alphazero_agent.save_model('./current_policy.model')
                    if win_ratio > self.best_win_ratio:
                        print('New best policy!!!!!!!!')
                        self.best_win_ratio = win_ratio
                        self.alphazero_agent.save_model('./best_policy.model')
                        if self.best_win_ratio == 1.0 and self.pure_mcts_playout_num < 5000:
                            self.pure_mcts_playout_num += 1000
                            self.best_win_ratio = 0.0
        except KeyboardInterrupt:
            print('\n\rquit')


if __name__ == '__main__':
    TrainPipeline().run()
