"""Policy-value networks: parameter containers (torch modules, state_dict compatible with the
reference) and ``NativeForward``, the CUDA inference path that the search uses.

* ``PolicyValueNet``       = rlzero/games/gomoku/policy_value_net.py:6-52, same parameter names
                             and shapes, so reference checkpoints load unchanged
                             (alphazero_agent.py:99-125).
* ``ResNetPolicyValueNet`` = the benchmark trunk SURVEY.md section 7 defines (the reference has no
                             ResNet): stem conv3x3(4->C)+ReLU, N blocks of
                             2x[conv3x3(C->C)+BN] + skip + ReLU, reference heads unchanged.

``forward`` of the modules is plain PyTorch (training side and fp32 checker).  Inference for the
search never goes through it: ``NativeForward`` packs the weights (BatchNorm folded) into the
layouts of include/rlzero_b200.h and runs the hand-written kernels -- tcgen05 tensor-core
convolutions in bf16 for 128-channel trunks on boards up to 15x15, the fp32 CUDA-core path for
the stock network / other shapes.
"""
import ctypes as C

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from ... import _lib as L


class PolicyValueNet(nn.Module):
    """policy-value network module (reference architecture and parameter names)."""

    def __init__(self, board_size):
        super().__init__()
        self.board_size = board_size
        hw = board_size * board_size
        self.conv1 = nn.Conv2d(4, 32, kernel_size=3, padding=1)
        self.conv2 = nn.Conv2d(32, 64, kernel_size=3, padding=1)
        self.conv3 = nn.Conv2d(64, 128, kernel_size=3, padding=1)
        self.act_conv1 = nn.Conv2d(128, 4, kernel_size=1)
        self.act_fc1 = nn.Linear(4 * hw, hw)
        self.val_conv1 = nn.Conv2d(128, 2, kernel_size=1)
        self.val_fc1 = nn.Linear(2 * hw, 64)
        self.val_fc2 = nn.Linear(64, 1)

    def trunk(self, obs):
        x = F.relu(self.conv1(obs))
        x = F.relu(self.conv2(x))
        return F.relu(self.conv3(x))

    def heads(self, x):
        hw = self.board_size * getattr(self, 'board_width', self.board_size)
        a = F.relu(self.act_conv1(x)).reshape(-1, 4 * hw)
        logp = F.log_softmax(self.act_fc1(a), dim=1)
        v = F.relu(self.val_conv1(x)).reshape(-1, 2 * hw)
        v = torch.tanh(self.val_fc2(F.relu(self.val_fc1(v))))
        return logp, v

    def forward(self, obs):
        return self.heads(self.trunk(obs))

    def trunk_layers(self):
        """[(conv, bn_or_None, residual_from_layer_index_or_None, relu)] in execution order."""
        return [(self.conv1, None, None, True), (self.conv2, None, None, True),
                (self.conv3, None, None, True)]


class _ResBlock(nn.Module):

    def __init__(self, c):
        super().__init__()
        self.conv1 = nn.Conv2d(c, c, 3, padding=1)
        self.bn1 = nn.BatchNorm2d(c)
        self.conv2 = nn.Conv2d(c, c, 3, padding=1)
        self.bn2 = nn.BatchNorm2d(c)

    def forward(self, x):
        y = F.relu(self.bn1(self.conv1(x)))
        return F.relu(self.bn2(self.conv2(y)) + x)


class ResNetPolicyValueNet(PolicyValueNet):
    """ResNet-N trunk (C channels) with the reference's heads."""

    def __init__(self, board_size, n_blocks=10, channels=128, board_width=None, n_actions=None, in_planes=4):
        """``board_size`` rows x ``board_width`` columns (square by default, like the reference);
        ``n_actions`` policy outputs (rows*columns by default; the columns for Connect Four;
        rows*columns + 1 for Go, whose last action is the pass); ``in_planes`` observation planes
        (4 = GomokuEnv.current_state, 17 = GoEnv.observe)."""
        nn.Module.__init__(self)
        if channels != 128:
            raise ValueError('the reference heads take 128 trunk channels (policy_value_net.py:19,23)')
        self.board_size = board_size
        self.board_width = board_size if board_width is None else board_width
        self.n_blocks = n_blocks
        hw = self.board_size * self.board_width
        self.n_actions = hw if n_actions is None else n_actions
        self.in_planes = in_planes
        self.stem = nn.Conv2d(in_planes, channels, 3, padding=1)
        self.blocks = nn.ModuleList([_ResBlock(channels) for _ in range(n_blocks)])
        self.act_conv1 = nn.Conv2d(channels, 4, kernel_size=1)
        self.act_fc1 = nn.Linear(4 * hw, self.n_actions)
        self.val_conv1 = nn.Conv2d(channels, 2, kernel_size=1)
        self.val_fc1 = nn.Linear(2 * hw, 64)
        self.val_fc2 = nn.Linear(64, 1)

    def trunk(self, obs):
        x = F.relu(self.stem(obs))
        for blk in self.blocks:
            x = blk(x)
        return x

    def trunk_layers(self):
        layers = [(self.stem, None, None, True)]
        for blk in self.blocks:
            skip = len(layers) - 1           # output of the previous layer
            layers.append((blk.conv1, blk.bn1, None, True))
            layers.append((blk.conv2, blk.bn2, skip, True))
        return layers

    def flops_per_eval(self):
        hw = self.board_size * self.board_width
        c = 128
        trunk = 2 * hw * (self.in_planes * c * 9) + self.n_blocks * 2 * 2 * hw * c * c * 9
        heads = 2 * hw * c * 6 + 2 * (4 * hw) * self.n_actions + 2 * (2 * hw) * 64 + 2 * 64
        return trunk + heads


def _fold_bn(conv, bn):
    """Conv weight/bias with an eval-mode BatchNorm folded in (float64 arithmetic)."""
    w = conv.weight.detach().double()
    b = conv.bias.detach().double() if conv.bias is not None else torch.zeros(w.shape[0], dtype=torch.float64,
                                                                              device=w.device)
    if bn is not None:
        s = bn.weight.detach().double() / torch.sqrt(bn.running_var.detach().double() + bn.eps)
        w = w * s[:, None, None, None]
        b = (b - bn.running_mean.detach().double()) * s + bn.bias.detach().double()
    return w, b


class NativeForward(object):
    """CUDA forward of a policy-value module through the C ABI (no PyTorch ops on the hot path).

    mode 'tc'  : bf16 tensor-core trunk (trunk convs of at most 128 channels, the last one exactly 128; narrower
                 layers -- the stock PolicyValueNet's 4 -> 32 -> 64 -> 128 -- run zero-padded to 128 channels:
                 a padded 128 -> 128 layer on the tensor cores is still ~50x faster than the fp32 CUDA-core path;
                 boards up to 19x19; outputs within 1e-3 of fp32.  Opt-in for the stock network, whose default
                 stays 'f32')
    mode 'f32' : fp32 CUDA-core trunk (any channel counts, any board <= 19)
    mode 'tc32': the reference's own PolicyValueNet (4 -> 32 -> 64 -> 128, policy_value_net.py:14-16) on the tensor
                 cores at float32-level accuracy: every activation and weight travels as a bf16 (high, low) pair
                 (x = hi + lo, 16 mantissa bits) and every convolution forms hi*Whi + lo*Whi + hi*Wlo (+ lo*Wlo
                 where it is free) in the fp32 accumulators -- the recipe of the tensor-core heads.  conv1 is the
                 fused encoder/stem kernel with the filters' high parts and residues as separate output columns;
                 conv2 is ONE ordinary K = 128 pass over [hi | lo | hi | lo] x [Whi | Whi | Wlo | Wlo]; conv3 runs
                 three products per tap and feeds the heads' 1x1 convolutions from the fp32 accumulators.  Boards
                 up to 15x15 (16-stride layout).  The default for the stock network on such boards.
    """
    graph_capturable = True
    prior_is_log = True       # the network emits log-probabilities (policy_value_net.py:44)

    def __init__(self, module, mode=None, max_batch=1, device='cuda', n_ctas=0, fused_head=True, game_type=None,
                 row_stride=None):
        if not torch.cuda.is_available():
            raise L.NativeLibraryError('NativeForward needs a CUDA device (no CPU fallback)')
        self.lib = L.load()
        self.module = module
        self.device = torch.device(device)
        self.H = int(module.board_size)
        self.W = int(getattr(module, 'board_width', self.H))
        self.HW = self.H * self.W                      # squares (inputs of the FC heads)
        self.A = int(getattr(module, 'n_actions', self.HW))   # policy outputs
        self.AS = (self.A + 31) // 32 * 32
        if game_type is None:   # a policy head over the columns of a non-square board = a gravity game
            game_type = L.GAME_CONNECT4 if (self.A == self.W and self.A != self.HW) else (
                L.GAME_GO if self.A == self.HW + 1 else L.GAME_GOMOKU)
        self.game_type = int(game_type)
        layers = module.trunk_layers()
        all128 = all(l[0].out_channels == 128 for l in layers)
        # narrower trunks fit the tensor-core kernels zero-padded to 128 channels (opt-in: mode='tc')
        tc_able = (all(l[0].out_channels <= 128 and l[0].in_channels <= 128 for l in layers)
                   and layers[-1][0].out_channels == 128 and (all128 or layers[0][0].in_channels in (4, 17)))
        fits = self.H <= 19 and self.W <= 19
        # padded position layout of the tensor-core path: row = board*S*S + y*S + x, S the smallest of 8 / 16 / 20
        # with a zero column and a zero row left (Connect Four 6x7 and other boards up to 7x7: S = 8, 64 rows per
        # board instead of 256); the Go stem stages at most two boards per tile and keeps 16 / 20
        auto = L.row_stride(self.H, self.W)
        if self.game_type == L.GAME_GO:
            auto = max(auto, 16)
        self.S = int(row_stride) if row_stride else (auto or 20)
        if fits and L.row_stride(self.H, self.W, self.S) != self.S:
            raise ValueError('row_stride %r does not hold a %dx%d board (8, 16 or 20, > max(H, W))' % (
                row_stride, self.H, self.W))
        self.P = self.S * self.S
        stock = (len(layers) == 3 and [l[0].in_channels for l in layers] == [4, 32, 64]
                 and [l[0].out_channels for l in layers] == [32, 64, 128] and all(l[1] is None and l[2] is None for l in layers)
                 and self.game_type != L.GAME_GO)
        if mode is None:
            mode = 'tc' if (all128 and fits) else ('tc32' if (stock and max(self.H, self.W) <= 15) else 'f32')
        if mode == 'tc32':
            if not (stock and max(self.H, self.W) <= 15):
                raise ValueError("mode 'tc32' serves the stock 4 -> 32 -> 64 -> 128 PolicyValueNet on boards up to 15x15")
            if row_stride not in (None, 0, 16):
                raise ValueError("mode 'tc32' uses the 16-stride layout")
            self.S, self.P = 16, 256
        if mode == 'tc' and not (tc_able and fits):
            raise ValueError("mode 'tc' needs trunk layers of at most 128 channels (the last one 128) and a board of "
                             "at most 19x19")
        if mode == 'f32' and self.W != self.H:
            raise ValueError('the fp32 CUDA-core path handles square boards only')
        if self.game_type == L.GAME_GO and mode != 'tc':
            raise ValueError('Go runs on the tensor-core path only (128-channel trunk, 17 input planes)')
        self.mode = mode
        self.n_ctas = int(n_ctas)
        # the heads' 1x1 convolutions inside the last trunk layer's epilogue (rz_net_tc2.cu, kHead)
        self.fused_head = bool(fused_head)
        self.weights_version = 0
        # boards up to which the one-launch trunk of rz_net_trunk_small.cu is used (one CTA pair per board, 74 pairs at a
        # time on 148 SMs; measured crossover with the per-layer kernels near 200 boards, profiles/r2_run43_crossover.log)
        self.small_batch_max = 148
        # boards from which the batched trunk runs in one launch (rz_net_trunk_tc2.cu: CTA pairs carry chunks of
        # `trunk_chunk` boards through every layer, the activations in an L2-sized scratch); below it, one launch per
        # layer.  The batched trunk is the faster one at every measured count from 300 boards up (ResNet-10 15x15: 22 %
        # at 300, 4.6 % at 8192, profiles/r3_run1_trunk_probe.jsonl), so it starts right above the 300-board batch that
        # keeps the per-layer kernels as the reference the small-batch path is checked against.  Chunks of 6 boards
        # (55 MB of scratch on 74 pairs) measured fastest at 8192 boards among 4..16.  Set batched_trunk_min on an
        # instance to a larger count to force the per-layer kernels.
        self.batched_trunk_min = 301
        self.trunk_chunk = 6
        self.scratch = None
        # flags of the 128 -> 128 rz_net_conv3x3_tc2 launches, read by bench.py too: 512 = static weights
        # (include/rlzero_b200.h); bit 1 (2) is accepted and ignored
        self.conv_flags = 514
        self.max_batch = 0
        self.refresh_weights()
        self._alloc(max_batch)

    # ------------------------------------------------------------------ weights
    def refresh_weights(self):
        """(Re)pack the module's current parameters for the kernels (after load / a training step)."""
        dev = self.device
        m = self.module
        self.layers = []
        if self.mode == 'tc32':
            self._pack_tc32()
        for conv, bn, skip, relu in (m.trunk_layers() if self.mode != 'tc32' else []):
            if (self.mode == 'tc' and conv.in_channels == 128 and conv.out_channels == 128 and len(self.layers) > 0
                    and conv.weight.is_cuda and conv.weight.dtype == torch.float32 and conv.weight.is_contiguous()):
                # a 128 -> 128 trunk layer whose parameters live on the device: folded and packed by one kernel
                wd = torch.empty(9, 128, 128, dtype=torch.bfloat16, device=dev)
                bd = torch.empty(128, dtype=torch.float32, device=dev)
                cb = conv.bias.detach() if conv.bias is not None else None
                L.check(self.lib.rz_net_pack_conv_bn_tc(
                    L.ptr(conv.weight.detach()), L.ptr(cb), L.ptr(bn.weight.detach()) if bn is not None else None,
                    L.ptr(bn.bias.detach()) if bn is not None else None, L.ptr(bn.running_mean) if bn is not None else None,
                    L.ptr(bn.running_var) if bn is not None else None, float(bn.eps) if bn is not None else 0.0,
                    L.ptr(wd), L.ptr(bd), L.stream_ptr()), 'rz_net_pack_conv_bn_tc')
                self.layers.append(dict(w=wd, b=bd, cin=128, cout=128, skip=skip, relu=bool(relu)))
                continue
            w, b = _fold_bn(conv, bn)                      # [Cout][Cin][3][3]
            cout, cin = w.shape[0], w.shape[1]
            if self.mode == 'tc':
                # [tap][cout][cin], zero-padded to 128 output channels (a narrower layer's extra channels come
                # out as relu(0) = 0) and to the 128 channels the previous layer wrote (64 for the plane input)
                # (packed where the parameters live: after a training step that is the device -- no host round trip)
                cin_p = 128 if len(self.layers) > 0 else (64 if cin <= 64 else 128)
                wt = torch.zeros(9, 128, cin_p, dtype=torch.float64, device=w.device)
                wt[:, :cout, :cin] = w.permute(2, 3, 0, 1).reshape(9, cout, cin)
                wd = wt.to(torch.bfloat16).contiguous().to(dev)
                bpad = torch.zeros(128, dtype=b.dtype, device=b.device)
                bpad[:cout] = b
                b, cout = bpad, 128
            else:
                cin_p = cin
                wd = w.permute(2, 3, 1, 0).reshape(9, cin, cout).float().contiguous().to(dev)  # [tap][cin][cout]
            self.layers.append(dict(w=wd, b=b.float().contiguous().to(dev), cin=cin_p, cout=cout,
                                    skip=skip, relu=bool(relu)))
        # small-batch latency path (rz_net_trunk_small.cu): the 128 -> 128 layers behind the stem in one stacked buffer
        # [layer][tap][cout][cin]; the per-layer tensors become views of it, so both paths read the same bytes
        self.trunk_small = None
        if self.mode == 'tc32' and self.S == 16:
            # conv2 (64 channels, split output) and conv3 (split input, float32 head features) of the reference's own net
            l2, l3 = self.layers[1], self.layers[2]
            wst = torch.stack([l2['w'], l3['w']]).contiguous()
            bst = torch.stack([l2['b'], l3['b']]).contiguous()
            l2['w'], l2['b'], l3['w'], l3['b'] = wst[0], bst[0], wst[1], bst[1]
            self.trunk_small = dict(w=wst, b=bst, n=2, relu_mask=int(bool(l2['relu'])) | (int(bool(l3['relu'])) << 1),
                                    res_mask=0, n64_mask=1, split_in_mask=2, head_f32=1)
        if (self.mode == 'tc' and self.S == 16 and 2 <= len(self.layers) <= 25
                and all(l['cin'] == 128 and l['cout'] == 128 for l in self.layers[1:])
                and self.layers[1]['skip'] is None):
            tail = self.layers[1:]
            wst = torch.stack([l['w'] for l in tail]).contiguous()
            bst = torch.stack([l['b'] for l in tail]).contiguous()
            relu_mask = res_mask = 0
            for i, l in enumerate(tail):
                l['w'], l['b'] = wst[i], bst[i]
                relu_mask |= int(bool(l['relu'])) << i
                res_mask |= int(l['skip'] is not None) << i
            self.trunk_small = dict(w=wst, b=bst, n=len(tail), relu_mask=relu_mask, res_mask=res_mask,
                                    b_host=np.ascontiguousarray(bst.float().cpu().numpy().reshape(-1)))
        # fused encoder + stem (rz_net_stem.cu): weight [cout][k = tap*4 + plane], k padded to 64
        conv0 = m.trunk_layers()[0][0]
        if self.mode != 'tc32':
            self.stem = None
        if self.mode == 'tc32':
            pass
        elif self.game_type == L.GAME_GO:
            # fused GoEnv.observe + stem (rz_net_stem.cu): weight [cout][k = tap*17 + plane], k padded to 192
            if conv0.in_channels != 17 or m.trunk_layers()[0][1] is not None:
                raise ValueError('the Go stem takes the 17 planes of GoEnv.observe (go_env.py:156-166)')
            w0, b0 = _fold_bn(conv0, None)
            ws = torch.zeros(128, 192, dtype=torch.float64, device=w0.device)
            ws[:, :153] = w0.permute(0, 2, 3, 1).reshape(128, 153)    # [cout][kh][kw][plane]
            self.stem = dict(w=ws.to(torch.bfloat16).contiguous().to(dev), b=b0.float().contiguous().to(dev),
                             relu=bool(m.trunk_layers()[0][3]))
        elif self.mode == 'tc' and conv0.in_channels == 4 and m.trunk_layers()[0][1] is None:
            w0, b0 = _fold_bn(conv0, None)
            c0 = w0.shape[0]
            ws = torch.zeros(128, 64, dtype=torch.float64, device=w0.device)
            ws[:c0, :36] = w0.permute(0, 2, 3, 1).reshape(c0, 36)     # [cout][kh][kw][plane], cout padded to 128
            bs = torch.zeros(128, dtype=b0.dtype, device=b0.device)
            bs[:c0] = b0
            self.stem = dict(w=ws.to(torch.bfloat16).contiguous().to(dev), b=bs.float().contiguous().to(dev),
                             relu=bool(m.trunk_layers()[0][3]))
        hw, AS = self.HW, self.AS
        f32 = torch.float32
        w1 = torch.cat([m.act_conv1.weight.detach().reshape(4, 128), m.val_conv1.weight.detach().reshape(2, 128)])
        b1 = torch.cat([m.act_conv1.bias.detach(), m.val_conv1.bias.detach()])
        pdev = m.act_fc1.weight.device
        wp = torch.zeros(4 * hw + 4, AS, dtype=f32, device=pdev)      # + 4 zero rows: the kernel prefetches past the end
        wp[:4 * hw, :self.A] = m.act_fc1.weight.detach().t().float()
        bp = torch.zeros(AS, dtype=f32, device=pdev)
        bp[:self.A] = m.act_fc1.bias.detach().float()
        self.heads = dict(
            w1x1=w1.float().contiguous().to(dev), b1x1=b1.float().contiguous().to(dev),
            wp=wp.contiguous().to(dev), bp=bp.to(dev),
            wv1=torch.cat([m.val_fc1.weight.detach().t().float(), torch.zeros(2, 64, device=pdev)]).contiguous().to(dev),
            bv1=m.val_fc1.bias.detach().float().contiguous().to(dev),
            wv2=m.val_fc2.weight.detach().reshape(64).float().contiguous().to(dev),
            bv2=m.val_fc2.bias.detach().float().contiguous().to(dev))
        if self.mode != 'f32':
            # both FCs as one K-major matrix over the padded feature row k' = f*P + y*S + x (rz_heads_desc.wtc_hi)
            S, Pp, A = self.S, self.P, self.A
            KP = (6 * Pp + 63) // 64 * 64
            wall = torch.zeros(AS + 64, KP, dtype=torch.float32, device=pdev)
            wpol = torch.zeros(A, 4, S, S, dtype=torch.float32, device=pdev)
            wpol[:, :, :self.H, :self.W] = m.act_fc1.weight.detach().float().reshape(A, 4, self.H, self.W)
            wall[:A, :4 * Pp] = wpol.reshape(A, 4 * Pp)
            wval = torch.zeros(64, 2, S, S, dtype=torch.float32, device=pdev)
            wval[:, :, :self.H, :self.W] = m.val_fc1.weight.detach().float().reshape(64, 2, self.H, self.W)
            wall[AS:AS + 64, 4 * Pp:6 * Pp] = wval.reshape(64, 2 * Pp)
            whi = wall.to(torch.bfloat16)
            wlo = (wall - whi.float()).to(torch.bfloat16)
            self.heads['wtc_hi'] = whi.contiguous().to(dev)
            self.heads['wtc_lo'] = wlo.contiguous().to(dev)
        # host copies of the 1x1 filters: they travel in the launch parameters of the fused last layer.  (The .cpu()
        # below also synchronises the stream: every pack kernel above has finished before a forward pass can be
        # launched, which the static-weights flag of the convolutions relies on -- include/rlzero_b200.h.)
        self.w1x1_host = np.ascontiguousarray(w1.float().cpu().numpy().reshape(-1))
        self.b1x1_host = np.ascontiguousarray(b1.float().cpu().numpy().reshape(-1))
        self.weights_version += 1
        hd = L.HeadsDesc()
        hd.board_size, hd.action_stride, hd.width, hd.n_actions = self.H, AS, self.W, self.A
        hd.row_stride = self.S if self.mode in ('tc', 'tc32') else 0
        for k, v in self.heads.items():
            setattr(hd, k, v.data_ptr())
        self.hdesc = hd

    @staticmethod
    def _split(w):
        """float64/float32 tensor -> (hi, lo) bf16 with hi + lo = w to 16 mantissa bits."""
        w = w.float()
        hi = w.to(torch.bfloat16)
        lo = (w - hi.float()).to(torch.bfloat16)
        return hi, lo

    def _pack_tc32(self):
        """Weights of the float32-accurate tensor-core path (mode 'tc32', see the class docstring); packed where the
        parameters live (the device after a training step)."""
        dev = self.device
        (c1, _, _, r1), (c2, _, _, r2), (c3, _, _, r3) = self.module.trunk_layers()
        pdev = c1.weight.device
        # conv1 through the fused stem: weight [128 rows][64 k], k = tap*4 + plane; rows 0..31 = high parts, rows
        # 32..63 = residues of the 32 filters
        w1 = c1.weight.detach().double().permute(0, 2, 3, 1).reshape(32, 36)
        hi, lo = self._split(w1)
        ws = torch.zeros(128, 64, dtype=torch.bfloat16, device=pdev)
        ws[:32, :36], ws[32:64, :36] = hi, lo
        b1 = torch.zeros(128, device=pdev)
        b1[:32] = c1.bias.detach().float()
        self.stem = dict(w=ws.contiguous().to(dev), b=b1.to(dev), relu=int(bool(r1)) | 2)
        # conv2: [tap][cout][cin = hi | lo | hi | lo of the 32 inputs] x [Whi | Whi | Wlo | Wlo] (all four partial
        # products: with the heads scaled up the lo*lo block is what keeps |dv| under 1e-5), N = 64 MMAs (flag 256): each
        # CTA of the pair supplies the first 32 rows of its weight tiles, so output channels 0..31 sit in rows 0..31 and
        # 32..63 in rows 64..95
        w2 = c2.weight.detach().double().permute(2, 3, 0, 1).reshape(9, 64, 32)
        hi, lo = self._split(w2)
        wt = torch.zeros(9, 128, 128, dtype=torch.bfloat16, device=pdev)
        for rows, sl in ((slice(0, 32), slice(0, 32)), (slice(64, 96), slice(32, 64))):
            wt[:, rows, 0:32], wt[:, rows, 32:64], wt[:, rows, 64:96], wt[:, rows, 96:128] = (
                hi[:, sl], hi[:, sl], lo[:, sl], lo[:, sl])
        b2 = torch.zeros(128, device=pdev)
        b2[:64] = c2.bias.detach().float()
        # conv3: [tap][cout 128][cin = Whi (64) | Wlo (64)], three products per tap in the kernel
        w3 = c3.weight.detach().double().permute(2, 3, 0, 1).reshape(9, 128, 64)
        hi, lo = self._split(w3)
        wt3 = torch.cat([hi, lo], dim=2).contiguous()
        self.layers = [dict(w=None, b=None, cin=64, cout=128, skip=None, relu=bool(r1)),      # the stem
                       dict(w=wt.contiguous().to(dev), b=b2.to(dev), cin=128, cout=128, skip=None, relu=bool(r2)),
                       dict(w=wt3.to(dev), b=c3.bias.detach().float().contiguous().to(dev), cin=128, cout=128,
                            skip=None, relu=bool(r3))]

    def _alloc(self, n):
        if self._route(n) == 'batched' and self.scratch is None:
            # [2][pairs][chunk][256][128] bf16, zeroed: the batched trunk keeps its pad rows zero
            pairs = (self.n_ctas or 148) // 2
            self.scratch = torch.zeros(2 * pairs * self.trunk_chunk * 256, 128, dtype=torch.bfloat16, device=self.device)
        if n <= self.max_batch:
            return
        dev = self.device
        if self.max_batch:
            # a captured wave graph holds the old buffers' addresses by value: growing them invalidates it, exactly
            # like repacked weights do, so the same version word makes every holder re-capture
            self.weights_version += 1
        self.max_batch = n
        if self.mode in ('tc', 'tc32'):
            bf = torch.bfloat16
            rows = (n * self.P + 255) // 256 * 256          # the convolutions work on pairs of 128-row tiles
            self.bufs = [torch.zeros(rows, 128, dtype=bf, device=dev) for _ in range(2)]
            self.feat = torch.zeros(n, 6, self.P, dtype=torch.float32, device=dev)
        else:
            cmax = max(max(l['cin'], l['cout']) for l in self.layers)
            self.act0 = torch.zeros(n, self.HW, self.layers[0]['cin'], dtype=torch.float32, device=dev)
            self.bufs = [torch.zeros(n, self.HW, cmax, dtype=torch.float32, device=dev) for _ in range(3)]
        self.logp = torch.zeros(n, self.AS, dtype=torch.float32, device=dev)
        self.value = torch.zeros(n, dtype=torch.float32, device=dev)

    # ------------------------------------------------------------------ forward
    def _gdesc(self, k=5):
        rs = self.S if self.mode in ('tc', 'tc32') else 0
        if self.game_type == L.GAME_GO:
            return L.GameDesc(self.H, 1, self.A, self.AS, self.W, self.game_type, 0.0, 0, rs)
        return L.GameDesc(self.H, min(k, max(self.H, self.W)), self.A, self.AS, self.W, self.game_type, 0.0, 0, rs)

    def _tc_stem(self):
        """The fused encoder + first convolution (rz_net_stem.cu) that starts every tensor-core forward."""
        if self.stem is None:
            raise ValueError("mode 'tc' needs a first layer the fused stem takes: 4 input planes without BatchNorm, "
                             "or Go's 17 planes")
        return self.stem

    def _route(self, n):
        """How ``n`` boards run the trunk behind the stem: 'small' = one launch, one CTA pair per board
        (rz_net_trunk_small.cu: few boards, a sequential search evaluates ONE); 'batched' = one launch, CTA pairs carrying
        chunks of boards through every layer (rz_net_trunk_tc2.cu: a search wave's thousands of leaves); 'layers' = one
        launch per layer.  Both one-launch kernels need a layout they take and, in mode 'tc', the fused heads epilogue,
        which they always apply.  kernels_per_forward reads the same answer."""
        if self.trunk_small is None or not (self.mode == 'tc32' or self.fused_head):
            return 'layers'
        if n <= self.small_batch_max:
            return 'small'
        if self.mode == 'tc' and n >= self.batched_trunk_min:
            return 'batched'
        return 'layers'

    def _conv(self, layer, inp, res, out, n):
        """One 128 -> 128 trunk layer on the tensor cores.  The layer layout picks the kernel: rz_net_tc2.cu for
        stride 16, rz_net_tc3.cu otherwise (bit 1 of its `relu`, like flag 512 of tc2: static weights)."""
        s = L.stream_ptr()
        if self.S == 16:
            L.check(self.lib.rz_net_conv3x3_tc2(L.ptr(inp), L.ptr(layer['w']), L.ptr(layer['b']), L.ptr(res),
                                                L.ptr(out), n, self.H, self.W, layer['cin'], int(layer['relu']), 2,
                                                self.conv_flags, self.n_ctas, s), 'rz_net_conv3x3_tc2')
        else:
            L.check(self.lib.rz_net_conv3x3_tc3(L.ptr(inp), L.ptr(layer['w']), L.ptr(layer['b']), L.ptr(res),
                                                L.ptr(out), n, self.H, self.W, self.S, int(layer['relu']) | 2,
                                                self.n_ctas, s), 'rz_net_conv3x3_tc3')

    def _conv_head(self, layer, inp, res, n):
        """``_conv`` of the last trunk layer with the heads' 1x1 convolutions in its epilogue: writes ``self.feat``."""
        s = L.stream_ptr()
        w1p = self.w1x1_host.ctypes.data_as(C.c_void_p)
        b1p = self.b1x1_host.ctypes.data_as(C.c_void_p)
        if self.S == 16:
            L.check(self.lib.rz_net_conv3x3_tc2_head_ex(
                L.ptr(inp), L.ptr(layer['w']), L.ptr(layer['b']), L.ptr(res), n, self.H, self.W, layer['cin'],
                int(layer['relu']), 512, w1p, b1p, L.ptr(self.feat), self.n_ctas, s), 'rz_net_conv3x3_tc2_head_ex')
        else:
            L.check(self.lib.rz_net_conv3x3_tc3_head(
                L.ptr(inp), L.ptr(layer['w']), L.ptr(layer['b']), L.ptr(res), n, self.H, self.W, self.S,
                int(layer['relu']) | 2, w1p, b1p, L.ptr(self.feat), self.n_ctas, s), 'rz_net_conv3x3_tc3_head')

    def _trunk_and_heads(self, n, logp, value):
        s = L.stream_ptr()
        lib = self.lib
        if self.mode == 'f32':
            outs = self.bufs
            hist = []   # buffer index holding the output of layer i
            inp = self.act0
            for i, l in enumerate(self.layers):
                busy = {hist[-1]} if hist else set()
                if l['skip'] is not None:
                    busy.add(hist[l['skip']])
                dst = [j for j in range(3) if j not in busy][0]
                res = outs[hist[l['skip']]] if l['skip'] is not None else None
                L.check(lib.rz_net_conv3x3_f32(L.ptr(inp), L.ptr(l['w']), L.ptr(l['b']), L.ptr(res),
                                               L.ptr(outs[dst]), n, self.H, l['cin'], l['cout'],
                                               int(l['relu']), s), 'rz_net_conv3x3_f32')
                hist.append(dst)
                inp = outs[dst]
            L.check(lib.rz_net_heads(C.byref(self.hdesc), L.ptr(inp), L.ptr(logp), L.ptr(value), n, s), 'rz_net_heads')
            return
        # the tensor-core modes: trunk behind the stem (which wrote bufs[0]) -> head features in self.feat -> FC heads
        w1p = self.w1x1_host.ctypes.data_as(C.c_void_p)
        b1p = self.b1x1_host.ctypes.data_as(C.c_void_p)
        route = self._route(n)
        if route == 'small':
            # the whole trunk in one launch, one CTA pair per board (tc32: conv2 + conv3 + the 1x1 heads)
            ts = self.trunk_small
            if self.mode == 'tc32':
                L.check(lib.rz_net_trunk_small_ex(
                    L.ptr(self.bufs[0]), L.ptr(ts['w']), L.ptr(ts['b']), ts['n'], ts['relu_mask'], ts['res_mask'],
                    ts['n64_mask'], ts['split_in_mask'], ts['head_f32'], n, self.H, self.W, w1p, b1p,
                    L.ptr(self.feat), s), 'rz_net_trunk_small_ex')
            else:
                L.check(lib.rz_net_trunk_small(
                    L.ptr(self.bufs[0]), L.ptr(ts['w']), L.ptr(ts['b']), ts['n'], ts['relu_mask'], ts['res_mask'], n,
                    self.H, self.W, w1p, b1p, L.ptr(self.feat), s), 'rz_net_trunk_small')
        elif route == 'batched':
            ts = self.trunk_small
            L.check(lib.rz_net_trunk_tc2(
                L.ptr(self.bufs[0]), L.ptr(ts['w']), ts['b_host'].ctypes.data_as(C.c_void_p), ts['n'], ts['relu_mask'],
                ts['res_mask'], L.ptr(self.scratch), self.trunk_chunk, n, self.H, self.W, w1p, b1p, L.ptr(self.feat),
                self.n_ctas, s), 'rz_net_trunk_tc2')
        elif self.mode == 'tc32':
            # conv2 (one K = 128 pass, split output) and conv3 (three products per tap, fp32 features)
            l2, l3 = self.layers[1], self.layers[2]
            L.check(lib.rz_net_conv3x3_tc2(L.ptr(self.bufs[0]), L.ptr(l2['w']), L.ptr(l2['b']), None, L.ptr(self.bufs[1]),
                                           n, self.H, self.W, 128, int(l2['relu']), 2, 2 | 8 | 256 | 512, self.n_ctas, s),
                    'rz_net_conv3x3_tc2')
            L.check(lib.rz_net_conv3x3_tc2_head_ex(
                L.ptr(self.bufs[1]), L.ptr(l3['w']), L.ptr(l3['b']), None, n, self.H, self.W, 128, int(l3['relu']),
                16 | 32 | 512, w1p, b1p, L.ptr(self.feat), self.n_ctas, s), 'rz_net_conv3x3_tc2_head_ex')
        else:
            # ping-pong: the residual of a block is the buffer its second conv overwrites
            outs = self.bufs
            cur = 0   # index in outs holding the latest activation
            for i, l in enumerate(self.layers[1:], 1):
                # skip always refers to the activation two layers back = the other buffer
                res = outs[1 - cur] if l['skip'] is not None else None
                if self.fused_head and i == len(self.layers) - 1:
                    self._conv_head(l, outs[cur], res, n)
                    break
                self._conv(l, outs[cur], res, outs[1 - cur], n)
                cur = 1 - cur
            else:
                L.check(lib.rz_net_head_features(C.byref(self.hdesc), L.ptr(outs[cur]), L.ptr(self.feat), n, s),
                        'rz_net_head_features')
        L.check(lib.rz_net_heads_tc(C.byref(self.hdesc), L.ptr(self.feat), L.ptr(logp), L.ptr(value), n, s),
                'rz_net_heads_tc')

    def kernels_per_forward(self, n=None):
        """Kernel launches of one forward_boards call of ``n`` boards (for bench.py's gpu_launches)."""
        if n is not None and self._route(n) != 'layers':
            return 3                                        # stem, one-launch trunk + 1x1 heads, FC heads
        if self.mode == 'tc32':
            return 4                                        # stem, conv2, conv3 + 1x1 heads, FC heads
        if self.mode == 'f32':
            return 1 + len(self.layers) + 1                 # encode, convs, heads
        return len(self.layers) + (1 if self.fused_head else 2)   # stem + convs, [1x1 features +] FC heads

    def forward_boards(self, rows, meta, n, logp=None, value=None, hist=None):
        """Positions in the device board layout -> (logp [n][AS], value [n]) float32 tensors.
        ``hist``: the Go history planes [n][14][H] (required for Go)."""
        self._alloc(n)
        logp = self.logp if logp is None else logp
        value = self.value if value is None else value
        g = self._gdesc()
        if self.game_type == L.GAME_GO:
            st = self.stem
            if hist is None:
                raise ValueError('Go positions need their history planes (hist=)')
            L.check(self.lib.rz_net_stem_go_tc(C.byref(g), L.ptr(rows), L.ptr(hist), L.ptr(meta), L.ptr(st['w']),
                                               L.ptr(st['b']), L.ptr(self.bufs[0]), n, int(st['relu']), 0,
                                               L.stream_ptr()), 'rz_net_stem_go_tc')
        elif self.mode in ('tc', 'tc32'):
            st = self._tc_stem()
            L.check(self.lib.rz_net_stem_tc(C.byref(g), L.ptr(rows), L.ptr(meta), L.ptr(st['w']), L.ptr(st['b']),
                                            L.ptr(self.bufs[0]), n, int(st['relu']), 0, L.stream_ptr()),
                    'rz_net_stem_tc')
        else:
            L.check(self.lib.rz_gomoku_encode_nhwc_f32(C.byref(g), L.ptr(rows), L.ptr(meta), L.ptr(self.act0),
                                                       n, L.stream_ptr()), 'rz_gomoku_encode_nhwc_f32')
        self._trunk_and_heads(n, logp, value)
        return logp[:n], value[:n]

    def forward_planes(self, planes):
        """[n,4,H,W] float planes (current_state format) -> (logp [n][A], value [n]).  Used by
        AlphaZeroAgent.policy_value / predict (alphazero_agent.py:48-57,88-97)."""
        x = torch.as_tensor(planes, dtype=torch.float32, device=self.device)
        n = x.shape[0]
        self._alloc(n)
        if self.game_type == L.GAME_GO:
            st = self.stem
            xc = x.contiguous()
            g = self._gdesc()
            L.check(self.lib.rz_net_stem_go_tc_planes(C.byref(g), L.ptr(xc), L.ptr(st['w']), L.ptr(st['b']),
                                                      L.ptr(self.bufs[0]), n, int(st['relu']), 0, L.stream_ptr()),
                    'rz_net_stem_go_tc_planes')
        elif self.mode in ('tc', 'tc32'):
            # same kernel (and therefore bit-identical stem outputs) as forward_boards
            st = self._tc_stem()
            xc = x.contiguous()
            g = self._gdesc()
            L.check(self.lib.rz_net_stem_tc_planes(C.byref(g), L.ptr(xc), L.ptr(st['w']), L.ptr(st['b']),
                                                   L.ptr(self.bufs[0]), n, int(st['relu']), 0, L.stream_ptr()),
                    'rz_net_stem_tc_planes')
        else:
            self.act0[:n] = x.permute(0, 2, 3, 1).reshape(n, self.HW, 4)
        self._trunk_and_heads(n, self.logp, self.value)
        return self.logp[:n, :self.A], self.value[:n]

    def __call__(self, forest):
        """Evaluator protocol of engine.SearchForest.run_waves: evaluate the wave's leaves."""
        self.forward_boards(forest.leaf_rows, forest.leaf_meta, forest.n_leaves, forest.prior, forest.value,
                            hist=getattr(forest, 'leaf_hist', None))
