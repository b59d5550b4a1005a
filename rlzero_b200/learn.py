"""``NativeTrainer``: the training step of ``AlphaZeroAgent.learn``
(rlzero/games/gomoku/alphazero_agent.py:59-86) on the hand-written kernels of ``csrc/rz_learn.cu``.

    forward (activations saved) -> loss / entropy -> analytic backward -> Adam(weight_decay)

for the reference's own ``PolicyValueNet`` (policy_value_net.py:6-52) in float32: no autograd, no
cuDNN, no cuBLAS on the path.  The module stays the parameter container -- its parameters are re-pointed
at slices of ONE flat device buffer, so ``state_dict()``, ``save_model`` / ``restore`` and the inference
path's ``refresh_weights`` see every update, and Adam is a single launch over the flat buffer.  Gradients
and both Adam moments are flat buffers with the same offsets; ``optimizer_state_dict()`` hands them out in
``torch.optim.Adam``'s format (alphazero_agent.py:104-111 saves exactly that).

PyTorch is used for device memory only.  The checker is ``oracle/train_oracle.py`` (numpy float64, pinned
to autograd and to the live reference agent): ``tests/test_gpu_learn.py``.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L


class NativeTrainer(object):
    """The reference's PolicyValueNet (conv 4 -> 32 -> 64 -> 128, float32 on CUDA cores).  The heads, the loss, the
    flat parameter buffers and Adam are shared with ``ResNetTrainer`` (tensor-core trunk) through the ``_trunk_*``
    hooks."""

    def __init__(self, module, learning_rate=1e-3, weight_decay=1e-4, betas=(0.9, 0.999), eps=1e-8, device='cuda'):
        if not torch.cuda.is_available():
            raise L.NativeLibraryError('NativeTrainer needs a CUDA device (no CPU fallback)')
        self.lib = L.load()
        self.module = module
        self.device = torch.device(device)
        self.H = int(module.board_size)
        self.HW = self.H * self.H
        self.A = self.HW
        self.AS = (self.A + 31) // 32 * 32
        self.lr, self.wd, self.betas, self.eps = float(learning_rate), float(weight_decay), tuple(betas), float(eps)
        self.step = 0
        for n in ['act_conv1', 'act_fc1', 'val_conv1', 'val_fc1', 'val_fc2']:
            if not hasattr(module, n):
                raise ValueError('the native trainers need the reference heads (missing %s)' % n)
        self._check_module(module)
        # ---- one flat buffer for the parameters, in parameters() order (= torch.optim.Adam's param order)
        params = list(module.parameters())
        self.names = [n for n, _ in module.named_parameters()]
        sizes = [p.numel() for p in params]
        self.offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        n_total = int(self.offsets[-1])
        f32 = torch.float32
        self.flat = torch.empty(n_total, dtype=f32, device=self.device)
        self.grad = torch.zeros(n_total, dtype=f32, device=self.device)
        self.exp_avg = torch.zeros(n_total, dtype=f32, device=self.device)
        self.exp_avg_sq = torch.zeros(n_total, dtype=f32, device=self.device)
        for p, o in zip(params, self.offsets[:-1]):
            view = self.flat[int(o):int(o) + p.numel()].view(p.shape)
            view.copy_(p.data.to(self.device, f32))
            p.data = view                                   # the module's tensors ARE the flat buffer from here on
        self._views = {n: (self.flat[int(o):int(o) + s], self.grad[int(o):int(o) + s])
                       for n, o, s in zip(self.names, self.offsets[:-1], sizes)}
        self._shapes = {n: tuple(p.shape) for n, p in zip(self.names, params)}
        self.zero_bias = torch.zeros(128, dtype=f32, device=self.device)
        self.B = 0
        self._init_trunk()
        self._repack()

    # ------------------------------------------------------------------ the stock trunk (float32, CUDA cores)
    def _check_module(self, module):
        for n in ['conv1', 'conv2', 'conv3']:
            if not hasattr(module, n):
                raise ValueError('NativeTrainer trains the reference PolicyValueNet (missing %s)' % n)
        self.chan = [(module.conv1.in_channels, module.conv1.out_channels),
                     (module.conv2.in_channels, module.conv2.out_channels),
                     (module.conv3.in_channels, module.conv3.out_channels)]
        if self.chan != [(4, 32), (32, 64), (64, 128)]:
            raise ValueError('NativeTrainer trains the 4 -> 32 -> 64 -> 128 trunk of the reference')

    use_tc_wgrad = True        # False: the float32 CUDA-core weight-gradient kernel (any board size)
    use_tc_trunk = False       # True ('native_tc'): forward AND data-gradient convolutions on the tensor cores too, on
                               # 16-mantissa-bit pairs: 3x faster at batch 512.  Forward within 1e-5 as before; the
                               # gradients within ~1e-3..1e-2 of the float64 oracle instead of 1e-5 (ReLU masks of
                               # pre-activations within 2e-6 of zero flip) -- tighter than PyTorch's default TF32.
                               # With the oracle's ReLU masks pinned to the device's, the gradients are within 1.9e-5
                               # of their largest entry on a B200 (act_fc1.weight: up to 2.6e-4 when almost no policy
                               # feature is positive, the cost of 16-bit weights; tests/test_gpu_learn_split.py)

    def _init_trunk(self):
        f32 = torch.float32
        # packed convolution weights (forward and data-gradient layouts), refreshed after every update
        self.wf = [torch.empty(9 * ci * co, dtype=f32, device=self.device) for ci, co in self.chan]
        self.wb = [torch.empty(9 * ci * co, dtype=f32, device=self.device) for ci, co in self.chan]

    def _repack(self):
        s = L.stream_ptr()
        for i, (ci, co) in enumerate(self.chan):
            L.check(self.lib.rz_learn_pack_conv(L.ptr(self._p('conv%d.weight' % (i + 1))), L.ptr(self.wf[i]),
                                                L.ptr(self.wb[i]), ci, co, s), 'rz_learn_pack_conv')
        if self.H <= 15 and self.use_tc_trunk:
            self._repack_tc()

    @staticmethod
    def _split(w):
        w = w.float()
        hi = w.to(torch.bfloat16)
        return hi, (w - hi.float()).to(torch.bfloat16)

    def _repack_tc(self):
        """bf16 (high, low) weight tiles of the float32-accurate tensor-core trunk (the layouts of NativeForward's mode
        'tc32' for the forward pass; mirrored taps and swapped channel roles for the data gradients)."""
        dev, bf = self.device, torch.bfloat16
        w1 = self._p('conv1.weight').view(32, 4, 3, 3).double().permute(0, 2, 3, 1).reshape(32, 36)
        hi, lo = self._split(w1)
        ws = torch.zeros(128, 64, dtype=bf, device=dev)
        ws[:32, :36], ws[32:64, :36] = hi, lo
        b1 = torch.zeros(128, device=dev)
        b1[:32] = self._p('conv1.bias')
        w2 = self._p('conv2.weight').view(64, 32, 3, 3).double()
        hi, lo = self._split(w2.permute(2, 3, 0, 1).reshape(9, 64, 32))                  # [tap][co][ci]
        wt2 = torch.zeros(9, 128, 128, dtype=bf, device=dev)
        for rows, sl in ((slice(0, 32), slice(0, 32)), (slice(64, 96), slice(32, 64))):     # N = 64 MMAs (flag 256)
            wt2[:, rows, 0:32], wt2[:, rows, 32:64], wt2[:, rows, 64:96], wt2[:, rows, 96:128] = (
                hi[:, sl], hi[:, sl], lo[:, sl], lo[:, sl])
        b2 = torch.zeros(128, device=dev)
        b2[:64] = self._p('conv2.bias')
        w3 = self._p('conv3.weight').view(128, 64, 3, 3).double()
        hi, lo = self._split(w3.permute(2, 3, 0, 1).reshape(9, 128, 64))
        wt3 = torch.cat([hi, lo], dim=2).contiguous()
        # data gradients: wT[8 - tap][ci][co] = w[co][ci][tap]; conv3 in two passes over the halves of its 128 output
        # channels (the kernel's K is 128 = [hi 64 | lo 64] of one half), conv2 in one
        flip = lambda w: torch.flip(w.permute(2, 3, 1, 0).reshape(9, w.shape[1], w.shape[0]), dims=[0])   # [8-tap][ci][co]
        w3t = flip(w3)                                                                   # [9][64 ci][128 co]
        d3 = []
        for h in range(2):
            hi, lo = self._split(w3t[:, :, 64 * h:64 * h + 64])
            t = torch.zeros(9, 128, 128, dtype=bf, device=dev)
            t[:, :64, :64], t[:, :64, 64:] = hi, lo
            d3.append(t.contiguous())
        hi, lo = self._split(flip(w2))                                                   # [9][32 ci][64 co]
        d2 = torch.zeros(9, 128, 128, dtype=bf, device=dev)
        d2[:, :32, :64], d2[:, :32, 64:] = hi, lo
        self.tcw = dict(stem=ws.contiguous(), b1=b1, w2=wt2.contiguous(), b2=b2, w3=wt3,
                        b3=self._p('conv3.bias'), d3=d3, d2=d2.contiguous())

    def _alloc_trunk(self, B):
        z = lambda *shape: torch.zeros(*shape, dtype=torch.float32, device=self.device)
        HW = self.HW
        self.x = z(B, HW, 4)
        self.a = [z(B, HW, 32), z(B, HW, 64), z(B, HW, 128)]
        self.d = [z(B, HW, 32), z(B, HW, 64), z(B, HW, 128)]     # gradients at the activations
        self.a_last, self.d_last = self.a[2], self.d[2]
        # the float32-accurate tensor-core trunk: activations as bf16 pair tiles, conv3's output and the data gradients
        # as float32 tiles
        self.tc = None
        if self.H <= 15 and self.use_tc_trunk and self.use_tc_wgrad:
            bft = lambda: torch.zeros(B * 256, 128, dtype=torch.bfloat16, device=self.device)
            f32t = lambda: torch.zeros(B * 256, 128, dtype=torch.float32, device=self.device)
            self.tc = dict(T1=bft(), T2=bft(), X0=bft(), XP=bft(), A3=f32t(), P1=f32t(), P2=f32t())
            self.gdesc = L.GameDesc(self.H, min(5, self.H), self.HW, self.AS, self.H, L.GAME_GOMOKU, 0.0, 0, 16)
        # operands of the tensor-core weight gradient: one [hi | lo] input tile, the high and the low gradient tile
        self.wg_tiles = None
        if self.H <= 15 and self.use_tc_wgrad:
            bf = torch.bfloat16
            self.wg_tiles = [torch.zeros(B * 256, 128, dtype=bf, device=self.device) for _ in range(3)]
            self.dw_a = torch.zeros(128 * 128 * 9, dtype=torch.float32, device=self.device)
            self.dw_b = torch.zeros(128 * 128 * 9, dtype=torch.float32, device=self.device)

    def _tc_conv(self, inp, w, bias, out, relu, flags):
        L.check(self.lib.rz_net_conv3x3_tc2(L.ptr(inp), L.ptr(w), L.ptr(bias), None, L.ptr(out), self.B, self.H, self.H, 128,
                                            int(relu), 2, flags, 0, L.stream_ptr()), 'rz_net_conv3x3_tc2')

    def _trunk_forward_tc(self, st):
        """The three convolutions on the tensor cores at float32-level accuracy (mode 'tc32' of the inference path):
        split stem -> one-pass conv2 with split output -> three-product conv3 with float32 output."""
        lib, s, B, H, t, w = self.lib, L.stream_ptr(), self.B, self.H, self.tc, self.tcw
        self.planes = st
        L.check(lib.rz_net_stem_tc_planes(C.byref(self.gdesc), L.ptr(st), L.ptr(w['stem']), L.ptr(w['b1']), L.ptr(t['T1']), B,
                                          1 | 2, 0, s), 'rz_net_stem_tc_planes')
        self._tc_conv(t['T1'], w['w2'], w['b2'], t['T2'], True, 2 | 8 | 256)
        self._tc_conv(t['T2'], w['w3'], w['b3'], t['A3'], True, 2 | 16 | 64)
        L.check(lib.rz_learn_tile_f32_to_nhwc(L.ptr(t['A3']), L.ptr(self.a[2]), 128, B, H, H, s), 'rz_learn_tile_f32_to_nhwc')

    def _wgrad_pair(self, xt, dhi, dlo, ci, co, gw):
        scr, nscr, s = L.ptr(self.scratch), self.scratch.numel(), L.stream_ptr()
        L.check(self.lib.rz_learn_conv_wgrad_tc(L.ptr(xt), L.ptr(dhi), L.ptr(self.dw_a), scr, nscr, self.B, 0, s),
                'rz_learn_conv_wgrad_tc')
        L.check(self.lib.rz_learn_conv_wgrad_tc(L.ptr(xt), L.ptr(dlo), L.ptr(self.dw_b), scr, nscr, self.B, 0, s),
                'rz_learn_conv_wgrad_tc')
        da, db = self.dw_a.view(128, 128, 9), self.dw_b.view(128, 128, 9)
        torch.add(da[:co, :ci] + da[:co, ci:2 * ci], db[:co, :ci] + db[:co, ci:2 * ci], out=gw.view(co, ci, 9))

    def _trunk_backward_tc(self):
        lib, s, B, H, HW, t, w = self.lib, L.stream_ptr(), self.B, self.H, self.HW, self.tc, self.tcw
        xt, dhi, dlo = self.wg_tiles
        # conv3: ReLU mask in channels-last float32 (where the heads left the gradient), weight gradient against the
        # stored [hi | lo] tile of a2, bias gradient
        L.check(lib.rz_learn_relu_bwd(L.ptr(self.a[2]), L.ptr(self.d[2]), B * HW * 128, s), 'rz_learn_relu_bwd')
        L.check(lib.rz_learn_nhwc_to_tile_hilo(L.ptr(self.d[2]), 128, L.ptr(dhi), L.ptr(dlo), 1, B, H, H, s),
                'rz_learn_nhwc_to_tile_hilo')
        self._wgrad_pair(t['T2'], dhi, dlo, 64, 128, self._g('conv3.weight'))
        self._colsum(self.d[2], B * HW, 128, 128, self._g('conv3.bias'), slices=96)
        # data gradient of conv3 in two passes over the halves of its output channels, float32 out
        for h, out in ((0, t['P1']), (1, t['P2'])):
            L.check(lib.rz_learn_nhwc_to_tile_hilo_slice(L.ptr(self.d[2]), 128, 64 * h, 64, L.ptr(t['XP']), B, H, H, s),
                    'rz_learn_nhwc_to_tile_hilo_slice')
            self._tc_conv(t['XP'], w['d3'][h], self.zero_bias, out, False, 2 | 16 | 64)
        # dz2 = (P1 + P2) * (a2 > 0): float32 back into P1, [hi | lo] pair tile for the next data gradient, hi / lo tiles
        L.check(lib.rz_learn_tile_grad_mask_split(L.ptr(t['P1']), L.ptr(t['P2']), L.ptr(t['T2']), 64, L.ptr(t['XP']), L.ptr(dhi),
                                                  L.ptr(dlo), B, s), 'rz_learn_tile_grad_mask_split')
        self._wgrad_pair(t['T1'], dhi, dlo, 32, 64, self._g('conv2.weight'))
        self._colsum(t['P1'], B * 256, 64, 128, self._g('conv2.bias'), slices=96)
        # conv2's data gradient (one pass: 64 channels in = one [hi | lo] tile), then dz1 and conv1's gradients
        self._tc_conv(t['XP'], w['d2'], self.zero_bias, t['P2'], False, 2 | 16 | 64)
        L.check(lib.rz_learn_tile_grad_mask_split(L.ptr(t['P2']), None, L.ptr(t['T1']), 32, None, L.ptr(dhi), L.ptr(dlo), B, s),
                'rz_learn_tile_grad_mask_split')
        L.check(lib.rz_learn_planes_to_tile(L.ptr(self.planes), L.ptr(t['X0']), B, H, H, s), 'rz_learn_planes_to_tile')
        self._wgrad_pair(t['X0'], dhi, dlo, 4, 32, self._g('conv1.weight'))
        self._colsum(t['P2'], B * 256, 32, 128, self._g('conv1.bias'), slices=96)

    def _trunk_forward(self, st):
        if self.tc is not None:
            return self._trunk_forward_tc(st)
        L.check(self.lib.rz_learn_nchw_to_nhwc(L.ptr(st), L.ptr(self.x), self.B, 4, self.HW, L.stream_ptr()),
                'rz_learn_nchw_to_nhwc')
        inp = self.x
        for i, (ci, co) in enumerate(self.chan):
            self._conv(inp, self.wf[i], self._p('conv%d.bias' % (i + 1)), self.a[i], ci, co, True)
            inp = self.a[i]

    def _wgrad_tc_split(self, x, dz, ci, co, gw, gb):
        """The float32 weight gradient of a 3x3 convolution on the tensor cores: input and output gradient travel as
        bf16 (high, low) pairs (16 mantissa bits), two launches of the tcgen05 weight-gradient kernel form all four
        partial products in fp32 accumulators (a [hi | lo] input tile against the high and the low gradient tile).
        Boards up to 15x15; the CUDA-core kernel serves larger ones."""
        lib, s, B, H = self.lib, L.stream_ptr(), self.B, self.H
        xt, dhi, dlo = self.wg_tiles
        L.check(lib.rz_learn_nhwc_to_tile_hilo(L.ptr(x), ci, L.ptr(xt), None, 0, B, H, H, s), 'rz_learn_nhwc_to_tile_hilo')
        L.check(lib.rz_learn_nhwc_to_tile_hilo(L.ptr(dz), co, L.ptr(dhi), L.ptr(dlo), 1, B, H, H, s), 'rz_learn_nhwc_to_tile_hilo')
        scr, nscr = L.ptr(self.scratch), self.scratch.numel()
        L.check(lib.rz_learn_conv_wgrad_tc(L.ptr(xt), L.ptr(dhi), L.ptr(self.dw_a), scr, nscr, B, 0, s), 'rz_learn_conv_wgrad_tc')
        L.check(lib.rz_learn_conv_wgrad_tc(L.ptr(xt), L.ptr(dlo), L.ptr(self.dw_b), scr, nscr, B, 0, s), 'rz_learn_conv_wgrad_tc')
        da, db = self.dw_a.view(128, 128, 9), self.dw_b.view(128, 128, 9)
        # fixed order of the four partial products: (hi*hi + hi*lo) + (lo*hi + lo*lo)
        torch.add(da[:co, :ci] + da[:co, ci:2 * ci], db[:co, :ci] + db[:co, ci:2 * ci], out=gw.view(co, ci, 9))
        self._colsum(dz, B * self.HW, co, co, gb, slices=96)

    def _trunk_backward(self):
        if self.tc is not None:
            return self._trunk_backward_tc()
        # last layer first: ReLU mask, weight/bias gradient, data gradient
        lib, s, B, HW = self.lib, L.stream_ptr(), self.B, self.HW
        inputs = [self.x, self.a[0], self.a[1]]
        for i in (2, 1, 0):
            ci, co = self.chan[i]
            L.check(lib.rz_learn_relu_bwd(L.ptr(self.a[i]), L.ptr(self.d[i]), B * HW * co, s), 'rz_learn_relu_bwd')
            gw, gb = self._g('conv%d.weight' % (i + 1)), self._g('conv%d.bias' % (i + 1))
            if self.wg_tiles is not None:
                self._wgrad_tc_split(inputs[i], self.d[i], ci, co, gw, gb)
            else:
                L.check(lib.rz_learn_conv_wgrad(L.ptr(inputs[i]), L.ptr(self.d[i]), L.ptr(gw), L.ptr(gb), L.ptr(self.scratch),
                                                self.scratch.numel(), B, self.H, ci, co, s), 'rz_learn_conv_wgrad')
            if i > 0:
                self._conv(self.d[i], self.wb[i], self.zero_bias, self.d[i - 1], co, ci, False)

    # ------------------------------------------------------------------ plumbing
    def _p(self, name):
        return self._views[name][0]

    def _g(self, name):
        return self._views[name][1]

    def _alloc(self, B):
        if B == self.B:
            return
        dev, f32, HW, AS = self.device, torch.float32, self.HW, self.AS
        self.B = B
        z = lambda *shape: torch.zeros(*shape, dtype=f32, device=dev)
        self._alloc_trunk(B)
        self.feat, self.dfeat = z(B, 6, HW), z(B, 6, HW)
        self.logp, self.dlogits = z(B, AS), z(B, AS)
        self.h, self.dh = z(B, 64), z(B, 64)
        self.v, self.dpre2 = z(B), z(B)
        self.terms, self.loss3 = z(B, 3), z(3)
        self.pi, self.z = z(B, self.A), z(B)
        rows = B * HW
        n_scr = max(96 * 9 * 64 * 128, ((rows + 63) // 64 + 64) * 774, 96 * AS, 1024, 49 * 9 * 128 * 128,
                    self._trunk_scratch_floats())
        self.scratch = z(n_scr)

    def _trunk_scratch_floats(self):
        return 0

    def _sgemm(self, M, N, K, A, sam, sak, Bm, sbk, sbn, Cm, ldc, alpha=1.0, accumulate=False):
        L.check(self.lib.rz_learn_sgemm(M, N, K, L.ptr(A), sam, sak, L.ptr(Bm), sbk, sbn, L.ptr(Cm), ldc, float(alpha),
                                        int(accumulate), L.stream_ptr()), 'rz_learn_sgemm')

    def _colsum(self, t, rows, cols, ld, out, slices=32):
        L.check(self.lib.rz_learn_colsum(L.ptr(t), rows, cols, ld, L.ptr(out), 1.0, L.ptr(self.scratch), slices,
                                         L.stream_ptr()), 'rz_learn_colsum')

    def _conv(self, inp, w, b, out, ci, co, relu):
        L.check(self.lib.rz_net_conv3x3_f32(L.ptr(inp), L.ptr(w), L.ptr(b), None, L.ptr(out), self.B, self.H, ci, co,
                                            int(relu), L.stream_ptr()), 'rz_net_conv3x3_f32')

    # ------------------------------------------------------------------ the step
    def forward(self, states):
        """states [B,4,H,W] float32 device tensor -> (logp [B,AS], v [B]); activations are kept for backward()."""
        B = int(states.shape[0])
        self._alloc(B)
        s = L.stream_ptr()
        lib, HW, AS, A = self.lib, self.HW, self.AS, self.A
        st = states.to(self.device, torch.float32).contiguous()
        self._trunk_forward(st)
        # the two 1x1 head convolutions, stacked: rows 0..3 act_conv1, 4..5 val_conv1
        w1 = torch.cat([self._p('act_conv1.weight'), self._p('val_conv1.weight')])
        b1 = torch.cat([self._p('act_conv1.bias'), self._p('val_conv1.bias')])
        self._w1x1 = w1
        L.check(lib.rz_learn_head_feat_fwd(L.ptr(self.a_last), L.ptr(w1), L.ptr(b1), L.ptr(self.feat), B, HW, s),
                'rz_learn_head_feat_fwd')
        # logits = pf . Wp^T (pf = feat[b][0:4HW]), log_softmax
        self._sgemm(B, A, 4 * HW, self.feat, 6 * HW, 1, self._p('act_fc1.weight'), 1, 4 * HW, self.logp, AS)
        L.check(lib.rz_learn_logsoftmax(L.ptr(self.logp), L.ptr(self._p('act_fc1.bias')), B, A, AS, s),
                'rz_learn_logsoftmax')
        # hidden = relu(vf . Wv1^T + bv1) (vf = feat[b][4HW:6HW]), v = tanh(h . wv2 + bv2)
        vf = self.feat.view(-1)[4 * HW:]
        self._sgemm(B, 64, 2 * HW, vf, 6 * HW, 1, self._p('val_fc1.weight'), 1, 2 * HW, self.h, 64)
        L.check(lib.rz_learn_value_fwd(L.ptr(self.h), L.ptr(self._p('val_fc1.bias')), L.ptr(self._p('val_fc2.weight')),
                                       L.ptr(self._p('val_fc2.bias')), L.ptr(self.v), B, s), 'rz_learn_value_fwd')
        return self.logp, self.v

    def backward(self, mcts_probs, target_vs):
        """Loss, entropy and every parameter gradient (into ``self.grad``) for the batch of the last forward()."""
        B, HW, AS, A = self.B, self.HW, self.AS, self.A
        lib, s = self.lib, L.stream_ptr()
        self.pi.copy_(mcts_probs.to(self.device, torch.float32).reshape(B, -1)[:, :A])
        self.z.copy_(target_vs.to(self.device, torch.float32).reshape(B))
        L.check(lib.rz_learn_loss_bwd(L.ptr(self.logp), L.ptr(self.pi), A, L.ptr(self.v), L.ptr(self.z), L.ptr(self.h),
                                      L.ptr(self._p('val_fc2.weight')), L.ptr(self.dlogits), L.ptr(self.dpre2),
                                      L.ptr(self.dh), L.ptr(self.terms), L.ptr(self.loss3), L.ptr(self.scratch), B, A, AS,
                                      s), 'rz_learn_loss_bwd')
        vf = self.feat.view(-1)[4 * HW:]
        # value head: val_fc2 (weight [1][64], bias [1]), val_fc1 (weight [64][2HW])
        self._sgemm(1, 64, B, self.dpre2, 0, 1, self.h, 64, 1, self._g('val_fc2.weight'), 64)
        self._colsum(self.dpre2, B, 1, 1, self._g('val_fc2.bias'))
        self._sgemm(64, 2 * HW, B, self.dh, 1, 64, vf, 6 * HW, 1, self._g('val_fc1.weight'), 2 * HW)
        self._colsum(self.dh, B, 64, 64, self._g('val_fc1.bias'))
        # policy head: act_fc1 (weight [A][4HW])
        self._sgemm(A, 4 * HW, B, self.dlogits, 1, AS, self.feat, 6 * HW, 1, self._g('act_fc1.weight'), 4 * HW)
        self._colsum(self.dlogits, B, A, AS, self._g('act_fc1.bias'))
        # gradients at the head features: dpf = dlogits . Wp, dvf = dh . Wv1, then the ReLU mask of the 1x1 convolutions
        self._sgemm(B, 4 * HW, A, self.dlogits, AS, 1, self._p('act_fc1.weight'), 4 * HW, 1, self.dfeat, 6 * HW)
        dvf = self.dfeat.view(-1)[4 * HW:]
        self._sgemm(B, 2 * HW, 64, self.dh, 64, 1, self._p('val_fc1.weight'), 2 * HW, 1, dvf, 6 * HW)
        L.check(lib.rz_learn_relu_bwd(L.ptr(self.feat), L.ptr(self.dfeat), B * 6 * HW, s), 'rz_learn_relu_bwd')
        dw1 = torch.empty(6 * 128, dtype=torch.float32, device=self.device)
        db1 = torch.empty(6, dtype=torch.float32, device=self.device)
        L.check(lib.rz_learn_head_feat_bwd(L.ptr(self.dfeat), L.ptr(self.a_last), L.ptr(self._w1x1), L.ptr(self.d_last),
                                           L.ptr(dw1), L.ptr(db1), L.ptr(self.scratch), self.scratch.numel(), B, HW, s),
                'rz_learn_head_feat_bwd')
        self._g('act_conv1.weight').copy_(dw1[:4 * 128])
        self._g('val_conv1.weight').copy_(dw1[4 * 128:])
        self._g('act_conv1.bias').copy_(db1[:4])
        self._g('val_conv1.bias').copy_(db1[4:])
        self._trunk_backward()
        return self.loss3

    def adam_step(self):
        self.step += 1
        L.check(self.lib.rz_learn_adam(L.ptr(self.flat), L.ptr(self.grad), L.ptr(self.exp_avg), L.ptr(self.exp_avg_sq),
                                       self.flat.numel(), self.lr, self.betas[0], self.betas[1], self.eps, self.wd,
                                       self.step, L.stream_ptr()), 'rz_learn_adam')
        self._repack()

    def learn(self, state_batch, mcts_probs, target_vs):
        """One training step; returns (loss, entropy) as Python floats (alphazero_agent.py:86)."""
        self.forward(state_batch)
        loss3 = self.backward(mcts_probs, target_vs)
        self.adam_step()
        vl, pl, ent = loss3.tolist()          # the one device -> host read of the step
        return vl + pl, ent

    # ------------------------------------------------------------------ views for callers and tests
    def grads(self):
        """{parameter name: gradient tensor in the state_dict's shape} (views of the flat gradient buffer)."""
        return {n: self._g(n).view(self._shapes[n]) for n in self.names}

    def optimizer_state_dict(self):
        """``torch.optim.Adam.state_dict()`` format (alphazero_agent.py:108-111 saves it)."""
        state = {}
        for i, n in enumerate(self.names):
            o, e = int(self.offsets[i]), int(self.offsets[i + 1])
            if self.step > 0:
                state[i] = {'step': torch.tensor(float(self.step)), 'exp_avg': self.exp_avg[o:e].view(self._shapes[n]).clone(),
                            'exp_avg_sq': self.exp_avg_sq[o:e].view(self._shapes[n]).clone()}
        group = {'lr': self.lr, 'betas': self.betas, 'eps': self.eps, 'weight_decay': self.wd, 'amsgrad': False,
                 'maximize': False, 'foreach': None, 'capturable': False, 'differentiable': False, 'fused': None,
                 'params': list(range(len(self.names)))}
        return {'state': state, 'param_groups': [group]}

    def load_optimizer_state_dict(self, sd):
        g = sd['param_groups'][0]
        self.lr, self.wd, self.eps = float(g['lr']), float(g['weight_decay']), float(g['eps'])
        self.betas = tuple(g['betas'])
        self.exp_avg.zero_()
        self.exp_avg_sq.zero_()
        self.step = 0
        for i, st in sd['state'].items():
            i = int(i)
            o, e = int(self.offsets[i]), int(self.offsets[i + 1])
            self.exp_avg[o:e].copy_(st['exp_avg'].reshape(-1))
            self.exp_avg_sq[o:e].copy_(st['exp_avg_sq'].reshape(-1))
            self.step = int(float(st['step']))

    def weights_changed(self):
        """Call after the module's parameters were written from outside (load_state_dict, a broadcast)."""
        self._repack()


class ResNetTrainer(NativeTrainer):
    """The same step for ``ResNetPolicyValueNet`` (stem conv3x3(P -> 128) + ReLU, N blocks of 2 x [conv3x3 +
    BatchNorm2d] + skip + ReLU, the reference heads) with the trunk on the tensor cores (``csrc/rz_learn_tc.cu``):
    bf16 activations / gradients in the padded position layout, forward convolution and data gradient through the
    inference path's convolution, weight gradient through the tcgen05 MN-major kernel, BatchNorm in training mode with
    float32 statistics.  Heads, loss and Adam are the float32 kernels of ``NativeTrainer`` (the trunk output crosses
    into float32 channels-last once per step).

    Square boards up to 19x19 in two forms: 4 input planes (GomokuEnv.current_state) with H*W actions, or 17 planes
    (GoEnv.observe) with H*W + 1 actions, the last one the pass.  The layout follows the board: row stride S = 16 up to
    15x15 (``rz_net_conv3x3_tc2``, [B*256][128] tensors) and S = 20 for 16x16 to 19x19 (``rz_net_conv3x3_tc3``,
    [round_up(B*400, 256)][128]).  The stem's forward is the inference path's fused stem fed from float32 planes
    (``rz_net_stem_tc_planes`` / ``rz_net_stem_go_tc_planes``)."""

    def _check_module(self, module):
        if not (hasattr(module, 'stem') and hasattr(module, 'blocks')):
            raise ValueError('ResNetTrainer trains ResNetPolicyValueNet')
        if not resnet_trainer_fits(module):
            raise ValueError('ResNetTrainer: square boards up to 19x19, with 4 input planes and H*W actions or 17 input '
                             'planes (Go) and H*W + 1 actions')
        self.in_planes = int(module.stem.in_channels)
        self.A = int(module.n_actions)               # policy outputs (the pass included); the heads read HW squares
        self.AS = (self.A + 31) // 32 * 32
        self.S = 16 if self.H <= 15 else 20          # row stride of the padded layout
        self.n_blocks = len(module.blocks)

    def _init_trunk(self):
        dev, bf = self.device, torch.bfloat16
        self.w_stem = torch.empty(128 * (64 if self.in_planes == 4 else 192), dtype=bf, device=dev)
        n_conv = 2 * self.n_blocks
        self.wf = [torch.empty(9 * 128 * 128, dtype=bf, device=dev) for _ in range(n_conv)]
        self.wb = [torch.empty(9 * 128 * 128, dtype=bf, device=dev) for _ in range(n_conv)]
        self.stats = [torch.zeros(4 * 128, dtype=torch.float32, device=dev) for _ in range(n_conv)]
        self.dw_full = torch.zeros(128 * 128 * 9, dtype=torch.float32, device=dev)
        if self.in_planes == 17:
            self.gdesc = L.GameDesc(self.H, 1, self.A, self.AS, self.H, L.GAME_GO, 0.0, 0, self.S)
        else:
            self.gdesc = L.GameDesc(self.H, min(5, self.H), self.HW, self.AS, self.H, L.GAME_GOMOKU, 0.0, 0, self.S)
        self.conv_names = []
        for i in range(self.n_blocks):
            self.conv_names += [('blocks.%d.conv1' % i, 'blocks.%d.bn1' % i), ('blocks.%d.conv2' % i, 'blocks.%d.bn2' % i)]
        self.bns = []
        for blk in self.module.blocks:
            self.bns += [blk.bn1, blk.bn2]

    def _repack(self):
        s = L.stream_ptr()
        L.check(self.lib.rz_learn_pack_stem_tc_ex(L.ptr(self._p('stem.weight')), self.in_planes, L.ptr(self.w_stem), s),
                'rz_learn_pack_stem_tc_ex')
        for j, (cn, _) in enumerate(self.conv_names):
            L.check(self.lib.rz_learn_pack_conv_tc(L.ptr(self._p(cn + '.weight')), L.ptr(self.wf[j]), L.ptr(self.wb[j]), s),
                    'rz_learn_pack_conv_tc')

    def _trunk_scratch_floats(self):
        return max(49 * 9 * 128 * 128, 148 * 4 * 256 + 256, 96 * 9 * 4 * 128)

    def _alloc_trunk(self, B):
        dev, bf, HW = self.device, torch.bfloat16, self.HW
        rows = (B * self.S * self.S + 255) // 256 * 256
        t = lambda: torch.zeros(rows, 128, dtype=bf, device=dev)
        n_conv = 2 * self.n_blocks
        self.act0 = t()                                  # stem output
        self.ybuf = [t() for _ in range(n_conv)]         # raw convolution outputs (inputs of the BatchNorms)
        self.abuf = [t() for _ in range(n_conv)]         # activations after BatchNorm (+ skip) + ReLU
        self.gbuf = [t() for _ in range(4)]              # gradient ping-pong
        z = lambda *shape: torch.zeros(*shape, dtype=torch.float32, device=dev)
        self.x = z(B, HW, 4)
        self.a_last, self.d_last = z(B, HW, 128), z(B, HW, 128)
        self.planes = None

    def _tc_conv(self, inp, w, bias, res, out):
        if self.S == 16:
            L.check(self.lib.rz_net_conv3x3_tc2(L.ptr(inp), L.ptr(w), L.ptr(bias), L.ptr(res), L.ptr(out), self.B, self.H,
                                                self.H, 128, 0, 2, 2, 0, L.stream_ptr()), 'rz_net_conv3x3_tc2')
        else:
            L.check(self.lib.rz_net_conv3x3_tc3(L.ptr(inp), L.ptr(w), L.ptr(bias), L.ptr(res), L.ptr(out), self.B, self.H,
                                                self.H, self.S, 0, 0, L.stream_ptr()), 'rz_net_conv3x3_tc3')

    def _trunk_forward(self, st):
        lib, s, B, H, S = self.lib, L.stream_ptr(), self.B, self.H, self.S
        self.planes = st
        stem = lib.rz_net_stem_go_tc_planes if self.in_planes == 17 else lib.rz_net_stem_tc_planes
        L.check(stem(C.byref(self.gdesc), L.ptr(st), L.ptr(self.w_stem), L.ptr(self._p('stem.bias')), L.ptr(self.act0), B, 1,
                     0, s), 'rz_net_stem_go_tc_planes' if self.in_planes == 17 else 'rz_net_stem_tc_planes')
        cur = self.act0
        for j, (cn, bn) in enumerate(self.conv_names):
            self._tc_conv(cur if j % 2 == 0 else self.abuf[j - 1], self.wf[j], self._p(cn + '.bias'), None, self.ybuf[j])
            m = self.bns[j]
            L.check(lib.rz_learn_bn_forward_ex(L.ptr(self.ybuf[j]), L.ptr(cur) if j % 2 == 1 else None, L.ptr(self.abuf[j]),
                                               L.ptr(self._p(bn + '.weight')), L.ptr(self._p(bn + '.bias')),
                                               L.ptr(m.running_mean), L.ptr(m.running_var), float(m.eps),
                                               float(m.momentum if m.momentum is not None else 0.1), L.ptr(self.stats[j]),
                                               L.ptr(self.scratch), B, H, H, S, s), 'rz_learn_bn_forward_ex')
            if j % 2 == 1:
                cur = self.abuf[j]
                m.num_batches_tracked += 1
            else:
                m.num_batches_tracked += 1
        self.trunk_out = cur
        L.check(lib.rz_learn_tile_to_nhwc_ex(L.ptr(cur), L.ptr(self.a_last), B, H, H, S, s), 'rz_learn_tile_to_nhwc_ex')

    def _trunk_backward(self):
        lib, s, B, H, S = self.lib, L.stream_ptr(), self.B, self.H, self.S
        g, dy, dz, da = self.gbuf
        L.check(lib.rz_learn_nhwc_to_tile_ex(L.ptr(self.d_last), L.ptr(g), B, H, H, S, s), 'rz_learn_nhwc_to_tile_ex')
        scr, nscr = L.ptr(self.scratch), self.scratch.numel()
        for i in reversed(range(self.n_blocks)):
            j1, j2 = 2 * i, 2 * i + 1
            block_in = self.act0 if i == 0 else self.abuf[j1 - 1]
            (c1, b1), (c2, b2) = self.conv_names[j1], self.conv_names[j2]
            # second half of the block: BatchNorm2 + skip + ReLU, conv2
            L.check(lib.rz_learn_bn_backward_ex(L.ptr(g), L.ptr(self.abuf[j2]), L.ptr(self.ybuf[j2]), L.ptr(self.stats[j2]),
                                                L.ptr(self._g(b2 + '.weight')), L.ptr(self._g(b2 + '.bias')), L.ptr(dy),
                                                L.ptr(dz), scr, B, H, H, S, s), 'rz_learn_bn_backward_ex')
            L.check(lib.rz_learn_conv_wgrad_tc_ex(L.ptr(self.abuf[j1]), L.ptr(dy), L.ptr(self._g(c2 + '.weight')), scr, nscr, B,
                                                  S, 0, s), 'rz_learn_conv_wgrad_tc_ex')
            self._tc_conv(dy, self.wb[j2], self.zero_bias, None, da)
            # first half: BatchNorm1 + ReLU, conv1; the skip gradient dz joins the data gradient
            L.check(lib.rz_learn_bn_backward_ex(L.ptr(da), L.ptr(self.abuf[j1]), L.ptr(self.ybuf[j1]), L.ptr(self.stats[j1]),
                                                L.ptr(self._g(b1 + '.weight')), L.ptr(self._g(b1 + '.bias')), L.ptr(dy), None,
                                                scr, B, H, H, S, s), 'rz_learn_bn_backward_ex')
            L.check(lib.rz_learn_conv_wgrad_tc_ex(L.ptr(block_in), L.ptr(dy), L.ptr(self._g(c1 + '.weight')), scr, nscr, B, S,
                                                  0, s), 'rz_learn_conv_wgrad_tc_ex')
            self._tc_conv(dy, self.wb[j1], self.zero_bias, dz, g)
            # a convolution bias in front of a BatchNorm has no gradient (the batch mean absorbs it)
            self._g(c1 + '.bias').zero_()
            self._g(c2 + '.bias').zero_()
        # stem: ReLU mask on the tile; its weight gradient through the same tensor-core kernel with the observation
        # planes as channels 0..P-1 of a tile (0/1 values: exact), its bias gradient = the column sums of dz
        P = self.in_planes
        L.check(lib.rz_learn_relu_bwd_bf16_ex(L.ptr(g), L.ptr(self.act0), L.ptr(dy), B, S, s), 'rz_learn_relu_bwd_bf16_ex')
        L.check(lib.rz_learn_planes_to_tile_ex(L.ptr(self.planes), P, L.ptr(da), B, H, H, S, s), 'rz_learn_planes_to_tile_ex')
        L.check(lib.rz_learn_conv_wgrad_tc_ex(L.ptr(da), L.ptr(dy), L.ptr(self.dw_full), scr, nscr, B, S, 0, s),
                'rz_learn_conv_wgrad_tc_ex')
        self._g('stem.weight').view(128, P, 9).copy_(self.dw_full.view(128, 128, 9)[:, :P, :])
        L.check(lib.rz_learn_tile_colsum_ex(L.ptr(dy), L.ptr(self._g('stem.bias')), scr, B, S, s), 'rz_learn_tile_colsum_ex')


def resnet_trainer_fits(module):
    """Whether ``ResNetTrainer`` trains ``module``: square boards up to 19x19, 4 planes with H*W actions or 17 (Go) with
    H*W + 1."""
    H = int(module.board_size)
    W = int(getattr(module, 'board_width', H))
    P, A = int(module.stem.in_channels), int(module.n_actions)
    return W == H and H <= 19 and ((P == 4 and A == H * H) or (P == 17 and A == H * H + 1))


def make_trainer(module, tc_trunk=False, requested=False, **kw):
    """The native trainer that fits ``module``, or None (the caller then falls back to its autograd path).
    ``tc_trunk``: the reference's own network with the whole trunk on the tensor cores (``NativeTrainer.use_tc_trunk``).
    ``requested``: the caller asked for a native trainer.  Without it only the shapes that have trained natively by
    default all along get one (4 planes, boards up to 15x15); Go networks and 16x16 .. 19x19 boards stay on autograd
    unless asked, because the bf16 trunk's value error on trained networks (DESIGN section 3.4) is not measured there."""
    from .games.gomoku.policy_value_net import PolicyValueNet, ResNetPolicyValueNet
    if type(module) is PolicyValueNet:
        t = NativeTrainer(module, **kw)
        t.use_tc_trunk = bool(tc_trunk)
        t._repack()
        return t
    if isinstance(module, ResNetPolicyValueNet) and resnet_trainer_fits(module):
        if requested or (module.board_size <= 15 and module.stem.in_channels == 4):
            return ResNetTrainer(module, **kw)
    return None
