"""GPU tests of the float32-accurate tensor-core training step of the reference's own network (``NativeTrainer`` with
``use_tc_trunk = True``, ``AlphaZeroAgent(trainer='native_tc')``), layer by layer and end to end, against float64.

Every operand of that step is a bf16 (high, low) pair, 16 mantissa bits.  Against the true oracle
(tests/test_gpu_learn.py) its gradients can only be held to 2e-2: a pre-activation within rounding of zero may fall on
the other side of the ReLU on the device, and each such flip is a 100 % error on that element.  A product dropped from
the pairs (hi * Wlo, lo * Whi) costs about 2^-9 of the affected terms -- well inside 2e-2.  These tests separate the
two:

  a. the conversion kernels between float32 and pair tiles equal their definitions written in torch, bit for bit;
  b. each forward layer, with the weights packed by ``NativeTrainer._repack_tc``, against a float64 convolution of the
     values the kernel consumed: its input tile's hi + lo, and Whi + Wlo split here from the float32 weights;
  c. each data-gradient pass against ``_conv3x3_backward`` of oracle/train_oracle.py in float64;
  d. the whole step against ``train_oracle.loss_and_grads`` with the ReLU masks pinned to those the device produced,
     so that the device and the reference differ by rounding alone;
  e. mutation controls: one partial product dropped from the packed weights or from an input tile, and the check of
     b, c or d fails by a wide margin.

Errors are relative to the reference tensor's largest entry, max |dev - ref| / max |ref|; the gradients of d are also
held in ||dev - ref|| / ||ref||, which sees a small error spread over the whole tensor.  Every error is printed
(``pytest -s``).  Each bound is at least 3x the worst clean error measured on an NVIDIA B200 (1000 W power limit) over
every shape below, and the smallest error of a mutation is at least 3x the bound it is checked against; the figures are
beside each bound.  The shapes put boards of 3, 6, 9 and 15 squares a side in the 16-stride tile layout and cover
batches of 1, 8, 48 and 130 boards.
"""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

BOARDS = (3, 6, 9, 15)
BATCHES = (1, 8, 48, 130)
SHAPES = [(3, 130), (6, 8), (9, 48), (15, 1), (15, 48)]

# Bounds.  In brackets: the worst clean error measured on an NVIDIA B200 (1000 W power limit) over SHAPES, then the
# smallest error of the mutations checked against that bound.
# b. forward layers, max |dev - ref| / max |ref|
BOUND_LAYER = {'stem': 2e-5,        # [5.4e-6 at 9x9 B=48]
               'conv2': 2e-5,       # [5.7e-6 at 3x3 B=130]
               'conv3': 2e-5}       # [4.2e-6 at 9x9 B=48; hi*Wlo dropped: 1.7e-3]
# c. data-gradient passes, max |dev - ref| / max |ref|
BOUND_DGRAD = 1.5e-5                # [4.0e-6, conv3 half 0 at 6x6 B=8; lo*Whi dropped: 1.5e-3]
# d. the whole step against the mask-pinned oracle, every gradient in two metrics, and the outputs
BOUND_GRAD_MAX = 6e-5               # max |dev - ref| / max |ref|  [1.9e-5, val_fc1.weight at 15x15 B=48; a data-gradient
                                    #                               hi*Wlo dropped: 1.5e-3]
BOUND_GRAD_L2 = 5e-5                # ||dev - ref|| / ||ref||      [1.6e-5, val_fc1.weight at 15x15 B=48; dropped: 1.5e-3]
# act_fc1.weight alone is held to 1e-3 [2.6e-4 in both metrics at 6x6 B=8].  The reason is measured, and it is not the
# kernels: in that batch 2 of the 1152 policy features are positive, the largest 4.3e-4, sums of conv3 outputs of order
# 1e-1 that nearly cancel.  The mode carries the convolution weights as Whi + Wlo, 16 mantissa bits, and in float64
# that substitution alone moves this gradient by 3.4e-4 of its largest entry (every other gradient by at most 7e-6).
# No mutation here reaches this tensor: the policy head runs in float32 on the CUDA cores.
BOUND_GRAD_OVERRIDE = {'act_fc1.weight': 1e-3}
BOUND_LOGP_V = 3e-6                 # log p and v, absolute        [7.6e-7]
BOUND_LOSS = 2e-6                   # loss and entropy, absolute   [4.6e-7]

SENTINEL = -7.25                    # fills the board past the last one: the kernels must leave it alone
BF16 = torch.bfloat16


def _lib():
    from rlzero_b200 import _lib as L
    return L, L.load()


def _split(x):
    """float32 -> its bf16 (high, low) pair: hi = bf16_rn(x), lo = bf16_rn(x - hi)."""
    hi = x.to(BF16)
    return hi, (x - hi.float()).to(BF16)


def _pair_value(x):
    """float64 value of the pair of float32 x: what a kernel fed with that pair consumes."""
    hi, lo = _split(x.float())
    return hi.double() + lo.double()


def _on_board(B, H):
    """bool [B*256]: the rows of the padded layout (row = board*256 + y*16 + x) that are board squares."""
    pos = torch.arange(256, device='cuda')
    return (((pos // 16) < H) & ((pos % 16) < H)).repeat(B)


def _rows(x, B, H):
    """[B, H*H, C] channels-last -> [B*256, C] in the padded layout, zero pad squares."""
    t = torch.zeros(B, 16, 16, x.shape[-1], dtype=x.dtype, device=x.device)
    t[:, :H, :H] = x.view(B, H, H, -1)
    return t.view(B * 256, -1)


def _board(t, B, H, c0, c1):
    """Channels c0..c1-1 of the board squares of a padded tile -> [B, c1 - c0, H, H]."""
    return t[:B * 256].view(B, 16, 16, -1)[:, :H, :H, c0:c1].permute(0, 3, 1, 2)


def _filled(B, dtype):
    """A [(B + 1) * 256, 128] tile: B boards for a kernel to write and one spare board of SENTINEL after them."""
    return torch.full(((B + 1) * 256, 128), SENTINEL, dtype=dtype, device='cuda')


def _assert_tail_untouched(t, B):
    assert (t[B * 256:].float() == SENTINEL).all(), 'a kernel wrote past its last board'


def _rand_f32(shape, g):
    """Random float32 over 30 binades with a quarter exact zeros, a quarter bf16 values (zero low part), both signs."""
    x = torch.randn(shape, generator=g, device='cuda')
    x = x * torch.exp2(torch.randint(-20, 10, shape, generator=g, device='cuda').float())
    sel = torch.randint(0, 4, shape, generator=g, device='cuda')
    x = torch.where(sel == 0, torch.zeros_like(x), x)
    return torch.where(sel == 1, x.to(BF16).float(), x)


def _rel(got, ref):
    return (got - ref).abs().max().item() / ref.abs().max().item()


def _assert_nearest_pair(hi, lo, what):
    """hi is the bf16 value nearest hi + lo: |lo| <= ulp(hi) / 2, and lo = 0 where hi = 0."""
    h, lo_ = hi.float(), lo.float()
    _, e = torch.frexp(h)                                   # |h| in [2^(e-1), 2^e): the bf16 spacing there is 2^(e-8)
    ok = torch.where(h == 0, lo_ == 0, lo_.abs() <= torch.ldexp(torch.ones_like(h), e - 9))
    assert ok.all(), (what, int((~ok).sum()))


# ---------------------------------------------------------------------------------------------- a. conversions, exact
@pytest.mark.parametrize('H', BOARDS)
@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('mode,Ch', [(0, 4), (0, 32), (0, 64), (1, 32), (1, 64), (1, 128)])
def test_nhwc_to_tile_hilo_is_the_pair_split(H, B, mode, Ch):
    """mode 0: tile_a = [hi C | lo C | 0]; mode 1: tile_a = [hi C | 0], tile_b = [lo C | 0]; pad squares zero."""
    L, lib = _lib()
    g = torch.Generator(device='cuda').manual_seed(1000 * H + 10 * B + Ch + mode)
    x = _rand_f32((B, H * H, Ch), g)
    a, b = _filled(B, BF16), _filled(B, BF16)
    L.check(lib.rz_learn_nhwc_to_tile_hilo(L.ptr(x), Ch, L.ptr(a), L.ptr(b), mode, B, H, H, L.stream_ptr()),
            'rz_learn_nhwc_to_tile_hilo')
    hi, lo = _split(x)
    want_a = torch.zeros(B * 256, 128, dtype=BF16, device='cuda')
    want_b = torch.zeros_like(want_a)
    want_a[:, :Ch] = _rows(hi, B, H)
    (want_a[:, Ch:2 * Ch] if mode == 0 else want_b[:, :Ch]).copy_(_rows(lo, B, H))
    assert torch.equal(a[:B * 256], want_a)
    _assert_tail_untouched(a, B)
    if mode == 1:
        assert torch.equal(b[:B * 256], want_b)
        _assert_tail_untouched(b, B)
    else:
        assert (b.float() == SENTINEL).all()                # mode 0 has no second tile
    assert (a[:B * 256][~_on_board(B, H)].float() == 0).all()


@pytest.mark.parametrize('H,B', SHAPES)
@pytest.mark.parametrize('offset', [0, 64])
def test_nhwc_to_tile_hilo_slice_is_the_pair_split_of_the_slice(H, B, offset):
    """The halves of conv3's output gradient (128 channels, offsets 0 and 64) as [hi 64 | lo 64] tiles."""
    L, lib = _lib()
    g = torch.Generator(device='cuda').manual_seed(100 * H + B + offset)
    x = _rand_f32((B, H * H, 128), g)
    t = _filled(B, BF16)
    L.check(lib.rz_learn_nhwc_to_tile_hilo_slice(L.ptr(x), 128, offset, 64, L.ptr(t), B, H, H, L.stream_ptr()),
            'rz_learn_nhwc_to_tile_hilo_slice')
    hi, lo = _split(x[..., offset:offset + 64].contiguous())
    assert torch.equal(t[:B * 256], torch.cat([_rows(hi, B, H), _rows(lo, B, H)], dim=1))
    _assert_tail_untouched(t, B)


@pytest.mark.parametrize('H,B', SHAPES)
@pytest.mark.parametrize('Ch', [32, 64])
@pytest.mark.parametrize('with_b,with_pair', [(True, True), (False, True), (True, False), (False, False)])
def test_tile_grad_mask_split_is_its_definition(H, B, Ch, with_b, with_pair):
    """g = (grad_a + grad_b) * (act_hi > 0) on channels < C, in float32: written back into grad_a (channels >= C keep
    their values), as hi / lo tiles [bf16(g) | 0], [bf16(g - hi) | 0] and as the pair tile [hi C | lo C | 0].  The
    mask reads the high part only (hi = 0 with lo > 0 is masked); pad rows, where the activation is zero, leave zero."""
    L, lib = _lib()
    g = torch.Generator(device='cuda').manual_seed(10 * H + B + Ch + 2 * with_b + with_pair)
    rows = B * 256
    on = _on_board(B, H)
    ga = torch.randn(rows, 128, generator=g, device='cuda')            # stale values everywhere, pad rows included
    gb = torch.randn(rows, 128, generator=g, device='cuda') if with_b else None
    act_hi = torch.randn(rows, Ch, generator=g, device='cuda').to(BF16)
    act_hi[torch.rand(rows, Ch, generator=g, device='cuda') < 0.3] = 0
    act_lo = (torch.rand(rows, Ch, generator=g, device='cuda') * 1e-3).to(BF16)   # > 0 where hi = 0
    act = torch.zeros(rows, 128, dtype=BF16, device='cuda')
    act[:, :Ch], act[:, Ch:2 * Ch] = act_hi, act_lo
    if Ch == 32:
        act[:, 64:] = act[:, :64]                        # the stem's [hi | lo | hi | lo]
    act[~on] = 0
    ga0 = ga.clone()
    hi_out, lo_out, pair_out = _filled(B, BF16), _filled(B, BF16), _filled(B, BF16)
    L.check(lib.rz_learn_tile_grad_mask_split(L.ptr(ga), L.ptr(gb) if with_b else None, L.ptr(act), Ch,
                                              L.ptr(pair_out) if with_pair else None, L.ptr(hi_out), L.ptr(lo_out), B,
                                              L.stream_ptr()), 'rz_learn_tile_grad_mask_split')
    s = ga0[:, :Ch] + gb[:, :Ch] if with_b else ga0[:, :Ch]
    gm = torch.where(act[:, :Ch].float() > 0, s, torch.zeros_like(s))
    hi, lo = _split(gm)
    want_a = ga0.clone()
    want_a[:, :Ch] = gm
    assert torch.equal(ga, want_a)
    z = torch.zeros(rows, 128, dtype=BF16, device='cuda')
    want_hi, want_lo, want_pair = z.clone(), z.clone(), z.clone()
    want_hi[:, :Ch], want_lo[:, :Ch] = hi, lo
    want_pair[:, :Ch], want_pair[:, Ch:2 * Ch] = hi, lo
    assert torch.equal(hi_out[:rows], want_hi) and torch.equal(lo_out[:rows], want_lo)
    _assert_tail_untouched(hi_out, B)
    _assert_tail_untouched(lo_out, B)
    if with_pair:
        assert torch.equal(pair_out[:rows], want_pair)
        _assert_tail_untouched(pair_out, B)
    else:
        assert (pair_out.float() == SENTINEL).all()
    assert (ga[~on][:, :Ch] == 0).all() and (hi_out[:rows][~on].float() == 0).all()
    assert ((act_hi.float() == 0) & (s != 0)).any() and ((act_hi.float() < 0) & (s != 0)).any()


@pytest.mark.parametrize('H,B', SHAPES)
@pytest.mark.parametrize('Ch', [128, 64, 5])
def test_tile_f32_to_nhwc_gathers_the_board_squares(H, B, Ch):
    L, lib = _lib()
    g = torch.Generator(device='cuda').manual_seed(H + B + Ch)
    t = _rand_f32((B * 256, 128), g)
    out = torch.full((B + 1, H * H, Ch), SENTINEL, device='cuda')
    L.check(lib.rz_learn_tile_f32_to_nhwc(L.ptr(t), L.ptr(out), Ch, B, H, H, L.stream_ptr()), 'rz_learn_tile_f32_to_nhwc')
    assert torch.equal(out[:B], t.view(B, 16, 16, 128)[:, :H, :H, :Ch].reshape(B, H * H, Ch))
    assert (out[B:] == SENTINEL).all()


# ------------------------------------------------------------------------------------ the trainer and its layers
def _batch(H, B, seed):
    """Game-like observation planes (stones of both players, the last move, the colour plane), pi and z."""
    rs = np.random.RandomState(seed)
    x = np.zeros((B, 4, H, H), dtype=np.float32)
    for i in range(B):
        k = rs.randint(0, H * H // 2 + 1)
        sq = rs.permutation(H * H)[:k]
        for j, s in enumerate(sq):
            x[i, j % 2, s // H, s % H] = 1.0
        if k:
            x[i, 2, sq[-1] // H, sq[-1] % H] = 1.0
        if k % 2 == 0:
            x[i, 3] = 1.0
    pi = rs.dirichlet(0.3 * np.ones(H * H), size=B).astype(np.float32)
    z = rs.choice([-1.0, 0.0, 1.0], size=B).astype(np.float32)
    return x, pi, z


def _trainer(H):
    from rlzero_b200.games.gomoku.policy_value_net import PolicyValueNet
    from rlzero_b200.learn import NativeTrainer
    torch.manual_seed(H)
    tr = NativeTrainer(PolicyValueNet(H).cuda())
    tr.use_tc_trunk = True
    tr._repack()
    return tr


def _conv(inp, w, bias, out, B, H, relu, flags):
    L, lib = _lib()
    L.check(lib.rz_net_conv3x3_tc2(L.ptr(inp), L.ptr(w), L.ptr(bias), None, L.ptr(out), B, H, H, 128, int(relu), 2, flags, 0,
                                   L.stream_ptr()), 'rz_net_conv3x3_tc2')


def _forward_layers(tr, planes, B, H):
    """The three launches of NativeTrainer._trunk_forward_tc, each into a tile with a spare SENTINEL board."""
    L, lib = _lib()
    w = tr.tcw
    T1, T2, A3 = _filled(B, BF16), _filled(B, BF16), _filled(B, torch.float32)
    gdesc = L.GameDesc(H, min(5, H), H * H, tr.AS, H, L.GAME_GOMOKU, 0.0, 0, 16)
    L.check(lib.rz_net_stem_tc_planes(C.byref(gdesc), L.ptr(planes), L.ptr(w['stem']), L.ptr(w['b1']), L.ptr(T1), B, 1 | 2, 0,
                                      L.stream_ptr()), 'rz_net_stem_tc_planes')
    _conv(T1[:B * 256].clone(), w['w2'], w['b2'], T2, B, H, True, 2 | 8 | 256)
    _conv(T2[:B * 256].clone(), w['w3'], w['b3'], A3, B, H, True, 2 | 16 | 64)
    return T1, T2, A3


def _layer_errors(tr, planes, T1, T2, A3, B, H):
    """Each layer against float64 on the values it consumed: the hi + lo of its input tile, Whi + Wlo of its weight."""
    m = tr.module
    W = [_pair_value(c.weight.detach()) for c in (m.conv1, m.conv2, m.conv3)]
    b = [c.bias.detach().double() for c in (m.conv1, m.conv2, m.conv3)]
    a1 = _board(T1, B, H, 0, 32).double() + _board(T1, B, H, 32, 64).double()
    a2 = _board(T2, B, H, 0, 64).double() + _board(T2, B, H, 64, 128).double()
    a3 = _board(A3, B, H, 0, 128).double()
    return dict(stem=_rel(a1, F.relu(F.conv2d(planes.double(), W[0], b[0], padding=1))),
                conv2=_rel(a2, F.relu(F.conv2d(a1, W[1], b[1], padding=1))),
                conv3=_rel(a3, F.relu(F.conv2d(a2, W[2], b[2], padding=1))))


@pytest.mark.parametrize('H,B', SHAPES)
def test_forward_layers_against_float64(H, B):
    """Stem (relu bits 1|2): [hi32 | lo32 | hi32 | lo32]; conv2 (flags 2|8|256): [hi64 | lo64] with hi the bf16 nearest
    hi + lo; conv3 (flags 2|16|64): float32.  Pad squares exactly zero; the board past the last one untouched."""
    tr = _trainer(H)
    x = torch.from_numpy(_batch(H, B, H + B)[0]).cuda()
    T1, T2, A3 = _forward_layers(tr, x, B, H)
    tr.forward(x)                                           # the trainer runs the same launches
    assert torch.equal(tr.tc['T1'], T1[:B * 256]) and torch.equal(tr.tc['T2'], T2[:B * 256])
    assert torch.equal(tr.tc['A3'], A3[:B * 256])
    off = ~_on_board(B, H)
    for t in (T1, T2, A3):
        assert (t[:B * 256][off].float() == 0).all()
        _assert_tail_untouched(t, B)
    assert torch.equal(T1[:, 64:], T1[:, :64])
    _assert_nearest_pair(T1[:B * 256, :32], T1[:B * 256, 32:64], 'stem')
    _assert_nearest_pair(T2[:B * 256, :64], T2[:B * 256, 64:], 'conv2')
    assert (T1[:B * 256, :32].float() >= 0).all() and (T2[:B * 256, :64].float() >= 0).all()
    errs = _layer_errors(tr, x, T1, T2, A3, B, H)
    print('forward layers %dx%d B=%d: ' % (H, H, B) +
          ', '.join('%s %.2e (bound %.1e)' % (k, e, BOUND_LAYER[k]) for k, e in errs.items()))
    for k, e in errs.items():
        assert e <= BOUND_LAYER[k], (k, e)


@pytest.mark.parametrize('H,B', [(3, 130), (15, 48)])
def test_dropping_hi_wlo_from_the_forward_conv3_fails_the_layer_check(H, B):
    """tcw['w3'][..., 64:] = 0 removes the hi * Wlo product of conv3's forward."""
    tr = _trainer(H)
    tr.tcw['w3'][..., 64:] = 0
    x = torch.from_numpy(_batch(H, B, H + B)[0]).cuda()
    e = _layer_errors(tr, x, *_forward_layers(tr, x, B, H), B, H)['conv3']
    print('mutation w3 hi*Wlo %dx%d B=%d: conv3 %.2e = %.0fx its bound %.1e' % (H, H, B, e, e / BOUND_LAYER['conv3'],
                                                                               BOUND_LAYER['conv3']))
    assert e >= 3 * BOUND_LAYER['conv3']


# ------------------------------------------------------------------------------------------- c. data-gradient passes
def _dgrad_passes(tr, dz3, dz2, B, H, drop_lo=False):
    """conv3's two data-gradient halves and conv2's one pass, as NativeTrainer._trunk_backward_tc launches them, from
    float32 output gradients dz3 [B, HW, 128] and dz2 [B, HW, 64].  drop_lo: zero the lo half of each input tile."""
    L, lib = _lib()
    w, s = tr.tcw, L.stream_ptr()
    XP = torch.zeros(B * 256, 128, dtype=BF16, device='cuda')
    outs = []
    for h in range(3):
        if h < 2:
            L.check(lib.rz_learn_nhwc_to_tile_hilo_slice(L.ptr(dz3), 128, 64 * h, 64, L.ptr(XP), B, H, H, s),
                    'rz_learn_nhwc_to_tile_hilo_slice')
        else:
            L.check(lib.rz_learn_nhwc_to_tile_hilo(L.ptr(dz2), 64, L.ptr(XP), None, 0, B, H, H, s), 'rz_learn_nhwc_to_tile_hilo')
        if drop_lo:
            XP[:, 64:] = 0
        out = _filled(B, torch.float32)
        _conv(XP, w['d3'][h] if h < 2 else w['d2'], tr.zero_bias, out, B, H, False, 2 | 16 | 64)
        outs.append(out)
    return outs


def _dgrad_refs(tr, dz3, dz2, B, H):
    """dx of oracle/train_oracle.py's _conv3x3_backward in float64 on the pair values of the weights and gradients."""
    from oracle.train_oracle import _conv3x3_backward
    nchw = lambda t: _pair_value(t).view(B, H, H, -1).permute(0, 3, 1, 2).cpu().numpy()
    W3, W2 = (_pair_value(c.weight.detach()).cpu().numpy() for c in (tr.module.conv3, tr.module.conv2))
    dy3, dy2 = nchw(dz3), nchw(dz2)
    x64, x32 = np.zeros((B, 64, H, H)), np.zeros((B, 32, H, H))
    return [_conv3x3_backward(x64, W3[:64], dy3[:, :64])[0], _conv3x3_backward(x64, W3[64:], dy3[:, 64:])[0],
            _conv3x3_backward(x32, W2, dy2)[0]]


def _grad_inputs(H, B):
    g = torch.Generator(device='cuda').manual_seed(7 * H + B)
    dz = lambda c: (torch.randn(B, H * H, c, generator=g, device='cuda')
                    * (torch.rand(B, H * H, c, generator=g, device='cuda') < 0.6))    # ReLU-masked: many exact zeros
    return dz(128), dz(64)


_PASSES = ('conv3 half 0 (d3[0])', 'conv3 half 1 (d3[1])', 'conv2 (d2)')


@pytest.mark.parametrize('H,B', SHAPES)
def test_data_gradient_passes_against_float64(H, B):
    """Each pass (flags 2|16|64: hi*Whi + lo*Whi + hi*Wlo, float32 out) against float64; the output channels past the
    layer's input channels (64 for conv3, 32 for conv2) and the pad squares exactly zero."""
    tr = _trainer(H)
    dz3, dz2 = _grad_inputs(H, B)
    outs = _dgrad_passes(tr, dz3, dz2, B, H)
    refs = _dgrad_refs(tr, dz3, dz2, B, H)
    off = ~_on_board(B, H)
    errs = []
    for out, ref, ci in zip(outs, refs, (64, 64, 32)):
        assert (out[:B * 256, ci:] == 0).all() and (out[:B * 256][off] == 0).all()
        _assert_tail_untouched(out, B)
        errs.append(_rel(_board(out, B, H, 0, ci).double().cpu(), torch.from_numpy(ref)))
    print('data gradient %dx%d B=%d: ' % (H, H, B) + ', '.join('%s %.2e' % (n, e) for n, e in zip(_PASSES, errs)) +
          ' (bound %.1e)' % BOUND_DGRAD)
    assert max(errs) <= BOUND_DGRAD, errs


@pytest.mark.parametrize('H,B', [(3, 130), (15, 48)])
def test_dropping_lo_whi_from_a_data_gradient_pass_fails_the_pass_check(H, B):
    """The lo half of each pass's input pair tile zeroed: the lo * Whi product is gone."""
    tr = _trainer(H)
    dz3, dz2 = _grad_inputs(H, B)
    outs = _dgrad_passes(tr, dz3, dz2, B, H, drop_lo=True)
    refs = _dgrad_refs(tr, dz3, dz2, B, H)
    errs = [_rel(_board(out, B, H, 0, ci).double().cpu(), torch.from_numpy(ref))
            for out, ref, ci in zip(outs, refs, (64, 64, 32))]
    print('mutation lo*Whi %dx%d B=%d: ' % (H, H, B) +
          ', '.join('%s %.2e = %.0fx' % (n, e, e / BOUND_DGRAD) for n, e in zip(_PASSES, errs)) + ' the bound %.1e' % BOUND_DGRAD)
    assert min(errs) >= 3 * BOUND_DGRAD, errs


# --------------------------------------------------------------------------- d. the whole step, mask-pinned oracle
def _device_masks(tr, B, H):
    """The ReLU masks the device applied, read from the activations the trainer keeps: a1 / a2 = sign of the high part
    of the pair tiles T1 / T2, a3 = the float32 conv3 output, pa / va = the head features, h = the value hidden layer."""
    f = tr.feat.view(B, 6, H, H)
    m = dict(a1=_board(tr.tc['T1'], B, H, 0, 32), a2=_board(tr.tc['T2'], B, H, 0, 64),
             a3=tr.a[2].view(B, H, H, 128).permute(0, 3, 1, 2), pa=f[:, :4], va=f[:, 4:], h=tr.h)
    return {k: (v.float() > 0).cpu().numpy() for k, v in m.items()}


def _step(tr, x, pi, z):
    B, H = x.shape[0], x.shape[2]
    logp, v = tr.forward(torch.from_numpy(x).cuda())
    masks = _device_masks(tr, B, H)
    vl, pl, ent = tr.backward(torch.from_numpy(pi).cuda(), torch.from_numpy(z).cuda()).tolist()
    after = _device_masks(tr, B, H)
    assert all(np.array_equal(masks[k], after[k]) for k in masks), 'backward overwrote an activation the masks come from'
    grads = {n: g.double().cpu().numpy() for n, g in tr.grads().items()}
    return logp[:, :H * H].double().cpu().numpy(), v.double().cpu().numpy(), vl + pl, ent, grads, masks


def _grad_errors(grads, ref):
    """{name: (max |d| / max |ref|, ||d|| / ||ref||)}"""
    return {n: (np.abs(grads[n] - r).max() / np.abs(r).max(), np.linalg.norm(grads[n] - r) / np.linalg.norm(r))
            for n, r in ref.items()}


def _grad_bounds(name):
    """(bound of max |d| / max |ref|, bound of ||d|| / ||ref||) for one gradient."""
    if name in BOUND_GRAD_OVERRIDE:
        return BOUND_GRAD_OVERRIDE[name], BOUND_GRAD_OVERRIDE[name]
    return BOUND_GRAD_MAX, BOUND_GRAD_L2


def _oracle_params(tr):
    return {k: v.detach().double().cpu().numpy() for k, v in tr.module.state_dict().items()}


@pytest.mark.parametrize('H,B', SHAPES)
def test_the_whole_step_against_the_mask_pinned_oracle(H, B):
    """forward + backward of the tensor-core step against loss_and_grads(..., masks=the device's masks): log p, v,
    loss, entropy and all 16 gradients, each gradient in both metrics."""
    from oracle import train_oracle
    tr = _trainer(H)
    x, pi, z = _batch(H, B, 3 * H + B)
    logp, v, loss, ent, grads, masks = _step(tr, x, pi, z)
    p = _oracle_params(tr)
    x64, pi64, z64 = x.astype(np.float64), pi.astype(np.float64), z.astype(np.float64)
    logp_o, v_o, _ = train_oracle.forward(p, x64, masks=masks)
    loss_o, ent_o, g_o = train_oracle.loss_and_grads(p, x64, pi64, z64, masks=masks)
    _, _, free = train_oracle.forward(p, x64)
    flips = {k: int((masks[k] != (free[k] > 0)).sum()) for k in masks}
    e_lv = max(np.abs(logp - logp_o).max(), np.abs(v - v_o.reshape(-1)).max())
    e_loss = max(abs(loss - loss_o), abs(ent - ent_o))
    errs = _grad_errors(grads, g_o)
    print('step %dx%d B=%d: mask elements that differ from the unpinned oracle: %s' % (H, H, B, flips))
    print('  log p / v %.2e (bound %.1e), loss / entropy %.2e (bound %.1e)' % (e_lv, BOUND_LOGP_V, e_loss, BOUND_LOSS))
    for n, (em, e2) in errs.items():
        print('  %-18s max %.2e  l2 %.2e  (bounds %.1e, %.1e)' % ((n, em, e2) + _grad_bounds(n)))
    assert e_lv <= BOUND_LOGP_V and e_loss <= BOUND_LOSS
    for n, (em, e2) in errs.items():
        bm, b2 = _grad_bounds(n)
        assert em <= bm and e2 <= b2, (n, em, e2)


@pytest.mark.parametrize('mutation', ['d3[1] hi*Wlo', 'd2 hi*Wlo'])
@pytest.mark.parametrize('H,B', [(3, 130), (15, 48)])
def test_a_dropped_data_gradient_product_fails_the_pinned_step(H, B, mutation):
    """hi * Wlo dropped from the second half of conv3's data gradient (tcw['d3'][1][:, :64, 64:] = 0) or from conv2's
    (tcw['d2'][:, :32, 64:] = 0): the mask-pinned comparison fails by at least 3x, while the metric of the unpinned
    comparison in tests/test_gpu_learn.py (max error over max(largest entry, 1e-3), bound 2e-2) is printed beside it."""
    from oracle import train_oracle
    tr = _trainer(H)
    if mutation.startswith('d3'):
        tr.tcw['d3'][1][:, :64, 64:] = 0
    else:
        tr.tcw['d2'][:, :32, 64:] = 0
    x, pi, z = _batch(H, B, 3 * H + B)
    _, _, _, _, grads, masks = _step(tr, x, pi, z)
    p = _oracle_params(tr)
    x64, pi64, z64 = x.astype(np.float64), pi.astype(np.float64), z.astype(np.float64)
    _, _, g_o = train_oracle.loss_and_grads(p, x64, pi64, z64, masks=masks)
    _, _, g_free = train_oracle.loss_and_grads(p, x64, pi64, z64)
    errs = _grad_errors(grads, g_o)
    over_max = max(em / _grad_bounds(n)[0] for n, (em, _) in errs.items())     # in multiples of each tensor's bound
    over_l2 = max(e2 / _grad_bounds(n)[1] for n, (_, e2) in errs.items())
    unpinned = max(np.abs(grads[n] - r).max() / max(np.abs(r).max(), 1e-3) for n, r in g_free.items())
    print('mutation %s %dx%d B=%d: pinned max metric %.0fx its bound, l2 metric %.0fx its bound; the unpinned metric '
          '%.2e %s its bound 2e-2' % (mutation, H, H, B, over_max, over_l2, unpinned,
                                      'passes' if unpinned <= 2e-2 else 'fails'))
    for n, (em, e2) in errs.items():
        bm, b2 = _grad_bounds(n)
        if em > bm or e2 > b2:
            print('  %-18s max %.2e  l2 %.2e  (bounds %.1e, %.1e)' % (n, em, e2, bm, b2))
    assert over_max >= 3 and over_l2 >= 3
