"""GPU tests of the tensor-core training step on the 20-stride layout (boards of 16x16 to 19x19) and with the 17-plane Go
stem and the pass action: the _ex entry points of csrc/rz_learn_tc.cu against plain PyTorch on the same bf16 values and
against their 16-stride forms, ResNetTrainer against autograd, and AlphaZeroAgent(trainer='native') on a Go network."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _rows(n, S):
    return (n * S * S + 255) // 256 * 256


def _tile(x_nchw, S):
    """float [n,C,H,W] -> bf16 padded layout of stride S, [round_up(n*S*S, 256), C] (zero pad squares and tail rows)."""
    n, c, h, w = x_nchw.shape
    t = torch.zeros(_rows(n, S), c, device=x_nchw.device)
    t[:n * S * S].view(n, S, S, c)[:, :h, :w, :] = x_nchw.permute(0, 2, 3, 1)
    return t.to(torch.bfloat16).contiguous()


def _untile(t, n, h, w, S):
    return t.float()[:n * S * S].reshape(n, S, S, -1)[:, :h, :w, :].permute(0, 3, 1, 2).contiguous()


def _off_board_max(t, n, h, w, S):
    """Largest |value| on the pad squares and the tail rows of a tile."""
    f = t.float()
    b = f[:n * S * S].reshape(n, S, S, -1)
    m = max(b[:, h:, :, :].abs().max().item() if h < S else 0.0, b[:, :, w:, :].abs().max().item() if w < S else 0.0)
    if f.shape[0] > n * S * S:
        m = max(m, f[n * S * S:].abs().max().item())
    return m


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield


@pytest.mark.parametrize('n,h', [(1, 19), (5, 19), (7, 19), (130, 19), (1, 17), (5, 17), (7, 17), (130, 17)])
def test_weight_gradient_at_row_stride_20(n, h):
    """rz_learn_conv_wgrad_tc_ex at S = 20 == d/dW of F.conv2d(x, W, padding=1) contracted with dy, in float64 on the
    bf16 values.  n = 7 ends in a partial 128-row tile; the tiles straddle boards."""
    from rlzero_b200 import _lib as L
    lib = L.load()
    S = 20
    g = torch.Generator(device='cuda').manual_seed(n + h)
    x = torch.randn(n, 128, h, h, device='cuda', generator=g)
    dy = torch.randn(n, 128, h, h, device='cuda', generator=g)
    xt, dyt = _tile(x, S), _tile(dy, S)
    ref = torch.nn.grad.conv2d_weight(_untile(xt, n, h, h, S).double(), (128, 128, 3, 3), _untile(dyt, n, h, h, S).double(),
                                      padding=1)
    dw = torch.empty(128, 128, 3, 3, device='cuda')
    scratch = torch.empty(49 * 9 * 128 * 128, device='cuda')
    L.check(lib.rz_learn_conv_wgrad_tc_ex(L.ptr(xt), L.ptr(dyt), L.ptr(dw), L.ptr(scratch), scratch.numel(), n, S, 0,
                                          L.stream_ptr()), 'rz_learn_conv_wgrad_tc_ex')
    err = (dw.double() - ref).abs().max().item()
    scale = ref.abs().max().item()
    assert err <= 2e-5 * scale, (err, scale)
    dw2 = torch.empty_like(dw)
    L.check(lib.rz_learn_conv_wgrad_tc_ex(L.ptr(xt), L.ptr(dyt), L.ptr(dw2), L.ptr(scratch), scratch.numel(), n, S, 0,
                                          L.stream_ptr()), 'rz_learn_conv_wgrad_tc_ex')
    assert torch.equal(dw, dw2)


@pytest.mark.parametrize('n,h', [(7, 15), (64, 9)])
def test_weight_gradient_ex_at_row_stride_16_is_the_legacy_entry_point(n, h):
    from rlzero_b200 import _lib as L
    lib = L.load()
    g = torch.Generator(device='cuda').manual_seed(n)
    xt = _tile(torch.randn(n, 128, h, h, device='cuda', generator=g), 16)
    dyt = _tile(torch.randn(n, 128, h, h, device='cuda', generator=g), 16)
    scratch = torch.empty(49 * 9 * 128 * 128, device='cuda')
    a, b = torch.empty(128 * 128 * 9, device='cuda'), torch.empty(128 * 128 * 9, device='cuda')
    L.check(lib.rz_learn_conv_wgrad_tc(L.ptr(xt), L.ptr(dyt), L.ptr(a), L.ptr(scratch), scratch.numel(), n, 0,
                                       L.stream_ptr()), 'rz_learn_conv_wgrad_tc')
    L.check(lib.rz_learn_conv_wgrad_tc_ex(L.ptr(xt), L.ptr(dyt), L.ptr(b), L.ptr(scratch), scratch.numel(), n, 16, 0,
                                          L.stream_ptr()), 'rz_learn_conv_wgrad_tc_ex')
    assert torch.equal(a, b)


def _bn_case(n, h, w, S, seed=11):
    g = torch.Generator(device='cuda').manual_seed(seed)
    y = torch.randn(n, 128, h, w, device='cuda', generator=g) * 2 + 0.5
    skip = torch.randn(n, 128, h, w, device='cuda', generator=g)
    dout = torch.randn(n, 128, h, w, device='cuda', generator=g)
    bn = torch.nn.BatchNorm2d(128).cuda().train()
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5, generator=g)
        bn.bias.uniform_(-0.5, 0.5, generator=g)
    return _tile(y, S), _tile(skip, S), _tile(dout, S), bn


def _bn_run(lib, L, fwd, bwd, extra, yt, skt, dt, bn, n, h, w, with_skip):
    """One BatchNorm forward + backward through the given entry points; outputs start as garbage."""
    rm, rv = bn.running_mean.clone(), bn.running_var.clone()
    stats = torch.empty(4 * 128, device='cuda')
    scratch = torch.empty(148 * 4 * 256 + 256, device='cuda')
    out = torch.full_like(yt, 7.0)
    L.check(fwd(L.ptr(yt), L.ptr(skt) if with_skip else None, L.ptr(out), L.ptr(bn.weight.data), L.ptr(bn.bias.data),
                L.ptr(rm), L.ptr(rv), bn.eps, bn.momentum, L.ptr(stats), L.ptr(scratch), n, h, w, *extra, L.stream_ptr()),
            'bn forward')
    dgamma, dbeta = torch.empty(128, device='cuda'), torch.empty(128, device='cuda')
    dy, dz = torch.full_like(yt, 7.0), torch.full_like(yt, 7.0)
    L.check(bwd(L.ptr(dt), L.ptr(out), L.ptr(yt), L.ptr(stats), L.ptr(dgamma), L.ptr(dbeta), L.ptr(dy), L.ptr(dz),
                L.ptr(scratch), n, h, w, *extra, L.stream_ptr()), 'bn backward')
    return dict(out=out, rm=rm, rv=rv, stats=stats, dgamma=dgamma, dbeta=dbeta, dy=dy, dz=dz)


@pytest.mark.parametrize('n,h,w,with_skip', [(9, 19, 19, True), (5, 17, 17, False), (3, 16, 16, True)])
def test_batchnorm_training_forward_and_backward_at_row_stride_20(n, h, w, with_skip):
    """rz_learn_bn_forward_ex / _backward_ex at S = 20 against nn.BatchNorm2d (the bounds of the 16-stride test); pad
    squares and the tail rows are written as exact zeros."""
    from rlzero_b200 import _lib as L
    lib = L.load()
    S = 20
    yt, skt, dt, bn = _bn_case(n, h, w, S)
    r = _bn_run(lib, L, lib.rz_learn_bn_forward_ex, lib.rz_learn_bn_backward_ex, (S,), yt, skt, dt, bn, n, h, w, with_skip)
    yr = _untile(yt, n, h, w, S).requires_grad_(True)
    sr = _untile(skt, n, h, w, S).requires_grad_(True)
    ref = F.relu(bn(yr) + (sr if with_skip else 0.0))
    got = _untile(r['out'], n, h, w, S)
    assert (got - ref).abs().max().item() <= 2e-2
    assert torch.allclose(r['rm'], bn.running_mean, atol=1e-5) and torch.allclose(r['rv'], bn.running_var, rtol=1e-4,
                                                                                  atol=1e-5)
    ref.backward(_untile(dt, n, h, w, S))
    assert (r['dgamma'] - bn.weight.grad).abs().max().item() <= 2e-3 * bn.weight.grad.abs().max().item() + 2e-2
    assert (r['dbeta'] - bn.bias.grad).abs().max().item() <= 2e-3 * bn.bias.grad.abs().max().item() + 2e-2
    assert (_untile(r['dy'], n, h, w, S) - yr.grad).abs().max().item() <= 2e-2 * yr.grad.abs().max().item()
    if with_skip:
        assert (_untile(r['dz'], n, h, w, S) - sr.grad).abs().max().item() <= 1e-2 * sr.grad.abs().max().item()
    for k in ('out', 'dy', 'dz'):
        assert _off_board_max(r[k], n, h, w, S) == 0.0, k


@pytest.mark.parametrize('n,h,w,with_skip', [(9, 15, 15, True), (64, 6, 6, False)])
def test_batchnorm_ex_at_row_stride_16_is_the_legacy_entry_point(n, h, w, with_skip):
    from rlzero_b200 import _lib as L
    lib = L.load()
    yt, skt, dt, bn = _bn_case(n, h, w, 16)
    a = _bn_run(lib, L, lib.rz_learn_bn_forward, lib.rz_learn_bn_backward, (), yt, skt, dt, bn, n, h, w, with_skip)
    b = _bn_run(lib, L, lib.rz_learn_bn_forward_ex, lib.rz_learn_bn_backward_ex, (16,), yt, skt, dt, bn, n, h, w, with_skip)
    for k in a:
        assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize('n_planes,n,h,S', [(17, 5, 19, 20), (17, 3, 9, 16), (17, 7, 16, 20), (4, 6, 17, 20),
                                              (4, 6, 15, 16)])
def test_planes_to_tile_ex(n_planes, n, h, S):
    """The stem's weight-gradient operand: channels 0..n_planes-1 are the planes, everything else is zero (exact)."""
    from rlzero_b200 import _lib as L
    lib = L.load()
    g = torch.Generator(device='cuda').manual_seed(n)
    planes = (torch.rand(n, n_planes, h, h, device='cuda', generator=g) < 0.3).float()
    want = torch.zeros(n, 128, h, h, device='cuda')
    want[:, :n_planes] = planes
    tile = torch.full((_rows(n, S), 128), 7.0, dtype=torch.bfloat16, device='cuda')
    L.check(lib.rz_learn_planes_to_tile_ex(L.ptr(planes), n_planes, L.ptr(tile), n, h, h, S, L.stream_ptr()),
            'rz_learn_planes_to_tile_ex')
    assert torch.equal(tile, _tile(want, S))
    if n_planes == 4 and S == 16:
        legacy = torch.full_like(tile, 7.0)
        L.check(lib.rz_learn_planes_to_tile(L.ptr(planes), L.ptr(legacy), n, h, h, L.stream_ptr()), 'rz_learn_planes_to_tile')
        assert torch.equal(tile, legacy)


@pytest.mark.parametrize('n,h', [(5, 19), (7, 17), (2, 16)])
def test_tile_nhwc_round_trip_at_row_stride_20(n, h):
    from rlzero_b200 import _lib as L
    lib = L.load()
    S = 20
    g = torch.Generator(device='cuda').manual_seed(n)
    x = torch.randn(n, h * h, 128, device='cuda', generator=g).to(torch.bfloat16).float()     # exact in bf16
    tile = torch.full((_rows(n, S), 128), 7.0, dtype=torch.bfloat16, device='cuda')
    L.check(lib.rz_learn_nhwc_to_tile_ex(L.ptr(x), L.ptr(tile), n, h, h, S, L.stream_ptr()), 'rz_learn_nhwc_to_tile_ex')
    assert torch.equal(tile, _tile(x.view(n, h, h, 128).permute(0, 3, 1, 2), S))
    back = torch.empty_like(x)
    L.check(lib.rz_learn_tile_to_nhwc_ex(L.ptr(tile), L.ptr(back), n, h, h, S, L.stream_ptr()), 'rz_learn_tile_to_nhwc_ex')
    assert torch.equal(back, x)


def test_stem_packing_matches_the_inference_weights():
    """pack_stem_tc_ex(17) is exactly the weight NativeForward builds for rz_net_stem_go_tc; pack_stem_tc_ex(4) is
    rz_learn_pack_stem_tc."""
    from rlzero_b200 import _lib as L
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    lib = L.load()
    torch.manual_seed(0)
    net = ResNetPolicyValueNet(19, n_blocks=1, n_actions=362, in_planes=17).cuda().eval()
    nf = NativeForward(net)
    out = torch.full((128 * 192,), 7.0, dtype=torch.bfloat16, device='cuda')
    L.check(lib.rz_learn_pack_stem_tc_ex(L.ptr(net.stem.weight.detach()), 17, L.ptr(out), L.stream_ptr()),
            'rz_learn_pack_stem_tc_ex')
    assert torch.equal(out.view(128, 192), nf.stem['w'])
    w4 = torch.randn(128, 4, 3, 3, device='cuda')
    a = torch.full((128 * 64,), 7.0, dtype=torch.bfloat16, device='cuda')
    b = torch.full_like(a, 3.0)
    L.check(lib.rz_learn_pack_stem_tc(L.ptr(w4), L.ptr(a), L.stream_ptr()), 'rz_learn_pack_stem_tc')
    L.check(lib.rz_learn_pack_stem_tc_ex(L.ptr(w4), 4, L.ptr(b), L.stream_ptr()), 'rz_learn_pack_stem_tc_ex')
    assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------- the whole step
def _batch(size, B, seed, planes):
    """Synthetic positions: 4 Gomoku planes, or the 17 GoEnv.observe planes (8 pairs of stone planes + the player
    plane); targets over H*W actions, or H*W + 1 with the pass."""
    rs = np.random.RandomState(seed)
    x = np.zeros((B, planes, size, size), dtype=np.float32)
    for i in range(B):
        k = rs.randint(0, size * size // 2)
        sq = rs.permutation(size * size)[:k]
        if planes == 4:
            for j, s in enumerate(sq):
                x[i, j % 2, s // size, s % size] = 1.0
            if k:
                x[i, 2, sq[-1] // size, sq[-1] % size] = 1.0
            if k % 2 == 0:
                x[i, 3] = 1.0
        else:
            for t in range(8):                      # history: the position t moves ago has fewer stones
                for j, s in enumerate(sq[:max(0, k - t)]):
                    x[i, 2 * t + j % 2, s // size, s % size] = 1.0
            x[i, 16] = float(k % 2)
    A = size * size + (1 if planes == 17 else 0)
    pi = rs.dirichlet(0.3 * np.ones(A), size=B).astype(np.float32)
    z = rs.choice([-1.0, 0.0, 1.0], size=B).astype(np.float32)
    return x, pi, z


def _net(size, blocks, planes):
    from rlzero_b200.games.gomoku.policy_value_net import ResNetPolicyValueNet
    if planes == 17:
        return ResNetPolicyValueNet(size, n_blocks=blocks, n_actions=size * size + 1, in_planes=17).cuda()
    return ResNetPolicyValueNet(size, n_blocks=blocks).cuda()


class _RoundBF16(torch.autograd.Function):
    """Round to bf16 in the forward pass and the gradient in the backward pass: where the kernels store a tensor."""

    @staticmethod
    def forward(ctx, x):
        return x.to(torch.bfloat16).float()

    @staticmethod
    def backward(ctx, g):
        return g.to(torch.bfloat16).float()


def _emulated_forward(net, x):
    """The training-mode forward with the kernels' storage points emulated: conv weights and every stored tensor rounded
    to bf16, everything else fp32."""
    r = _RoundBF16.apply
    wq = lambda conv: conv.weight + (conv.weight.to(torch.bfloat16).float() - conv.weight).detach()
    a = r(F.relu(F.conv2d(x, wq(net.stem), net.stem.bias, padding=1)))
    for blk in net.blocks:
        y1 = r(F.conv2d(a, wq(blk.conv1), blk.conv1.bias, padding=1))
        a1 = r(F.relu(blk.bn1(y1)))
        y2 = r(F.conv2d(a1, wq(blk.conv2), blk.conv2.bias, padding=1))
        a = r(F.relu(blk.bn2(y2) + a))
    return net.heads(a)


@pytest.mark.parametrize('size,blocks,B,planes', [(9, 2, 16, 17), (13, 1, 16, 17), (19, 2, 16, 17), (19, 1, 7, 17),
                                                  (17, 1, 8, 4)])
def test_resnet_training_step_go_and_row_stride_20_against_autograd(size, blocks, B, planes):
    """ResNetTrainer on Go networks (17-plane stem, H*W + 1 actions; 9x9 and 13x13 at S = 16, 19x19 at S = 20) and on a
    4-plane 17x17 network (S = 20) against fp32 autograd and the bf16-storage emulation, with the method and bounds of
    test_gpu_learn_tc.py::test_resnet_training_step_against_autograd.  Go 19x19 with B = 7 (a partial last tile of the
    weight gradient) takes the strict branch."""
    from rlzero_b200.learn import ResNetTrainer
    torch.manual_seed(size + blocks)
    net = _net(size, blocks, planes)
    ref = _net(size, blocks, planes)
    emu = _net(size, blocks, planes)
    ref.load_state_dict(net.state_dict())
    emu.load_state_dict(net.state_dict())
    tr = ResNetTrainer(net)
    assert tr.S == (16 if size <= 15 else 20) and tr.A == net.n_actions
    x, pi, z = _batch(size, B, 2, planes)
    xt, pit, zt = (torch.from_numpy(t).cuda() for t in (x, pi, z))

    def loss_of(lp, v):
        return F.mse_loss(v.view(-1), zt) - torch.mean(torch.sum(pit * lp, dim=1))
    ref.train()
    emu.train()
    lp_ref, v_ref = ref(xt)
    loss_ref = loss_of(lp_ref, v_ref)
    ent_ref = -torch.mean(torch.sum(torch.exp(lp_ref) * lp_ref, dim=1))
    loss_ref.backward()
    lp_emu, v_emu = _emulated_forward(emu, xt)
    loss_of(lp_emu, v_emu).backward()
    logp, v = tr.forward(xt)
    A = net.n_actions
    p_err = (logp[:, :A].exp() - lp_ref.exp()).abs().max().item()
    v_err = (v - v_ref.view(-1)).abs().max().item()
    vl, pl, ent = tr.backward(pit, zt).tolist()
    print('resnet-%d %dx%d %d planes B=%d: |dp| %.2e |dv| %.2e loss %.5f vs %.5f; vs the emulation |dp| %.2e |dv| %.2e' % (
        blocks, size, size, planes, B, p_err, v_err, vl + pl, loss_ref.item(),
        (logp[:, :A].exp() - lp_emu.exp()).abs().max().item(), (v - v_emu.view(-1)).abs().max().item()))
    assert p_err < 5e-3 and v_err < 3e-2
    assert abs((vl + pl) - loss_ref.item()) < 2e-2 and abs(ent - ent_ref.item()) < 1e-2
    for blk_n, blk_r in zip(net.blocks, ref.blocks):
        for bn_n, bn_r in ((blk_n.bn1, blk_r.bn1), (blk_n.bn2, blk_r.bn2)):
            assert (bn_n.running_mean - bn_r.running_mean).abs().max().item() < 5e-3
            assert (bn_n.running_var - bn_r.running_var).abs().max().item() < 5e-3
            assert int(bn_n.num_batches_tracked) == 1
    grads = tr.grads()
    same_forward = (v - v_emu.view(-1)).abs().max().item() < 2e-4
    e_ref, e_emu, cos, ratio = {}, {}, {}, {}
    for (name, prm), (_, pe) in zip(ref.named_parameters(), emu.named_parameters()):
        g, r, q = grads[name].double(), prm.grad.double(), pe.grad.double()
        if name.startswith('blocks.') and name.endswith(('conv1.bias', 'conv2.bias')):
            assert g.abs().max().item() == 0.0 and r.abs().max().item() < 1e-4
            continue
        e_ref[name] = ((g - r).norm() / (r.norm() + 1e-12)).item()
        e_emu[name] = ((g - q).norm() / (q.norm() + 1e-12)).item()
        cos[name] = (torch.dot(g.flatten(), q.flatten()) / (g.norm() * q.norm() + 1e-30)).item()
        ratio[name] = (g.norm() / (q.norm() + 1e-30)).item()
    short = lambda d: ' '.join('%s=%.3f' % (k.replace('blocks.', 'b'), e) for k, e in d.items())
    print('same forward as the emulation:', same_forward)
    print('relative gradient errors vs fp32 autograd:', short(e_ref))
    print('relative gradient errors vs the bf16-storage emulation:', short(e_emu))
    if same_forward:
        assert max(e_emu.values()) < 0.03, max(e_emu.items(), key=lambda kv: kv[1])
    else:
        print('cosines:', short(cos))
        print('norm ratios:', short(ratio))
        assert min(cos.values()) > 0.93, min(cos.items(), key=lambda kv: kv[1])
        assert all(0.85 < r < 1.18 for k, r in ratio.items() if grads[k].numel() >= 16), ratio
    assert (size, blocks, B, planes) != (19, 1, 7, 17) or same_forward      # this S = 20 case takes the strict branch
    assert max(e_ref.values()) < 0.5, max(e_ref.items(), key=lambda kv: kv[1])


def test_go_agent_learns_on_the_native_step_and_tracks_autograd():
    """AlphaZeroAgent(Go ResNet-2 9x9, trainer='native').learn for 20 steps on one batch: the loss falls and follows the
    fp32 autograd agent's; policy_value sees the updated weights and agrees with the module's PyTorch eval forward.  The
    default trainer keeps Go networks on autograd."""
    from rlzero_b200.games.gomoku.alphazero_agent import AlphaZeroAgent
    from rlzero_b200.learn import ResNetTrainer
    x, pi, z = _batch(9, 64, 5, 17)
    torch.manual_seed(4)
    a = AlphaZeroAgent(9, net=_net(9, 2, 17), trainer='native')
    torch.manual_seed(4)
    b = AlphaZeroAgent(9, net=_net(9, 2, 17), trainer='autograd')
    c = AlphaZeroAgent(9, net=_net(9, 2, 17))
    assert isinstance(a.trainer, ResNetTrainer) and b.trainer is None and c.trainer is None
    p0, _ = a.policy_value(x)
    assert p0.shape == (64, 82)
    la, lb = [], []
    for _ in range(20):
        la.append(a.learn(x, pi, z)[0])
        lb.append(b.learn(x, pi, z)[0])
    print('native', ['%.3f' % u for u in la])
    print('autograd', ['%.3f' % u for u in lb])
    assert la[-1] < la[0] - 0.3 and lb[-1] < lb[0] - 0.3
    assert max(abs(u - w) for u, w in zip(la, lb)) < 0.15
    p1, v1 = a.policy_value(x)
    assert not np.allclose(p0, p1)
    net = a.policy_value_net
    net.eval()
    with torch.no_grad():
        lp, v = net(torch.from_numpy(x).cuda())
    dp = np.abs(p1 - lp.exp().cpu().numpy()).max()
    print('policy_value vs the PyTorch eval forward: |dp| %.2e |dv| %.2e' % (dp, np.abs(v1 - v.cpu().numpy()).max()))
    assert dp < 1e-3
