"""GPU tests of the policy-value forward: tcgen05 convolution and heads against PyTorch, the
stock network against the reference's golden outputs, and search parity with the real net."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _to_tile(x_nchw):
    """[n,C,H,W] float -> bf16 tile layout [n,256,C] (p = y*16+x, zero padded)."""
    n, c, h, w = x_nchw.shape
    t = torch.zeros(n, 16, 16, c, dtype=torch.bfloat16, device=x_nchw.device)
    t[:, :h, :w, :] = x_nchw.permute(0, 2, 3, 1).to(torch.bfloat16)
    return t.reshape(n, 256, c).contiguous()


def _from_tile(t, h):
    n, _, c = t.shape
    return t.reshape(n, 16, 16, c)[:, :h, :h, :].permute(0, 3, 1, 2).float()


@pytest.mark.parametrize('rev', ['v2_pair', 'v3'])
@pytest.mark.parametrize('n,h,cin,relu,res', [(1, 15, 128, 1, 0), (3, 15, 128, 1, 1), (5, 9, 64, 0, 0),
                                              (300, 15, 128, 1, 1), (2, 3, 64, 1, 0), (37, 15, 64, 1, 0)])
def test_conv3x3_tc_matches_torch(n, h, cin, relu, res, rev):
    from rlzero_b200 import _lib as L
    lib = L.load()
    torch.manual_seed(n * 100 + h)
    dev = 'cuda'
    x = (torch.randn(n, cin, h, h, device=dev) * 0.5).to(torch.bfloat16).float()
    w = (torch.randn(128, cin, 3, 3, device=dev) / (3.0 * cin ** 0.5)).to(torch.bfloat16).float()
    b = torch.randn(128, device=dev) * 0.1
    r = (torch.randn(n, 128, h, h, device=dev) * 0.5).to(torch.bfloat16).float() if res else None
    ref = torch.nn.functional.conv2d(x.double(), w.double(), b.double(), padding=1)
    if res:
        ref = ref + r.double()
    if relu:
        ref = torch.relu(ref)
    xt = _to_tile(x)
    wt = w.permute(2, 3, 0, 1).reshape(9, 128, cin).to(torch.bfloat16).contiguous()
    out = torch.full((n, 256, 128), 7.0, dtype=torch.bfloat16, device=dev)
    rt = None
    if res:
        out.copy_(_to_tile(r))   # residual aliases the output buffer, as in the trunk
        rt = out
    if rev == 'v3':
        if cin != 128:
            pytest.skip('revision 3 is the 128 -> 128 trunk layer')
        if n % 2:   # tensors padded to a multiple of 256 rows (pairs of 128-row tiles)
            pad = torch.zeros(1, 256, 128, dtype=torch.bfloat16, device=dev)
            xt = torch.cat([xt, pad])
            out = torch.cat([out, pad + 7.0]) if not res else torch.cat([out, pad])
            rt = out if res else None
        L.check(lib.rz_net_conv3x3_tc3(L.ptr(xt), L.ptr(wt), L.ptr(b.contiguous()), L.ptr(rt), L.ptr(out),
                                       n, h, h, 16, relu, 0, L.stream_ptr()), 'conv3')
        out = out[:n]
    else:
        L.check(lib.rz_net_conv3x3_tc2(L.ptr(xt), L.ptr(wt), L.ptr(b.contiguous()), L.ptr(rt), L.ptr(out),
                                       n, h, h, cin, relu, 2, 0, 0, L.stream_ptr()), 'conv2')
    torch.cuda.synchronize()
    got = _from_tile(out, h).double()
    err = (got - ref).abs().max().item()
    scale = ref.abs().max().item()
    assert err <= 2e-2 * max(scale, 1.0), (err, scale)   # bf16 output rounding: 2^-9 relative
    # relative to bf16 rounding of the exact result the error is tiny
    ref_bf = ref.float().to(torch.bfloat16).double()
    frac_exact = ((got - ref_bf).abs() <= 1e-6).double().mean().item()
    assert frac_exact > 0.97, frac_exact
    # padding squares must be exactly zero (they are the halo of the next layer)
    full = out.reshape(n, 16, 16, 128).float()
    assert full[:, h:, :, :].abs().max().item() == 0.0
    assert full[:, :, h:, :].abs().max().item() == 0.0


@pytest.mark.parametrize('mode', ['tc32', 'f32'])
@pytest.mark.parametrize('size', [3, 6])
def test_stock_net_matches_reference_golden(size, mode):
    """PolicyValueNet == the reference's own outputs (tests/golden/net_pvn_*.npz) within 1e-5: through the default
    path -- the tensor cores at float32-level accuracy (mode 'tc32': bf16 high/low pairs, three products per
    convolution) -- and through the fp32 CUDA-core path."""
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, PolicyValueNet
    z = np.load(os.path.join(HERE, 'golden', 'net_pvn_%d.npz' % size))
    net = PolicyValueNet(size)
    net.load_state_dict({k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith('w_')})
    net.cuda().eval()
    assert NativeForward(net).mode == 'tc32'           # the default for the reference's network
    nf = NativeForward(net, mode=mode)
    logp, v = nf.forward_planes(z['x'])
    np.testing.assert_allclose(logp.cpu().numpy(), z['logp'], atol=1e-5, rtol=0)
    np.testing.assert_allclose(v.cpu().numpy().reshape(-1, 1), z['v'], atol=1e-5, rtol=0)


@pytest.mark.parametrize('size,n,scale', [(15, 70, 1.0), (15, 300, 4.0), (15, 64, 8.0), (15, 64, 30.0), (9, 5, 1.0),
                                          (6, 130, 2.0), (3, 9, 1.0)])
def test_stock_net_float32_accurate_tensor_core_path(size, n, scale):
    """mode 'tc32' against PyTorch fp32 on the CPU (cuDNN would use TF32): action probabilities and values within 1e-5
    (the north star's fp32 tolerance), also with the heads scaled up to trained-like logit ranges; the search through
    the reference API runs on it.  The pairs carry 16 mantissa bits, so the error grows with the magnitude of the
    logits: measured |d logp| ~ 1.1e-5 x (logit range).  At an extreme range of 30 (one move with probability ~1) the
    1e-5 bound on the probabilities no longer holds and the test asserts the relative bound instead -- mode 'f32'
    (CUDA cores) is the path for that regime."""
    from rlzero_b200.games.gomoku import GomokuEnv
    from rlzero_b200.games.gomoku.alphazero_agent import AlphaZeroAgent
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, PolicyValueNet
    from rlzero_b200.mcts import AlphaZeroMCTS
    torch.manual_seed(size)
    net = PolicyValueNet(size)
    with torch.no_grad():
        for prm in net.parameters():
            prm.mul_(scale ** 0.25)
        if scale > 1.0:                      # trained-like heads: logits and value pre-activations spread out
            net.act_fc1.weight.mul_(scale)
            net.val_fc2.weight.mul_(scale)
    ref = PolicyValueNet(size).eval()
    ref.load_state_dict(net.state_dict())
    net.cuda().eval()
    nf = NativeForward(net, max_batch=n)
    assert nf.mode == 'tc32' and nf.kernels_per_forward() == 4
    x = _random_boards(n, size, 9)
    logp, v = (t.cpu() for t in nf.forward_planes(x))
    with torch.no_grad():
        lt, vt = ref(torch.from_numpy(x))
    p_err = (logp.exp() - lt.exp()).abs().max().item()
    v_err = (v - vt.reshape(-1)).abs().max().item()
    l_err = (logp - lt).abs().max().item()
    print('tc32 %dx%d n=%d scale %.1f: max |dp| %.2e  |dv| %.2e  |dlogp| %.2e (logp range %.2f)' % (
        size, size, n, scale, p_err, v_err, l_err, float(lt.max() - lt.min())))
    rng = float(lt.max() - lt.min())
    if scale <= 4.0:
        assert p_err < 1e-5 and v_err < 1e-5 and l_err < max(1e-5, 2e-5 * rng)
    elif scale <= 8.0:          # val_fc2 scaled by 8 as well: the value's pre-activation error is scaled with it
        assert p_err < 1e-5 and v_err < 3e-5 and l_err < max(1e-5, 2e-5 * rng)
    else:
        assert l_err < 2e-5 * rng and p_err < 1e-4 and v_err < 3e-4
    if scale == 1.0:
        agent = AlphaZeroAgent(size, net=net)
        env = GomokuEnv(size, min(5, size))
        env.reset()
        acts, probs = AlphaZeroMCTS(agent.policy_value_fn, n_playout=40).simulate(env, 1.0)
        assert len(acts) == size * size and abs(probs.sum() - 1.0) < 1e-9


def _random_boards(n, size, seed):
    rs = np.random.RandomState(seed)
    x = np.zeros((n, 4, size, size), dtype=np.float32)
    for i in range(n):
        k = rs.randint(0, size * size // 2)
        sq = rs.permutation(size * size)[:k]
        for j, s in enumerate(sq):
            x[i, j % 2, s // size, s % size] = 1.0
        if k:
            x[i, 2, sq[-1] // size, sq[-1] % size] = 1.0
        if k % 2 == 0:
            x[i, 3] = 1.0
    return x


@pytest.mark.parametrize('size,blocks,n', [(15, 10, 64), (9, 3, 17), (6, 2, 5)])
def test_resnet_tc_forward_vs_torch(size, blocks, n):
    """bf16 tensor-core trunk: probabilities and value within 1e-3 of the fp32 PyTorch forward."""
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    torch.manual_seed(0)
    net = ResNetPolicyValueNet(size, n_blocks=blocks).cuda().eval()
    nf = NativeForward(net)
    assert nf.mode == 'tc'
    x = _random_boards(n, size, 1)
    logp, v = (t.cpu() for t in nf.forward_planes(x))
    # plain PyTorch fp32 reference on the CPU (cuDNN would silently use TF32)
    ref = ResNetPolicyValueNet(size, n_blocks=blocks).eval()
    ref.load_state_dict({k: t.cpu() for k, t in net.state_dict().items()})
    with torch.no_grad():
        lt, vt = ref(torch.from_numpy(x))
    p_err = (logp.exp() - lt.exp()).abs().max().item()
    v_err = (v - vt.reshape(-1)).abs().max().item()
    print('resnet%d %dx%d bf16: max |dp| %.3e  max |dv| %.3e' % (blocks, size, size, p_err, v_err))
    assert p_err < 1e-3 and v_err < 1e-3          # north_star tolerance for bf16
    assert torch.allclose(logp.exp().sum(1), torch.ones(n), atol=1e-4)
    # fp32 CUDA-core path of the same net: 1e-5 on the same outputs
    nf32 = NativeForward(net, mode='f32')
    l32, v32 = (t.cpu() for t in nf32.forward_planes(x[:6]))
    p32 = (l32.exp() - lt[:6].exp()).abs().max().item()
    v32e = (v32 - vt[:6].reshape(-1)).abs().max().item()
    print('resnet%d %dx%d fp32: max |dp| %.3e  max |dv| %.3e  max |dlogp| %.3e' % (
        blocks, size, size, p32, v32e, (l32 - lt[:6]).abs().max().item()))
    assert p32 < 1e-5 and v32e < 1e-5             # north_star tolerance for fp32


def test_forward_is_batch_invariant():
    """A board's outputs do not depend on its batch neighbours (needed for search parity)."""
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    torch.manual_seed(1)
    net = ResNetPolicyValueNet(9, n_blocks=2).cuda().eval()
    nf = NativeForward(net)
    x = _random_boards(33, 9, 2)
    l_all, v_all = (t.clone() for t in nf.forward_planes(x))
    for i in (0, 7, 32):
        l1, v1 = nf.forward_planes(x[i:i + 1])
        assert torch.equal(l1[0], l_all[i]) and torch.equal(v1[0], v_all[i])


@pytest.mark.parametrize('kind', ['stock', 'resnet'])
def test_search_with_native_net_matches_oracle(kind):
    """Visit counts with the real network on the device == the oracle search fed the same
    network outputs (its policy_value_fn calls the same CUDA forward board by board)."""
    from oracle import pyoracle
    from rlzero_b200.games.gomoku import GomokuEnv
    from rlzero_b200.games.gomoku.alphazero_agent import AlphaZeroAgent
    from rlzero_b200.games.gomoku.policy_value_net import ResNetPolicyValueNet
    from rlzero_b200.mcts import AlphaZeroMCTS
    size, k, n_playout = 6, 4, 150
    torch.manual_seed(3)
    agent = AlphaZeroAgent(size, net=ResNetPolicyValueNet(size, n_blocks=2) if kind == 'resnet' else None)
    agent.policy_value_net.eval()
    env = GomokuEnv(size, k)
    env.reset()
    for m in (14, 15, 20):
        env.step(m)
    mcts = AlphaZeroMCTS(agent.policy_value_fn, n_playout=n_playout, c_puct=5)
    acts, probs = mcts.simulate(env, 1.0)
    board = pyoracle.Board(size, k)
    board.reset()
    for m in (14, 15, 20):
        board.step(m)
    s = pyoracle.Search(agent.policy_value_fn, n_playout, 5)
    acts2, probs2 = s.simulate(board, 1.0)
    assert tuple(acts) == tuple(acts2)
    root = mcts._root
    assert [root._children[a].explore_count for a in acts] == [s.root.children[a].n for a in acts]
    assert [float(root._children[a].total_reward).hex() for a in acts] == [
        float(s.root.children[a].w).hex() for a in acts]
    assert [float(p).hex() for p in probs] == [float(p).hex() for p in probs2]
    # priors stored on the device are exp(log p) of the same forward
    pri = np.array([root._children[a].prior for a in acts])
    ref = np.array([s.root.children[a].prior for a in acts], dtype=np.float64)
    np.testing.assert_allclose(pri, ref, rtol=2e-6)


def test_agent_api_shapes():
    from rlzero_b200.games.gomoku import GomokuEnv
    from rlzero_b200.games.gomoku.alphazero_agent import AlphaZeroAgent
    torch.manual_seed(0)
    agent = AlphaZeroAgent(5)
    env = GomokuEnv(5, 4)
    env.reset()
    env.step(12)
    ap, v = agent.policy_value_fn(env)
    ap = list(ap)
    assert len(ap) == 24 and -1.0 <= v <= 1.0 and all(a != 12 for a, _ in ap)
    probs, vals = agent.policy_value([env.current_state()] * 3)
    assert probs.shape == (3, 25) and vals.shape == (3, 1)
    np.testing.assert_allclose(probs.sum(1), 1.0, atol=1e-5)
    loss, ent = agent.learn([env.current_state()] * 4, [np.full(25, 0.04)] * 4, [1.0, -1.0, 0.0, 1.0])
    assert np.isfinite(loss) and np.isfinite(ent)
    probs2, _ = agent.predict(np.array([env.current_state()]))
    assert not np.allclose(probs2[0], probs[0])   # weights were refreshed after the step


@pytest.mark.parametrize('size,n', [(15, 70), (9, 33), (6, 5)])
def test_stem_kernel_matches_torch_and_planes_stem(size, n):
    """rz_net_stem_tc (planes built from the bitboards inside the kernel, K = 36) against PyTorch on
    current_state planes, with zero pad squares, and bit-identical to the planes-fed stem."""
    from oracle import pyoracle
    from rlzero_b200 import _lib as L
    from rlzero_b200.games.gomoku.gomoku_env import GomokuEnv
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    torch.manual_seed(size)
    net = ResNetPolicyValueNet(size, n_blocks=1).cuda().eval()
    rs = np.random.RandomState(size)
    envs = []
    for i in range(n):
        e = GomokuEnv(size, min(5, size))
        e.reset()
        for m in rs.permutation(size * size)[:(0 if i == 0 else rs.randint(0, size * size - 1))]:
            e.step(int(m))
            if e.game_end_winner()[0]:
                break
        envs.append(e)
    rows = torch.cat([e.device_state()[0] for e in envs]).cuda()
    meta = torch.cat([e.device_state()[1] for e in envs]).cuda()
    # row_stride=16: the 8-stride layout a 6x6 board would otherwise use is covered by test_row_stride_8_*
    nf = NativeForward(net, max_batch=n, row_stride=16)
    lib, g = L.load(), nf._gdesc()
    st = nf.stem
    fused = torch.full((n, 256, 128), 3.0, dtype=torch.bfloat16, device='cuda')
    L.check(lib.rz_net_stem_tc(C.byref(g), L.ptr(rows), L.ptr(meta), L.ptr(st['w']), L.ptr(st['b']), L.ptr(fused),
                               n, 1, 0, L.stream_ptr()), 'stem')
    torch.cuda.synchronize()
    full = fused.reshape(n, 16, 16, 128).float()
    assert full[:, size:].abs().max().item() == 0.0 and full[:, :, size:].abs().max().item() == 0.0
    # against PyTorch on the reference's observation planes (weights rounded to bf16 like the kernel's)
    planes = torch.tensor(np.stack([e.current_state() for e in envs]), dtype=torch.float32, device='cuda')
    wq = net.stem.weight.detach().to(torch.bfloat16).float()
    ref = torch.relu(torch.nn.functional.conv2d(planes, wq, net.stem.bias.detach(), padding=1))
    got = _from_tile(fused, size)
    assert (got - ref).abs().max().item() <= 2.0 ** -8 * max(1.0, ref.abs().max().item()) + 1e-6
    lp1, v1 = nf.forward_boards(rows, meta, n)
    lp1, v1 = lp1.clone(), v1.clone()
    # the planes-fed variant of the kernel (AlphaZeroAgent.policy_value_fn on a host env) is
    # bit-identical to the bitboard-fed one: search parity with a Python-side evaluator relies on it
    lp3, v3 = nf.forward_planes(planes.cpu().numpy())
    assert torch.equal(lp3[:, :size * size], lp1[:, :size * size]) and torch.equal(v3, v1)


@pytest.mark.parametrize('size,blocks,n', [(15, 2, 70), (9, 1, 37), (6, 1, 3)])
def test_fused_head_matches_separate_heads(size, blocks, n):
    """The 1x1 head convolutions inside the last layer's epilogue (rz_net_conv3x3_tc2_head_ex) give
    the same logits / values as storing the trunk output and running the heads kernel on it."""
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    torch.manual_seed(size + 1)
    net = ResNetPolicyValueNet(size, n_blocks=blocks).cuda().eval()
    x = _random_boards(n, size, 3)
    a = NativeForward(net, max_batch=n, fused_head=True)
    b = NativeForward(net, max_batch=n, fused_head=False)
    la, va = (t.clone() for t in a.forward_planes(x))
    lb, vb = (t.clone() for t in b.forward_planes(x))
    # same bf16 activations, same fp32 FMA order over channels: identical features; the FC sums are
    # split over two k halves in both, so the results are bit-identical
    assert torch.equal(la, lb) and torch.equal(va, vb)


@pytest.mark.parametrize('size,blocks,n', [(15, 10, 1), (15, 3, 5), (15, 2, 74), (15, 1, 148), (9, 2, 3), (8, 1, 2), (11, 1, 1)])
def test_one_launch_trunk_is_bit_identical_to_the_layer_kernels(size, blocks, n):
    """rz_net_trunk_small (one CTA pair keeps a board's activation in shared memory through the whole trunk, the seam
    rows exchanged through distributed shared memory) against the same layers launched one by one: the same MMAs in the
    same order and the same epilogue arithmetic, so the logits and values are equal bit for bit -- which is what keeps
    a single-position evaluation (the sequential search, alphazero_mcts.py:73-94) consistent with the batched one."""
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    torch.manual_seed(size + blocks)
    net = ResNetPolicyValueNet(size, n_blocks=blocks).cuda().eval()
    with torch.no_grad():
        for m in net.modules():            # non-trivial BatchNorm statistics, so that folded scales and biases matter
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.normal_(0.0, 0.2)
                m.running_var.uniform_(0.5, 1.5)
                m.weight.uniform_(0.5, 1.5)
                m.bias.normal_(0.0, 0.2)
    x = _random_boards(n, size, 3)
    a = NativeForward(net, max_batch=n)
    assert a.trunk_small is not None and a.small_batch_max >= n and a.kernels_per_forward(n) == 3
    b = NativeForward(net, max_batch=n)
    b.small_batch_max = 0
    la, va = (t.clone() for t in a.forward_planes(x))
    lb, vb = (t.clone() for t in b.forward_planes(x))
    assert torch.isfinite(la[:, :size * size]).all() and torch.equal(la, lb) and torch.equal(va, vb)
    # and twice in a row (the ring and the barriers start from scratch in every launch)
    la2, va2 = a.forward_planes(x)
    assert torch.equal(la2, la) and torch.equal(va2, va)


def test_one_launch_trunk_on_a_rectangular_board_and_at_the_layer_limit():
    """The one-launch trunk with H != W (9 rows x 11 columns in the 16-stride layout), with 24 layers behind the stem
    (its limit: the biases of all layers sit in shared memory), and the fallback to the per-layer kernels beyond it."""
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    torch.manual_seed(3)
    rect = ResNetPolicyValueNet(9, n_blocks=2, board_width=11).cuda().eval()
    a = NativeForward(rect, max_batch=3)
    b = NativeForward(rect, max_batch=3)
    b.small_batch_max = 0
    x = (np.random.RandomState(0).rand(3, 4, 9, 11) < 0.3).astype(np.float32)
    la, va = (t.clone() for t in a.forward_planes(x))
    lb, vb = (t.clone() for t in b.forward_planes(x))
    assert a.kernels_per_forward(3) == 3 and torch.equal(la, lb) and torch.equal(va, vb)
    deep = ResNetPolicyValueNet(8, n_blocks=12).cuda().eval()          # 24 layers behind the stem
    a = NativeForward(deep, max_batch=2)
    b = NativeForward(deep, max_batch=2)
    b.small_batch_max = 0
    x = _random_boards(2, 8, 1)
    la, va = (t.clone() for t in a.forward_planes(x))
    lb, vb = (t.clone() for t in b.forward_planes(x))
    assert a.trunk_small is not None and a.trunk_small['n'] == 24 and torch.equal(la, lb) and torch.equal(va, vb)
    deeper = ResNetPolicyValueNet(8, n_blocks=13).cuda().eval()        # 26 layers: per-layer kernels
    c = NativeForward(deeper, max_batch=2)
    assert c.trunk_small is None
    lc, vc = c.forward_planes(x)
    assert torch.isfinite(lc[:, :64]).all() and torch.isfinite(vc).all()


@pytest.mark.parametrize('size,n', [(15, 1), (15, 9), (9, 3), (6, 2), (3, 1)])
def test_one_launch_trunk_of_the_reference_net_is_bit_identical(size, n):
    """The float32-accurate path of the reference's own PolicyValueNet for a few boards: conv2 (64 channels, split
    output), conv3 (split input) and the 1x1 head convolutions in ONE launch (rz_net_trunk_small_ex) against the two
    per-layer launches -- equal bit for bit, so a single-game search evaluates exactly what a batched one does."""
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, PolicyValueNet
    torch.manual_seed(size)
    net = PolicyValueNet(size).cuda().eval()
    a = NativeForward(net, max_batch=n)
    b = NativeForward(net, max_batch=n)
    b.small_batch_max = 0
    assert a.mode == 'tc32' and a.trunk_small is not None and a.kernels_per_forward(n) == 3 and b.kernels_per_forward(n) == 4
    x = _random_boards(n, size, 7)
    la, va = (t.clone() for t in a.forward_planes(x))
    lb, vb = (t.clone() for t in b.forward_planes(x))
    assert torch.isfinite(la[:, :size * size]).all() and torch.equal(la, lb) and torch.equal(va, vb)


def test_small_and_large_batch_paths_agree_bit_for_bit():
    """Batch invariance ACROSS the path boundary: a board evaluated alone or among 100 (one-launch trunk, one CTA pair per
    board) gives exactly the logits and value it gets among 300 (one launch per layer, persistent CTA pairs over
    tiles) -- what lets the oracle's board-by-board evaluations check a search that evaluates 8192 boards at once."""
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    torch.manual_seed(5)
    net = ResNetPolicyValueNet(15, n_blocks=4).cuda().eval()
    nf = NativeForward(net, max_batch=300)
    assert nf.trunk_small is not None and 100 <= nf.small_batch_max < 300
    x = _random_boards(300, 15, 11)
    l_all, v_all = (t.clone() for t in nf.forward_planes(x))
    assert nf.kernels_per_forward(300) > 3 and nf.kernels_per_forward(100) == 3 and nf.kernels_per_forward(1) == 3
    for i in (0, 17, 148, 299):
        l1, v1 = nf.forward_planes(x[i:i + 1])
        assert torch.equal(l1[0], l_all[i]) and torch.equal(v1[0], v_all[i]), i
    l100, v100 = nf.forward_planes(x[150:250])
    assert torch.equal(l100[:100], l_all[150:250]) and torch.equal(v100[:100], v_all[150:250])


def test_graph_recaptured_after_weight_refresh():
    """A CUDA-graph-captured wave holds weight pointers by value: after AlphaZeroAgent.learn /
    refresh_weights the self-play driver must capture again (stale weights otherwise)."""
    from rlzero_b200.games.gomoku.policy_value_net import ResNetPolicyValueNet
    from rlzero_b200.selfplay import BatchedSelfPlay
    torch.manual_seed(2)
    net = ResNetPolicyValueNet(6, n_blocks=1).cuda().eval()
    sp = BatchedSelfPlay(4, 6, 4, net=net, n_playout=8, add_noise=False, seed=1)
    rows, meta = sp.forest.boards()
    _, _, v1 = sp.get_actions(rows, meta)
    with torch.no_grad():
        for p in net.parameters():
            p.add_(torch.randn_like(p) * 0.5)
    sp.evaluator.refresh_weights()
    _, _, v2 = sp.get_actions(rows, meta)
    sp_new = BatchedSelfPlay(4, 6, 4, net=net, n_playout=8, add_noise=False, seed=1)
    _, _, v3 = sp_new.get_actions(rows, meta)
    assert np.array_equal(v2, v3)


def _to_pad(x_nchw, S):
    """[n,C,H,W] float -> bf16 padded layout [round_up(n*S*S, 256)][C] (row = b*S*S + y*S + x)."""
    n, c, h, w = x_nchw.shape
    t = torch.zeros(n, S, S, c, dtype=torch.bfloat16, device=x_nchw.device)
    t[:, :h, :w, :] = x_nchw.permute(0, 2, 3, 1).to(torch.bfloat16)
    rows = (n * S * S + 255) // 256 * 256
    out = torch.zeros(rows, c, dtype=torch.bfloat16, device=x_nchw.device)
    out[:n * S * S] = t.reshape(n * S * S, c)
    return out


@pytest.mark.parametrize('n,h,w,relu,res,S', [(1, 19, 19, 1, 0, 20), (5, 19, 19, 1, 1, 20), (131, 19, 19, 1, 1, 20),
                                              (3, 17, 18, 0, 0, 20), (2, 6, 7, 1, 1, 16), (2, 6, 7, 1, 1, 8),
                                              (1, 7, 7, 0, 0, 8), (301, 6, 7, 1, 1, 8), (9, 3, 3, 1, 0, 8),
                                              (1200, 6, 7, 1, 1, 8)])
def test_conv3x3_tc3_any_stride_matches_torch(n, h, w, relu, res, S):
    """Revision 3 at row stride 20 (19x19 and other boards > 15: tiles straddling boards), 16, and 8 (Connect
    Four 6x7 and other boards up to 7x7: two whole boards per 128-row tile, 4 per CTA-pair item)."""
    from rlzero_b200 import _lib as L
    lib = L.load()
    torch.manual_seed(n * 10 + h)
    dev = 'cuda'
    assert L.row_stride(h, w, S) == S
    x = (torch.randn(n, 128, h, w, device=dev) * 0.5).to(torch.bfloat16).float()
    wgt = (torch.randn(128, 128, 3, 3, device=dev) / (3.0 * 128 ** 0.5)).to(torch.bfloat16).float()
    b = torch.randn(128, device=dev) * 0.1
    r = (torch.randn(n, 128, h, w, device=dev) * 0.5).to(torch.bfloat16).float() if res else None
    ref = torch.nn.functional.conv2d(x.double(), wgt.double(), b.double(), padding=1)
    if res:
        ref = ref + r.double()
    if relu:
        ref = torch.relu(ref)
    xt = _to_pad(x, S)
    wt = wgt.permute(2, 3, 0, 1).reshape(9, 128, 128).to(torch.bfloat16).contiguous()
    out = torch.full_like(xt, 7.0)
    rt = None
    if res:
        out.copy_(_to_pad(r, S))
        rt = out
    L.check(lib.rz_net_conv3x3_tc3(L.ptr(xt), L.ptr(wt), L.ptr(b.contiguous()), L.ptr(rt), L.ptr(out), n, h, w, S,
                                   relu, 0, L.stream_ptr()), 'conv3')
    torch.cuda.synchronize()
    full = out[:n * S * S].reshape(n, S, S, 128).float()
    got = full[:, :h, :w, :].permute(0, 3, 1, 2).double()
    err = (got - ref).abs().max().item()
    scale = ref.abs().max().item()
    assert err <= 2e-2 * max(scale, 1.0), (err, scale)
    ref_bf = ref.float().to(torch.bfloat16).double()
    assert ((got - ref_bf).abs() <= 1e-6).double().mean().item() > 0.97
    assert full[:, h:, :, :].abs().max().item() == 0.0 and full[:, :, w:, :].abs().max().item() == 0.0
    assert out[n * S * S:].abs().max().item() == 0.0 if out.shape[0] > n * S * S else True


def test_resnet_forward_rev3_19x19_vs_torch():
    """Whole 19x19 forward on the revision-3 convolution (row stride 20) against PyTorch fp32 (1e-3)."""
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    size, blocks, n = 19, 3, 9
    torch.manual_seed(size)
    net = ResNetPolicyValueNet(size, n_blocks=blocks).cuda().eval()
    nf = NativeForward(net, max_batch=n)
    assert nf.mode == 'tc' and nf.S == 20
    x = _random_boards(n, size, 5)
    logp, v = (t.cpu() for t in nf.forward_planes(x))
    ref = ResNetPolicyValueNet(size, n_blocks=blocks).eval()
    ref.load_state_dict({k: t.cpu() for k, t in net.state_dict().items()})
    with torch.no_grad():
        lt, vt = ref(torch.from_numpy(x))
    assert (logp.exp() - lt.exp()).abs().max().item() < 1e-3
    assert (v - vt.reshape(-1)).abs().max().item() < 1e-3
    # fused head on/off agree exactly on this path too
    nf_b = NativeForward(net, max_batch=n, fused_head=False)
    lb, vb = (t.cpu() for t in nf_b.forward_planes(x))
    assert torch.equal(lb, logp) and torch.equal(vb, v)


def test_tc_trunk_without_a_fusable_stem_is_rejected():
    """Mode 'tc' starts every forward with the fused stem (4 planes without BatchNorm, or Go's 17): a trunk with any
    other first layer still constructs -- MuZeroNative packs its dynamics trunk this way -- but does not run."""
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    from rlzero_b200.games.gomoku.gomoku_env import GomokuEnv
    nf = NativeForward(ResNetPolicyValueNet(9, n_blocks=1, in_planes=8).cuda().eval())
    assert nf.mode == 'tc' and nf.stem is None
    e = GomokuEnv(9, 5)
    e.reset()
    rows, meta = e.device_state()[0].cuda(), e.device_state()[1].cuda()
    with pytest.raises(ValueError, match='fused stem'):
        nf.forward_boards(rows, meta, 1)
    with pytest.raises(ValueError, match='fused stem'):
        nf.forward_planes(np.zeros((1, 8, 9, 9), dtype=np.float32))


@pytest.mark.parametrize('h,w,a,blocks,n', [(6, 7, 7, 3, 300), (6, 6, None, 2, 5), (3, 3, None, 1, 17), (7, 7, None, 1, 130)])
def test_row_stride_8_forward_vs_torch_and_tc2_stride_16(h, w, a, blocks, n):
    """Boards up to 7x7 (Connect Four 6x7 = BASELINE config 2, TicTacToe 3x3) run on the 8-stride padded layout
    (64 rows per board instead of 256, revision 3): whole forward within 1e-3 of PyTorch fp32, fused head on/off and
    planes-/bitboard-fed stems bit-identical, and the same network forced onto the 16-stride layout, where revision 2
    runs, agrees (same bf16 products; revision 2 sums them tap-outer, revision 3 k-block-outer)."""
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    torch.manual_seed(h * 10 + w)
    kw = dict(board_width=w, n_actions=a) if a is not None else dict(board_width=w)
    net = ResNetPolicyValueNet(h, n_blocks=blocks, **kw).cuda().eval()
    nf = NativeForward(net, max_batch=n)
    assert nf.mode == 'tc' and nf.S == 8 and nf.P == 64
    rs = np.random.RandomState(n)
    x = rs.randint(0, 2, size=(n, 4, h, w)).astype(np.float32)
    logp, v = (t.cpu().clone() for t in nf.forward_planes(x))
    ref = ResNetPolicyValueNet(h, n_blocks=blocks, **kw).eval()
    ref.load_state_dict({k: t.cpu() for k, t in net.state_dict().items()})
    with torch.no_grad():
        lt, vt = ref(torch.from_numpy(x))
    A = nf.A
    assert (logp[:, :A].exp() - lt.exp()).abs().max().item() < 1e-3
    assert (v - vt.reshape(-1)).abs().max().item() < 1e-3
    nf_b = NativeForward(net, max_batch=n, fused_head=False)
    assert nf_b.S == 8
    lb, vb = (t.cpu() for t in nf_b.forward_planes(x))
    assert torch.equal(lb[:, :A], logp[:, :A]) and torch.equal(vb, v)
    nf16 = NativeForward(net, max_batch=n, row_stride=16)
    assert nf16.S == 16
    l16, v16 = (t.cpu() for t in nf16.forward_planes(x))
    assert (l16[:, :A].exp() - logp[:, :A].exp()).abs().max().item() < 1e-4 and (v16 - v).abs().max().item() < 1e-3
    # padding squares and the rows beyond the last board stay zero (they are every tap's halo)
    full = nf_b.bufs[0][:n * 64].reshape(n, 8, 8, 128).float()
    assert full[:, h:].abs().max().item() == 0.0 and full[:, :, w:].abs().max().item() == 0.0
    with pytest.raises(ValueError):
        NativeForward(ResNetPolicyValueNet(9, n_blocks=1).cuda().eval(), row_stride=8)


@pytest.mark.parametrize('size,n', [(6, 37), (3, 4)])
def test_row_stride_8_stem_bitboards_vs_planes_and_torch(size, n):
    """The fused encoder + stem on the 8-stride layout: positions fed as device bitboards and as current_state
    planes give bit-identical outputs, equal to PyTorch's conv on the reference's planes (bf16 weights)."""
    from rlzero_b200 import _lib as L
    from rlzero_b200.games.gomoku.gomoku_env import GomokuEnv
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    torch.manual_seed(size)
    net = ResNetPolicyValueNet(size, n_blocks=1).cuda().eval()
    rs = np.random.RandomState(size)
    envs = []
    for i in range(n):
        e = GomokuEnv(size, min(4, size))
        e.reset()
        for m in rs.permutation(size * size)[:(0 if i == 0 else rs.randint(0, size * size - 1))]:
            e.step(int(m))
            if e.game_end_winner()[0]:
                break
        envs.append(e)
    rows = torch.cat([e.device_state()[0] for e in envs]).cuda()
    meta = torch.cat([e.device_state()[1] for e in envs]).cuda()
    nf = NativeForward(net, max_batch=n)
    assert nf.S == 8
    lib, g = L.load(), nf._gdesc()
    st = nf.stem
    rows_alloc = (n * 64 + 255) // 256 * 256
    fused = torch.full((rows_alloc, 128), 3.0, dtype=torch.bfloat16, device='cuda')
    L.check(lib.rz_net_stem_tc(C.byref(g), L.ptr(rows), L.ptr(meta), L.ptr(st['w']), L.ptr(st['b']), L.ptr(fused),
                               n, 1, 0, L.stream_ptr()), 'stem')
    planes = torch.tensor(np.stack([e.current_state() for e in envs]), dtype=torch.float32, device='cuda')
    fused_p = torch.full((rows_alloc, 128), 5.0, dtype=torch.bfloat16, device='cuda')
    L.check(lib.rz_net_stem_tc_planes(C.byref(g), L.ptr(planes.contiguous()), L.ptr(st['w']), L.ptr(st['b']),
                                      L.ptr(fused_p), n, 1, 0, L.stream_ptr()), 'stem planes')
    torch.cuda.synchronize()
    assert torch.equal(fused, fused_p)
    assert fused[n * 64:].abs().max().item() == 0.0 if rows_alloc > n * 64 else True
    full = fused[:n * 64].reshape(n, 8, 8, 128).float()
    assert full[:, size:].abs().max().item() == 0.0 and full[:, :, size:].abs().max().item() == 0.0
    wq = net.stem.weight.detach().to(torch.bfloat16).float()
    ref = torch.relu(torch.nn.functional.conv2d(planes, wq, net.stem.bias.detach(), padding=1))
    got = full[:, :size, :size].permute(0, 3, 1, 2)
    assert (got - ref).abs().max().item() <= 2.0 ** -8 * max(1.0, ref.abs().max().item()) + 1e-6
    lp1, v1 = (t.clone() for t in nf.forward_boards(rows, meta, n))
    lp3, v3 = nf.forward_planes(planes.cpu().numpy())
    assert torch.equal(lp3[:, :size * size], lp1[:, :size * size]) and torch.equal(v3, v1)


@pytest.mark.parametrize('h,w,a,planes,n', [(15, 15, None, 4, 300), (15, 15, None, 4, 1), (19, 19, 362, 17, 131),
                                            (6, 7, 7, 4, 257), (3, 3, None, 4, 5), (9, 9, None, 4, 128)])
def test_heads_on_the_tensor_cores_match_float64_heads(h, w, a, planes, n):
    """rz_net_heads_tc (both FCs as one tcgen05 GEMM over the padded feature row, bf16 hi/lo split) against the
    heads' FC layers in float64 on the same features: float32-level agreement (the split drops only the lo*lo term),
    for every padded layout (S = 8 / 16 / 20), AS = 32 ... 384 (two N pieces for Go), partial last tile;
    fused-head and separate-feature routes are bit-identical."""
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    torch.manual_seed(h * 31 + n)
    kw = dict(board_width=w, in_planes=planes)
    if a is not None:
        kw['n_actions'] = a
    net = ResNetPolicyValueNet(h, n_blocks=1, **kw).cuda().eval()
    with torch.no_grad():   # heads with some dynamic range: a peaked policy, a value away from 0
        net.act_fc1.weight.mul_(8.0)
        net.val_fc1.weight.mul_(4.0)
        net.val_fc2.weight.mul_(4.0)
    x = np.random.RandomState(n).randint(0, 2, size=(n, planes, h, w)).astype(np.float32)
    tc = NativeForward(net, max_batch=n)
    lt, vt = (t.clone() for t in tc.forward_planes(x))
    A = tc.A
    assert torch.isfinite(lt).all() and torch.isfinite(vt).all()
    # the features the kernel consumed, at the board squares of the padded layout, in the reference's flatten order
    fe = tc.feat[:n].double().view(n, 6, tc.S, tc.S)[:, :, :h, :w]
    with torch.no_grad():
        d = {k: t.double() for k, t in net.state_dict().items()}
        lc = torch.log_softmax(fe[:, :4].reshape(n, -1) @ d['act_fc1.weight'].t() + d['act_fc1.bias'], dim=1)
        hid = torch.relu(fe[:, 4:].reshape(n, -1) @ d['val_fc1.weight'].t() + d['val_fc1.bias'])
        vc = torch.tanh(hid @ d['val_fc2.weight'].t() + d['val_fc2.bias']).reshape(-1)
    # a few float32 ulps of the largest |log p| (the scaled heads reach ~30)
    assert (lt[:, :A] - lc).abs().max().item() < 1e-4, (lt[:, :A] - lc).abs().max().item()
    assert (lt[:, :A].double().exp() - lc.exp()).abs().max().item() < 1e-5
    assert (vt.double() - vc).abs().max().item() < 1e-5
    assert torch.allclose(lt[:, :A].exp().sum(1), torch.ones(n, device='cuda'), atol=1e-4)
    assert tc.logp[:n, A:].abs().max().item() == 0.0 if tc.AS > A else True
    tb = NativeForward(net, max_batch=n, fused_head=False)
    lb, vb = tb.forward_planes(x)
    assert torch.equal(lb, lt) and torch.equal(vb, vt)
    # against PyTorch fp32 end to end
    ref = ResNetPolicyValueNet(h, n_blocks=1, **kw).eval()
    ref.load_state_dict({k: t.cpu() for k, t in net.state_dict().items()})
    with torch.no_grad():
        lr, vr = ref(torch.from_numpy(x))
    # (the scaled-up head weights amplify the bf16 error of the trunk: looser than the 1e-3 of the stock scale)
    assert (lt[:, :A].exp().cpu() - lr.exp()).abs().max().item() < 1e-2
    assert (vt.cpu() - vr.reshape(-1)).abs().max().item() < 2e-2


@pytest.mark.parametrize('size,n', [(15, 37), (9, 5), (6, 130)])
def test_stock_net_on_the_tensor_core_path(size, n):
    """The reference's PolicyValueNet (4 -> 32 -> 64 -> 128) zero-padded onto the bf16 tensor-core trunk (mode 'tc',
    opt-in): within the north star's bf16 tolerance (1e-3) of PyTorch fp32, padding channels exactly zero, search
    through the reference API works with it."""
    from rlzero_b200.games.gomoku import GomokuEnv
    from rlzero_b200.games.gomoku.alphazero_agent import AlphaZeroAgent
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, PolicyValueNet
    from rlzero_b200.mcts import AlphaZeroMCTS
    torch.manual_seed(size)
    net = PolicyValueNet(size).cuda().eval()
    nf = NativeForward(net, max_batch=n, mode='tc')
    assert nf.mode == 'tc' and all(l['cout'] == 128 for l in nf.layers)
    assert NativeForward(net, max_batch=1).mode == 'tc32'       # the default: float32-accurate tensor-core path
    x = _random_boards(n, size, 9)
    logp, v = (t.cpu() for t in nf.forward_planes(x))
    ref = PolicyValueNet(size).eval()
    ref.load_state_dict({k: t.cpu() for k, t in net.state_dict().items()})
    with torch.no_grad():
        lt, vt = ref(torch.from_numpy(x))
    assert (logp.exp() - lt.exp()).abs().max().item() < 1e-3
    assert (v - vt.reshape(-1)).abs().max().item() < 1e-3
    nb = NativeForward(net, max_batch=n, mode='tc', fused_head=False)
    nb.forward_planes(x)
    P = nb.P
    mid = nb.bufs[1][:n * P].float()           # output of the padded 32 -> 64 layer (ping-pong buffer 1): channels 64.. are zero
    assert mid[:, 64:].abs().max().item() == 0.0 and mid[:, :64].abs().max().item() > 0.0
    agent = AlphaZeroAgent(size, net=net, mode='tc')
    env = GomokuEnv(size, min(5, size))
    env.reset()
    acts, probs = AlphaZeroMCTS(agent.policy_value_fn, n_playout=40).simulate(env, 1.0)
    assert len(acts) == size * size and abs(probs.sum() - 1.0) < 1e-9


@pytest.mark.parametrize('h,cin,cout,relu,res', [(15, 64, 128, 1, 0), (15, 4, 32, 1, 0), (9, 32, 64, 0, 1), (19, 64, 128, 1, 1)])
def test_fp32_conv_tiled_and_scalar_kernels_are_bit_identical(h, cin, cout, relu, res):
    """rz_net_conv3x3_f32 picks the register-tiled kernel for batches (>= 64 boards) and the scalar one for a handful
    of boards: the same boards through both give the same bits (same fmaf order per output), and match PyTorch."""
    from rlzero_b200 import _lib as L
    lib = L.load()
    torch.manual_seed(h + cin)
    n = 96
    x = torch.randn(n, h * h, cin, device='cuda')
    w = (torch.randn(9, cin, cout, device='cuda') / (3.0 * cin ** 0.5)).contiguous()
    b = torch.randn(cout, device='cuda') * 0.1
    r = torch.randn(n, h * h, cout, device='cuda') if res else None
    big = torch.full((n, h * h, cout), 7.0, device='cuda')
    L.check(lib.rz_net_conv3x3_f32(L.ptr(x), L.ptr(w), L.ptr(b), L.ptr(r), L.ptr(big), n, h, cin, cout, relu,
                                   L.stream_ptr()), 'tiled')
    small = torch.full((n, h * h, cout), 5.0, device='cuda')
    for i in range(0, n, 32):
        rr = r[i:i + 32].contiguous() if res else None
        xi, oi = x[i:i + 32].contiguous(), torch.empty(32, h * h, cout, device='cuda')
        L.check(lib.rz_net_conv3x3_f32(L.ptr(xi), L.ptr(w), L.ptr(b), L.ptr(rr), L.ptr(oi), 32, h, cin, cout, relu,
                                       L.stream_ptr()), 'scalar')
        small[i:i + 32] = oi
    torch.cuda.synchronize()
    assert torch.equal(big, small)
    xt = x.reshape(n, h, h, cin).permute(0, 3, 1, 2).double()
    wt = w.reshape(3, 3, cin, cout).permute(3, 2, 0, 1).double()
    ref = torch.nn.functional.conv2d(xt, wt, b.double(), padding=1).permute(0, 2, 3, 1).reshape(n, h * h, cout)
    if res:
        ref = ref + r.double()
    if relu:
        ref = torch.relu(ref)
    assert (big.double() - ref).abs().max().item() < 1e-4
