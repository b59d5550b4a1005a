"""GPU tests of the batched one-launch trunk (rz_net_trunk_tc2.cu): CTA pairs carry chunks of boards through every layer
behind the stem.  Per board it issues the per-layer kernel's MMAs and epilogue arithmetic, so its features, log-policy
and value must equal those of one launch per layer bit for bit."""
import numpy as np
import pytest
import torch
import torch.nn as nn

pytestmark = pytest.mark.gpu
FORCE_LAYERS = 1 << 30


def _random_planes(n, size, seed, width=None):
    """Positions with a random number of stones of both colours (vectorised: thousands of boards)."""
    width = width or size
    rs = np.random.RandomState(seed)
    x = np.zeros((n, 4, size, width), dtype=np.float32)
    fill = rs.rand(n, 1, 1) * 0.6
    u = rs.rand(n, size, width)
    x[:, 0] = u < fill[:, :, :] / 2
    x[:, 1] = (u >= fill / 2) & (u < fill)
    x[:, 3] = (np.arange(n) % 2)[:, None, None]
    last = rs.randint(0, size * width, n)
    x[np.arange(n), 2, last // width, last % width] = 1.0
    return x


def _perturbed(net, seed):
    """Non-trivial BatchNorm statistics, so that folded scales and biases matter."""
    g = torch.Generator(device='cpu').manual_seed(seed)
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.2)
                m.running_var.copy_(torch.rand(m.running_var.shape, generator=g) + 0.5)
                m.weight.copy_(torch.rand(m.weight.shape, generator=g) + 0.5)
                m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.2)
    return net


def _pair(net, n, **kw):
    """The same net twice: `a` on the batched trunk, `b` forced onto one launch per layer."""
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward
    a = NativeForward(net, max_batch=n, **kw)
    b = NativeForward(net, max_batch=n, **kw)
    b.batched_trunk_min = FORCE_LAYERS
    assert a._route(n) == 'batched' and a.kernels_per_forward(n) == 3
    assert b._route(n) == 'layers' and b.kernels_per_forward(n) > 3
    return a, b


def _run(nf, x):
    lp, v = nf.forward_planes(x)
    return nf.feat[:x.shape[0]].clone(), lp.clone(), v.clone()


def _assert_equal(a, b, x):
    fa, la, va = _run(a, x)
    fb, lb, vb = _run(b, x)
    n, hw = x.shape[0], x.shape[2] * x.shape[3]
    assert torch.isfinite(la[:, :hw]).all() and torch.isfinite(va).all()
    assert torch.equal(fa, fb), (fa - fb).abs().max()
    assert torch.equal(la, lb) and torch.equal(va, vb)
    return fa, la, va


@pytest.mark.parametrize('size,blocks,n', [(15, 10, 8192), (15, 10, 1500), (9, 2, 1100), (12, 3, 1037)])
def test_batched_trunk_equals_the_layer_kernels(size, blocks, n):
    """ResNet-10 at the headline's 8192 boards; 1500 boards leave ragged pairs (20 or 21 boards) and ragged chunks;
    9x9 and 12x12 put pad squares inside the 16x16 tile."""
    from rlzero_b200.games.gomoku.policy_value_net import ResNetPolicyValueNet
    torch.manual_seed(size + blocks)
    net = _perturbed(ResNetPolicyValueNet(size, n_blocks=blocks).cuda().eval(), size)
    a, b = _pair(net, n)
    x = _random_planes(n, size, n)
    _assert_equal(a, b, x)
    # a second launch on the same scratch gives the same bits
    fa2, la2, va2 = _run(a, x)
    fb, lb, vb = _run(b, x)
    assert torch.equal(fa2, fb) and torch.equal(la2, lb) and torch.equal(va2, vb)


class _OddTrunk(nn.Module):
    """ResNet blocks + one more 3x3 layer without skip and without ReLU: an odd number of layers behind the stem."""

    def __init__(self, size, n_blocks):
        super().__init__()
        from rlzero_b200.games.gomoku.policy_value_net import ResNetPolicyValueNet
        self.net = ResNetPolicyValueNet(size, n_blocks=n_blocks)
        self.extra = nn.Conv2d(128, 128, 3, padding=1)
        self.board_size = size
        for k in ('act_conv1', 'act_fc1', 'val_conv1', 'val_fc1', 'val_fc2'):
            setattr(self, k, getattr(self.net, k))

    def trunk_layers(self):
        return self.net.trunk_layers() + [(self.extra, None, None, False)]


@pytest.mark.parametrize('chunk,n_ctas', [(8, 0), (1, 0), (5, 6), (16, 148)])
def test_batched_trunk_with_an_odd_layer_count_and_other_chunks(chunk, n_ctas):
    """5 layers behind the stem, the last one without skip or ReLU; chunks of 1 (a weight reload after every tile),
    5 and 16 boards; 3 CTA pairs (every pair walks many chunks)."""
    torch.manual_seed(11)
    net = _perturbed(_OddTrunk(15, 2).cuda().eval(), 11)
    n = 1111
    a, b = _pair(net, n, n_ctas=n_ctas)
    a.trunk_chunk = chunk
    a.scratch = None               # re-sized for the new chunk on the next forward
    assert a.trunk_small['n'] == 5 and a.trunk_small['res_mask'] == 0b01010 and a.trunk_small['relu_mask'] == 0b01111
    _assert_equal(a, b, _random_planes(n, 15, 3))


def test_one_board_alone_equals_the_same_board_in_the_batch():
    """The board-by-board path (one-launch trunk_small) and the batched trunk agree bit for bit: what lets the oracle's
    single-board evaluations check a search that evaluates 8192 boards at once."""
    from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet
    torch.manual_seed(4)
    net = _perturbed(ResNetPolicyValueNet(15, n_blocks=10).cuda().eval(), 4)
    n = 8192
    nf = NativeForward(net, max_batch=n)
    x = _random_planes(n, 15, 21)
    assert nf._route(n) == 'batched' and nf._route(1) == 'small'
    f_all, l_all, v_all = _run(nf, x)
    for i in (0, 1, 110, 111, 4095, 8191):
        f1, l1, v1 = _run(nf, x[i:i + 1])
        assert torch.equal(f1[0], f_all[i]) and torch.equal(l1[0], l_all[i]) and torch.equal(v1[0], v_all[i]), i


def test_captured_batched_trunk_replays_and_recaptures_after_refresh():
    """A CUDA graph of the trunk + heads on the batched route replays the eager result; after refresh_weights
    (new weight tensors, new biases in the launch parameters) a new capture gives the new network's outputs."""
    from rlzero_b200 import _lib as L
    from rlzero_b200.games.gomoku.policy_value_net import ResNetPolicyValueNet
    torch.manual_seed(6)
    net = _perturbed(ResNetPolicyValueNet(15, n_blocks=3).cuda().eval(), 6)
    n = 2000
    a, b = _pair(net, n)
    x = _random_planes(n, 15, 8)

    def captured(nf):
        nf.forward_planes(x)                  # the stem's output in bufs[0], buffers and scratch allocated
        eager = (nf.logp[:n].clone(), nf.value[:n].clone())
        torch.cuda.synchronize()
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                assert L.stream_ptr().value == s.cuda_stream
                nf._trunk_and_heads(n, nf.logp, nf.value)
        nf.logp.zero_()
        nf.value.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(nf.logp[:n], eager[0]) and torch.equal(nf.value[:n], eager[1])
        return g, eager

    g1, e1 = captured(a)
    with torch.no_grad():
        for p in net.parameters():
            p.add_(torch.randn_like(p) * 0.05)
    version = a.weights_version
    a.refresh_weights()
    b.refresh_weights()
    assert a.weights_version > version
    g2, e2 = captured(a)
    _, lb, vb = _run(b, x)
    A = lb.shape[1]
    assert torch.equal(e2[0][:, :A], lb) and torch.equal(e2[1], vb) and not torch.equal(e1[0], e2[0])
