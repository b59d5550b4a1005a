"""CPU tests: the numpy restatement of the reference's training step (oracle/train_oracle.py: forward, hand-derived
backward, Adam) against PyTorch autograd / torch.optim.Adam in float64 -- and against the LIVE reference's
AlphaZeroAgent.learn where RLZERO_REFERENCE_ROOT names an RLZero checkout."""
import numpy as np
import pytest
import torch

from oracle import ref_loader, train_oracle


def _module(size, seed):
    from rlzero_b200.games.gomoku.policy_value_net import PolicyValueNet
    torch.manual_seed(seed)
    return PolicyValueNet(size).double()


def _batch(size, n, seed):
    rs = np.random.RandomState(seed)
    x = (rs.rand(n, 4, size, size) < 0.35).astype(np.float64)
    pi = rs.dirichlet(np.ones(size * size), size=n)
    z = rs.choice([-1.0, 0.0, 1.0], size=n)
    return x, pi, z


@pytest.mark.parametrize('size,n', [(3, 5), (6, 8), (9, 3)])
def test_loss_and_gradients_match_autograd(size, n):
    net = _module(size, size)
    x, pi, z = _batch(size, n, size + 1)
    p = {k: v.detach().numpy().copy() for k, v in net.state_dict().items()}
    loss, entropy, g = train_oracle.loss_and_grads(p, x, pi, z)
    log_p, v = net(torch.from_numpy(x))
    tl = torch.nn.functional.mse_loss(v.view(-1), torch.from_numpy(z)) - torch.mean(torch.sum(torch.from_numpy(pi) * log_p, dim=1))
    tl.backward()
    te = -torch.mean(torch.sum(torch.exp(log_p) * log_p, dim=1))
    assert abs(loss - tl.item()) < 1e-12 and abs(entropy - te.item()) < 1e-12
    for k, prm in net.named_parameters():
        assert g[k].shape == tuple(prm.shape), k
        assert np.abs(g[k] - prm.grad.numpy()).max() < 1e-12, k


def test_pinning_the_oracles_own_masks_changes_nothing():
    """masks= set to the masks the unpinned oracle forms itself: the same log p, v, loss, entropy and gradients."""
    size, n = 6, 8
    net = _module(size, 3)
    x, pi, z = _batch(size, n, 4)
    p = {k: v.detach().numpy().copy() for k, v in net.state_dict().items()}
    log_p, v, c = train_oracle.forward(p, x)
    loss, entropy, g = train_oracle.loss_and_grads(p, x, pi, z)
    masks = {k: c[k] > 0 for k in ('a1', 'a2', 'a3', 'pa', 'va', 'h')}
    assert all(0 < m.mean() < 1 for m in masks.values())
    log_p2, v2, _ = train_oracle.forward(p, x, masks=masks)
    loss2, entropy2, g2 = train_oracle.loss_and_grads(p, x, pi, z, masks=masks)
    assert np.array_equal(log_p, log_p2) and np.array_equal(v, v2)
    assert loss == loss2 and entropy == entropy2
    for k in g:
        assert np.array_equal(g[k], g2[k]), k


def _masked_torch_net(net, masks):
    """PolicyValueNet's forward (policy_value_net.py:34-52) with every ReLU replaced by the product with a fixed mask."""
    F = torch.nn.functional
    m = {k: torch.from_numpy(v.astype(np.float64)) for k, v in masks.items()}

    def run(obs):
        a = F.conv2d(obs, net.conv1.weight, net.conv1.bias, padding=1) * m['a1']
        a = F.conv2d(a, net.conv2.weight, net.conv2.bias, padding=1) * m['a2']
        a = F.conv2d(a, net.conv3.weight, net.conv3.bias, padding=1) * m['a3']
        pa = net.act_conv1(a) * m['pa']
        log_p = F.log_softmax(net.act_fc1(pa.reshape(obs.shape[0], -1)), dim=1)
        va = net.val_conv1(a) * m['va']
        h = net.val_fc1(va.reshape(obs.shape[0], -1)) * m['h']
        return log_p, torch.tanh(net.val_fc2(h))
    return run


@pytest.mark.parametrize('size,n', [(3, 5), (6, 8)])
def test_pinned_masks_match_autograd_of_the_masked_network(size, n):
    """Random masks, independent of the signs of the pre-activations: loss, entropy and all 16 gradients equal float64
    autograd of the network whose ReLUs are multiplications by those masks."""
    net = _module(size, size + 20)
    x, pi, z = _batch(size, n, size + 21)
    p = {k: v.detach().numpy().copy() for k, v in net.state_dict().items()}
    rs = np.random.RandomState(size)
    shapes = dict(a1=(n, 32, size, size), a2=(n, 64, size, size), a3=(n, 128, size, size), pa=(n, 4, size, size),
                  va=(n, 2, size, size), h=(n, 64))
    masks = {k: rs.rand(*s) < 0.6 for k, s in shapes.items()}
    loss, entropy, g = train_oracle.loss_and_grads(p, x, pi, z, masks=masks)
    _, _, c = train_oracle.forward(p, x)
    unpinned = sum(int((masks[k] != (c[k] > 0)).sum()) for k in shapes)
    assert unpinned > 0.3 * sum(int(np.prod(s)) for s in shapes.values())     # the masks are not the ReLUs' own
    log_p, v = _masked_torch_net(net, masks)(torch.from_numpy(x))
    tl = torch.nn.functional.mse_loss(v.view(-1), torch.from_numpy(z)) - torch.mean(torch.sum(torch.from_numpy(pi) * log_p, dim=1))
    tl.backward()
    te = -torch.mean(torch.sum(torch.exp(log_p) * log_p, dim=1))
    assert abs(loss - tl.item()) < 1e-12 and abs(entropy - te.item()) < 1e-12
    named = dict(net.named_parameters())
    assert len(named) == len(g) == 16
    for k, prm in named.items():
        assert g[k].shape == tuple(prm.shape), k
        assert np.abs(g[k] - prm.grad.numpy()).max() < 1e-12, k


def test_three_adam_steps_match_torch_optim():
    size, n = 6, 8
    net = _module(size, 1)
    opt = torch.optim.Adam(net.parameters(), lr=2e-3, weight_decay=1e-4)
    p = {k: v.detach().numpy().copy() for k, v in net.state_dict().items()}
    state = {}
    for step in range(3):
        x, pi, z = _batch(size, n, 10 + step)
        loss, _, g = train_oracle.loss_and_grads(p, x, pi, z)
        p = train_oracle.adam_step(p, g, state, lr=2e-3, weight_decay=1e-4)
        log_p, v = net(torch.from_numpy(x))
        tl = torch.nn.functional.mse_loss(v.view(-1), torch.from_numpy(z)) - torch.mean(torch.sum(torch.from_numpy(pi) * log_p, dim=1))
        opt.zero_grad()
        tl.backward()
        opt.step()
        assert abs(loss - tl.item()) < 1e-11
    for k, prm in net.named_parameters():
        assert np.abs(p[k] - prm.detach().numpy()).max() < 1e-11, k


@pytest.mark.skipif(not ref_loader.available(), reason='no RLZero checkout (set RLZERO_REFERENCE_ROOT)')
def test_one_learn_step_matches_the_live_reference_agent():
    """AlphaZeroAgent.learn of the UNMODIFIED reference (float32, its own Adam) against the oracle in float64 from the
    same initial weights: loss / entropy within float32 accuracy, updated weights within 1e-5."""
    ref = ref_loader.load()
    size, n = 6, 16
    torch.manual_seed(4)
    agent = ref.AlphaZeroAgent(size, device='cpu')
    p = {k: v.detach().numpy().astype(np.float64) for k, v in agent.policy_value_net.state_dict().items()}
    x, pi, z = _batch(size, n, 5)
    loss, entropy, g = train_oracle.loss_and_grads(p, x, pi, z)
    p = train_oracle.adam_step(p, g, {}, lr=agent.optimizer.param_groups[0]['lr'],
                               weight_decay=agent.optimizer.param_groups[0]['weight_decay'])
    rl, re_ = agent.learn(list(x.astype(np.float32)), list(pi.astype(np.float32)), list(z.astype(np.float32)))
    assert abs(rl - loss) < 1e-5 and abs(re_ - entropy) < 1e-5
    for k, v in agent.policy_value_net.state_dict().items():
        assert np.abs(v.numpy() - p[k]).max() < 1e-5, k
