"""TEST INFRASTRUCTURE ONLY -- numpy (float64) restatement of the reference's training step.

Follows ``AlphaZeroAgent.learn`` (rlzero/games/gomoku/alphazero_agent.py:59-86) on the stock
``PolicyValueNet`` (rlzero/games/gomoku/policy_value_net.py:6-52):

    loss = mse(v, z) - mean_b sum_a pi[b, a] * log p[b, a]          (:70-75; the L2 term lives in Adam's weight_decay)
    entropy = -mean_b sum_a p * log p                               (:83-85, monitoring only)
    Adam(lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4)       (:22-24, torch.optim.Adam semantics)

with the forward pass, the analytic backward pass and the optimiser update written out by hand -- no autograd -- so
that a hand-written backward pass on the device (a next-round item: today the product's ``learn`` is PyTorch autograd
on device tensors) has an oracle to be checked against.  Pinned by ``tests/test_train_oracle.py`` against PyTorch
autograd in float64 on the CPU.  Parameters use the module's own names and layouts (``state_dict``).
"""
import numpy as np


def _conv3x3(x, w, b):
    """x [B,Cin,H,W], w [Cout,Cin,3,3], b [Cout] -> [B,Cout,H,W], zero padding 1 (nn.Conv2d(..., 3, padding=1))."""
    B, C, H, W = x.shape
    xp = np.zeros((B, C, H + 2, W + 2), dtype=x.dtype)
    xp[:, :, 1:-1, 1:-1] = x
    out = np.zeros((B, w.shape[0], H, W), dtype=x.dtype)
    for kh in range(3):
        for kw in range(3):
            out += np.einsum('bchw,oc->bohw', xp[:, :, kh:kh + H, kw:kw + W], w[:, :, kh, kw])
    return out + b[None, :, None, None]


def _conv3x3_backward(x, w, dy):
    """Gradients of _conv3x3: (dx, dw, db)."""
    B, C, H, W = x.shape
    xp = np.zeros((B, C, H + 2, W + 2), dtype=x.dtype)
    xp[:, :, 1:-1, 1:-1] = x
    dxp = np.zeros_like(xp)
    dw = np.zeros_like(w)
    for kh in range(3):
        for kw in range(3):
            patch = xp[:, :, kh:kh + H, kw:kw + W]
            dw[:, :, kh, kw] = np.einsum('bohw,bchw->oc', dy, patch)
            dxp[:, :, kh:kh + H, kw:kw + W] += np.einsum('bohw,oc->bchw', dy, w[:, :, kh, kw])
    return dxp[:, :, 1:-1, 1:-1], dw, dy.sum(axis=(0, 2, 3))


_MASKED = ('a1', 'a2', 'a3', 'pa', 'va', 'h')


def _relu(z, masks, name):
    """max(z, 0), or z times the fixed 0/1 mask ``masks[name]`` (a ReLU pinned to given masks)."""
    if masks is None:
        return np.maximum(z, 0.0)
    m = np.asarray(masks[name], dtype=bool)
    if m.shape != z.shape:
        raise ValueError('mask %s has shape %s, the activation %s' % (name, m.shape, z.shape))
    return z * m


def forward(p, x, masks=None):
    """The stock network (policy_value_net.py:34-52).  Returns (log_p [B,HW], v [B,1], cache of activations).

    ``masks``: None, or {'a1', 'a2', 'a3', 'pa', 'va', 'h': boolean arrays in the shapes of those activations}; each
    ReLU then multiplies by its mask instead of testing the sign (and ``loss_and_grads`` back-propagates through the same
    masks).  With the masks a device produced, the float64 result differs from the device's only by rounding: a
    pre-activation within rounding of zero cannot land on the other side of the ReLU than on the device."""
    B = x.shape[0]
    a1 = _relu(_conv3x3(x, p['conv1.weight'], p['conv1.bias']), masks, 'a1')
    a2 = _relu(_conv3x3(a1, p['conv2.weight'], p['conv2.bias']), masks, 'a2')
    a3 = _relu(_conv3x3(a2, p['conv3.weight'], p['conv3.bias']), masks, 'a3')
    pa = _relu(np.einsum('bchw,oc->bohw', a3, p['act_conv1.weight'][:, :, 0, 0])
               + p['act_conv1.bias'][None, :, None, None], masks, 'pa')
    pf = pa.reshape(B, -1)                                   # x.view(-1, 4*H*W): channel-major flatten
    logits = pf @ p['act_fc1.weight'].T + p['act_fc1.bias']
    m = logits.max(axis=1, keepdims=True)
    log_p = logits - m - np.log(np.exp(logits - m).sum(axis=1, keepdims=True))
    va = _relu(np.einsum('bchw,oc->bohw', a3, p['val_conv1.weight'][:, :, 0, 0])
               + p['val_conv1.bias'][None, :, None, None], masks, 'va')
    vf = va.reshape(B, -1)
    h = _relu(vf @ p['val_fc1.weight'].T + p['val_fc1.bias'], masks, 'h')
    v = np.tanh(h @ p['val_fc2.weight'].T + p['val_fc2.bias'])
    if masks is None:
        relu_masks = dict(a1=a1 > 0, a2=a2 > 0, a3=a3 > 0, pa=pa > 0, va=va > 0, h=h > 0)
    else:
        relu_masks = {k: np.asarray(masks[k], dtype=bool) for k in _MASKED}
    return log_p, v, dict(x=x, a1=a1, a2=a2, a3=a3, pa=pa, pf=pf, va=va, vf=vf, h=h, v=v, log_p=log_p, masks=relu_masks)


def loss_and_grads(p, x, pi, z, masks=None):
    """(loss, entropy, grads) of alphazero_agent.py:66-85; grads keyed like the state_dict.  ``masks``: as in
    ``forward`` (the backward pass uses the same masks as the forward)."""
    B = x.shape[0]
    log_p, v, c = forward(p, x, masks)
    m = c['masks']
    value_loss = np.mean((v.reshape(-1) - z) ** 2)
    policy_loss = -np.mean(np.sum(pi * log_p, axis=1))
    loss = value_loss + policy_loss
    prob = np.exp(log_p)
    entropy = -np.mean(np.sum(prob * log_p, axis=1))
    g = {}
    # value head
    dv = (2.0 * (v.reshape(-1) - z) / B).reshape(B, 1)
    dpre2 = dv * (1.0 - v ** 2)                              # tanh'
    g['val_fc2.weight'] = dpre2.T @ c['h']
    g['val_fc2.bias'] = dpre2.sum(axis=0)
    dh = (dpre2 @ p['val_fc2.weight']) * m['h']
    g['val_fc1.weight'] = dh.T @ c['vf']
    g['val_fc1.bias'] = dh.sum(axis=0)
    dva = (dh @ p['val_fc1.weight']).reshape(c['va'].shape) * m['va']
    g['val_conv1.weight'] = np.einsum('bohw,bchw->oc', dva, c['a3'])[:, :, None, None]
    g['val_conv1.bias'] = dva.sum(axis=(0, 2, 3))
    da3 = np.einsum('bohw,oc->bchw', dva, p['val_conv1.weight'][:, :, 0, 0])
    # policy head: d(-mean sum pi log_softmax) / dlogits = (softmax * sum_a pi - pi) / B
    dlogits = (prob * pi.sum(axis=1, keepdims=True) - pi) / B
    g['act_fc1.weight'] = dlogits.T @ c['pf']
    g['act_fc1.bias'] = dlogits.sum(axis=0)
    dpa = (dlogits @ p['act_fc1.weight']).reshape(c['pa'].shape) * m['pa']
    g['act_conv1.weight'] = np.einsum('bohw,bchw->oc', dpa, c['a3'])[:, :, None, None]
    g['act_conv1.bias'] = dpa.sum(axis=(0, 2, 3))
    da3 = da3 + np.einsum('bohw,oc->bchw', dpa, p['act_conv1.weight'][:, :, 0, 0])
    # trunk
    dz3 = da3 * m['a3']
    da2, g['conv3.weight'], g['conv3.bias'] = _conv3x3_backward(c['a2'], p['conv3.weight'], dz3)
    dz2 = da2 * m['a2']
    da1, g['conv2.weight'], g['conv2.bias'] = _conv3x3_backward(c['a1'], p['conv2.weight'], dz2)
    dz1 = da1 * m['a1']
    _, g['conv1.weight'], g['conv1.bias'] = _conv3x3_backward(c['x'], p['conv1.weight'], dz1)
    return float(loss), float(entropy), g


def adam_step(p, g, state, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4):
    """torch.optim.Adam (L2 weight decay folded into the gradient, bias-corrected moments):
    g += wd * p; m = b1 m + (1 - b1) g; v = b2 v + (1 - b2) g^2; p -= lr / (1 - b1^t) * m / (sqrt(v) / sqrt(1 - b2^t) + eps).
    ``state``: {'step': t, 'm': {...}, 'v': {...}} updated in place (created on first use)."""
    if 'step' not in state:
        state.update(step=0, m={k: np.zeros_like(v) for k, v in p.items()}, v={k: np.zeros_like(v) for k, v in p.items()})
    state['step'] += 1
    t = state['step']
    b1, b2 = betas
    for k in p:
        grad = g[k] + weight_decay * p[k]
        state['m'][k] = b1 * state['m'][k] + (1 - b1) * grad
        state['v'][k] = b2 * state['v'][k] + (1 - b2) * grad * grad
        denom = np.sqrt(state['v'][k]) / np.sqrt(1 - b2 ** t) + eps
        p[k] = p[k] - (lr / (1 - b1 ** t)) * state['m'][k] / denom
    return p
