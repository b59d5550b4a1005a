"""``AlphaZeroAgent`` with the reference's API (rlzero/games/gomoku/alphazero_agent.py:12-125).

Inference (``policy_value_fn``, ``policy_value``, ``predict``) runs on the hand-written CUDA
forward (``NativeForward``); ``policy_value_fn`` additionally carries a ``device_evaluator`` so
that ``AlphaZeroMCTS`` evaluates whole waves of leaves on the device without the per-leaf
host round trip the reference makes (alphazero_agent.py:41-45).  ``learn`` (:59-86) runs on the
hand-written training kernels (``rlzero_b200.learn.NativeTrainer``: forward with saved activations,
analytic backward, loss / entropy, Adam -- no autograd, cuDNN or cuBLAS) for the reference's own
``PolicyValueNet``; ``learn_autograd`` is the same step in plain PyTorch, kept as the checker and for
other modules.  The packed inference weights are refreshed after every step.
"""
import os

import numpy as np
import torch
import torch.nn.functional as F
import torch.optim as optim

from ...learn import make_trainer
from .policy_value_net import NativeForward, PolicyValueNet


class _PolicyValueFn(object):
    """Callable ``policy_value_fn(game_env) -> (zip(legal, probs), value)`` (:31-46)."""

    def __init__(self, agent):
        self._agent = agent

    @property
    def device_evaluator(self):
        return self._agent.native

    def __call__(self, game_env):
        agent = self._agent
        legal_positions = game_env.leagel_actions()
        state = np.ascontiguousarray(game_env.current_state()[None])     # [1,4,H,W] (:38-39)
        logp, value = agent.native.forward_planes(state)
        act_probs = np.exp(logp[0].cpu().numpy())
        return zip(legal_positions, act_probs[legal_positions]), float(value[0].item())


class AlphaZeroAgent(object):

    def __init__(self, board_size, learning_rate=0.001, weight_decay=1e-4, device='cuda',
                 net=None, mode=None, trainer=None):
        """``trainer``: 'native' (hand-written kernels: the float32 step for the reference's PolicyValueNet, the
        tensor-core step for ResNetPolicyValueNet on square boards up to 19x19 -- 4 input planes with H*W actions, or the
        17 planes of GoEnv.observe with H*W + 1 actions, the pass last) or 'autograd' (plain PyTorch: the checker, and
        any other module).  The default (None) is the native step for the reference's PolicyValueNet and for 4-plane
        ResNets up to 15x15, and autograd for everything else, Go networks and 16x16 .. 19x19 boards included: ask for
        'native' to train those on the tensor cores (the bf16 trunk's value error on trained networks, DESIGN section
        3.4, is measured at 15x15 only)."""
        self.board_size = board_size
        self.policy_value_net = net if net is not None else PolicyValueNet(board_size)
        self.policy_value_net.to(device)
        self.optimizer = optim.Adam(self.policy_value_net.parameters(), lr=learning_rate,
                                    weight_decay=weight_decay)
        self.device = device
        if trainer not in (None, 'native', 'native_tc', 'autograd'):
            raise ValueError("trainer must be 'native', 'native_tc' or 'autograd'")
        self.trainer = None
        if trainer != 'autograd':
            # re-points the module's parameters at one flat device buffer (state_dict / optimizer see the same tensors)
            # 'native_tc': the reference's own network with forward and data-gradient convolutions on the tensor cores as
            # well (16-mantissa-bit pairs: forward still within 1e-5, gradients within 1e-3..1e-2 of the float64 oracle
            # instead of 1e-5 -- tighter than PyTorch's default TF32 convolutions -- and 3x faster at batch 512)
            self.trainer = make_trainer(self.policy_value_net, tc_trunk=(trainer == 'native_tc'),
                                        requested=trainer in ('native', 'native_tc'),
                                        learning_rate=learning_rate, weight_decay=weight_decay, device=device)
            if self.trainer is None and trainer in ('native', 'native_tc'):
                raise ValueError('no native trainer fits this module (use trainer="autograd")')
        self.native = NativeForward(self.policy_value_net, mode=mode, device=device)
        self.policy_value_fn = _PolicyValueFn(self)

    def policy_value(self, state_batch):
        """a batch of states -> (action probabilities [B,HW], state values [B,1]) (:48-57)."""
        logp, value = self.native.forward_planes(np.array(state_batch))
        return np.exp(logp.cpu().numpy()), value.cpu().numpy().reshape(-1, 1)

    def policy_value_device(self, state_batch):
        """``policy_value`` for a device tensor [B,4,H,W], results left on the device (the batched training
        path: mini-batches gathered from the device replay buffer never visit the host)."""
        logp, value = self.native.forward_planes(state_batch)
        return torch.exp(logp).clone(), value.reshape(-1, 1).clone()

    def _f32(self, x):
        if isinstance(x, torch.Tensor):
            return x.to(device=self.device, dtype=torch.float32)
        return torch.FloatTensor(np.array(x)).to(self.device)

    def predict(self, state_batch):
        """(:88-97)"""
        return self.policy_value(state_batch)

    def learn(self, state_batch, mcts_probs, target_vs):
        """perform a training step: loss = (z - v)^2 - pi^T log p (+ L2 in the optimizer) (:59-86)."""
        if self.trainer is None:
            return self.learn_autograd(state_batch, mcts_probs, target_vs)
        loss, entropy = self.trainer.learn(self._f32(state_batch), self._f32(mcts_probs), self._f32(target_vs))
        self.native.refresh_weights()
        return loss, entropy

    def learn_autograd(self, state_batch, mcts_probs, target_vs):
        """The same step through PyTorch autograd (the checker of the native trainer; other network modules)."""
        net = self.policy_value_net
        net.train()
        dev = self.device
        state_batch = self._f32(state_batch)          # lists / numpy as in the reference, or device tensors
        mcts_probs = self._f32(mcts_probs)
        target_batch = self._f32(target_vs)
        log_act_probs, value = net(state_batch)
        value_loss = F.mse_loss(value.view(-1), target_batch)
        policy_loss = -torch.mean(torch.sum(mcts_probs * log_act_probs, dim=1))
        loss = value_loss + policy_loss
        self.optimizer.zero_grad()
        loss.backward()
        self.optimizer.step()
        entropy = -torch.mean(torch.sum(torch.exp(log_act_probs) * log_act_probs, dim=1))
        net.eval()
        self.native.refresh_weights()
        return loss.item(), entropy.item()

    def save_model(self, save_dir, model_name='model.th', opt_name='optimizer.th'):
        """(:99-111) same files and state_dict keys as the reference."""
        if not os.path.exists(save_dir):
            os.mkdir(save_dir)
        torch.save(self.policy_value_net.state_dict(), os.path.join(save_dir, model_name))
        opt_state = self.trainer.optimizer_state_dict() if self.trainer is not None else self.optimizer.state_dict()
        torch.save(opt_state, os.path.join(save_dir, opt_name))
        print('save model successfully!')

    def restore(self, save_dir, model_name='model.th', opt_name='optimizer.th'):
        """(:113-125)"""
        if not os.path.exists(save_dir):
            os.mkdir(save_dir)
        self.policy_value_net.load_state_dict(torch.load(os.path.join(save_dir, model_name)))
        opt_state = torch.load(os.path.join(save_dir, opt_name))
        if self.trainer is not None:
            self.trainer.load_optimizer_state_dict(opt_state)
            self.trainer.weights_changed()
        else:
            self.optimizer.load_state_dict(opt_state)
        self.native.refresh_weights()
        print('restore model successfully!')
