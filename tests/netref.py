"""Plain float64 references of the network and of the root prior rules, shared by the network and search tests."""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

from oracle import kv_oracle as O


def bnrand_net(seed=0, **kw):
    """ChessNet with the weights of oracle/gen_golden.py's recipe: non-trivial BN statistics, so folding is exercised."""
    from knightvision_b200.model import ChessNet
    torch.manual_seed(seed)
    net = ChessNet(**kw).eval()
    g = torch.Generator().manual_seed(1)
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.05)
            m.running_var.copy_(1.0 + 0.2 * torch.rand(m.running_var.shape, generator=g))
            m.weight.data.copy_(1.0 + 0.1 * torch.randn(m.weight.shape, generator=g))
            m.bias.data.copy_(0.05 * torch.randn(m.bias.shape, generator=g))
    return net


def live_heads(net):
    """Shift the BatchNorm of both 1x1 heads up by 0.5: with the default initialisation their two / one channels are
    often negative at every square after the ReLU, and policy and value then do not depend on the tower at all."""
    with torch.no_grad():
        net.policy_bn.bias.add_(0.5)
        net.value_bn.bias.add_(0.5)
    return net


class Fp64Net:
    """float64 copy of model._fp32_graph (the graph of ai/model.py:51-77, eval-mode BatchNorm) on `device`."""

    def __init__(self, net, device):
        self.sd = {k: v.detach().to(device, torch.float64) for k, v in net.state_dict().items()}
        self.arch = net.arch
        self.eps = {n + ".": m.eps for n, m in net.named_modules() if isinstance(m, torch.nn.BatchNorm2d)}

    def bn(self, p, t):
        s = self.sd
        return F.batch_norm(t, s[p + ".running_mean"], s[p + ".running_var"], s[p + ".weight"], s[p + ".bias"], False, 0.0,
                            self.eps[p + "."])

    def conv(self, p, t, pad=1):
        return F.conv2d(t, self.sd[p + ".weight"], self.sd[p + ".bias"], padding=pad)

    def tower_layers(self):
        """[(conv, bn, residual input = k convs back or None)] in the order of kv_net_forward_partial."""
        L = [("conv2", "bn2", None)] if self.arch[3] else []
        for i in range(self.arch[2]):
            L += [(f"res_blocks.{i}.conv1", f"res_blocks.{i}.bn1", None), (f"res_blocks.{i}.conv2", f"res_blocks.{i}.bn2", 2)]
        return L

    def stem(self, x):
        return F.relu(self.bn("bn1", self.conv("conv1", x.double())))

    def layer(self, k, h, res=None):
        conv, bn, _ = self.tower_layers()[k]
        t = self.bn(bn, self.conv(conv, h))
        return F.relu(t + res if res is not None else t)

    def heads(self, h):
        s = self.sd
        p = F.relu(self.bn("policy_bn", self.conv("policy_conv", h, 0))).flatten(1)
        p = F.linear(p, s["policy_fc.weight"], s["policy_fc.bias"])
        v = F.relu(self.bn("value_bn", self.conv("value_conv", h, 0))).flatten(1)
        v = F.relu(F.linear(v, s["value_fc1.weight"], s["value_fc1.bias"]))
        v = torch.tanh(F.linear(v, s["value_fc2.weight"], s["value_fc2.bias"]))
        return p, v

    def forward(self, x):
        h = self.stem(x)
        acts = [h]
        for k, (_, _, r) in enumerate(self.tower_layers()):
            h = self.layer(k, h, acts[-r] if r else None)
            acts.append(h)
        return self.heads(h)


def reference_rule_priors(logits, moves, alpha, eps, seed, game_id, ply):
    """scripts/self_play.py:150-167 in float64 (see tests/test_emu_mcts.py): softmax over all 4096 logits, Dirichlet
    noise over all 4096 indices, mixed with eps, the legal entries renormalised."""
    p = np.exp(logits.astype(np.float64) - logits.max())
    p /= p.sum()
    if eps > 0:
        g = O.root_noise(alpha, seed, game_id, ply).astype(np.float64)
        p = (1 - eps) * p + eps * g / g.sum()
    w = p[[O.lib().kvo_move_index(int(m)) for m in moves]]
    return w / w.sum()
