"""float64 torch restatement of the reference critics, differentiable by autograd - TEST INFRASTRUCTURE.

The same network as oracle/critic_ref.py (rls/model/ac_network_multi_gumbel.py:70-148 and
ac_network_model_multi_gumbel.py:69-143) spelled with the reference's building blocks - ``nn.Linear`` per agent,
``nn.LSTM(64, 64, batch_first=True)`` over the agent axis, ``bmm`` attention with the final hidden state, softmax over
agents - so that autograd gives the gradients the critic's backward kernel is compared with.  Never imported by the
product.
"""
import numpy as np
import torch
import torch.nn as nn

H = 64
KEYS = ['dense1.module.weight', 'dense1.module.bias', 'lstm.weight_ih_l0', 'lstm.weight_hh_l0', 'lstm.bias_ih_l0',
        'lstm.bias_hh_l0', 'dense2.weight', 'dense2.bias']
KEYS3 = ['dense3.weight', 'dense3.bias']


class _TimeDistributed(nn.Module):
    def __init__(self, module):
        super().__init__()
        self.module = module

    def forward(self, x):
        return self.module(x.reshape(-1, x.shape[-1])).reshape(*x.shape[:-1], -1)


class Critic64(nn.Module):
    """``Critic64(sd)``: float64 copy of the weights in ``sd`` (the reference's state_dict keys).  ``forward(obs,
    action)`` -> q, or (q, r) when ``sd`` has ``dense3``."""

    def __init__(self, sd, device='cpu'):
        super().__init__()
        din, out = np.shape(sd['dense1.module.weight'])[1], np.shape(sd['dense2.weight'])[0]
        self.model = 'dense3.weight' in sd
        self.dense1 = _TimeDistributed(nn.Linear(din, H))
        self.lstm = nn.LSTM(H, H, batch_first=True)
        self.dense2 = nn.Linear(H, out)
        if self.model:
            self.dense3 = nn.Linear(H, out)
        self.double().to(device)
        self.load_state_dict({k: torch.as_tensor(np.asarray(v, np.float64)) for k, v in _numpy(sd).items()})

    def keys(self):
        return KEYS + (KEYS3 if self.model else [])

    def pre_activations(self, obs, action):
        """(dense1 pre-activation [B,N,64], attention output before the relu [B,64]) - where relu kinks are."""
        z1 = self.dense1(torch.cat([obs, action], -1))
        out, (hn, _) = self.lstm(torch.relu(z1))
        return z1, self._attend(out, hn)

    @staticmethod
    def _attend(out, hn):
        hidden = hn.squeeze(0).unsqueeze(2)                              # [B,64,1]
        attn = torch.softmax(torch.bmm(out, hidden).squeeze(2), dim=1)   # [B,N]
        return torch.bmm(out.transpose(1, 2), attn.unsqueeze(2)).squeeze(2)

    def forward(self, obs, action):
        if isinstance(action, (list, tuple)):
            action = torch.cat(list(action), -1)
        x = torch.relu(self.dense1(torch.cat([obs, action], -1)))
        out, (hn, _) = self.lstm(x)
        n = self._attend(out, hn)
        if not self.model:
            return self.dense2(torch.relu(n))
        return self.dense2(n), self.dense3(n)


def _numpy(sd):
    return {k: (v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in sd.items()}


def grads(sd, obs, action, dq, dr=None, device='cpu'):
    """float64 gradients of sum(q * dq) (+ sum(r * dr)) with respect to obs, action and every weight:
    {'obs', 'action', <state_dict key>...} as numpy arrays, plus 'q' (and 'r')."""
    net = Critic64(sd, device)
    o = torch.as_tensor(np.asarray(obs, np.float64), device=device).requires_grad_(True)
    a = torch.as_tensor(np.asarray(action, np.float64), device=device).requires_grad_(True)
    res = net(o, a)
    q, r = res if net.model else (res, None)
    loss = (q * torch.as_tensor(np.asarray(dq, np.float64), device=device)).sum()
    if dr is not None:
        loss = loss + (r * torch.as_tensor(np.asarray(dr, np.float64), device=device)).sum()
    loss.backward()
    params = dict(net.named_parameters())
    out = {'obs': o.grad.cpu().numpy(), 'action': a.grad.cpu().numpy(), 'q': q.detach().cpu().numpy()}
    if r is not None:
        out['r'] = r.detach().cpu().numpy()
    for k in net.keys():  # a head the loss does not use (dr None) has no .grad: its gradient is zero
        g = params[k].grad
        out[k] = np.zeros(tuple(params[k].shape)) if g is None else g.cpu().numpy()
    return out


def kink_free(sd, obs, action, eps=1e-5):
    """Mask [B] of the samples whose float64 relu pre-activations (dense1, and the attention output of the relu
    critic) are all farther than eps from zero: there fp32 and float64 agree on which side of every kink they are."""
    net = Critic64(sd)
    with torch.no_grad():
        z1, n = net.pre_activations(torch.as_tensor(np.asarray(obs, np.float64)),
                                    torch.as_tensor(np.asarray(action, np.float64)))
    ok = (z1.abs() > eps).all(-1).all(-1)
    if not net.model:
        ok &= (n.abs() > eps).all(-1)
    return ok.numpy()
