"""float64 torch restatement of the reference actors, differentiable by autograd - TEST INFRASTRUCTURE.

The same network as oracle/actor_ref.py (rls/model/ac_network_multi_gumbel.py:24-67 and
ac_network_model_multi_gumbel.py:23-66) spelled with the reference's building blocks - ``nn.Linear`` per agent,
``nn.LSTM(64, 32, bidirectional=True, batch_first=True)`` over the agent axis, relu, the head(s) - so that autograd
gives the gradients the actor's backward kernel is compared with.  Never imported by the product.
"""
import numpy as np
import torch
import torch.nn as nn

H = 64


class _TimeDistributed(nn.Module):
    def __init__(self, module):
        super().__init__()
        self.module = module

    def forward(self, x):
        return self.module(x.reshape(-1, x.shape[-1])).reshape(*x.shape[:-1], -1)


def _numpy(sd):
    return {k: (v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in sd.items()}


class Actor64(nn.Module):
    """``Actor64(sd)``: float64 copy of the weights in ``sd`` (the reference's state_dict keys).  ``forward(obs)`` ->
    (logits [B,N,A] with both heads concatenated, next_state [B,N,D] or None)."""

    def __init__(self, sd, device='cpu'):
        super().__init__()
        D = np.shape(sd['dense1.module.weight'])[1]
        self.multi = 'dense2_1.module.weight' in sd
        self.model = 'dense3.module.weight' in sd
        self.dense1 = _TimeDistributed(nn.Linear(D, H))
        self.bilstm = nn.LSTM(H, 32, batch_first=True, bidirectional=True)
        if self.multi:
            self.dense2_1 = _TimeDistributed(nn.Linear(H, np.shape(sd['dense2_1.module.weight'])[0]))
            self.dense2_2 = _TimeDistributed(nn.Linear(H, np.shape(sd['dense2_2.module.weight'])[0]))
        else:
            self.dense2 = _TimeDistributed(nn.Linear(H, np.shape(sd['dense2.module.weight'])[0]))
        if self.model:
            self.dense3 = _TimeDistributed(nn.Linear(H, D))
        self.double().to(device)
        self.load_state_dict({k: torch.as_tensor(np.asarray(v, np.float64)) for k, v in _numpy(sd).items()})

    def keys(self):
        return [k for k, _ in self.named_parameters()]

    def pre_activations(self, obs):
        """(dense1 pre-activation [B,N,64], BiLSTM output [B,N,64]) - where the relu kinks are."""
        z1 = self.dense1(obs)
        out, _ = self.bilstm(torch.relu(z1))
        return z1, out

    def forward(self, obs):
        out, _ = self.bilstm(torch.relu(self.dense1(obs)))
        hid = torch.relu(out)
        logits = torch.cat([self.dense2_1(hid), self.dense2_2(hid)], -1) if self.multi else self.dense2(hid)
        return logits, (self.dense3(hid) if self.model else None)


def grads(sd, obs, dlogits, dnext_state=None, device='cpu'):
    """float64 gradients of sum(logits * dlogits) (+ sum(next_state * dnext_state)) with respect to obs and every
    weight: {'obs', <state_dict key>...} as numpy arrays, plus 'logits' (and 'next_state')."""
    net = Actor64(sd, device)
    o = torch.as_tensor(np.asarray(obs, np.float64), device=device).requires_grad_(True)
    logits, ns = net(o)
    loss = (logits * torch.as_tensor(np.asarray(dlogits, np.float64), device=device)).sum()
    if dnext_state is not None:
        loss = loss + (ns * torch.as_tensor(np.asarray(dnext_state, np.float64), device=device)).sum()
    loss.backward()
    params = dict(net.named_parameters())
    out = {'obs': o.grad.cpu().numpy(), 'logits': logits.detach().cpu().numpy()}
    if ns is not None:
        out['next_state'] = ns.detach().cpu().numpy()
    for k in net.keys():  # a head the loss does not use (dnext_state None) has no .grad: its gradient is zero
        g = params[k].grad
        out[k] = np.zeros(tuple(params[k].shape)) if g is None else g.cpu().numpy()
    return out


def kink_free(sd, obs, eps=1e-5):
    """Mask [B] of the samples whose float64 relu inputs (dense1's pre-activation and the BiLSTM output) are all
    farther than eps from zero: there fp32 and float64 agree on which side of every kink they are."""
    net = Actor64(sd)
    with torch.no_grad():
        z1, out = net.pre_activations(torch.as_tensor(np.asarray(obs, np.float64)))
    return ((z1.abs() > eps).all(-1).all(-1) & (out.abs() > eps).all(-1).all(-1)).numpy()
