"""The reference's ``CriticNetwork`` (LSTM over the agent axis + dot-product attention) as CUDA kernels: the forward
for TD targets / imagined rollouts that should not leave the GPU (SURVEY 8f-2), and its backward, so that
``Trainer.optimize()`` can train the critic through the kernels.

Mirrors ``rls/model/ac_network_multi_gumbel.py:70-148`` and ``rls/model/ac_network_model_multi_gumbel.py:69-143``
(state_dict key names are kept so a reference checkpoint - ``Trainer.save_models``, ddpg_gumbel_fix.py:221-229 - loads
as is).  ``FusedCritic`` is the handle-level interface; ``FusedCriticNetwork`` is an ``nn.Module`` with the reference
class's constructor, parameters and forward, differentiable through ``critic_backward``.
"""
import ctypes as C

import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from . import _lib
from .networks import _PerAgent

_KEYS = [('dense1_w', 'dense1.module.weight'), ('dense1_b', 'dense1.module.bias'),
         ('w_ih', 'lstm.weight_ih_l0'), ('w_hh', 'lstm.weight_hh_l0'), ('b_ih', 'lstm.bias_ih_l0'),
         ('b_hh', 'lstm.bias_hh_l0'), ('dense2_w', 'dense2.weight'), ('dense2_b', 'dense2.bias')]
_KEYS3 = [('dense3_w', 'dense3.weight'), ('dense3_b', 'dense3.bias')]
_H, _G = 64, 256


class FusedCritic(object):
    """``FusedCritic(critic.state_dict(), obs_dim)``; ``forward(obs[B,N,D], action[B,N,A] | [a0, a1]) -> q[B,1]``
    (``(q, r)`` for the "+model" critic, whose state_dict carries ``dense3``)."""

    def __init__(self, state_dict, obs_dim, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError('multiagent_rl_b200 needs a CUDA device: the critic runs only as an sm_100a kernel')
        self._lib = _lib.load()
        self.device = torch.device(device if device is not None else 'cuda:%d' % torch.cuda.current_device())
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        sd = dict(state_dict)
        din = int(_lib.np32(sd['dense1.module.weight']).shape[1])
        self.obs_dim, self.act_dim = int(obs_dim), din - int(obs_dim)
        self.out_dim = int(_lib.np32(sd['dense2.weight']).shape[0])
        self.model = 'dense3.weight' in sd
        cfg = _lib.CriticConfig(obs_dim=self.obs_dim, act_dim=self.act_dim, out_dim=self.out_dim,
                                has_reward_head=1 if self.model else 0, relu_attention=0 if self.model else 1,
                                device=self.device.index)
        h = C.c_void_p()
        _lib.check(self._lib.critic_create(C.byref(cfg), C.byref(h)), 'critic_create')
        self._h = h
        self.load_state_dict(sd)

    def __del__(self):
        h = getattr(self, '_h', None)
        if h is not None and self._lib is not None:
            self._lib.critic_destroy(h)
            self._h = None

    def _shapes(self):
        H, G, O = _H, _G, self.out_dim
        return {'dense1_w': (H, self.obs_dim + self.act_dim), 'dense1_b': (H,), 'w_ih': (G, H), 'w_hh': (G, H),
                'b_ih': (G,), 'b_hh': (G,), 'dense2_w': (O, H), 'dense2_b': (O,), 'dense3_w': (O, H), 'dense3_b': (O,)}

    def _names(self):
        return list(_KEYS) + (_KEYS3 if self.model else [])

    def load_state_dict(self, sd):
        """``critic.load_state_dict``.  CUDA tensors on the critic's device are packed by one kernel on torch's current
        stream without a host synchronisation (critic forwards enqueued on that stream afterwards see the new weights;
        other streams are ordered by the caller); anything else is read on the host.  KeyError for a missing key,
        ValueError for a tensor of the wrong shape."""
        w, keep, on_device = _lib.weights(_lib.CriticWeights, sd, self._names(), self._shapes(), self.device)
        fn = 'critic_load_device' if on_device else 'critic_load'
        _lib.check(getattr(self._lib, fn)(self._h, C.byref(w), _lib.current_stream(self.device)), fn)
        del keep

    def _inputs(self, obs, action):
        obs = torch.as_tensor(obs, dtype=torch.float32, device=self.device).contiguous()
        if isinstance(action, (list, tuple)):  # ac_network_multi_gumbel.py:131-132
            action = torch.cat([torch.as_tensor(a, dtype=torch.float32, device=self.device) for a in action], dim=-1)
        action = torch.as_tensor(action, dtype=torch.float32, device=self.device).contiguous()
        B, N, D = obs.shape
        if D != self.obs_dim or tuple(action.shape) != (B, N, self.act_dim):
            raise ValueError('expected obs [B,N,%d] and action [B,N,%d]' % (self.obs_dim, self.act_dim))
        return obs, action

    def forward(self, obs, action):
        obs, action = self._inputs(obs, action)
        B, N, _ = obs.shape
        q = torch.empty((B, self.out_dim), dtype=torch.float32, device=self.device)
        r = torch.empty((B, self.out_dim), dtype=torch.float32, device=self.device) if self.model else None
        _lib.check(self._lib.critic_forward(self._h, _lib.ptr(obs), _lib.ptr(action), B, N, _lib.ptr(q), _lib.ptr(r),
                                            _lib.current_stream(self.device)), 'critic_forward')
        return (q, r) if self.model else q

    def backward(self, obs, action, dq, dr=None, want_obs=False, want_action=True, want_weights=True):
        """Gradients of ``forward(obs, action)`` with the loaded weights, for upstream gradients ``dq`` [B,out] and, for
        the "+model" critic, ``dr`` [B,out] (None: zero).  Returns ``{'obs': [B,N,D] | None, 'action': [B,N,A] |
        None, 'weights': {state_dict key: gradient} (empty unless want_weights)}``; ``lstm.bias_ih_l0`` and
        ``lstm.bias_hh_l0`` get the same gradient.  Outputs and workspace come from torch's allocator; the kernels
        run on torch's current stream without a host synchronisation."""
        obs, action = self._inputs(obs, action)
        B, N, _ = obs.shape
        dq = torch.as_tensor(dq, dtype=torch.float32, device=self.device).contiguous()
        if tuple(dq.shape) != (B, self.out_dim):
            raise ValueError('expected dq [%d,%d]' % (B, self.out_dim))
        if dr is not None:
            if not self.model:
                raise ValueError('dr is the gradient of the reward head, which this critic does not have')
            dr = torch.as_tensor(dr, dtype=torch.float32, device=self.device).contiguous()
            if tuple(dr.shape) != (B, self.out_dim):
                raise ValueError('expected dr [%d,%d]' % (B, self.out_dim))
        dobs = torch.empty_like(obs) if want_obs else None
        dact = torch.empty_like(action) if want_action else None
        grads, g = {}, _lib.CriticGrads()
        if want_weights:
            shapes = self._shapes()
            for field, key in self._names():
                grads[key] = torch.empty(shapes[field], dtype=torch.float32, device=self.device)
                setattr(g, field, grads[key].data_ptr())
        nbytes = self._lib.critic_backward_workspace(self._h, B, N)
        if nbytes < 0:
            _lib.check(nbytes, 'critic_backward_workspace')
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=self.device)
        _lib.check(self._lib.critic_backward(self._h, _lib.ptr(obs), _lib.ptr(action), B, N, _lib.ptr(dq), _lib.ptr(dr),
                                             _lib.ptr(dobs), _lib.ptr(dact), C.byref(g), _lib.ptr(ws), nbytes,
                                             _lib.current_stream(self.device)), 'critic_backward')
        return {'obs': dobs, 'action': dact, 'weights': grads}


class _CriticFunction(torch.autograd.Function):
    """q (, r) = critic(obs, action) with the weights ``params``: the forward kernel after a repack of ``params``; the
    backward repacks the saved ``params`` and runs critic_backward for the gradients autograd asks for."""

    @staticmethod
    def forward(ctx, critic, keys, obs, action, *params):
        critic.load_state_dict(dict(zip(keys, params)))
        out = critic.forward(obs, action)
        ctx.critic, ctx.keys = critic, keys
        ctx.save_for_backward(obs, action, *params)
        ctx.set_materialize_grads(False)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, dq, dr=None):
        obs, action = ctx.saved_tensors[:2]
        params = ctx.saved_tensors[2:]
        need = ctx.needs_input_grad
        want_w = any(need[4:])
        none = (None,) * len(need)
        if not (need[2] or need[3] or want_w) or (dq is None and dr is None):
            return none
        critic = ctx.critic
        unused = set()  # a head whose output the loss does not use gets no gradient, as under autograd
        if dq is None:
            dq = torch.zeros((obs.shape[0], critic.out_dim), dtype=torch.float32, device=obs.device)
            unused = {'dense2.weight', 'dense2.bias'}
        elif critic.model and dr is None:
            unused = {'dense3.weight', 'dense3.bias'}
        critic.load_state_dict(dict(zip(ctx.keys, params)))
        g = critic.backward(obs, action, dq, dr, want_obs=need[2], want_action=need[3], want_weights=want_w)
        wg = [g['weights'][k] if n and k not in unused else None for k, n in zip(ctx.keys, need[4:])]
        return (None, None, g['obs'], g['action']) + tuple(wg)


class FusedCriticNetwork(nn.Module):
    """Drop-in for the reference ``CriticNetwork(input_dim=D + A, out_dim=1)`` (main.py:61), or with ``model=True``
    for the "+model" critic of ac_network_model_multi_gumbel.py (no relu after the attention, reward head dense3),
    that runs forward and backward as CUDA kernels.

    Parameters are plain ``nn.Parameter`` s under the reference's names and created in its order (``dense1.module``,
    ``lstm`` - an ``nn.LSTM(64, 64)`` that only holds ``*_l0`` and is never called - ``dense2``, ``dense3``), so a
    seed gives the reference's initial weights, and state_dict / load_state_dict / optimizers / clip_grad_norm_ work
    as for the reference.  ``forward(obs [B,N,D], action [B,N,A] | [a0, a1])`` returns ``q [B,out]`` (``(q, r)`` for
    the model critic).  Every forward repacks the parameters into the kernel's weight image on the current stream
    (a soft update written through ``.data`` is seen by the next call); the backward repacks the parameters it saved.
    Parameters must be float32 on a CUDA device; there is no CPU path."""

    def __init__(self, input_dim, out_dim, model=False):
        super().__init__()
        input_dim, out_dim = int(input_dim), int(out_dim)
        if not 2 <= input_dim <= 64:
            raise ValueError('FusedCriticNetwork: input_dim = obs_dim + action width must be 2..64 (the kernel holds '
                             'one input row per lane pair), got %d' % input_dim)
        if not 1 <= out_dim <= 4:
            raise ValueError('FusedCriticNetwork: out_dim must be 1..4, got %d' % out_dim)
        self.input_dim, self.out_dim, self.model = input_dim, out_dim, bool(model)
        self.dense1 = _PerAgent(nn.Linear(input_dim, _H))
        self.lstm = nn.LSTM(_H, _H, batch_first=True)
        self.dense2 = nn.Linear(_H, out_dim)
        if self.model:
            self.dense3 = nn.Linear(_H, out_dim)
        self._handle = _lib.ModuleHandle('critic')

    def _keys(self):
        return [k for _, k in _KEYS] + ([k for _, k in _KEYS3] if self.model else [])

    def forward(self, obs, action):
        sd = dict(self.named_parameters())
        keys = self._keys()
        params = [sd[k] for k in keys]
        dev = params[0].device
        if dev.type != 'cuda' or any(p.device != dev or p.dtype != torch.float32 for p in params):
            raise RuntimeError('FusedCriticNetwork runs only as a CUDA kernel: its parameters must be float32 tensors '
                               'on one CUDA device (call .cuda()); got %s %s' % (params[0].dtype, dev))
        if isinstance(action, (list, tuple)):  # ac_network_multi_gumbel.py:131-132; autograd splits the gradient
            action = torch.cat([torch.as_tensor(a, device=dev).float() for a in action], dim=-1)
        obs = torch.as_tensor(obs, device=dev).float()
        action = torch.as_tensor(action, device=dev).float()
        if obs.dim() != 3 or action.dim() != 3 or action.shape[:2] != obs.shape[:2]:
            raise ValueError('expected obs [B,N,D] and action [B,N,A], got %s and %s'
                             % (tuple(obs.shape), tuple(action.shape)))
        B, N, D = obs.shape
        if D + action.shape[2] != self.input_dim:
            raise ValueError('obs_dim + action width = %d, the critic was built for %d'
                             % (D + action.shape[2], self.input_dim))
        if not 1 <= N <= 16:
            raise ValueError('FusedCriticNetwork: 1..16 agents (the kernel keeps a step per register), got %d' % N)
        h = self._handle
        if h.critic is None or h.critic.obs_dim != D or h.critic.device != dev:
            h.critic = FusedCritic({k: p.detach() for k, p in zip(keys, params)}, obs_dim=D, device=dev)
        return _CriticFunction.apply(h.critic, keys, obs.contiguous(), action.contiguous(), *params)
