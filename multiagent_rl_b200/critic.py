"""Critic forward on the device: the reference's ``CriticNetwork`` (LSTM over the agent axis + dot-product attention)
as one CUDA kernel, for TD targets / imagined rollouts that should not leave the GPU (SURVEY 8f-2).

Mirrors ``rls/model/ac_network_multi_gumbel.py:70-148`` and ``rls/model/ac_network_model_multi_gumbel.py:69-143``
(state_dict key names are kept so a reference checkpoint - ``Trainer.save_models``, ddpg_gumbel_fix.py:221-229 - loads
as is).  Acting never calls the critic; ``Trainer.optimize()`` (autograd, out of scope) is where the reference does.
"""
import ctypes as C

import torch

from . import _lib

_KEYS = [('dense1_w', 'dense1.module.weight'), ('dense1_b', 'dense1.module.bias'),
         ('w_ih', 'lstm.weight_ih_l0'), ('w_hh', 'lstm.weight_hh_l0'), ('b_ih', 'lstm.bias_ih_l0'),
         ('b_hh', 'lstm.bias_hh_l0'), ('dense2_w', 'dense2.weight'), ('dense2_b', 'dense2.bias')]


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

    def load_state_dict(self, sd):
        """``critic.load_state_dict``.  CUDA tensors on the critic's device are packed by one kernel on torch's current
        stream without a host synchronisation (critic forwards enqueued on that stream afterwards see the new weights;
        other streams are ordered by the caller); anything else is read on the host.  KeyError for a missing key,
        ValueError for a tensor of the wrong shape."""
        H, G = 64, 256
        names = list(_KEYS) + ([('dense3_w', 'dense3.weight'), ('dense3_b', 'dense3.bias')] if self.model else [])
        shapes = {'dense1_w': (H, self.obs_dim + self.act_dim), 'dense1_b': (H,), 'w_ih': (G, H), 'w_hh': (G, H),
                  'b_ih': (G,), 'b_hh': (G,), 'dense2_w': (self.out_dim, H), 'dense2_b': (self.out_dim,),
                  'dense3_w': (self.out_dim, H), 'dense3_b': (self.out_dim,)}
        w, keep, on_device = _lib.weights(_lib.CriticWeights, sd, names, shapes, self.device)
        fn = 'critic_load_device' if on_device else 'critic_load'
        _lib.check(getattr(self._lib, fn)(self._h, C.byref(w), _lib.current_stream(self.device)), fn)
        del keep

    def forward(self, obs, action):
        obs = torch.as_tensor(obs, dtype=torch.float32, device=self.device).contiguous()
        if isinstance(action, (list, tuple)):  # ac_network_multi_gumbel.py:131-132
            action = torch.cat([torch.as_tensor(a, dtype=torch.float32, device=self.device) for a in action], dim=-1)
        action = torch.as_tensor(action, dtype=torch.float32, device=self.device).contiguous()
        B, N, D = obs.shape
        if D != self.obs_dim or tuple(action.shape) != (B, N, self.act_dim):
            raise ValueError('expected obs [B,N,%d] and action [B,N,%d]' % (self.obs_dim, self.act_dim))
        q = torch.empty((B, self.out_dim), dtype=torch.float32, device=self.device)
        r = torch.empty((B, self.out_dim), dtype=torch.float32, device=self.device) if self.model else None
        _lib.check(self._lib.critic_forward(self._h, _lib.ptr(obs), _lib.ptr(action), B, N, _lib.ptr(q), _lib.ptr(r),
                                            _lib.current_stream(self.device)), 'critic_forward')
        return (q, r) if self.model else q
