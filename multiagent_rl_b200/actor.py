"""Acting surface: the reference's ``ActorNetwork`` forward + hard Gumbel-softmax sampling as one
CUDA kernel, behind the names the reference uses.

Mirrors
  * ``rls/model/ac_network_multi_gumbel.py:24-67`` (ActorNetwork; state_dict key names are kept so a
    reference checkpoint loads as is) and ``ac_network_model_multi_gumbel.py:23-66`` (dense3 head);
  * ``rls/agent/multiagent/ddpg_gumbel_fix.py:86-107`` ``Trainer.get_exploration_action`` and
    ``:109-116`` ``gumbel_softmax(hard=True)``.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib

_KEYS = [('dense1_w', 'dense1.module.weight'), ('dense1_b', 'dense1.module.bias'),
         ('w_ih', 'bilstm.weight_ih_l0'), ('w_hh', 'bilstm.weight_hh_l0'),
         ('b_ih', 'bilstm.bias_ih_l0'), ('b_hh', 'bilstm.bias_hh_l0'),
         ('w_ih_r', 'bilstm.weight_ih_l0_reverse'), ('w_hh_r', 'bilstm.weight_hh_l0_reverse'),
         ('b_ih_r', 'bilstm.bias_ih_l0_reverse'), ('b_hh_r', 'bilstm.bias_hh_l0_reverse')]


class FusedActor(object):
    """Device-resident copy of an ActorNetwork's weights + the fused forward/sample kernel.

    ``state_dict``: mapping with the reference's key names (torch tensors or numpy arrays).
    """

    IMPLS = {'auto': 0, 'simt': 1, 'tc': 2}

    def __init__(self, state_dict, device=None, seed=0, impl='auto'):
        if not torch.cuda.is_available():
            raise RuntimeError('multiagent_rl_b200 needs a CUDA device: the actor runs only as an sm_100a kernel')
        self._lib = _lib.load()
        self.device = torch.device(device if device is not None else 'cuda:%d' % torch.cuda.current_device())
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        sd = dict(state_dict)
        self.obs_dim = int(_lib.np32(sd['dense1.module.weight']).shape[1])
        self.multi = 'dense2_1.module.weight' in sd
        if self.multi:
            self.act_dims = [int(sd['dense2_1.module.weight'].shape[0]), int(sd['dense2_2.module.weight'].shape[0])]
        else:
            self.act_dims = [int(sd['dense2.module.weight'].shape[0])]
        self.has_model = 'dense3.module.weight' in sd
        self.A = sum(self.act_dims)
        self.seed = int(seed)
        cfg = _lib.ActorConfig(obs_dim=self.obs_dim, act0=self.act_dims[0],
                               act1=self.act_dims[1] if self.multi else 0,
                               has_model_head=1 if self.has_model else 0, device=self.device.index, reserved0=0)
        h = C.c_void_p()
        _lib.check(self._lib.actor_create(C.byref(cfg), C.byref(h)), 'actor_create')
        self._h = h
        self.set_impl(impl)
        self.load_state_dict(sd)

    def __del__(self):
        h = getattr(self, '_h', None)
        if h is not None and self._lib is not None:
            self._lib.actor_destroy(h)
            self._h = None

    def set_impl(self, impl):
        """'auto' (tensor cores where supported), 'simt' (fp32 FFMA) or 'tc' (tcgen05, fp16 hi/lo split)."""
        _lib.check(self._lib.actor_set_impl(self._h, self.IMPLS[impl]), 'actor_set_impl')
        self.impl = impl

    def load_state_dict(self, sd):
        """``actor.load_state_dict`` (rls/agent/multiagent/ddpg_gumbel_fix.py:231-241).

        CUDA tensors on the actor's device - a learner's ``state_dict()`` - are packed by one kernel on torch's current
        stream, without a host synchronisation: forwards and rollouts enqueued on that stream afterwards see the new
        weights, and in-place changes made to the tensors earlier on it are what gets loaded.  The weights are
        overwritten in place, so work on other streams that uses this actor must be ordered with events.  Anything
        else (numpy arrays, CPU tensors, another device) is read on the host; the call returns when it has been
        loaded.  KeyError for a missing key, ValueError for a tensor of the wrong shape."""
        H = 64
        names = list(_KEYS)
        shapes = {'dense1_w': (H, self.obs_dim), 'dense1_b': (H,)}
        for d in ('', '_r'):
            shapes.update({'w_ih' + d: (4 * 32, H), 'w_hh' + d: (4 * 32, 32), 'b_ih' + d: (4 * 32,), 'b_hh' + d: (4 * 32,)})
        if self.multi:
            names += [('dense2_w', 'dense2_1.module.weight'), ('dense2_b', 'dense2_1.module.bias'),
                      ('dense2b_w', 'dense2_2.module.weight'), ('dense2b_b', 'dense2_2.module.bias')]
            shapes.update({'dense2b_w': (self.act_dims[1], H), 'dense2b_b': (self.act_dims[1],)})
        else:
            names += [('dense2_w', 'dense2.module.weight'), ('dense2_b', 'dense2.module.bias')]
        shapes.update({'dense2_w': (self.act_dims[0], H), 'dense2_b': (self.act_dims[0],)})
        if self.has_model:
            names += [('dense3_w', 'dense3.module.weight'), ('dense3_b', 'dense3.module.bias')]
            shapes.update({'dense3_w': (self.obs_dim, H), 'dense3_b': (self.obs_dim,)})
        w, keep, on_device = _lib.weights(_lib.ActorWeights, sd, names, shapes, self.device)
        fn = 'actor_load_device' if on_device else 'actor_load'
        _lib.check(getattr(self._lib, fn)(self._h, C.byref(w), _lib.current_stream(self.device)), fn)
        del keep  # the host path has copied the arrays; device tensors are released in stream order by torch

    # ------------------------------------------------------------------ device tensors
    def forward(self, obs, gumbel=None, step=0, env_id_offset=0, want_logits=False, want_onehot=False,
                want_next_state=False, seed=None):
        """obs [B,N,D] fp32 cuda tensor -> dict(act_u[B,N] int32, act_c, logits, onehot, next_state).
        ``gumbel`` [B,N,A] injects the noise (parity tests); otherwise Philox(seed, env id, step, agent)."""
        obs = torch.as_tensor(obs, dtype=torch.float32, device=self.device).contiguous()
        B, N, D = obs.shape
        if D != self.obs_dim:
            raise ValueError('obs has D=%d, actor expects %d' % (D, self.obs_dim))
        if gumbel is not None:
            gumbel = torch.as_tensor(gumbel, dtype=torch.float32, device=self.device).contiguous()
            if gumbel.numel() != B * N * self.A:
                raise ValueError('gumbel must be [B,N,%d]' % self.A)
        dev = self.device
        out = {'act_u': torch.empty((B, N), dtype=torch.int32, device=dev)}
        out['act_c'] = torch.empty((B, N), dtype=torch.int32, device=dev) if self.multi else None
        out['logits'] = torch.empty((B, N, self.A), dtype=torch.float32, device=dev) if want_logits else None
        out['onehot'] = torch.empty((B, N, self.A), dtype=torch.float32, device=dev) if want_onehot else None
        out['next_state'] = torch.empty((B, N, D), dtype=torch.float32, device=dev) if want_next_state else None
        _lib.check(self._lib.actor_forward(
            self._h, _lib.ptr(obs), B, N, _lib.ptr(gumbel), C.c_uint64(self.seed if seed is None else int(seed)),
            C.c_uint64(int(step)), int(env_id_offset), _lib.ptr(out['logits']), _lib.ptr(out['next_state']),
            _lib.ptr(out['act_u']), _lib.ptr(out['act_c']), _lib.ptr(out['onehot']),
            _lib.current_stream(dev)), 'actor_forward')
        return out

    # ------------------------------------------------------------------ host buffers
    def act_host(self, obs_host, step=0, env_id_offset=0, act_u=None, act_c=None, onehot=None, seed=None):
        """obs_host: float32 numpy / pinned tensor [B,N,D]; outputs are written into the given host
        buffers (H2D + kernel + D2H + sync: ddpg_gumbel_fix.py:93-100)."""
        B, N, D = obs_host.shape
        _lib.check(self._lib.actor_forward_host(
            self._h, _lib.ptr(obs_host), B, N, C.c_uint64(self.seed if seed is None else int(seed)),
            C.c_uint64(int(step)), int(env_id_offset), _lib.ptr(act_u), _lib.ptr(act_c), _lib.ptr(onehot),
            _lib.current_stream(self.device)), 'actor_forward_host')


class FusedActingMixin(object):
    """Drop-in for ``Trainer.get_exploration_action``: mix into the reference's Trainer
    (``class Trainer(FusedActingMixin, rls.agent.multiagent.ddpg_gumbel_fix.Trainer)``), or use
    ``ActingTrainer`` below when only acting is needed.  Needs ``self.actor`` (a module with the
    reference's parameter names) and ``self.action_type``."""

    _fused = None
    _fused_version = None
    _act_step = 0

    def _weights_version(self):
        return tuple(int(p._version) for p in self.actor.parameters())

    def _sync_fused(self):
        v = self._weights_version()
        if self._fused is None:
            dev = next(self.actor.parameters()).device
            self._fused = FusedActor(self.actor.state_dict(), device=dev if dev.type == 'cuda' else None,
                                     seed=getattr(self, 'sample_seed', torch.initial_seed() & (2 ** 63 - 1)))
        elif v != self._fused_version:  # optimize() stepped the actor (ddpg_gumbel_fix.py:196-199)
            # a CUDA actor reloads on the device, in stream order after the update (no host round trip)
            self._fused.load_state_dict(self.actor.state_dict())
        self._fused_version = v
        return self._fused

    def get_exploration_action(self, state):
        """state: list of N arrays (one env, the reference call) or array [B,N,D].
        Returns float32 one-hot array (B,N,A) - (1,N,A) for the reference call - or, for
        'MultiDiscrete', a list of two such arrays (ddpg_gumbel_fix.py:96-105)."""
        fused = self._sync_fused()
        if isinstance(state, (list, tuple)):
            obs = np.array([np.stack(state)], dtype='float32')  # process_obs (ddpg_gumbel_fix.py:59-61)
        else:
            obs = np.ascontiguousarray(state, dtype='float32')
        B, N, _ = obs.shape
        onehot = np.empty((B, N, fused.A), dtype=np.float32)
        fused.act_host(obs, step=self._act_step, onehot=onehot)
        self._act_step += 1
        if self.action_type == 'Discrete':
            return onehot
        a0 = fused.act_dims[0]
        return [np.ascontiguousarray(onehot[..., :a0]), np.ascontiguousarray(onehot[..., a0:])]


class ActingTrainer(FusedActingMixin):
    """Acting-only stand-in with the reference Trainer's constructor signature
    (rls/agent/multiagent/ddpg_gumbel_fix.py:14): ``Trainer(actor, critic, memory, action_type)``.
    ``optimize()`` is out of scope for the kernels and not provided here."""

    def __init__(self, actor, critic=None, memory=None, action_type='Discrete', device=None, sample_seed=None):
        self.device = torch.device(device if device is not None else 'cuda:0')
        self.actor = actor.to(self.device)
        self.critic = critic
        self.memory = memory
        self.action_type = action_type
        self.nb_actions = 5
        if sample_seed is not None:
            self.sample_seed = int(sample_seed)

    def load_models(self, fname):
        """rls/agent/multiagent/ddpg_gumbel_fix.py:231-236 (actor only): the caller passes the full stem -
        experiments/run.py:117 already prepends ``arglist.appx`` - so the path is './Models/<fname>_actor.pt'."""
        self.actor.load_state_dict(torch.load('./Models/' + str(fname) + '_actor.pt', map_location=self.device))

    def save_models(self, fname):
        """rls/agent/multiagent/ddpg_gumbel_fix.py:221-229 (actor only; this stand-in has no target network)."""
        torch.save(self.actor.state_dict(), './Models/' + str(fname) + '_actor.pt')
