"""Acting surface: the reference's ``ActorNetwork`` forward + hard Gumbel-softmax sampling as one
CUDA kernel, behind the names the reference uses; and the actor's backward, so that ``Trainer.optimize()`` can train
the actor through the kernels (``FusedActorNetwork``).

Mirrors
  * ``rls/model/ac_network_multi_gumbel.py:24-67`` (ActorNetwork; state_dict key names are kept so a
    reference checkpoint loads as is) and ``ac_network_model_multi_gumbel.py:23-66`` (dense3 head);
  * ``rls/agent/multiagent/ddpg_gumbel_fix.py:86-107`` ``Trainer.get_exploration_action`` and
    ``:109-116`` ``gumbel_softmax(hard=True)``.
"""
import ctypes as C

import numpy as np
import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from . import _lib
from .networks import _PerAgent

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

    def _names(self):
        """(ActorWeights field, state_dict key) of every tensor this actor has."""
        names = list(_KEYS)
        if self.multi:
            names += [('dense2_w', 'dense2_1.module.weight'), ('dense2_b', 'dense2_1.module.bias'),
                      ('dense2b_w', 'dense2_2.module.weight'), ('dense2b_b', 'dense2_2.module.bias')]
        else:
            names += [('dense2_w', 'dense2.module.weight'), ('dense2_b', 'dense2.module.bias')]
        if self.has_model:
            names += [('dense3_w', 'dense3.module.weight'), ('dense3_b', 'dense3.module.bias')]
        return names

    def _shapes(self):
        H = 64
        shapes = {'dense1_w': (H, self.obs_dim), 'dense1_b': (H,)}
        for d in ('', '_r'):
            shapes.update({'w_ih' + d: (4 * 32, H), 'w_hh' + d: (4 * 32, 32), 'b_ih' + d: (4 * 32,), 'b_hh' + d: (4 * 32,)})
        shapes.update({'dense2_w': (self.act_dims[0], H), 'dense2_b': (self.act_dims[0],)})
        if self.multi:
            shapes.update({'dense2b_w': (self.act_dims[1], H), 'dense2b_b': (self.act_dims[1],)})
        if self.has_model:
            shapes.update({'dense3_w': (self.obs_dim, H), 'dense3_b': (self.obs_dim,)})
        return shapes

    def load_state_dict(self, sd):
        """``actor.load_state_dict`` (rls/agent/multiagent/ddpg_gumbel_fix.py:231-241).

        CUDA tensors on the actor's device - a learner's ``state_dict()`` - are packed by one kernel on torch's current
        stream, without a host synchronisation: forwards and rollouts enqueued on that stream afterwards see the new
        weights, and in-place changes made to the tensors earlier on it are what gets loaded.  The weights are
        overwritten in place, so work on other streams that uses this actor must be ordered with events.  Anything
        else (numpy arrays, CPU tensors, another device) is read on the host; the call returns when it has been
        loaded.  KeyError for a missing key, ValueError for a tensor of the wrong shape."""
        w, keep, on_device = _lib.weights(_lib.ActorWeights, sd, self._names(), self._shapes(), self.device)
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

    def backward(self, obs, dlogits, dnext_state=None, want_obs=False, want_weights=True):
        """Gradients of the fp32 FFMA forward (``impl='simt'``) of ``obs`` [B,N,D] with the loaded weights, for
        upstream gradients ``dlogits`` [B,N,A] (both heads concatenated) and, for the "+model" actor, ``dnext_state``
        [B,N,D] (None: zero).  Returns ``{'obs': [B,N,D] | None, 'weights': {state_dict key: gradient} (empty unless
        want_weights)}``; ``bias_ih*`` and ``bias_hh*`` of a direction get the same gradient.  Outputs and workspace
        come from torch's allocator; the kernels run on torch's current stream without a host synchronisation."""
        obs = torch.as_tensor(obs, dtype=torch.float32, device=self.device).contiguous()
        B, N, D = obs.shape
        if D != self.obs_dim:
            raise ValueError('obs has D=%d, actor expects %d' % (D, self.obs_dim))
        dlogits = torch.as_tensor(dlogits, dtype=torch.float32, device=self.device).contiguous()
        if tuple(dlogits.shape) != (B, N, self.A):
            raise ValueError('expected dlogits [%d,%d,%d]' % (B, N, self.A))
        if dnext_state is not None:
            if not self.has_model:
                raise ValueError('dnext_state is the gradient of the dense3 head, which this actor does not have')
            dnext_state = torch.as_tensor(dnext_state, dtype=torch.float32, device=self.device).contiguous()
            if tuple(dnext_state.shape) != (B, N, D):
                raise ValueError('expected dnext_state [%d,%d,%d]' % (B, N, D))
        dobs = torch.empty_like(obs) if want_obs else None
        grads, g = {}, _lib.ActorGrads()
        if want_weights:
            shapes = self._shapes()
            for field, key in self._names():
                grads[key] = torch.empty(shapes[field], dtype=torch.float32, device=self.device)
                setattr(g, field, grads[key].data_ptr())
        nbytes = self._lib.actor_backward_workspace(self._h, B, N)
        if nbytes < 0:
            _lib.check(nbytes, 'actor_backward_workspace')
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=self.device)
        _lib.check(self._lib.actor_backward(self._h, _lib.ptr(obs), B, N, _lib.ptr(dlogits), _lib.ptr(dnext_state),
                                            _lib.ptr(dobs), C.byref(g), _lib.ptr(ws), nbytes,
                                            _lib.current_stream(self.device)), 'actor_backward')
        return {'obs': dobs, 'weights': grads}

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


class _ActorFunction(torch.autograd.Function):
    """logits (, next_state) = actor(obs) with the weights ``params``: the FFMA forward kernel after a repack of
    ``params``; the backward repacks the saved ``params`` and runs actor_backward for the gradients autograd asks for."""

    @staticmethod
    def forward(ctx, actor, keys, obs, *params):
        actor.load_state_dict(dict(zip(keys, params)))
        out = actor.forward(obs, want_logits=True, want_next_state=actor.has_model)
        ctx.actor, ctx.keys = actor, keys
        ctx.save_for_backward(obs, *params)
        ctx.set_materialize_grads(False)
        return (out['logits'], out['next_state']) if actor.has_model else out['logits']

    @staticmethod
    @once_differentiable
    def backward(ctx, dlogits, dnext_state=None):
        obs, params = ctx.saved_tensors[0], ctx.saved_tensors[1:]
        need = ctx.needs_input_grad
        want_w = any(need[3:])
        if not (need[2] or want_w) or (dlogits is None and dnext_state is None):
            return (None,) * len(need)
        actor = ctx.actor
        unused = set()  # an output the loss does not use gets no gradient, as under autograd
        if dlogits is None:
            dlogits = torch.zeros(tuple(obs.shape[:2]) + (actor.A,), dtype=torch.float32, device=obs.device)
            unused = {k for k in ctx.keys if k.startswith('dense2')}
        elif actor.has_model and dnext_state is None:
            unused = {'dense3.module.weight', 'dense3.module.bias'}
        actor.load_state_dict(dict(zip(ctx.keys, params)))
        g = actor.backward(obs, dlogits, dnext_state, want_obs=need[2], want_weights=want_w)
        wg = [g['weights'][k] if n and k not in unused else None for k, n in zip(ctx.keys, need[3:])]
        return (None, None, g['obs']) + tuple(wg)


class FusedActorNetwork(nn.Module):
    """Drop-in for the reference ``ActorNetwork(input_dim, out_dim)`` (rls/model/ac_network_multi_gumbel.py:24-67;
    ``out_dim`` an int or a list of two head widths), or with ``model_head=True`` for the actor of
    ac_network_model_multi_gumbel.py (dense3 head), that runs forward and backward as CUDA kernels.

    Parameters are plain ``nn.Parameter`` s under the reference's names and created in its order (``dense1.module``,
    ``bilstm`` - an ``nn.LSTM(64, 32, bidirectional=True)`` that only holds the parameters and is never called -
    ``dense2`` or ``dense2_1`` / ``dense2_2``, ``dense3``), so a seed gives the reference's initial weights, and
    state_dict / load_state_dict / optimizers work as for the reference.  ``forward(obs [B,N,D])`` returns what the
    reference returns: logits [B,N,A] (a list of two for two heads; ``(policy, next_state)`` with the model head).
    Every forward repacks the parameters into the kernel's weight image on the current stream (a soft update written
    through ``.data`` is seen by the next call) and runs the fp32 FFMA forward, which the backward differentiates; the
    backward repacks the parameters it saved.  Parameters must be float32 on a CUDA device; there is no CPU path."""

    def __init__(self, input_dim, out_dim, model_head=False):
        super().__init__()
        input_dim = int(input_dim)
        heads = [int(a) for a in out_dim] if isinstance(out_dim, (list, tuple)) else [int(out_dim)]
        if not 1 <= input_dim <= 64:
            raise ValueError('FusedActorNetwork: input_dim must be 1..64 (the kernel stages one observation row per '
                             'lane pair), got %d' % input_dim)
        if len(heads) not in (1, 2) or min(heads) < 1 or sum(heads) > 16:
            raise ValueError('FusedActorNetwork: one or two heads of at least one entry and at most 16 in total, '
                             'got %s' % (out_dim,))
        self.input_dim, self.out_dim, self.model_head = input_dim, out_dim, bool(model_head)
        self.dense1 = _PerAgent(nn.Linear(input_dim, 64))
        self.bilstm = nn.LSTM(64, 32, num_layers=1, batch_first=True, bidirectional=True)
        if len(heads) == 2:
            self.dense2_1 = _PerAgent(nn.Linear(64, heads[0]))
            self.dense2_2 = _PerAgent(nn.Linear(64, heads[1]))
        else:
            self.dense2 = _PerAgent(nn.Linear(64, heads[0]))
        if self.model_head:
            self.dense3 = _PerAgent(nn.Linear(64, input_dim))
        self._heads = heads
        self._handle = _lib.ModuleHandle('actor')

    def forward(self, obs):
        sd = dict(self.named_parameters())
        keys = list(sd)
        params = [sd[k] for k in keys]
        dev = params[0].device
        if dev.type != 'cuda' or any(p.device != dev or p.dtype != torch.float32 for p in params):
            raise RuntimeError('FusedActorNetwork runs only as a CUDA kernel: its parameters must be float32 tensors '
                               'on one CUDA device (call .cuda()); got %s %s' % (params[0].dtype, dev))
        obs = torch.as_tensor(obs, device=dev).float()
        if obs.dim() != 3 or obs.shape[2] != self.input_dim:
            raise ValueError('expected obs [B,N,%d], got %s' % (self.input_dim, tuple(obs.shape)))
        if not 1 <= obs.shape[1] <= 12:
            raise ValueError('FusedActorNetwork: 1..12 agents (the kernel unrolls the agent axis), got %d'
                             % obs.shape[1])
        h = self._handle
        if h.actor is None or h.actor.device != dev:
            h.actor = FusedActor({k: p.detach() for k, p in zip(keys, params)}, device=dev, impl='simt')
        out = _ActorFunction.apply(h.actor, keys, obs.contiguous(), *params)
        logits, next_state = out if self.model_head else (out, None)
        policy = [logits[..., :self._heads[0]], logits[..., self._heads[0]:]] if len(self._heads) == 2 else logits
        return (policy, next_state) if self.model_head else policy
