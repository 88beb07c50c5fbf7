"""ctypes binding of libmpe_b200.so (the C ABI in include/mpe_b200.h).

There is NO fallback: if the library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('MPE_B200_LIB', os.path.join(HERE, 'libmpe_b200.so'))  # override: A/B builds
ABI_VERSION = 9

MPE_OK, MPE_EINVAL, MPE_ECUDA, MPE_EUNSUPPORTED = 0, -1, -2, -3
SCENARIO_IDS = {'simple_spread': 0, 'simple_reference': 1, 'simple_speaker_listener': 2, 'fullobs_collect_treasure': 3}
F32, F64 = 0, 1
STATS_LEN = 5  # MPE_STATS_LEN


class MpeConfig(C.Structure):
    _fields_ = [('scenario', C.c_int32), ('num_agents', C.c_int32), ('precision', C.c_int32),
                ('device', C.c_int32), ('num_envs', C.c_int64), ('env_id_offset', C.c_int64),
                ('seed', C.c_uint64), ('max_episode_len', C.c_int32), ('reserved0', C.c_int32),
                ('max_speed', C.c_double), ('accel', C.c_double)]


class MpeDims(C.Structure):
    _fields_ = [('num_agents', C.c_int32), ('num_landmarks', C.c_int32), ('obs_dim', C.c_int32),
                ('dim_c', C.c_int32), ('act_u', C.c_int32), ('act_c', C.c_int32),
                ('precision', C.c_int32), ('device', C.c_int32), ('num_envs', C.c_int64),
                ('env_id_offset', C.c_int64)]


class MpeHostBlockLayout(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ('off_act_u', 'off_act_c', 'off_obs', 'off_rew', 'off_done', 'bytes')]


class ReplayConfig(C.Structure):
    _fields_ = [('capacity', C.c_int64), ('num_agents', C.c_int32), ('obs_dim', C.c_int32), ('act0', C.c_int32),
                ('act1', C.c_int32), ('device', C.c_int32), ('reserved0', C.c_int32)]


class ActorConfig(C.Structure):
    _fields_ = [('obs_dim', C.c_int32), ('act0', C.c_int32), ('act1', C.c_int32),
                ('has_model_head', C.c_int32), ('device', C.c_int32), ('reserved0', C.c_int32)]


class CriticConfig(C.Structure):
    _fields_ = [('obs_dim', C.c_int32), ('act_dim', C.c_int32), ('out_dim', C.c_int32), ('has_reward_head', C.c_int32),
                ('relu_attention', C.c_int32), ('device', C.c_int32)]


class CriticWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('dense1_w', 'dense1_b', 'w_ih', 'w_hh', 'b_ih', 'b_hh', 'dense2_w', 'dense2_b',
                                          'dense3_w', 'dense3_b')]


class CriticGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('dense1_w', 'dense1_b', 'w_ih', 'w_hh', 'b_ih', 'b_hh', 'dense2_w', 'dense2_b',
                                          'dense3_w', 'dense3_b')]


_WEIGHT_FIELDS = ['dense1_w', 'dense1_b', 'w_ih', 'w_hh', 'b_ih', 'b_hh', 'w_ih_r', 'w_hh_r', 'b_ih_r',
                  'b_hh_r', 'dense2_w', 'dense2_b', 'dense2b_w', 'dense2b_b', 'dense3_w', 'dense3_b']


class ActorWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in _WEIGHT_FIELDS]


class ActorGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in _WEIGHT_FIELDS]


P = C.c_void_p
# name -> (restype, argtypes); must list EVERY symbol include/mpe_b200.h declares
SIGNATURES = {
    'mpe_abi_version': (C.c_int, []),
    'mpe_last_error': (C.c_char_p, []),
    'mpe_create': (C.c_int, [C.POINTER(MpeConfig), C.POINTER(P)]),
    'mpe_destroy': (C.c_int, [P]),
    'mpe_query': (C.c_int, [P, C.POINTER(MpeDims)]),
    'mpe_seed': (C.c_int, [P, C.c_uint64, P]),
    'mpe_reset': (C.c_int, [P, P, P, P]),
    'mpe_set_state': (C.c_int, [P, P, P, P, P, P]),
    'mpe_get_state': (C.c_int, [P, P, P, P, P, P]),
    'mpe_observe': (C.c_int, [P, P, P]),
    'mpe_step': (C.c_int, [P, P, P, P, P, P, P, P, P, P]),
    'mpe_step_host': (C.c_int, [P, P, P, P, P, P, P]),
    'mpe_reset_host_async': (C.c_int, [P, P, P]),
    'mpe_host_wait': (C.c_int, [P]),
    'mpe_host_block_layout': (C.c_int, [P, C.POINTER(MpeHostBlockLayout)]),
    'mpe_act_step_host_async': (C.c_int, [P, P, P, C.c_uint64, P, P]),
    'mpe_host_alloc': (C.c_int, [C.POINTER(P), C.c_uint64]),
    'mpe_host_free': (C.c_int, [P]),
    'mpe_track_returns': (C.c_int, [P, C.c_int32]),
    'mpe_stats_read': (C.c_int, [P, C.POINTER(C.c_double), C.c_int32, P]),
    'mpe_stats_ptr': (C.c_int, [P, C.POINTER(P)]),
    'actor_create': (C.c_int, [C.POINTER(ActorConfig), C.POINTER(P)]),
    'actor_destroy': (C.c_int, [P]),
    'actor_load': (C.c_int, [P, C.POINTER(ActorWeights), P]),
    'actor_load_device': (C.c_int, [P, C.POINTER(ActorWeights), P]),
    'actor_set_impl': (C.c_int, [P, C.c_int32]),
    'actor_forward': (C.c_int, [P, P, C.c_int64, C.c_int32, P, C.c_uint64, C.c_uint64, C.c_int64, P, P, P, P, P, P]),
    'actor_forward_host': (C.c_int, [P, P, C.c_int64, C.c_int32, C.c_uint64, C.c_uint64, C.c_int64, P, P, P, P]),
    'actor_backward_workspace': (C.c_int64, [P, C.c_int64, C.c_int32]),
    'actor_backward': (C.c_int, [P, P, C.c_int64, C.c_int32, P, P, P, C.POINTER(ActorGrads), P, C.c_int64, P]),
    'mpe_rollout': (C.c_int, [P, P, C.c_int32, C.c_uint64, P, P, P, P, P, P, P]),
    'critic_create': (C.c_int, [C.POINTER(CriticConfig), C.POINTER(P)]),
    'critic_destroy': (C.c_int, [P]),
    'critic_load': (C.c_int, [P, C.POINTER(CriticWeights), P]),
    'critic_load_device': (C.c_int, [P, C.POINTER(CriticWeights), P]),
    'critic_forward': (C.c_int, [P, P, P, C.c_int64, C.c_int32, P, P, P]),
    'critic_backward_workspace': (C.c_int64, [P, C.c_int64, C.c_int32]),
    'critic_backward': (C.c_int, [P, P, P, C.c_int64, C.c_int32, P, P, P, P, C.POINTER(CriticGrads), P, C.c_int64, P]),
    'replay_create': (C.c_int, [C.POINTER(ReplayConfig), C.POINTER(P)]),
    'replay_destroy': (C.c_int, [P]),
    'replay_clear': (C.c_int, [P]),
    'replay_len': (C.c_int64, [P]),
    'replay_next_idx': (C.c_int64, [P]),
    'replay_add': (C.c_int, [P, P, P, P, P, P, P, C.c_int64, P]),
    'replay_sample': (C.c_int, [P, C.c_int64, P, C.c_uint64, P, P, P, P, P, P, P]),
    'mpe_rollout_replay': (C.c_int, [P, P, P, C.c_int32, C.c_uint64, P, P, P, P, P, P, P]),
}
# ABI version 9 added the info_i / info_f outputs just before the stream; a call from Python may still pass the
# version-8 argument list without them, which records no benchmark_data
_INFO_BEFORE_STREAM = ('mpe_rollout', 'mpe_rollout_replay')


def _info_optional(fn, nargs):
    def call(*args):
        if len(args) == nargs - 2:
            args = args[:-1] + (None, None) + args[-1:]
        return fn(*args)
    call.__name__ = fn.__name__
    return call

_lib = None


def load():
    """Load the shared library (once).  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            'libmpe_b200.so is not built (%s). Run `python -m multiagent_rl_b200.build`; there is no '
            'CPU or PyTorch fallback for the particle-env / actor kernels.' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
        if name in _INFO_BEFORE_STREAM:
            setattr(lib, name, _info_optional(fn, len(args)))
    v = lib.mpe_abi_version()
    if v != ABI_VERSION:
        raise RuntimeError('libmpe_b200.so ABI version %d, python binding expects %d: rebuild' % (v, ABI_VERSION))
    _lib = lib
    return lib


def check(rc, what):
    if rc != MPE_OK:
        msg = load().mpe_last_error()
        raise RuntimeError('%s failed (%d): %s' % (what, rc, msg.decode() if msg else '?'))


def ptr(t):
    """Device/host pointer of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return None
    if hasattr(t, 'data_ptr'):
        return C.c_void_p(t.data_ptr())
    return C.c_void_p(t.ctypes.data)


def np32(v):
    """A C-contiguous float32 numpy copy (or view) of a torch tensor, numpy array or nested list."""
    import numpy as np
    import torch
    if isinstance(v, torch.Tensor):
        v = v.detach().to('cpu', torch.float32).numpy()
    return np.ascontiguousarray(np.asarray(v, dtype=np.float32))


def weights(cls, sd, names, shapes, device):
    """Fill a weight struct (``ActorWeights`` / ``CriticWeights``) from the state_dict ``sd``.

    ``names``: (struct field, state_dict key) pairs; ``shapes``: field -> the shape the handle's layout expects.
    When every entry is a CUDA tensor on ``device`` the struct holds device pointers for ``*_load_device``
    (``.to(float32).contiguous()``, a no-op for a learner's parameters); otherwise host pointers to float32 copies for
    ``*_load``.  Returns ``(struct, keep, on_device)``, where ``keep`` owns the memory the pointers refer to.
    KeyError for a missing key and ValueError for a wrong shape, both before anything is launched."""
    import torch
    for _, key in names:
        if key not in sd:
            raise KeyError('state_dict is missing %r' % key)
    vals = [sd[key] for _, key in names]
    on_device = all(isinstance(v, torch.Tensor) and v.device == device for v in vals)
    keep = [v.detach().to(torch.float32).contiguous() if on_device else np32(v) for v in vals]
    w = cls()
    for (field, key), a in zip(names, keep):
        if tuple(a.shape) != tuple(shapes[field]):
            raise ValueError('%r has shape %s, expected %s' % (key, tuple(a.shape), tuple(shapes[field])))
        setattr(w, field, a.data_ptr() if on_device else a.ctypes.data)
    return w, keep, on_device


def current_stream(device):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class ModuleHandle(object):
    """The device handle of one fused network module (``FusedCriticNetwork``, ``FusedActorNetwork``), kept in the
    attribute named ``slot`` (None until the module's first forward creates it).  A deep copy (how learners build
    target networks) or a pickle starts without one, so copies never share or double-free a handle."""

    def __init__(self, slot):
        self._slot = slot
        setattr(self, slot, None)

    def __deepcopy__(self, memo):
        return ModuleHandle(self._slot)

    def __getstate__(self):
        return {'_slot': self._slot, self._slot: None}


class HostBlock(object):
    """Page-locked host memory from cudaHostAlloc (``mpe_host_alloc``), carved into torch tensors.

    Use this - not ``tensor.pin_memory()`` - for the buffers handed to the ``*_host`` entry points: on the B200 pool
    the copy engine uploads from torch's pinned blocks at 14 - 18 GB/s and from cudaHostAlloc memory at 54 GB/s
    (tools/h2d_probe.py).  The tensors are views: they are valid until ``free()`` / garbage collection of the block."""

    def __init__(self, nbytes):
        self.nbytes = int(nbytes)
        p = C.c_void_p()
        check(load().mpe_host_alloc(C.byref(p), self.nbytes), 'mpe_host_alloc')
        self.ptr = p.value
        self._used = 0
        self._views = []

    def tensor(self, shape, dtype, offset=None):
        """A slice of the block as a tensor of the given shape / torch dtype: at byte ``offset``, or (default) the
        next unused 256 B-aligned position."""
        import torch
        n = 1
        for d in shape:
            n *= int(d)
        size = n * torch.empty((), dtype=dtype).element_size()
        off = (self._used + 255) // 256 * 256 if offset is None else int(offset)
        if off + size > self.nbytes:
            raise ValueError('HostBlock of %d bytes is full' % self.nbytes)
        if offset is None:
            self._used = off + size
        if size == 0:
            return torch.empty(shape, dtype=dtype)
        buf = (C.c_uint8 * size).from_address(self.ptr + off)
        t = torch.frombuffer(buf, dtype=torch.uint8).view(dtype).view(*shape)
        self._views.append(buf)
        return t

    @staticmethod
    def size_for(specs):
        """Bytes needed for a list of (shape, torch dtype), each 256 B aligned."""
        import torch
        total = 0
        for shape, dtype in specs:
            n = 1
            for d in shape:
                n *= int(d)
            total = (total + 255) // 256 * 256 + n * torch.empty((), dtype=dtype).element_size()
        return total + 256

    def free(self):
        if getattr(self, 'ptr', None):
            ptr, self.ptr = self.ptr, None
            try:
                load().mpe_host_free(C.c_void_p(ptr))
            except Exception:  # noqa: BLE001 - interpreter shutdown: the library may already be gone
                pass

    __del__ = free
