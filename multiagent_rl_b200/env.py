"""Host-side mirror of the reference's env surface on top of the CUDA kernels.

Mirrors ``experiments/scenarios.py:124-192`` (``make_env``) and the upstream ``MultiAgentEnv``
object it returns (``reset`` / ``step`` / ``seed`` / ``render`` / ``n`` / ``observation_space`` /
``action_space`` / ``force_discrete_action`` ...), so that ``main.py:39-65`` and
``experiments/run.py:28,44,60`` run against it unchanged.

Two surfaces (SURVEY.md section 8b):
  * ``num_envs == 1`` (default): the reference's list-of-numpy surface.
  * ``num_envs > 1`` or ``batched=True``: device tensors, ``step(act_u[B,N] int32, act_c=None)``
    -> ``obs[B,N,D], rew[B,N], done[B,N], info``; nothing leaves the GPU.
All compute is in libmpe_b200.so; without it (or without a GPU) construction raises.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .spaces import Box, Discrete, MultiDiscrete

SCENARIOS = ('simple_spread', 'simple_reference', 'simple_speaker_listener', 'fullobs_collect_treasure')


class _World(object):
    """The attributes of upstream ``World`` that callers read (``env.world.dim_c``)."""

    def __init__(self, dim_c, n_agents, n_landmarks):
        self.dim_c = dim_c
        self.dim_p = 2
        self.dim_color = 3
        self.dt = 0.1
        self.damping = 0.25
        self.contact_force = 1e+2
        self.contact_margin = 1e-3
        self.collaborative = False  # experiments/scenarios.py:171
        self.num_agents = n_agents
        self.num_landmarks = n_landmarks


class BatchedMultiAgentEnv(object):
    def __init__(self, scenario_name, n=None, benchmark=False, discrete_action=True, num_envs=1,
                 device=None, precision='fp32', seed=0, env_id_offset=0, rng=None, batched=None,
                 max_episode_len=25, max_speed=None, accel=None):
        if scenario_name not in SCENARIOS:
            raise ValueError('unsupported scenario %r (supported: %s)' % (scenario_name, ', '.join(SCENARIOS)))
        if not discrete_action:
            raise NotImplementedError('continuous action spaces are not on the reference path '
                                      '(main.py:39 passes discrete_action=True)')
        if not torch.cuda.is_available():
            raise RuntimeError('multiagent_rl_b200 needs a CUDA device: the particle env runs only as '
                               'sm_100a kernels (no CPU fallback)')
        self._lib = _lib.load()
        self.device = torch.device(device if device is not None else 'cuda:%d' % torch.cuda.current_device())
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        self.scenario_name = scenario_name
        self.num_envs = int(num_envs)
        self.batched = bool(batched) if batched is not None else self.num_envs > 1
        self.precision = precision
        self.dtype = {'fp32': torch.float32, 'fp64': torch.float64}[precision]
        self.benchmark = benchmark
        self.max_episode_len = int(max_episode_len)  # rls/arglist.py:5; EpisodeHistory.for_env reads it
        self.rng = rng if rng is not None else ('numpy' if not self.batched else 'philox')
        self.env_id_offset = int(env_id_offset)
        cfg = _lib.MpeConfig(scenario=_lib.SCENARIO_IDS[scenario_name], num_agents=0 if n is None else int(n),
                             precision=_lib.F32 if precision == 'fp32' else _lib.F64,
                             device=self.device.index, num_envs=self.num_envs, env_id_offset=self.env_id_offset,
                             seed=int(seed) & (2 ** 64 - 1), max_episode_len=int(max_episode_len), reserved0=0,
                             max_speed=-1.0 if max_speed is None else float(max_speed),
                             accel=-1.0 if accel is None else float(accel))
        h = C.c_void_p()
        _lib.check(self._lib.mpe_create(C.byref(cfg), C.byref(h)), 'mpe_create')
        self._h = h
        dims = _lib.MpeDims()
        _lib.check(self._lib.mpe_query(self._h, C.byref(dims)), 'mpe_query')
        self.n = dims.num_agents
        self.num_landmarks = dims.num_landmarks
        self.obs_dim = dims.obs_dim
        self.dim_c = dims.dim_c
        self.act_c = dims.act_c  # width of the message head (0: single Discrete(5) head)
        self.world = _World(self.dim_c, self.n, self.num_landmarks)
        self.shared_reward = False  # world.collaborative = False (experiments/scenarios.py:171)
        # writable attributes of upstream MultiAgentEnv
        self.discrete_action_space = True
        self.discrete_action_input = False
        self.force_discrete_action = True  # experiments/scenarios.py:191
        self.time = 0
        if self.act_c > 0:
            self.action_space = [MultiDiscrete([[0, 4], [0, self.act_c - 1]]) for _ in range(self.n)]
        else:
            self.action_space = [Discrete(5) for _ in range(self.n)]
        self.observation_space = [Box(-np.inf, +np.inf, (self.obs_dim,), np.float32) for _ in range(self.n)]
        self._seed = int(seed)
        self.global_step = 0

    # ------------------------------------------------------------------ plumbing
    def __del__(self):
        h = getattr(self, '_h', None)
        if h is not None and self._lib is not None:
            self._lib.mpe_destroy(h)
            self._h = None

    close = __del__

    def _stream(self):
        return _lib.current_stream(self.device)

    def _empty(self, *shape, dtype=None):
        return torch.empty(shape, dtype=dtype or self.dtype, device=self.device)

    def _as_dev(self, x, dtype):
        if x is None:
            return None
        t = torch.as_tensor(x, dtype=dtype, device=self.device)
        return t.contiguous()

    # ------------------------------------------------------------------ reference surface
    def seed(self, seed=None):
        """main.py:45.  The MAAC-fork ``_seed`` reseeds numpy's global RNG; the Philox key follows."""
        seed = 1 if seed is None else int(seed)
        np.random.seed(seed)
        self._seed = seed
        _lib.check(self._lib.mpe_seed(self._h, C.c_uint64(seed & (2 ** 64 - 1)), self._stream()), 'mpe_seed')
        return [seed]

    def render(self, mode='human', close=False):
        """No viewer on a headless GPU box (``arglist.display`` is False on the reference path)."""
        return []

    def reset(self, mask=None):
        if self.rng == 'numpy':
            self._reset_numpy(mask)
            obs = self.observe()
        else:
            obs = self._empty(self.num_envs, self.n, self.obs_dim)
            m = self._as_dev(mask, torch.uint8)
            _lib.check(self._lib.mpe_reset(self._h, _lib.ptr(m), _lib.ptr(obs), self._stream()), 'mpe_reset')
        return obs if self.batched else self._obs_list(obs)

    def _reset_numpy(self, mask=None):
        """Draw like upstream ``reset_world`` from numpy's GLOBAL RNG, in upstream's order (goal
        landmarks via np.random.choice first, then agents, then landmarks), env by env."""
        B, N, L = self.num_envs, self.n, self.num_landmarks
        idx = range(B) if mask is None else [b for b in range(B) if mask[b]]
        pos, vel, lm, goal = self.get_state()
        pos, vel, lm, goal = pos.cpu().numpy(), vel.cpu().numpy(), lm.cpu().numpy(), goal.cpu().numpy()
        if self.scenario_name == 'fullobs_collect_treasure':
            # MAAC fork reset_world: agents, then per treasure its type (np.random.choice) and its position
            for b in idx:
                for i in range(N):
                    pos[b, i] = np.random.uniform(low=-1, high=1, size=2)
                    vel[b, i] = 0.0
                types = 0
                for l in range(L):
                    types |= int(np.random.choice(2)) << l
                    lm[b, l] = np.random.uniform(low=-0.95, high=0.95, size=2)
                goal[b, 0] = types | (0x3F << 6)  # all alive, nobody holds anything
            self.set_state(pos, vel, lm, goal)
            self._tr_flags = goal[:, 0].copy()
            return
        for b in idx:
            if self.scenario_name == 'simple_reference':
                goal[b, 0] = np.random.choice(L)
                goal[b, 1] = np.random.choice(L)
            elif self.scenario_name == 'simple_speaker_listener':
                goal[b, 0] = np.random.choice(L)
                goal[b, 1] = -1
            for i in range(N):
                pos[b, i] = np.random.uniform(-1, +1, 2)
                vel[b, i] = 0.0
            for l in range(L):
                lm[b, l] = np.random.uniform(-1, +1, 2)
        self.set_state(pos, vel, lm, goal)

    def step(self, action_n, act_c=None, out=None, info=False):
        if self.batched:
            return self.step_tensor(action_n, act_c, out=out, info=info)
        return self._step_list(action_n)

    # ------------------------------------------------------------------ list surface (num_envs == 1)
    def _obs_list(self, obs):
        o = obs.detach().to('cpu', torch.float64).numpy()
        return [o[0, i].copy() for i in range(self.n)]

    def _step_list(self, action_n):
        """upstream MultiAgentEnv.step on one env: list of N action vectors (len 5 or 5 + dim_c)."""
        N = self.n
        if len(action_n) != N:
            raise ValueError('expected %d actions, got %d' % (N, len(action_n)))
        act_u = np.zeros((1, N), dtype=np.int32)
        comm = np.zeros((1, N, max(self.dim_c, 1)), dtype=np.float64)
        for i, a in enumerate(action_n):
            if self.discrete_action_input:
                # upstream's index branch: 1 -> u[0] = -1, 2 -> +1, 3 -> u[1] = -1, 4 -> +1
                parts = list(a) if self.act_c > 0 else [a]
                act_u[0, i] = {0: 0, 1: 2, 2: 1, 3: 4, 4: 3}[int(np.asarray(parts[0]).reshape(-1)[0])]
                if self.act_c > 0:
                    comm[0, i, int(parts[1])] = 1.0
                continue
            a = np.asarray(a) if not isinstance(a, np.ndarray) else a
            if a.shape[0] != 5 + self.act_c:
                raise AssertionError('action of agent %d has %d entries, expected %d' % (i, a.shape[0], 5 + self.act_c))
            d = int(np.argmax(a[:5]))
            movable = not (self.scenario_name == 'simple_speaker_listener' and i == 0)  # the speaker
            if movable and self.force_discrete_action and a.dtype.kind == 'f':
                a[:5] = 0.0  # in place, like upstream: the caller's arrays become exact one-hots
                a[d] = 1.0
            act_u[0, i] = d
            if self.act_c > 0:
                comm[0, i, :self.dim_c] = a[5:5 + self.dim_c]
        obs, rew, done, info = self.step_tensor(torch.from_numpy(act_u), None,
                                                comm_vec=comm if self.act_c > 0 else None, info=self.benchmark)
        self.time += 1
        if self.scenario_name == 'fullobs_collect_treasure' and self.rng == 'numpy':
            self._respawn_numpy()
        o = obs.detach().to('cpu', torch.float64).numpy()
        r = rew.detach().to('cpu', torch.float64).numpy()
        obs_n = [o[0, i].copy() for i in range(N)]
        rew_n = [r[0, i] for i in range(N)]
        done_n = [False] * N
        if self.benchmark and self.scenario_name == 'simple_spread':
            ii = info['info_i'].cpu().numpy()
            md = float(info['info_f'].cpu().numpy()[0])
            info_n = {'n': [(rew_n[i], int(ii[0, i]), md, int(ii[0, N])) for i in range(N)]}
        elif self.benchmark and self.scenario_name == 'fullobs_collect_treasure':
            ii = info['info_i'].cpu().numpy()
            info_n = {'n': [int(ii[0, i]) for i in range(N)]}
        elif self.benchmark:
            info_n = {'n': [rew_n[i] for i in range(N)]}
        else:
            info_n = {'n': [{} for _ in range(N)]}
        if self.shared_reward:  # upstream MultiAgentEnv.step: world.collaborative -> every agent gets the sum
            rew_n = [np.sum(rew_n)] * N
        return obs_n, rew_n, done_n, info_n

    def _respawn_numpy(self):
        """rng='numpy' (the one-env drop-in): the treasures that post_step respawned in this step (dead one step
        earlier) get the draws upstream would have taken from numpy's GLOBAL generator, in upstream's order per
        treasure: probability, position, type."""
        prev = getattr(self, '_tr_flags', None)
        pos, vel, lm, goal = self.get_state()
        lm, goal = lm.cpu().numpy(), goal.cpu().numpy()
        if prev is not None:
            changed = False
            for b in range(self.num_envs):
                for l in range(self.num_landmarks):
                    if not (int(prev[b]) >> (6 + l)) & 1:
                        np.random.uniform()  # <= respawn_prob (1.0)
                        lm[b, l] = np.random.uniform(low=-0.95, high=0.95, size=2)
                        goal[b, 0] = (int(goal[b, 0]) & ~(1 << l)) | (int(np.random.choice(2)) << l)
                        changed = True
            if changed:
                self.set_state(None, None, lm, goal)
        self._tr_flags = goal[:, 0].copy()

    def _check_out(self, out, host):
        """``out`` = (obs[B,N,D], rew[B,N], done[B,N] uint8): each entry None (that output is skipped) or a
        C-contiguous buffer of exactly that shape and dtype, on the env's device (``host=False``: torch tensors) or
        in host memory (``host=True``: numpy arrays or CPU tensors).  The kernels write B*N*D / B*N elements through
        the raw pointer, so anything else would be written out of bounds or misread: refuse it before any launch."""
        B, N = self.num_envs, self.n
        if not isinstance(out, (tuple, list)) or len(out) != 3:
            raise ValueError('out must be a tuple (obs, rew, done)')
        real = np.float32 if self.precision == 'fp32' else np.float64
        want = (('obs', (B, N, self.obs_dim), real), ('rew', (B, N), real), ('done', (B, N), np.uint8))
        for x, (name, shape, dt) in zip(out, want):
            if x is None:
                continue
            if isinstance(x, torch.Tensor):
                if x.device.type == 'cpu':
                    where = 'host'
                elif x.device == self.device:
                    where = 'device'
                else:
                    where = str(x.device)
                dtype_ok = x.dtype == {np.float32: torch.float32, np.float64: torch.float64, np.uint8: torch.uint8}[dt]
                contiguous = x.is_contiguous()
                got = (tuple(x.shape), x.dtype)
            elif isinstance(x, np.ndarray) and host:
                where, dtype_ok, contiguous = 'host', x.dtype == dt, bool(x.flags['C_CONTIGUOUS'])
                got = (x.shape, x.dtype)
            else:
                raise ValueError('out %s must be a %s or None, got %s' % (name, 'numpy array / CPU tensor' if host
                                                                         else 'torch tensor', type(x).__name__))
            if where != ('host' if host else 'device'):
                raise ValueError('out %s must be in %s, got a tensor on %s' % (
                    name, 'host memory' if host else str(self.device), where))
            if tuple(got[0]) != shape or not dtype_ok:
                raise ValueError('out %s must be %s %s, got %s %s' % (name, np.dtype(dt).name, shape, got[1], got[0]))
            if not contiguous:
                raise ValueError('out %s must be contiguous' % name)
        return tuple(out)

    # ------------------------------------------------------------------ tensor surface
    def step_tensor(self, act_u, act_c=None, comm_vec=None, out=None, info=False):
        """act_u [B,N] int (index of the movement head), act_c [B,N] int (message head) or
        comm_vec [B,N,dim_c] real.  Returns (obs[B,N,D], rew[B,N], done[B,N] uint8, info dict).
        ``out`` = (obs, rew, done) writes into the caller's device tensors instead (see ``_check_out``)."""
        B, N = self.num_envs, self.n
        if out is not None:
            out = self._check_out(out, host=False)
        if self.discrete_action_input:
            remap = torch.tensor([0, 2, 1, 4, 3], device=self.device, dtype=torch.int32)
            act_u = remap[torch.as_tensor(act_u, device=self.device).long()]
        au = self._as_dev(act_u, torch.int32)
        if au.numel() != B * N:
            raise ValueError('act_u must have %d entries' % (B * N))
        ac = self._as_dev(act_c, torch.int32)
        cv = self._as_dev(comm_vec, self.dtype)
        if self.scenario_name == 'simple_reference' and ac is None and cv is None:
            raise ValueError('simple_reference needs act_c or comm_vec')
        if out is None:
            obs = self._empty(B, N, self.obs_dim)
            rew = self._empty(B, N)
            done = self._empty(B, N, dtype=torch.uint8)
        else:
            obs, rew, done = out
        info_i = self._empty(B, N + 1, dtype=torch.int32) if info else None
        info_f = self._empty(B) if info else None
        _lib.check(self._lib.mpe_step(self._h, _lib.ptr(au), _lib.ptr(ac), _lib.ptr(cv), _lib.ptr(obs),
                                      _lib.ptr(rew), _lib.ptr(done), _lib.ptr(info_i), _lib.ptr(info_f),
                                      self._stream()), 'mpe_step')
        self.global_step += 1
        return obs, rew, done, ({'info_i': info_i, 'info_f': info_f} if info else {})

    def step_host(self, act_u, act_c=None, out=None):
        """Same step through HOST buffers (numpy / pinned torch tensors): H2D actions, kernel, D2H
        obs/rew/done, synchronise.  This is the cost a list-of-numpy caller pays per step."""
        B, N = self.num_envs, self.n
        if out is None:
            dt = np.float32 if self.precision == 'fp32' else np.float64
            out = (np.empty((B, N, self.obs_dim), dt), np.empty((B, N), dt), np.empty((B, N), np.uint8))
        else:
            out = self._check_out(out, host=True)
        obs, rew, done = out
        _lib.check(self._lib.mpe_step_host(self._h, _lib.ptr(act_u), _lib.ptr(act_c), _lib.ptr(obs), _lib.ptr(rew),
                                           _lib.ptr(done), self._stream()), 'mpe_step_host')
        self.global_step += 1
        return obs, rew, done

    def observe(self):
        obs = self._empty(self.num_envs, self.n, self.obs_dim)
        _lib.check(self._lib.mpe_observe(self._h, _lib.ptr(obs), self._stream()), 'mpe_observe')
        return obs

    def set_state(self, pos=None, vel=None, lm=None, goal=None):
        """pos/vel [B,N,2], lm [B,L,2], goal [B,N] (-1 = None)."""
        p, v, l = (self._as_dev(x, self.dtype) for x in (pos, vel, lm))
        g = self._as_dev(goal, torch.int32)
        _lib.check(self._lib.mpe_set_state(self._h, _lib.ptr(p), _lib.ptr(v), _lib.ptr(l), _lib.ptr(g),
                                           self._stream()), 'mpe_set_state')

    def get_state(self):
        B, N, L = self.num_envs, self.n, self.num_landmarks
        pos, vel, lm = self._empty(B, N, 2), self._empty(B, N, 2), self._empty(B, L, 2)
        goal = self._empty(B, N, dtype=torch.int32)
        _lib.check(self._lib.mpe_get_state(self._h, _lib.ptr(pos), _lib.ptr(vel), _lib.ptr(lm), _lib.ptr(goal),
                                           self._stream()), 'mpe_get_state')
        return pos, vel, lm, goal

    # ------------------------------------------------------------------ episode statistics
    def track_returns(self, enable=True):
        _lib.check(self._lib.mpe_track_returns(self._h, 1 if enable else 0), 'mpe_track_returns')

    def stats_tensor(self):
        """Zero-copy float64[5] CUDA tensor aliasing the shard's statistics (for NCCL reductions without a host
        sync): [sum(return), sum(return^2), n_episodes, n_steps, n_nonfinite_episodes].  Valid while the env is alive."""
        p = C.c_void_p()
        _lib.check(self._lib.mpe_stats_ptr(self._h, C.byref(p)), 'mpe_stats_ptr')

        class _Alias(object):
            __cuda_array_interface__ = {'shape': (_lib.STATS_LEN,), 'typestr': '<f8', 'data': (int(p.value), False), 'version': 2}
        with torch.cuda.device(self.device):
            t = torch.as_tensor(_Alias(), device=self.device)
        t._mpe_owner = self  # keep the env (and the device buffer) alive
        return t

    def read_stats(self, clear=False):
        """-> np.array([sum(return), sum(return^2), n_episodes, n_steps, n_nonfinite_episodes]) for this shard
        (host sync).  Episodes with a NaN/inf return (coincident agents, like upstream) are counted in [4] only."""
        out = (C.c_double * _lib.STATS_LEN)()
        _lib.check(self._lib.mpe_stats_read(self._h, out, 1 if clear else 0, self._stream()), 'mpe_stats_read')
        return np.array(list(out), dtype=np.float64)

    # ------------------------------------------------------------------ fused rollout
    def rollout(self, actor, T, step0=None, record=False, replay=None, info=False):
        """T fused iterations of experiments/run.py:36-65 (act -> step -> reward -> auto-reset).
        ``record`` returns per-step (obs_next[T,B,N,D], rew[T,B,N], act_u[T,B,N], act_c[T,B,N] | None).
        ``info`` also records upstream's ``benchmark_data`` of every step, bit for bit what ``step(info=True)`` returns
        for it: the call returns (obs_next, rew, act_u, act_c, {'info_i': int32 [T,B,N+1], 'info_f': fp32 [T,B]}),
        the first four None without ``record``.  info_i holds the collisions per agent and the occupied landmarks
        (fullobs_collect_treasure: the 0 / 1 flags per agent and a zero), info_f the sum of min distances (None for
        fullobs_collect_treasure).
        ``replay`` (a DeviceReplayBuffer) receives every env-step's transition (obs_t, act, sum of rewards, obs_t+1,
        done = 0) in step-major, then env order, as ``T`` calls of ``replay.add`` with ``B`` transitions each would:
        obs_t is the observation the actor acted on, the post-reset one at an episode's first step.
        Memory: on envs whose episodes are aligned (small teams on the tensor cores), the recordings not requested here
        go to a scratch buffer the env keeps until it is destroyed - one segment's worth, at most 1 GiB (144 B per env
        and step for simple_spread N = 3 without ``record``); other envs keep two observation buffers and a reward
        buffer of one step."""
        if self.precision != 'fp32':
            raise RuntimeError('rollout is fp32 only')
        B, N = self.num_envs, self.n
        if replay is not None:
            self._check_replay(replay)
        step0 = self.global_step if step0 is None else int(step0)
        obs = rew = au = ac = None
        if record:
            obs = self._empty(T, B, N, self.obs_dim)
            rew = self._empty(T, B, N)
            au = self._empty(T, B, N, dtype=torch.int32)
            ac = self._empty(T, B, N, dtype=torch.int32) if self.act_c > 0 else None
        info_i = self._empty(T, B, N + 1, dtype=torch.int32) if info else None
        info_f = self._empty(T, B) if info and self.scenario_name != 'fullobs_collect_treasure' else None
        if replay is None:
            _lib.check(self._lib.mpe_rollout(self._h, actor._h, int(T), C.c_uint64(step0), _lib.ptr(obs), _lib.ptr(rew),
                                             _lib.ptr(au), _lib.ptr(ac), _lib.ptr(info_i), _lib.ptr(info_f),
                                             self._stream()), 'mpe_rollout')
        else:
            _lib.check(self._lib.mpe_rollout_replay(self._h, actor._h, replay._h, int(T), C.c_uint64(step0),
                                                    _lib.ptr(obs), _lib.ptr(rew), _lib.ptr(au), _lib.ptr(ac),
                                                    _lib.ptr(info_i), _lib.ptr(info_f), self._stream()),
                       'mpe_rollout_replay')
        self.global_step = step0 + int(T)
        if info:
            return obs, rew, au, ac, {'info_i': info_i, 'info_f': info_f}
        return (obs, rew, au, ac) if record else None

    def _check_replay(self, replay):
        """The ring stores this env's transitions: same device, agents, observation width and action heads, and room
        for one step of every env."""
        from .replay import DeviceReplayBuffer
        if not isinstance(replay, DeviceReplayBuffer):
            raise ValueError('replay must be a DeviceReplayBuffer, got %s' % type(replay).__name__)
        if replay.device != self.device:
            raise ValueError('replay is on %s, the env on %s' % (replay.device, self.device))
        if (replay.N, replay.D) != (self.n, self.obs_dim):
            raise ValueError('replay stores %d agents x %d observations, the env has %d x %d'
                             % (replay.N, replay.D, self.n, self.obs_dim))
        if (replay.act_dims[0], replay.A1) != (5, self.act_c):
            raise ValueError('replay action heads %s do not match the env (5, %d)' % (replay.act_dims, self.act_c))
        if self.num_envs > replay._maxsize:
            raise ValueError('replay holds %d transitions, fewer than one step of %d envs' % (replay._maxsize, self.num_envs))


def make_env(scenario_name, n=None, local_observation=True, benchmark=False, discrete_action=True, **kw):
    """Signature of experiments/scenarios.py:124 plus keyword-only batching options
    (num_envs, device, precision, seed, env_id_offset, rng, batched, max_episode_len).

    Only the reference's partial observations are implemented: ``local_observation`` must be True,
    which is what main.py:39 and main_scalability_1.py:36 pass."""
    if not local_observation:
        raise NotImplementedError('only local_observation=True (the reference path) is implemented')
    return BatchedMultiAgentEnv(scenario_name, n=n, benchmark=benchmark, discrete_action=discrete_action, **kw)
