"""Every env kernel instantiation through every store path it picks at run time, against the float64 oracle.

Each output of k_step / k_reset / k_observe (one thread per env, 32 envs per warp), k_step_grp / k_reset_grp (G lanes
per env, EPW = 32 / G envs per warp) and k_treasure (4 lanes per env, 8 envs per warp) leaves one of three ways:
  * full warp, 16 B-aligned output: rows staged in shared memory, one TMA bulk store per warp (emit_outputs; grp_emit,
    per env in the fp64 group build; k_treasure).  Variants (a) and (b) of test_step_store_paths_agree_and_match_the_oracle,
    the full resets of test_masked_resets_and_observe_into_caller_buffers;
  * full warp, output not 16 B-aligned: a coalesced copy out of staging (emit_outputs, k_treasure) or rows stored
    straight from registers (grp_emit); `done` by bytes instead of 32-bit words (k_step).  Variant (c) of the step test,
    every masked reset and observe of the reset test;
  * the ragged last warp: every env writes its own rows.  B = 4,099 (prime) leaves a partial last warp in every family,
    after several full CTAs; _assert_geometry checks that.
simple_spread n = 5 in fp64 is the per-agent staging path (32 rows of 70 doubles exceed the 16 KB staging tile).
test_null_output_subsets drives each NULL output the header allows, test_real_valued_messages the comm_vec branch of
simple_reference, test_out_is_validated the host-side checks of BatchedMultiAgentEnv's `out` buffers.

Caller buffers sit inside a guard band and are pre-filled with a sentinel (NaN for reals, 0xA5 for done, -7 for
info_i) before every call: the guard must stay untouched (no overrun past either end) and no sentinel may remain
inside (no skipped row), except info_f of fullobs_collect_treasure, which the kernel never writes.  The Philox keys
use a 64-bit seed with a non-zero high word and env ids that cross 2^32 inside the batch (env_id_offset = 2^32 - 2000).

Tolerances.  The three store paths of one computation are compared BIT for bit.  fp64 build against the float64
oracle: 1e-12 absolute on observations, rewards and state, flags and state words bit-exact, free-running.
fp32 build: the oracle is re-synchronised from the device state before every step and one step is compared (the
single-step tolerances of test_gpu_treasure.py's fixture test): 2e-5 on positions, 2e-4 on velocities, observations
and rewards; a collision / occupancy flag may differ only where the deciding distance lies within 1e-5 of its
threshold, and such envs are left out of the reward comparison (a flipped flag moves a reward by 1).  Philox resets
are bit-exact in both builds; observations of a reset state match to 1e-12 (fp64) / 1e-6 (fp32), as in
test_gpu_env.py, and offsets to a dead treasure (about -999) to 1e-4 in fp32.
"""
import numpy as np
import pytest
import torch

from oracle import maac_vec, mpe_vec, philox
from tests.test_gpu_treasure import _near_threshold

pytestmark = pytest.mark.gpu

B = 4099                    # prime: a ragged last warp in every family, after many full CTAs
SEED = 2 ** 40 + 9          # high key word non-zero
OFF = 2 ** 32 - 2000        # env ids cross into the counter's high word at env 2,000
TR = 'fullobs_collect_treasure'
F64_ATOL = 1e-12
F32_POS, F32_VEL, F32_REW, F32_BAND = 2e-5, 2e-4, 2e-4, 1e-5
NAN, DONE_FILL, INFO_FILL = float('nan'), 0xA5, -7

FAMILIES = ([('simple_spread', n) for n in range(1, 13)] +
            [('simple_reference', None), ('simple_speaker_listener', None), (TR, None)])
FAMILY_IDS = ['spread%d' % n for n in range(1, 13)] + ['reference', 'speaker_listener', 'treasure']
PRECISIONS = ['fp32', 'fp64']

GROUP_LANES = {6: 2, 7: 7, 8: 4, 9: 3, 10: 5, 11: 11, 12: 4}   # env_group.cuh group_lanes()
_INT = {torch.float32: torch.int32, torch.float64: torch.int64, torch.uint8: torch.uint8, torch.int32: torch.int32}


def _envs_per_warp(scenario, n):
    if scenario == TR:
        return 8                                   # env_treasure.cuh kTrEpw
    if scenario == 'simple_spread' and n >= 6:
        return 32 // GROUP_LANES[n]                # GroupLayout::EPW
    return 32                                      # one thread per env


def _assert_geometry(scenario, n):
    """128 threads per CTA in every family: several full CTAs, then a last warp that is only partly filled."""
    epw = _envs_per_warp(scenario, n)
    assert B // (4 * epw) >= 8 and 0 < B % epw < epw, (scenario, n, epw)


def _mk(scenario, n, precision, **kw):
    import multiagent_rl_b200 as m
    return m.make_env(scenario, n=n, num_envs=B, batched=True, precision=precision, seed=SEED, env_id_offset=OFF, **kw)


def _np(t):
    return t.detach().cpu().numpy().astype(np.float64)


def _bits(t):
    return t.view(_INT[t.dtype])


def _same(a, b):
    return torch.equal(_bits(a), _bits(b))


def _same_state(e1, e2):
    return all(_same(x, y) for x, y in zip(e1.get_state(), e2.get_state()))


class _Guarded(object):
    """A caller buffer inside a guard band, pre-filled with a sentinel: offset 0 starts it 16 B-aligned, offset 1 one
    element past that (4 B / 8 B for reals, 1 B for done, 4 B for info_i)."""

    def __init__(self, shape, dtype, fill, offset):
        es = torch.empty((), dtype=dtype).element_size()
        self.n = int(np.prod(shape))
        self.lo = 16 // es + offset
        self.buf = torch.full((self.lo + self.n + 16 // es,), fill, dtype=dtype, device='cuda')
        assert self.buf.data_ptr() % 16 == 0
        self.t = self.buf[self.lo:self.lo + self.n].view(shape)
        assert (self.t.data_ptr() % 16 == 0) == (offset == 0)
        self.fill = fill
        self.fill_bits = _bits(torch.full((1,), fill, dtype=dtype, device='cuda'))

    def refill(self):
        self.buf.fill_(self.fill)

    def check(self, what, written=True):
        guard = torch.cat([self.buf[:self.lo], self.buf[self.lo + self.n:]])
        assert bool((_bits(guard) == self.fill_bits).all()), (what, 'guard band overwritten')
        left = _bits(self.t) == self.fill_bits
        if written:
            assert not bool(left.any()), (what, 'elements left unwritten', int(left.sum()))
        else:
            assert bool(left.all()), (what, 'written although the kernel never writes it')


OUTPUTS = ('obs', 'rew', 'done', 'info_i', 'info_f')


def _out_specs(env):
    Bn, N, D = env.num_envs, env.n, env.obs_dim
    return {'obs': ((Bn, N, D), env.dtype, NAN), 'rew': ((Bn, N), env.dtype, NAN),
            'done': ((Bn, N), torch.uint8, DONE_FILL), 'info_i': ((Bn, N + 1), torch.int32, INFO_FILL),
            'info_f': ((Bn,), env.dtype, NAN)}


class _Outputs(object):
    """The five outputs of mpe_step: 'default' = fresh torch.empty tensors, 'aligned' / 'offset' = _Guarded buffers."""

    def __init__(self, env, kind, names=OUTPUTS):
        self.kind, self.scenario = kind, env.scenario_name
        specs = _out_specs(env)
        self.g = {}
        self.t = {k: None for k in OUTPUTS}
        for k in names:
            shape, dt, fill = specs[k]
            if kind == 'default':
                self.t[k] = torch.empty(shape, dtype=dt, device='cuda')
            else:
                self.g[k] = _Guarded(shape, dt, fill, 0 if kind == 'aligned' else 1)
                self.t[k] = self.g[k].t
        if kind == 'offset' and 'done' in self.g:
            assert self.t['done'].data_ptr() % 4 != 0   # k_step's per-byte done stores

    def refill(self):
        for g in self.g.values():
            g.refill()

    def check(self, what):
        for k, g in self.g.items():
            g.check((what, self.kind, k), written=not (k == 'info_f' and self.scenario == TR))


def _step(env, act, ac, cv, out):
    from multiagent_rl_b200 import _lib
    t = out.t
    _lib.check(env._lib.mpe_step(env._h, _lib.ptr(act), _lib.ptr(ac), _lib.ptr(cv), _lib.ptr(t['obs']),
                                 _lib.ptr(t['rew']), _lib.ptr(t['done']), _lib.ptr(t['info_i']), _lib.ptr(t['info_f']),
                                 env._stream()), 'mpe_step')


def _actions(env, rng):
    act = torch.from_numpy(rng.randint(0, 5, (B, env.n)).astype(np.int32)).cuda()
    ac = torch.from_numpy(rng.randint(0, 10, (B, env.n)).astype(np.int32)).cuda() \
        if env.scenario_name == 'simple_reference' else None
    return act, ac


def _oracle_act_c(scenario, act, ac):
    """simple_reference: the message head; the speaker's message is the first dim_c entries of its width-5 one-hot."""
    if scenario == 'simple_reference':
        return ac.cpu().numpy()
    if scenario == 'simple_speaker_listener':
        return act.cpu().numpy()
    return None


def _make_oracle(scenario, n, state):
    pos, vel, lm, goal = (x.cpu().numpy() for x in state)
    if scenario == TR:
        v = maac_vec.VecTreasure(B, seed=SEED, gid0=OFF)
        v.reset()                                  # episode 0, step counter 0: the keys of the respawn draws
        v.set_state(pos, vel, lm, goal[:, 0])
    else:
        v = mpe_vec.VecEnv(mpe_vec.Spec(scenario, n), B)
        v.set_state(pos, vel, lm, goal)
    return v


def _sync_oracle(v, scenario, state):
    pos, vel, lm, goal = (x.cpu().numpy() for x in state)
    v.set_state(pos, vel, lm, goal[:, 0] if scenario == TR else goal)


def _spread_flag_band(v, ii, coll, occ):
    """fp32: env mask of flags that agree with the oracle; a flag may differ only within F32_BAND of its threshold."""
    N = v.spec.N
    bad = ii[:, :N] != coll
    d = np.linalg.norm(v.pos[:, :, None] - v.pos[:, None, :], axis=-1)
    near = (np.abs(d - 0.3) < F32_BAND).any(axis=2)
    assert np.all(near[bad]), ('collision flag away from its threshold', np.argwhere(bad & ~near)[:5])
    bad_o = ii[:, N] != occ
    dl = np.linalg.norm(v.pos[:, :, None] - v.lm[:, None, :], axis=-1).min(axis=1)
    near_o = (np.abs(dl - 0.1) < F32_BAND).any(axis=1)
    assert np.all(near_o[bad_o]), ('occupied flag away from its threshold', np.nonzero(bad_o & ~near_o)[0][:5])
    return ~bad.any(axis=1) & ~bad_o


def _dead_apart(tr):
    """dead treasures all sit at (-999, -999): move them apart so that they do not read as ties of the sorted list"""
    tr = tr.copy()
    for l in range(tr.shape[1]):
        tr[tr[:, l, 0] < -900, l] = 1000.0 * (l + 2)
    return tr


def _check_step_against_oracle(scenario, precision, v, act, ac, t, state, respawns):
    """Step the oracle and compare the outputs `t` and the device state after the step."""
    o_dev = _np(t['obs'])
    r_dev = _np(t['rew'])
    ii = t['info_i'].cpu().numpy()
    pos, vel, lm, goal = state
    if scenario == TR:
        tr_before = _dead_apart(v.tr)
        hi = v.gid >= np.uint64(2 ** 32)
        dead = ~v.alive                            # these respawn in this step's post_step (respawn_prob = 1)
        respawns[0] += int(dead[~hi].sum())
        respawns[1] += int(dead[hi].sum())
        o, r, info = v.step(act.cpu().numpy())
        far = np.abs(o) > 100                      # offsets to a dead treasure
        if precision == 'fp64':
            ok = np.ones(B, dtype=bool)
            tol_o = tol_far = tol_p = tol_v = tol_tr = F64_ATOL
            tol_r = np.full(B, F64_ATOL)
        else:
            ok = ~_near_threshold(v.pos, tr_before, F32_BAND)
            assert ok.mean() > 0.9, ok.mean()
            tol_o, tol_far, tol_p, tol_v, tol_tr = F32_VEL, 1e-4, F32_POS, F32_VEL, 1e-4
            tol_r = 2e-5 + 1e-4 * far.any(axis=(1, 2))
        err = np.abs(o_dev - o)[ok]
        assert err[~far[ok]].max() <= tol_o and (not far[ok].any() or err[far[ok]].max() <= tol_far)
        assert np.all((np.abs(r_dev - r).max(axis=1) <= tol_r)[ok])
        assert np.array_equal(ii[:, :8][ok], info[ok]) and not ii[:, 8].any()
        assert np.abs(_np(pos) - v.pos).max() <= tol_p and np.abs(_np(vel) - v.vel).max() <= tol_v
        assert np.abs(_np(lm) - v.tr)[ok].max() <= tol_tr
        assert np.array_equal(goal[:, 0].cpu().numpy().astype(np.int64)[ok], v.flags()[ok])
        return
    o, r, (coll, occ) = v.step(act.cpu().numpy(), act_c=_oracle_act_c(scenario, act, ac))
    md = v.min_dists_sum() if scenario == 'simple_spread' else np.zeros(B)
    N = v.spec.N
    if precision == 'fp64':
        assert np.abs(o_dev - o).max() <= F64_ATOL and np.abs(r_dev - r).max() <= F64_ATOL
        assert np.array_equal(ii[:, :N], coll) and np.array_equal(ii[:, N], occ)
        assert np.abs(_np(t['info_f']) - md).max() <= F64_ATOL
        assert np.abs(_np(pos) - v.pos).max() <= F64_ATOL and np.abs(_np(vel) - v.vel).max() <= F64_ATOL
    else:
        ok = _spread_flag_band(v, ii, coll, occ)
        assert ok.mean() > 0.99, ok.mean()
        assert np.abs(o_dev - o).max() <= F32_VEL and np.abs(r_dev - r)[ok].max() <= F32_REW
        assert np.abs(_np(t['info_f']) - md).max() <= F32_REW
        assert np.abs(_np(pos) - v.pos).max() <= F32_POS and np.abs(_np(vel) - v.vel).max() <= F32_VEL
    assert np.array_equal(_np(lm), v.lm) and np.array_equal(goal.cpu().numpy(), v.goal)


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('scenario,n', FAMILIES, ids=FAMILY_IDS)
def test_step_store_paths_agree_and_match_the_oracle(scenario, n, precision):
    """Three identically seeded envs step into (a) fresh allocations, (b) 16 B-aligned caller buffers, (c) caller
    buffers one element off that alignment: the same computation through the TMA, coalesced-copy / direct-store and
    ragged-warp paths must give the same bits, and (a) must match the float64 oracle."""
    _assert_geometry(scenario, n)
    envs = [_mk(scenario, n, precision) for _ in range(3)]
    for e in envs:
        e.reset()
    pos, vel, lm, goal = envs[0].get_state()
    pos = pos * 0.35                               # crowd the agents so that contacts happen
    for e in envs:
        e.set_state(pos, vel, lm, goal)
    assert _same_state(envs[0], envs[1]) and _same_state(envs[0], envs[2])
    v = _make_oracle(scenario, n, envs[0].get_state())
    outs = [_Outputs(e, kind) for e, kind in zip(envs, ('default', 'aligned', 'offset'))]
    rng = np.random.RandomState(n or 0)
    T = 8 if scenario == TR else 10
    respawns = [0, 0]
    for t in range(T):
        act, ac = _actions(envs[0], rng)
        if precision == 'fp32':
            _sync_oracle(v, scenario, envs[0].get_state())
        for e, o in zip(envs, outs):
            o.refill()
            _step(e, act, ac, None, o)
        for o in outs[1:]:
            o.check(t)
        a = outs[0].t
        for o in outs[1:]:
            for k in OUTPUTS:
                if k == 'info_f' and scenario == TR:
                    continue
                assert _same(a[k], o.t[k]), (t, o.kind, k)
        assert not bool(a['done'].any())
        state = envs[0].get_state()
        for e in envs[1:]:
            assert all(_same(x, y) for x, y in zip(state, e.get_state())), t
        _check_step_against_oracle(scenario, precision, v, act, ac, a, state, respawns)
    if scenario == TR:                             # respawn draws keyed by ids on both sides of 2^32
        assert respawns[0] > 100 and respawns[1] > 100, respawns


_SUBSETS = [('obs',), ('rew',), ('done',), ('info_i', 'info_f'), ()]


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('scenario,n', FAMILIES, ids=FAMILY_IDS)
def test_null_output_subsets(scenario, n, precision):
    """mpe_step with each output alone and with none: what is produced equals an all-outputs call on a twin env, and
    the state afterwards is the same bits, also after a call that produces nothing."""
    env, twin = _mk(scenario, n, precision), _mk(scenario, n, precision)
    env.reset(); twin.reset()
    rng = np.random.RandomState(7)
    for names in _SUBSETS:
        act, ac = _actions(env, rng)
        part = _Outputs(env, 'aligned', names)
        part.refill()
        full = _Outputs(twin, 'default')
        _step(env, act, ac, None, part)
        _step(twin, act, ac, None, full)
        part.check(names)
        for k in names:
            if not (k == 'info_f' and scenario == TR):
                assert _same(part.t[k], full.t[k]), (names, k)
        assert _same_state(env, twin), names


def _expect_reset(scenario, n, precision, ep):
    """Philox reset of every env at its own episode index -> (pos, lm, goal[B, N]) as get_state returns them."""
    gid = np.arange(B, dtype=np.uint64) + np.uint64(OFF)
    if scenario == TR:
        a, t, ty = philox.treasure_reset(SEED, gid, ep)
        if precision == 'fp32':
            t = (t / 0.95).astype(np.float32) * np.float32(0.95)
        goal = -np.ones((B, 8), dtype=np.int64)
        goal[:, 0] = (ty << np.arange(6)).sum(axis=1) | (0x3F << 6)   # every treasure alive, nobody holds
        return a, t.astype(np.float64), goal
    spec = mpe_vec.Spec(scenario, n)
    want = philox.reset_positions(SEED, gid, ep, spec.N + spec.L)
    goal = -np.ones((B, spec.N), dtype=np.int64)
    if scenario == 'simple_reference':
        goal = philox.reset_goals(SEED, gid, ep, 2, 3)
    elif scenario == 'simple_speaker_listener':
        goal[:, 0] = philox.reset_goals(SEED, gid, ep, 1, 3)[:, 0]
    return want[:, :spec.N], want[:, spec.N:], goal


def _check_reset_obs(scenario, n, precision, state, obs, comm):
    """obs of EVERY row against the oracle's observation of the state the reset left (reset rows and loaded rows)."""
    pos, vel, lm, goal = (x.cpu().numpy() for x in state)
    o_dev = _np(obs)
    tol = F64_ATOL if precision == 'fp64' else 1e-6
    if scenario == TR:
        v = maac_vec.VecTreasure(B)
        v.set_state(pos, vel, lm, goal[:, 0])
        o = v.observe()
        ok = np.ones(B, dtype=bool) if precision == 'fp64' else ~_near_threshold(v.pos, _dead_apart(v.tr), F32_BAND)
        assert ok.mean() > 0.95, ok.mean()
        far = np.abs(o) > 100
        assert np.abs(o_dev - o)[ok][~far[ok]].max() <= tol
        assert not far[ok].any() or np.abs(o_dev - o)[ok][far[ok]].max() <= (tol if precision == 'fp64' else 1e-4)
        return
    v = mpe_vec.VecEnv(mpe_vec.Spec(scenario, n), B)
    v.set_state(pos, vel, lm, goal)
    if comm is not None:
        v.comm = comm
    assert np.abs(o_dev - v.observe()).max() <= tol


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('scenario,n', FAMILIES, ids=FAMILY_IDS)
def test_masked_resets_and_observe_into_caller_buffers(scenario, n, precision):
    """full reset, step, masked reset, step, masked reset: reset envs get the Philox draws of their own episode index,
    the others keep their state bits, every observation row matches the oracle, mpe_observe into a misaligned buffer
    repeats it, and the read-back statistics hold exactly the episodes each reset ended."""
    from multiagent_rl_b200 import _lib
    env = _mk(scenario, n, precision)
    env.track_returns(True)
    obs = env.reset()
    ep = np.zeros(B, dtype=np.int64)               # episode index of the first full reset
    p, l, g = _expect_reset(scenario, n, precision, ep)
    state = env.get_state()
    assert np.array_equal(_np(state[0]), p) and np.array_equal(_np(state[2]), l) and not state[1].any()
    assert np.array_equal(state[3].cpu().numpy(), g)
    _check_reset_obs(scenario, n, precision, state, obs, None)
    assert env.read_stats(clear=True)[2] == 0      # no episode had begun
    rng = np.random.RandomState(11)
    epw = _envs_per_warp(scenario, n)
    ret = np.zeros(B)
    tlen = np.zeros(B, dtype=np.int64)
    comm = None
    for k in range(2):
        act, ac = _actions(env, rng)
        _, rew, _, _ = env.step_tensor(act, ac)
        ret += _np(rew).sum(axis=1)
        tlen += 1
        if scenario == 'simple_reference':          # the messages the loaded rows observe
            comm = np.eye(10)[ac.cpu().numpy()]
        mask = (rng.rand(B) < 0.5).astype(np.uint8)
        mask[B // epw * epw] = 1 - k                # the ragged last warp: its first env reset in one call only
        spans = mask[:B // epw * epw].reshape(-1, epw).sum(axis=1)
        assert ((spans > 0) & (spans < epw)).mean() > 0.25      # reset and kept envs share warps
        before = [x.clone() for x in env.get_state()]
        out = _Guarded((B, env.n, env.obs_dim), env.dtype, NAN, 1)
        m = torch.from_numpy(mask).cuda()
        _lib.check(env._lib.mpe_reset(env._h, _lib.ptr(m), _lib.ptr(out.t), env._stream()), 'mpe_reset')
        out.check(('reset', k))
        after = env.get_state()
        sel = mask.astype(bool)
        keep = torch.from_numpy(~sel).cuda()
        for x, y in zip(before, after):
            assert _same(x[keep], y[keep]), k
        ep += mask
        p, l, g = _expect_reset(scenario, n, precision, ep)
        assert np.array_equal(_np(after[0])[sel], p[sel]) and np.array_equal(_np(after[2])[sel], l[sel])
        assert not after[1][~keep].any() and np.array_equal(after[3].cpu().numpy()[sel], g[sel])
        if comm is not None:
            comm[sel] = 0.0
        _check_reset_obs(scenario, n, precision, after, out.t, comm)
        again = _Guarded((B, env.n, env.obs_dim), env.dtype, NAN, 1)
        _lib.check(env._lib.mpe_observe(env._h, _lib.ptr(again.t), env._stream()), 'mpe_observe')
        again.check(('observe', k))
        assert _same(again.t, out.t)
        s = env.read_stats(clear=True)
        assert s[2] == sel.sum() and s[3] == tlen[sel].sum() and s[4] == 0, (k, s, sel.sum(), tlen[sel].sum())
        rtol = 1e-12 if precision == 'fp64' else 1e-5
        assert abs(s[0] - ret[sel].sum()) <= rtol * np.abs(ret[sel]).sum(), (k, s[0], ret[sel].sum())
        ret[sel] = 0.0
        tlen[sel] = 0
    assert (ep == 2).any() and (ep == 0).any()


@pytest.mark.parametrize('precision', PRECISIONS)
def test_real_valued_messages(precision):
    """simple_reference with real-valued messages comm_vec ~ U[-2, 2] (the one-env list surface sends these): against
    the oracle over an episode, the message part of each observation is the other agent's message exactly, and a
    comm_vec passed together with act_c wins over it."""
    env, twin = _mk('simple_reference', None, precision), _mk('simple_reference', None, precision)
    env.reset(); twin.reset()
    v = mpe_vec.VecEnv(mpe_vec.Spec('simple_reference'), B)
    v.set_state(*(x.cpu().numpy() for x in env.get_state()))
    rng = np.random.RandomState(3)
    real = np.float32 if precision == 'fp32' else np.float64
    for t in range(25):
        act = rng.randint(0, 5, (B, 2)).astype(np.int32)
        ac = rng.randint(0, 10, (B, 2)).astype(np.int32)
        cv = rng.uniform(-2, 2, (B, 2, 10)).astype(real).astype(np.float64)
        obs, rew, _, _ = env.step_tensor(act, ac, comm_vec=cv)
        obs2, rew2, _, _ = twin.step_tensor(act, None, comm_vec=cv)
        assert _same(obs, obs2) and _same(rew, rew2), t
        o, r, _ = v.step(act, act_c=ac, comm_vec=cv)
        od = _np(obs)
        assert np.array_equal(od[:, 0, 11:], cv[:, 1]) and np.array_equal(od[:, 1, 11:], cv[:, 0]), t
        if precision == 'fp64':
            assert np.abs(od - o).max() <= F64_ATOL and np.abs(_np(rew) - r).max() <= F64_ATOL, t
        else:                                      # test_gpu_env.py's fp32 tolerances over an episode
            assert np.abs(od - o).max() <= 5e-5 and np.abs(_np(rew) - r).max() <= 2e-4, t
    assert _same_state(env, twin)


def test_out_is_validated():
    """step_tensor / step_host refuse an `out` buffer of the wrong shape, dtype, layout or memory before any launch:
    the kernels would write B*N*D elements through its pointer whatever it is."""
    env = _mk('simple_spread', None, 'fp32')
    env.reset()
    N, D = env.n, env.obs_dim
    act = np.random.RandomState(0).randint(0, 5, (B, N)).astype(np.int32)
    before = [x.clone() for x in env.get_state()]
    steps = env.global_step

    def dev():
        return (torch.full((B, N, D), NAN, device='cuda'), torch.full((B, N), NAN, device='cuda'),
                torch.full((B, N), DONE_FILL, dtype=torch.uint8, device='cuda'))

    def host():
        return (np.full((B, N, D), np.nan, np.float32), np.full((B, N), np.nan, np.float32),
                np.full((B, N), DONE_FILL, np.uint8))

    def bad(good, i, x):
        o = list(good)
        o[i] = x
        return tuple(o)

    d, h = dev(), host()
    dev_cases = [bad(d, 0, torch.empty((B, N, D + 1), device='cuda')),                    # shape
                 bad(d, 1, torch.empty((B * N,), device='cuda')),
                 bad(d, 1, torch.empty((B, N), dtype=torch.float64, device='cuda')),      # dtype
                 bad(d, 2, torch.empty((B, N), dtype=torch.bool, device='cuda')),
                 bad(d, 0, torch.empty((B, D, N), device='cuda').transpose(1, 2)),        # not contiguous
                 bad(d, 1, torch.empty((B, 2 * N), device='cuda')[:, ::2]),
                 bad(d, 0, torch.empty((B, N, D))),                                       # host tensor
                 (d[0], d[1])]
    host_cases = [bad(h, 0, np.empty((B, N, D - 1), np.float32)),
                  bad(h, 1, np.empty((B, N), np.float64)),
                  bad(h, 2, np.empty((B, N), np.int32)),
                  bad(h, 0, np.empty((B, D, N), np.float32).transpose(0, 2, 1)),
                  bad(h, 1, torch.empty((B, N), device='cuda')),                          # device tensor
                  bad(h, 2, torch.empty((B, N), dtype=torch.uint8, device='cuda'))]
    for out in dev_cases:
        with pytest.raises(ValueError):
            env.step_tensor(torch.from_numpy(act).cuda(), out=out)
    for out in host_cases:
        with pytest.raises(ValueError):
            env.step_host(act, out=out)
    torch.cuda.synchronize()
    assert all(_same(x, y) for x, y in zip(before, env.get_state())) and env.global_step == steps
    assert bool(torch.isnan(d[0]).all() and torch.isnan(d[1]).all() and (d[2] == DONE_FILL).all())
    assert np.isnan(h[0]).all() and np.isnan(h[1]).all() and (h[2] == DONE_FILL).all()
    # None skips an output; well-formed buffers are written in place, on both surfaces
    obs, rew, done, _ = env.step_tensor(torch.from_numpy(act).cuda(), out=(None, d[1], d[2]))
    assert obs is None and rew is d[1] and not bool(torch.isnan(d[1]).any()) and not bool(d[2].any())
    twin = _mk('simple_spread', None, 'fp32')
    twin.reset()
    twin.set_state(*before)
    ho, hr, hd = twin.step_host(act, out=h)
    assert ho is h[0] and np.array_equal(hr, d[1].cpu().numpy()) and not hd.any() and not np.isnan(ho).any()
