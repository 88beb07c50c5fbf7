"""env.rollout(..., info=True): upstream's benchmark_data of every env-step, recorded by the rollout itself (the fused
k_tc2 kernel for teams of 2 / 3 on the tensor cores, the per-step kernels otherwise), bit for bit what
env.step(info=True) returns for the same step, and without changing anything else the rollout computes."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import actor_ref, mpe_vec
from tests.test_gpu_env import _flags_differ_only_at_the_threshold

pytestmark = pytest.mark.gpu

TR = 'fullobs_collect_treasure'
TC_TEAMS = (2, 3, 4, 6, 8, 9, 12)
GUARD = 4099  # elements past [T][B] that must stay untouched


def _N(scenario, n):
    return {'simple_reference': 2, 'simple_speaker_listener': 2, TR: 8}.get(scenario, n or 3)


def _actor(env, impl, seed, scale=3.0):
    import multiagent_rl_b200 as m
    heads = [5, env.act_c] if env.act_c else 5
    sd = actor_ref.init_state_dict(env.obs_dim, heads, 9)
    for k in sd:
        if 'dense2' in k:
            sd[k] = sd[k] * scale
    return m.FusedActor(sd, seed=seed, impl=impl)


def _envs(scenario, n, B, k, **kw):
    import multiagent_rl_b200 as m
    return [m.make_env(scenario, n=n, num_envs=B, batched=True, **kw) for _ in range(k)]


def _same(a, b):
    return (a is None and b is None) or torch.equal(a, b)


def _check_stepwise(step, obs, actor, rec, info, T, L, step0, seed, gid0=0, treasure=False):
    """rec / info of a rollout from the state `step` starts in (observation `obs`) == actor.forward +
    env.step(info=True) + reset."""
    for t in range(T):
        out = actor.forward(obs, step=step0 + t, seed=seed, env_id_offset=gid0)
        assert torch.equal(out['act_u'], rec[2][t]), t
        if out['act_c'] is not None:
            assert torch.equal(out['act_c'], rec[3][t]), t
        obs, rew, _, inf = step.step(out['act_u'], out['act_c'], info=True)
        assert torch.equal(obs, rec[0][t]) and torch.equal(rew, rec[1][t]), t
        assert torch.equal(inf['info_i'], info['info_i'][t]), t
        if not treasure:
            assert torch.equal(inf['info_f'], info['info_f'][t]), t
        if (t + 1) % L == 0:
            obs = step.reset()


# the matrix of tests/test_gpu_actor.py::test_fused_rollout_equals_stepwise_path, plus fullobs_collect_treasure
CASES = [('simple_spread', None, 10_000 + 13), ('simple_spread', 6, 2000), ('simple_spread', 9, 1000),
         ('simple_spread', 12, 500), ('simple_reference', None, 3000), ('simple_speaker_listener', None, 3000),
         ('simple_spread', 2, 3001), ('simple_spread', 4, 2000), ('simple_spread', 8, 1000), (TR, None, 1000)]


@pytest.mark.parametrize('impl', ['simt', 'tc'])
@pytest.mark.parametrize('scenario,n,B', CASES)
def test_rollout_info_equals_stepwise_path(scenario, n, B, impl):
    """T = 30, episodes of 7 steps, step0 = 100: info_i / info_f of rollout(info=True, record=True) equal
    env.step(info=True) step by step, and the recordings equal those of a rollout without info on a twin env."""
    T, seed, L, step0 = 30, 2024, 7, 100
    if impl == 'tc' and _N(scenario, n) not in TC_TEAMS:
        pytest.skip('not covered by the tensor-core path')
    env, twin, step = _envs(scenario, n, B, 3, seed=seed, max_episode_len=L)
    actor = _actor(env, impl, seed)
    env.reset(); twin.reset()
    obs = step.reset()
    *rec, info = env.rollout(actor, T, step0=step0, record=True, info=True)
    want = twin.rollout(actor, T, step0=step0, record=True)
    assert all(_same(a, b) for a, b in zip(rec, want))
    N = env.n
    assert info['info_i'].shape == (T, B, N + 1) and info['info_i'].dtype == torch.int32
    if scenario == TR:
        assert info['info_f'] is None
        assert bool((info['info_i'][..., N] == 0).all()) and bool(((info['info_i'] == 0) | (info['info_i'] == 1)).all())
    else:
        assert info['info_f'].shape == (T, B) and info['info_f'].dtype == torch.float32
    if scenario in ('simple_reference', 'simple_speaker_listener'):
        assert int(info['info_i'].abs().max()) == 0 and float(info['info_f'].abs().max()) == 0.0
    _check_stepwise(step, obs, actor, rec, info, T, L, step0, seed, treasure=scenario == TR)
    for a, b, c in zip(env.get_state(), twin.get_state(), step.get_state()):
        assert torch.equal(a, b) and torch.equal(a, c)
    s1, s0 = env.read_stats(), twin.read_stats()
    assert s1[2] == s0[2] and s1[3] == s0[3]


def _prefilled(T, B, N, offset_elems, dev):
    """info_i (-1) / info_f (NaN) views of [T][B] entries starting `offset_elems` elements into a larger buffer, with
    GUARD sentinel elements after them."""
    ii = torch.full((offset_elems + T * B * (N + 1) + GUARD,), -1, dtype=torch.int32, device=dev)
    fi = torch.full((offset_elems + T * B + GUARD,), float('nan'), dtype=torch.float32, device=dev)
    return ii, fi, ii[offset_elems:offset_elems + T * B * (N + 1)].view(T, B, N + 1), \
        fi[offset_elems:offset_elems + T * B].view(T, B)


def _c_rollout(env, actor, T, step0, rec, ii, fi):
    from multiagent_rl_b200 import _lib
    lib = _lib.load()
    rc = lib.mpe_rollout(env._h, actor._h, T, C.c_uint64(step0), *[_lib.ptr(x) for x in rec], _lib.ptr(ii),
                         _lib.ptr(fi), _lib.current_stream(env.device))
    _lib.check(rc, 'mpe_rollout')
    env.global_step = step0 + T


@pytest.mark.parametrize('scenario,n', [('simple_spread', 2), ('simple_spread', None), ('simple_reference', None),
                                        ('simple_speaker_listener', None)])
def test_fused_rollout_info_past_the_first_wave(scenario, n):
    """The fused kernels at B = 6 * SMs * 128 + 77 (every CTA walks several tile pairs and ends on a ragged one), 9 steps
    with episodes of 4, into caller buffers pre-filled with -1 / NaN, once aligned and once at a 4-byte offset: every
    entry of [T][B] is written, nothing after it, and the values equal the stepwise calls."""
    dev = torch.device('cuda', torch.cuda.current_device())
    nsm = torch.cuda.get_device_properties(dev).multi_processor_count
    B, T, L, step0, seed, gid0 = 6 * nsm * 128 + 77, 9, 4, 100, 2 ** 40 + 9, 2 ** 32 - 5000
    ntiles = -(-B // 128)
    assert (ntiles + 1) // 2 // nsm >= 3 and ntiles % 2 == 1
    for offset in (0, 1):
        env, twin, step = _envs(scenario, n, B, 3, seed=seed, max_episode_len=L, env_id_offset=gid0)
        actor = _actor(env, 'tc', seed)
        env.reset(); twin.reset()
        obs = step.reset()
        N = env.n
        rec = [torch.empty(T, B, N, env.obs_dim, device=dev), torch.empty(T, B, N, device=dev),
               torch.empty(T, B, N, dtype=torch.int32, device=dev),
               torch.empty(T, B, N, dtype=torch.int32, device=dev) if env.act_c else None]
        ii_all, fi_all, ii, fi = _prefilled(T, B, N, offset, dev)
        _c_rollout(env, actor, T, step0, rec, ii, fi)
        assert (ii.data_ptr() % 16 == 0) == (offset == 0)
        assert not bool((ii == -1).any()) and not bool(torch.isnan(fi).any())
        assert bool((ii_all[:offset] == -1).all()) and bool((ii_all[offset + ii.numel():] == -1).all())
        assert bool(torch.isnan(fi_all[:offset]).all()) and bool(torch.isnan(fi_all[offset + fi.numel():]).all())
        want = twin.rollout(actor, T, step0=step0, record=True)
        assert all(_same(a, b) for a, b in zip(rec, want))
        _check_stepwise(step, obs, actor, rec, {'info_i': ii, 'info_f': fi}, T, L, step0, seed, gid0)


def test_fused_rollout_info_vs_float64_oracle_directly():
    """A 25-step simple_spread N = 3 rollout of 65,536 envs replayed by oracle/mpe_vec.py with the recorded actions:
    collision counts and occupied landmarks equal except where a flag's float64 distance sits within the band the env's
    fp32 position error explains; the sum of min distances within what that error allows (each landmark's nearest
    distance moves by at most sqrt(2) x the largest coordinate error, plus fp32 rounding)."""
    import multiagent_rl_b200 as m
    B, T, seed = 65_536, 25, 4242
    spec = mpe_vec.Spec('simple_spread')
    env = m.make_env('simple_spread', num_envs=B, batched=True, seed=seed, max_episode_len=T)
    actor = m.FusedActor(actor_ref.init_state_dict(spec.obs_dim, 5, 17), seed=seed, impl='auto')
    env.reset()
    pos, vel, lm, goal = env.get_state()
    v = mpe_vec.VecEnv(spec, B)
    v.set_state(pos.cpu().numpy().astype(np.float64), vel.cpu().numpy().astype(np.float64),
                lm.cpu().numpy().astype(np.float64), goal.cpu().numpy())
    obs, _, act_u, _, info = env.rollout(actor, T, step0=0, record=True, info=True)
    obs, act_u = obs.cpu().numpy().astype(np.float64), act_u.cpu().numpy()
    ii, md = info['info_i'].cpu().numpy(), info['info_f'].cpu().numpy().astype(np.float64)
    lm0 = lm.cpu().numpy().astype(np.float64)
    for t in range(T):
        v.step(act_u[t])
        coll, occ = v.flags()
        pos32 = obs[t][:, :, 2:4]  # simple_spread observations carry the agent's own position after its velocity
        g = {'pos': {t: v.pos}, 'lm0': lm0, 'coll': {t: coll}, 'occ': {t: occ}}
        _flags_differ_only_at_the_threshold(ii[t], g, t, pos32)
        err = np.abs(pos32 - v.pos).max(axis=(1, 2))
        dmd = np.abs(md[t] - v.min_dists_sum())
        assert np.all(dmd <= spec.L * np.sqrt(2.0) * err + 1e-5), (t, dmd.max())
        assert dmd.max() <= 2e-4, (t, dmd.max())
    assert ii[..., :3].max() >= 2 and ii[..., 3].max() >= 1  # collisions and occupied landmarks do occur


def _ring_case(scenario, n, B, L, T, step0, record, warm=0, mask=None):
    """Three identical envs: rollout(replay=buf, info=True), rollout(replay=buf) and rollout(info=True); the first
    two rings must hold the same bytes, and the info of the first and the third must be equal."""
    import multiagent_rl_b200 as m
    seed = 7
    envs = _envs(scenario, n, B, 3, seed=seed, max_episode_len=L)
    e = envs[0]
    heads = [5, e.act_c] if e.act_c else 5
    actor = _actor(e, 'auto', seed, scale=1.0)
    bufs = [m.DeviceReplayBuffer(2 * B + 3, e.n, e.obs_dim, heads, seed=1) for _ in range(2)]
    for x in envs:
        x.reset()
        if warm:
            x.rollout(actor, warm, step0=0)
    if mask is not None:
        mt = torch.from_numpy(mask.astype(np.uint8)).cuda()
        for x in envs:
            x.reset(mask=mt)
    got = envs[0].rollout(actor, T, step0=step0, record=record, replay=bufs[0], info=True)
    plain = envs[1].rollout(actor, T, step0=step0, record=record, replay=bufs[1])
    ref = envs[2].rollout(actor, T, step0=step0, record=record, info=True)
    assert torch.equal(got[4]['info_i'], ref[4]['info_i']) and _same(got[4]['info_f'], ref[4]['info_f'])
    if record:
        assert all(_same(a, b) for a, b in zip(got[:4], plain))
        assert all(_same(a, b) for a, b in zip(got[:4], ref[:4]))
    assert len(bufs[0]) == len(bufs[1]) and bufs[0]._next_idx == bufs[1]._next_idx
    idx = torch.arange(len(bufs[0]), device='cuda')
    for a, b in zip(bufs[0].sample_index(idx), bufs[1].sample_index(idx)):
        assert torch.equal(a, b)
    for a, b, c in zip(*(x.get_state() for x in envs)):
        assert torch.equal(a, b) and torch.equal(a, c)
    return got[4]


def test_ring_fused_segments_across_an_episode_end_and_the_scratch_budget():
    """Synced envs, no recordings: at 400,000 envs of simple_spread N = 3 the 1 GiB scratch holds 18 steps, so T = 30
    from the episode start runs as segments of 18, 7 (episode end) and 5 steps, each writing its own rows of info."""
    info = _ring_case('simple_spread', None, 400_000, 25, 30, 0, record=False)
    assert bool((info['info_i'][..., :3] >= 1).all())  # every agent collides with itself: every row was written


@pytest.mark.parametrize('scenario,n', [('simple_spread', None), ('simple_reference', None), ('simple_spread', 6)])
def test_ring_fused_segments_with_recordings(scenario, n):
    _ring_case(scenario, n, 300, 7, 19, 11, record=True, warm=3)


@pytest.mark.parametrize('scenario,n', [('simple_spread', None), ('simple_speaker_listener', None),
                                        ('simple_spread', 9)])
def test_ring_per_step_path_after_a_masked_reset(scenario, n):
    mask = np.random.RandomState(4).rand(300) < 0.4
    _ring_case(scenario, n, 300, 7, 19, 50, record=True, warm=3, mask=mask)


def test_contract_details():
    """info=False returns what it always did; fp64 envs still refuse; on fullobs_collect_treasure info_f is None and
    a caller's info_f buffer is left as it was; info=True without record gives None for the recordings."""
    import multiagent_rl_b200 as m
    B, T = 257, 5
    env = m.make_env('simple_spread', num_envs=B, batched=True, seed=1, max_episode_len=7)
    actor = _actor(env, 'auto', 1)
    env.reset()
    assert env.rollout(actor, T) is None
    r = env.rollout(actor, T, record=True)
    assert isinstance(r, tuple) and len(r) == 4 and r[3] is None
    r = env.rollout(actor, T, info=True)
    assert isinstance(r, tuple) and len(r) == 5 and r[:4] == (None, None, None, None)
    assert set(r[4]) == {'info_i', 'info_f'} and r[4]['info_i'].shape == (T, B, 4) and r[4]['info_f'].shape == (T, B)
    f64 = m.make_env('simple_spread', num_envs=B, batched=True, seed=1, precision='fp64')
    f64.reset()
    with pytest.raises(RuntimeError):
        f64.rollout(actor, T, info=True)
    tr = m.make_env(TR, num_envs=B, batched=True, seed=1, max_episode_len=7)
    ta = _actor(tr, 'auto', 1)
    tr.reset()
    *_, info = tr.rollout(ta, T, info=True)
    assert info['info_f'] is None and info['info_i'].shape == (T, B, 9)
    dev = torch.device('cuda', torch.cuda.current_device())
    _, fi_all, ii, fi = _prefilled(T, B, 8, 0, dev)
    _c_rollout(tr, ta, T, 0, [None] * 4, ii, fi)
    assert not bool((ii == -1).any()) and bool(torch.isnan(fi_all).all())
