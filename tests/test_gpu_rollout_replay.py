"""env.rollout(..., replay=buf): every env-step's transition goes to the device ring, bit-identical to the stepwise
loop built from public calls (actor.forward -> env.step -> buf.add -> reset of the envs whose episode ended), on the
fused path (synced envs, teams of 2 / 3 on the tensor cores) and the per-step path (everything else)."""
import numpy as np
import pytest
import torch

from oracle import actor_ref

pytestmark = pytest.mark.gpu

TEAMS = [('simple_spread', n) for n in range(1, 13)] + [('simple_reference', None), ('simple_speaker_listener', None),
                                                         ('fullobs_collect_treasure', None)]
TC_TEAMS = (2, 3, 4, 6, 8, 9, 12)


def _teams_impls():
    out = []
    for scenario, n in TEAMS:
        N = {'simple_reference': 2, 'simple_speaker_listener': 2, 'fullobs_collect_treasure': 8}.get(scenario, n)
        out.append((scenario, n, 'simt'))
        if N in TC_TEAMS:
            out.append((scenario, n, 'auto'))
    return out


class _Case(object):
    """Three identical envs: `env` runs rollout(replay=buf), `plain` rollout without a ring, `ref` the stepwise loop
    into `ref_buf`.  `tstep` is the host's view of every env's episode step (for the reference's resets)."""

    def __init__(self, scenario, n, impl, B, L, cap, seed=7, gid0=0, warm=0, mask=None, prefill=0):
        import multiagent_rl_b200 as m
        self.L, self.seed, self.gid0, self.B = L, seed, gid0, B
        mk = lambda: m.make_env(scenario, n=n, num_envs=B, batched=True, seed=seed, max_episode_len=L,  # noqa: E731
                                env_id_offset=gid0)
        self.env, self.plain, self.ref = mk(), mk(), mk()
        e = self.env
        heads = [5, e.act_c] if e.act_c else 5
        self.actor = m.FusedActor(actor_ref.init_state_dict(e.obs_dim, heads, 5), seed=seed, impl=impl)
        self.buf = m.DeviceReplayBuffer(cap, e.n, e.obs_dim, heads, seed=1)
        self.ref_buf = m.DeviceReplayBuffer(cap, e.n, e.obs_dim, heads, seed=1)
        self.tstep = np.zeros(B, np.int64)
        for x in (self.env, self.plain, self.ref):
            x.reset()
            if warm:
                x.rollout(self.actor, warm, step0=0)
        self.tstep[:] = warm % L
        if mask is not None:
            mt = torch.from_numpy(mask.astype(np.uint8)).cuda()
            for x in (self.env, self.plain, self.ref):
                x.reset(mask=mt)
            self.tstep[mask] = 0
        if prefill:  # the call starts at a ring position other than 0
            g = torch.Generator(device='cuda').manual_seed(3)
            o = torch.randn(prefill, e.n, e.obs_dim, device='cuda', generator=g)
            a = torch.randint(0, 5, (prefill, e.n), device='cuda', generator=g)
            ac = torch.randint(0, max(e.act_c, 1), (prefill, e.n), device='cuda', generator=g) if e.act_c else None
            for b in (self.buf, self.ref_buf):
                b.add(o, a, o[:, :, 0], o * 2, act_c=ac)

    def run(self, T, step0, record=True):
        got = self.env.rollout(self.actor, T, step0=step0, record=record, replay=self.buf)
        want = self.plain.rollout(self.actor, T, step0=step0, record=record)
        obs = self.ref.observe()
        for t in range(T):
            out = self.actor.forward(obs, step=step0 + t, env_id_offset=self.gid0, seed=self.seed)
            nxt, rew, _, _ = self.ref.step(out['act_u'], out['act_c'])
            self.ref_buf.add(obs, out['act_u'], rew, nxt, act_c=out['act_c'])
            self.tstep += 1
            ended = self.tstep >= self.L
            if ended.any():
                obs = self.ref.reset(mask=torch.from_numpy(ended.astype(np.uint8)).cuda())
                self.tstep[ended] = 0
            else:
                obs = nxt
        return got, want

    def check(self, got, want):
        assert len(self.buf) == len(self.ref_buf) and self.buf._next_idx == self.ref_buf._next_idx
        idx = torch.arange(len(self.buf), device='cuda')
        for a, b in zip(self.buf.sample_index(idx), self.ref_buf.sample_index(idx)):
            assert torch.equal(a, b)
        for a, b, c in zip(self.env.get_state(), self.plain.get_state(), self.ref.get_state()):
            assert torch.equal(a, b) and torch.equal(a, c)
        s1, s0 = self.env.read_stats(), self.plain.read_stats()
        assert s1[2] == s0[2] and s1[3] == s0[3] and s1[4] == s0[4]
        assert np.allclose(s1[:2], s0[:2], rtol=1e-12, atol=0)  # double atomics: summation order may differ
        if got is not None:
            for a, b in zip(got, want):
                assert (a is None and b is None) or torch.equal(a, b)


@pytest.mark.parametrize('scenario,n,impl', _teams_impls())
def test_every_team_mid_episode_long_call(scenario, n, impl):
    """T = 2L + 5 starting mid-episode (episode step 3, step0 unrelated to it): several in-call resets, and the ring
    starts at a position other than 0."""
    c = _Case(scenario, n, impl, B=300, L=7, cap=300 * 40, warm=3, prefill=77)
    c.check(*c.run(19, step0=11))
    c.check(*c.run(5, step0=30, record=False))  # a second call continues the episodes where the first left them


@pytest.mark.parametrize('T', [3, 7])
@pytest.mark.parametrize('scenario,n,impl', [('simple_spread', None, 'auto'), ('simple_spread', None, 'simt'),
                                             ('simple_reference', None, 'auto'), ('simple_spread', 6, 'auto'),
                                             ('fullobs_collect_treasure', None, 'auto')])
def test_short_and_one_episode_calls(scenario, n, impl, T):
    c = _Case(scenario, n, impl, B=257, L=7, cap=257 * 20)
    c.check(*c.run(T, step0=0))
    c.check(*c.run(T, step0=T))


@pytest.mark.parametrize('scenario,n,impl', [('simple_spread', None, 'auto'), ('simple_spread', 2, 'simt'),
                                             ('simple_reference', None, 'auto'), ('simple_speaker_listener', None, 'auto'),
                                             ('simple_spread', 9, 'auto')])
def test_envs_unsynced_by_a_masked_reset(scenario, n, impl):
    """Not fullobs_collect_treasure: on envs whose episodes are not aligned the rollout re-emits every env's
    observation after each step, and a treasure env's observation after post_step (pick-up / respawn) is not the one
    its step returned, so the rollout itself already differs from the stepwise loop there."""
    mask = np.random.RandomState(4).rand(300) < 0.4
    c = _Case(scenario, n, impl, B=300, L=7, cap=300 * 40, warm=3, mask=mask)
    c.check(*c.run(19, step0=50))


@pytest.mark.parametrize('record', [True, False])
@pytest.mark.parametrize('scenario,n,impl', [('simple_spread', None, 'auto'), ('simple_spread', None, 'simt'),
                                             ('simple_reference', None, 'auto'), ('simple_spread', 6, 'auto')])
def test_call_wraps_the_ring_several_times(scenario, n, impl, record):
    """T * B = 2,451 transitions into 500 slots (not a multiple of B): only the last 500 survive, as with adds."""
    c = _Case(scenario, n, impl, B=129, L=7, cap=500, warm=2, prefill=31)
    c.check(*c.run(19, step0=4, record=record))


@pytest.mark.parametrize('scenario,n,impl', [('simple_spread', None, 'auto'), ('simple_reference', None, 'auto'),
                                             ('simple_spread', 4, 'auto')])
def test_ragged_batches(scenario, n, impl):
    """1 env, 129 envs (a tile pair whose second tile has one row), and one env past the first wave of k_tc2's
    tile pairs (two tiles of 128 envs per SM)."""
    nsm = torch.cuda.get_device_properties(0).multi_processor_count
    for B in (1, 129, nsm * 256 + 1):
        c = _Case(scenario, n, impl, B=B, L=5, cap=B * 13 + 3, warm=1)
        c.check(*c.run(12, step0=2))


@pytest.mark.parametrize('scenario,n,impl', [('simple_spread', None, 'auto'), ('simple_spread', 6, 'auto'),
                                             ('simple_reference', None, 'simt')])
def test_64_bit_seed_and_env_ids_across_2_to_the_32(scenario, n, impl):
    c = _Case(scenario, n, impl, B=300, L=7, cap=300 * 20, seed=(1 << 63) + 12345, gid0=(1 << 32) - 100)
    c.check(*c.run(10, step0=(1 << 33) + 1))


def test_scratch_budget_splits_an_episode():
    """Without recordings the fused path keeps one segment's recordings in a 1 GiB scratch: at 400,000 envs of
    simple_spread N = 3 (144 B per env-step) an episode of 25 steps runs as 18 + 7 steps, and step 18's obs_t is the
    last observation of the first segment."""
    B = 400_000
    c = _Case('simple_spread', None, 'auto', B=B, L=25, cap=B * 8)
    c.check(*c.run(25, step0=0, record=False))


def test_transitions_chain_and_open_episodes_with_the_reset_observation():
    """Inside an episode obs_next of step t is obs of step t + 1; at an episode's first step obs is the env's
    post-reset observation (episode k of an env = its (k + 1)-th reset)."""
    import multiagent_rl_b200 as m
    B, L, T, seed = 200, 7, 19, 21
    env = m.make_env('simple_spread', num_envs=B, batched=True, seed=seed, max_episode_len=L)
    actor = m.FusedActor(actor_ref.init_state_dict(env.obs_dim, 5, 2), seed=seed)
    buf = m.DeviceReplayBuffer(B * T, env.n, env.obs_dim, 5)
    first = env.reset()
    env.rollout(actor, T, step0=0, replay=buf)
    s0, _, _, s1, d = buf.sample_index(torch.arange(B * T, device='cuda'))
    s0, s1 = s0.view(T, B, env.n, -1), s1.view(T, B, env.n, -1)
    assert float(d.abs().max()) == 0.0
    fresh = m.make_env('simple_spread', num_envs=B, batched=True, seed=seed, max_episode_len=L)
    resets = [fresh.reset() for _ in range(T // L + 1)]
    assert torch.equal(s0[0], first) and torch.equal(s0[0], resets[0])
    for t in range(T - 1):
        if (t + 1) % L == 0:
            assert torch.equal(s0[t + 1], resets[(t + 1) // L]), t
            assert not torch.equal(s0[t + 1], s1[t]), t
        else:
            assert torch.equal(s0[t + 1], s1[t]), t


def test_refused_calls_leave_the_ring_and_the_env_unchanged():
    import multiagent_rl_b200 as m
    from multiagent_rl_b200 import _lib
    B = 64
    mk = lambda: m.make_env('simple_spread', num_envs=B, batched=True, seed=1, max_episode_len=7)  # noqa: E731
    env, twin = mk(), mk()
    actor = m.FusedActor(actor_ref.init_state_dict(env.obs_dim, 5, 2), seed=1)
    good, twin_buf = m.DeviceReplayBuffer(1000, 3, 10, 5), m.DeviceReplayBuffer(1000, 3, 10, 5)
    for e, b in ((env, good), (twin, twin_buf)):
        e.reset()
        e.rollout(actor, 2, step0=0, replay=b)
    idx = torch.arange(len(good), device='cuda')
    before = [x.clone() for x in good.sample_index(idx)], len(good), good._next_idx
    state0, stats0, gstep0 = env.get_state(), env.read_stats(), env.global_step
    bad = [m.DeviceReplayBuffer(1000, 4, 10, 5), m.DeviceReplayBuffer(1000, 3, 12, 5),
           m.DeviceReplayBuffer(1000, 3, 10, [5, 10]), m.DeviceReplayBuffer(1000, 3, 10, 6),
           m.DeviceReplayBuffer(B - 1, 3, 10, 5)]
    for rb in bad:
        n0 = rb._next_idx
        with pytest.raises(ValueError):
            env.rollout(actor, 3, replay=rb)
        # the C entry point refuses them as well, before any launch
        rc = _lib.load().mpe_rollout_replay(env._h, actor._h, rb._h, 3, 0, None, None, None, None,
                                            _lib.current_stream(env.device))
        assert rc == _lib.MPE_EINVAL and len(rb) == 0 and rb._next_idx == n0
    with pytest.raises(ValueError):
        env.rollout(actor, 3, replay=object())
    f64 = m.make_env('simple_spread', num_envs=B, batched=True, seed=1, precision='fp64')
    f64.reset()
    with pytest.raises(RuntimeError):
        f64.rollout(actor, 3, replay=good)
    rc = _lib.load().mpe_rollout_replay(f64._h, actor._h, good._h, 3, 0, None, None, None, None,
                                        _lib.current_stream(env.device))
    assert rc == _lib.MPE_EUNSUPPORTED
    if torch.cuda.device_count() > 1:
        other = m.DeviceReplayBuffer(1000, 3, 10, 5, device='cuda:1')
        with pytest.raises(ValueError):
            env.rollout(actor, 3, replay=other)
    after = good.sample_index(idx), len(good), good._next_idx
    assert after[1:] == before[1:] and all(torch.equal(a, b) for a, b in zip(after[0], before[0]))
    assert env.global_step == gstep0 and np.array_equal(env.read_stats(), stats0)
    assert all(torch.equal(a, b) for a, b in zip(env.get_state(), state0))
    # the episode counters did not move either: the next accepted call (across the episode end at step 7) gives the
    # transitions of a twin env that never saw the refused calls
    for e, b in ((env, good), (twin, twin_buf)):
        e.rollout(actor, 9, step0=2, replay=b)
    idx = torch.arange(len(good), device='cuda')
    assert len(good) == len(twin_buf) == 11 * B
    assert all(torch.equal(a, b) for a, b in zip(good.sample_index(idx), twin_buf.sample_index(idx)))
    assert all(torch.equal(a, b) for a, b in zip(env.get_state(), twin.get_state()))


def _kernels(fn):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.key for e in prof.key_averages() if e.device_time_total > 0]


def test_aligned_small_teams_take_the_fused_path():
    """The path is chosen from observable state: envs whose episodes are aligned with the tensor-core actor of a small
    team run k_tc2 and the multi-step ring writer (no per-step replay_add); after a masked reset the same envs run the
    per-step loop with one replay_add per step."""
    import multiagent_rl_b200 as m
    B, L = 300, 7
    env = m.make_env('simple_spread', num_envs=B, batched=True, seed=2, max_episode_len=L)
    actor = m.FusedActor(actor_ref.init_state_dict(env.obs_dim, 5, 2), seed=2)
    buf = m.DeviceReplayBuffer(B * 40, env.n, env.obs_dim, 5)
    env.reset()
    env.rollout(actor, 1, replay=buf)  # module loads outside the profiled calls
    names = _kernels(lambda: env.rollout(actor, 19, replay=buf))
    writer = [k for k in names if 'k_replay_add_steps' in k]
    adds = [k for k in names if 'k_replay_add' in k and 'k_replay_add_steps' not in k]
    assert writer and not adds and any('k_tc2' in k for k in names), names
    env.reset(mask=torch.ones(B, dtype=torch.uint8, device='cuda'))
    names = _kernels(lambda: env.rollout(actor, 5, replay=buf))
    writer = [k for k in names if 'k_replay_add_steps' in k]
    adds = [k for k in names if 'k_replay_add' in k and 'k_replay_add_steps' not in k]
    assert adds and not writer, names
