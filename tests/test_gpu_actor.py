"""GPU parity tests of the actor forward / sampling kernel and of the fused rollout kernel.

Tolerances: logits of the fp32 kernel vs the reference network's fp32 CPU logits (committed under
tests/golden/actor_*.npz) and vs the float64 oracle: 1e-5 absolute.  Sampled indices under injected
identical Gumbel noise are bit-exact except where the two best perturbed logits are closer than
1e-5 (the kernel and torch round differently there).
"""
import os

import numpy as np
import pytest
import torch

from oracle import actor_ref, mpe_vec, philox

pytestmark = pytest.mark.gpu

LOGIT_ATOL = 1e-5
GAP = 1e-5

TAGS = [('spread_n3', 3), ('spread_n12', 12), ('reference', 2), ('speaker', 2), ('model_n6', 6)]


def _load(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, 'actor_%s.npz' % tag))
    sd = {k[3:]: g[k] for k in g.files if k.startswith('sd/')}
    return g, sd


def _impls(N, model=False, wide=False):
    # tensor-core path: 2-3 agents (resident operands, fused env), 4/6/8/9/12 agents (just-in-time operands, single
    # head of <= 8 entries); the dense3 model head is one small kernel on the relu(hcat) the tensor-core forward emits
    if N in (2, 3) or (N in (4, 6, 8, 9, 12) and not wide):
        return ['simt', 'tc']
    return ['simt']


@pytest.mark.parametrize('impl', ['simt', 'tc'])
@pytest.mark.parametrize('tag,N', TAGS)
def test_actor_matches_reference_network(golden_dir, tag, N, impl):
    import multiagent_rl_b200 as m
    g, sd = _load(golden_dir, tag)
    if impl not in _impls(N, 'next_state' in g.files):
        pytest.skip('not covered by the tensor-core path')
    actor = m.FusedActor(sd, impl=impl)
    heads = [g['logits0']] + ([g['logits1']] if 'logits1' in g.files else [])
    gum = np.concatenate([g['gumbel0']] + ([g['gumbel1']] if 'gumbel1' in g.files else []), axis=-1)
    ref_logits = np.concatenate(heads, axis=-1)
    out = actor.forward(torch.from_numpy(g['obs'].astype(np.float32)), gumbel=gum, want_logits=True,
                        want_onehot=True, want_next_state='next_state' in g.files)
    logits = out['logits'].cpu().numpy()
    assert np.abs(logits - ref_logits).max() <= LOGIT_ATOL
    assert np.abs(logits - np.concatenate(actor_ref.forward(sd, g['obs'])['logits'], -1)).max() <= LOGIT_ATOL
    a0 = heads[0].shape[-1]
    ref_u = np.argmax(g['action0'], -1)
    gap = actor_ref.top2_gap(heads[0], g['gumbel0'])
    got_u = out['act_u'].cpu().numpy()
    assert np.all((got_u == ref_u) | (gap < GAP)) and (got_u == ref_u).mean() > 0.999
    onehot = out['onehot'].cpu().numpy()
    assert np.array_equal(np.argmax(onehot[..., :a0], -1), got_u) and np.all(onehot[..., :a0].sum(-1) == 1)
    if len(heads) == 2:
        ref_c = np.argmax(g['action1'], -1)
        gap = actor_ref.top2_gap(heads[1], g['gumbel1'])
        got_c = out['act_c'].cpu().numpy()
        assert np.all((got_c == ref_c) | (gap < GAP))
        assert np.array_equal(np.argmax(onehot[..., a0:], -1), got_c)
    if 'next_state' in g.files:
        assert np.abs(out['next_state'].cpu().numpy() - g['next_state']).max() <= LOGIT_ATOL


@pytest.mark.parametrize('impl', ['simt', 'tc'])
@pytest.mark.parametrize('N,D,A,B', [(3, 10, 5, 70_001), (6, 16, 5, 5000), (9, 22, 5, 3000), (12, 28, 5, 3000),
                                     (2, 21, [5, 10], 5000), (4, 12, 5, 999), (2, 11, 5, 257)])
def test_actor_vs_oracle_random_weights_and_philox_sampling(N, D, A, B, impl):
    """Ragged tile counts (B not a multiple of the tile), scaled-up weights for sharper logits,
    Philox-drawn noise checked against oracle/philox.py."""
    import multiagent_rl_b200 as m
    sd = actor_ref.init_state_dict(D, A, 5)
    for k in sd:
        if 'dense2' in k:
            sd[k] = sd[k] * 4.0
    if impl not in _impls(N):
        pytest.skip('not covered by the tensor-core path')
    obs = np.random.RandomState(1).uniform(-2, 2, (B, N, D)).astype(np.float32)
    actor = m.FusedActor(sd, seed=777, impl=impl)
    off, step = 1_000_000, 41
    out = actor.forward(torch.from_numpy(obs), step=step, env_id_offset=off, want_logits=True)
    want = np.concatenate(actor_ref.forward(sd, obs)['logits'], -1)
    logits = out['logits'].cpu().numpy()
    assert np.abs(logits - want).max() <= LOGIT_ATOL
    width = want.shape[-1]
    gum = philox.gumbel_noise(777, np.arange(off, off + B), step, N, width)
    a0 = A[0] if isinstance(A, list) else A
    ref_u = actor_ref.sample_hard(want[..., :a0], gum[..., :a0])
    gap = actor_ref.top2_gap(want[..., :a0], gum[..., :a0])
    got = out['act_u'].cpu().numpy()
    assert np.all((got == ref_u) | (gap < GAP)) and (got == ref_u).mean() > 0.9995
    assert len(np.unique(got)) == a0  # all actions get sampled
    if isinstance(A, list):
        ref_c = actor_ref.sample_hard(want[..., a0:], gum[..., a0:])
        gap = actor_ref.top2_gap(want[..., a0:], gum[..., a0:])
        assert np.all((out['act_c'].cpu().numpy() == ref_c) | (gap < GAP))
    # a different step or seed gives a different draw
    out2 = actor.forward(torch.from_numpy(obs), step=step + 1, env_id_offset=off)
    assert (out2['act_u'].cpu().numpy() != got).mean() > 0.2


def test_get_exploration_action_surface(golden_dir):
    """ddpg_gumbel_fix.py:86-107 return shapes: (1,N,A) float32 one-hot; MultiDiscrete -> list of two."""
    import multiagent_rl_b200 as m
    g, sd = _load(golden_dir, 'spread_n3')
    net = m.ActorNetwork(10, 5)
    net.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    tr = m.ActingTrainer(net, None, None, action_type='Discrete')
    obs_n = [g['obs'][0, i] for i in range(3)]
    a = tr.get_exploration_action(obs_n)
    assert a.shape == (1, 3, 5) and a.dtype == np.float32 and np.all(a.sum(-1) == 1)
    action_n_env = [np.array(x) for x in a[0].tolist()]  # experiments/run.py:37-38
    assert len(action_n_env) == 3 and action_n_env[0].shape == (5,)
    # weights edited in place (what optimize() does) are picked up
    with torch.no_grad():
        net.dense2.module.bias.add_(torch.tensor([0, 0, 0, 50.0, 0], device=net.dense2.module.bias.device))
    a = tr.get_exploration_action(obs_n)
    assert np.all(np.argmax(a, -1) == 3)
    g, sd = _load(golden_dir, 'reference')
    net = m.ActorNetwork(21, [5, 10])
    net.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    tr = m.ActingTrainer(net, None, None, action_type='MultiDiscrete')
    a = tr.get_exploration_action([g['obs'][0, i] for i in range(2)])
    assert isinstance(a, list) and a[0].shape == (1, 2, 5) and a[1].shape == (1, 2, 10)
    env_act = [np.concatenate([x, y], axis=-1) for x, y in zip(a[0][0], a[1][0])]  # experiments/run.py:41
    assert env_act[0].shape == (15,)
    # batched call: [B,N,D] in, [B,N,A] out
    a = tr.get_exploration_action(g['obs'][:64])
    assert a[0].shape == (64, 2, 5)


@pytest.mark.parametrize('impl', ['simt', 'tc'])
@pytest.mark.parametrize('scenario,n,B', [('simple_spread', None, 10_000 + 13), ('simple_spread', 6, 2000),
                                          ('simple_spread', 9, 1000), ('simple_spread', 12, 500),
                                          ('simple_reference', None, 3000), ('simple_speaker_listener', None, 3000),
                                          ('simple_spread', 2, 3001), ('simple_spread', 4, 2000),
                                          ('simple_spread', 8, 1000)])
def test_fused_rollout_equals_stepwise_path(scenario, n, B, impl):
    """mpe_rollout (one kernel, T steps, in-kernel auto-reset) == actor_forward + mpe_step + mpe_reset
    called step by step with the same Philox keys: actions bit-exact, values bit-exact."""
    import multiagent_rl_b200 as m
    T, seed, L = 30, 2024, 7  # episodes of 7 steps so that several auto-resets happen inside T
    spec = mpe_vec.Spec(scenario, n)
    A = [5, 10] if scenario == 'simple_reference' else 5
    sd = actor_ref.init_state_dict(spec.obs_dim, A, 9)
    for k in sd:
        if 'dense2' in k:
            sd[k] = sd[k] * 3.0
    if impl not in _impls(spec.N):
        pytest.skip('not covered by the tensor-core path')
    actor = m.FusedActor(sd, seed=seed, impl=impl)
    fused = m.make_env(scenario, n=n, num_envs=B, batched=True, seed=seed, max_episode_len=L)
    step = m.make_env(scenario, n=n, num_envs=B, batched=True, seed=seed, max_episode_len=L)
    fused.reset(); obs = step.reset()
    step.track_returns(True)
    rec = fused.rollout(actor, T, step0=100, record=True)
    for t in range(T):
        out = actor.forward(obs, step=100 + t, seed=seed)
        assert torch.equal(out['act_u'], rec[2][t]), t
        if spec.act_c:
            assert torch.equal(out['act_c'], rec[3][t]), t
        obs, rew, _, _ = step.step(out['act_u'], out['act_c'])
        assert torch.equal(obs, rec[0][t]), t
        assert torch.equal(rew, rec[1][t]), t
        if (t + 1) % L == 0:
            obs = step.reset()
    for a, b in zip(fused.get_state(), step.get_state()):
        assert torch.equal(a, b)
    sf, ss = fused.read_stats(), step.read_stats()
    assert sf[2] == ss[2] == B * (T // L) and sf[3] == ss[3]
    assert abs(sf[0] - ss[0]) <= 1e-6 * abs(ss[0]) and abs(sf[1] - ss[1]) <= 1e-6 * abs(ss[1])
    assert bool(torch.isfinite(rec[1]).all())  # the float64 oracle check of the fused kernel is the next test


@pytest.mark.parametrize('scenario,n,B', [('simple_spread', None, 65_536), ('simple_spread', 6, 8_192),
                                          ('simple_spread', 12, 2_048), ('simple_reference', None, 16_384),
                                          ('simple_speaker_listener', None, 16_384), ('simple_spread', 4, 8_192),
                                          ('simple_spread', 9, 4_096)])
def test_fused_rollout_vs_float64_oracle_directly(scenario, n, B):
    """The rollout's env phase against the float64 oracle, not via the stepwise calls: a full 25-step episode of
    ``rollout(record=True)`` (the fused kernel for teams of 2 / 3, actor + step kernels per step for larger teams) at
    the bench size (65,536 envs) is replayed by oracle/mpe_vec.py from the same initial state with the RECORDED actions.  fp32 tolerances of tests/test_gpu_env.py: positions 5e-5 worst case and 1e-5
    at p99.99 per env, velocities 5e-4, rewards 2e-4 (a reward may be off by whole units only where a collision flag sits on its
    threshold: |dist - 0.30| within the band that env's position error explains)."""
    import multiagent_rl_b200 as m
    T, seed = 25, 4242
    spec = mpe_vec.Spec(scenario, n)
    A = [5, 10] if scenario == 'simple_reference' else 5
    sd = actor_ref.init_state_dict(spec.obs_dim, A, 17)
    env = m.make_env(scenario, n=n, num_envs=B, batched=True, seed=seed, max_episode_len=T)
    actor = m.FusedActor(sd, seed=seed, impl='auto')
    obs0 = env.reset()
    pos, vel, lm, goal = env.get_state()
    v = mpe_vec.VecEnv(spec, B)
    v.set_state(pos.cpu().numpy().astype(np.float64), vel.cpu().numpy().astype(np.float64),
                lm.cpu().numpy().astype(np.float64), goal.cpu().numpy())
    assert np.abs(obs0.cpu().numpy() - v.observe()).max() <= 1e-6
    obs, rew, act_u, act_c = env.rollout(actor, T, step0=0, record=True)
    obs, rew, act_u = obs.cpu().numpy().astype(np.float64), rew.cpu().numpy().astype(np.float64), act_u.cpu().numpy()
    # the speaker's message is the first dim_c entries of its width-5 one-hot action (oracle/mpe_ref.py, ambiguity 3)
    act_c = act_c.cpu().numpy() if act_c is not None else (act_u if scenario == 'simple_speaker_listener' else None)
    worst = np.zeros(B)
    for t in range(T):
        o, r, _ = v.step(act_u[t], act_c[t] if act_c is not None else None)
        err = np.abs(obs[t] - o)[:, :, 2:].max(axis=(1, 2))     # positions and relative landmark positions
        worst = np.maximum(worst, err)
        assert np.abs(obs[t] - o)[:, :, :2].max() <= 5e-4          # velocities (= position differences / dt)
        dr = np.abs(rew[t] - r)
        if scenario == 'simple_spread':
            band = 2.0 * np.sqrt(2.0) * err + 1e-6
            d = np.linalg.norm(v.pos[:, :, None] - v.pos[:, None, :], axis=-1)
            near = (np.abs(d - 0.3) <= band[:, None, None]).any(axis=(1, 2))
            assert dr[~near].max() <= 2e-4, (t, dr[~near].max())
            assert near.mean() < 1e-3
        else:
            assert dr.max() <= 2e-4, (t, dr.max())
    # Stiff contacts (contact_margin 1e-3, contact_force 100) multiply a position difference by up to
    # 100 / 1e-3 * dt^2 = 1e3 per step while two agents overlap, so an fp32 rounding difference of 3e-8 can grow for
    # as long as a contact lasts; crowded teams (6 - 12 agents in the same arena) spend more steps in contact.
    # N <= 3: 5e-5 worst case, 1e-5 at p99.99 (SURVEY 7).  Larger teams: 5e-4 worst case, 2e-5 at p99, 2e-6 median.
    if spec.N <= 3:
        assert worst.max() <= 5e-5 and np.quantile(worst, 0.9999) <= 1e-5, (worst.max(), np.quantile(worst, 0.9999))
    else:
        assert worst.max() <= 5e-4 and np.quantile(worst, 0.99) <= 2e-5 and np.median(worst) <= 2e-6, \
            (worst.max(), np.quantile(worst, 0.99), np.median(worst))
    assert len(np.unique(act_u)) == 5


def test_host_buffer_acting_matches_device_acting():
    import multiagent_rl_b200 as m
    sd = actor_ref.init_state_dict(10, 5, 1)
    actor = m.FusedActor(sd, seed=5, impl='auto')
    obs = np.random.RandomState(0).uniform(-1, 1, (4097, 3, 10)).astype(np.float32)
    dev = actor.forward(torch.from_numpy(obs), step=3, want_onehot=True)
    au = np.empty((4097, 3), np.int32); oh = np.empty((4097, 3, 5), np.float32)
    actor.act_host(obs, step=3, act_u=au, onehot=oh)
    assert np.array_equal(au, dev['act_u'].cpu().numpy()) and np.array_equal(oh, dev['onehot'].cpu().numpy())


@pytest.mark.parametrize('N,D,A,B', [(3, 10, 5, 33_000), (2, 21, [5, 10], 9_000), (2, 11, 5, 4_100),
                                     (4, 12, 5, 3_000), (6, 16, 5, 5_000), (9, 22, 5, 2_100), (12, 28, 5, 1_537),
                                     (8, 30, 5, 1_300)])
def test_tensor_core_and_simt_paths_agree(N, D, A, B):
    """Same weights, same injected noise: logits within 1e-5, sampled indices equal outside the gap band - for
    every team size / head layout the tensor-core kernel covers (resident operands, operand ring + scratch shares,
    two heads through scratch rows), at batch sizes that are not multiples of the 128-env tile."""
    import multiagent_rl_b200 as m
    sd = actor_ref.init_state_dict(D, A, 11)
    for k in sd:  # larger weights (trained policies are sharper than the default init)
        sd[k] = sd[k] * 2.0
    width = sum(A) if isinstance(A, list) else A
    a0 = A[0] if isinstance(A, list) else A
    rng = np.random.RandomState(3)
    obs = rng.uniform(-2, 2, (B, N, D)).astype(np.float32)
    gum = -np.log(-np.log(rng.uniform(1e-6, 1 - 1e-6, (B, N, width)))).astype(np.float32)
    outs = {}
    for impl in ('simt', 'tc'):
        a = m.FusedActor(sd, impl=impl)
        outs[impl] = a.forward(torch.from_numpy(obs), gumbel=gum, want_logits=True)
        nolog = a.forward(torch.from_numpy(obs), gumbel=gum)  # the path that does not materialise the logits
        same = nolog['act_u'].cpu().numpy() == outs[impl]['act_u'].cpu().numpy()
        want = np.concatenate(actor_ref.forward(sd, obs)['logits'], -1)
        assert np.all(same | (actor_ref.top2_gap(want[..., :a0], gum[..., :a0]) < GAP))
    ls, lt = outs['simt']['logits'].cpu().numpy(), outs['tc']['logits'].cpu().numpy()
    assert np.abs(ls - want).max() <= LOGIT_ATOL and np.abs(lt - want).max() <= LOGIT_ATOL
    gap = actor_ref.top2_gap(want[..., :a0], gum[..., :a0])
    same = outs['simt']['act_u'].cpu().numpy() == outs['tc']['act_u'].cpu().numpy()
    assert np.all(same | (gap < GAP))
    if isinstance(A, list):
        gap = actor_ref.top2_gap(want[..., a0:], gum[..., a0:])
        same = outs['simt']['act_c'].cpu().numpy() == outs['tc']['act_c'].cpu().numpy()
        assert np.all(same | (gap < GAP))


@pytest.mark.parametrize('impl,N', [('tc', 3), ('tc', 6), ('simt', 3)])
def test_sampler_draws_from_softmax_of_the_logits(impl, N):
    """F.gumbel_softmax(hard=True) draws index a with probability softmax(logits)[a]
    (rls/agent/multiagent/ddpg_gumbel_fix.py:109-116).  262,144 rows with the SAME observation, Philox noise keyed by
    the row: the empirical action frequencies of every agent must match softmax(logits) within 5 sigma, and two
    different steps must be (nearly) independent draws."""
    import multiagent_rl_b200 as m
    D = 4 + 2 * N
    sd = actor_ref.init_state_dict(D, 5, 21)
    for k in sd:
        if 'dense2' in k:
            sd[k] = sd[k] * 6.0
    B = 1 << 18
    one = np.random.RandomState(5).uniform(-1, 1, (1, N, D)).astype(np.float32)
    obs = torch.from_numpy(np.repeat(one, B, 0))
    actor = m.FusedActor(sd, seed=99, impl=impl)
    lg = actor_ref.forward(sd, one)['logits'][0][0].astype(np.float64)  # [N, 5]
    p = np.exp(lg - lg.max(-1, keepdims=True))
    p /= p.sum(-1, keepdims=True)
    a1 = actor.forward(obs, step=7)['act_u'].cpu().numpy()
    a2 = actor.forward(obs, step=8)['act_u'].cpu().numpy()
    for t in range(N):
        freq = np.bincount(a1[:, t], minlength=5) / B
        sigma = np.sqrt(p[t] * (1 - p[t]) / B)
        assert np.all(np.abs(freq - p[t]) <= 5 * sigma + 1e-6), (t, freq, p[t])
        agree = (a1[:, t] == a2[:, t]).mean()  # independent draws agree with probability sum p^2
        assert abs(agree - (p[t] ** 2).sum()) < 0.01


@pytest.mark.parametrize('B', [65_536, 1 << 20])
def test_fused_rollout_full_size_properties(B):
    """BASELINE sizes (the bench's 65,536 envs and the north-star's 1,048,576): size-independent invariants of the
    fused kernel's recorded transitions instead of the oracle -
      * rewards are what the float64 reward formula gives on the recorded next observations (SURVEY 8a8: nearest-agent
        distance per landmark, -1 per agent within 0.30 including itself);
      * the recorded velocity/position pair obeys integrate_state: pos' - pos = 0.1 vel' (from consecutive records);
      * momentum: sum_i vel'_i = 0.75 sum_i vel_i + 0.1 sum_i u(action_i) (pair forces cancel);
      * every action is drawn, Philox draws differ from step to step."""
    import multiagent_rl_b200 as m
    sd = actor_ref.init_state_dict(10, 5, 33)
    actor = m.FusedActor(sd, seed=12)
    env = m.make_env('simple_spread', num_envs=B, batched=True, seed=12, max_episode_len=25)
    env.reset()
    T = 3
    obs, rew, act_u, _ = env.rollout(actor, T, step0=5, record=True)  # [T,B,N,D], [T,B,N], [T,B,N]
    table = torch.tensor([[0, 0], [5, 0], [-5, 0], [0, 5], [0, -5]], dtype=torch.float64, device='cuda')
    for t in range(T):
        o = obs[t].double()
        vel, pos = o[:, :, 0:2], o[:, :, 2:4]
        lm = pos[:, 0:1, None, :] + o[:, 0:1, 4:].reshape(B, 1, 3, 2)          # landmarks from agent 0's relative rows
        d = (pos[:, :, None, :] - lm).norm(dim=-1)                               # [B, agent, landmark]
        base = -d.min(dim=1).values.sum(-1)                                      # -sum_l min_a dist
        dd = (pos[:, :, None, :] - pos[:, None, :, :]).norm(dim=-1)              # [B, i, j], diagonal 0
        coll = (dd < 0.30).sum(-1).double()
        want = base[:, None] - coll
        near = ((dd - 0.30).abs() < 1e-5).any(-1)                                # fp32 vs fp64 flag flips at the threshold
        assert float(((rew[t].double() - want).abs() * (~near)).max()) < 2e-4
        if t > 0:
            prev = obs[t - 1].double()
            assert float((pos - prev[:, :, 2:4] - 0.1 * vel).abs().max()) < 1e-6
            u = table[act_u[t].long()].sum(1)
            assert float((vel.sum(1) - 0.75 * prev[:, :, 0:2].sum(1) - 0.1 * u).abs().max()) < 1e-4
    a = act_u.reshape(-1)
    assert int(a.min()) == 0 and int(a.max()) == 4 and len(torch.unique(a)) == 5
    assert float((act_u[0] != act_u[1]).float().mean()) > 0.2


@pytest.mark.parametrize('impl', ['auto', 'simt'])
@pytest.mark.parametrize('scenario,n,A', [('simple_spread', None, 5), ('simple_reference', None, [5, 10]),
                                          ('simple_speaker_listener', None, 5), ('simple_spread', 6, 5)])
def test_fused_rollout_equals_stepwise_path_tiny_batches(scenario, n, A, impl):
    """Batches of 1, 2 and 129 envs (one row of one tile, a tile pair whose second tile has one row): the rollout
    (one kernel for small teams on the tensor cores, actor + step kernels for large teams and for the FFMA actor)
    equals the step-by-step calls bit for bit, across auto-resets."""
    import multiagent_rl_b200 as m
    for B in (1, 2, 129):
        env = m.make_env(scenario, n=n, num_envs=B, batched=True, seed=3, max_episode_len=4)
        env2 = m.make_env(scenario, n=n, num_envs=B, batched=True, seed=3, max_episode_len=4)
        actor = m.FusedActor(actor_ref.init_state_dict(env.obs_dim, A, 1), seed=3, impl=impl)  # the rollout draws with the env's seed
        env.reset()
        obs = env2.reset()
        rec = env.rollout(actor, 9, step0=0, record=True)
        for t in range(9):
            out = actor.forward(obs, step=t)
            assert torch.equal(out['act_u'], rec[2][t]), (B, t)
            obs, rew, _, _ = env2.step(out['act_u'], out['act_c'])
            assert torch.equal(obs, rec[0][t]) and torch.equal(rew, rec[1][t]), (B, t)
            if (t + 1) % 4 == 0:
                obs = env2.reset()


@pytest.mark.parametrize('scenario,shards,B', [('simple_spread', 3, 5001), ('simple_spread', 1, 700),
                                               ('simple_reference', 2, 2050), ('simple_spread', 4, 3),
                                               ('fullobs_collect_treasure', 2, 515),
                                               ('fullobs_collect_treasure', 4, 20_011),
                                               ('simple_reference', 2, 113_801),
                                               ('fullobs_collect_treasure', 2, 113_801)])
def test_host_rollout_shards_match_the_blocking_calls(scenario, shards, B):
    """HostRollout (non-blocking mpe_act_step_host_async per shard and stream) gives, for every shard count, exactly
    the transitions of the device-tensor calls on one env handle: same Philox keys (global env id, step), same
    kernels.  Both ends of each transition are on the host: obs_prev -> (act, rew) -> obs.  The two 113,801-env
    configurations give each shard 445 tiles of 128 envs, more than one wave of tile pairs on a 148-SM part, so the
    per-stream dense2-share scratch rows of the two-head and the 8-agent tensor-core actors are reused by CTAs that
    walk a second pair."""
    import multiagent_rl_b200 as m
    L, seed = 4, 31
    n = None
    A = [5, 10] if scenario == 'simple_reference' else 5
    D = {'simple_reference': 21, 'fullobs_collect_treasure': 30}.get(scenario, 10)
    actor = m.FusedActor(actor_ref.init_state_dict(D, A, 2), seed=seed)
    hr = m.HostRollout(scenario, B, actor, shards=shards, n=n, seed=seed, max_episode_len=L, track_returns=True)
    env = m.make_env(scenario, n=n, num_envs=B, batched=True, seed=seed, max_episode_len=L)
    env.track_returns(True)
    seen = []
    cb = lambda k, tr: seen.append((tr.step, k, float(tr.rew_np.sum()), float(tr.obs_prev.sum()), float(tr.obs.sum())))  # noqa: E731
    want = []
    obs = None
    for t in range(10):
        hr.step(cb)
        hr.wait()
        if t % L == 0:
            obs = env.reset()
        out = actor.forward(obs, step=t)
        assert np.array_equal(hr.obs_prev.numpy(), obs.cpu().numpy()), t
        assert np.array_equal(hr.act_u.numpy(), out['act_u'].cpu().numpy()), t
        if hr.two_heads:
            assert np.array_equal(hr.act_c.numpy(), out['act_c'].cpu().numpy()), t
        prev = obs
        obs, rew, done, _ = env.step(out['act_u'], out['act_c'])
        assert np.array_equal(hr.obs.numpy(), obs.cpu().numpy()) and np.array_equal(hr.rew.numpy(), rew.cpu().numpy()), t
        assert int(hr.done.sum()) == 0
        for k, sh in enumerate(hr.shards):
            sl = slice(sh.offset, sh.offset + sh.num_envs)
            want.append((t, k, float(rew[sl].cpu().numpy().sum()), float(prev[sl].cpu().sum()), float(obs[sl].cpu().sum())))
    hr.flush(cb)
    # the callbacks (delivered `depth` steps late, the rest by flush) saw every shard-step once, in step order, with
    # both ends of the transition intact
    assert [x[:2] for x in seen] == [x[:2] for x in want]
    assert np.allclose(np.array(seen), np.array(want), rtol=1e-5, atol=1e-3)
    env.reset()
    hr.reset()
    hr.step()
    assert np.allclose(hr.read_stats(), env.read_stats(), rtol=1e-9)


@pytest.mark.parametrize('n', [1, 5, 7, 8, 10, 11])
def test_actor_and_rollout_for_every_team_size(n):
    """Team sizes without a tensor-core instantiation run the fp32 FFMA actor; their rollout is actor + step (+ reset)
    kernels per step.  Logits vs the float64 restatement, and the rollout equals the step-by-step calls bit for bit."""
    import multiagent_rl_b200 as m
    D, B, L = 4 + 2 * n, 777, 4
    sd = actor_ref.init_state_dict(D, 5, n)
    obs = np.random.RandomState(n).uniform(-2, 2, (B, n, D)).astype(np.float32)
    actor = m.FusedActor(sd, seed=9)
    out = actor.forward(torch.from_numpy(obs), want_logits=True, step=3)
    want = actor_ref.forward(sd, obs)['logits'][0]
    assert np.abs(out['logits'].cpu().numpy() - want).max() <= LOGIT_ATOL
    env = m.make_env('simple_spread', n=n, num_envs=B, batched=True, seed=9, max_episode_len=L)
    env2 = m.make_env('simple_spread', n=n, num_envs=B, batched=True, seed=9, max_episode_len=L)
    env.reset()
    o = env2.reset()
    rec = env.rollout(actor, 9, step0=0, record=True)
    for t in range(9):
        a = actor.forward(o, step=t)
        assert torch.equal(a['act_u'], rec[2][t]), t
        o, rew, _, _ = env2.step(a['act_u'])
        assert torch.equal(o, rec[0][t]) and torch.equal(rew, rec[1][t]), t
        if (t + 1) % L == 0:
            o = env2.reset()


@pytest.mark.parametrize('N,D,B', [(3, 10, 1000), (2, 21, 129), (6, 16, 4097), (12, 28, 300)])
def test_model_head_next_state_on_both_paths(N, D, B):
    """ac_network_model_multi_gumbel.py:49,65: next_state = dense3(relu(hcat)).  The tensor-core forward emits
    relu(hcat) and one small kernel applies dense3; the fp32 FFMA kernel computes it in place.  Both vs the float64
    restatement (1e-5), at batch sizes that leave the last tile partly empty."""
    import multiagent_rl_b200 as m
    sd = actor_ref.init_state_dict(D, 5, 4, model_head=True)
    for k in sd:
        sd[k] = sd[k] * 2.0
    obs = np.random.RandomState(N).uniform(-2, 2, (B, N, D)).astype(np.float32)
    want = actor_ref.forward(sd, obs)
    for impl in ('tc', 'simt'):
        out = m.FusedActor(sd, impl=impl).forward(torch.from_numpy(obs), want_next_state=True, want_logits=True)
        assert np.abs(out['next_state'].cpu().numpy() - want['next_state']).max() <= LOGIT_ATOL * 2, impl
        assert np.abs(out['logits'].cpu().numpy() - want['logits'][0]).max() <= LOGIT_ATOL * 2, impl


def test_host_block_layout_and_argument_checks():
    """mpe_host_block_layout / mpe_act_step_host_async: offsets are 256 B aligned and ordered, the message head only
    takes room when the env has one; mismatched handles are rejected, not launched."""
    import ctypes as C
    import multiagent_rl_b200 as m
    from multiagent_rl_b200 import _lib
    lib = _lib.load()
    for scen, heads in (('simple_spread', 1), ('simple_reference', 2)):
        env = m.make_env(scen, num_envs=1000, batched=True)
        lay = _lib.MpeHostBlockLayout()
        _lib.check(lib.mpe_host_block_layout(env._h, C.byref(lay)), 'layout')
        rows = 1000 * env.n
        offs = [lay.off_act_u, lay.off_act_c, lay.off_obs, lay.off_rew, lay.off_done, lay.bytes]
        assert all(o % 256 == 0 for o in offs) and offs == sorted(offs)
        assert lay.off_act_c - lay.off_act_u >= rows * 4 and lay.off_rew - lay.off_obs >= rows * env.obs_dim * 4
        assert (lay.off_obs == lay.off_act_c) == (heads == 1)
    env64 = m.make_env('simple_spread', num_envs=8, batched=True, precision='fp64')
    actor = m.FusedActor(actor_ref.init_state_dict(10, 5, 0))
    blk = _lib.HostBlock(1 << 20)
    obs = blk.tensor((8, 3, 10), torch.float32)
    out = blk.tensor((4096,), torch.uint8)
    st = _lib.current_stream(actor.device)
    assert lib.mpe_act_step_host_async(env64._h, actor._h, _lib.ptr(obs), 0, _lib.ptr(out), st) == _lib.MPE_EUNSUPPORTED
    env6 = m.make_env('simple_spread', n=6, num_envs=8, batched=True)
    assert lib.mpe_act_step_host_async(env6._h, actor._h, _lib.ptr(obs), 0, _lib.ptr(out), st) == _lib.MPE_EINVAL
    assert b'observation' in lib.mpe_last_error()
    with pytest.raises(ValueError):
        m.HostRollout('simple_spread', 8, actor, n=6)
    blk.free()

