"""CPU tests that pin the oracle: Philox known answers, hand-derived contact
forces, loop-vs-vectorised bit equality on the committed trajectories, and the
actor restatement against the reference ActorNetwork's committed outputs."""
import os

import numpy as np
import pytest

from oracle import actor_ref, critic_ref, mpe_ref, mpe_vec, philox

MPE_FILES = [('simple_spread', None), ('simple_spread', 6), ('simple_spread', 9), ('simple_spread', 12),
             ('simple_reference', None), ('simple_speaker_listener', None)]


def _gold(golden_dir, scenario, n):
    return np.load(os.path.join(golden_dir, 'mpe_%s%s.npz' % (scenario, '' if n is None else '_n%d' % n)))


def test_philox_known_answers():
    # Random123 kat_vectors, philox4x32 10 rounds
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in kat:
        got = philox.philox4x32_10([np.array([c]) for c in ctr], [np.array([k]) for k in key])
        assert tuple(int(g[0]) for g in got) == want


def test_philox_float_maps():
    r = np.array([0, 0xffffffff, 0x80000000], dtype=np.uint32)
    p = philox.bits_to_pos(r)
    assert p[0] == -1.0 and p[1] == 1.0 - 2.0 ** -23 and p[2] == 0.0
    assert np.all(p.astype(np.float32).astype(np.float64) == p)  # exact in fp32
    g = philox.bits_to_gumbel(r)
    assert np.all(np.isfinite(g))
    pos = philox.reset_positions(7, np.arange(1000), 3, 6)
    assert pos.shape == (1000, 6, 2) and pos.min() >= -1 and pos.max() < 1
    assert abs(pos.mean()) < 0.05
    goals = philox.reset_goals(7, np.arange(3000), 0, 2, 3)
    assert set(np.unique(goals)) == {0, 1, 2}


def _two_agent_force(dist):
    w = mpe_ref.World()
    a, b = mpe_ref.Agent(), mpe_ref.Agent()
    a.size = b.size = 0.15
    a.state.p_pos = np.array([0.0, 0.0]); b.state.p_pos = np.array([dist, 0.0])
    return w.get_collision_force(a, b)


def test_contact_force_known_answers():
    # SURVEY 8c: dist == dist_min -> pen = k ln2, |f| = 100 * k * ln2
    fa, fb = _two_agent_force(0.3)
    assert np.isclose(-fa[0], 100 * 1e-3 * np.log(2.0), rtol=1e-9) and fa[1] == 0.0
    assert np.all(fb == -fa)
    # 1 cm penetration -> |f| ~ 1.0 (pen = 0.01 + k*log1p(exp(-10)))
    fa, _ = _two_agent_force(0.29)
    assert np.isclose(-fa[0], 100 * (0.01 + 1e-3 * np.log1p(np.exp(-10.0))), rtol=1e-9)
    assert abs(-fa[0] - 1.0) < 1e-4
    # far pairs: exactly zero once exp(-x/k) underflows
    fa, _ = _two_agent_force(0.3 + 0.75)
    assert fa[0] == 0.0 and fa[1] == 0.0
    # float32 underflow threshold used by the fp32 kernel's early-out
    assert np.float32(np.exp(np.float32(-104.0))) == 0.0


def test_action_table_and_self_collision():
    env = mpe_ref.make_env('simple_spread')
    mpe_ref.set_state(env, [[0, 0], [1, 1], [-1, -1]], np.zeros((3, 2)), np.zeros((3, 2)) + 5)
    table = {0: (0, 0), 1: (5, 0), 2: (-5, 0), 3: (0, 5), 4: (0, -5)}
    for idx, u in table.items():
        a = np.zeros(5); a[idx] = 0.7  # force_discrete_action: argmax -> exact one-hot, in place
        env._set_action(a, env.world.agents[0], env.action_space[0])
        assert tuple(env.world.agents[0].action.u) == u
        assert a[idx] == 1.0 and a.sum() == 1.0
    # reward contains the constant -1 self collision
    _, rew, done, info = env.step([np.eye(5)[0]] * 3)
    md = sum(min(np.linalg.norm(a.state.p_pos - l.state.p_pos) for a in env.world.agents)
             for l in env.world.landmarks)
    assert np.allclose(rew, -md - 1.0) and done == [False] * 3 and info == {'n': [{}, {}, {}]}


def test_make_env_surface():
    e = mpe_ref.make_env('simple_spread')
    assert e.n == 3 and e.observation_space[0].shape[0] == 10 and e.action_space[0].n == 5
    assert e.shared_reward is False and e.force_discrete_action is True
    e = mpe_ref.make_env('simple_spread', n=12)
    assert e.n == 12 and e.observation_space[0].shape[0] == 28
    e = mpe_ref.make_env('simple_reference')
    assert e.n == 2 and e.observation_space[0].shape[0] == 21
    assert (e.action_space[0].high + 1).tolist() == [5, 10]
    e = mpe_ref.make_env('simple_speaker_listener')
    assert e.n == 2 and e.observation_space[0].shape[0] == 11 and e.action_space[0].n == 5
    np.random.seed(3)
    obs = e.reset()
    assert len(obs) == 2 and obs[0].shape == (11,) and np.all(obs[1][8:] == 0)


@pytest.mark.parametrize('scenario,n', MPE_FILES)
def test_vectorised_oracle_matches_loop_oracle_bit_exactly(golden_dir, scenario, n):
    g = _gold(golden_dir, scenario, n)
    spec = mpe_vec.Spec(scenario, n)
    B = g['pos0'].shape[0]
    env = mpe_vec.VecEnv(spec, B)
    env.set_state(g['pos0'], g['vel0'], g['lm0'], g['goal0'])
    assert np.array_equal(env.observe(), g['obs0'])
    for t in range(g['act_u'].shape[0]):
        obs, rew, (coll, occ) = env.step(g['act_u'][t], g['act_c'][t])
        assert np.array_equal(env.pos, g['pos'][t]), t
        assert np.array_equal(env.vel, g['vel'][t]), t
        assert np.array_equal(obs, g['obs'][t]), t
        assert np.array_equal(rew, g['rew'][t]), t
        if scenario == 'simple_spread':
            assert np.array_equal(coll, g['coll'][t]) and np.array_equal(occ, g['occ'][t])


def test_golden_has_contacts_and_momentum_symmetry(golden_dir):
    g = _gold(golden_dir, 'simple_spread', None)
    assert (g['coll'].sum(-1) > 3).sum() > 10
    # f_a = -f_b: with zero action and equal masses total momentum only decays by damping
    spec = mpe_vec.Spec('simple_spread')
    env = mpe_vec.VecEnv(spec, g['pos0'].shape[0])
    env.set_state(g['pos0'], g['vel0'], g['lm0'])
    p0 = env.vel.sum(axis=1)
    env.step(np.zeros((env.B, 3), dtype=np.int64))
    assert np.allclose(env.vel.sum(axis=1), 0.75 * p0, atol=1e-12)


def test_max_speed_clip_loop_vs_vec():
    rng = np.random.RandomState(5)
    env = mpe_ref.make_env('simple_spread')
    for a in env.world.agents:
        a.max_speed = 0.3
    spec = mpe_vec.Spec('simple_spread', max_speed=0.3)
    B = 16
    pos = rng.uniform(-1, 1, (B, 3, 2)); vel = rng.uniform(-1, 1, (B, 3, 2)); lm = rng.uniform(-1, 1, (B, 3, 2))
    act = rng.randint(0, 5, (B, 3))
    v = mpe_vec.VecEnv(spec, B); v.set_state(pos, vel, lm)
    obs, rew, _ = v.step(act)
    for b in range(B):
        mpe_ref.set_state(env, pos[b], vel[b], lm[b])
        o, r, _, _ = env.step([np.eye(5)[act[b, i]] for i in range(3)])
        assert np.array_equal(np.stack(o), obs[b]) and np.array_equal(np.array(r), rew[b])
    assert np.all(np.linalg.norm(v.vel, axis=-1) <= 0.3 + 1e-12)


def test_numpy_reset_order_matches_loop_oracle():
    env = mpe_ref.make_env('simple_reference')
    np.random.seed(42)
    env.reset()
    np.random.seed(42)
    g0, g1 = np.random.choice(3), np.random.choice(3)
    pts = [np.random.uniform(-1, +1, 2) for _ in range(5)]
    w = env.world
    assert w.agents[0].goal_b is w.landmarks[g0] and w.agents[1].goal_b is w.landmarks[g1]
    for ent, p in zip(w.agents + w.landmarks, pts):
        assert np.array_equal(ent.state.p_pos, p)


ACTOR_FILES = ['spread_n3', 'spread_n12', 'reference', 'speaker', 'model_n6']


@pytest.mark.parametrize('tag', ACTOR_FILES)
def test_actor_restatement_matches_reference_network(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, 'actor_%s.npz' % tag))
    sd = {k[3:]: g[k] for k in g.files if k.startswith('sd/')}
    out = actor_ref.forward(sd, g['obs'])
    for hi, logits in enumerate(out['logits']):
        ref = g['logits%d' % hi]
        assert logits.shape == ref.shape
        # reference runs fp32 on CPU; the float64 restatement agrees to fp32 rounding
        assert np.max(np.abs(logits - ref)) < 2e-6
        gum = g['gumbel%d' % hi]
        idx = actor_ref.sample_hard(ref, gum)
        ref_idx = np.argmax(g['action%d' % hi], axis=-1)
        gap = actor_ref.top2_gap(ref, gum)
        assert np.all((idx == ref_idx) | (gap < 1e-6))
        assert (idx == ref_idx).mean() > 0.999
        # hard one-hot up to 1 ulp (y_hard - y_soft.detach() + y_soft)
        assert np.allclose(g['action%d' % hi].sum(-1), 1.0, atol=1e-6)
    if 'next_state' in g.files:
        assert np.max(np.abs(out['next_state'] - g['next_state'])) < 2e-6


def test_init_state_dict_shapes():
    sd = actor_ref.init_state_dict(21, [5, 10], 0, model_head=True)
    assert sd['dense2_2.module.weight'].shape == (10, 64) and sd['dense3.module.weight'].shape == (21, 64)
    assert sum(v.size for v in actor_ref.init_state_dict(10, 5, 0).values()) == 26117


@pytest.mark.parametrize('tag', ['spread_n3', 'reference', 'model_n12'])
def test_critic_restatement_matches_reference_network(golden_dir, tag):
    """tests/golden/critic_*.npz are outputs of the reference's CriticNetwork classes (fp32, CPU)."""
    g = np.load(os.path.join(golden_dir, 'critic_%s.npz' % tag))
    sd = {k[3:]: g[k] for k in g.files if k.startswith('sd/')}
    out = critic_ref.forward(sd, g['obs'], g['action'])
    assert out['q'].shape == g['q'].shape and np.abs(out['q'] - g['q']).max() < 1e-6
    assert ('r' in out) == ('r' in g.files)
    if 'r' in out:
        assert np.abs(out['r'] - g['r']).max() < 1e-6


def _replay_batch(rng, B, N, D, act_dims, with_done):
    obs, nxt = rng.randn(B, N, D).astype(np.float32), rng.randn(B, N, D).astype(np.float32)
    rew = rng.randn(B, N).astype(np.float32)
    au = rng.randint(0, act_dims[0], (B, N))
    ac = rng.randint(0, act_dims[1], (B, N)) if len(act_dims) > 1 else None
    done = (rng.rand(B) < 0.3).astype(np.float32) if with_done else None
    return obs, au, ac, rew, nxt, done


@pytest.mark.parametrize('cap,batches,act_dims', [
    (50, [7, 13], [5]),                # partial fill
    (50, [30, 31], [5]),               # the second add wraps
    (50, [11, 50, 50], [5]),           # batches equal to the capacity, head != 0
    (37, [20, 9, 37, 1, 25], [5, 10]),  # two heads, several wraps
])
def test_vectorised_replay_model_matches_reference_ring(cap, batches, act_dims):
    """oracle/replay_ref.BatchedRing (index arithmetic) equals ReplayRing fed one transition at a time."""
    from oracle import replay_ref
    rng = np.random.RandomState(cap + len(batches))
    N, D = 3, 4
    model, ring = replay_ref.BatchedRing(cap, act_dims), replay_ref.ReplayRing(cap)
    for i, B in enumerate(batches):
        obs, au, ac, rew, nxt, done = _replay_batch(rng, B, N, D, act_dims, with_done=i % 2 == 0)
        model.add(obs, au, rew, nxt, done, act_c=ac)
        onehot = np.eye(act_dims[0], dtype=np.float32)[au]
        if ac is not None:
            onehot = np.concatenate([onehot, np.eye(act_dims[1], dtype=np.float32)[ac]], axis=-1)
        replay_ref.add_batched_step(ring, obs, onehot, rew, nxt, done)
        assert len(model) == len(ring) and model._next_idx == ring._next_idx
        n = len(ring)
        idx = np.concatenate([np.arange(n), rng.randint(-n, n, 40), [-n, n - 1, -1]])
        got, want = model.sample_index(idx), ring.sample_index(idx)
        for k in (0, 1, 3, 4):
            assert np.array_equal(got[k], want[k].astype(np.float32)), k
        # np.sum adds the agents in its own order; the model adds them the way the kernel does
        assert np.allclose(got[2], want[2], rtol=1e-6, atol=1e-6)
        with pytest.raises(IndexError):
            model.sample_index([n])
        with pytest.raises(IndexError):
            model.sample_index([-n - 1])
        # device indices: negatives wrap once, anything still out of range is clamped
        assert np.array_equal(model.slots([n, 10 * n, -1, -n - 1, -10 * n], clamp=True), [n - 1, n - 1, n - 1, 0, 0])
    for k, c in enumerate(model.collect()):
        assert len(c) == len(ring), k


def test_shared_reward_is_a_sequential_fp32_sum():
    from oracle import replay_ref
    rng = np.random.RandomState(3)
    rew = (rng.randn(200, 12) * 10.0 ** rng.randint(-3, 4, (200, 12))).astype(np.float32)
    want = []
    for row in rew:
        s = np.float32(0.0)
        for v in row:
            s = np.float32(s + v)
        want.append(s)
    assert np.array_equal(replay_ref.shared_reward(rew), np.array(want, dtype=np.float32))


def test_replay_index_matches_big_integer_arithmetic():
    """philox.replay_index against the formula in Python integers: mulhi64((r0 << 32) | r1, size)."""
    for seed, draw, size in [(0, 0, 1), (1, 0, 3000), (7, 5, 1000003), (2 ** 40 + 9, 2 ** 33 + 17, 12345),
                             (123, 1, 2 ** 20), (5, 2, 2 ** 63 - 25)]:
        batch = 300
        got = philox.replay_index(seed, draw, batch, size)
        r = philox.raw(seed, np.arange(batch, dtype=np.uint64), draw & 0xFFFFFFFF, philox.DOMAIN_REPLAY,
                       (draw >> 32) & 0xFFFF)
        want = [((int(r[0][j]) << 32 | int(r[1][j])) * size) >> 64 for j in range(batch)]
        assert got.tolist() == want
        assert got.min() >= 0 and got.max() < size
    # the replay stream is its own domain: no block is shared with the treasure env's respawn draws
    r = philox.raw(1, np.arange(8, dtype=np.uint64), 0, philox.DOMAIN_REPLAY, 0)
    q = philox.raw(1, np.arange(8, dtype=np.uint64), 0, philox.DOMAIN_RESPAWN, 0)
    assert not np.array_equal(r[0], q[0])
