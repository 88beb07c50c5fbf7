"""Generate the committed fixtures under tests/golden/.

TEST INFRASTRUCTURE (see oracle/__init__.py).  Run in the authoring container:

    python -m oracle.gen_golden            # writes tests/golden/*.npz

Two families:
  * ``mpe_<scenario>[_n<N>].npz`` - trajectories produced by the LOOP oracle
    (oracle/mpe_ref.py), env by env, 25 steps (rls/arglist.py:5) of seeded
    random one-hot actions from seeded initial states.  No reference
    implementation of the physics exists in /root/reference (it imports the
    un-vendored ``multiagent`` package), so these pin the *restatement*, not
    the reference: parity unpinned.
  * ``critic_*.npz`` - outputs of the REFERENCE's own CriticNetwork classes (same two files, :70-148 / :69-143).
  * ``actor_*.npz`` - outputs of the REFERENCE's own ActorNetwork
    (/root/reference/rls/model/ac_network_multi_gumbel.py:24-67 and
    ac_network_model_multi_gumbel.py:23-66) and of the reference's sampling
    recipe (rls/agent/multiagent/ddpg_gumbel_fix.py:92-100,109-116) run on CPU
    with torch.manual_seed; needs /root/reference, which only exists here.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLD = os.path.join(ROOT, 'tests', 'golden')
T = 25


def gen_mpe(scenario, n, B, seed):
    from oracle import mpe_ref
    rng = np.random.RandomState(seed)
    env = mpe_ref.make_env(scenario, n=n)
    N = env.n
    L = len(env.world.landmarks)
    D = env.observation_space[0].shape[0]
    dim_c = env.world.dim_c
    multi = isinstance(env.action_space[0], mpe_ref.MultiDiscrete)
    pos0 = rng.uniform(-1, 1, (B, N, 2))
    lm0 = rng.uniform(-1, 1, (B, L, 2))
    vel0 = np.zeros((B, N, 2))
    # make a share of the envs start in (or near) contact so the softplus branch is exercised
    for b in range(0, B, 3):
        for i in range(1, N):
            ang = rng.uniform(0, 2 * np.pi)
            rad = rng.uniform(0.2, 0.34)
            pos0[b, i] = pos0[b, i - 1] + rad * np.array([np.cos(ang), np.sin(ang)])
    # and a share start with non-zero velocity
    vel0[1::4] = rng.uniform(-1, 1, vel0[1::4].shape)
    if scenario == 'simple_reference':
        goal0 = rng.randint(0, L, (B, N))
    elif scenario == 'simple_speaker_listener':
        goal0 = np.stack([rng.randint(0, L, B), -np.ones(B, dtype=np.int64)], axis=1)
    else:
        goal0 = -np.ones((B, N), dtype=np.int64)
    act_u = rng.randint(0, 5, (T, B, N))
    act_c = rng.randint(0, max(dim_c, 1), (T, B, N))
    pos = np.zeros((T, B, N, 2)); vel = np.zeros((T, B, N, 2))
    obs = np.zeros((T, B, N, D)); rew = np.zeros((T, B, N))
    coll = np.zeros((T, B, N), dtype=np.int32); occ = np.zeros((T, B), dtype=np.int32)
    obs0 = np.zeros((B, N, D))
    bench_env = mpe_ref.make_env(scenario, n=n, benchmark=True) if scenario == 'simple_spread' else None
    for b in range(B):
        mpe_ref.set_state(env, pos0[b], vel0[b], lm0[b], goal0[b])
        obs0[b] = np.stack(mpe_ref.get_obs(env))
        for t in range(T):
            action_n = []
            for i in range(N):
                a = np.zeros(5); a[act_u[t, b, i]] = 1.0
                if multi:
                    c = np.zeros(dim_c); c[act_c[t, b, i]] = 1.0
                    a = np.concatenate([a, c])
                action_n.append(a)
            o, r, d, info = env.step(action_n)
            assert not any(d)
            obs[t, b] = np.stack(o); rew[t, b] = np.array(r)
            pos[t, b] = np.stack([a.state.p_pos for a in env.world.agents])
            vel[t, b] = np.stack([a.state.p_vel for a in env.world.agents])
            if bench_env is not None:
                mpe_ref.set_state(bench_env, pos[t, b], vel[t, b], lm0[b], goal0[b])
                for i, ag in enumerate(bench_env.world.agents):
                    bd = bench_env.scenario.benchmark_data(ag, bench_env.world)
                    assert bd[0] == rew[t, b, i]
                    coll[t, b, i] = bd[1]; occ[t, b] = bd[3]
    name = 'mpe_%s%s.npz' % (scenario, '' if n is None else '_n%d' % n)
    np.savez_compressed(os.path.join(GOLD, name), pos0=pos0, vel0=vel0, lm0=lm0, goal0=goal0,
                        act_u=act_u, act_c=act_c, obs0=obs0, pos=pos, vel=vel, obs=obs, rew=rew,
                        coll=coll, occ=occ)
    print('wrote', name, 'contacts:', int((coll.sum(-1) > N).sum()))


TREASURE_SEED = 20240607  # Philox key of the fixture's respawn draws (global env id = row index, episode 0)


def gen_treasure(B, seed, T=T, keep=24):
    """``mpe_fullobs_collect_treasure.npz``: the loop oracle of the MAAC-fork scenario (oracle/maac_ref.py) from
    crafted initial states - collectors on / next to treasures, collectors that hold a treasure next to the matching
    (and the wrong) deposit, a dead treasure that respawns in the first post_step, agents in contact across the three
    mass pairings - under seeded random actions.  Respawn draws come from the kernels' Philox stream
    (seed TREASURE_SEED, env id = row, episode 0, step t), so a CUDA env seeded alike reproduces the file.
    Only the first ``keep`` of the B envs are stored (four of each of the six kinds of crafted state at 24), which
    keeps the file under 1 MB; rows are independent, so they are the same as in a run of ``keep`` envs."""
    from oracle import maac_ref, mpe_ref
    rng = np.random.RandomState(seed)
    env = mpe_ref.make_env('fullobs_collect_treasure')
    bench = mpe_ref.make_env('fullobs_collect_treasure', benchmark=True)
    N, L, D = 8, 6, 30
    pos0 = rng.uniform(-1, 1, (B, N, 2)); vel0 = np.zeros((B, N, 2))
    tr0 = rng.uniform(-0.95, 0.95, (B, L, 2))
    flags0 = np.zeros(B, dtype=np.int64)
    for b in range(B):
        types = rng.randint(0, 2, L); alive = [True] * L; hold = [-1] * 6
        kind = b % 6
        if kind == 1:    # collectors right at treasures (inside / just outside the 0.075 contact radius)
            for i in range(6):
                ang = rng.uniform(0, 2 * np.pi)
                pos0[b, i] = tr0[b, rng.randint(L)] + rng.uniform(0.0, 0.12) * np.array([np.cos(ang), np.sin(ang)])
        elif kind == 2:  # holders next to the deposits
            for i in range(6):
                hold[i] = int(rng.randint(-1, 2))
                ang = rng.uniform(0, 2 * np.pi)
                pos0[b, i] = pos0[b, 6 + rng.randint(2)] + rng.uniform(0.0, 0.2) * np.array([np.cos(ang), np.sin(ang)])
        elif kind == 3:  # dead treasures (they respawn in the first post_step), some holders
            for l in rng.choice(L, 2, replace=False):
                alive[l] = False
                tr0[b, l] = -999.0
            hold[0] = int(types[0])
        elif kind == 4:  # contacts between collectors, collector / deposit and the two deposits; moving agents
            pos0[b, 1] = pos0[b, 0] + np.array([0.09, 0.01])
            pos0[b, 2] = pos0[b, 6] + np.array([0.05, 0.1])
            pos0[b, 7] = pos0[b, 6] + np.array([-0.1, 0.1])
            vel0[b] = rng.uniform(-1.2, 1.2, (N, 2))
        elif kind == 5:  # everything at once
            vel0[b] = rng.uniform(-0.5, 0.5, (N, 2))
            for i in range(6):
                hold[i] = int(rng.randint(-1, 2))
                pos0[b, i] = (tr0[b, i] if hold[i] < 0 else pos0[b, 6 + hold[i]]) + rng.uniform(-0.08, 0.08, 2)
        flags0[b] = maac_ref.pack_flags(types, alive, hold)
    act_u = rng.randint(0, 5, (T, B, N))
    pos = np.zeros((T, B, N, 2)); vel = np.zeros((T, B, N, 2)); tr = np.zeros((T, B, L, 2))
    obs = np.zeros((T, B, N, D)); rew = np.zeros((T, B, N)); flags = np.zeros((T, B), dtype=np.int64)
    info = np.zeros((T, B, N), dtype=np.int32); obs0 = np.zeros((B, N, D))
    for b in range(B):
        for e in (env, bench):
            e.scenario.draws = maac_ref.PhiloxDraws(TREASURE_SEED, b)
            maac_ref.set_state(e, pos0[b], vel0[b], tr0[b], flags0[b])
        obs0[b] = np.stack(mpe_ref.get_obs(env))
        for t in range(T):
            for e in (env, bench):
                e.scenario.draws.tstep = t
            acts = [np.eye(5)[act_u[t, b, i]] for i in range(N)]
            o, r, d, _ = env.step([a.copy() for a in acts])
            o2, r2, _, inf = bench.step([a.copy() for a in acts])
            assert r == r2 and not any(d)
            obs[t, b] = np.stack(o); rew[t, b] = np.array(r); info[t, b] = np.array(inf['n'])
            pos[t, b] = np.stack([a.state.p_pos for a in env.world.agents])
            vel[t, b] = np.stack([a.state.p_vel for a in env.world.agents])
            tr[t, b] = np.stack([l.state.p_pos for l in env.world.landmarks])
            flags[t, b] = maac_ref.get_flags(env)
    pos0, vel0, tr0, flags0, obs0 = pos0[:keep], vel0[:keep], tr0[:keep], flags0[:keep], obs0[:keep]
    act_u, pos, vel, tr, obs, rew, flags, info = (x[:, :keep] for x in (act_u, pos, vel, tr, obs, rew, flags, info))
    name = 'mpe_fullobs_collect_treasure.npz'
    np.savez_compressed(os.path.join(GOLD, name), pos0=pos0, vel0=vel0, tr0=tr0, flags0=flags0, act_u=act_u, obs0=obs0,
                        pos=pos, vel=vel, tr=tr, obs=obs, rew=rew, flags=flags, info=info, seed=np.int64(TREASURE_SEED))
    ev = (np.diff(np.concatenate([flags0[None], flags]), axis=0) != 0).sum()
    print('wrote', name, 'state-word changes (pick-up / respawn / deposit):', int(ev), 'reward range', rew.min(), rew.max())


def gen_actor(tag, D, A, N, B, seed, model_head):
    sys.path.insert(0, '/root/reference')
    import torch
    import torch.nn.functional as F
    if model_head:
        from rls.model.ac_network_model_multi_gumbel import ActorNetwork
    else:
        from rls.model.ac_network_multi_gumbel import ActorNetwork
    torch.manual_seed(seed)
    np.random.seed(seed)
    actor = ActorNetwork(input_dim=D, out_dim=A)
    # scale the output layers up so logits are not all ~0 (trained policies are sharper)
    sd = actor.state_dict()
    obs = np.random.uniform(-1.5, 1.5, (B, N, D))  # float64, like the env returns
    # ddpg_gumbel_fix.py:59-61,92-94 with batch B instead of 1
    state = torch.from_numpy(np.array(obs, dtype='float32'))
    with torch.no_grad():
        res = actor.forward(state)
    nxt = None
    if model_head:
        res, nxt = res
    heads = res if isinstance(res, list) else [res]
    out = {'obs': obs}
    for k, v in sd.items():
        out['sd/' + k] = v.numpy()
    for hi, logits in enumerate(heads):
        logits = logits.detach()
        n, t = logits.size(0), logits.size(1)
        flat = logits.contiguous().view(n * t, logits.size(2))
        torch.manual_seed(seed + 100 + hi)
        y = F.gumbel_softmax(flat, hard=True).view(n, t, -1)  # ddpg_gumbel_fix.py:113
        torch.manual_seed(seed + 100 + hi)
        g = -torch.empty_like(flat).exponential_().log()  # same first draw as F.gumbel_softmax
        out['logits%d' % hi] = logits.numpy()
        out['gumbel%d' % hi] = g.view(n, t, -1).numpy()
        out['action%d' % hi] = y.numpy()
    if nxt is not None:
        out['next_state'] = nxt.detach().numpy()
    name = 'actor_%s.npz' % tag
    np.savez_compressed(os.path.join(GOLD, name), **out)
    print('wrote', name)


def gen_critic(tag, D, A, N, B, seed, model):
    """Outputs of the REFERENCE's own CriticNetwork (rls/model/ac_network_multi_gumbel.py:70-148 or
    ac_network_model_multi_gumbel.py:69-143) on seeded observations and one-hot / soft actions."""
    sys.path.insert(0, '/root/reference')
    import torch
    import torch.nn.functional as F
    if model:
        from rls.model.ac_network_model_multi_gumbel import CriticNetwork
    else:
        from rls.model.ac_network_multi_gumbel import CriticNetwork
    torch.manual_seed(seed)
    np.random.seed(seed)
    widths = A if isinstance(A, list) else [A]
    critic = CriticNetwork(input_dim=D + int(np.sum(widths)), out_dim=1)   # main.py:61
    obs = np.random.uniform(-1.5, 1.5, (B, N, D)).astype(np.float32)
    acts = []
    for w in widths:  # half the rows exact one-hots (replay), half soft Gumbel-softmax samples (optimize())
        logits = torch.randn(B, N, w)
        soft = F.gumbel_softmax(logits.view(B * N, w), hard=False).view(B, N, w)
        hard = F.one_hot(logits.argmax(-1), w).float()
        a = torch.where((torch.arange(B) % 2 == 0).view(B, 1, 1), hard, soft)
        acts.append(a.numpy().astype(np.float32))
    with torch.no_grad():
        res = critic.forward(torch.from_numpy(obs), [torch.from_numpy(a) for a in acts] if len(acts) > 1 else torch.from_numpy(acts[0]))
    out = {'obs': obs, 'action': np.concatenate(acts, -1)}
    for k, v in critic.state_dict().items():
        out['sd/' + k] = v.numpy()
    if model:
        out['q'], out['r'] = res[0].numpy(), res[1].numpy()
    else:
        out['q'] = res.numpy()
    name = 'critic_%s.npz' % tag
    np.savez_compressed(os.path.join(GOLD, name), **out)
    print('wrote', name)


def main():
    os.makedirs(GOLD, exist_ok=True)
    gen_mpe('simple_spread', None, 48, 101)
    gen_mpe('simple_spread', 6, 24, 102)
    gen_mpe('simple_spread', 9, 12, 103)
    gen_mpe('simple_spread', 12, 12, 104)
    gen_mpe('simple_reference', None, 48, 105)
    gen_mpe('simple_speaker_listener', None, 48, 106)
    gen_treasure(48, 107)
    if os.path.isdir('/root/reference'):
        gen_actor('spread_n3', 10, 5, 3, 256, 12345678, False)
        gen_actor('spread_n12', 28, 5, 12, 64, 12345679, False)
        gen_actor('reference', 21, [5, 10], 2, 256, 12345680, False)
        gen_actor('speaker', 11, 5, 2, 256, 12345681, False)
        gen_actor('model_n6', 16, 5, 6, 64, 12345682, True)
        gen_critic('spread_n3', 10, 5, 3, 256, 12345683, False)
        gen_critic('reference', 21, [5, 10], 2, 256, 12345684, False)
        gen_critic('model_n12', 28, 5, 12, 64, 12345685, True)
    else:
        print('no /root/reference: actor fixtures not regenerated')


if __name__ == '__main__':
    main()
