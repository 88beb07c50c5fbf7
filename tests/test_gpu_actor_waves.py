"""Every actor kernel instantiation past its first wave, at every head layout the launchers accept, against the
float64 oracle.

The actor kernels are persistent: k_tc2 launches min(tile pairs, SMs) CTAs of two 128-env tiles, k_actor_forward
min(tiles, SMs) CTAs of TB-env tiles, k_dense3x2 at most 5 x SMs CTAs of 128 rows, and each CTA walks the rest in a
grid-stride loop.  A CTA's second and later pairs (tiles) carry state across iterations - mbarrier phase bits, the
operand ring's fill bits, the pending TMA store, the per-CTA dense2-share scratch rows - that a batch of one wave
never exercises.  The tests here therefore run at B = 6 * SMs * 128 + 77 envs (113,741 on a 148-SM B200), read from
the device so the file means the same on any part: 6 * SMs + 1 tiles of 128, so every k_tc2 CTA walks at least three
tile pairs and the last pair holds one ragged tile and one empty one; every FFMA CTA walks 12 or more 64-env tiles
(48 or more 16-env tiles).  Each test asserts its geometry.

The observations are periodic, obs[b] = pool[b % P] with P = 4,099 distinct rows (prime, more than the tiles), so the
float64 oracle runs only on the pool while every one of the B rows is checked: its logits against the oracle row, and
bit for bit against the first row of the batch with the same observation.  That catches a row that picks up another
pair's data far below the 1e-5 tolerance, and logits that depend on where an env sits in the batch (which warpgroup of
the tile pair owns its tile): HostRollout shards start at any env, and their trajectories must not depend on the
shard count.  Outputs are caller-allocated and
pre-filled with NaN / -1, so a row the kernel skips cannot pass on bytes a previous call left in torch's allocator.
The sampling noise is Philox with a 64-bit seed and env ids that cross 2^32 inside the batch, against oracle/philox.py.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import actor_ref, mpe_vec, philox

pytestmark = pytest.mark.gpu

LOGIT_ATOL = 1e-5
GAP = 1e-5
P = 4099
SEED = 2 ** 40 + 9           # high key word non-zero
OFF = 2 ** 32 - 5000         # env ids cross into the counter's high word at row 5,000
STEP = 41
TC_TEAMS = (2, 3, 4, 6, 8, 9, 12)


def _nsm():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _wave_batch():
    return 6 * _nsm() * 128 + 77


def _ffma_tile(N):
    return 64 if N <= 3 else (32 if N <= 6 else 16)


def _assert_waves(B, N, impl):
    """The launch geometry of actor_kernels.cu / tc_kernels.cu at batch B: every CTA walks several tiles."""
    nsm = _nsm()
    if impl == 'tc':
        ntiles = -(-B // 128)
        pairs = (ntiles + 1) // 2
        grid = min(pairs, nsm)
        assert grid == nsm and pairs // grid >= 3, (B, pairs, grid)
        assert ntiles % 2 == 1 and 0 < B - (ntiles - 1) * 128 < 128  # last pair: a ragged tile and an empty one
    else:
        tb = _ffma_tile(N)
        ntiles = -(-B // tb)
        grid = min(ntiles, nsm)
        assert grid == nsm and ntiles // grid >= 12 * 64 // tb and B % tb != 0, (B, ntiles, grid)


def _impls(N, width):
    if N in (2, 3) or (N in TC_TEAMS and width <= 8):
        return ['simt', 'tc']
    return ['simt']


def _pool(N, D, seed):
    return np.random.RandomState(seed).uniform(-2, 2, (P, N, D)).astype(np.float32)


def _periodic(pool_dev, B):
    return pool_dev[torch.arange(B, device=pool_dev.device) % P].contiguous()


def _misaligned(x):
    """The same values at an address 4 bytes past a 16-byte boundary (no float2 / float4 / TMA loads)."""
    buf = torch.empty(x.numel() + 1, dtype=x.dtype, device=x.device)
    buf[1:] = x.reshape(-1)
    v = buf[1:].view(x.shape)
    assert v.data_ptr() % 16 == 4
    return v


def _forward(actor, obs, step=STEP, seed=SEED, off=OFF, next_state=False):
    """actor_forward into caller-allocated outputs pre-filled with NaN / -1."""
    from multiagent_rl_b200 import _lib
    B, N, D = obs.shape
    dev = obs.device
    nan = lambda *s: torch.full(s, float('nan'), dtype=torch.float32, device=dev)  # noqa: E731
    out = {'act_u': torch.full((B, N), -1, dtype=torch.int32, device=dev),
           'act_c': torch.full((B, N), -1, dtype=torch.int32, device=dev) if actor.multi else None,
           'logits': nan(B, N, actor.A), 'onehot': nan(B, N, actor.A),
           'next_state': nan(B, N, D) if next_state else None}
    _lib.check(actor._lib.actor_forward(
        actor._h, _lib.ptr(obs), B, N, None, C.c_uint64(seed), C.c_uint64(step), int(off), _lib.ptr(out['logits']),
        _lib.ptr(out['next_state']), _lib.ptr(out['act_u']), _lib.ptr(out['act_c']), _lib.ptr(out['onehot']),
        _lib.current_stream(dev)), 'actor_forward')
    torch.cuda.synchronize()
    return out


def _first_of_class(B):
    """Index of the first row of the batch with the same observation as row b."""
    b = np.arange(B)
    _, first, inv = np.unique(b % P, return_index=True, return_inverse=True)
    return torch.from_numpy(first[inv.reshape(-1)])


def _bits_equal(x, ref_idx):
    return torch.equal(x.view(torch.int32), x[ref_idx.to(x.device)].view(torch.int32))


def _heads(A):
    return list(A) if isinstance(A, list) else [A]


def _oracle_picks(want_rows, gum, heads):
    """Per head: Gumbel-max index of (float64 logits + float64 noise) and the top-2 gap."""
    res, a0 = [], 0
    for w in heads:
        z = want_rows[..., a0:a0 + w] + gum[..., a0:a0 + w]
        top = torch.topk(z, 2, dim=-1).values
        res.append((z.argmax(-1), top[..., 0] - top[..., 1]))
        a0 += w
    return res


def _check_actions(out, picks, heads, tag):
    a0 = 0
    oh = out['onehot']
    assert bool(((oh == 0) | (oh == 1)).all()), tag
    for key, (want, gap), w in zip(('act_u', 'act_c'), picks, heads):
        got = out[key].long()
        bad = (got != want) & (gap >= GAP)
        assert int(bad.sum()) == 0, (tag, key, int(bad.sum()))
        assert float((got == want).double().mean()) > 0.999, (tag, key)
        assert len(torch.unique(got)) == w, (tag, key)  # every entry of the head gets drawn
        assert torch.equal(oh[..., a0:a0 + w].argmax(-1), got) and bool((oh[..., a0:a0 + w].sum(-1) == 1).all()), tag
        a0 += w


MATRIX = ([(2, D, A) for D in (11, 21) for A in (5, 3, 12, [5, 10], [3, 4])] +
          [(3, 10, A) for A in (5, 8, 16, [5, 10], [3, 4])] +
          [(N, 4 + 2 * N, A) for N in (4, 6, 8, 9, 12) for A in (5, 3, [3, 4])] + [(4, 13, 5)] +
          [(N, 4 + 2 * N, 5) for N in (1, 5, 7, 10, 11)])


@pytest.mark.parametrize('N,D,A', MATRIX)
def test_actor_past_the_first_wave_vs_oracle(N, D, A):
    """Every path that covers (N, D, heads): logits of all B rows within 1e-5 of the float64 oracle and bit-identical
    to the row with the same observation; actions = argmax(oracle logits + oracle Philox noise) per head outside the
    top-2 gap band; one-hot consistent with the actions."""
    import multiagent_rl_b200 as m
    B = _wave_batch()
    heads = _heads(A)
    width = sum(heads)
    sd = actor_ref.init_state_dict(D, A, 5 + N)
    for k in sd:
        if 'dense2' in k:
            sd[k] = sd[k] * 3.0
    pool = _pool(N, D, N * 100 + D)
    want = torch.from_numpy(np.concatenate(actor_ref.forward(sd, pool)['logits'], -1)).cuda()  # [P,N,A] float64
    idx = torch.arange(B, device='cuda') % P
    want_rows = want[idx]
    gum = torch.from_numpy(philox.gumbel_noise(SEED, np.arange(OFF, OFF + B, dtype=np.uint64), STEP, N, width)).cuda()
    picks = _oracle_picks(want_rows, gum, heads)
    del gum
    obs = _periodic(torch.from_numpy(pool).cuda(), B)
    for impl in _impls(N, width):
        _assert_waves(B, N, impl)
        tag = (impl, N, D, A)
        out = _forward(m.FusedActor(sd, seed=0, impl=impl), obs)  # the seed argument of actor_forward wins
        lg = out['logits']
        assert float((lg.double() - want_rows).abs().max()) <= LOGIT_ATOL, tag  # NaN (a skipped row) fails too
        assert _bits_equal(lg, _first_of_class(B)), tag
        _check_actions(out, picks, heads, tag)
        if len(heads) == 1:
            assert out['act_c'] is None


@pytest.mark.parametrize('N,D,A', [(3, 10, 5), (2, 11, [3, 4]), (6, 16, 5), (9, 22, [3, 4])])
def test_misaligned_observations_give_the_same_outputs(N, D, A):
    """The same batch through an aligned tensor and through a view one float past it: the large-team operand warp
    then loads scalars instead of float2, the FFMA kernel stages tiles with plain loads instead of TMA bulk copies.
    Every output is bit-identical."""
    import multiagent_rl_b200 as m
    B = _wave_batch()
    sd = actor_ref.init_state_dict(D, A, 3)
    obs = _periodic(torch.from_numpy(_pool(N, D, 7)).cuda(), B)
    mis = _misaligned(obs)
    for impl in _impls(N, sum(_heads(A))):
        _assert_waves(B, N, impl)
        actor = m.FusedActor(sd, impl=impl)
        a, b = _forward(actor, obs), _forward(actor, mis)
        assert bool(torch.isfinite(a['logits']).all()), impl
        for k in ('logits', 'onehot', 'act_u', 'act_c'):
            if a[k] is not None:
                assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), (impl, k)


@pytest.mark.parametrize('N', [3, 6])
def test_model_head_past_the_first_wave(N):
    """next_state of the "+model" actor at the wave size, where k_dense3x2 (after the tensor-core forward) takes 3 or
    more grid-stride steps, and of the FFMA kernel's in-kernel head.  Three calls on one actor - B, a smaller batch,
    a larger one - reuse and then grow its relu(hcat) buffer.  Each call vs the float64 oracle (2e-5), rows
    bit-identical to the row with the same observation."""
    import multiagent_rl_b200 as m
    D = 4 + 2 * N
    B = _wave_batch()
    sizes = (B, B // 3 + 5, B + 3001)
    rows = B * N
    grid = min(-(-rows // 128), 5 * _nsm())
    assert (-(-rows // 128)) // grid >= 3
    sd = actor_ref.init_state_dict(D, 5, 4, model_head=True)
    for k in sd:
        sd[k] = sd[k] * 2.0
    pool = _pool(N, D, 11)
    ref = actor_ref.forward(sd, pool)
    want_ns = torch.from_numpy(ref['next_state']).cuda()
    want_lg = torch.from_numpy(ref['logits'][0]).cuda()
    obs = _periodic(torch.from_numpy(pool).cuda(), max(sizes))
    for impl in ('tc', 'simt'):
        actor = m.FusedActor(sd, impl=impl)
        for i, Bk in enumerate(sizes):
            idx = torch.arange(Bk, device='cuda') % P
            out = _forward(actor, obs[:Bk], step=i, next_state=True)
            ns = out['next_state']
            assert float((ns.double() - want_ns[idx]).abs().max()) <= 2 * LOGIT_ATOL, (impl, Bk)
            assert float((out['logits'].double() - want_lg[idx]).abs().max()) <= 2 * LOGIT_ATOL, (impl, Bk)
            assert _bits_equal(ns, _first_of_class(Bk)), (impl, Bk)


def _rollout_sample_rows(B, nsm, seed):
    """Env rows whose actions are checked against the float64 actor: a few rows of both tiles of every CTA's last
    pair, the whole ragged last tile, the rows where the env id crosses 2^32, and a random sample."""
    ntiles = -(-B // 128)
    npairs = (ntiles + 1) // 2
    rows = set(range((ntiles - 1) * 128, B))
    for c in range(min(npairs, nsm)):
        last = c + (npairs - 1 - c) // nsm * nsm
        for tile in (2 * last, 2 * last + 1):
            rows.update(r for r in (tile * 128, tile * 128 + 63, tile * 128 + 127) if r < B)
    rows.update(range(2 ** 32 - OFF - 3, 2 ** 32 - OFF + 3))
    rows.update(np.random.RandomState(seed).randint(0, B, 512).tolist())
    return np.array(sorted(rows))


@pytest.mark.parametrize('scenario,n', [('simple_spread', 2), ('simple_spread', None), ('simple_reference', None),
                                        ('simple_speaker_listener', None)])
def test_fused_rollout_past_the_first_wave(scenario, n):
    """The four fused k_tc2 rollouts at the wave size, 9 steps with episodes of 4 (two in-kernel auto-resets), a
    64-bit env seed and env ids crossing 2^32:
      * the rollout equals the stepwise actor / step / reset calls bit for bit;
      * its env phase matches oracle/mpe_vec.py replayed with the recorded actions from each episode's start state
        (tolerances of test_fused_rollout_vs_float64_oracle_directly);
      * on sampled env rows (every CTA's last pair, the ragged last tile) the recorded actions are the float64
        actor's Gumbel-max picks under the oracle's Philox noise, outside the top-2 gap band."""
    import multiagent_rl_b200 as m
    B, T, L, step0 = _wave_batch(), 9, 4, 100
    spec = mpe_vec.Spec(scenario, n)
    _assert_waves(B, spec.N, 'tc')
    heads = [5, 10] if scenario == 'simple_reference' else [5]
    sd = actor_ref.init_state_dict(spec.obs_dim, heads if len(heads) == 2 else 5, 9)
    for k in sd:
        if 'dense2' in k:
            sd[k] = sd[k] * 3.0
    actor = m.FusedActor(sd, seed=SEED, impl='tc')
    kw = dict(n=n, num_envs=B, batched=True, seed=SEED, env_id_offset=OFF, max_episode_len=L)
    fused, step = m.make_env(scenario, **kw), m.make_env(scenario, **kw)
    fused.reset()
    obs = step.reset()
    rec = fused.rollout(actor, T, step0=step0, record=True)
    sample = _rollout_sample_rows(B, _nsm(), 1)
    sample_dev = torch.from_numpy(sample).cuda()
    starts, seen = {}, []
    for t in range(T):
        if t % L == 0:
            starts[t] = [x.cpu().numpy() for x in step.get_state()]
        seen.append(obs[sample_dev].cpu().numpy())
        out = actor.forward(obs, step=step0 + t, seed=SEED, env_id_offset=OFF)
        assert torch.equal(out['act_u'], rec[2][t]), t
        if spec.act_c:
            assert torch.equal(out['act_c'], rec[3][t]), t
        obs, rew, _, _ = step.step(out['act_u'], out['act_c'])
        assert torch.equal(obs, rec[0][t]) and torch.equal(rew, rec[1][t]), t
        if (t + 1) % L == 0:
            obs = step.reset()
    for a, b in zip(fused.get_state(), step.get_state()):
        assert torch.equal(a, b)

    # env phase vs the float64 oracle, each episode replayed from its start state with the recorded actions
    v = mpe_vec.VecEnv(spec, B)
    worst = np.zeros(B)
    for t in range(T):
        if t in starts:
            pos, vel, lm, goal = starts[t]
            v.set_state(pos.astype(np.float64), vel.astype(np.float64), lm.astype(np.float64), goal)
        au = rec[2][t].cpu().numpy()
        ac = rec[3][t].cpu().numpy() if spec.act_c else (au if scenario == 'simple_speaker_listener' else None)
        o, r, _ = v.step(au, ac)
        ob = rec[0][t].cpu().numpy().astype(np.float64)
        err = np.abs(ob - o)[:, :, 2:].max(axis=(1, 2))
        worst = np.maximum(worst, err)
        assert np.abs(ob - o)[:, :, :2].max() <= 5e-4, t
        dr = np.abs(rec[1][t].cpu().numpy().astype(np.float64) - r)
        if scenario == 'simple_spread':
            band = 2.0 * np.sqrt(2.0) * err + 1e-6
            d = np.linalg.norm(v.pos[:, :, None] - v.pos[:, None, :], axis=-1)
            near = (np.abs(d - 0.3) <= band[:, None, None]).any(axis=(1, 2))
            assert dr[~near].max() <= 2e-4, (t, dr[~near].max())
            assert near.mean() < 1e-3
        else:
            assert dr.max() <= 2e-4, (t, dr.max())
    assert worst.max() <= 5e-5 and np.quantile(worst, 0.9999) <= 1e-5, (worst.max(), np.quantile(worst, 0.9999))

    # recorded actions of the sampled rows vs the float64 actor and the oracle's Philox noise
    width = sum(heads)
    gids = (OFF + sample).astype(np.uint64)
    for t in range(T):
        lg = np.concatenate(actor_ref.forward(sd, seen[t])['logits'], -1)
        gum = philox.gumbel_noise(SEED, gids, step0 + t, spec.N, width)
        a0 = 0
        for w, got in zip(heads, (rec[2][t], rec[3][t] if spec.act_c else None)):
            want = actor_ref.sample_hard(lg[..., a0:a0 + w], gum[..., a0:a0 + w])
            gap = actor_ref.top2_gap(lg[..., a0:a0 + w], gum[..., a0:a0 + w])
            got = got[sample_dev].cpu().numpy()
            assert np.all((got == want) | (gap < GAP)), (t, w, int(((got != want) & (gap >= GAP)).sum()))
            a0 += w
