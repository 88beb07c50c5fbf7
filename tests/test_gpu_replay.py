"""GPU tests of the device replay ring against oracle/replay_ref.py (the reference ReplayBuffer's semantics):
ring overwrite order, shared-reward sum, one-hot actions, gather by index, uniform sampling - on every launch path of
csrc/replay_kernels.cu, exactly, and the index stream against oracle/philox.py."""
import numpy as np
import pytest
import torch

from oracle import philox, replay_ref

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('N,D,A', [(3, 10, [5]), (2, 21, [5, 10]), (12, 28, [5])])
def test_ring_matches_reference_semantics(N, D, A):
    import multiagent_rl_b200 as m
    cap, B = 1000, 333
    buf = m.DeviceReplayBuffer(cap, N, D, A, seed=1)
    ring = replay_ref.ReplayRing(cap)
    rng = np.random.RandomState(0)
    for step in range(5):  # 1665 transitions through a ring of 1000: wraps
        obs = rng.randn(B, N, D).astype(np.float32); nxt = rng.randn(B, N, D).astype(np.float32)
        rew = rng.randn(B, N).astype(np.float32); done = (rng.rand(B) < 0.1).astype(np.float32)
        au = rng.randint(0, A[0], (B, N)); ac = rng.randint(0, A[1], (B, N)) if len(A) > 1 else None
        onehot = np.eye(A[0], dtype=np.float32)[au]
        if ac is not None:
            onehot = np.concatenate([onehot, np.eye(A[1], dtype=np.float32)[ac]], axis=-1)
        buf.add(obs, au, rew, nxt, done, act_c=ac)
        replay_ref.add_batched_step(ring, obs, onehot, rew, nxt, done)
        assert len(buf) == len(ring) and buf._next_idx == ring._next_idx
    idx = rng.randint(0, cap, 257)
    got = buf.sample_index(idx)
    want = ring.sample_index(idx)
    assert np.array_equal(got[0].cpu().numpy(), want[0]) and np.array_equal(got[3].cpu().numpy(), want[3])
    assert np.array_equal(got[1].cpu().numpy(), want[1])
    assert np.allclose(got[2].cpu().numpy(), want[2], atol=1e-6)  # fp32 sum over agents in agent order
    assert np.array_equal(got[4].cpu().numpy(), want[4])
    allv = buf.collect()
    assert allv[0].shape == (cap, N, D)
    buf.clear()
    assert len(buf) == 0


def test_uniform_sampling_and_errors():
    import multiagent_rl_b200 as m
    buf = m.DeviceReplayBuffer(5000, 3, 10, 5, seed=7)
    with pytest.raises(RuntimeError, match='empty'):
        buf.sample(4)
    z = torch.zeros(3000, 3, 10, device='cuda')
    buf.add(z, torch.zeros(3000, 3, dtype=torch.int32), torch.arange(9000, dtype=torch.float32).reshape(3000, 3), z)
    i1, i2 = buf.make_index(200_000), buf.make_index(200_000)
    assert int(i1.min()) >= 0 and int(i1.max()) < 3000 and not torch.equal(i1, i2)
    hist = torch.bincount(i1, minlength=3000).float()
    assert abs(float(hist.mean()) - 200_000 / 3000) < 1e-3 and float(hist.std()) < 12  # ~sqrt(66.7) = 8.2
    obs, act, rew, nxt, done = buf.sample(1024)
    assert obs.shape == (1024, 3, 10) and act.shape == (1024, 3, 5) and bool((act.sum(-1) == 1).all())
    assert bool(((rew / 3 - (rew / 3).round()).abs() < 1e-3).all())  # rew_shared = 3*(3i+1): every i in range
    latest = buf.make_latest_index(10)
    assert sorted(latest.tolist()) == list(range(2990, 3000))


def test_rollout_feeds_replay():
    """env.rollout(record=True) + replay: the transition stream of experiments/run.py:36-65 without leaving HBM."""
    import multiagent_rl_b200 as m
    from oracle import actor_ref
    B, T = 2048, 6
    env = m.make_env('simple_spread', num_envs=B, batched=True, seed=5, max_episode_len=25)
    actor = m.FusedActor(actor_ref.init_state_dict(10, 5, 0), seed=5)
    buf = m.DeviceReplayBuffer(B * T, 3, 10, 5)
    obs = env.reset()
    nxt, rew, au, _ = env.rollout(actor, T, record=True)
    prev = obs
    for t in range(T):
        buf.add(prev, au[t], rew[t], nxt[t])
        prev = nxt[t]
    assert len(buf) == B * T
    o, a, r, n, d = buf.sample_index(torch.arange(B, 2 * B))  # the transitions of step 1
    assert torch.equal(o, nxt[0]) and torch.equal(n, nxt[1]) and torch.allclose(r, rew[1].sum(1), atol=1e-5)
    assert torch.equal(a.argmax(-1).int(), au[1]) and float(d.abs().max()) == 0.0


def test_replay_rejects_mismatched_tensors_and_bad_indices():
    import multiagent_rl_b200 as m
    rb = m.DeviceReplayBuffer(64, 3, 10, 5)
    obs = torch.zeros((8, 3, 10), device='cuda')
    act = torch.zeros((8, 3), dtype=torch.int32, device='cuda')
    rew = torch.zeros((8, 3), device='cuda')
    with pytest.raises(ValueError):
        rb.add(obs, act[:4], rew, obs)
    with pytest.raises(ValueError):
        rb.add(obs, act, rew[:, :2], obs)
    with pytest.raises(ValueError):
        rb.add(obs[:, :2], act, rew, obs)
    # records over 48 KB cannot be staged by add: such a ring is refused when it is created
    with pytest.raises(RuntimeError, match='49232 bytes'):
        m.DeviceReplayBuffer(16, 32, 192, 5)
    rb.add(obs + torch.arange(8, device='cuda').view(8, 1, 1), act, rew, obs)
    with pytest.raises(IndexError):
        rb.sample_index([0, 8])
    with pytest.raises(IndexError):
        rb.sample_index(np.array([-9]))
    o = rb.sample_index([-1, 0])[0]   # Python list indexing: -1 is the newest transition
    assert float(o[0, 0, 0]) == 7.0 and float(o[1, 0, 0]) == 0.0
    # device-resident indices cannot raise without a sync: out-of-range values are clamped into the ring
    o = rb.sample_index(torch.tensor([1000, -1000, -2], device='cuda'))[0]
    assert [float(x) for x in o[:, 0, 0]] == [7.0, 0.0, 6.0]


# Ring shapes, one per launch path of csrc/replay_kernels.cu.  record = record_bytes(N, D): [obs][obs_next][rew][done]
# [act_u bytes][act_c bytes] padded to 16 B.  add: k_replay_add<2> when N*D is even and both sources are 8 B aligned,
# else <1>; records per block (rpb) = 128 halved until rpb * record <= 32 KB.  gather: k_replay_gather_tile<2 / 1> (same
# rule) with rpb = 64 halved until rpb * record <= 16 KB; records over 16 KB go to the element-parallel k_replay_gather.
RINGS = [
    pytest.param(3, 10, [5], id='n3d10_256B_tile2_rpb128_64'),
    pytest.param(3, 7, [5], id='n3d7_192B_tile1_odd_R'),
    pytest.param(1, 5, [5], id='n1d5_64B_tile1_smallest_team'),
    pytest.param(2, 21, [5, 10], id='n2d21_352B_two_heads'),
    pytest.param(2, 9, [127, 127], id='n2d9_160B_widest_int8_action'),
    pytest.param(12, 28, [5], id='n12d28_2720B_rpb8_4'),
    pytest.param(32, 64, [5], id='n32d64_16464B_add_rpb1_gather_elem2'),
    pytest.param(31, 67, [5], id='n31d67_16688B_add_rpb1_gather_elem1'),
    pytest.param(32, 191, [5], id='n32d191_48976B_largest_record'),
]


def _batch(rng, B, N, D, A, with_done):
    obs = rng.randn(B, N, D).astype(np.float32)
    nxt = rng.randn(B, N, D).astype(np.float32)
    rew = (rng.randn(B, N) * 10.0 ** rng.randint(-3, 4, (B, N))).astype(np.float32)  # magnitudes that round in the sum
    au = rng.randint(0, A[0], (B, N))
    ac = rng.randint(0, A[1], (B, N)) if len(A) > 1 else None
    if A[0] == 127:  # the largest index a 127-wide head stores in its int8 action byte
        au[:, 0] = 126
        if ac is not None:
            ac[:, -1] = 126
    done = (rng.rand(B) < 0.3).astype(np.float32) if with_done else None
    return obs, au, ac, rew, nxt, done


def _assert_same(got, want, what):
    names = ('obs', 'act_onehot', 'rew', 'obs_next', 'done')
    for g, w, name in zip(got, want, names):
        g = g.cpu().numpy()
        assert g.shape == w.shape and g.dtype == w.dtype, (what, name, g.shape, w.shape)
        assert np.array_equal(g, w), (what, name, int((g != w).sum()))


@pytest.mark.parametrize('N,D,A', RINGS)
def test_ring_matches_vectorised_model_on_every_launch_path(N, D, A):
    """A partial fill, a batch that crosses the end of the ring, a batch of the ring's capacity starting at head != 0,
    and one more small add: contents, shared reward (fp32, agent order), one-hot rebuild and index rules are exact."""
    import multiagent_rl_b200 as m
    cap = 300
    buf = m.DeviceReplayBuffer(cap, N, D, A, seed=3)
    model = replay_ref.BatchedRing(cap, A)
    rng = np.random.RandomState(N * 1000 + D)
    for i, B in enumerate([70, 250, cap, 33]):
        obs, au, ac, rew, nxt, done = _batch(rng, B, N, D, A, with_done=i % 2 == 0)
        buf.add(obs, au, rew, nxt, done, act_c=ac)
        model.add(obs, au, rew, nxt, done, act_c=ac)
        assert len(buf) == len(model) and buf._next_idx == model._next_idx, i
        _assert_same(buf.collect(), model.collect(), 'collect after add %d' % i)
        n = len(model)
        # host indices: Python list indexing, negatives included; 1500 rows take the element-parallel gather of the
        # largest records through more than one grid stride
        idx = np.concatenate([rng.randint(-n, n, 1500), [-n, -1, 0, n - 1]])
        _assert_same(buf.sample_index(idx), model.sample_index(idx), 'host indices after add %d' % i)
        # device indices: negatives wrap once, anything still outside [0, len) is clamped
        big = np.iinfo(np.int64)
        didx = np.array([n, n + 1, 10 * n, -n - 1, -10 * n, big.max, big.min, -1, 0, n - 1], dtype=np.int64)
        _assert_same(buf.sample_index(torch.from_numpy(didx).cuda()), model.sample_index(didx, clamp=True),
                     'device indices after add %d' % i)


def test_misaligned_sources_take_the_scalar_add_path():
    """obs / obs_next that start 4 B into a larger tensor (N * D even) go through k_replay_add<1> by the alignment
    test; the ring must hold exactly what an aligned add stores."""
    import multiagent_rl_b200 as m
    N, D, B, cap = 3, 10, 333, 500
    rng = np.random.RandomState(9)
    obs, au, _, rew, nxt, done = _batch(rng, B, N, D, [5], with_done=True)
    o_mis, n_mis = (torch.cat([torch.zeros(1), torch.from_numpy(x).reshape(-1)]).cuda()[1:].view(B, N, D)
                    for x in (obs, nxt))
    assert o_mis.is_contiguous() and o_mis.data_ptr() % 8 == 4 and n_mis.data_ptr() % 8 == 4
    aligned, mis = m.DeviceReplayBuffer(cap, N, D, 5), m.DeviceReplayBuffer(cap, N, D, 5)
    for _ in range(2):  # the second add wraps
        aligned.add(obs, au, rew, nxt, done)
        mis.add(o_mis, au, rew, n_mis, done)
    for g, w in zip(mis.collect(), aligned.collect()):
        assert torch.equal(g, w)
    model = replay_ref.BatchedRing(cap, [5])
    model.add(obs, au, rew, nxt, done)
    model.add(obs, au, rew, nxt, done)
    _assert_same(mis.collect(), model.collect(), 'misaligned add')


def test_bench_size_ring_drives_every_grid_stride_loop():
    """Capacity 2^20, two adds of 2^19 + 3 transitions (the second wraps): the add and tile-gather grids cover the
    rows in more than one stride.  Expectations are gathered on the device from the added tensors."""
    import multiagent_rl_b200 as m
    N, D, cap, B = 3, 10, 1 << 20, (1 << 19) + 3
    g = torch.Generator(device='cuda')
    g.manual_seed(5)
    buf = m.DeviceReplayBuffer(cap, N, D, 5, seed=2)
    model = replay_ref.BatchedRing(cap, [5])
    adds = []
    for k in range(2):
        obs = torch.randn(B, N, D, device='cuda', generator=g)
        nxt = torch.randn(B, N, D, device='cuda', generator=g)
        rew = torch.randn(B, N, device='cuda', generator=g)
        au = torch.randint(0, 5, (B, N), device='cuda', dtype=torch.int32, generator=g)
        done = (torch.rand(B, device='cuda', generator=g) < 0.1).float()
        buf.add(obs, au, rew, nxt, done)
        assert model.add_rows(B) == k
        shared = rew[:, 0].clone()
        for n in range(1, N):  # the kernel's fp32 sum, agent by agent
            shared = shared + rew[:, n]
        adds.append((obs, torch.nn.functional.one_hot(au.long(), 5).float(), shared, nxt, done))
    assert len(buf) == cap and buf._next_idx == 6 == model._next_idx
    idx = np.random.RandomState(1).randint(-cap, cap, cap)
    add, row = (torch.from_numpy(x).cuda() for x in model.source(idx))
    got = buf.sample_index(torch.from_numpy(idx).cuda())
    for f in range(5):
        want = torch.where((add == 0).view((-1,) + (1,) * (adds[0][f].dim() - 1)), adds[0][f][row], adds[1][f][row])
        assert torch.equal(got[f], want), f
    allv = buf.collect()  # slot order: slots 0..5 hold the wrapped tail of the second add
    assert torch.equal(allv[0][:6], adds[1][0][B - 6:]) and torch.equal(allv[0][6:B], adds[0][0][6:])
    assert torch.equal(allv[3][B:], adds[1][3][:cap - B]) and torch.equal(allv[2][B:], adds[1][2][:cap - B])
    del allv, got
    # make_index over more samples than one grid of k_replay_make_index covers (4736 blocks x 256 threads)
    big = (1 << 21) + 5
    want = philox.replay_index(2, 0, big, cap)
    assert np.array_equal(buf.make_index(big).cpu().numpy(), want)


@pytest.mark.parametrize('N,D,offset', [
    pytest.param(3, 10, 0, id='tile2'), pytest.param(3, 10, 1, id='tile1_misaligned_out'),
    pytest.param(3, 7, 0, id='tile1_odd_R'), pytest.param(32, 64, 0, id='elem2'),
    pytest.param(32, 64, 1, id='elem1_misaligned_out'), pytest.param(31, 67, 0, id='elem1_odd_R')])
def test_gather_writes_nothing_past_the_batch(N, D, offset):
    """replay_sample called directly with output buffers of B + 64 rows filled with a NaN sentinel: rows past B
    stay untouched, rows below B equal sample_index (outputs `offset` floats into their allocation)."""
    import ctypes as C
    import multiagent_rl_b200 as m
    from multiagent_rl_b200 import _lib
    cap, B, A, pad = 400, 333, 5, 64
    rng = np.random.RandomState(N + D + offset)
    buf = m.DeviceReplayBuffer(cap, N, D, A, seed=4)
    obs, au, _, rew, nxt, done = _batch(rng, cap, N, D, [A], with_done=True)
    buf.add(obs, au, rew, nxt, done)
    nan = float('nan')

    def out(*shape):
        t = torch.full((int(np.prod((B + pad,) + shape)) + offset,), nan, device='cuda')
        return t[offset:].view((B + pad,) + shape)
    for idx in (torch.from_numpy(rng.randint(-cap, cap, B)).cuda(), None):
        o, a, r, x, d = out(N, D), out(N, A), out(), out(N, D), out()
        iout = torch.full((B + pad,), -7, dtype=torch.int64, device='cuda')
        if offset:
            assert o.data_ptr() % 8 == 4 and x.data_ptr() % 8 == 4
        _lib.check(buf._lib.replay_sample(buf._h, B, _lib.ptr(idx), C.c_uint64(buf.seed), _lib.ptr(o), _lib.ptr(a),
                                          _lib.ptr(r), _lib.ptr(x), _lib.ptr(d), _lib.ptr(iout),
                                          _lib.current_stream(buf.device)), 'replay_sample')
        for t in (o, a, r, x, d):
            assert bool(torch.isnan(t[B:]).all())
        assert bool((iout[B:] == -7).all())
        used = iout[:B] if idx is None else idx
        if idx is not None:
            assert torch.equal(iout[:B], idx)
        for g, w in zip((o, a, r, x, d), buf.sample_index(used)):
            assert torch.equal(g[:B], w)


def test_index_stream_is_the_specified_philox_stream():
    """The k-th index draw of a ring (make_index or sample(batch)) is philox.replay_index(seed, k, batch, len):
    domain 5 of the Philox stream layout; sample_index and collect() draw nothing."""
    import multiagent_rl_b200 as m
    N, D, A, cap, seed = 3, 10, 5, 1000, 11
    rng = np.random.RandomState(0)
    buf = m.DeviceReplayBuffer(cap, N, D, A, seed=seed)
    model = replay_ref.BatchedRing(cap, [A])

    def add(B):
        obs, au, _, rew, nxt, done = _batch(rng, B, N, D, [A], with_done=True)
        buf.add(obs, au, rew, nxt, done)
        model.add(obs, au, rew, nxt, done)
    add(300)  # partial fill: len 300
    assert np.array_equal(buf.make_index(257).cpu().numpy(), philox.replay_index(seed, 0, 257, 300))
    want_idx = philox.replay_index(seed, 1, 100, 300)
    _assert_same(buf.sample(100), model.sample_index(want_idx), 'sample(100) draws index set 1')
    buf.sample_index(np.arange(5))
    buf.sample_index(torch.arange(5, device='cuda'))
    buf.collect()
    assert np.array_equal(buf.make_index(64).cpu().numpy(), philox.replay_index(seed, 2, 64, 300))
    add(777)  # wraps: len 1000, head 77
    assert len(buf) == cap and buf._next_idx == 77
    assert np.array_equal(buf.make_index(1001).cpu().numpy(), philox.replay_index(seed, 3, 1001, 1000))
    _assert_same(buf.sample(3), model.sample_index(philox.replay_index(seed, 4, 3, 1000)), 'sample(3) after wrap')
    assert np.array_equal(buf.make_index(5).cpu().numpy(), philox.replay_index(seed, 5, 5, 1000))
