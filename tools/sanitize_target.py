"""Small workload touching every kernel (ragged sizes) for compute-sanitizer runs:
    compute-sanitizer --tool memcheck python tools/sanitize_target.py"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import multiagent_rl_b200 as m  # noqa: E402
from multiagent_rl_b200.networks import random_state_dict  # noqa: E402

for scen, n, B, A in [('simple_spread', None, 333, 5), ('simple_spread', 6, 70, 5), ('simple_spread', 9, 41, 5),
                      ('simple_spread', 12, 37, 5), ('simple_reference', None, 200, [5, 10]),
                      ('simple_speaker_listener', None, 129, 5), ('simple_spread', 1, 33, 5), ('simple_spread', 5, 65, 5),
                      ('simple_spread', 7, 29, 5), ('simple_spread', 8, 31, 5), ('simple_spread', 10, 27, 5),
                      ('simple_spread', 11, 23, 5), ('fullobs_collect_treasure', None, 77, 5)]:
    for precision in ('fp32', 'fp64'):
        env = m.make_env(scen, n=n, num_envs=B, batched=True, seed=3, precision=precision, max_episode_len=3)
        env.track_returns(True)
        env.reset()
        for t in range(4):
            au = torch.randint(0, 5, (B, env.n), dtype=torch.int32, device='cuda')
            ac = torch.randint(0, 10, (B, env.n), dtype=torch.int32, device='cuda') if env.act_c else None
            env.step(au, ac, info=True)
        env.reset(mask=torch.ones(B, dtype=torch.uint8))
        env.observe(); env.get_state(); env.read_stats()
    env = m.make_env(scen, n=n, num_envs=B, batched=True, seed=3, max_episode_len=3)
    obs = env.reset()
    tc_ok = env.n in (2, 3, 4, 6, 8, 9, 12)
    for impl in ['simt'] + (['tc'] if tc_ok else []):
        actor = m.FusedActor(random_state_dict(env.obs_dim, A, 1), impl=impl)
        actor.forward(obs, want_logits=True, want_onehot=True)
        env.rollout(actor, 5, record=True)
        env.rollout(actor, 2)
# the tensor-core actor at tile-boundary batch sizes (1 tile, 1 tile + 1 row, odd numbers of tiles / tile pairs),
# small and large teams: same actions as the fp32 SIMT kernel under the same Philox keys except at near-ties
for n, D in ((3, 10), (4, 12), (6, 16), (12, 28)):
    sd = random_state_dict(D, 5, 2)
    tc, simt = m.FusedActor(sd, impl='tc', seed=4), m.FusedActor(sd, impl='simt', seed=4)
    for B in (1, 127, 128, 129, 255, 257, 300, 385):
        obs = torch.from_numpy(np.random.RandomState(B).uniform(-1, 1, (B, n, D)).astype(np.float32)).cuda()
        a, b = tc.forward(obs, step=B)['act_u'], simt.forward(obs, step=B)['act_u']
        assert int(a.min()) >= 0 and int(a.max()) <= 4
        assert float((a == b).float().mean()) > 0.995, (n, B)
# model head (dense3 on top of the tensor-core forward), critic, host-buffer rollouts at ragged sizes
for n, D, B in ((3, 10, 130), (6, 16, 257), (12, 28, 65)):
    sd = random_state_dict(D, 5, 3, model_head=True)
    obs = torch.from_numpy(np.random.RandomState(n).uniform(-1, 1, (B, n, D)).astype(np.float32)).cuda()
    for impl in ('tc', 'simt'):
        out = m.FusedActor(sd, impl=impl).forward(obs, want_next_state=True)
        assert bool(torch.isfinite(out['next_state']).all())
    rng = np.random.RandomState(0)
    csd = {'dense1.module.weight': rng.randn(64, D + 5).astype(np.float32) * 0.1, 'dense1.module.bias': np.zeros(64, np.float32),
           'lstm.weight_ih_l0': rng.randn(256, 64).astype(np.float32) * 0.1, 'lstm.weight_hh_l0': rng.randn(256, 64).astype(np.float32) * 0.1,
           'lstm.bias_ih_l0': np.zeros(256, np.float32), 'lstm.bias_hh_l0': np.zeros(256, np.float32),
           'dense2.weight': rng.randn(1, 64).astype(np.float32), 'dense2.bias': np.zeros(1, np.float32)}
    q = m.FusedCritic(csd, obs_dim=D).forward(obs, torch.eye(5, device='cuda')[torch.randint(0, 5, (B, n), device='cuda')])
    assert q.shape == (B, 1) and bool(torch.isfinite(q).all())
for scen, B, shards in (('simple_spread', 1001, 3), ('simple_reference', 130, 2), ('simple_spread', 5, 4)):
    A = [5, 10] if scen == 'simple_reference' else 5
    D = 21 if scen == 'simple_reference' else 10
    hr = m.HostRollout(scen, B, m.FusedActor(random_state_dict(D, A, 1), seed=2), shards=shards, seed=2, max_episode_len=3)
    for _ in range(7):
        hr.step(lambda k, tr: float(tr.rew_np.sum()))
    hr.flush()
    hr.close()
# replay ring: scalar (odd N*D) and vector tile paths, the element-parallel gather of records over 16 KB; adds across
# the end of the ring, uniform samples, device indices out of range (clamped)
for n, D, cap, B in ((3, 7, 331, 203), (3, 10, 331, 203), (31, 67, 53, 37)):
    rng = np.random.RandomState(D)
    rb = m.DeviceReplayBuffer(cap, n, D, 5, seed=1)
    for _ in range(3):
        rb.add(rng.randn(B, n, D).astype(np.float32), rng.randint(0, 5, (B, n)), rng.randn(B, n).astype(np.float32),
               rng.randn(B, n, D).astype(np.float32), (rng.rand(B) < 0.5).astype(np.float32))
    o = rb.sample(129)
    assert bool(torch.isfinite(o[0]).all()) and bool(torch.isfinite(o[2]).all())
    idx = rb.make_index(1001)
    assert int(idx.min()) >= 0 and int(idx.max()) < len(rb)
    rb.sample_index(torch.tensor([-1, 0, cap - 1, cap, -10 * cap, 7], device='cuda'))
    rb.collect()
# rollouts into the ring at ragged sizes: the multi-step writer (synced envs, fused kernel) with and without
# recordings, the per-step path after a masked reset, and calls that wrap the ring
for scen, n, B, cap in (('simple_spread', None, 129, 300), ('simple_reference', None, 33, 1000), ('simple_spread', 6, 65, 100)):
    env = m.make_env(scen, n=n, num_envs=B, batched=True, seed=3, max_episode_len=3)
    A = [5, env.act_c] if env.act_c else 5
    actor = m.FusedActor(random_state_dict(env.obs_dim, A, 1), seed=3)
    rb = m.DeviceReplayBuffer(cap, env.n, env.obs_dim, A)
    env.reset()
    env.rollout(actor, 7, record=True, replay=rb)
    env.rollout(actor, 5, replay=rb)
    env.reset(mask=(torch.arange(B, device='cuda') % 2).to(torch.uint8))
    env.rollout(actor, 4, replay=rb)
    rb.collect()
# rollouts that record benchmark_data (info_i / info_f) at ragged sizes: the fused kernel, the per-step path (large
# team, FFMA actor, treasure) and the ring on both of its paths
for scen, n, B, impl in (('simple_spread', None, 129, 'auto'), ('simple_reference', None, 257, 'auto'),
                         ('simple_spread', 9, 41, 'auto'), ('simple_spread', None, 33, 'simt'),
                         ('fullobs_collect_treasure', None, 77, 'auto')):
    env = m.make_env(scen, n=n, num_envs=B, batched=True, seed=3, max_episode_len=3)
    A = [5, env.act_c] if env.act_c else 5
    actor = m.FusedActor(random_state_dict(env.obs_dim, A, 1), seed=3, impl=impl)
    rb = m.DeviceReplayBuffer(2 * B + 1, env.n, env.obs_dim, A)
    env.reset()
    env.rollout(actor, 5, record=True, info=True)
    env.rollout(actor, 4, replay=rb, info=True)
    env.reset(mask=(torch.arange(B, device='cuda') % 2).to(torch.uint8))
    env.rollout(actor, 4, replay=rb, info=True)
    rb.collect()
# weight loads from CUDA tensors: every actor image layout (tensor-core image written, D > 32 where it is not, the
# dense3 region past the staged blob), sources at 4 B-aligned offsets of one flat buffer; the critic with both heads
for D, A, model in ((10, 5, False), (21, [5, 10], False), (28, 5, True), (57, 5, True)):
    sd = random_state_dict(D, A, 4, model_head=model)
    flat = torch.empty(1 + sum(v.size for v in sd.values()), device='cuda')
    dev, off = {}, 1
    for k, v in sd.items():
        dev[k] = flat[off:off + v.size].view(v.shape)
        dev[k].copy_(torch.from_numpy(v))
        off += v.size
    actor = m.FusedActor(random_state_dict(D, A, 5, model_head=model))
    actor.load_state_dict(dev)
    actor.forward(torch.zeros((33, 1 if D > 32 else 2, D), device='cuda'), want_next_state=model)
for model in (False, True):
    rng = np.random.RandomState(1)
    csd = {'dense1.module.weight': rng.randn(64, 15), 'dense1.module.bias': rng.randn(64),
           'lstm.weight_ih_l0': rng.randn(256, 64), 'lstm.weight_hh_l0': rng.randn(256, 64),
           'lstm.bias_ih_l0': rng.randn(256), 'lstm.bias_hh_l0': rng.randn(256),
           'dense2.weight': rng.randn(1, 64), 'dense2.bias': rng.randn(1)}
    if model:
        csd['dense3.weight'], csd['dense3.bias'] = rng.randn(1, 64), rng.randn(1)
    critic = m.FusedCritic(csd, obs_dim=10)
    critic.load_state_dict({k: torch.from_numpy(v).float().cuda() for k, v in csd.items()})
    critic.forward(torch.zeros((17, 3, 10), device='cuda'), torch.zeros((17, 3, 5), device='cuda'))
    # the backward kernel and both gradient reductions at ragged sizes: one sample, a partial last CTA, 16 agents
    for B, N in ((1, 1), (17, 3), (1031, 16)):
        o = torch.randn((B, N, 10), device='cuda')
        a = torch.randn((B, N, 5), device='cuda')
        dq = torch.randn((B, 1), device='cuda')
        critic.backward(o, a, dq, torch.randn((B, 1), device='cuda') if model else None, want_obs=True)
    net = m.FusedCriticNetwork(15, 1, model=model).cuda()
    out = net(torch.randn((33, 3, 10), device='cuda'), torch.randn((33, 3, 5), device='cuda'))
    (out[0].sum() + out[1].sum() if model else out.sum()).backward()
# the actor backward and its reductions at ragged sizes for every head layout: one head, two heads, the model head
# with and without dnext_state, D = 64; one sample, a partial last CTA, 12 agents
for D, A, model in ((10, 5, False), (21, [5, 10], False), (16, 5, True), (64, [6, 10], True)):
    actor = m.FusedActor(random_state_dict(D, A, 7, model_head=model), impl='simt')
    width = sum(A) if isinstance(A, list) else A
    for B, N in ((1, 1), (17, 3), (1031, 12)):
        o = torch.randn((B, N, D), device='cuda')
        actor.backward(o, torch.randn((B, N, width), device='cuda'),
                       torch.randn((B, N, D), device='cuda') if model else None, want_obs=True)
        if model:
            actor.backward(o, torch.randn((B, N, width), device='cuda'), None, want_obs=True)
net = m.FusedActorNetwork(10, 5).cuda()
net(torch.randn((33, 3, 10), device='cuda')).sum().backward()
torch.cuda.synchronize()
print('sanitize target done')
