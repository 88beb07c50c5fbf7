"""Short, fixed workload for ncu captures (run under gpurun; see profiles/README.md):
5 launches each of the env-only step kernel at 1,048,576 envs, the fused rollout kernel (T=1) at
65,536 envs and the actor-forward kernel at 65,536 envs, simple_spread N=3, plus the N=6/12 steps."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import multiagent_rl_b200 as m  # noqa: E402
from multiagent_rl_b200.networks import random_state_dict  # noqa: E402

which = sys.argv[1] if len(sys.argv) > 1 else 'all'
dev = torch.device('cuda:0')
actor = m.FusedActor(random_state_dict(10, 5, 12345678), device=dev, seed=1)
if which in ('all', 'step'):
    B = 1 << 20
    env = m.make_env('simple_spread', num_envs=B, batched=True, seed=1)
    env.reset()
    act = torch.randint(0, 5, (B, 3), dtype=torch.int32, device=dev)
    # four rotating output sets (566 MB > the 126 MB L2): a launch's output lines are written back to DRAM instead of
    # being overwritten in L2 by the next launch, so ncu's dram__bytes is the traffic the byte model counts
    outs = [(torch.empty((B, 3, 10), device=dev), torch.empty((B, 3), device=dev),
             torch.empty((B, 3), dtype=torch.uint8, device=dev)) for _ in range(4)]
    for i in range(8):
        env.step(act, out=outs[i % 4])
    torch.cuda.synchronize()
if which in ('all', 'rollout', 'actor'):
    B = 65536
    env = m.make_env('simple_spread', num_envs=B, batched=True, seed=1)
    obs = env.reset()
    if which != 'actor':
        for _ in range(5):
            env.rollout(actor, 1, record=True)
    if which != 'rollout':
        for _ in range(5):
            actor.forward(obs)
    torch.cuda.synchronize()
if which in ('all', 'bign'):
    actor6 = m.FusedActor(random_state_dict(16, 5, 1), device=dev, seed=1)
    env6 = m.make_env('simple_spread', n=6, num_envs=65536, batched=True, seed=1)
    obs6 = env6.reset()
    for _ in range(3):
        actor6.forward(obs6)
    torch.cuda.synchronize()
    for n, D in ((6, 16), (12, 28)):
        B = 1 << 18
        env = m.make_env('simple_spread', n=n, num_envs=B, batched=True, seed=1)
        env.reset()
        act = torch.randint(0, 5, (B, n), dtype=torch.int32, device=dev)
        for _ in range(3):
            env.step(act)
        torch.cuda.synchronize()
if which == 'critic':
    import numpy as np
    rng = np.random.RandomState(0)
    D, N, B = 10, 3, 65536
    csd = {'dense1.module.weight': rng.randn(64, D + 5).astype(np.float32) * 0.1, 'dense1.module.bias': np.zeros(64, np.float32),
           'lstm.weight_ih_l0': rng.randn(256, 64).astype(np.float32) * 0.1, 'lstm.weight_hh_l0': rng.randn(256, 64).astype(np.float32) * 0.1,
           'lstm.bias_ih_l0': np.zeros(256, np.float32), 'lstm.bias_hh_l0': np.zeros(256, np.float32),
           'dense2.weight': rng.randn(1, 64).astype(np.float32), 'dense2.bias': np.zeros(1, np.float32)}
    critic = m.FusedCritic(csd, obs_dim=D)
    obs = torch.randn((B, N, D), device=dev)
    act = torch.eye(5, device=dev)[torch.randint(0, 5, (B, N), device=dev)]
    for _ in range(3):
        critic.forward(obs, act)
    am = m.FusedActor(random_state_dict(16, 5, 1, model_head=True), device=dev, seed=1)
    o6 = torch.randn((B, 6, 16), device=dev)
    for _ in range(2):
        am.forward(o6, want_next_state=True)
    torch.cuda.synchronize()
if which == 'treasure':
    B = 1 << 18
    env = m.make_env('fullobs_collect_treasure', num_envs=B, batched=True, seed=1)
    env.reset()
    act = torch.randint(0, 5, (B, 8), dtype=torch.int32, device=dev)
    outs = [(torch.empty((B, 8, 30), device=dev), torch.empty((B, 8), device=dev),
             torch.empty((B, 8), dtype=torch.uint8, device=dev)) for _ in range(3)]
    for i in range(6):
        env.step(act, out=outs[i % 3])
    torch.cuda.synchronize()
print('profile target done')
