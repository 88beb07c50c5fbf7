"""Fused rollout (mpe_rollout, T=25 per call) across scenarios / team sizes: ms per env step and G agent-steps/s."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import multiagent_rl_b200 as m  # noqa: E402
from multiagent_rl_b200.networks import random_state_dict  # noqa: E402


def _gpu_spin(torch, cycles=20_000_000):
    """~10 ms of GPU-side spinning before a timed launch loop, so that the host enqueues ahead of the GPU and the
    kernels run back to back (torch.cuda._sleep is a private helper: skipped quietly where it does not exist)."""
    spin = getattr(torch.cuda, '_sleep', None)
    if spin is not None:
        spin(cycles)

CONFIGS = [('simple_spread', None, 65536), ('simple_spread', 6, 65536), ('simple_spread', 9, 32768),
           ('simple_spread', 12, 32768), ('simple_reference', None, 65536), ('simple_speaker_listener', None, 65536),
           ('fullobs_collect_treasure', None, 32768)]
# SURVEY 8d configs 3-5: the same at 1,048,576 envs per GPU (no tail quantisation: thousands of tile pairs per SM)
CONFIGS += [(s, n, 1 << 20 if s != 'fullobs_collect_treasure' else 1 << 19) for s, n, _ in CONFIGS]
IMPL = sys.argv[1] if len(sys.argv) > 1 else 'auto'  # a key of FusedActor.IMPLS: 'auto', 'simt' or 'tc'
for scen, n, B in CONFIGS:
    env = m.make_env(scen, n=n, num_envs=B, batched=True, seed=1, max_episode_len=25)
    A = [5, 10] if scen == 'simple_reference' else 5
    actor = m.FusedActor(random_state_dict(env.obs_dim, A, 1), seed=1, impl=IMPL)
    env.reset()
    T = 25
    env.rollout(actor, T)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    _gpu_spin(torch)  # ~10 ms GPU spin: the timed launches below are all queued before the first one starts
    e0.record()
    for _ in range(4):
        env.rollout(actor, T)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / (4 * T)
    print(json.dumps({'scenario': scen, 'N': env.n, 'envs': B, 'impl': IMPL, 'ms_per_env_step': round(ms, 4),
                      'G_agent_steps_per_s': round(B * env.n / ms / 1e6, 3)}))
    del env, actor
