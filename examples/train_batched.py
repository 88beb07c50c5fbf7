"""Batched training loop: thousands of particle envs on the GPU feeding the REFERENCE's own learner.

What runs where:
  * acting + env stepping: `env.rollout(fused_actor, 25, record=True, replay=memory)` - one fused CUDA kernel per
    episode (experiments/run.py:36-65 for B envs at once) and one launch that appends its transitions to the ring;
  * replay: `DeviceReplayBuffer` (the reference ReplayBuffer's surface, rls/replay_buffer.py:9-91) - transitions
    never leave HBM;
  * learning: the reference's `Trainer.optimize()` (rls/agent/multiagent/ddpg_gumbel_fix.py:131-219) UNCHANGED, with the
    device replay as its `memory`; after every update the fused actor reloads the weights.  With `--fused-critic` the
    learner's critic is `FusedCriticNetwork`, whose forward and backward are the critic kernels; with `--fused-actor`
    the learner's actor is `FusedActorNetwork`, whose forward and backward are the actor kernels.

Needs the reference on the import path (PYTHONPATH=/path/to/multiagent_rl, or the compiled copy `python -m
oracle.build_ref` leaves in oracle/_ref).  Example:

    python examples/train_batched.py --envs 4096 --episodes 20
"""
import argparse
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import multiagent_rl_b200 as m  # noqa: E402


def import_reference():
    try:
        import rls  # noqa: F401 - the reference tree is on the path
    except ImportError:
        from oracle import build_ref  # examples / tests only: the byte-compiled reference
        build_ref.add_to_path()
    from rls import arglist
    from rls.agent.multiagent.ddpg_gumbel_fix import Trainer
    from rls.model.ac_network_multi_gumbel import ActorNetwork, CriticNetwork
    return arglist, Trainer, ActorNetwork, CriticNetwork


def train(num_envs=4096, episodes=20, updates_per_episode=4, scenario='simple_spread', n=None, seed=12345678,
          batch_size=1024, lr=1e-2, log=print, fused_critic=False, fused_actor=False):
    arglist, Trainer, ActorNetwork, CriticNetwork = import_reference()
    arglist.actor_learning_rate = arglist.critic_learning_rate = lr   # main.py:34-35
    arglist.batch_size = batch_size
    torch.manual_seed(seed)
    np.random.seed(seed)
    T = arglist.max_episode_len
    env = m.make_env(scenario, n=n, num_envs=num_envs, batched=True, seed=seed, max_episode_len=T)
    N, D = env.n, env.obs_dim
    A = 5
    actor = (m.FusedActorNetwork if fused_actor else ActorNetwork)(D, A)
    critic = (m.FusedCriticNetwork if fused_critic else CriticNetwork)(D + A, 1)
    memory = m.DeviceReplayBuffer(max(1_000_000, 2 * num_envs * T), N, D, A, seed=seed)
    learner = Trainer(actor, critic, memory, action_type='Discrete')        # the reference's class, cuda:0
    fused = m.FusedActor(learner.actor.state_dict(), seed=seed)
    hist = m.EpisodeHistory.for_env(env)
    returns = []
    t0 = time.time()
    for ep in range(episodes):
        env.reset()
        # T * B transitions go straight into the replay ring; rew [T,B,N] is kept for the episode history
        _, rew, _, _ = env.rollout(fused, T, step0=ep * T, record=True, replay=memory)
        hist.add_rollout(rew)
        returns.append(float(rew.sum((0, 2)).mean()))
        if len(memory) >= batch_size:
            for _ in range(updates_per_episode):
                learner.optimize()                                           # reference code, device replay
            fused.load_state_dict(learner.actor.state_dict())  # CUDA parameters: packed on the device, in stream order
        log('episode %d: mean return %.2f over %d envs, %d transitions in replay, %.1f s'
            % (ep, returns[-1], num_envs, len(memory), time.time() - t0))
    return returns, learner, hist


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--envs', type=int, default=4096)
    ap.add_argument('--episodes', type=int, default=20)
    ap.add_argument('--scenario', default='simple_spread')
    ap.add_argument('--n', type=int, default=None)
    ap.add_argument('--fused-critic', action='store_true', help='train the critic through the CUDA kernels')
    ap.add_argument('--fused-actor', action='store_true', help='train the actor through the CUDA kernels')
    a = ap.parse_args()
    train(a.envs, a.episodes, scenario=a.scenario, n=a.n, fused_critic=a.fused_critic, fused_actor=a.fused_actor)
