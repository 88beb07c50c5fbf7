"""Reloading actor / critic weights from a learner's CUDA state_dict: what the call costs the host and the device.

    python tools/bench_weight_load.py [--tree DIR] [--label NAME] [--reps 50] [--iters 60] [--quick] [--out FILE]

Per configuration (actor: simple_spread N = 3, simple_reference with heads [5, 10], simple_spread N = 12 with the
dense3 head; critic: simple_spread N = 3 and the "+model" critic of N = 12), ``load_state_dict`` of CUDA tensors as a
learner holds them (``ActorNetwork(...).cuda().state_dict()``; fp32 contiguous parameters):
  host_return_us  host time until the call returns, the GPU idle before it;
  host_block_us   the same with about 5 ms of GPU work (``torch.cuda._sleep``) enqueued just before the call: a call
                  that waits for the stream shows the wait here, one that only enqueues does not;
  device_us       CUDA events on the current stream around the call, the GPU idle before it.
Medians over ``--reps`` calls.  One loop row at 65,536 simple_spread N = 3 envs: per iteration
``env.rollout(actor, 25, replay=buf)``, one Adam step of ``ActorNetwork`` on a 1,024-transition sample of ``buf`` and
the reload; iterations are enqueued back to back without a synchronize, an event marks each iteration's start on the
stream, and the median gap between consecutive events is reported (host stalls that starve the GPU are in it).

``--tree`` imports ``multiagent_rl_b200`` from another checkout with its library built, so that two builds can be
compared by running this file once per build, alternating, in one session.  Rows are printed as JSON lines and
appended to ``--out``, with the GPU's name and power limit read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or 'unknown'
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    return name, power


def sleep_cycles(ms):
    """torch.cuda._sleep argument for about `ms` milliseconds on this GPU (calibrated with events)."""
    import torch
    torch.cuda._sleep(1_000_000)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 20_000_000
    e0.record()
    torch.cuda._sleep(n)
    e1.record()
    torch.cuda.synchronize()
    return int(n * ms / e0.elapsed_time(e1))


def time_load(load, reps, busy):
    import torch
    host, block, dev = [], [], []
    for _ in range(3):
        load()
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        load()
        host.append(time.perf_counter() - t0)
        torch.cuda.synchronize()
        torch.cuda._sleep(busy)
        t0 = time.perf_counter()
        load()
        block.append(time.perf_counter() - t0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        load()
        e1.record()
        torch.cuda.synchronize()
        dev.append(e0.elapsed_time(e1) * 1e-3)
    us = lambda x: round(statistics.median(x) * 1e6, 1)  # noqa: E731
    return {'host_return_us': us(host), 'host_block_us': us(block), 'device_us': us(dev)}


def critic_state_dict(D, A, model, seed):
    import numpy as np
    import torch
    rng = np.random.RandomState(seed)
    U = lambda *s: torch.from_numpy(rng.uniform(-0.1, 0.1, s).astype(np.float32)).cuda()  # noqa: E731
    sd = {'dense1.module.weight': U(64, D + A), 'dense1.module.bias': U(64), 'lstm.weight_ih_l0': U(256, 64),
          'lstm.weight_hh_l0': U(256, 64), 'lstm.bias_ih_l0': U(256), 'lstm.bias_hh_l0': U(256),
          'dense2.weight': U(1, 64), 'dense2.bias': U(1)}
    if model:
        sd['dense3.weight'], sd['dense3.bias'] = U(1, 64), U(1)
    return sd


def loop_row(m, envs, iters):
    import torch
    torch.manual_seed(0)
    T, N, D = 25, 3, 10
    env = m.make_env('simple_spread', n=N, num_envs=envs, batched=True, seed=1, max_episode_len=T)
    net = m.ActorNetwork(D, 5).cuda()
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    actor = m.FusedActor(net.state_dict(), seed=1)
    buf = m.DeviceReplayBuffer(T * envs, N, D, 5, seed=1)
    env.reset()

    def iteration(t):
        env.rollout(actor, T, step0=t * T, replay=buf)
        obs, act, _, _, _ = buf.sample(1024)
        loss = torch.nn.functional.cross_entropy(net(obs).reshape(-1, 5), act.argmax(-1).reshape(-1))
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        actor.load_state_dict(net.state_dict())

    for t in range(5):
        iteration(t)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(iters + 1)]
    for t in range(iters):
        ev[t].record()
        iteration(5 + t)
    ev[iters].record()
    torch.cuda.synchronize()
    gaps = [ev[i].elapsed_time(ev[i + 1]) for i in range(iters)]
    return {'kind': 'loop', 'config': 'simple_spread N=3 rollout(T=25, replay) + Adam step (batch 1024) + reload',
            'envs': envs, 'iters': iters, 'median_ms': round(statistics.median(gaps), 3),
            'min_ms': round(min(gaps), 3), 'max_ms': round(max(gaps), 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--tree', default=ROOT, help='checkout whose multiagent_rl_b200 (with its built library) is timed')
    ap.add_argument('--label', default=None)
    ap.add_argument('--reps', type=int, default=50)
    ap.add_argument('--iters', type=int, default=60)
    ap.add_argument('--quick', action='store_true', help='small sizes (a smoke run of the tool)')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    sys.path.insert(0, os.path.abspath(a.tree))
    import torch
    import multiagent_rl_b200 as m
    from multiagent_rl_b200.networks import ActorNetwork
    if not torch.cuda.is_available():
        raise SystemExit('bench_weight_load needs a CUDA device')
    name, power = card()
    base = {'gpu': name, 'power_limit': power, 'label': a.label or os.path.basename(os.path.abspath(a.tree))}
    reps = 5 if a.quick else a.reps
    busy = sleep_cycles(5.0)
    rows = []
    for cfg, D, A, model in (('actor simple_spread N=3', 10, 5, False), ('actor simple_reference [5,10]', 21, [5, 10], False),
                             ('actor simple_spread N=12 +model', 28, 5, True)):
        sd = ActorNetwork(D, A, model_head=model).cuda().state_dict()
        actor = m.FusedActor(sd, seed=1)
        rows.append(dict(base, kind='actor', config=cfg, **time_load(lambda: actor.load_state_dict(sd), reps, busy)))
    for cfg, D, model in (('critic simple_spread N=3', 10, False), ('critic +model N=12', 28, True)):
        sd = critic_state_dict(D, 5, model, 1)
        critic = m.FusedCritic(sd, obs_dim=D)
        rows.append(dict(base, kind='critic', config=cfg, **time_load(lambda: critic.load_state_dict(sd), reps, busy)))
    rows.append(dict(base, **loop_row(m, 4096 if a.quick else 65536, 10 if a.quick else max(50, a.iters))))
    for r in rows:
        print(json.dumps(r))
    if a.out:
        with open(a.out, 'a') as fp:
            for r in rows:
                fp.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
