"""Rollout into the device replay ring: today's caller-side pattern against rollout(replay=...) on each path.

    python tools/bench_rollout_replay.py [--quick] [--out profiles/rollout_replay.jsonl]

(a) ``record``: rollout(record=True), torch.cat of the shifted observations, T x replay.add - what a caller did before
    the ring could be filled by the rollout (correct only for a call that starts at an episode start and spans one
    episode, which is what is timed here);
(b) ``replay_fused``: rollout(replay=buf) on synced envs (fused kernel + one ring-writer launch per segment), teams of
    2 / 3 on the tensor cores only;
(c) ``replay_stepwise``: rollout(replay=buf) on the same envs after a masked reset of every env (the envs are the same,
    the host no longer knows that their episodes are aligned): actor + step kernels and one replay_add per step; on
    such envs the loop also launches the reset kernel after every step, not only at the episode end, so this column
    carries 24 reset launches a per-step run on aligned envs would not;
(d) ``plain``: rollout() without recordings or ring, the floor.
Every timed call is T = 25 steps (one episode) from a fresh reset, done outside the timed window; the ring holds
T * B transitions, so every variant writes all of them (the fused writer skips nothing).  CUDA events around each call,
variants alternated, the median of the repeats kept.  The ring writer's share of HBM comes from a separate
torch.profiler run of (b) / (c): algorithmic bytes (record written, obs_t / obs_t+1 / actions / rewards read) over the
writer kernels' summed time.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import multiagent_rl_b200 as m  # noqa: E402
from multiagent_rl_b200.networks import random_state_dict  # noqa: E402

T = 25


def card():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or 'unknown'
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    return name, power


def hbm_peak():
    p = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return json.load(open(p))['hbm_gbs'], 'MEASURED_PEAKS.json'
    return 6528.4, 'copy-kernel measurement of tools/bench_replay.py'


def one_config(scenario, n, B, reps):
    env = m.make_env(scenario, n=n, num_envs=B, batched=True, seed=5, max_episode_len=T)
    N, D, act_c = env.n, env.obs_dim, env.act_c
    heads = [5, act_c] if act_c else 5
    actor = m.FusedActor(random_state_dict(D, heads, 1), seed=5)
    buf = m.DeviceReplayBuffer(T * B, N, D, heads)  # nothing is overwritten within one call
    fused_ok = N in (2, 3)
    all_envs = torch.ones(B, dtype=torch.uint8, device='cuda')

    state = {}

    def p_reset():
        state['obs0'] = env.reset()

    def p_unsync():
        env.reset()
        env.reset(mask=all_envs)  # same envs, but the host no longer knows their episodes are aligned

    def v_record():
        obs0 = state['obs0']
        obs_next, rew, au, ac = env.rollout(actor, T, step0=0, record=True)
        obs_t = torch.cat([obs0[None], obs_next[:-1]], 0)
        for t in range(T):
            buf.add(obs_t[t], au[t], rew[t], obs_next[t], act_c=None if ac is None else ac[t])

    def v_replay():
        env.rollout(actor, T, step0=0, replay=buf)

    def v_plain():
        env.rollout(actor, T, step0=0)

    variants = [('record', p_reset, v_record)] + ([('replay_fused', p_reset, v_replay)] if fused_ok else []) + \
               [('replay_stepwise', p_unsync, v_replay), ('plain', p_reset, v_plain)]
    times = {k: [] for k, _, _ in variants}
    for _, prep, fn in variants:  # warm-up: module loads, scratch allocations, caching allocator
        prep()
        fn()
    torch.cuda.synchronize()
    for _ in range(reps):
        for k, prep, fn in variants:
            prep()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) * 1e-3)
            torch.cuda.empty_cache()
    # writer kernels' time in a profiled call of each replay path
    writer = {}
    for k, prep, kern in (('replay_fused', p_reset, 'k_replay_add_steps'), ('replay_stepwise', p_unsync, 'k_replay_add')):
        if k not in times:
            continue
        prep()
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            v_replay()
            torch.cuda.synchronize()
        us = sum(e.device_time_total for e in prof.key_averages()
                 if kern in e.key and (kern != 'k_replay_add' or 'steps' not in e.key))
        writer[k] = us * 1e-6
    rec = (N * D * 8 + 8 + 2 * N + 15) // 16 * 16  # ReplayDev::record_bytes (256 B for N = 3, D = 10)
    per_tr = rec + 2 * N * D * 4 + N * 4 * (2 if act_c else 1) + N * 4  # + obs_t, obs_t+1, actions, rewards read
    del buf, env
    torch.cuda.empty_cache()
    return N, D, times, writer, per_tr


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--quick', action='store_true', help='small sizes (a smoke run of the tool)')
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_rollout_replay needs a CUDA device')
    name, power = card()
    peak, peak_src = hbm_peak()
    sizes = (4096,) if a.quick else (65_536, 1_048_576)
    lines = []
    for scenario, n in (('simple_spread', 3), ('simple_spread', 9), ('fullobs_collect_treasure', None)):
        for B in sizes:
            N, D, times, writer, per_tr = one_config(scenario, n, B, a.reps)
            med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
            row = {'gpu': name, 'power_limit': power, 'scenario': scenario, 'N': N, 'D': D, 'envs': B, 'T': T,
                   'reps': a.reps}
            for k, t in med.items():
                row[k + '_ms'] = round(t * 1e3, 3)
                row[k + '_G_agent_steps_per_s'] = round(T * B * N / t / 1e9, 3)
            for k, t in writer.items():
                gbs = T * B * per_tr / t / 1e9
                row[k + '_writer_ms'] = round(t * 1e3, 3)
                row[k + '_writer_GBps'] = round(gbs, 1)
                row[k + '_writer_frac_of_measured_hbm'] = round(gbs / peak, 3)
            row['writer_bytes_per_transition'] = per_tr
            row['hbm_peak_GBps'] = peak
            row['hbm_peak_source'] = peak_src
            print(json.dumps(row), flush=True)
            lines.append(row)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as fp:
            for row in lines:
                fp.write(json.dumps(row) + '\n')


if __name__ == '__main__':
    main()
