"""Cost of recording benchmark_data in a rollout: env.rollout(actor, 25) with and without info=True.

    python tools/bench_rollout_info.py [--quick] [--reps 7] [--parent DIR] [--out profiles/r3_rollout_info.jsonl]

info=True writes 4 (N + 1) + 4 bytes per env-step more (20 B at N = 3, 4 (N + 1) B for fullobs_collect_treasure, whose
info_f is not written).  Configurations: simple_spread N = 3 at 65,536 and 1,048,576 envs (the fused k_tc2 kernel),
N = 9 at 65,536 (tensor-core actor + step kernel per step) and fullobs_collect_treasure at 262,144 (the same per-step
loop).  Every timed call is T = 25 steps (one episode) from a reset done outside the timed window; the two variants are
alternated on the same env, CUDA events around each call, the median of the repeats kept.  The output buffers of a
variant are allocated once, outside the timed window, and passed through the C entry point, so both variants time
the rollout and nothing else.

With --parent DIR (a checkout of the parent commit, its library built), `bench.py --gpus 1 --no-extras` of this tree
and of DIR are run alternately, --bench-runs times each, and their `value` lines are reported in the same file.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import multiagent_rl_b200 as m  # noqa: E402
from multiagent_rl_b200 import _lib  # noqa: E402
from multiagent_rl_b200.networks import random_state_dict  # noqa: E402

T = 25
CONFIGS = [('simple_spread', 3, 65_536), ('simple_spread', 3, 1_048_576), ('simple_spread', 9, 65_536),
           ('fullobs_collect_treasure', None, 262_144)]
QUICK = [('simple_spread', 3, 4096), ('simple_spread', 9, 1024), ('fullobs_collect_treasure', None, 1024)]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or 'unknown'
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    return name, power


def one_config(scenario, n, B, reps):
    env = m.make_env(scenario, n=n, num_envs=B, batched=True, seed=5, max_episode_len=T)
    N, D = env.n, env.obs_dim
    actor = m.FusedActor(random_state_dict(D, 5, 1), seed=5)
    lib = _lib.load()
    info_i = torch.empty(T, B, N + 1, dtype=torch.int32, device='cuda')
    info_f = torch.empty(T, B, device='cuda') if scenario != 'fullobs_collect_treasure' else None
    stream = _lib.current_stream(env.device)

    def run(with_info):
        ii, fi = (info_i, info_f) if with_info else (None, None)
        _lib.check(lib.mpe_rollout(env._h, actor._h, T, C.c_uint64(0), None, None, None, None, _lib.ptr(ii),
                                   _lib.ptr(fi), stream), 'mpe_rollout')

    variants = [('plain', False), ('info', True)]
    for _, w in variants:  # warm-up: module loads, scratch allocations
        env.reset()
        run(w)
    torch.cuda.synchronize()
    times = {k: [] for k, _ in variants}
    for _ in range(reps):
        for k, w in variants:
            env.reset()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run(w)
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1))
    extra = 4 * (N + 1) + (4 if info_f is not None else 0)
    del env, info_i, info_f
    torch.cuda.empty_cache()
    return N, times, extra


def bench_values(parent, runs, steps, warmup):
    """bench.py --no-extras of this tree and of `parent`, alternated; the `value` of every run."""
    out = {'this': [], 'parent': []}
    for _ in range(runs):
        for k, root in (('this', ROOT), ('parent', parent)):
            r = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--gpus', '1', '--steps', str(steps),
                                '--warmup', str(warmup), '--no-extras', '--cpu-seconds', '1'],
                               cwd=root, capture_output=True, text=True)
            if r.returncode != 0:
                raise SystemExit('bench.py in %s failed:\n%s' % (root, r.stderr[-3000:]))
            line = json.loads([x for x in r.stdout.splitlines() if x.startswith('{')][-1])
            out[k].append(line['value'])
            print(k, line['value'], flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--quick', action='store_true', help='small sizes (a smoke run of the tool)')
    ap.add_argument('--reps', type=int, default=7)
    ap.add_argument('--parent', default=None, help='checkout of the parent commit with its library built')
    ap.add_argument('--bench-runs', type=int, default=3)
    ap.add_argument('--bench-steps', type=int, default=2000)
    ap.add_argument('--bench-warmup', type=int, default=50)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_rollout_info needs a CUDA device')
    name, power = card()
    lines = []
    for scenario, n, B in (QUICK if a.quick else CONFIGS):
        N, times, extra = one_config(scenario, n, B, a.reps)
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        row = {'gpu': name, 'power_limit': power, 'scenario': scenario, 'N': N, 'envs': B, 'T': T, 'reps': a.reps,
               'path': 'fused k_tc2' if N in (2, 3) else 'actor + step kernels per step',
               'info_bytes_per_env_step': extra}
        for k, t in med.items():
            row[k + '_ms'] = round(t, 3)
            row[k + '_G_agent_steps_per_s'] = round(T * B * N / (t * 1e-3) / 1e9, 3)
            row[k + '_ms_all'] = [round(x, 3) for x in times[k]]
        row['info_overhead_pct'] = round((med['info'] / med['plain'] - 1) * 100, 2)
        print(json.dumps(row), flush=True)
        lines.append(row)
    if a.parent:
        vals = bench_values(os.path.abspath(a.parent), a.bench_runs, a.bench_steps, a.bench_warmup)
        row = {'gpu': name, 'power_limit': power, 'measurement': 'bench.py --gpus 1 --no-extras value, alternated',
               'steps': a.bench_steps, 'warmup': a.bench_warmup, 'unit': 'agent-steps/s',
               'this_build': vals['this'], 'parent_build': vals['parent']}
        print(json.dumps(row), flush=True)
        lines.append(row)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as fp:
            for row in lines:
                fp.write(json.dumps(row) + '\n')


if __name__ == '__main__':
    main()
