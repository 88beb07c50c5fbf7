"""bench.py - agent-steps/sec of the fused MPE step + observe + reward + actor path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs B_per_gpu] [--impl reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  Workload = BASELINE.json configs[1]: simple_spread, N = L = 3,
65,536 env instances per GPU, one launch of the fused kernel (observe -> actor forward -> hard Gumbel
sample -> World.step -> reward -> auto-reset every 25 steps) per "step"; weak scaling (per-GPU
work fixed).  See DESIGN.md "Measurement" for how every field is derived.

--dump-outputs DIR writes what the last timed step returned (obs_next, rew, act of rank 0) as DIR/<name>.npy.
The env, the actor weights and the sampling noise are seeded, so two builds run with the same arguments can be
compared output for output.  The bench writes nothing into the source tree (no bytecode either).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # the bench writes nothing into the tree: tools/ and oracle/ modules build() never
#                                 imported would otherwise leave __pycache__ directories there
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _gpu_spin(torch, cycles=20_000_000):
    """~10 ms of GPU-side spinning before a timed launch loop, so that the host enqueues ahead of the GPU and the
    kernels run back to back (torch.cuda._sleep is a private helper: skipped quietly where it does not exist)."""
    spin = getattr(torch.cuda, '_sleep', None)
    if spin is not None:
        spin(cycles)

SCENARIO, N_AGENTS, OBS_DIM, ACT_DIM, EP_LEN = 'simple_spread', 3, 10, 5, 25
SEED = 12345678  # main.py:41
# algorithmic bytes of one env step (SURVEY.md 8d): 41N + 8L + 4ND with N = L = 3, D = 10
BYTES_PER_ENV_STEP = 41 * 3 + 8 * 3 + 4 * 3 * 10
# algorithmic FLOPs of one actor forward per env (SURVEY.md 8d): N (128 D + 49152 + 128 A)
# DRAM traffic per launch of the two kernels the rooflines are quoted for, from the committed ncu --set full captures
NCU_DRAM_BYTES_FUSED = 5.455e6   # k_tc2<0,3,1,8>, 65,536 envs: 5.455 MB read + 0 written (outputs stay in the 126 MB L2)
NCU_DRAM_BYTES_STEP = 221.9e6    # k_step<float,0,3>, 1,048,576 envs, rotating outputs: 88.1 MB read + 133.8 MB written
#   inside the kernel's window (algorithmic 88 + 192 MB: ~58 MB of dirty lines are still in L2 when the kernel ends
#   and ncu flushes before the next replay; back to back they are written during the next launch)
# MUFU (XU pipe) warp instructions per launch of k_tc2<0,3,1,8> at 65,536 envs: smsp__inst_executed_pipe_xu.sum in
# profiles/r2_ncu_tc2_counters.txt = 989 transcendental evaluations per env step; XU issue rate 0.5 warp inst / clk / SM
NCU_XU_WARP_INST_FUSED = 2025472
XU_WARP_INST_PER_CLK_PER_SM = 0.5
# all warp instructions per launch of the same kernel (smsp__inst_executed.sum, same file); issue rate 1 / clk / sub-partition
NCU_WARP_INST_FUSED = 26181167
FLOPS_PER_ENV_STEP = N_AGENTS * (128 * OBS_DIM + 49152 + 128 * ACT_DIM)
FP32_SIMT_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12  # FFMA peak at max clock (not a measured number)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=2000)
    ap.add_argument('--warmup', type=int, default=50)
    ap.add_argument('--envs', type=int, default=None,
                    help='env instances per GPU (default: 65,536 at --gpus 1 = BASELINE configs[1]; 131,072 at '
                         '--gpus N > 1, so that 8 GPUs carry configs[4]\'s >= 1M envs)')
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--cpu-seconds', type=float, default=12.0, help='budget of the cpu_baseline sample')
    ap.add_argument('--no-extras', action='store_true', help='skip the env-only / 1M-env side measurements')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step as DIR/<name>.npy (float32)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200')
    return args


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Each array (env rows first) as out_dir/<name>.npy in float32; the action indices 0..4 are exact in it.  Above
    DUMP_MAX_BYTES in all, the same fixed, seeded sample of env rows is kept from every array, and its row numbers go
    to out_dir/env_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    rows = next(iter(arrays.values())).shape[0]
    row_bytes = sum(4 * a[0].numel() for a in arrays.values())
    keep = min(rows, (DUMP_MAX_BYTES - 8 * rows) // row_bytes)
    idx = None
    if keep < rows:
        idx = np.sort(np.random.RandomState(0).choice(rows, keep, replace=False))
        np.save(os.path.join(out_dir, 'env_index.npy'), idx.astype(np.float64))
    for name, a in arrays.items():
        a = a.detach().float().cpu().numpy()
        np.save(os.path.join(out_dir, name + '.npy'), a if idx is None else a[idx])


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return {'hbm_gbs': d['hbm_gbs'], 'bf16_tflops': d['bf16_tflops'],
                'bf16_tflops_sustained': d.get('bf16_tflops_sustained', d['bf16_tflops']), 'source': 'measured'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback'}


# --------------------------------------------------------------------------------------------------
# CPU arm: the reference's loop body (experiments/run.py:36-65 without replay/optimize) on the oracle
# --------------------------------------------------------------------------------------------------
def cpu_loop(n_env_steps, seed, threads=1):
    """Runs the reference-shaped rollout loop on the CPU oracle; returns (agent_steps, seconds)."""
    import torch
    import torch.nn.functional as F
    from oracle import build_ref, mpe_ref
    if build_ref.available():  # the reference's own ActorNetwork (rls/model/ac_network_multi_gumbel.py:24-67), compiled
        build_ref.add_to_path()  # into oracle/_ref by `python -m oracle.build_ref`
        from rls.model.ac_network_multi_gumbel import ActorNetwork
    else:
        from multiagent_rl_b200.networks import ActorNetwork  # same layers and parameter names, this repo's mirror
    torch.set_num_threads(threads)
    np.random.seed(seed)
    torch.manual_seed(seed)
    env = mpe_ref.make_env(SCENARIO)
    actor = ActorNetwork(OBS_DIM, ACT_DIM)
    obs_n = env.reset()
    episode_step = 0
    t0 = time.perf_counter()
    for _ in range(n_env_steps):
        state = torch.from_numpy(np.array([np.stack(obs_n)], dtype='float32'))  # process_obs
        with torch.no_grad():
            logits = actor(state)
        a = F.gumbel_softmax(logits.view(N_AGENTS, ACT_DIM), hard=True).view(1, N_AGENTS, ACT_DIM).numpy()
        action_n_env = [np.array(x) for x in a[0].tolist()]
        obs_n, rew_n, done_n, _ = env.step(action_n_env)
        _ = np.sum(rew_n)
        episode_step += 1
        if all(done_n) or episode_step >= EP_LEN:
            obs_n = env.reset()
            episode_step = 0
    return n_env_steps * N_AGENTS, time.perf_counter() - t0


def _cpu_worker(args):
    n, seed = args
    return cpu_loop(n, seed, threads=1)


def _cpu_actor_kind():
    """Which ActorNetwork cpu_loop imports: the reference's own class when oracle/_ref was built."""
    have = os.path.exists(os.path.join(ROOT, 'oracle', '_ref', 'rls', 'model', 'ac_network_multi_gumbel.refpyc'))
    return 'reference ActorNetwork (oracle/_ref)' if have else 'torch mirror of the reference ActorNetwork'


def cpu_baseline(seconds):
    """1 core, bounded sample of the same workload (rank 0, N = 1 only)."""
    cpu_loop(100, SEED)  # warm-up
    _, dt = cpu_loop(300, SEED)
    n = max(500, int(300 * seconds / max(dt, 1e-6)))
    steps, dt = cpu_loop(n, SEED)
    return {'value': steps / dt, 'unit': 'agent-steps/s', 'cores': 1, 'kind': 'port',
            'sample': '%d env steps (25-step episodes) of the float64 loop oracle + %s on torch CPU + '
                      'F.gumbel_softmax, 1 thread, %.1f s' % (n, _cpu_actor_kind(), dt)}


def run_reference(args):
    """--impl reference: the reference's own (Python/numpy + torch CPU) implementation of the path,
    restated in oracle/ because the physics package is not vendored, on all host cores."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    ctx = mp.get_context('fork')
    with ctx.Pool(cores) as pool:
        t0 = time.perf_counter()
        for _ in range(max(args.warmup, 1)):
            pool.map(_cpu_worker, [(20, SEED + i) for i in range(cores)])
        rate = 20 * max(args.warmup, 1) / (time.perf_counter() - t0)  # env steps / s / process
        # bounded sample: env steps per process per bench step, sized so that K steps take <= ~90 s
        per_step = int(max(5, min(150, rate * 90.0 / max(args.steps, 1))))
        t0 = time.perf_counter()
        total = 0
        for k in range(args.steps):
            res = pool.map(_cpu_worker, [(per_step, SEED + k * cores + i) for i in range(cores)])
            total += sum(r[0] for r in res)
        dt = time.perf_counter() - t0
    val = total / dt
    line = {
        'impl': 'reference', 'metric': 'agent-steps/sec', 'value': val, 'unit': 'agent-steps/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': 'simple_spread N=3 L=3 D=10 A=5, 25-step episodes, act+step loop '
                               '(experiments/run.py:36-65), %d independent CPU processes x %d env steps per bench step'
                               % (cores, per_step)},
        'cpu_baseline': {'value': val, 'unit': 'agent-steps/s', 'cores': cores, 'kind': 'port',
                         'sample': '%d processes x %d steps x %d env steps; env = float64 loop oracle (the physics package '
                                   'is not in the reference tree), actor = %s' % (cores, args.steps, per_step, _cpu_actor_kind())},
        'e2e': {'value': val, 'unit': 'agent-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# clocks sampler
# --------------------------------------------------------------------------------------------------
class Clocks(object):
    """Samples SM clock and clock-event (throttle) reasons of one GPU through NVML from a thread,
    every few ms, between start() and stop() - i.e. DURING the timed region."""
    REASONS = {0x8: 'hw_slowdown', 0x40: 'hw_thermal_slowdown', 0x20: 'sw_thermal_slowdown', 0x4: 'sw_power_cap',
               0x80: 'hw_power_brake_slowdown'}

    def __init__(self, index, period_s=0.004):
        self.index, self.period = index, period_s
        self.sm, self.reasons, self.power = [], set(), []
        self.sm_max = None
        self._stop = threading.Event()
        self._thr = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001 - any NVML failure just leaves the record empty
            self.err = repr(e)
            return
        self._thr = threading.Thread(target=self._loop, daemon=True)
        self._thr.start()

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception as e:  # noqa: BLE001
                self.err = repr(e)
                return
            time.sleep(self.period)

    def stop(self):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=1.0)
        out = {'sm_mhz': float(np.median(self.sm)) if self.sm else None, 'sm_max_mhz': self.sm_max,
               'reasons': sorted(self.reasons), 'samples': len(self.sm),
               'power_w_max': max(self.power) if self.power else None, 'source': 'nvml, sampled inside the timed region'}
        if self.err:
            out['error'] = self.err
        return out


def _lib_stats_len():
    from multiagent_rl_b200 import _lib
    return _lib.STATS_LEN


def physical_gpu_index(local_rank):
    vis = os.environ.get('CUDA_VISIBLE_DEVICES')
    if vis:
        try:
            return int(vis.split(',')[local_rank])
        except (ValueError, IndexError):
            pass
    return local_rank


# --------------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    import multiagent_rl_b200 as m
    from multiagent_rl_b200 import distributed as D
    from multiagent_rl_b200.networks import random_state_dict  # reference architecture, default-init distribution

    rank, world, local = D.init_from_env()
    if world != args.gpus:
        raise SystemExit('--gpus %d but WORLD_SIZE=%d (launch with torchrun)' % (args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    numa_cores = D.bind_to_gpu_numa(physical_gpu_index(local))  # before any pinned allocation (first touch)
    B = args.envs if args.envs else (65536 if world == 1 else 131072)
    off = rank * B
    pk = peaks()

    env = m.make_env(SCENARIO, num_envs=B, batched=True, seed=SEED, env_id_offset=off, max_episode_len=EP_LEN)
    actor = m.FusedActor(random_state_dict(OBS_DIM, ACT_DIM, SEED), device=dev, seed=SEED)
    env.reset()
    # per-step outputs of the fused kernel (what a replay writer consumes)
    obs_next = torch.empty((1, B, N_AGENTS, OBS_DIM), device=dev)
    rew = torch.empty((1, B, N_AGENTS), device=dev)
    act = torch.empty((1, B, N_AGENTS), dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stats = torch.zeros(_lib_stats_len(), dtype=torch.float64, device=dev)
    stats_dev = env.stats_tensor()  # aliases the device statistics of this shard
    from multiagent_rl_b200 import _lib
    lib = _lib.load()

    def fused_step(t):
        _lib.check(lib.mpe_rollout(env._h, actor._h, 1, t, _lib.ptr(obs_next), _lib.ptr(rew), _lib.ptr(act), None,
                                   _lib.current_stream(dev)), 'mpe_rollout')

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # The path's only collective - the all-reduce of the episode-return statistics, once per episode - runs on a SIDE
    # stream behind an event, never on the step stream (SURVEY 8e: nothing on the per-step path).
    side = torch.cuda.Stream(device=dev)
    reduces = [0]

    def reduce_stats_off_stream():
        ready = torch.cuda.Event()
        ready.record()
        with torch.cuda.stream(side):
            side.wait_event(ready)
            stats.copy_(stats_dev, non_blocking=True)
            dist.all_reduce(stats)
        reduces[0] += 1

    t = 0
    for _ in range(max(args.warmup, 3)):
        flush.zero_()
        fused_step(t)
        t += 1
        if world > 1 and t % EP_LEN == 0:
            reduce_stats_off_stream()
    clocks = Clocks(physical_gpu_index(local))
    clocks.start()
    side.synchronize()
    sync_all()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches = 0
    _gpu_spin(torch)  # ~10 ms GPU spin (outside every event pair): the host enqueues ahead of the GPU, so no
    #                                event pair contains a wait for a launch that Python had not issued yet
    for k in range(args.steps):
        flush.zero_()  # L2 flush between timed iterations (outside the event pair)
        ev[k][0].record()
        fused_step(t)
        launches += 1
        t += 1
        ev[k][1].record()
        if world > 1 and t % EP_LEN == 0:
            reduce_stats_off_stream()
    side.synchronize()
    sync_all()
    per_step = [a.elapsed_time(b) for a, b in ev]
    if args.dump_outputs and rank == 0:  # 65,536 envs: 7.9 MB of observations, 0.8 MB each of rewards and actions
        dump_outputs(args.dump_outputs, {'obs_next': obs_next[0], 'rew': rew[0], 'act': act[0]})
    ms = sum(per_step)
    ms = D.max_over_ranks(ms, device=dev)
    clk = clocks.stop()
    stats_now = D.reduce_return_stats(env.read_stats(), device=dev)
    value = world * B * N_AGENTS * args.steps / (ms * 1e-3)
    kernel_s = ms * 1e-3 / args.steps
    tflops = B * FLOPS_PER_ENV_STEP / kernel_s / 1e12

    # ---- e2e: the reference-facing host-buffer path (get_exploration_action + env.step with HOST tensors).
    # Every step uploads every env's observations and actions and downloads its actions, observations, rewards and
    # dones.  HostRollout keeps `shards` independent shards in different phases on their own streams, so the two PCIe
    # directions are busy at the same time; the blocking pair (actor_forward_host + mpe_step_host) is timed beside it.
    rows = B * N_AGENTS
    e2e_steps = max(25, min(args.steps, 100))
    del env
    best = None
    for shards in (3, 4, 2, 1):  # 1 = one direction at a time: the better schedule when many ranks oversubscribe the host
        hr = m.HostRollout(SCENARIO, B, actor, shards=shards, seed=SEED, env_id_offset=off, device=dev,
                           max_episode_len=EP_LEN)
        seen = [0.0]

        def consume(k, tr, seen=seen):  # every step's result is read on the host: a slice of the rewards
            seen[0] += float(tr.rew_np[:64].sum())
        for _ in range(5):
            hr.step(consume)
        hr.flush(consume)
        sync_all()
        w0 = time.perf_counter()
        for k in range(e2e_steps):
            hr.step(consume)
        hr.flush(consume)
        wall = time.perf_counter() - w0
        sync_all()
        if best is None or wall < best[0]:
            best = (wall, shards)
        assert np.isfinite(seen[0])
        del hr
    e2e_ms = D.max_over_ranks(best[0] * 1e3, device=dev)
    resets = e2e_steps // EP_LEN
    e2e = {'value': world * rows * e2e_steps / (e2e_ms * 1e-3), 'unit': 'agent-steps/s',
           'h2d_bytes_per_step': rows * OBS_DIM * 4,
           'd2h_bytes_per_step': rows * 4 + rows * OBS_DIM * 4 + rows * 4 + rows + resets * rows * OBS_DIM * 4 // e2e_steps,
           'steps': e2e_steps, 'shards': best[1], 'depth': 2,
           'timing': 'host wall clock around K steps incl. delivering every step\'s results to the host callback, max over ranks',
           'api': 'HostRollout.step: mpe_act_step_host_async per shard on its own stream (H2D observations, actor, env '
                  'step, one D2H of {actions, observations, rewards, dones}), cudaHostAlloc host buffers, mpe_host_wait '
                  'before a shard\'s results are read'}
    # the blocking pair of calls, for comparison (what round 1 reported as e2e)
    env = m.make_env(SCENARIO, num_envs=B, batched=True, seed=SEED, env_id_offset=off, max_episode_len=EP_LEN)
    blk = _lib.HostBlock(rows * (OBS_DIM * 4 + 4 + 1 + 4) + 4096)  # cudaHostAlloc staging (not tensor.pin_memory())
    h_obs = blk.tensor((B, N_AGENTS, OBS_DIM), torch.float32)
    h_rew = blk.tensor((B, N_AGENTS), torch.float32)
    h_done = blk.tensor((B, N_AGENTS), torch.uint8)
    h_act = blk.tensor((B, N_AGENTS), torch.int32)
    h_obs.copy_(env.reset())
    for _ in range(3):
        actor.act_host(h_obs, step=t, env_id_offset=off, act_u=h_act)
        env.step_host(h_act, out=(h_obs, h_rew, h_done))
    sync_all()
    w0 = time.perf_counter()
    for k in range(25):
        actor.act_host(h_obs, step=t + k, env_id_offset=off, act_u=h_act)  # H2D obs, kernel, D2H actions
        env.step_host(h_act, out=(h_obs, h_rew, h_done))                  # H2D actions, kernel, D2H obs/rew/done
    blocking_ms = D.max_over_ranks((time.perf_counter() - w0) * 1e3, device=dev)
    e2e['blocking_calls_value'] = world * rows * 25 / (blocking_ms * 1e-3)
    torch.cuda.synchronize()
    del h_obs, h_rew, h_done, h_act
    blk.free()
    e2e['pcie_probe'] = pcie_probe(torch, dev, world, D, _lib)

    extras = {}
    if not args.no_extras:
        extras = side_measurements(m, actor, dev, pk, off)

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    line = {
        'metric': 'agent-steps/sec', 'value': value, 'unit': 'agent-steps/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': ms / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'simple_spread N=3 L=3 D=10 A=5, %d envs per GPU, fused observe+actor+sample+'
                               'step+reward kernel (mpe_rollout T=1), in-kernel reset every 25 steps; per-step '
                               'obs_next/rew/act written to HBM' % B,
                   'envs_per_gpu': B, 'l2': 'flushed between timed iterations (256 MiB memset outside the events)',
                   'actor_weights': 'random init, reference architecture (26,117 params)', 'seed': SEED},
        'roofline': {'bound': 'tensor', 'achieved': tflops, 'peak': pk['bf16_tflops_sustained'],
                     'unit': 'TFLOP/s', 'frac': tflops / pk['bf16_tflops_sustained'],
                     'traffic': NCU_DRAM_BYTES_FUSED if B == 65536 else None,
                     'traffic_source': 'dram__bytes_read.sum + dram__bytes_write.sum per launch at 65,536 envs, '
                                       'profiles/r2_ncu_full_summary_tc2_step.txt (state + weights in, outputs stay in L2)',
                     'xu_frac': (NCU_XU_WARP_INST_FUSED / kernel_s) / (148 * XU_WARP_INST_PER_CLK_PER_SM * (clk.get('sm_mhz') or 1965.0) * 1e6)
                                if B == 65536 else None,
                     'issue_frac': NCU_WARP_INST_FUSED / kernel_s / (148 * 4 * (clk.get('sm_mhz') or 1965.0) * 1e6)
                                   if B == 65536 else None,
                     'xu_source': 'smsp__inst_executed_pipe_xu.sum = 2,025,472 warp instructions per launch (989 MUFU ops per '
                                  'env step), profiles/r2_ncu_tc2_counters.txt; peak = 0.5 warp inst/clk/SM x 148 SMs x the SM '
                                  'clock sampled during the run (ncu itself reads 25.9 % of XU peak over the CTA-active cycles, '
                                  'tensor pipe 21.4 %, issue slots 41.9 % cold / 52.8 % warm); issue_frac = smsp__inst_executed.sum (26,181,167 warp '
                                  'instructions per launch) / time / (4 sub-partitions x 148 SMs x the SM clock): the kernel is '
                                  'bound by instruction issue + dependency latency at 2 epilogue warps per sub-partition, and by '
                                  'the 13.5 % tile-quantisation tail of this batch size (DESIGN.md 4.3)',
                     'kernel': 'k_tc2<simple_spread,3,fused> (tcgen05 kind::f16, fp16 hi/lo split operands, fp32 TMEM accum)',
                     'peak_source': pk['source'] + ' bf16 sustained',
                     'flops_per_env_step': FLOPS_PER_ENV_STEP,
                     'note': 'algorithmic (fp32-equivalent) FLOPs; every product is issued as 3 fp16 MMAs for fp32-level '
                             'accuracy, so tensor-pipe work is 3x this; the kernel is bound by the MUFU/issue cost of the '
                             'LSTM cell math between the GEMMs (see DESIGN.md 4.3), not by the tensor pipe'},
        'step_ms_percentiles': {'p50': float(np.percentile(per_step, 50)), 'p99': float(np.percentile(per_step, 99)),
                                'max': float(np.max(per_step))},
        'stats_allreduces': {'count': reduces[0], 'where': 'side stream behind an event, once per %d steps; not inside '
                             'any step\'s event pair' % EP_LEN},
        'e2e': e2e, 'gpu_launches': launches, 'clocks': clk, 'host_cores_bound': len(numa_cores),
        'episode_stats': {k: stats_now[k] for k in ('episodes', 'mean_return', 'std_return')},
    }
    line.update(extras)
    if world == 1:
        line['cpu_baseline'] = cpu_baseline(args.cpu_seconds)
    print(json.dumps(line), flush=True)


def pcie_probe(torch, dev, world, D, _lib):
    """Plain pinned-memory copies, 8 MiB each way: one direction alone, then both at once on two streams - the
    ceiling of the host-buffer path on this box (all ranks run it at the same time, like the e2e loop)."""
    n = 8 << 20
    blk = _lib.HostBlock(2 * n + 1024)
    h_in, h_out = blk.tensor((n,), torch.uint8), blk.tensor((n,), torch.uint8)
    d_in, d_out = torch.empty(n, dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    reps = 40

    def run(up, down):
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            if up:
                with torch.cuda.stream(s1):
                    d_in.copy_(h_in, non_blocking=True)
            if down:
                with torch.cuda.stream(s2):
                    h_out.copy_(d_out, non_blocking=True)
        torch.cuda.synchronize()
        return D.max_over_ranks(time.perf_counter() - t0, device=dev)
    run(True, True)
    t_up, t_down, t_both = run(True, False), run(False, True), run(True, True)
    gb = reps * n / 1e9
    del h_in, h_out
    blk.free()
    return {'h2d_gbs': gb / t_up, 'd2h_gbs': gb / t_down, 'duplex_gbs_each_way': gb / t_both,
            'note': 'per GPU, all ranks copying at once, 8 MiB cudaHostAlloc buffers'}


def side_measurements(m, actor, dev, pk, off):
    """Env-only step kernel (the HBM-bound half of the path) at 1,048,576 envs, and the actor kernel alone."""
    import torch
    out = {}
    B = 1 << 20
    env = m.make_env(SCENARIO, num_envs=B, batched=True, seed=SEED, env_id_offset=off)
    env.reset()
    act = torch.randint(0, 5, (B, N_AGENTS), dtype=torch.int32, device=dev)
    # four rotating output sets (566 MB > the 126 MB L2): every launch's obs / rew / done lines really go to DRAM
    # instead of being overwritten in L2 by the next launch
    rot = [(torch.empty((B, N_AGENTS, OBS_DIM), device=dev), torch.empty((B, N_AGENTS), device=dev),
            torch.empty((B, N_AGENTS), dtype=torch.uint8, device=dev)) for _ in range(4)]
    bufs = rot[0]
    for i in range(8):
        env.step(act, out=rot[i % 4])
    torch.cuda.synchronize()
    reps = 48
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    _gpu_spin(torch)  # ~10 ms GPU spin: the timed launches below are all queued before the first one starts
    e0.record()
    for i in range(reps):
        env.step(act, out=rot[i % 4])  # 280 MB of algorithmic traffic per launch, outputs rotate over 566 MB
    e1.record()
    torch.cuda.synchronize()
    s = e0.elapsed_time(e1) * 1e-3 / reps
    gbs = B * BYTES_PER_ENV_STEP / s / 1e9
    out['roofline_env_step'] = {'bound': 'hbm', 'achieved': gbs, 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
                                'frac': gbs / pk['hbm_gbs'], 'traffic': NCU_DRAM_BYTES_STEP,
                                'frac_dram': NCU_DRAM_BYTES_STEP / s / 1e9 / pk['hbm_gbs'],
                                'traffic_source': 'profiles/r2_ncu_full_summary_tc2_step.txt, 1,048,576 envs per launch, '
                                                  'rotating outputs: 88.1 MB read + 133.8 MB written inside the kernel window; '
                                                  'the remaining ~58 MB of the 192 MB of output are dirty L2 lines written '
                                                  'back after the kernel ends (ncu flushes between replays), so frac_dram is a '
                                                  'lower bound of the DRAM rate and frac (algorithmic bytes) the steady-state one',
                                'outputs': '4 rotating sets, 566 MB > L2',
                                'kernel': 'k_step<float,simple_spread,3>',
                                'envs': B, 'agent_steps_per_s': B * N_AGENTS / s, 'us_per_launch': s * 1e6,
                                'bytes_per_env_step': BYTES_PER_ENV_STEP, 'peak_source': pk['source']}
    obs = bufs[0]
    for _ in range(2):
        actor.forward(obs[:262144])
    torch.cuda.synchronize()
    _gpu_spin(torch)  # ~10 ms GPU spin: the timed launches below are all queued before the first one starts
    e0.record()
    for _ in range(5):
        actor.forward(obs[:262144])
    e1.record()
    torch.cuda.synchronize()
    s = e0.elapsed_time(e1) * 1e-3 / 5
    out['actor_forward_only'] = {'envs': 262144, 'agent_steps_per_s': 262144 * N_AGENTS / s,
                                 'tflops': 262144 * FLOPS_PER_ENV_STEP / s / 1e12}
    # the fused step at the north-star size (>= 1M envs per GPU): 4,096 tile pairs per launch, so the 13.5 % tail of
    # the 65,536-env launch (256 pairs on 148 SMs) is gone; 240 MB of state + outputs per launch > L2, no flush needed
    env.reset()
    rec = (torch.empty((1, B, N_AGENTS, OBS_DIM), device=dev), torch.empty((1, B, N_AGENTS), device=dev),
           torch.empty((1, B, N_AGENTS), dtype=torch.int32, device=dev))
    from multiagent_rl_b200 import _lib
    lib = _lib.load()

    def fused(t):
        _lib.check(lib.mpe_rollout(env._h, actor._h, 1, t, _lib.ptr(rec[0]), _lib.ptr(rec[1]), _lib.ptr(rec[2]), None,
                                   _lib.current_stream(dev)), 'mpe_rollout')
    for t in range(3):
        fused(t)
    torch.cuda.synchronize()
    _gpu_spin(torch)  # ~10 ms GPU spin: the timed launches below are all queued before the first one starts
    e0.record()
    for t in range(20):
        fused(3 + t)
    e1.record()
    torch.cuda.synchronize()
    s = e0.elapsed_time(e1) * 1e-3 / 20
    out['fused_step_1m_envs'] = {'envs': B, 'ms_per_step': s * 1e3, 'agent_steps_per_s': B * N_AGENTS / s,
                                 'tflops': B * FLOPS_PER_ENV_STEP / s / 1e12,
                                 'frac_of_bf16_sustained': B * FLOPS_PER_ENV_STEP / s / 1e12 / pk['bf16_tflops_sustained']}
    del env
    # The headline step again with INPUTS LARGER THAN L2 instead of a flush: 16 independent shards of 65,536 envs
    # (16 x 17.5 MB of state + outputs = 280 MB > 126 MB) stepped round-robin, one launch per step, per-step event
    # pairs.  Every launch finds its data cold in L2 but the kernel's code and the 106 KB weight image warm - what a
    # rollout loop sees - so the difference to `value` is what the flush costs in instruction / weight refetch.
    nsh, Bs = 16, 65536
    shards = []
    for k in range(nsh):
        e = m.make_env(SCENARIO, num_envs=Bs, batched=True, seed=SEED, env_id_offset=k * Bs, max_episode_len=EP_LEN)
        e.reset()
        shards.append((e, torch.empty((1, Bs, N_AGENTS, OBS_DIM), device=dev), torch.empty((1, Bs, N_AGENTS), device=dev),
                       torch.empty((1, Bs, N_AGENTS), dtype=torch.int32, device=dev)))

    def fused_shard(k, t):
        e, o, r, a = shards[k]
        _lib.check(lib.mpe_rollout(e._h, actor._h, 1, t, _lib.ptr(o), _lib.ptr(r), _lib.ptr(a), None,
                                   _lib.current_stream(dev)), 'mpe_rollout')
    for i in range(2 * nsh):
        fused_shard(i % nsh, i // nsh)
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10 * nsh)]
    _gpu_spin(torch)
    for i, (a, b) in enumerate(evs):
        a.record()
        fused_shard(i % nsh, 2 + i // nsh)
        b.record()
    torch.cuda.synchronize()
    per = sorted(a.elapsed_time(b) for a, b in evs)
    s = sum(per) / len(per) * 1e-3
    out['fused_step_rotating_shards'] = {'envs_per_launch': Bs, 'shards': nsh, 'ms_per_step': s * 1e3,
                                         'p50_ms': per[len(per) // 2], 'agent_steps_per_s': Bs * N_AGENTS / s,
                                         'l2': 'no flush: %d shards x 17.5 MB rotate (inputs larger than L2)' % nsh}
    del shards
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    import bench_env_configs
    out['env_step_configs'] = bench_env_configs.run(dev, pk['hbm_gbs'])  # configs 3/4: env-only HBM fractions
    import bench_replay
    out['replay'] = bench_replay.run(dev, pk['hbm_gbs'])  # SURVEY 8f-1: device replay ring, add / uniform sample
    return out


def main():
    args = parse()
    if args.gpus > 1 and 'WORLD_SIZE' not in os.environ:
        cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(args.gpus),
               '--master-addr', '127.0.0.1', '--master-port', '29531', os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
