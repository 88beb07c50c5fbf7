"""Critic forward + backward on the device: FusedCriticNetwork (the critic kernels) against the same network in torch.

    python tools/bench_critic_grad.py [--reps 30] [--iters 20] [--quick] [--out FILE]

The torch side is the reference ``CriticNetwork`` (rls/model/ac_network_multi_gumbel.py:70-148, or the "+model"
class) when the reference is importable, otherwise the same layers spelled here: per-agent ``nn.Linear``,
``nn.LSTM(64, 64)`` (cuDNN) over the agent axis, ``bmm`` attention, softmax.  Per configuration - B = 1,024 (the
reference's batch_size) at N = 3 and N = 12 ("+model" critic), B = 65,536 at N = 3 - one step is: zero the grads,
forward on (obs, action) with action requiring grad, loss = sum(q) (+ sum(r)), backward (weight and action
gradients), as ``Trainer.optimize()`` asks of its critic; TF32 is off, so both sides compute in fp32.  Before anything
is timed the two implementations' gradients are compared (weights within 1e-3 of max(1, max|g|); action gradients
within 1e-4 for all but 0.1 % of the samples, which may sit at a relu kink).  Timing: ``--iters`` steps back to back between two CUDA events, the two implementations
alternating ``--reps`` times after a warm-up of every shape; medians per step.  Also the repack alone (the
``critic_load_device`` every FusedCriticNetwork forward does), and one ``Trainer.optimize()`` of the reference with
each critic where the reference is importable.  Rows are printed as JSON lines and appended to ``--out``, with the
GPU's name and power limit read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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


def torch_critic(input_dim, model):
    """The reference class when importable, else the same layers."""
    import torch
    import torch.nn as nn
    try:
        if model:
            from rls.model.ac_network_model_multi_gumbel import CriticNetwork
        else:
            from rls.model.ac_network_multi_gumbel import CriticNetwork
        return CriticNetwork(input_dim=input_dim, out_dim=1), 'reference CriticNetwork'
    except ImportError:
        pass
    from multiagent_rl_b200.networks import _PerAgent

    class Critic(nn.Module):
        def __init__(self):
            super().__init__()
            self.dense1 = _PerAgent(nn.Linear(input_dim, 64))
            self.lstm = nn.LSTM(64, 64, batch_first=True)
            self.dense2 = nn.Linear(64, 1)
            if model:
                self.dense3 = nn.Linear(64, 1)

        def forward(self, obs, action):
            out, (hn, _) = self.lstm(torch.relu(self.dense1(torch.cat([obs, action], -1))))
            attn = torch.softmax(torch.bmm(out, hn.squeeze(0).unsqueeze(2)).squeeze(2), 1)
            n = torch.bmm(out.transpose(1, 2), attn.unsqueeze(2)).squeeze(2)
            return (self.dense2(n), self.dense3(n)) if model else self.dense2(torch.relu(n))
    return Critic(), 'torch nn.LSTM + bmm restatement'


def step(net, obs, act):
    net.zero_grad(set_to_none=True)
    act = act.detach().requires_grad_(True)
    out = net(obs, act)
    loss = out[0].sum() + out[1].sum() if isinstance(out, tuple) else out.sum()
    loss.backward()
    return act.grad


def time_steps(fn, iters):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def critic_row(m, base, N, B, model, reps, iters):
    import numpy as np
    import torch
    D, A = {3: 10, 12: 28}[N], 5
    torch.manual_seed(0)
    fused = m.FusedCriticNetwork(D + A, 1, model=model).cuda()
    ref, ref_kind = torch_critic(D + A, model)
    ref = ref.cuda()
    ref.load_state_dict(fused.state_dict())
    rng = np.random.RandomState(1)
    obs = torch.from_numpy(rng.uniform(-1.5, 1.5, (B, N, D)).astype(np.float32)).cuda()
    z = torch.from_numpy(rng.randn(B, N, A).astype(np.float32)).cuda()
    act = torch.softmax(2 * z, -1)
    # the two implementations agree before anything is timed: every weight gradient within 1e-3 of max(1, max|g|);
    # action gradients within 1e-4 for all but 0.1 % of the samples (a sample whose dense1 or attention output sits
    # at a relu kink may take the other side in either fp32 implementation)
    ga, gb = step(fused, obs, act), step(ref, obs, act)
    pr = dict(ref.named_parameters())
    worst = 0.0
    for k, p in fused.named_parameters():
        worst = max(worst, float((p.grad - pr[k].grad).abs().max()) / max(1.0, float(pr[k].grad.abs().max())))
    dev = (ga - gb).abs().flatten(1).max(1).values / max(1.0, float(gb.abs().max()))
    off = float((dev > 1e-4).float().mean())
    if not (worst <= 1e-3 and off <= 1e-3):
        raise SystemExit('gradients disagree at N=%d B=%d: weights %.3g, %.3g of the samples\' action gradients'
                         % (N, B, worst, off))
    fa, fb = [], []
    for _ in range(3):
        step(fused, obs, act), step(ref, obs, act)
    for _ in range(reps):
        fa.append(time_steps(lambda: step(fused, obs, act), iters))
        fb.append(time_steps(lambda: step(ref, obs, act), iters))
    params = dict(fused.named_parameters())
    h = fused._handle.critic
    load = lambda: h.load_state_dict(params)  # noqa: E731
    for _ in range(3):
        load()
    rp = [time_steps(load, iters) for _ in range(reps)]
    med = lambda x: round(statistics.median(x), 4)  # noqa: E731
    return dict(base, kind='critic_fwd_bwd', config='N=%d B=%d %s' % (N, B, '+model' if model else 'relu'),
                N=N, B=B, torch_side=ref_kind, weight_grad_max_rel_diff=float('%.3g' % worst),
                action_grad_max_diff=float('%.3g' % float(dev.max())), action_grad_samples_off=off,
                fused_ms=med(fa), torch_ms=med(fb), speedup=round(statistics.median(fb) / statistics.median(fa), 3),
                fused_ms_min=round(min(fa), 4), torch_ms_min=round(min(fb), 4), repack_ms=med(rp), reps=reps,
                iters=iters)


def optimize_rows(m, base, reps):
    """One reference Trainer.optimize() (ddpg_gumbel_fix.py:131-219) with each critic over a DeviceReplayBuffer."""
    import numpy as np
    import torch
    try:
        from rls import arglist
        from rls.agent.multiagent.ddpg_gumbel_fix import Trainer
        from rls.model.ac_network_multi_gumbel import ActorNetwork, CriticNetwork
    except ImportError:
        return [dict(base, kind='optimize', status='not measured: the reference is not importable')]
    N, D, A, B = 3, 10, 5, 1024
    arglist.batch_size = B
    env = m.make_env('simple_spread', num_envs=4096, batched=True, seed=1, max_episode_len=25)
    memory = m.DeviceReplayBuffer(4096 * 25, N, D, A, seed=1)
    torch.manual_seed(0)
    actor = m.FusedActor(m.networks.random_state_dict(D, A, 0), seed=1)
    env.reset()
    env.rollout(actor, 25, replay=memory)
    rows, learners = [], {}
    for kind in ('fused', 'torch'):
        torch.manual_seed(0)
        a = ActorNetwork(input_dim=D, out_dim=A)
        c = m.FusedCriticNetwork(D + A, 1) if kind == 'fused' else CriticNetwork(input_dim=D + A, out_dim=1)
        learners[kind] = Trainer(a, c, memory, action_type='Discrete')
    times = {k: [] for k in learners}
    for k, lr in learners.items():
        for _ in range(3):
            lr.optimize()
    for _ in range(reps):
        for k, lr in learners.items():
            times[k].append(time_steps(lr.optimize, 5))
    rows.append(dict(base, kind='optimize', config='ddpg_gumbel_fix Trainer.optimize() N=3 B=1024',
                     fused_ms=round(statistics.median(times['fused']), 4),
                     torch_ms=round(statistics.median(times['torch']), 4), reps=reps, iters=5))
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=30)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--quick', action='store_true', help='small sizes (a smoke run of the tool)')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    import torch
    import multiagent_rl_b200 as m
    if not torch.cuda.is_available():
        raise SystemExit('bench_critic_grad needs a CUDA device')
    # both sides in fp32: cuDNN's LSTM and the matmuls would otherwise round their inputs to TF32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    name, power = card()
    base = {'gpu': name, 'power_limit': power}
    reps, iters = (3, 3) if a.quick else (a.reps, a.iters)
    rows = []
    for N, B, model in ((3, 1024, False), (12, 1024, True), (3, 4096 if a.quick else 65536, False)):
        rows.append(critic_row(m, base, N, B, model, reps, iters))
        print(json.dumps(rows[-1]), flush=True)
    for r in optimize_rows(m, base, reps):
        rows.append(r)
        print(json.dumps(r), flush=True)
    if a.out:
        with open(a.out, 'a') as fp:
            for r in rows:
                fp.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
