"""Actor forward + backward on the device: FusedActorNetwork (the actor kernels) against the same network in torch.

    python tools/bench_actor_grad.py [--reps 30] [--iters 20] [--quick] [--out FILE]

The torch side is ``networks.ActorNetwork`` - per-agent ``nn.Linear``, ``nn.LSTM(64, 32, bidirectional=True)``
(cuDNN) over the agent axis, the head(s) - with the weights of the fused network.  Per configuration - B = 1,024 (the
reference's batch_size) at N = 3, simple_reference's two heads [5, 10] at N = 2, the N = 12 "+model" actor, and
B = 65,536 at N = 3 - one step is: zero the grads, forward on obs, loss = sum(logits) (+ sum(next_state)), backward
(weight gradients), as ``Trainer.optimize()`` asks of its actor; TF32 is off, so both sides compute in fp32.  Before
anything is timed the two implementations' weight gradients are compared (within 1e-3 of max(1, max|g|)).  Timing:
``--iters`` steps back to back between two CUDA events, the two implementations alternating ``--reps`` times after a
warm-up of every shape; medians per step.  The fused step is also timed in parts: the repack alone
(``actor_load_device``, done by every forward and every backward), the forward kernel alone and the backward
(kernel + reductions) alone.

Then one whole DDPG update (target actor soft Gumbel -> target critic -> SmoothL1 TD -> critic Adam with gradient
clip 0.5 -> actor -Q(soft Gumbel) + 1e-3 L2 -> actor Adam -> tau = 0.01 soft updates) at N = 3, B = 1,024 for
stock / stock, fused critic / stock actor and fused / fused networks: the reference ``Trainer.optimize()`` over a
``DeviceReplayBuffer`` where the reference is importable, otherwise the same update restated here; each row says which.
Rows are printed as JSON lines and appended to ``--out``, with the GPU's name and power limit read in the same run.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from bench_critic_grad import card, time_steps  # noqa: E402


def step(net, obs):
    net.zero_grad(set_to_none=True)
    out = net(obs)
    policy, ns = out if isinstance(out, tuple) else (out, None)
    loss = sum(p.sum() for p in policy) if isinstance(policy, list) else policy.sum()
    if ns is not None:
        loss = loss + ns.sum()
    loss.backward()


def actor_row(m, base, N, D, heads, model, B, reps, iters):
    import numpy as np
    import torch
    torch.manual_seed(0)
    fused = m.FusedActorNetwork(D, heads, model_head=model).cuda()
    ref = m.ActorNetwork(D, heads, model_head=model).cuda()
    ref.load_state_dict(fused.state_dict())
    obs = torch.from_numpy(np.random.RandomState(1).uniform(-1.5, 1.5, (B, N, D)).astype(np.float32)).cuda()
    # the two implementations agree before anything is timed
    step(fused, obs), step(ref, obs)
    pr = dict(ref.named_parameters())
    worst = 0.0
    for k, p in fused.named_parameters():
        worst = max(worst, float((p.grad - pr[k].grad).abs().max()) / max(1.0, float(pr[k].grad.abs().max())))
    if not worst <= 1e-3:
        raise SystemExit('gradients disagree at N=%d B=%d: %.3g' % (N, B, worst))
    h = fused._handle.actor
    params = dict(fused.named_parameters())
    A = sum(heads) if isinstance(heads, list) else heads
    dl = torch.ones((B, N, A), device='cuda')
    dn = torch.ones_like(obs) if model else None
    parts = {'repack': lambda: h.load_state_dict(params),
             'forward': lambda: h.forward(obs, want_logits=True, want_next_state=model),
             'backward': lambda: h.backward(obs, dl, dn)}
    for _ in range(3):
        step(fused, obs), step(ref, obs)
        for f in parts.values():
            f()
    fa, fb, pt = [], [], {k: [] for k in parts}
    for _ in range(reps):
        fa.append(time_steps(lambda: step(fused, obs), iters))
        fb.append(time_steps(lambda: step(ref, obs), iters))
        for k, f in parts.items():
            pt[k].append(time_steps(f, iters))
    med = lambda x: round(statistics.median(x), 4)  # noqa: E731
    name = 'N=%d B=%d heads=%s%s' % (N, B, heads, ' +model' if model else '')
    return dict(base, kind='actor_fwd_bwd', config=name, N=N, D=D, B=B, torch_side='networks.ActorNetwork (cuDNN BiLSTM)',
                weight_grad_max_rel_diff=float('%.3g' % worst), fused_ms=med(fa), torch_ms=med(fb),
                speedup=round(statistics.median(fb) / statistics.median(fa), 3), fused_ms_min=round(min(fa), 4),
                torch_ms_min=round(min(fb), 4), fused_repack_ms=med(pt['repack']),
                fused_forward_ms=med(pt['forward']), fused_backward_ms=med(pt['backward']), reps=reps, iters=iters)


def ddpg_update(actor, critic, tactor, tcritic, aopt, copt, batch, gamma=0.95, tau=0.01):
    """One update as Trainer.optimize() (ddpg_gumbel_fix.py:131-219) does it, for tools where the reference is not
    importable."""
    import torch
    import torch.nn.functional as F
    s1, a1, r1, s2 = batch
    with torch.no_grad():
        a2 = F.gumbel_softmax(tactor(s2), hard=False)
        y = r1 + gamma * tcritic(s2, a2).squeeze(-1)
    q = critic(s1, a1).squeeze(-1)
    loss_c = F.smooth_l1_loss(q, y)
    copt.zero_grad()
    loss_c.backward()
    torch.nn.utils.clip_grad_norm_(critic.parameters(), 0.5)
    copt.step()
    logits = actor(s1)
    loss_a = -critic(s1, F.gumbel_softmax(logits, hard=False)).mean() + 1e-3 * (logits ** 2).mean()
    aopt.zero_grad()
    loss_a.backward()
    aopt.step()
    for tn, n in ((tactor, actor), (tcritic, critic)):
        for tp, p in zip(tn.parameters(), n.parameters()):
            tp.data.copy_(tp.data * (1.0 - tau) + p.data * tau)


def optimize_rows(m, base, reps):
    import copy
    import torch
    N, D, A, B = 3, 10, 5, 1024
    kinds = {'stock/stock': (False, False), 'fused critic/stock actor': (True, False), 'fused/fused': (True, True)}
    try:
        from rls import arglist
        from rls.agent.multiagent.ddpg_gumbel_fix import Trainer
        from rls.model.ac_network_multi_gumbel import ActorNetwork, CriticNetwork
        source = 'reference Trainer.optimize()'
    except ImportError:
        Trainer = None
        ActorNetwork, CriticNetwork = m.ActorNetwork, None
        source = 'restated in tools/bench_actor_grad.py (reference not importable)'
    if Trainer is not None:
        arglist.batch_size = B
        env = m.make_env('simple_spread', num_envs=4096, batched=True, seed=1, max_episode_len=25)
        memory = m.DeviceReplayBuffer(4096 * 25, N, D, A, seed=1)
        env.reset()
        env.rollout(m.FusedActor(m.networks.random_state_dict(D, A, 0), seed=1), 25, replay=memory)
    else:
        g = torch.Generator(device='cuda').manual_seed(1)
        s1 = torch.rand((B, N, D), device='cuda', generator=g) * 3 - 1.5
        s2 = torch.rand((B, N, D), device='cuda', generator=g) * 3 - 1.5
        a1 = torch.nn.functional.one_hot(torch.randint(0, A, (B, N), device='cuda', generator=g), A).float()
        r1 = torch.randn((B,), device='cuda', generator=g)
        batch = (s1, a1, r1, s2)
    updates = {}
    for kind, (fc, fa) in kinds.items():
        torch.manual_seed(0)
        actor = (m.FusedActorNetwork if fa else ActorNetwork)(D, A)
        if fc:
            critic = m.FusedCriticNetwork(D + A, 1)
        elif CriticNetwork is not None:
            critic = CriticNetwork(input_dim=D + A, out_dim=1)
        else:
            critic = _torch_critic(D + A)
        if Trainer is not None:
            updates[kind] = Trainer(actor, critic, memory, action_type='Discrete').optimize
        else:
            actor, critic = actor.cuda(), critic.cuda()
            ta, tc = copy.deepcopy(actor), copy.deepcopy(critic)
            ao, co = torch.optim.Adam(actor.parameters(), 1e-2), torch.optim.Adam(critic.parameters(), 1e-2)
            updates[kind] = (lambda a=actor, c=critic, ta=ta, tc=tc, ao=ao, co=co:
                             ddpg_update(a, c, ta, tc, ao, co, batch))
    times = {k: [] for k in updates}
    for f in updates.values():
        for _ in range(3):
            f()
    for _ in range(reps):
        for k, f in updates.items():
            times[k].append(time_steps(f, 5))
    return [dict(base, kind='optimize', config='DDPG update N=3 B=1024 ' + k, update=source,
                 ms=round(statistics.median(times[k]), 4), ms_min=round(min(times[k]), 4), reps=reps, iters=5)
            for k in updates]


def _torch_critic(input_dim):
    from bench_critic_grad import torch_critic
    return torch_critic(input_dim, False)[0]


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
        raise SystemExit('bench_actor_grad needs a CUDA device')
    # both sides in fp32: cuDNN's LSTM and the matmuls would otherwise round their inputs to TF32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    name, power = card()
    base = {'gpu': name, 'power_limit': power}
    reps, iters = (3, 3) if a.quick else (a.reps, a.iters)
    rows = []
    configs = ((3, 10, 5, False, 1024), (2, 21, [5, 10], False, 1024), (12, 28, 5, True, 1024),
               (3, 10, 5, False, 4096 if a.quick else 65536))
    for N, D, heads, model, B in configs:
        rows.append(actor_row(m, base, N, D, heads, model, B, reps, iters))
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
