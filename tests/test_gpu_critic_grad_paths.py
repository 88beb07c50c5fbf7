"""GPU tests of the critic backward (critic_grad_kernels.cu) past what a float64 tolerance can see:

1. k_critic_backward recomputes the attention output n the heads read bit for bit as k_critic_forward computes it (so
   it differentiates the forward's function, relu masks included), read on both sides through exact probes;
2. exact relu kinks (z1 = 0, h = 0 in fp32 and float64) with no sample dropped, relu'(0) = 0 as in torch;
3. exact invariants of the chunked reductions (a constant input column or LSTM input, linearity, zero upstream);
4. each sample's rows land exactly once in the weight gradients (one-hot upstream against a batch of one, and the
   heads' gradients against a rigorous float64 summation bound);
5. the ABI's workspace / output / stream / graph-capture promises and the autograd paths of FusedCriticNetwork;
6. record and output offsets past 2^31 floats.

Where a probe is aimed at the chunking of the weight-gradient sums, ``_plan`` mirrors it; every assertion holds for
any chunking, only where the probes land depends on it."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

from tests import _critic_torch as ct
from tests.test_gpu_critic import _actions, _sharp_critic

pytestmark = pytest.mark.gpu

H = 64
EPS = 2.0 ** -24  # unit roundoff of fp32
_FIELDS = [('dense1_w', 'dense1.module.weight'), ('dense1_b', 'dense1.module.bias'), ('w_ih', 'lstm.weight_ih_l0'),
           ('w_hh', 'lstm.weight_hh_l0'), ('b_ih', 'lstm.bias_ih_l0'), ('b_hh', 'lstm.bias_hh_l0'),
           ('dense2_w', 'dense2.weight'), ('dense2_b', 'dense2.bias'), ('dense3_w', 'dense3.weight'),
           ('dense3_b', 'dense3.bias')]  # CriticGrads field -> state_dict key
HEADS = ('dense2.weight', 'dense2.bias', 'dense3.weight', 'dense3.bias')

# The chunking of the weight-gradient sums (critic_grad_kernels.cu: kMaxChunks, kChunkRows, grad_plan): the B * N
# (sample, agent) rows are cut into nchunk = min(ceil(rows / 64), 64) chunks of ceil(rows / nchunk) rows, each summed
# by one CTA that stages 32 rows at a time; the dense2 / dense3 tiles cut the B samples into the same nchunk chunks
# (of ceil(B / nchunk) samples, so some may be empty); the chunk partials are then summed in chunk order.
K_MAX_CHUNKS, K_CHUNK_ROWS, K_STAGE_ROWS = 64, 64, 32


def _plan(B, N):
    """(rows, nchunk, rows per chunk, samples per dense2 / dense3 chunk)"""
    rows = B * N
    nchunk = max(1, min(-(-rows // K_CHUNK_ROWS), K_MAX_CHUNKS))
    return rows, nchunk, -(-rows // nchunk), -(-B // nchunk)


def _one_chunk(b, N, cs):
    """Whether sample b's N rows lie in one chunk of cs rows."""
    return b * N // cs == ((b + 1) * N - 1) // cs


def _probes(B, N, nsm):
    """Samples aimed at the edges of the plan: the first and last rows of chunks (the first four, a middle one and the
    last), a sample across each of those chunk boundaries, the 32-row staging edges inside them, the first and last
    samples of dense2 chunks, the first sample of k_critic_backward's second pass (8 warps x nsm CTAs) and B - 1."""
    rows, nchunk, cs, csb = _plan(B, N)
    want = {0, B - 1}
    for c in sorted({0, 1, 2, 3, nchunk // 2, nchunk - 1}):
        r0, r1 = c * cs, min((c + 1) * cs, rows)
        if r0 >= rows:
            continue
        want.update([r0 // N, (r1 - 1) // N, min(r0 + K_STAGE_ROWS, r1 - 1) // N,
                     min(r0 + K_STAGE_ROWS - 1, r1 - 1) // N])
        s0, s1 = c * csb, min((c + 1) * csb, B)
        if s0 < s1:
            want.update([s0, s1 - 1])
    if B > nsm * 8:
        want.add(nsm * 8)
    return sorted(want)


def _nsm():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _weights(kind, seed, D, A, model, out):
    """float32 numpy state_dict: 'default' is FusedCriticNetwork's (the reference's) initialisation under `seed`,
    'sharp' the saturating weights of tests/test_gpu_critic.py."""
    import multiagent_rl_b200 as m
    if kind == 'sharp':
        return _sharp_critic(np.random.RandomState(seed), D, A, model, out)
    torch.manual_seed(seed)
    return {k: v.numpy().copy() for k, v in m.FusedCriticNetwork(D + A, out, model=model).state_dict().items()}


def _inputs(rng, B, N, D, A, action='softmax'):
    obs = torch.from_numpy(rng.uniform(-2, 2, (B, N, D)).astype(np.float32)).cuda()
    return obs, torch.from_numpy(_actions(rng, B, N, A, action)).cuda()


def _upstream(rng, B, out, model):
    dq = torch.from_numpy(rng.randn(B, out).astype(np.float32)).cuda()
    return dq, (torch.from_numpy(rng.randn(B, out).astype(np.float32)).cuda() if model else None)


def _nan_outputs(sd, obs, act):
    nan = float('nan')
    return {'obs': torch.full_like(obs, nan), 'action': torch.full_like(act, nan),
            'weights': {k: torch.full(np.shape(sd[k]), nan, device=obs.device) for _, k in _FIELDS if k in sd}}


def _raw_backward(critic, sd, obs, act, dq, dr=None, ws=None, offset=0):
    """critic_backward through the C ABI with every output requested, each filled with NaN first (an output that is
    accumulated into or left unwritten shows); the workspace is `ws` from byte `offset`, or a fresh one."""
    from multiagent_rl_b200 import _lib
    B, N = obs.shape[:2]
    nbytes = critic._lib.critic_backward_workspace(critic._h, B, N)
    if ws is None:
        ws = torch.empty(nbytes, dtype=torch.uint8, device=obs.device)
    assert ws.numel() * ws.element_size() >= offset + nbytes
    out = _nan_outputs(sd, obs, act)
    g = _lib.CriticGrads(**{f: out['weights'][k].data_ptr() for f, k in _FIELDS if k in out['weights']})
    _lib.check(critic._lib.critic_backward(critic._h, _lib.ptr(obs), _lib.ptr(act), B, N, _lib.ptr(dq), _lib.ptr(dr),
                                           _lib.ptr(out['obs']), _lib.ptr(out['action']), C.byref(g),
                                           C.c_void_p(ws.data_ptr() + offset), nbytes,
                                           _lib.current_stream(obs.device)), 'critic_backward')
    return out


def _same(got, want, what=''):
    """Bit for bit (== on every element, so -0 and +0 are equal and a NaN never is)."""
    for k in ('obs', 'action'):
        if want[k] is not None:
            assert torch.equal(got[k], want[k]), (what, k)
    assert sorted(got['weights']) == sorted(want['weights']), what
    for k, v in want['weights'].items():
        assert torch.equal(got['weights'][k], v), (what, k)


def _check(got, want, tol, what):
    """The float64 tolerance of tests/test_gpu_critic_grad.py."""
    scale = max(1.0, float(np.abs(want).max()))
    err = float(np.abs(np.asarray(got, np.float64) - want).max())
    assert err <= tol * scale, (what, err, scale)


# ---- 1. the backward's forward is the forward's ----

def _selectors(sd, units):
    """`sd` with head rows that are unit selectors e_k (bias 0): q_o = n_{units[o]} and r_o = n_{units[out + o]}
    exactly (one product by 1, the warp sum adds exact zeros)."""
    sd = dict(sd)
    out = np.shape(sd['dense2.weight'])[0]
    eye = np.eye(H, dtype=np.float32)
    sd['dense2.weight'], sd['dense2.bias'] = eye[units[:out]], np.zeros(out, np.float32)
    if 'dense3.weight' in sd:
        sd['dense3.weight'], sd['dense3.bias'] = eye[units[out:2 * out]], np.zeros(out, np.float32)
    return sd


def _forward_n(critic, sd, obs, act):
    """n [B,64], the attention output the heads read (after the relu of the relu critic), as k_critic_forward computes
    it: the critic's heads are reloaded as selectors until every unit has been read.  Leaves selector heads loaded."""
    out = critic.out_dim
    per = out * (2 if critic.model else 1)
    n = torch.empty(obs.shape[0], H, device=obs.device)
    for k0 in range(0, H, per):
        critic.load_state_dict(_selectors(sd, list(range(k0, k0 + per))))
        res = critic.forward(obs, act)
        if critic.model:
            n[:, k0:k0 + out], n[:, k0 + out:k0 + per] = res
        else:
            n[:, k0:k0 + out] = res
    return n


def _backward_n(critic, obs, act, s):
    """n [4,64] of samples s..s+3 as k_critic_backward recomputes it (out_dim 4): with dq = I_4 on those samples and 0
    elsewhere, row o of the dense2.weight gradient is n of sample s + o (one product by 1 plus exact zeros)."""
    dq = torch.zeros(obs.shape[0], 4, device=obs.device)
    dq[s:s + 4] = torch.eye(4, device=obs.device)
    return critic.backward(obs, act, dq, want_action=False)['weights']['dense2.weight']


@pytest.mark.parametrize('weights', ['default', 'sharp'])
@pytest.mark.parametrize('D,A', [(10, 5), (59, 5)], ids=['din15', 'din64'])
@pytest.mark.parametrize('N', [1, 3, 16])
@pytest.mark.parametrize('model', [False, True], ids=['relu', 'model'])
def test_backward_recomputes_the_forwards_attention_output_bit_for_bit(model, N, D, A, weights):
    """n from k_critic_forward (through selector heads) and from k_critic_backward (through the dense2 gradient) are
    the same bits, for 4-sample launches aimed at the samples with the most units near a relu kink and for 4-sample
    groups inside a batch that takes every warp of the backward through a second pass."""
    import multiagent_rl_b200 as m
    seed = 100 * N + D + (7 if model else 0) + (1 if weights == 'sharp' else 0)
    rng = np.random.RandomState(seed)
    sd = _weights(weights, seed, D, A, model, 4)
    pass1 = _nsm() * 8  # k_critic_backward: one sample per warp, 8 warps per CTA, at most one CTA per SM
    B = 2 * pass1 + 37
    obs, act = _inputs(rng, B, N, D, A)
    critic = m.FusedCritic(sd, obs_dim=D)
    n_fwd = _forward_n(critic, sd, obs, act)
    with torch.no_grad():
        z1, n64 = ct.Critic64(sd).pre_activations(obs.cpu().double(), act.cpu().double())
    near_n, near_z = (n64.abs() <= 1e-5).numpy(), (z1.abs() <= 1e-5).numpy()
    per_sample = near_n.sum(-1) + near_z.sum((-1, -2))
    groups = np.argsort(-per_sample[:B // 4 * 4].reshape(-1, 4).sum(1), kind='stable')[:13] * 4
    compared = []
    for s in groups:  # 4-sample launches
        got = _backward_n(critic, obs[s:s + 4], act[s:s + 4], 0)
        assert torch.equal(got, n_fwd[s:s + 4]), ('launch of 4', int(s), int((got != n_fwd[s:s + 4]).sum()))
        compared.extend(range(s, s + 4))
    for s in (0, pass1 - 2, B - 4):  # inside the full batch: first group, across the second pass's start, last
        got = _backward_n(critic, obs, act, s)
        assert torch.equal(got, n_fwd[s:s + 4]), ('in the batch', s, int((got != n_fwd[s:s + 4]).sum()))
        compared.extend(range(s, s + 4))
    kn, kz = int(near_n[compared].sum()), int(near_z[compared].sum())
    print('compared %d samples x 64 units: %d units of n and %d dense1 pre-activations within 1e-5 of a relu kink'
          % (len(compared), kn, kz))
    assert kn + kz > 0


# ---- 2. exact kinks ----

DEAD_ROWS = [0, 17, 40, 63]  # dense1 rows with zero weights and bias: z1 = 0 exactly for every input
DEAD_UNITS = [3, 32, 50]  # LSTM units whose output gate sees exactly -100: h = o * tanh(c) = 0 exactly in fp32


def _kill(sd, units):
    """Output gate of `units` = sigmoid(-100): zero weights, bias -100.  In fp32 expf(100) = inf, so o = 1 / inf = 0 and
    h = 0 exactly; in float64 o is about 4e-44 and every gradient it scales is negligible."""
    sd = {k: np.array(v, np.float32, copy=True) for k, v in sd.items()}
    rows = [3 * H + u for u in units]  # torch's gate order i, f, g, o
    for k in ('lstm.weight_ih_l0', 'lstm.weight_hh_l0', 'lstm.bias_hh_l0'):
        sd[k][rows] = 0.0
    sd['lstm.bias_ih_l0'][rows] = -100.0
    return sd


@pytest.mark.parametrize('model', [False, True], ids=['relu', 'model'])
def test_exact_relu_kinks_with_no_sample_dropped(model):
    """Every gradient against float64 autograd on the whole batch (no kink filter) where some dense1 units sit exactly
    on the relu's kink and some LSTM units are exactly 0; torch's relu'(0) = 0 gives exact zeros where the gradient
    can only pass through a dead unit.  A critic whose every output gate is dead has exactly zero gradients for
    dobs, daction and every weight that feeds the LSTM."""
    import multiagent_rl_b200 as m
    N, D, A, B, out = 3, 10, 5, 1500, 2
    rng = np.random.RandomState(31 + model)
    sd = _kill(_weights('default', 31, D, A, model, out), DEAD_UNITS)
    sd['dense1.module.weight'][DEAD_ROWS] = 0.0
    sd['dense1.module.bias'][DEAD_ROWS] = 0.0
    obs, act = _inputs(rng, B, N, D, A, 'onehot')
    dq, dr = _upstream(rng, B, out, model)
    tol = 1e-4
    for case, w in (('some dead', sd), ('all dead', _kill(sd, range(H)))):
        critic = m.FusedCritic(w, obs_dim=D)
        got = critic.backward(obs, act, dq, dr, want_obs=True)
        want = ct.grads(w, obs.cpu().numpy(), act.cpu().numpy(), dq.cpu().numpy(),
                        None if dr is None else dr.cpu().numpy())
        _check(got['obs'].cpu().numpy(), want['obs'], tol, (case, 'obs'))
        _check(got['action'].cpu().numpy(), want['action'], tol, (case, 'action'))
        for k, v in got['weights'].items():
            _check(v.cpu().numpy(), want[k], tol, (case, k))
        g = got['weights']
        # relu'(0) = 0: the dense1 rows on the kink get no gradient, and the LSTM sees x = 0 there
        assert bool((g['dense1.module.weight'][DEAD_ROWS] == 0).all()), case
        assert bool((g['dense1.module.bias'][DEAD_ROWS] == 0).all()), case
        assert bool((g['lstm.weight_ih_l0'][:, DEAD_ROWS] == 0).all()), case
        # h = 0 for a dead unit: W_hh's column for it multiplies h_{t-1} = 0, and its output gate gets o (1 - o) = 0
        assert bool((g['lstm.weight_hh_l0'][:, DEAD_UNITS] == 0).all()), case
        rows = [3 * H + u for u in DEAD_UNITS]
        assert bool((g['lstm.weight_ih_l0'][rows] == 0).all()) and bool((g['lstm.bias_ih_l0'][rows] == 0).all()), case
        if case == 'all dead':
            for k in ('obs', 'action'):
                assert bool((got[k] == 0).all()), (case, k)
            for k in ('dense1.module.weight', 'dense1.module.bias') + tuple(k for k in ct.KEYS if k.startswith('lstm')):
                assert bool((g[k] == 0).all()), (case, k)


# ---- 3. exact invariants of the reductions ----

# B * N = 1, 63, 64, 65 (one chunk and the first ragged one), 4095, 4096, 4097 (the most chunks of 64 rows and one
# past), B = 257 x 16 (12 of the dense2 / dense3 tiles' 64 chunks empty) and 65,539 x 3 (64 chunks of 3,073 rows)
SHAPES = [(1, 1, False), (21, 3, True), (4, 16, False), (13, 5, True), (1365, 3, False), (256, 16, True),
          (4097, 1, False), (257, 16, True), (65539, 3, False), (65539, 3, True)]
CONST_UNITS = [0, 31, 32, 63]  # dense1 rows with zero weights and bias 1: x_j = 1 exactly


@pytest.mark.parametrize('B,N,model', SHAPES, ids=['%dx%d-%s' % (b, n, 'model' if m else 'relu') for b, n, m in SHAPES])
def test_reductions_keep_exact_invariants(B, N, model):
    """No tolerance.  A constant input column k gives dense1.weight.grad[:, k] == dense1.bias.grad and a constant LSTM
    input j gives lstm.weight_ih_l0.grad[:, j] == bias_ih.grad == bias_hh.grad (each product is exact and both sums
    take the same rows in the same order); scaling dq and dr by 2^4 scales every output by 2^4; dq = dr = 0 gives
    exact zeros in outputs that were NaN."""
    import multiagent_rl_b200 as m
    D, A, out = 59, 5, 2
    rng = np.random.RandomState(B + N)
    sd = _weights('default', 41 + N, D, A, model, out)
    sd['dense1.module.weight'][CONST_UNITS] = 0.0
    sd['dense1.module.bias'][CONST_UNITS] = 1.0
    obs, act = _inputs(rng, B, N, D, A, 'uniform')
    cols = [0, D - 1, D, D + A - 1]  # first and last obs column, first and last action column
    for k in cols:
        (obs[..., k] if k < D else act[..., k - D]).fill_(1.0)
    dq, dr = _upstream(rng, B, out, model)
    critic = m.FusedCritic(sd, obs_dim=D)
    g = _raw_backward(critic, sd, obs, act, dq, dr)
    w = g['weights']
    for k in cols:
        assert torch.equal(w['dense1.module.weight'][:, k], w['dense1.module.bias']), k
    for j in CONST_UNITS:
        assert torch.equal(w['lstm.weight_ih_l0'][:, j], w['lstm.bias_ih_l0']), j
        assert torch.equal(w['lstm.weight_ih_l0'][:, j], w['lstm.bias_hh_l0']), j
    g16 = _raw_backward(critic, sd, obs, act, dq * 16.0, None if dr is None else dr * 16.0)
    for k in ('obs', 'action'):
        assert torch.equal(g16[k], g[k] * 16.0), k
    for k, v in w.items():
        assert torch.equal(g16['weights'][k], v * 16.0), k
    g0 = _raw_backward(critic, sd, obs, act, torch.zeros_like(dq), None if dr is None else torch.zeros_like(dr))
    for k in ('obs', 'action'):
        assert bool((g0[k] == 0).all()), k
    for k, v in g0['weights'].items():
        assert bool((v == 0).all()), k


# ---- 4. each sample's contribution lands exactly once ----

def _batch_of_one(critic, obs, act, dq, dr, b):
    return critic.backward(obs[b:b + 1], act[b:b + 1], dq[b:b + 1], None if dr is None else dr[b:b + 1],
                           want_obs=True)


@pytest.mark.parametrize('B,N,model', [(65539, 3, False), (65539, 3, True), (257, 16, False), (257, 16, True)])
def test_each_samples_rows_land_exactly_once(B, N, model):
    """dq (and dr) on one sample b only: the full batch's weight gradients are those of the batch [b] alone (bit for bit
    where b's rows lie in one chunk and for the heads, else within 1e-6 of max|g|; a dropped row gives 0, a doubled
    one 2x), dobs / daction are exactly 0 for every other sample and b's are the same bits.  Then one sample in each
    chunk: the result is the float64 sum of their batch-of-one gradients within (nchunk + 1) * 2^-24 * sum |g_b|."""
    import multiagent_rl_b200 as m
    D, A, out = 10, 5, 2
    rng = np.random.RandomState(B * N + model)
    sd = _weights('default', 51 + model, D, A, model, out)
    obs, act = _inputs(rng, B, N, D, A)
    critic = m.FusedCritic(sd, obs_dim=D)
    rows, nchunk, cs, _ = _plan(B, N)
    v, vr = _upstream(rng, 1, out, model)
    probes = _probes(B, N, _nsm())
    print('probes at B = %d, N = %d (%d chunks of %d rows): %s' % (B, N, nchunk, cs, probes))
    for b in probes:
        dq = torch.zeros(B, out, device='cuda')
        dq[b] = v[0]
        dr = None
        if model:
            dr = torch.zeros(B, out, device='cuda')
            dr[b] = vr[0]
        full = critic.backward(obs, act, dq, dr, want_obs=True)
        one = _batch_of_one(critic, obs, act, dq, dr, b)
        for k in ('obs', 'action'):
            assert torch.equal(full[k][b:b + 1], one[k]), (b, k)
            assert bool((full[k][:b] == 0).all()) and bool((full[k][b + 1:] == 0).all()), (b, k)
        exact = _one_chunk(b, N, cs)
        for k, g1 in one['weights'].items():
            g = full['weights'][k]
            if exact or k in HEADS:
                assert torch.equal(g, g1), (b, k)
            else:
                err = float((g - g1).abs().max())
                assert err <= 1e-6 * float(g1.abs().max()), (b, k, err)
    # one sample wholly inside each chunk, all in one call
    picks = [b for b in (-(-c * cs // N) for c in range(nchunk)) if b < B and _one_chunk(b, N, cs)]
    assert len(set(b * N // cs for b in picks)) == len(picks)
    sel = torch.zeros(B, 1, device='cuda')
    sel[picks] = 1.0
    dq, dr = _upstream(rng, B, out, model)
    dq = dq * sel
    dr = None if dr is None else dr * sel
    full = critic.backward(obs, act, dq, dr, want_obs=True)
    ones = [_batch_of_one(critic, obs, act, dq, dr, b) for b in picks]
    for k in ('obs', 'action'):
        assert torch.equal(full[k][picks], torch.cat([o[k] for o in ones])), k
        assert bool((full[k][sel[:, 0] == 0] == 0).all()), k
    gamma = (nchunk + 1) * EPS
    for k, g in full['weights'].items():
        terms = torch.stack([o['weights'][k].double() for o in ones])
        err = (g.double() - terms.sum(0)).abs()
        bound = gamma * terms.abs().sum(0)
        assert bool((err <= bound).all()), (k, float((err - bound).max()))


@pytest.mark.parametrize('B,N,model', [(4097, 1, False), (1365, 3, True), (257, 16, False), (13, 5, True)])
def test_head_gradients_within_the_rigorous_summation_bound(B, N, model):
    """dense2 / dense3 weight gradients = sum_b dq_b n_b^T with n read from the forward (bit for bit what the backward
    sums, by the first test), summed in float64: the kernel's error stays within (cs + nchunk) * 2^-24 * sum |dq_b n_b|
    (cs samples per chunk summed by FFMA, then nchunk partials), which at these sizes resolves a single sample;
    likewise the biases against sum_b dq_b."""
    import multiagent_rl_b200 as m
    D, A, out = 10, 5, 4
    rng = np.random.RandomState(B + 7 * N)
    sd = _weights('default', 61 + N, D, A, model, out)
    obs, act = _inputs(rng, B, N, D, A)
    critic = m.FusedCritic(sd, obs_dim=D)
    n = _forward_n(critic, sd, obs, act).double()
    critic.load_state_dict(sd)
    dq, dr = _upstream(rng, B, out, model)
    g = critic.backward(obs, act, dq, dr, want_action=False)['weights']
    _, nchunk, _, csb = _plan(B, N)
    m_ = csb + nchunk
    gamma = m_ * EPS / (1 - m_ * EPS)
    for up, wk, bk in ((dq, 'dense2.weight', 'dense2.bias'), (dr, 'dense3.weight', 'dense3.bias')):
        if up is None:
            continue
        terms = up.double()[:, :, None] * n[:, None, :]  # [B, out, 64]
        err = (g[wk].double() - terms.sum(0)).abs()
        bound = gamma * terms.abs().sum(0)
        assert bool((err <= bound).all()), (wk, float((err - bound).max()))
        # one sample's share is above the bound, so a dropped or doubled sample cannot hide in it
        assert float((terms.abs().max(0).values - bound).max()) > 0, wk
        err = (g[bk].double() - up.double().sum(0)).abs()
        assert bool((err <= gamma * up.double().abs().sum(0)).all()), bk


# ---- 5. the ABI and autograd contracts ----

@pytest.mark.parametrize('model', [False, True], ids=['relu', 'model'])
def test_workspace_is_borrowed_and_outputs_are_overwritten(model):
    """Against fresh FusedCritic.backward calls, bit for bit: a NaN-filled workspace, one workspace used for B = 65,539
    and then for B = 1,000 (64 and 47 chunks), a workspace 4 bytes into a larger buffer; every output NaN-filled."""
    import multiagent_rl_b200 as m
    N, D, A, out, B1, B2 = 3, 10, 5, 2, 65539, 1000
    rng = np.random.RandomState(71 + model)
    sd = _weights('sharp', 71, D, A, model, out)
    obs, act = _inputs(rng, B1, N, D, A)
    dq, dr = _upstream(rng, B1, out, model)
    sl = slice(0, B2)
    drs = None if dr is None else dr[sl]
    critic = m.FusedCritic(sd, obs_dim=D)
    fresh1 = critic.backward(obs, act, dq, dr, want_obs=True)
    fresh2 = critic.backward(obs[sl], act[sl], dq[sl], drs, want_obs=True)
    nb1 = critic._lib.critic_backward_workspace(critic._h, B1, N)
    nb2 = critic._lib.critic_backward_workspace(critic._h, B2, N)
    assert _plan(B1, N)[1] != _plan(B2, N)[1] and nb2 < nb1
    ws = torch.full((nb1 // 4 + 1,), float('nan'), device='cuda')
    _same(_raw_backward(critic, sd, obs, act, dq, dr, ws), fresh1, 'NaN workspace')
    _same(_raw_backward(critic, sd, obs[sl], act[sl], dq[sl], drs, ws), fresh2, 'reused for a smaller batch')
    big = torch.full((nb2 // 4 + 2,), float('nan'), device='cuda')
    _same(_raw_backward(critic, sd, obs[sl], act[sl], dq[sl], drs, big, offset=4), fresh2, 'at a 4-byte offset')


def test_load_and_backward_are_stream_ordered_without_a_host_sync():
    """sleep on a side stream -> load_state_dict(CUDA tensors) -> FusedCritic.backward on that stream: the calls return
    while the sleep still runs, and the gradients are those of an eager call with the loaded weights."""
    import multiagent_rl_b200 as m
    if not hasattr(torch.cuda, '_sleep'):
        pytest.skip('torch.cuda._sleep is not available')
    N, D, A, B, out = 6, 16, 5, 2000, 1
    rng = np.random.RandomState(81)
    w0, w1 = _weights('default', 81, D, A, True, out), _weights('sharp', 82, D, A, True, out)
    obs, act = _inputs(rng, B, N, D, A)
    dq, dr = _upstream(rng, B, out, True)
    want = m.FusedCritic(w1, obs_dim=D).backward(obs, act, dq, dr, want_obs=True)
    critic = m.FusedCritic(w0, obs_dim=D)
    params = {k: torch.from_numpy(v).cuda() for k, v in w1.items()}
    critic.backward(obs, act, dq, dr, want_obs=True)  # the first launches of the process may wait for the device
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(1_000_000_000)  # about 0.5 s at the B200's clocks
        critic.load_state_dict(params)
        got = critic.backward(obs, act, dq, dr, want_obs=True)
        ev = torch.cuda.Event()
        ev.record()
        pending = not ev.query()
    assert pending, 'load_state_dict / backward waited for the GPU'
    torch.cuda.synchronize()
    _same(got, want)


def test_raw_backward_captures_in_a_cuda_graph():
    """critic_backward with static inputs, outputs and a preallocated workspace captured in a graph: each replay after
    new obs / action / dq / dr are copied into the inputs gives an eager call's gradients bit for bit."""
    import multiagent_rl_b200 as m
    from multiagent_rl_b200 import _lib
    N, D, A, B, out = 3, 10, 5, 3000, 2
    rng = np.random.RandomState(91)
    sd = _weights('default', 91, D, A, True, out)
    critic = m.FusedCritic(sd, obs_dim=D)
    obs, act = _inputs(rng, B, N, D, A)
    dq, dr = _upstream(rng, B, out, True)
    nbytes = critic._lib.critic_backward_workspace(critic._h, B, N)
    ws = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
    res = _nan_outputs(sd, obs, act)
    g = _lib.CriticGrads(**{f: res['weights'][k].data_ptr() for f, k in _FIELDS})

    def call():
        return critic._lib.critic_backward(critic._h, _lib.ptr(obs), _lib.ptr(act), B, N, _lib.ptr(dq), _lib.ptr(dr),
                                           _lib.ptr(res['obs']), _lib.ptr(res['action']), C.byref(g), _lib.ptr(ws),
                                           nbytes, _lib.current_stream(obs.device))
    assert call() == _lib.MPE_OK
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        assert call() == _lib.MPE_OK
    for it in range(2):
        o2, a2 = _inputs(rng, B, N, D, A, 'onehot' if it else 'uniform')
        q2, r2 = _upstream(rng, B, out, True)
        for dst, src in ((obs, o2), (act, a2), (dq, q2), (dr, r2)):
            dst.copy_(src)
        for v in [res['obs'], res['action']] + list(res['weights'].values()):
            v.fill_(float('nan'))
        graph.replay()
        torch.cuda.synchronize()
        _same(res, critic.backward(o2, a2, q2, r2, want_obs=True), 'replay %d' % it)


def _train_step(net, opt, obs, act, y):
    out = net(obs, act)
    q = out[0] if net.model else out
    loss = torch.nn.functional.smooth_l1_loss(q, y)
    if net.model:
        loss = loss + out[1].abs().mean()
    loss.backward()
    opt.step()


@pytest.mark.parametrize('model', [False, True], ids=['relu', 'model'])
def test_a_training_step_captures_in_a_cuda_graph(model):
    """One whole FusedCriticNetwork step (forward, SmoothL1 loss, loss.backward(), SGD.step()) captured by torch's
    whole-network recipe (warm-up on a side stream): three replays on three batches end with the parameters of three
    eager steps, bit for bit."""
    import multiagent_rl_b200 as m
    N, D, A, B, lr = 3, 10, 5, 1024, 0.05
    torch.manual_seed(101 + model)
    net = m.FusedCriticNetwork(D + A, 1, model=model).cuda()
    eager = copy.deepcopy(net)
    rng = np.random.RandomState(101)
    batches = []
    for _ in range(3):
        obs, act = _inputs(rng, B, N, D, A)
        batches.append((obs, act, torch.from_numpy(rng.randn(B, 1).astype(np.float32)).cuda()))
    opt_e = torch.optim.SGD(eager.parameters(), lr=lr)
    for obs, act, y in batches:
        opt_e.zero_grad(set_to_none=True)
        _train_step(eager, opt_e, obs, act, y)
    p0 = [p.detach().clone() for p in net.parameters()]
    opt = torch.optim.SGD(net.parameters(), lr=lr)
    s_obs, s_act, s_y = (t.clone() for t in batches[0])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            opt.zero_grad(set_to_none=True)
            _train_step(net, opt, s_obs, s_act, s_y)
    torch.cuda.current_stream().wait_stream(side)
    with torch.no_grad():  # undo the warm-up's updates in place (the graph keeps the parameters' addresses)
        for p, v in zip(net.parameters(), p0):
            p.copy_(v)
    opt.zero_grad(set_to_none=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _train_step(net, opt, s_obs, s_act, s_y)
    for obs, act, y in batches:
        s_obs.copy_(obs)
        s_act.copy_(act)
        s_y.copy_(y)
        graph.replay()
    torch.cuda.synchronize()
    moved = False
    for (k, p), (_, pe), v in zip(net.named_parameters(), eager.named_parameters(), p0):
        assert torch.equal(p, pe), k
        moved |= not torch.equal(p, v)
    assert moved


def test_autograd_asks_only_for_the_gradients_in_use(monkeypatch):
    """A loss on r alone (model critic): the dense2 gradients are None and the rest are critic_backward's with dq = 0
    (bit for bit, and float64 autograd's within 1e-4).  Frozen parameters with obs.requires_grad (relu critic): the
    backward asks for dobs alone, and obs.grad is FusedCritic.backward's dobs."""
    import multiagent_rl_b200 as m
    N, D, A, B = 3, 10, 5, 777
    rng = np.random.RandomState(111)
    torch.manual_seed(111)
    net = m.FusedCriticNetwork(D + A, 1, model=True).cuda()
    sd = {k: v.detach().cpu().numpy() for k, v in net.state_dict().items()}
    obs, act = _inputs(rng, B, N, D, A)
    keep = torch.from_numpy(ct.kink_free(sd, obs.cpu().numpy(), act.cpu().numpy())).cuda()
    obs, act = obs[keep], act[keep]
    B = obs.shape[0]
    _, dr = _upstream(rng, B, 1, True)
    o, a = obs.clone().requires_grad_(True), act.clone().requires_grad_(True)
    (net(o, a)[1] * dr).sum().backward()
    assert net.dense2.weight.grad is None and net.dense2.bias.grad is None
    direct = m.FusedCritic(sd, obs_dim=D).backward(obs, act, torch.zeros(B, 1, device='cuda'), dr, want_obs=True)
    want = ct.grads(sd, obs.cpu().numpy(), act.cpu().numpy(), np.zeros((B, 1)), dr.cpu().numpy())
    assert torch.equal(o.grad, direct['obs']) and torch.equal(a.grad, direct['action'])
    _check(o.grad.cpu().numpy(), want['obs'], 1e-4, 'obs')
    _check(a.grad.cpu().numpy(), want['action'], 1e-4, 'action')
    for k, p in net.named_parameters():
        if not k.startswith('dense2'):
            assert torch.equal(p.grad, direct['weights'][k]), k
            _check(p.grad.cpu().numpy(), want[k], 1e-4, k)

    torch.manual_seed(112)
    net = m.FusedCriticNetwork(D + A, 1).cuda()
    net.requires_grad_(False)
    sd = {k: v.detach().cpu().numpy() for k, v in net.state_dict().items()}
    calls = []
    real = m.FusedCritic.backward

    def spy(self, *args, **kw):
        calls.append(kw)
        return real(self, *args, **kw)
    monkeypatch.setattr(m.FusedCritic, 'backward', spy)
    dq, _ = _upstream(rng, B, 1, False)
    o = obs.clone().requires_grad_(True)
    (net(o, act) * dq).sum().backward()
    assert len(calls) == 1 and calls[0]['want_obs'] and not calls[0]['want_action'] and not calls[0]['want_weights']
    assert all(p.grad is None for p in net.parameters())
    monkeypatch.undo()
    assert torch.equal(o.grad, m.FusedCritic(sd, obs_dim=D).backward(obs, act, dq, want_obs=True)['obs'])


# ---- 6. offsets past 2^31 floats ----

def test_workspace_and_output_offsets_past_2_31_floats():
    """B = 262,145 x 16 agent rows: the per-row records span rows * 512 = 2,147,491,840 floats (the last sample's start
    at 2^31), an 8.6 GB workspace.  One-hot probes in the middle, across the last chunk's boundary and at B - 1 land
    exactly once; the last samples' dobs are those of batches of one; dobs past row B stays NaN."""
    import multiagent_rl_b200 as m
    from multiagent_rl_b200 import _lib
    B, N, D, A, out, pad = 262145, 16, 10, 5, 1, 16
    rows, nchunk, cs, _ = _plan(B, N)
    assert rows * 512 > 2 ** 31
    rng = np.random.RandomState(121)
    sd = _weights('default', 121, D, A, False, out)
    critic = m.FusedCritic(sd, obs_dim=D)
    nbytes = critic._lib.critic_backward_workspace(critic._h, B, N)
    assert nbytes > 2 ** 33
    obs, act = _inputs(rng, B, N, D, A)
    last = (nchunk - 1) * cs  # first row of the last chunk
    for b in ((nchunk // 2 * cs + N - 1) // N, (last - 1) // N, B - 1):
        dq = torch.zeros(B, out, device='cuda')
        dq[b] = 1.5
        full = critic.backward(obs, act, dq, want_obs=True)
        one = _batch_of_one(critic, obs, act, dq, None, b)
        for k in ('obs', 'action'):
            assert torch.equal(full[k][b:b + 1], one[k]), (b, k)
            assert bool((full[k][:b] == 0).all()) and bool((full[k][b + 1:] == 0).all()), (b, k)
        for k, g1 in one['weights'].items():
            g = full['weights'][k]
            if _one_chunk(b, N, cs) or k in HEADS:
                assert torch.equal(g, g1), (b, k)
            else:
                assert float((g - g1).abs().max()) <= 1e-6 * float(g1.abs().max()), (b, k)
        del full
    dq, _ = _upstream(rng, B, out, False)
    dobs = torch.full((B + pad, N, D), float('nan'), device='cuda')
    ws = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
    _lib.check(critic._lib.critic_backward(critic._h, _lib.ptr(obs), _lib.ptr(act), B, N, _lib.ptr(dq), None,
                                           _lib.ptr(dobs), None, None, _lib.ptr(ws), nbytes,
                                           _lib.current_stream(obs.device)), 'critic_backward')
    del ws
    assert bool(torch.isnan(dobs[B:]).all()) and not bool(torch.isnan(dobs[:B]).any())
    for b in (B - 9, B - 3, B - 2, B - 1):
        assert torch.equal(dobs[b:b + 1], _batch_of_one(critic, obs, act, dq, None, b)['obs']), b
    del dobs
    torch.cuda.empty_cache()
