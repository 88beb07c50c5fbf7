"""Philox4x32-10 counter-based RNG in numpy, and the exact bit->float maps the
CUDA kernels use for episode resets and Gumbel noise.

TEST INFRASTRUCTURE (see oracle/__init__.py).  The reference draws reset
positions from numpy's global Mersenne Twister (upstream ``reset_world``) and
Gumbel noise from torch's generator (rls/agent/multiagent/ddpg_gumbel_fix.py:113
-> ``F.gumbel_softmax``); neither stream can be reproduced inside a kernel, so
the batched path defines its own stream keyed by (seed, global env id, episode
or step, slot).  This file is the executable specification of that stream; the
known-answer vectors for Philox4x32-10 itself (Random123 ``kat_vectors``) are
checked in tests/test_oracle.py.

Stream layout (must match multiagent_rl_b200/csrc/common.cuh):
  key      = (seed_lo, seed_hi)
  counter  = (gid_lo, gid_hi, t, (domain << 16) | slot)
  domain 1 = reset positions, t = episode index of that env, slot = entity-pair index:
             call j gives (x, y) of entity 2j and of entity 2j+1, entities ordered
             agents then landmarks (upstream reset order).  pos = (r >> 8) * 2^-23 - 1.
  domain 2 = goal landmarks, t = episode index, slot 0: r0 -> goal of agent 0, r1 -> goal of
             agent 1 ; goal = mulhi(r, L).
  domain 3 = Gumbel noise, t = global step index, slot = agent * 8 + j: call j gives noise
             for head entries 4j..4j+3 of that agent's concatenated logits.
             u = ((r >> 9) + 0.5) * 2^-23 ;  g = -log(-log(u)).
  fullobs_collect_treasure (csrc/env_treasure.cuh):
  domain 1 = as above over 8 agents + 6 treasures; treasure positions are scaled by 0.95.
  domain 2 = treasure types at reset, t = episode: slot 0 gives types 0..3, slot 1 types 4, 5 ; type = r >> 31.
  domain 4 = respawn, t = episode, slot = (step within the episode & 0xFFF) << 4 | treasure:
             r0, r1 -> position (scaled by 0.95), r2 >> 31 -> type, r3 -> the probability draw (prob = 1: passes).
  replay ring (csrc/replay_kernels.cu, k_replay_make_index):
  domain 5 = sampled indices, counter = (j, 0, draw_lo, 5 << 16 | draw_hi & 0xFFFF) for sample j of the ring's
             draw-th make_index call: index = mulhi64((r0 << 32) | r1, len).
"""
import numpy as np

M0 = np.uint64(0xD2511F53)
M1 = np.uint64(0xCD9E8D57)
W0 = 0x9E3779B9
W1 = 0xBB67AE85
MASK = np.uint64(0xFFFFFFFF)

DOMAIN_RESET = 1
DOMAIN_GOAL = 2
DOMAIN_GUMBEL = 3
DOMAIN_RESPAWN = 4
DOMAIN_REPLAY = 5


def philox4x32_10(counter, key):
    """counter: 4 arrays (uint32-valued), key: 2 arrays.  Returns 4 uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint64) & MASK for x in counter]
    c = list(np.broadcast_arrays(*c))
    k0 = np.asarray(key[0], dtype=np.uint64) & MASK
    k1 = np.asarray(key[1], dtype=np.uint64) & MASK
    for r in range(10):
        p0 = M0 * c[0]
        p1 = M1 * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & MASK
        c = [(hi1 ^ c[1] ^ k0) & MASK, lo1, (hi0 ^ c[3] ^ k1) & MASK, lo0]
        k0 = (k0 + np.uint64(W0)) & MASK
        k1 = (k1 + np.uint64(W1)) & MASK
    return [x.astype(np.uint32) for x in c]


def _split64(x):
    x = np.asarray(x, dtype=np.uint64)
    return x & MASK, x >> np.uint64(32)


def raw(seed, gid, t, domain, slot):
    s_lo, s_hi = _split64(np.uint64(seed))
    g_lo, g_hi = _split64(gid)
    ctr3 = (np.uint64(domain) << np.uint64(16)) | np.asarray(slot, dtype=np.uint64)
    return philox4x32_10([g_lo, g_hi, np.asarray(t, dtype=np.uint64), ctr3], [s_lo, s_hi])


def bits_to_pos(r):
    """U[-1, 1): exactly representable in fp32 and fp64."""
    return (r >> np.uint32(8)).astype(np.float64) * (2.0 ** -23) - 1.0


def bits_to_gumbel(r, dtype=np.float64):
    u = ((r >> np.uint32(9)).astype(np.float64) + 0.5) * (2.0 ** -23)
    u = u.astype(dtype)
    return -np.log(-np.log(u))


def reset_positions(seed, gid, episode, n_entities):
    """-> [B, n_entities, 2] float64 positions, entities = agents then landmarks."""
    gid = np.asarray(gid, dtype=np.uint64)
    episode = np.broadcast_to(np.asarray(episode, dtype=np.uint64), gid.shape)
    out = np.zeros(gid.shape + (n_entities, 2))
    for j in range((n_entities + 1) // 2):
        r = raw(seed, gid, episode, DOMAIN_RESET, j)
        out[..., 2 * j, 0] = bits_to_pos(r[0])
        out[..., 2 * j, 1] = bits_to_pos(r[1])
        if 2 * j + 1 < n_entities:
            out[..., 2 * j + 1, 0] = bits_to_pos(r[2])
            out[..., 2 * j + 1, 1] = bits_to_pos(r[3])
    return out


def reset_goals(seed, gid, episode, n_goals, L):
    """-> [B, n_goals] int landmark indices (n_goals <= 4)."""
    gid = np.asarray(gid, dtype=np.uint64)
    episode = np.broadcast_to(np.asarray(episode, dtype=np.uint64), gid.shape)
    r = raw(seed, gid, episode, DOMAIN_GOAL, 0)
    out = np.zeros(gid.shape + (n_goals,), dtype=np.int64)
    for i in range(n_goals):
        out[..., i] = ((r[i].astype(np.uint64) * np.uint64(L)) >> np.uint64(32)).astype(np.int64)
    return out


def gumbel_noise(seed, gid, step, n_agents, width, dtype=np.float64):
    """-> [B, n_agents, width] Gumbel(0,1) noise for the concatenated logits of each agent."""
    gid = np.asarray(gid, dtype=np.uint64)
    step = np.broadcast_to(np.asarray(step, dtype=np.uint64), gid.shape)
    out = np.zeros(gid.shape + (n_agents, width), dtype=dtype)
    for a in range(n_agents):
        for j in range((width + 3) // 4):
            r = raw(seed, gid, step, DOMAIN_GUMBEL, a * 8 + j)
            for q in range(4):
                if 4 * j + q < width:
                    out[..., a, 4 * j + q] = bits_to_gumbel(r[q], dtype)
    return out


def treasure_reset(seed, gid, episode):
    """fullobs_collect_treasure reset -> (agent pos [B,8,2], treasure pos [B,6,2], treasure types [B,6])."""
    pos = reset_positions(seed, gid, episode, 14)
    gid = np.asarray(gid, dtype=np.uint64)
    episode = np.broadcast_to(np.asarray(episode, dtype=np.uint64), gid.shape)
    r0 = raw(seed, gid, episode, DOMAIN_GOAL, 0)
    r1 = raw(seed, gid, episode, DOMAIN_GOAL, 1)
    types = np.stack([(x >> np.uint32(31)).astype(np.int64) for x in (r0[0], r0[1], r0[2], r0[3], r1[0], r1[1])], axis=-1)
    return pos[..., :8, :], pos[..., 8:, :] * 0.95, types


def treasure_respawn(seed, gid, episode, tstep, treasure):
    """-> (position [.., 2], type) of a treasure that respawns in post_step of step `tstep` of episode `episode`."""
    slot = ((np.asarray(tstep, dtype=np.uint64) & np.uint64(0xFFF)) << np.uint64(4)) | np.asarray(treasure, dtype=np.uint64)
    r = raw(seed, gid, episode, DOMAIN_RESPAWN, slot)
    pos = np.stack([bits_to_pos(r[0]), bits_to_pos(r[1])], axis=-1) * 0.95
    return pos, (r[2] >> np.uint32(31)).astype(np.int64)


def mulhi64(x, y):
    """High 64 bits of the 128-bit product of two uint64 arrays (CUDA's __umul64hi), from 32-bit limbs."""
    x, y = np.asarray(x, dtype=np.uint64), np.asarray(y, dtype=np.uint64)
    s32 = np.uint64(32)
    xl, xh, yl, yh = x & MASK, x >> s32, y & MASK, y >> s32
    ll, lh, hl, hh = xl * yl, xl * yh, xh * yl, xh * yh
    mid = (ll >> s32) + (lh & MASK) + (hl & MASK)  # < 3 * 2^32: no overflow
    return hh + (lh >> s32) + (hl >> s32) + (mid >> s32)


def replay_index(seed, draw, batch, size):
    """-> [batch] int64: the indices of the replay ring's draw-th make_index call on a ring holding `size`
    transitions (uniform on [0, size) with replacement)."""
    draw = int(draw)
    r = raw(seed, np.arange(int(batch), dtype=np.uint64), draw & 0xFFFFFFFF, DOMAIN_REPLAY, (draw >> 32) & 0xFFFF)
    x = (r[0].astype(np.uint64) << np.uint64(32)) | r[1].astype(np.uint64)
    return mulhi64(x, np.uint64(size)).astype(np.int64)
