"""Restatement of the reference replay ring (rls/replay_buffer.py:9-60: ReplayBuffer.add / _encode_sample /
sample_index) fed the way experiments/run.py:46,52 feeds it.  TEST INFRASTRUCTURE (see oracle/__init__.py).
Pinned against the reference's own class in tests/test_reference_exec.py where it is compiled into oracle/_ref."""
import numpy as np


class ReplayRing(object):
    def __init__(self, size):
        self._storage = []
        self._maxsize = int(size)
        self._next_idx = 0

    def __len__(self):
        return len(self._storage)

    def add(self, obs_t, action, reward, obs_tp1, done):
        data = (obs_t, action, reward, obs_tp1, done)
        if self._next_idx >= len(self._storage):
            self._storage.append(data)
        else:
            self._storage[self._next_idx] = data
        self._next_idx = (self._next_idx + 1) % self._maxsize

    def sample_index(self, idxes):
        cols = [[], [], [], [], []]
        for i in idxes:
            for c, v in zip(cols, self._storage[i]):
                c.append(np.asarray(v))
        return tuple(np.array(c) for c in cols)


def add_batched_step(ring, obs, act_onehot, rew, obs_next, done=None):
    """What the reference loop does for every env of a batched step, in env order (run.py:46,52)."""
    for b in range(obs.shape[0]):
        ring.add(list(obs[b]), list(act_onehot[b]), np.sum(rew[b]), list(obs_next[b]),
                 float(done[b]) if done is not None else 0.0)
