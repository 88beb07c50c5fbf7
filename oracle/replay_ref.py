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


def shared_reward(rew):
    """[B, N] per-agent rewards -> [B] float32 shared reward, summed in fp32 one agent at a time in agent order (what
    the ring's add kernel computes; np.sum's pairwise order can differ from it in the last bit)."""
    rew = np.asarray(rew, dtype=np.float32)
    s = np.zeros(rew.shape[0], dtype=np.float32)
    for n in range(rew.shape[1]):
        s = s + rew[:, n]
    return s


class BatchedRing(object):
    """Vectorised model of the device replay ring: ``ReplayRing`` fed by ``add_batched_step``, by index arithmetic.

    A batched add of B transitions writes row b to slot (head + b) % capacity, the last writer winning; every slot
    remembers which add and which row of it wrote it (``source``), so expectations can be gathered from the added
    tensors themselves - numpy arrays kept by ``add``, or device tensors the caller holds after ``add_rows``."""

    def __init__(self, size, act_dims):
        self._maxsize = int(size)
        self.act_dims = [int(act_dims)] if np.isscalar(act_dims) else [int(a) for a in act_dims]
        self._next_idx = 0
        self._len = 0
        self._add = np.full(self._maxsize, -1, dtype=np.int64)  # slot -> add number
        self._row = np.full(self._maxsize, -1, dtype=np.int64)  # slot -> row within that add
        self._data = []

    def __len__(self):
        return self._len

    def add_rows(self, B):
        """The index arithmetic of one batched add of B transitions; returns the add's number."""
        k, B = len(self._data), int(B)
        rows = np.arange(max(0, B - self._maxsize), B)  # a batch longer than the ring keeps only its last rows
        slots = (self._next_idx + rows) % self._maxsize
        self._add[slots], self._row[slots] = k, rows
        self._next_idx = (self._next_idx + B) % self._maxsize
        self._len = min(self._maxsize, self._len + B)
        self._data.append(None)
        return k

    def add(self, obs, act_u, rew, obs_next, done=None, act_c=None):
        """obs / obs_next [B,N,D], act_u / act_c [B,N] head indices, rew [B,N], done [B] or None (stored as 0)."""
        obs = np.asarray(obs, dtype=np.float32)
        B = obs.shape[0]
        onehot = np.eye(self.act_dims[0], dtype=np.float32)[np.asarray(act_u)]
        if len(self.act_dims) > 1 and self.act_dims[1] > 0:
            onehot = np.concatenate([onehot, np.eye(self.act_dims[1], dtype=np.float32)[np.asarray(act_c)]], axis=-1)
        dn = np.zeros(B, np.float32) if done is None else np.asarray(done, dtype=np.float32)
        k = self.add_rows(B)
        self._data[k] = (obs, onehot, shared_reward(rew), np.asarray(obs_next, dtype=np.float32), dn)
        return k

    def slots(self, idxes, clamp=False):
        """Ring slots of ``_storage[i]``: Python list indexing (IndexError out of range), or with ``clamp`` the
        device-index rule of the gather kernels (negatives wrap once, whatever is still outside [0, len) is clamped)."""
        idx = np.asarray(idxes, dtype=np.int64).reshape(-1)
        n = self._len
        if not clamp and idx.size and (idx.min() < -n or idx.max() >= n):
            raise IndexError('replay index out of range (len %d)' % n)
        idx = np.where(idx < 0, idx + n, idx)
        return np.clip(idx, 0, n - 1)

    def source(self, idxes, clamp=False):
        """-> (add number, row) of the transition each index reads."""
        s = self.slots(idxes, clamp)
        return self._add[s], self._row[s]

    def sample_index(self, idxes, clamp=False):
        """-> (obs [n,N,D], act one-hot [n,N,A], rew_shared [n], obs_next [n,N,D], done [n]) float32 arrays."""
        add, row = self.source(idxes, clamp)
        out = None
        for k, data in enumerate(self._data):
            sel = add == k
            if out is None:
                out = [np.zeros((add.size,) + d.shape[1:], dtype=np.float32) for d in data]
            for o, d in zip(out, data):
                o[sel] = d[row[sel]]
        return tuple(out)

    def collect(self):
        return self.sample_index(np.arange(self._len))
