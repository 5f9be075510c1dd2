"""The host model of adaptive sampling (adaptive_model.py) restricted to one shard of pixels, as vk_adaptive_begin_shard
renders it: batch-wide pixel g belongs to shard (g // 32) % n_shards, a shard's pass loop lists only the pixels it owns,
and the others keep what they hold (zero in a shard session)."""
import numpy as np

import adaptive_model as am

SHARD_RUN = 32  # VK_SHARD_RUN


def owned(shape, shard, n_shards):
    """The pixels of a state of this shape (frames, rows bottom-up, columns: the accumulators' order) that shard `shard`
    of n_shards owns."""
    g = np.arange(int(np.prod(shape)), dtype=np.int64).reshape(shape)
    return (g // SHARD_RUN) % n_shards == shard


def predict_shard(states, target, M, shard, start=None):
    """am.predict over the pixels shard = (k, n_shards) owns, the others left at their start (zero for a fresh session).
    Every step of the pass loop is per pixel, so it runs am.predict on the owned pixels alone and puts them back."""
    shape = states[am.grid(M, target[0])[0]][0].shape[:-1]
    idx = np.flatnonzero(owned(shape, *shard).reshape(-1))
    if start is None:
        s0 = states[am.grid(M, target[0])[0]]
        start = (np.zeros(shape, np.uint32), np.zeros_like(s0[0]), np.zeros_like(s0[1]))
    n, S, Q = (np.array(a) for a in start)
    n = n.astype(np.uint32)
    sub = {b: (st[0].reshape(-1, 3)[idx], st[1].reshape(-1, 3)[idx]) for b, st in states.items()}
    n_o, S_o, Q_o = am.predict(sub, target, M, start=(n.reshape(-1)[idx], S.reshape(-1, 3)[idx], Q.reshape(-1, 3)[idx]))
    n.reshape(-1)[idx] = n_o
    S.reshape(-1, 3)[idx] = S_o
    Q.reshape(-1, 3)[idx] = Q_o
    return n, S, Q
