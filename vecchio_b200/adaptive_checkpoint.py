"""Checkpoint / resume of an adaptive render session (``Context.adaptive_session``).

A session's state is integers: per pixel the fixed-point sums and squares of its samples [0, n) and the count n, plus the
last target it reached.  Philox is keyed by (pixel, global sample), so a session that imports this state and refines on
renders exactly what an uninterrupted one would (include/vecchio_gpu.h, vk_adaptive_import).  The library cannot see
whether a state belongs to its scene, cameras and parameters, so the checkpoint carries that identity and refuses to load
into another one.  The format follows ``accumulate.FrameAccumulator``: one ``.npz`` written to a temporary name and renamed.

Nothing here renders: ``render_adaptive_resumable`` drives whatever object offers the session's methods.
"""
import json
import os

import numpy as np

from .accumulate import frame_key

_FORMAT = 1


def session_key(scene_name, scene_seed, cams, params, pass_spp, variant, scene_param=0, shard=None):
    """Identity of a session's state: ``frame_key`` of its first camera with the hashes of ALL its cameras, plus
    ``pass_spp`` (the pass grid the counts lie on) and the kernel that ran (``variant``: the render build's kernels may
    round differently).  ``params.spp`` in it is the session's limit.  A shard session's key adds ``"shard": [k, n]``, so
    its partial state never loads into a whole session; a whole state's key (one GPU or several) has no such entry."""
    cams = list(cams)
    if not cams:
        raise ValueError("session_key: at least one camera")
    keys = [frame_key(scene_name, scene_seed, c, params, scene_param) for c in cams]
    key = dict(keys[0])
    key["camera"] = [k["camera"] for k in keys]
    key["pass_spp"] = int(pass_spp)
    key["variant"] = int(variant)
    if shard is not None:
        key["shard"] = [int(shard[0]), int(shard[1])]
    return key


def _key_mismatch(a, b):
    return sorted(k for k in set(a) | set(b) if a.get(k) != b.get(k))


def save_state(path, key, sums, squares, counts, reached):
    """Writes the exported state (``reached`` = (spp, min_spp, max_error), or None for a session that reached no
    target) to ``path`` through a temporary file: an interrupted save leaves the previous checkpoint as it was."""
    reached = (0, 0, 0.0) if reached is None else reached
    meta = {"format": _FORMAT, "key": key, "reached": [int(reached[0]), int(reached[1]), float(np.float32(reached[2]))]}
    arrays = {"meta": np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8),
              "sums": np.ascontiguousarray(sums, dtype=np.int64), "squares": np.ascontiguousarray(squares, dtype=np.uint64),
              "counts": np.ascontiguousarray(counts, dtype=np.uint32)}
    tmp = f"{path}.tmp{os.getpid()}"
    try:
        with open(tmp, "wb") as f:
            np.savez(f, **arrays)
        os.replace(tmp, path)
    finally:
        if os.path.exists(tmp):
            os.remove(tmp)


def load_state(path, key):
    """(sums, squares, counts, reached) of a checkpoint written for ``key``; ValueError for another identity or
    format.  ``reached`` is None for a state that reached no target."""
    with np.load(path) as z:
        meta = json.loads(bytes(z["meta"]).decode())
        if meta.get("format") != _FORMAT:
            raise ValueError(f"{path}: unknown checkpoint format {meta.get('format')}")
        diff = _key_mismatch(meta["key"], dict(key))
        if diff:
            raise ValueError(f"{path}: the checkpoint is of another session (differs in {', '.join(diff)})")
        sums, squares, counts = z["sums"], z["squares"], z["counts"]
    if sums.shape != squares.shape or sums.shape[:-1] != counts.shape or sums.shape[-1:] != (3,):
        raise ValueError(f"{path}: array shapes {sums.shape}, {squares.shape}, {counts.shape} do not fit together")
    spp, min_spp, max_error = meta["reached"]
    reached = None if spp == 0 else (int(spp), int(min_spp), float(max_error))
    return sums, squares, counts, reached


def render_adaptive_resumable(session, targets, checkpoint_path, key):
    """Refines ``session`` through ``targets`` (each ``(max_error, spp, min_spp)``; spp None = the session's limit),
    saving to ``checkpoint_path`` after each.  When the checkpoint exists it is loaded first and the targets up to the
    one it reached are skipped, so a run interrupted at any point resumes where it stopped and ends with the state an
    uninterrupted run reaches.  Returns the number of refines run."""
    targets = [session.target(*t) for t in targets]
    start = 0
    if os.path.exists(checkpoint_path):
        session.load(checkpoint_path, key)
        if session.reached is not None and session.reached in targets:
            start = len(targets) - targets[::-1].index(session.reached)
    n = 0
    for t in targets[start:]:
        session.refine(t[2], spp=t[0], min_spp=t[1])
        session.save(checkpoint_path, key)
        n += 1
    return n
