"""Multi-GPU sharding of grasp candidates: contiguous blocks, labels gathered at the end.

Candidates are independent (the reference resets the simulation at the top of every loop
iteration, /root/reference/mgs/env/gravityless_object_grasping.py:158), so ranks exchange nothing
during the rollout; the only collective is an all_gather of the uint8 labels (SURVEY.md 8(e)).
Works with any torch.distributed backend (NCCL on the GPU box, gloo in the CPU tests).
"""
from __future__ import annotations

import numpy as np


def shard_range(n: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous block [lo, hi) of ceil(n/world) candidates for `rank` (keeps enough_stable's prefix
    semantics cheap: a rank's block is a contiguous piece of the sequential order)."""
    per = -(-n // world) if world > 0 else n
    lo = min(n, rank * per)
    return lo, min(n, lo + per)


def gather_labels(local: np.ndarray, n: int, group=None, device=None) -> np.ndarray:
    """all_gather of per-rank label blocks -> bool[n] on every rank (padding trimmed)."""
    import torch
    import torch.distributed as dist
    if not dist.is_available() or not dist.is_initialized():
        return np.asarray(local, dtype=bool)
    world = dist.get_world_size(group)
    per = -(-n // world)
    buf = torch.zeros(per, dtype=torch.uint8, device=device)
    buf[: len(local)] = torch.as_tensor(np.asarray(local, dtype=np.uint8), device=device)
    out = torch.empty(world * per, dtype=torch.uint8, device=device)
    dist.all_gather_into_tensor(out, buf, group=group)
    out = out.cpu().numpy().astype(bool)
    pieces = []
    for r in range(world):
        lo, hi = shard_range(n, r, world)
        pieces.append(out[r * per: r * per + (hi - lo)])
    return np.concatenate(pieces) if pieces else np.zeros(0, dtype=bool)


def apply_enough_stable(labels: np.ndarray, enough_stable) -> np.ndarray:
    """Sequential `enough_stable` semantics of the reference loop (:151-156, :278-279): once that many
    successes have been seen, every later candidate is labelled False."""
    labels = np.asarray(labels, dtype=bool)
    if enough_stable is None:
        return labels
    before = np.concatenate([[0], np.cumsum(labels)[:-1]])
    return labels & (before < enough_stable)


def dist_state():
    """(world, rank, device for collectives) of the initialised default process group, else (1, 0, None)."""
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            import torch
            dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else None
            return dist.get_world_size(), dist.get_rank(), dev
    except Exception:
        pass
    return 1, 0, None


def evaluate_sharded(n: int, run_range, enough_stable=None, chunk: int = 0) -> np.ndarray:
    """Labels bool[n] of candidates 0..n-1, evaluated by `run_range(lo, hi) -> bool[hi-lo]` on this rank's share.

    Without `enough_stable`: one contiguous block per rank, one label gather.  With it, the reference's early stop
    (gravityless_object_grasping.py:151-156: once `enough_stable` successes were seen the remaining candidates are
    labelled False WITHOUT being simulated) is kept: candidates are evaluated in sequential rounds of world x `chunk`
    (one chunk = what keeps one GPU full, so a smaller round would not finish sooner), the round's labels are gathered,
    and the loop stops as soon as the running success count reaches `enough_stable`.  The returned array equals the
    reference's sequential result."""
    world, rank, dev = dist_state()
    if enough_stable is None:
        if world == 1:
            return np.asarray(run_range(0, n), dtype=bool)
        lo, hi = shard_range(n, rank, world)
        return gather_labels(run_range(lo, hi), n, device=dev)
    chunk = max(1, int(chunk) if chunk else n)
    labels = np.zeros(n, dtype=bool)
    done, count = 0, 0
    while done < n and count < enough_stable:
        rn = min(n - done, world * chunk)
        lo, hi = shard_range(rn, rank, world)
        local = np.asarray(run_range(done + lo, done + hi), dtype=bool) if hi > lo else np.zeros(0, dtype=bool)
        got = gather_labels(local, rn, device=dev) if world > 1 else local
        labels[done:done + rn] = got
        count += int(got.sum())
        done += rn
    return apply_enough_stable(labels, enough_stable)


def scene_round_robin(scene_index) -> np.ndarray:
    """Launch order for candidates of several scenes: the first candidate of every scene (in scene order), then the second of
    every scene, and so on.  Each scene's own candidates keep their order, which is what the device enough_stable early stop
    needs (include/mgs_b200.h, mgs_clutter_scenes_*).  Returns `order` (launch position j runs candidate order[j]); results
    come back with `out[order] = launched`."""
    s = np.asarray(scene_index, dtype=np.int64).reshape(-1)
    if not len(s):
        return np.zeros(0, dtype=np.int64)
    by_scene = np.argsort(s, kind="stable")
    first = np.concatenate([[0], np.nonzero(np.diff(s[by_scene]))[0] + 1])
    rank = np.empty(len(s), dtype=np.int64)
    rank[by_scene] = np.arange(len(s)) - np.repeat(first, np.diff(np.concatenate([first, [len(s)]])))
    return np.lexsort((s, rank))


def plan_scenes(counts, world: int) -> list:
    """Whole scenes per rank, balanced by candidate count (longest-processing-time first; ties to the lower rank).  Returns per-rank
    sorted lists of scene indices."""
    load = [0] * world
    plan = [[] for _ in range(world)]
    for s in sorted(range(len(counts)), key=lambda s: (-int(counts[s]), s)):
        r = min(range(world), key=lambda r: (load[r], r))
        plan[r].append(s)
        load[r] += int(counts[s])
    return [sorted(p) for p in plan]


def evaluate_scenes_sharded(scene_index, nscene: int, run_scenes) -> np.ndarray:
    """Labels bool[n] of candidates of several scenes, each rank evaluating whole scenes: `run_scenes(candidates) -> bool[len]` runs the
    given candidate indices (in increasing order, all of this rank's scenes) on this rank's GPU.  A scene's enough_stable early stop
    never crosses ranks this way.  The labels are combined by one MAX all-reduce of the full uint8 array (every candidate is
    written by exactly one rank), as mixed.run_mixed does."""
    s = np.asarray(scene_index, dtype=np.int64).reshape(-1)
    world, rank, dev = dist_state()
    if world == 1:
        return np.asarray(run_scenes(np.arange(len(s))), dtype=bool)
    mine = plan_scenes(np.bincount(s, minlength=nscene), world)[rank]
    idx = np.nonzero(np.isin(s, mine))[0]
    local = np.zeros(len(s), dtype=np.uint8)
    if len(idx):
        local[idx] = np.asarray(run_scenes(idx), dtype=np.uint8)
    import torch
    import torch.distributed as dist
    flat = torch.as_tensor(local, device=dev)
    dist.all_reduce(flat, op=dist.ReduceOp.MAX)
    return flat.cpu().numpy().astype(bool)
