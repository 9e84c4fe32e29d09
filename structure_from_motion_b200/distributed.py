"""Multi-GPU plumbing for the two shardings of the path (SURVEY.md §8(e)).

* hypothesis-sharded (one large pair): correspondences replicated, rank r evaluates the
  global hypothesis indices [r*H, (r+1)*H); the per-rank winners are merged by ONE tiny
  collective (an all-gather of 12 doubles per rank) and every rank applies the reference's
  selection rule (lib/ransac/ransac.py:83: smallest error, earliest iteration on ties).
* pair-sharded (batches of independent pairs): no data-path communication at all.

torch.distributed is plumbing only (NCCL on the GPUs, gloo in the CPU tests); the merge
itself is a dozen scalar comparisons.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence

import numpy as np


def shard_range(total: int, rank: int, world: int):
    """Contiguous, balanced partition of ``total`` items: returns (start, stop) for ``rank``."""
    base, rem = divmod(int(total), int(world))
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def pack_local_best(err: float, index: int, count: int, E) -> np.ndarray:
    """12 doubles: err, global index (exact in a double up to 2^53), count, E[9]."""
    out = np.empty(12, dtype=np.float64)
    out[0] = err if index >= 0 else math.inf
    out[1] = float(index)
    out[2] = float(count)
    out[3:] = np.asarray(E, dtype=np.float64).reshape(9) if index >= 0 else 0.0
    return out


def merge_best(rows: np.ndarray, selection: str = "min_error"):
    """Pick the global winner from per-rank rows (see pack_local_best).

    min_error: smallest error, lowest global index on ties (ransac.py:83 keeps the earliest
    iteration; "msac" merges the same way, the error being the MSAC cost).  max_inliers: largest count,
    lowest index on ties.  Returns
    (owner_rank, err, index, count, E) or (-1, inf, -1, -1, None) when no rank has a candidate.
    """
    rows = np.asarray(rows, dtype=np.float64).reshape(-1, 12)
    best = -1
    for r in range(rows.shape[0]):
        if rows[r, 1] < 0:
            continue
        if best < 0:
            best = r
            continue
        if selection == "max_inliers":
            better = (rows[r, 2], -rows[r, 1]) > (rows[best, 2], -rows[best, 1])
        else:
            better = (rows[r, 0], rows[r, 1]) < (rows[best, 0], rows[best, 1])
        if better:
            best = r
    if best < 0:
        return -1, math.inf, -1, -1, None
    return best, float(rows[best, 0]), int(rows[best, 1]), int(rows[best, 2]), rows[best, 3:].reshape(3, 3).copy()


def all_gather_best(local: np.ndarray, group=None, device=None) -> np.ndarray:
    """The one collective of the hypothesis-sharded mode: all-gather of 12 doubles per rank."""
    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return np.asarray(local, dtype=np.float64).reshape(1, 12)
    world = dist.get_world_size(group)
    backend = dist.get_backend(group)
    dev = device if device is not None else (torch.device("cuda", torch.cuda.current_device())
                                             if backend == "nccl" else torch.device("cpu"))
    t = torch.from_numpy(np.asarray(local, dtype=np.float64).reshape(12)).to(dev)
    if backend == "nccl":
        out = torch.empty(world * 12, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(out, t, group=group)
        return out.view(world, 12).cpu().numpy()
    parts = [torch.empty(12, dtype=torch.float64) for _ in range(world)]
    dist.all_gather(parts, t, group=group)
    return torch.stack(parts).numpy()


def ransac_essential_sharded(camera_matrix, pts_a, pts_b, threshold, min_num_extra_inliers, aggregation,
                             hyps_per_rank: int, seed: int, *, engine, rank: int, world: int,
                             selection: str = "min_error", group=None, resident: bool = False):
    """One estimate with hypotheses sharded over ``world`` GPUs (device sampler).

    Every rank holds the full correspondence set (``resident=True``: already uploaded to
    ``engine``) and scores its own ``hyps_per_rank`` hypotheses; one all-gather merges the
    winners; every rank then adopts the global winner (so the inlier mask / pose /
    triangulation tail can run anywhere).  Returns dict(err, index, count, E, owner).
    """
    if not resident:
        engine.upload_pairs(pts_a, pts_b, camera_matrix)
    engine.sample_device(seed, hyps_per_rank, hyp_offset=rank * hyps_per_rank)
    best, _, _ = engine.ransac_essential(threshold, float(min_num_extra_inliers or 0), aggregation, selection,
                                         want_mask=False, want_sed=False)
    gidx = int(best.index) + rank * hyps_per_rank if best.index >= 0 else -1
    rows = all_gather_best(pack_local_best(best.err, gidx, best.count_extra, list(best.E)), group=group)
    owner, err, index, count, E = merge_best(rows, selection)
    if owner >= 0:
        if owner == rank:
            engine.set_winner(int(best.index))
        else:
            engine.set_winner(-1, E)
    return dict(err=err, index=index, count=count, E=E, owner=owner,
                num_invalid=int(best.num_invalid))


class _DeviceBuffer:
    """Zero-copy view of library-owned device memory for torch (``torch.as_tensor`` reads __cuda_array_interface__)."""

    def __init__(self, ptr: int, n_doubles: int):
        self.__cuda_array_interface__ = {"shape": (n_doubles,), "typestr": "<f8", "data": (ptr, False), "version": 3}


def two_view_sharded(threshold, min_num_extra_inliers, aggregation, hyps_per_rank: int, seed: int, *, engine, rank: int,
                     world: int, selection: str = "min_error", distance_threshold: float = 50.0, group=None,
                     native: bool = False):
    """One complete estimate (RANSAC E -> cheirality vote -> triangulation) with the hypotheses sharded over ``world``
    GPUs and NO host round trip between scoring and the final results: every rank scores its hypotheses
    (``sfm_score_async``), the 144-byte selection records are all-gathered device-to-device by NCCL on the engine's
    stream — the path's only collective — and merged by a kernel with the reference's rule (``sfm_sharded_tail``),
    which also enqueues the inlier mask, pose vote and triangulation of the global winner.  The correspondences must
    already be resident (``engine.upload_pairs``).  ``native=True``: the all-gather is issued by the library itself on the
    communicator of ``Engine.nccl_init`` (no torch involved); otherwise torch.distributed's NCCL group is used and the engine
    is put on torch's current stream.
    Returns dict(err, index (global), count, E, owner, num_invalid, poses, num_inliers, inlier_idx, pass_bits, points)."""
    if native:
        # the communicator lives behind the C ABI (Engine.nccl_init): sample -> fit -> score -> ncclAllGather ->
        # merge -> tail in ONE C call, no torch on the data path
        engine.two_view_sharded(seed, hyps_per_rank, threshold, float(min_num_extra_inliers or 0), aggregation, selection,
                                distance_threshold)
        best, owner, poses, num, idx, ok, X = engine.sharded_fetch()
        return dict(err=float(best.err), index=int(best.index), count=int(best.count_extra),
                    E=np.array(best.E, dtype=np.float64).reshape(3, 3), owner=owner, num_invalid=int(best.num_invalid),
                    poses=poses, num_inliers=num, inlier_idx=idx, pass_bits=ok, points=X)
    import torch
    import torch.distributed as dist

    n_doubles = engine.RECORD_BYTES // 8
    dev = torch.device("cuda", engine.device)
    # the all-gather reads the record K3 writes and the tail reads what the all-gather writes: everything has to be
    # enqueued on ONE stream - torch's current stream of the engine's device, which NCCL orders itself with
    engine.set_stream(torch.cuda.current_stream(dev).cuda_stream)
    engine.sample_device(seed, hyps_per_rank, hyp_offset=rank * hyps_per_rank)
    rec_ptr = engine.score_async(threshold, float(min_num_extra_inliers or 0), aggregation, selection)
    mine = torch.as_tensor(_DeviceBuffer(rec_ptr, n_doubles), device=dev)
    if world > 1:
        gathered = torch.empty(world * n_doubles, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(gathered, mine, group=group)
    else:
        gathered = mine
    engine.sharded_tail(gathered.data_ptr(), world, rank, hyps_per_rank, threshold, distance_threshold, selection)
    best, owner, poses, num, idx, ok, X = engine.sharded_fetch()
    return dict(err=float(best.err), index=int(best.index), count=int(best.count_extra),
                E=np.array(best.E, dtype=np.float64).reshape(3, 3), owner=owner, num_invalid=int(best.num_invalid),
                poses=poses, num_inliers=num, inlier_idx=idx, pass_bits=ok, points=X, _keep=gathered)


def shard_pairs(offsets: Sequence[int], rank: int, world: int):
    """Pair-sharded mode: the pairs [p0, p1) this rank owns and their re-based offsets."""
    offsets = np.asarray(offsets, dtype=np.int64)
    p0, p1 = shard_range(len(offsets) - 1, rank, world)
    return p0, p1, offsets[p0:p1 + 1] - offsets[p0]


def _merge_chunks(parts: list) -> dict:
    """The dicts of consecutive chunks of pairs as one dict: arrays concatenated, ``inlier_offsets`` re-based, nested
    dicts merged alike."""
    out = {}
    for key, v in parts[0].items():
        if isinstance(v, dict):
            out[key] = _merge_chunks([p[key] for p in parts])
        elif key == "inlier_offsets":
            base, segs = 0, [np.zeros(1, dtype=np.int64)]
            for p in parts:
                segs.append(p[key][1:] + base)
                base += int(p[key][-1])
            out[key] = np.concatenate(segs)
        else:
            out[key] = np.concatenate([p[key] for p in parts])
    return out


class PairPipeline:
    """Pair-sharded batches from HOST buffers with the H2D copy of one chunk hidden behind the kernels of another:
    the pairs are cut into chunks that alternate between ``depth`` contexts on the same GPU (each with its own
    non-blocking stream), driven by one thread per context (ctypes releases the GIL during the C call).  Results are
    identical to one ``Engine.batch_ransac`` call over all pairs: the device sampler is keyed by (seed, global pair
    id, hypothesis), not by the chunking."""

    def __init__(self, device: Optional[int] = None, depth: int = 2):
        from concurrent.futures import ThreadPoolExecutor

        from . import _native

        dev = _native.default_device() if device is None else int(device)
        self.engines = [_native.Engine(dev) for _ in range(depth)]
        self.pool = ThreadPoolExecutor(max_workers=depth)

    def set_score_variant(self, *a, **k):
        for e in self.engines:
            e.set_score_variant(*a, **k)

    def launches(self) -> int:
        return sum(e.get_timing()[1] for e in self.engines)

    def batch_ransac(self, pts_a, pts_b, offsets, Ks, h, seed, threshold, min_extra=0.0, aggregation="rms",
                     selection="min_error", pair_id0=0, chunk_pairs: Optional[int] = None):
        offsets = np.asarray(offsets, dtype=np.int64)
        P = len(offsets) - 1
        Ks = np.asarray(Ks, dtype=np.float64).reshape(P, 3, 3)
        depth = len(self.engines)
        if chunk_pairs is None:
            # uneven chunks de-phase the contexts: equal chunks would copy at the same time and compute at the same
            # time; a short first chunk lets context 0 compute while context 1 still copies, and so on
            fr = np.cumsum([0.0, 1 / 8, 3 / 8, 3 / 8, 1 / 8]) if depth == 2 else np.linspace(0.0, 1.0, 2 * depth + 1)
            bounds = sorted(set(int(round(f * P)) for f in fr))
        else:
            bounds = list(range(0, P, chunk_pairs)) + [P]

        def run(k):
            p0, p1 = bounds[k], bounds[k + 1]
            lo, hi = int(offsets[p0]), int(offsets[p1])
            return self.engines[k % depth].batch_ransac(pts_a[lo:hi], pts_b[lo:hi], offsets[p0:p1 + 1] - lo, Ks[p0:p1], h,
                                                        seed, threshold, min_extra, aggregation, selection,
                                                        pair_id0=pair_id0 + p0)

        # chunk k runs on engine k % depth; a worker thread keeps one engine busy with its chunks in order
        def worker(e):
            return [(k, run(k)) for k in range(e, len(bounds) - 1, depth)]

        parts = dict(kv for res in self.pool.map(worker, range(depth)) for kv in res)
        keys = parts[0].keys()
        return {key: np.concatenate([parts[k][key] for k in range(len(bounds) - 1)]) for key in keys}

    def _chunked(self, call, pts_a, pts_b, offsets, Ks, pair_id0, chunk_pairs):
        """call(engine, pts_a, pts_b, offsets, Ks, pair_id0) over chunks of pairs that alternate between the contexts,
        merged into the dict of one call over all pairs: per-pair and per-inlier arrays are concatenated,
        ``inlier_offsets`` re-based, nested dicts merged the same way."""
        offsets = np.asarray(offsets, dtype=np.int64)
        P = len(offsets) - 1
        Ks = np.asarray(Ks, dtype=np.float64).reshape(P, 3, 3)
        depth = len(self.engines)
        if chunk_pairs is None:
            chunk_pairs = max(1, -(-P // (4 * depth)))
        bounds = list(range(0, P, chunk_pairs)) + [P]

        def run(k):
            p0, p1 = bounds[k], bounds[k + 1]
            lo, hi = int(offsets[p0]), int(offsets[p1])
            return call(self.engines[k % depth], pts_a[lo:hi], pts_b[lo:hi], offsets[p0:p1 + 1] - lo, Ks[p0:p1],
                        pair_id0 + p0)

        def worker(e):
            return [(k, run(k)) for k in range(e, len(bounds) - 1, depth)]

        parts = dict(kv for res in self.pool.map(worker, range(depth)) for kv in res)
        return _merge_chunks([parts[k] for k in range(len(bounds) - 1)])

    def batch_two_view(self, pts_a, pts_b, offsets, Ks, h, seed, threshold, min_extra=0.0, aggregation="rms",
                       selection="min_error", distance_threshold=50.0, pair_id0=0, chunk_pairs: Optional[int] = None,
                       refine_iterations=0):
        """``Engine.batch_two_view`` (RANSAC E + inlier list + pose vote + triangulation per pair) over chunks of
        pairs that alternate between the contexts; identical to one call over all pairs (refinement included: a pair's
        refined model depends on its inliers only)."""
        return self._chunked(lambda e, a, b, o, K, p0: e.batch_two_view(a, b, o, K, h, seed, threshold, min_extra,
                                                                         aggregation, selection, distance_threshold,
                                                                         pair_id0=p0, refine_iterations=refine_iterations),
                             pts_a, pts_b, offsets, Ks, pair_id0, chunk_pairs)

    def batch_two_view_homography(self, pts_a, pts_b, offsets, Ks, h, seed, threshold, min_extra=0.0, aggregation="rms",
                                  selection="min_error", distance_threshold=50.0, rotation_tolerance=1e-2, pair_id0=0,
                                  chunk_pairs: Optional[int] = None, refine_iterations=0):
        """``Engine.batch_two_view_homography`` over chunks of pairs; identical to one call over all pairs."""
        return self._chunked(lambda e, a, b, o, K, p0: e.batch_two_view_homography(
            a, b, o, K, h, seed, threshold, min_extra, aggregation, selection, distance_threshold, rotation_tolerance,
            pair_id0=p0, refine_iterations=refine_iterations), pts_a, pts_b, offsets, Ks, pair_id0, chunk_pairs)

    def batch_two_view_select(self, pts_a, pts_b, offsets, Ks, essential_threshold, homography_threshold, h, seed,
                              pair_id0=0, chunk_pairs: Optional[int] = None, **kw):
        """``model_selection.batch_two_view_select_arrays`` (keyword arguments passed on) over chunks of pairs;
        identical to one call over all pairs."""
        from .model_selection import batch_two_view_select_arrays

        return self._chunked(lambda e, a, b, o, K, p0: batch_two_view_select_arrays(
            a, b, o, K, essential_threshold, homography_threshold, h, seed, pair_id0=p0, engine=e, **kw),
            pts_a, pts_b, offsets, Ks, pair_id0, chunk_pairs)

    def close(self):
        self.pool.shutdown()
        for e in self.engines:
            e.close()
