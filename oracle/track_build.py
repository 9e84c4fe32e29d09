"""TEST INFRASTRUCTURE ONLY — restatement of the track building from pairwise matches (csrc/sfm_track_build.cuh) with a
different algorithm: scipy's ``connected_components`` on the sparse match graph, then each component labelled by its
smallest global id, the features of components of >= 2 sorted by (label, id), and the status of every run.

``build_tracks(feature_offsets, pair_views, match_offsets, matches)`` takes the C ABI's arrays and returns a dict with
``offsets`` int64[T+1], ``status`` int32[T] (0 ok, 1 conflict, 2 long), ``view`` int32[M], ``feature`` int32[M] and
``track`` int32[N], the outputs of sfm_build_tracks trimmed to T and M.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components

OK, CONFLICT, LONG = 0, 1, 2
MAX_OBSERVATIONS = 64


def global_edges(feature_offsets, pair_views, match_offsets, matches):
    """int64[E][2]: every match as the pair of global ids (off[a] + i, off[b] + j)."""
    off = np.asarray(feature_offsets, dtype=np.int64)
    pv = np.asarray(pair_views, dtype=np.int64).reshape(-1, 2)
    mo = np.asarray(match_offsets, dtype=np.int64).reshape(-1)
    m = np.asarray(matches, dtype=np.int64).reshape(-1, 2)
    pair = np.repeat(np.arange(len(pv)), np.diff(mo)) if len(pv) else np.zeros(0, dtype=np.int64)
    return np.column_stack([off[pv[pair, 0]] + m[:, 0], off[pv[pair, 1]] + m[:, 1]])


def build_tracks(feature_offsets, pair_views, match_offsets, matches):
    off = np.asarray(feature_offsets, dtype=np.int64)
    N = int(off[-1])
    e = global_edges(feature_offsets, pair_views, match_offsets, matches)
    g = sp.coo_matrix((np.ones(len(e), dtype=np.int8), (e[:, 0], e[:, 1])), shape=(N, N))
    _, comp = connected_components(g, directed=False)
    ids = np.arange(N)
    low = np.full(comp.max() + 1 if N else 0, N, dtype=np.int64)
    np.minimum.at(low, comp, ids)
    label = low[comp]
    size = np.bincount(label, minlength=N) if N else np.zeros(0, dtype=np.int64)
    sel = ids[size[label] >= 2]
    order = np.lexsort((sel, label[sel]))
    feature = sel[order]
    lab = label[feature]
    head = np.ones(len(feature), dtype=bool)
    head[1:] = lab[1:] != lab[:-1]
    starts = np.flatnonzero(head)
    T = len(starts)
    offsets = np.append(starts, len(feature)).astype(np.int64)
    view = (np.searchsorted(off, feature, side="right") - 1).astype(np.int32)
    tix = np.cumsum(head) - 1
    same = np.zeros(len(feature), dtype=bool)
    same[1:] = (~head[1:]) & (view[1:] == view[:-1])
    status = np.zeros(T, dtype=np.int32)
    status[np.diff(offsets) > MAX_OBSERVATIONS] = LONG
    status[np.unique(tix[same])] = CONFLICT
    track = np.full(N, -1, dtype=np.int32)
    track[feature] = tix
    return {"offsets": offsets, "status": status, "view": view, "feature": feature.astype(np.int32), "track": track}
