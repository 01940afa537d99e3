"""numpy reference of dist_b200_regroup_batch: the stable compaction of live groups plus n_empty fresh ones."""
import numpy as np


def remap(sizes, n_empty):
    """(remap[G] old -> new or -1, counts_out[K+ + n_empty], G_new) from the group sizes"""
    sizes = np.asarray(sizes, dtype=np.int64)
    live = sizes > 0
    rm = np.where(live, np.cumsum(live) - 1, -1).astype(np.int32)
    counts_out = np.concatenate([sizes[live], np.zeros(n_empty, np.int64)]).astype(np.int32)
    return rm, counts_out, int(live.sum()) + n_empty


def relabel(assign, rm):
    """negative ids stay; ids >= G become -1; others their group's new id"""
    a = np.asarray(assign, dtype=np.int32)
    G = rm.size
    out = a.copy()
    valid = a >= 0
    inside = valid & (a < G)
    out[inside] = rm[a[inside]]
    out[valid & (a >= G)] = -1
    return out


def compact(arr, sizes, n_empty):
    """[G][...] per-group array -> survivors in order, then n_empty zero groups"""
    arr = np.asarray(arr)
    live = np.asarray(sizes) > 0
    fresh = np.zeros((n_empty,) + arr.shape[1:], arr.dtype)
    return np.concatenate([arr[live], fresh])
