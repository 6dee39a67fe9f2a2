"""numpy / scipy restatement of pcl::EuclideanClusterExtraction (TEST INFRASTRUCTURE ONLY), written from the component
formulation rather than PCL's loop: the neighbour pairs (cKDTree at a slightly larger radius, then the exact float test
(dx*dx + dy*dy) + dz*dz < r2 with every operation rounded to float32), the connected components of that graph
(scipy.sparse.csgraph), each component's smallest index as its seed, the size filter, and the cluster order of
std::sort(clusters.rbegin(), clusters.rend(), size <) -- libstdc++'s introsort, restated below step by step."""
from __future__ import annotations

import numpy as np

F32 = np.float32
INT_MAX = 2 ** 31 - 1


def r2_of(tolerance: float) -> np.float32:
    """(float)((double)tf * tf), tf = (float)tolerance: extract() narrows, KdTreeFLANN::radiusSearch squares in double."""
    tf = float(F32(tolerance))
    return F32(tf * tf)


def pairs(x, tolerance: float) -> np.ndarray:
    """(i, j), i < j, of the finite points strictly inside the tolerance in FLANN's float order."""
    from scipy.spatial import cKDTree
    x = np.asarray(x, F32).reshape(-1, 4)
    fin = np.nonzero(np.isfinite(x[:, :3]).all(axis=1))[0]
    if len(fin) < 2:
        return np.zeros((0, 2), np.int64)
    r2 = r2_of(tolerance)
    p = cKDTree(x[fin, :3].astype(np.float64)).query_pairs(float(np.sqrt(np.float64(r2))) * (1 + 1e-5) + 1e-30,
                                                          output_type="ndarray")
    if not len(p):
        return np.zeros((0, 2), np.int64)
    p = fin[p]
    d = x[p[:, 0], :3] - x[p[:, 1], :3]
    acc = ((d[:, 0] * d[:, 0]).astype(F32) + (d[:, 1] * d[:, 1]).astype(F32)).astype(F32)
    acc = (acc + (d[:, 2] * d[:, 2]).astype(F32)).astype(F32)
    return np.sort(p[acc < r2], axis=1)


# ---- libstdc++ std::sort (bits/stl_algo.h, bits/stl_heap.h), comparator `less` -----------------------------------------------
_THRESHOLD = 16


def _unguarded_linear_insert(a, last, less):
    val = a[last]
    nxt = last - 1
    while less(val, a[nxt]):
        a[last] = a[nxt]
        last = nxt
        nxt -= 1
    a[last] = val


def _insertion_sort(a, first, last, less):
    if first == last:
        return
    for i in range(first + 1, last):
        if less(a[i], a[first]):
            val = a[i]
            a[first + 1:i + 1] = a[first:i]
            a[first] = val
        else:
            _unguarded_linear_insert(a, i, less)


def _final_insertion_sort(a, first, last, less):
    if last - first > _THRESHOLD:
        _insertion_sort(a, first, first + _THRESHOLD, less)
        for i in range(first + _THRESHOLD, last):
            _unguarded_linear_insert(a, i, less)
    else:
        _insertion_sort(a, first, last, less)


def _push_heap(a, first, hole, top, value, less):
    parent = (hole - 1) // 2
    while hole > top and less(a[first + parent], value):
        a[first + hole] = a[first + parent]
        hole = parent
        parent = (hole - 1) // 2
    a[first + hole] = value


def _adjust_heap(a, first, hole, length, value, less):
    top = hole
    second = hole
    while second < (length - 1) // 2:
        second = 2 * (second + 1)
        if less(a[first + second], a[first + second - 1]):
            second -= 1
        a[first + hole] = a[first + second]
        hole = second
    if (length & 1) == 0 and second == (length - 2) // 2:
        second = 2 * (second + 1)
        a[first + hole] = a[first + second - 1]
        hole = second - 1
    _push_heap(a, first, hole, top, value, less)


def _heap_sort(a, first, last, less):  # __partial_sort(first, last, last): make_heap, then sort_heap
    n = last - first
    if n >= 2:
        parent = (n - 2) // 2
        while True:
            _adjust_heap(a, first, parent, n, a[first + parent], less)
            if parent == 0:
                break
            parent -= 1
    while last - first > 1:
        last -= 1
        value = a[last]
        a[last] = a[first]
        _adjust_heap(a, first, 0, last - first, value, less)


def _move_median_to_first(a, result, i, j, k, less):
    if less(a[i], a[j]):
        if less(a[j], a[k]):
            m = j
        elif less(a[i], a[k]):
            m = k
        else:
            m = i
    elif less(a[i], a[k]):
        m = i
    elif less(a[j], a[k]):
        m = k
    else:
        m = j
    a[result], a[m] = a[m], a[result]


def _unguarded_partition(a, first, last, pivot, less):
    while True:
        while less(a[first], a[pivot]):
            first += 1
        last -= 1
        while less(a[pivot], a[last]):
            last -= 1
        if not first < last:
            return first
        a[first], a[last] = a[last], a[first]
        first += 1


def _introsort_loop(a, first, last, depth, less):
    while last - first > _THRESHOLD:
        if depth == 0:
            _heap_sort(a, first, last, less)
            return
        depth -= 1
        mid = first + (last - first) // 2
        _move_median_to_first(a, first, first + 1, mid, last - 1, less)
        cut = _unguarded_partition(a, first + 1, last, first, less)
        _introsort_loop(a, cut, last, depth, less)
        last = cut


def std_sort(a: list, less) -> None:
    """libstdc++'s std::sort(a.begin(), a.end(), less), in place."""
    n = len(a)
    if n > 1:
        _introsort_loop(a, 0, n, 2 * (n.bit_length() - 1), less)
        _final_insertion_sort(a, 0, n, less)


def pcl_cluster_order(sizes) -> np.ndarray:
    """std::sort(clusters.rbegin(), clusters.rend(), comparePointClusters): the input position of the cluster at every
    rank. Sorting through reverse iterators is sorting the reversed sequence."""
    recs = [(int(s), k) for k, s in enumerate(sizes)][::-1]
    std_sort(recs, lambda p, q: p[0] < q[0])
    return np.array([k for _, k in recs[::-1]], np.int64)


def clusters_of(x, tolerance: float, min_size: int = 1, max_size: int = INT_MAX) -> list:
    """the clusters of one cloud in PCL's order: a list of int64 index arrays, ascending inside a cluster."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    x = np.asarray(x, F32).reshape(-1, 4)
    n = len(x)
    if n == 0:
        return []
    p = pairs(x, tolerance)
    g = coo_matrix((np.ones(len(p), np.int8), (p[:, 0], p[:, 1])), shape=(n, n))
    _, lab = connected_components(g, directed=False)
    fin = np.isfinite(x[:, :3]).all(axis=1)
    order = np.argsort(lab, kind="stable")                    # every component's indices, ascending
    lab_s = lab[order]
    cuts = np.nonzero(np.diff(lab_s))[0] + 1
    comps = [c for c in np.split(order, cuts) if fin[c[0]]]  # a non-finite point is a component of its own
    comps.sort(key=lambda c: int(c[0]))                       # seed order
    kept = [c.astype(np.int64) for c in comps if min_size <= len(c) <= max_size]
    return [kept[k] for k in pcl_cluster_order([len(c) for c in kept])]


def clusters(clouds, tolerance: float, min_size: int = 1, max_size: int = INT_MAX) -> list:
    return [clusters_of(c, tolerance, min_size, max_size) for c in clouds]
