"""CPU tests of famsa_b200/mst.py: the MST under MSTPrim's (distance, key) total order is unique, so Kruskal + the
Prim-order replay must reproduce the sequential Prim loop edge for edge -- and, through the reference's own
mst_to_dendogram, the reference's default guide tree."""
import numpy as np
import pytest

from famsa_b200 import mst, seqio
from oracle import pyoracle


def _distances(codes, offsets, lens, kind=0):
    n = len(lens)
    tri = pyoracle.lcs_triangle(codes, offsets, lens)
    out = np.zeros(len(tri), dtype=np.float64)
    at = 0
    for i in range(1, n):
        for j in range(i):
            out[at] = pyoracle.transform(kind, int(tri[at]), int(lens[i]), int(lens[j]), True)
            at += 1
    return out


def _prim_sequential(n, tri):
    """MSTPrim<>::run_view's relax / elect loop (MSTPrim.cpp:366-386, 492-503) on a symmetric distance triangle."""
    dist = [np.finfo(np.float64).max] * n
    key = [0] * n
    visited = [False] * n
    order = np.full(n, n, dtype=np.int32)
    v = 0
    visited[0] = True
    order[0] = 0
    ef, et, ed = [], [], []
    for step in range(1, n):
        best = -1
        for j in range(n):
            if visited[j]:
                continue
            hi, lo = (v, j) if v > j else (j, v)
            d = float(tri[hi * (hi - 1) // 2 + lo])
            if d <= dist[j]:
                k = mst.edge_key(v, j)
                if d < dist[j] or k < key[j]:
                    dist[j], key[j] = d, k
            if best < 0 or dist[j] < dist[best] or (dist[j] == dist[best] and key[j] < key[best]):
                best = j
        p = 0xFFFFFFFFFFFFFFFF ^ key[best]
        ef.append(p >> 32); et.append(p & 0xFFFFFFFF); ed.append(dist[best])
        order[best] = step
        visited[best] = True
        v = best
    return np.array(ef, np.int32), np.array(et, np.int32), np.array(ed), order


@pytest.mark.parametrize("n,length,seed,kind", [(120, 60, 3, 0), (90, 35, 4, 1), (40, 12, 5, 0)])
def test_kruskal_plus_replay_equals_sequential_prim(n, length, seed, kind):
    """Short sequences give many tied distances: the key component of the order decides, identically in both."""
    codes, offsets, lens = seqio.synth_family(n, length, seed)
    tri = _distances(codes, offsets, lens, kind)
    assert len(np.unique(tri)) < len(tri)                       # ties are present
    got = mst.prim_replay(n, mst.kruskal_total_order(n, tri))
    want = _prim_sequential(n, tri)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)


def test_replayed_mst_gives_the_reference_tree():
    """Through the reference's mst_to_dendogram where oracle/_ref is built; elsewhere the edges must be the ones that
    were checked to give the reference's tree when the stored answers were recorded."""
    import refgold
    codes, offsets, lens = seqio.synth_family(150, 80, seed=6)
    n = len(lens)
    tri = _distances(codes, offsets, lens, 0)
    ef, et, ed, order = mst.prim_replay(n, mst.kruskal_total_order(n, tri))
    letters = [seqio.decode(codes[int(o):int(o) + int(ln)]) for o, ln in zip(offsets, lens)]
    if refgold.live():
        want = pyoracle.RefSeqSet(letters).mst_prim_tree(2)
        assert np.array_equal(pyoracle.mst_to_dendogram(ef, et, ed, order), want)
    edges = np.concatenate([np.asarray(ef, np.float64), np.asarray(et, np.float64), np.asarray(ed, np.float64), np.asarray(order, np.float64)])
    assert refgold.crc(edges) == refgold.answer_crc("mst_host/edges/" + refgold.input_key(letters), lambda: edges)


def test_golden_sl_tree_edges_without_reference():
    """tests/golden/adeno_sl_tree.npz was generated with the assertion that these edges, through the reference's
    mst_to_dendogram, give the reference's MSTPrim tree and exactly the clades of the golden test/adeno_fiber/sl.dnd.
    Here (no oracle/_ref needed) the oracle's distances + Kruskal under MSTPrim's edge order + the visiting-order
    replay must reproduce them."""
    import os
    from conftest import GOLDEN
    z = np.load(os.path.join(GOLDEN, "adeno_sl_tree.npz"))
    codes, offsets, lens = seqio.pack([seqio.encode(str(s)) for s in z["seqs"]])
    n = len(lens)
    tri = _distances(codes, offsets, lens, 0)
    ef, et, ed, po = mst.prim_replay(n, mst.kruskal_total_order(n, tri))
    assert np.array_equal(ef, z["edge_from"]) and np.array_equal(et, z["edge_to"])
    assert np.array_equal(ed, z["edge_dist"]) and np.array_equal(po, z["prim_order"])
