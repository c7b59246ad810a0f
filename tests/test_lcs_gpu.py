"""GPU parity tests for HP-1 (all go through the C ABI).  Bit-exact: LCS lengths are integers."""
import os
import zlib

import numpy as np
import pytest

from conftest import GOLDEN, QUIRK_LCS, QUIRK_SEQS, random_set
from famsa_b200 import seqio
from famsa_b200.binding import Engine
from oracle import pyoracle

import refgold

pytestmark = pytest.mark.gpu


def tri_to_square(tri, n, base_row=0):
    sq = np.zeros((n, n), dtype=np.int64)
    i, j = np.tril_indices(n, -1)
    keep = i >= base_row
    i, j = i[keep], j[keep]
    sq[i, j] = tri[i * (i - 1) // 2 + j - base_row * (base_row - 1) // 2 * (base_row > 0)]
    return sq


def test_adeno_triangle_matches_golden(engine, adeno):
    """Unsorted input order (the -dist_export shape): every LCS pinned by pid.csv."""
    n = len(adeno["lens"])
    engine.upload(adeno["codes"], adeno["offsets"], adeno["lens"])
    for dtype in (np.uint16, np.uint32):
        tri = engine.triangle(dtype=dtype)
        i, j = np.tril_indices(n, -1)
        assert np.array_equal(tri[i * (i - 1) // 2 + j], adeno["lcs"][i, j])
    part = engine.triangle(57, 131)
    assert np.array_equal(part, tri[57 * 56 // 2:131 * 130 // 2])


def test_adeno_rows_match_golden_square(engine, adeno):
    """All 242 x 242 entries of pid_sq.csv incl. the diagonal, row = seq0."""
    n = len(adeno["lens"])
    engine.upload(adeno["codes"], adeno["offsets"], adeno["lens"])
    got = engine.rows(np.arange(n))
    assert np.array_equal(got, adeno["lcs"])
    cols = np.array([5, 5, 200, 0, 17, 241, 3], dtype=np.uint32)      # duplicates allowed
    got = engine.rows([7, 100, 7], cols, dtype=np.uint16)
    assert np.array_equal(got, adeno["lcs"][np.ix_([7, 100, 7], cols)])
    got = engine.rows([9], n_col=50)
    assert np.array_equal(got[0], adeno["lcs"][9, :50])


def test_carry_quirk_vector(engine):
    """The reference's dropped-carry corner (SURVEY.md section 7) is reproduced bit for bit."""
    codes, offsets, lens = seqio.pack([seqio.encode(s) for s in QUIRK_SEQS])
    engine.upload(codes, offsets, lens)
    assert np.array_equal(engine.rows(np.arange(4)), QUIRK_LCS)
    tri = engine.triangle(dtype=np.uint32)
    i, j = np.tril_indices(4, -1)
    assert np.array_equal(tri, QUIRK_LCS[i, j])


@pytest.mark.parametrize("seed,n,lo,hi", [(1, 150, 0, 90), (2, 97, 30, 700), (3, 40, 1000, 2300), (4, 33, 1, 1)])
def test_random_ragged_sets(engine, seed, n, lo, hi):
    """Ragged lengths incl. empty sequences, non-matching symbols (B Z X *), low-complexity runs,
    sequences beyond the register-resident kernel's 2048 residues."""
    rng = np.random.default_rng(seed)
    code_list = random_set(rng, n, lo, hi)
    code_list += random_set(rng, 6, max(lo, 1), max(hi // 2, 1), alphabet=2)
    code_list.append(np.zeros(min(hi, 200) + 1, np.int8))
    rng.shuffle(code_list)
    codes, offsets, lens = seqio.pack(code_list)
    m = len(code_list)
    engine.upload(codes, offsets, lens)
    assert np.array_equal(engine.triangle(dtype=np.uint32), pyoracle.lcs_triangle(codes, offsets, lens))
    refs = rng.permutation(m)[:9]
    cols = rng.permutation(m)[:31]
    assert np.array_equal(engine.rows(refs, cols), pyoracle.lcs_rows(codes, offsets, lens, refs, cols))
    assert np.array_equal(engine.rows(refs[:2]), pyoracle.lcs_rows(codes, offsets, lens, refs[:2]))


def test_sorted_set_partial_rows(engine):
    """Length-descending input (FAMSA's own order): identity permutation, row-range sharding."""
    codes, offsets, lens = seqio.synth_family(300, 120, seed=9)
    engine.upload(codes, offsets, lens)
    full = pyoracle.lcs_triangle(codes, offsets, lens)
    got = np.concatenate([engine.triangle(a, b, dtype=np.uint32) for a, b in [(0, 64), (64, 65), (65, 201), (201, 300)]])
    assert np.array_equal(got, full)


def test_edge_cases(engine):
    codes, offsets, lens = seqio.pack([seqio.encode("ACDEFGHIK")])
    engine.upload(codes, offsets, lens)
    assert engine.triangle().size == 0
    assert np.array_equal(engine.rows([0]), [[9]])
    codes, offsets, lens = seqio.pack([seqio.encode("ACD"), seqio.encode(""), seqio.encode("XXBZ*"), seqio.encode("DCA")])
    engine.upload(codes, offsets, lens)
    assert np.array_equal(engine.rows(np.arange(4)), pyoracle.lcs_rows(codes, offsets, lens, np.arange(4)))
    with pytest.raises(Exception):
        engine.rows([4])
    with pytest.raises(Exception):
        engine.triangle(0, 5)


@pytest.mark.parametrize("sort", [True, False])
def test_over_long_and_quirky_sequences(engine, sort):
    """5 % of the set longer than the register-resident kernel handles as the mask side (> 2048 aa, up to 4500 aa, one of
    7000 aa beyond the batched exact kernel), a few with a dropped-carry word: over-long x shorter pairs come from the tile
    kernel (shorter sequence as the mask side), over-long x over-long and dropped-carry rows from the exact kernels --
    triangle and row calls against the oracle."""
    rng = np.random.default_rng(91)
    cl = random_set(rng, 170, 40, 400, alphabet=6)
    cl += random_set(rng, 8, 2100, 4500, alphabet=6)
    cl += random_set(rng, 1, 7000, 7000, alphabet=6)
    q = np.full(300, 3, dtype=np.int8); q[70:90] = rng.integers(0, 6, 20)          # positions 128..191 all the same residue
    cl += [q, np.concatenate([np.full(64, 2, dtype=np.int8), rng.integers(0, 6, 2300).astype(np.int8)])]
    order = rng.permutation(len(cl))
    cl = [cl[i] for i in order]
    if sort:
        cl.sort(key=lambda c: -len(c))
    codes, offsets, lens = seqio.pack(cl)
    engine.upload(codes, offsets, lens)
    assert np.array_equal(engine.triangle(dtype=np.uint32), pyoracle.lcs_triangle(codes, offsets, lens))
    refs = [0, 3, 57, len(cl) - 1] + [int(i) for i in np.argsort(-lens.astype(np.int64))[:4]]
    assert np.array_equal(engine.rows(refs), pyoracle.lcs_rows(codes, offsets, lens, refs))


def test_full_size_properties(engine):
    """BASELINE config 2 shape (10k x 400 aa): size-independent properties + oracle spot checks."""
    codes, offsets, lens = seqio.synth_family(10000, 400, seed=1)
    n = len(lens)
    engine.upload(codes, offsets, lens)
    tri = engine.triangle(dtype=np.uint16)
    assert tri.size == n * (n - 1) // 2
    rng = np.random.default_rng(0)
    # (1) bounded by the shorter sequence, and > 0 for related sequences
    i, j = np.tril_indices(n, -1)
    sel = rng.integers(0, tri.size, size=200000)
    assert np.all(tri[sel] <= np.minimum(lens[i[sel]], lens[j[sel]]))
    # (2) symmetry of the true LCS: row mode (roles swapped) agrees with the triangle
    refs = rng.integers(0, n, size=8)
    rows = engine.rows(refs, dtype=np.uint16)
    for r, ref in enumerate(refs):
        below = tri[ref * (ref - 1) // 2: ref * (ref - 1) // 2 + ref]
        assert np.array_equal(rows[r, :ref], below)
        assert rows[r, ref] == lens[ref]
        above = np.arange(ref + 1, n)
        assert np.array_equal(rows[r, ref + 1:], tri[above * (above - 1) // 2 + ref])
    # (3) oracle on random rows
    for ref in rng.integers(1, n, size=3):
        cols = rng.integers(0, ref, size=300)
        want = pyoracle.lcs_rows(codes, offsets, lens, [ref], cols)[0]
        assert np.array_equal(tri[ref * (ref - 1) // 2 + cols], want)
    # (4) checksum of checksums is reproducible across a second run
    assert int(tri.astype(np.uint64).sum()) == int(engine.triangle(dtype=np.uint16).astype(np.uint64).sum())


def test_full_c2_triangle_equals_reference(engine):
    """BASELINE config 2 in full: all 49 995 000 LCS lengths of the 10k x 400 aa set against the unmodified reference
    (CLCSBP AVX2 through calculateDistanceVector, oracle/_ref; without it, the CRC32 of the reference's triangle)
    -- every pair, not a sample."""
    codes, offsets, lens = seqio.synth_family(10000, 400, seed=1)
    n = len(lens)

    def reference():
        letters = [seqio.decode(codes[int(o):int(o) + int(l)]) for o, l in zip(offsets, lens)]
        rs = pyoracle.RefSeqSet(letters)
        _, pairs, want = rs.triangle_mt(0, n, max(1, len(os.sched_getaffinity(0))), 2, want_lcs=True)
        rs.close()
        assert pairs == n * (n - 1) // 2
        return want.astype(np.uint16)
    want_crc = refgold.answer_crc("c2_triangle", reference)
    engine.upload(codes, offsets, lens)
    got = engine.triangle(dtype=np.uint16)
    assert got.size == n * (n - 1) // 2
    assert refgold.crc(got) == want_crc, "the C2 triangle differs from the reference's"


def _assign_reference(codes, offsets, lens, seeds, kind, lcs_rows):
    """FastTree<>::makeEvaluation (src/tree/FastTree.cpp:309-324) restated with the oracle's float Transform."""
    n = len(lens)
    best = np.zeros(n, dtype=np.float32)
    assign = np.zeros(n, dtype=np.uint32)
    for k, s in enumerate(seeds):
        row = np.array([pyoracle.transform(kind, int(lcs_rows[k, j]), int(lens[s]), int(lens[j]), double=False)
                        for j in range(n)], dtype=np.float32)
        if k == 0:
            best[:] = row
        else:
            better = row < best
            best[better] = row[better]
            assign[better] = k
    return assign, best


@pytest.mark.parametrize("kind", [0, 1, 2])
def test_medoid_assignment(engine, adeno, kind):
    """famsa_lcs_assign == seed rows -> float Transform -> strict-< running arg-min, bit for bit."""
    rng = np.random.default_rng(kind)
    codes, offsets, lens = adeno["codes"], adeno["offsets"], adeno["lens"]
    engine.upload(codes, offsets, lens)
    seeds = rng.permutation(len(lens))[:17]
    want_a, want_d = _assign_reference(codes, offsets, lens, seeds, kind, adeno["lcs"][seeds])
    got_a, got_d = engine.assign(seeds, kind)
    assert np.array_equal(got_a, want_a)
    assert np.array_equal(got_d.view(np.uint32), want_d.view(np.uint32))          # same float bits
    s = int(seeds[3])

    def reference():
        rs = pyoracle.RefSeqSet(adeno["seqs"])
        lib = pyoracle.ref()
        row = rs.row_prefix(s, len(lens), 2)
        return np.array([lib.ref_transform_f32(kind, int(row[j]), int(lens[s]), int(lens[j])) for j in range(len(lens))], dtype=np.float32)
    d = refgold.answer(f"adeno/assign_row/{kind}/{s}", reference)
    assert np.all(got_d <= d)
    assert np.array_equal(got_d[got_a == 3], d[got_a == 3])


def test_medoid_assignment_large(engine):
    """Config-5 shape at reduced N: two-level family, 100 seeds, duplicates of a seed's sequence tie to the first."""
    codes, offsets, lens = seqio.synth_family(20000, 250, seed=3, n_subroots=30)
    engine.upload(codes, offsets, lens)
    rng = np.random.default_rng(5)
    seeds = np.sort(rng.choice(len(lens), size=100, replace=False))
    a, d = engine.assign(seeds, 0)
    rows = engine.rows(seeds[:3], dtype=np.uint32)
    for j in rng.integers(0, len(lens), size=200):
        ds = [pyoracle.transform(0, int(pyoracle.lcs_rows(codes, offsets, lens, [int(s)], [int(j)])[0, 0]), int(lens[s]), int(lens[j]), False)
              for s in seeds]
        ds = np.array(ds, dtype=np.float32)
        assert a[j] == int(np.argmin(ds)) and d[j] == ds.min()
    assert np.all(a[seeds] == np.arange(100)) or np.all(d[seeds] == 0)
    cost = np.float32(0)
    for x in d[:1000]:
        cost = np.float32(cost + x)                     # the caller keeps std::accumulate's order
    assert np.isfinite(cost)


def test_medoid_assignment_sharded(engine):
    """famsa_lcs_assign_shard: three shards of one context, combined with an element-wise MIN (what the NCCL all-reduce
    does across GPUs), equal the unsharded famsa_lcs_assign bit for bit -- ragged lengths, unsorted input, a repeated seed."""
    import torch
    from famsa_b200.binding import unpack_assignment
    codes, offsets, lens = seqio.pack(random_set(np.random.default_rng(77), 1000, 30, 300))
    engine.upload(codes, offsets, lens)
    seeds = np.array([5, 900, 17, 5, 333, 64], dtype=np.uint32)
    for kind in (0, 2):
        want_a, want_d = engine.assign(seeds, kind)
        parts = []
        for sh in range(3):
            t = torch.empty(len(lens), dtype=torch.int64, device="cuda")
            engine.assign_shard(seeds, sh, 3, t.data_ptr(), kind)
            parts.append(t.cpu().numpy())
        owned = np.stack([p != np.iinfo(np.int64).max for p in parts])
        assert np.all(owned.sum(axis=0) == 1), "the shards must partition the sequences"
        a, d = unpack_assignment(np.minimum.reduce(parts))
        assert np.array_equal(a, want_a) and np.array_equal(d, want_d)


@pytest.mark.parametrize("modified", [False, True])
def test_gpu_driven_upgma_tree(engine, modified):
    """Drop-in proof for HP-1: GPU LCS triangle -> host Transform<float, indel075_div_lcs> -> the reference's own,
    unmodified UPGMA agglomeration (UPGMA<>::computeTree) gives exactly the guide tree the reference builds from
    its CPU LCS (and, on adeno_fiber, every distance of the golden dist_sq.csv)."""
    codes, offsets, lens = seqio.synth_family(400, 150, seed=21)
    n = len(lens)
    engine.upload(codes, offsets, lens)
    lcs = engine.triangle(dtype=np.uint32)
    i, j = np.tril_indices(n, -1)
    tri = np.zeros(lcs.size, dtype=np.float32)
    tri[i * (i - 1) // 2 + j] = [engine.transform(0, int(l), int(lens[a]), int(lens[b]), double=False)
                                 for l, a, b in zip(lcs[i * (i - 1) // 2 + j], i, j)]
    letters = [seqio.decode(codes[int(o):int(o) + int(ln)]) for o, ln in zip(offsets, lens)]
    if refgold.live():
        want = pyoracle.RefSeqSet(letters).upgma_tree(modified)
        got = pyoracle.upgma_tree_from_distances(tri, n, modified)
        assert np.array_equal(got, want)

    def reference_distances():                   # the reference's own LCS + Transform<float>: its UPGMA's input
        _, _, ref_lcs = pyoracle.RefSeqSet(letters).triangle_mt(0, n, 4, 2, want_lcs=True)
        f = pyoracle.ref().ref_transform_f32
        return np.array([f(0, int(ref_lcs[i * (i - 1) // 2 + j]), int(lens[i]), int(lens[j])) for i, j in zip(*np.tril_indices(n, -1))],
                        dtype=np.float32)
    assert refgold.crc(tri) == refgold.answer_crc("upgma_driven/distances/" + refgold.input_key(letters), reference_distances)


@pytest.mark.parametrize("modified", [False, True])
@pytest.mark.parametrize("case", ["family400", "ragged", "big"])
def test_device_upgma_tree(engine, modified, case):
    """famsa_lcs_upgma (distances + agglomeration on the device, SURVEY 8f-1): the tree is the reference's UPGMA<>::run
    tree pair for pair, plain and MAFFT-modified average, on a family, on a ragged random set full of distance ties and on
    3000 sequences (several thread blocks per scan)."""
    if case == "family400":
        codes, offsets, lens = seqio.synth_family(400, 150, seed=21)
    elif case == "ragged":
        cl = random_set(np.random.default_rng(5), 500, 20, 90, alphabet=4)
        cl.sort(key=lambda c: -len(c))
        codes, offsets, lens = seqio.pack(cl)
    else:
        codes, offsets, lens = seqio.synth_family(3000, 120, seed=23)
    n = len(lens)
    engine.upload(codes, offsets, lens)
    got = engine.upgma(0, modified)
    letters = [seqio.decode(codes[int(o):int(o) + int(ln)]) for o, ln in zip(offsets, lens)]
    want = refgold.answer(f"upgma_tree/{case}/{int(modified)}/" + refgold.input_key(letters),
                          lambda: pyoracle.RefSeqSet(letters).upgma_tree(modified, n_threads=8)[n:])
    assert got.shape == want.shape and np.array_equal(got, want)


def test_device_upgma_golden(engine):
    """The golden UPGMA tree of adeno_fiber (test/adeno_fiber/upgma.dnd, held as merges in the fixture): same clades."""
    z = np.load(os.path.join(GOLDEN, "adeno_upgma_merges.npz"))
    seqs = [str(s) for s in z["seqs"]]
    codes, offsets, lens = seqio.pack([seqio.encode(s) for s in seqs])
    n = len(seqs)
    engine.upload(codes, offsets, lens)

    def clades(merges):
        members = {i: frozenset([i]) for i in range(n)}
        out = set()
        for k, (a, b) in enumerate(merges):
            members[n + k] = members[int(a)] | members[int(b)]
            out.add(members[n + k])
        return out
    # the fixture's leaves are in the tree file's order, UPGMA needs FAMSA's own (length-descending) order: re-order
    order = sorted(range(n), key=lambda i: (-len(seqs[i]), seqio.encode(seqs[i]).tobytes()))
    codes, offsets, lens = seqio.pack([seqio.encode(seqs[i]) for i in order])
    engine.upload(codes, offsets, lens)
    got = engine.upgma(0, False)
    remap = lambda m: [(order[a] if a < n else a, order[b] if b < n else b) for a, b in m]
    assert clades(remap([(int(a), int(b)) for a, b in got])) == clades([(int(a), int(b)) for a, b in z["merges"]])


def test_gpu_distances_match_golden_dist_sq(engine, adeno):
    """test/adeno_fiber/dist_sq.csv: GPU LCS + host float Transform reproduce every printed distance."""
    n = len(adeno["lens"])
    engine.upload(adeno["codes"], adeno["offsets"], adeno["lens"])
    rows = engine.rows(np.arange(n))
    lens = adeno["lens"]
    for a in range(0, n, 3):
        for b in range(n):
            if a != b:
                d = engine.transform(0, int(rows[a, b]), int(lens[a]), int(lens[b]), double=False)
                assert abs(d - adeno["dist"][a, b]) < 1e-6 * max(1.0, abs(d)) + 6e-7


def test_blockwise_triangle_copy(engine, monkeypatch):
    """famsa_lcs_triangle's block-wise path (eight equal-pair row blocks, each copied back as soon as it is done;
    normally used above 4e8 pairs) forced on a small set."""
    codes, offsets, lens = seqio.synth_family(700, 90, seed=33)
    engine.upload(codes, offsets, lens)
    monkeypatch.setenv("FAMSA_LCS_BLOCK_MIN_PAIRS", "1000")
    want = pyoracle.lcs_triangle(codes, offsets, lens)
    assert np.array_equal(engine.triangle(dtype=np.uint16), want)
    assert np.array_equal(engine.triangle(dtype=np.uint32), want)


def test_concurrent_callers_share_one_context(engine, adeno):
    """The reference gives every worker thread its own CLCSBP; here all workers may share one context (calls are
    serialised inside the library).  Eight threads hammer rows() concurrently -- ctypes drops the GIL."""
    import threading
    n = len(adeno["lens"])
    engine.upload(adeno["codes"], adeno["offsets"], adeno["lens"])
    errors = []

    def work(tid):
        rng = np.random.default_rng(tid)
        for _ in range(6):
            refs = rng.permutation(n)[:3]
            cols = rng.permutation(n)[:40]
            got = engine.rows(refs, cols)
            if not np.array_equal(got, adeno["lcs"][np.ix_(refs, cols)]):
                errors.append(tid)

    threads = [threading.Thread(target=work, args=(t,)) for t in range(8)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors


from treeutil import prim_restated as _prim_restated  # noqa: E402


@pytest.mark.parametrize("case", ["family", "adeno", "quirky", "tiny"])
def test_gpu_prim_tree(engine, adeno, case):
    """Drop-in proof for the DEFAULT guide tree (-gt sl): famsa_lcs_prim's MST edges, passed to the reference's own
    unmodified mst_to_dendogram, give exactly the tree MSTPrim<indel075_div_lcs> builds on the CPU.  Without oracle/_ref the
    edges must be the ones that were checked to give that tree when the stored answers were recorded."""
    if case == "family":
        codes, offsets, lens = seqio.synth_family(700, 130, seed=41)
    elif case == "adeno":
        order = sorted(range(len(adeno["lens"])), key=lambda i: (-int(adeno["lens"][i]), adeno["code_list"][i].tobytes()))
        codes, offsets, lens = seqio.pack([adeno["code_list"][i] for i in order])      # FAMSA's own order (msa.cpp:245-256)
    elif case == "quirky":
        rng = np.random.default_rng(8)
        cl = random_set(rng, 60, 60, 260, alphabet=3)
        cl += [np.zeros(200, np.int8), np.zeros(130, np.int8), np.concatenate([np.ones(64, np.int8), np.zeros(70, np.int8)])]
        cl.sort(key=lambda c: (-len(c), c.tobytes()))
        codes, offsets, lens = seqio.pack(cl)
    else:
        codes, offsets, lens = seqio.pack([seqio.encode(s) for s in ["ACDEFGHIKL", "ACDEFGHIK", "ACDFGHIK"]])
    n = len(lens)
    engine.upload(codes, offsets, lens)
    ef, et, ed, order = engine.prim(0)
    letters = [seqio.decode(codes[int(o):int(o) + int(ln)]) for o, ln in zip(offsets, lens)]
    if refgold.live():
        want = pyoracle.RefSeqSet(letters).mst_prim_tree(3)
        got = pyoracle.mst_to_dendogram(ef, et, ed, order)
        assert np.array_equal(got, want)
    assert refgold.crc(_edges(ef, et, ed, order)) == refgold.answer_crc(f"prim_tree/{case}/" + refgold.input_key(letters),
                                                                        lambda: _edges(ef, et, ed, order))
    assert sorted(order.tolist()) == list(range(n))


def _edges(ef, et, ed, order):
    return np.concatenate([np.asarray(x, dtype=np.float64) for x in (ef, et, ed, order)])


@pytest.mark.parametrize("sequential", [False, True])
def test_gpu_prim_edges_match_restatement(engine, monkeypatch, sequential):
    """Both device implementations -- Boruvka rounds + host replay of the visiting order (default when no sequence has
    orientation-dependent LCS values) and the sequential vertex loop -- against the restated Prim, edge for edge."""
    if sequential:
        monkeypatch.setenv("FAMSA_PRIM_SEQUENTIAL", "1")
    codes, offsets, lens = seqio.synth_family(90, 70, seed=43)
    engine.upload(codes, offsets, lens)
    for kind in (0, 1):
        got = engine.prim(kind)
        want = _prim_restated(codes, offsets, lens, kind)
        for g, w in zip(got, want):
            assert np.array_equal(g, w)


@pytest.mark.parametrize("sequential", [False, True])
def test_gpu_prim_golden_sl_tree(engine, monkeypatch, sequential):
    """The reference's default guide tree golden (test/adeno_fiber/sl.dnd) without oracle/_ref: the fixture's MST edges
    were checked at generation to rebuild, through the reference's mst_to_dendogram, the reference's tree and the
    clades of sl.dnd; famsa_lcs_prim (both device implementations) must return exactly those edges."""
    if sequential:
        monkeypatch.setenv("FAMSA_PRIM_SEQUENTIAL", "1")
    z = np.load(os.path.join(GOLDEN, "adeno_sl_tree.npz"))
    codes, offsets, lens = seqio.pack([seqio.encode(str(s)) for s in z["seqs"]])
    engine.upload(codes, offsets, lens)
    ef, et, ed, order = engine.prim(0)
    assert np.array_equal(ef, z["edge_from"]) and np.array_equal(et, z["edge_to"])
    assert np.array_equal(ed, z["edge_dist"]) and np.array_equal(order, z["prim_order"])


def test_gpu_prim_lrr_golden_tree():
    """The reference's large default-guide-tree golden, test/LRR/sl.dnd (124 140 sequences; fixture lrr_sl.npz: the set in
    FAMSA's order and the CRC of the reference's MSTPrim tree, whose clades were checked against sl.dnd at generation).
    famsa_lcs_prim keeps the 7.7 G-pair triangle in HBM (15 GB as u16 + 62 GB of float64 distances for the Boruvka
    rounds); its edges, through the reference's own mst_to_dendogram, must give that tree (without oracle/_ref: must be
    the edges that were checked to give it when the stored answers were recorded)."""
    path = os.path.join(GOLDEN, "lrr_sl.npz")
    if not os.path.exists(path):
        pytest.skip("lrr_sl.npz not generated")
    z = np.load(path)
    seqs = bytes(z["seqs"]).decode().split("\n")
    n = int(z["n"][0])
    assert len(seqs) == n
    codes, offsets, lens = seqio.pack([seqio.encode(s) for s in seqs])
    eng = Engine()                                       # own context: tens of GB of scratch go away with it
    try:
        eng.upload(codes, offsets, lens)
        ef, et, ed, order = eng.prim(0)
    finally:
        eng.close()
    if refgold.live():
        tree = pyoracle.mst_to_dendogram(ef, et, ed, order)
        assert zlib.crc32(np.ascontiguousarray(tree[n:], dtype=np.int32).tobytes()) == int(z["tree_crc"][0])
    assert refgold.crc(_edges(ef, et, ed, order)) == refgold.answer_crc("prim_tree/lrr", lambda: _edges(ef, et, ed, order))


def test_gpu_prim_lower_bound_pruning_case(engine):
    """MSTPrim skips a candidate whose best possible distance -- LCS = the shorter length -- cannot beat its current one
    (MSTPrim.cpp:450-467).  With the dropped-carry corner the reference's LCS can exceed the shorter length, so the skip
    changes the tree; fixture prim_pruning_case.npz holds a 13-sequence set where it does (generation asserts the
    reference's tree equals the restated loop WITH the skip and differs from the one without) and the edges of that loop."""
    z = np.load(os.path.join(GOLDEN, "prim_pruning_case.npz"))
    codes, offsets, lens = seqio.pack([seqio.encode(str(s)) for s in z["seqs"]])
    engine.upload(codes, offsets, lens)
    ef, et, ed, order = engine.prim(0)
    assert np.array_equal(ef, z["edge_from"]) and np.array_equal(et, z["edge_to"])
    assert np.array_equal(ed, z["edge_dist"]) and np.array_equal(order, z["prim_order"])
