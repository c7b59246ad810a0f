"""CPU tests: oracle/dp_oracle.c against the reference's golden alignments and the reference itself."""
import os
import zlib

import numpy as np
import pytest

from conftest import GOLDEN
from dp_cases import check_against_reference, random_tree, reference_merges
from famsa_b200 import seqio
from oracle import pyoracle



def test_oracle_pp_golden():
    """test/adeno_fiber/upgma.pp.fasta: the reference's one pure profile-profile known answer."""
    z = np.load(os.path.join(GOLDEN, "adeno_pp.npz"))
    o = pyoracle.dp_align(z["s1"], z["c1"], int(z["k1"]), z["s2"], z["c2"], int(z["k2"]), z["gaps"])
    assert o["variant"] == 2 and o["swapped"] == bool(z["swapped"])
    assert o["total"] == int(z["total"])
    assert np.array_equal(o["path"], z["path"])
    d = o["dirs"]
    assert np.all(d[0, 1:] == 0x15) and np.all(d[1:, 0] == 0x2A) and d[0, 0] == 0


def test_oracle_all_merges_of_golden_upgma_tree():
    """All 241 merges (SeqSeq, SeqProf, ProfProf) behind test/adeno_fiber/upgma.no_refine.fasta."""
    z = np.load(os.path.join(GOLDEN, "adeno_upgma_merges.npz"))
    seqs = [str(s) for s in z["seqs"]]
    merges = [tuple(int(x) for x in m) for m in z["merges"]]
    g, recs = reference_merges(seqs, merges, threads=(1, 2))
    assert np.array_equal(g, z["gaps"])
    res = [pyoracle.dp_align(*r["job"], g) for r in recs]
    check_against_reference(res, recs)
    assert [r["total"] for r in res] == [int(t) for t in z["totals"]]
    assert np.array_equal(np.concatenate([r["path"] for r in res]), z["path"])
    assert sorted(set(r["variant"] for r in res)) == [0, 1, 2]


@pytest.mark.parametrize("seed,n,length,gaps", [(1, 60, 90, None), (2, 40, 300, None), (3, 50, 40, (-9000, -700, -300, -100)),
                                                (4, 30, 150, (-20000, -2000, -2500, -900))])
def test_oracle_random_families(seed, n, length, gaps):
    rng = np.random.default_rng(seed)
    codes, off, lens = seqio.synth_family(n, length, seed, sort_desc=False)
    seqs = [seqio.decode(codes[int(o):int(o) + int(l)]) for o, l in zip(off, lens)]
    seqs[0] = seqs[0][:5] + "XBZ" + seqs[0][8:]          # non-standard residues
    merges = random_tree(n, rng)
    g, recs = reference_merges(seqs, merges, threads=(1, 2), rng=rng, gaps=gaps)
    res = [pyoracle.dp_align(*r["job"], g) for r in recs]
    check_against_reference(res, recs)


def test_oracle_hemopexin_fixture_selfcheck():
    z = np.load(os.path.join(GOLDEN, "hemopexin_medoid_sl.npz"))
    assert len(z["seqs"]) == 4188 and len(z["merges"]) == 4187 and len(z["totals"]) == 4187


def test_oracle_hemopexin_first_levels():
    """Config 4 subset on CPU (the whole tree runs in the GPU test): first 400 merges of medoid-sl.dnd."""
    z = np.load(os.path.join(GOLDEN, "hemopexin_medoid_sl.npz"))
    seqs = [str(s) for s in z["seqs"]]
    merges = [tuple(int(x) for x in m) for m in z["merges"]]
    # keep a prefix that is closed under dependencies
    n = len(seqs)
    keep = []
    for k, (a, b) in enumerate(merges):
        if len(keep) >= 400:
            break
        if (a < n or (a - n) in keep) and (b < n or (b - n) in keep):
            keep.append(k)
    remap = {k: i for i, k in enumerate(keep)}
    sub = [tuple(x if x < n else n + remap[x - n] for x in merges[k]) for k in keep]
    g, recs = reference_merges(seqs, sub, n_seqs_for_rescale=n, threads=(1,), want_merged=True)
    assert np.array_equal(g, z["gaps"])
    res = []
    for k, r in zip(keep, recs):
        o = pyoracle.dp_align(*r["job"], g)
        assert o["total"] == int(z["totals"][k])
        assert zlib.crc32(o["path"].tobytes()) == int(z["path_crc"][k])
        res.append(o)
    _check_construct(res, recs, g)               # and the merged tables ConstructProfile builds from those paths


def test_oracle_driven_alignment_equals_reference():
    """The oracle's direction matrices drive the reference's own ConstructProfile through the whole upgma tree of
    adeno_fiber: the final alignment must be the reference's, row for row."""
    from dp_cases import driven_progressive_alignment
    z = np.load(os.path.join(GOLDEN, "adeno_upgma_merges.npz"))
    seqs = [str(s) for s in z["seqs"]]
    merges = [tuple(int(x) for x in m) for m in z["merges"]]
    rows, total = driven_progressive_alignment(
        seqs, merges, lambda jobs, g: [pyoracle.dp_align(*j, g) for j in jobs])
    _, recs = reference_merges(seqs, merges, threads=(1,))
    assert rows == recs[-1]["rows"] and total == recs[-1]["total"] == int(z["totals"][-1])


def _check_construct(res, recs, g):
    """oracle ConstructProfile merge part == the reference's merged scores/counters, merge by merge."""
    for k, (r, rec) in enumerate(zip(res, recs)):
        s1, c1, k1, s2, c2, k2 = rec["job"]
        rp, cp = ((s2, c2, k2), (s1, c1, k1)) if r["swapped"] else ((s1, c1, k1), (s2, c2, k2))
        s, c, g1, g2 = pyoracle.dp_construct(rp, cp, r["path"], g)
        ws, wc, wk = rec["merged"]
        assert wk == k1 + k2 and ws.shape == s.shape, f"merge {k}"
        assert np.array_equal(c, wc), f"merge {k}: counters differ"
        assert np.array_equal(s, ws), f"merge {k}: scores differ"
        # gap runs: exactly the H (resp. V) runs of the path, as (first merged column, length)
        for runs, d in ((g1, 1), (g2, 2)):
            mask = np.zeros(len(r["path"]) + 2, dtype=bool)
            for a, ln in runs:
                assert not mask[a:a + ln].any()
                mask[a:a + ln] = True
            assert np.array_equal(mask[1:-1], r["path"] == d)
            assert all(not mask[a - 1] and not mask[a + ln] for a, ln in runs), "runs must be maximal"


def test_oracle_construct_golden_upgma_tree():
    """Merged profile tables after each of the 241 merges behind upgma.no_refine.fasta (ConstructProfile,
    profile.cpp:784-1002) -- the widened row SURVEY 8f-2."""
    z = np.load(os.path.join(GOLDEN, "adeno_upgma_merges.npz"))
    seqs = [str(s) for s in z["seqs"]]
    merges = [tuple(int(x) for x in m) for m in z["merges"]]
    g, recs = reference_merges(seqs, merges, threads=(1,), want_merged=True)
    res = [pyoracle.dp_align(*r["job"], g) for r in recs]
    _check_construct(res, recs, g)


@pytest.mark.parametrize("seed,n,length,gaps", [(11, 50, 80, None), (12, 40, 200, (-9000, -700, -300, -100))])
def test_oracle_construct_random_families(seed, n, length, gaps):
    rng = np.random.default_rng(seed)
    codes, off, lens = seqio.synth_family(n, length, seed, sort_desc=False)
    seqs = [seqio.decode(codes[int(o):int(o) + int(l)]) for o, l in zip(off, lens)]
    seqs[1] = seqs[1][:3] + "XBZ" + seqs[1][6:]
    merges = random_tree(n, rng, caterpillar=0.5)
    g, recs = reference_merges(seqs, merges, threads=(1, 2), rng=rng, gaps=gaps, want_merged=True)
    res = [pyoracle.dp_align(*r["job"], g) for r in recs]
    _check_construct(res, recs, g)


def test_oracle_progressive_alignment_from_fixture_alone():
    """No oracle/_ref needed: leaves from the host mirror of CalculateCountersScores, DP + merged tables from the
    restatement, level by level over the 241 merges behind upgma.no_refine.fasta; totals, paths and the CRC32 of every
    merged profile's scores/counters must equal what the reference produced when the fixture was generated."""
    from famsa_b200 import profiles
    z = np.load(os.path.join(GOLDEN, "adeno_upgma_merges.npz"))
    seqs = [str(s) for s in z["seqs"]]
    merges = [tuple(int(x) for x in m) for m in z["merges"]]
    g, sm = z["gaps"], z["score_matrix"]
    n = len(seqs)
    node = {i: profiles.tables_from_rows(seqio.encode(seqs[i])[None, :], sm, g) for i in range(n)}
    at = 0
    for k, (a, b) in enumerate(merges):
        ta, tb = node.pop(a), node.pop(b)
        r = pyoracle.dp_align(*ta, *tb, g)
        assert r["total"] == int(z["totals"][k]) and r["swapped"] == bool(z["swapped"][k])
        assert np.array_equal(r["path"], z["path"][at:at + int(z["path_len"][k])])
        at += int(z["path_len"][k])
        rp, cp = (tb, ta) if r["swapped"] else (ta, tb)
        s, c, _, _ = pyoracle.dp_construct(rp, cp, r["path"], g)
        assert (zlib.crc32(s.tobytes()), zlib.crc32(c.tobytes())) == tuple(int(x) for x in z["merged_crc"][k]), f"merge {k}"
        node[n + k] = (s, c, ta[2] + tb[2])
