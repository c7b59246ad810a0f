"""GPU tests for the resident-profile path (SURVEY 8f-2): famsa_prof_merge_batch = CProfile::Align + the table
half of ConstructProfile with all profiles kept in HBM.  Every merged table is compared with the reference's own
ConstructProfile output (oracle/_ref) and with the CPU restatement; the alignment assembled from the returned
paths must be the reference's."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from dp_cases import (check_against_reference, random_tree, reference_merges, reference_score_matrix,
                      resident_progressive_alignment)
from famsa_b200 import seqio
from famsa_b200.binding import PROF_LEAF, Engine, FamsaError
from oracle import pyoracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    e = Engine()
    yield e
    e.close()


def _score_matrix(n):
    return reference_score_matrix(n)


def _run_and_check(engine, seqs, merges, g, recs, sm):
    """Resident run; after each level compares the merged tables with the reference's and the restatement's."""
    def on_level(lvl, ids, res):
        for k, pid, r in zip(lvl, ids, res):
            s, c, card = engine.prof_get(pid)
            ws, wc, wk = recs[k]["merged"]
            assert card == wk and s.shape == ws.shape, f"merge {k}"
            assert np.array_equal(c, wc), f"merge {k}: counters differ from the reference's ConstructProfile"
            assert np.array_equal(s, ws), f"merge {k}: scores differ from the reference's ConstructProfile"
            s1, c1, k1, s2, c2, k2 = recs[k]["job"]
            rp, cp = ((s2, c2, k2), (s1, c1, k1)) if r["swapped"] else ((s1, c1, k1), (s2, c2, k2))
            os_, oc, _, _ = pyoracle.dp_construct(rp, cp, r["path"], g)
            assert np.array_equal(os_, s) and np.array_equal(oc, c)
    rows, results, root = resident_progressive_alignment(engine, seqs, merges, g, sm, on_level)
    check_against_reference(results, recs)
    assert rows == recs[-1]["rows"], "alignment assembled from the GPU's paths differs from the reference's"
    assert engine.prof_stats()[0] == 1
    engine.prof_drop([root])
    assert engine.prof_stats() == (0, 0)
    return results


def test_resident_golden_upgma_tree(engine):
    """All 241 merges behind test/adeno_fiber/upgma.no_refine.fasta with profiles resident in HBM."""
    z = np.load(os.path.join(GOLDEN, "adeno_upgma_merges.npz"))
    seqs = [str(s) for s in z["seqs"]]
    merges = [tuple(int(x) for x in m) for m in z["merges"]]
    g, recs = reference_merges(seqs, merges, threads=(1,), want_merged=True)
    res = _run_and_check(engine, seqs, merges, g, recs, _score_matrix(len(seqs)))
    assert [r["total"] for r in res] == [int(t) for t in z["totals"]]
    assert np.array_equal(np.concatenate([r["path"] for r in res]), z["path"])


@pytest.mark.parametrize("seed,n,length,gaps,cat", [(31, 60, 70, None, 0.3), (32, 24, 400, None, 0.6),
                                                    (33, 40, 33, (-9000, -700, -300, -100), 0.2),
                                                    (34, 10, 1300, None, 0.5)])
def test_resident_random_families(engine, seed, n, length, gaps, cat):
    rng = np.random.default_rng(seed)
    codes, off, lens = seqio.synth_family(n, length, seed, sort_desc=False)
    seqs = [seqio.decode(codes[int(o):int(o) + int(l)]) for o, l in zip(off, lens)]
    seqs[1] = seqs[1][:3] + "XBZ*" + seqs[1][7:]
    merges = random_tree(n, rng, caterpillar=cat)
    g, recs = reference_merges(seqs, merges, threads=(1, 2), rng=rng, gaps=gaps, want_merged=True)
    _run_and_check(engine, seqs, merges, g, recs, _score_matrix(n))


def test_resident_hemopexin(engine):
    """4188 sequences / 94 levels (golden medoid-sl tree): totals and path checksums of every merge, and the final
    alignment assembled from the paths, equal the fixture the reference generated."""
    import zlib
    z = np.load(os.path.join(GOLDEN, "hemopexin_medoid_sl.npz"))
    seqs = [str(s) for s in z["seqs"]]
    merges = [tuple(int(x) for x in m) for m in z["merges"]]
    rows, res, root = resident_progressive_alignment(engine, seqs, merges, z["gaps"], _score_matrix(len(seqs)))
    assert [r["total"] for r in res] == [int(t) for t in z["totals"]]
    assert [zlib.crc32(r["path"].tobytes()) for r in res] == [int(c) for c in z["path_crc"]]
    assert len({len(v) for v in rows.values()}) == 1 and len(rows) == len(seqs)
    for i in (0, 17, 4187):
        assert rows[i].replace("-", "") == seqs[i]
    engine.prof_drop([root])
    assert engine.prof_stats() == (0, 0)


def test_prof_put_and_mixed_children(engine):
    """Host-built tables uploaded with famsa_prof_put merge exactly like the reference's; leaf + resident mixes."""
    rng = np.random.default_rng(5)
    codes, off, lens = seqio.synth_family(9, 120, 5, sort_desc=False)
    seqs = [seqio.decode(codes[int(o):int(o) + int(l)]) for o, l in zip(off, lens)]
    merges = [(0, 1), (2, 3), (9, 10), (11, 4), (5, 12), (6, 7), (14, 13), (15, 8)]
    g, recs = reference_merges(seqs, merges, threads=(1,), want_merged=True)
    engine.upload(codes, off, lens)
    engine.prof_set_scoring(_score_matrix(9))
    # merges 0 and 1 on the host side (reference tables), uploaded; merge 2 joins them on the device
    ids = engine.prof_put([recs[0]["merged"], recs[1]["merged"]])
    w = [recs[0]["merged"][0].shape[0] - 1, recs[1]["merged"][0].shape[0] - 1]
    assert engine.prof_get(ids[0], tables=False) == (w[0], 2)
    mid, res = engine.prof_merge_batch([(ids[0], ids[1])], g, [(w[0], w[1])])
    check_against_reference(res, [recs[2]])
    s, c, k = engine.prof_get(mid[0])
    assert np.array_equal(s, recs[2]["merged"][0]) and np.array_equal(c, recs[2]["merged"][1]) and k == 4
    # resident x leaf (SeqProf both ways), leaf x leaf in one batch
    m3, r3 = engine.prof_merge_batch([(mid[0], PROF_LEAF | 4), (PROF_LEAF | 6, PROF_LEAF | 7)], g,
                                     [(len(res[0]["path"]), len(seqs[4])), (len(seqs[6]), len(seqs[7]))])
    check_against_reference(r3, [recs[3], recs[5]])
    m4, r4 = engine.prof_merge_batch([(PROF_LEAF | 5, m3[0])], g, [(len(seqs[5]), len(r3[0]["path"]))])
    check_against_reference(r4, [recs[4]])
    for pid, k in ((m4[0], 4), (m3[1], 5)):
        s, c, _ = engine.prof_get(pid)
        assert np.array_equal(s, recs[k]["merged"][0]) and np.array_equal(c, recs[k]["merged"][1])
    engine.prof_drop([m4[0], m3[1]])
    assert engine.prof_stats() == (0, 0)


def test_prof_errors(engine):
    codes, off, lens = seqio.synth_family(4, 50, 1, sort_desc=False)
    engine.upload(codes, off, lens)
    engine.prof_set_scoring(np.eye(24, dtype=np.int64))
    g = np.array([-14000, -1200, -3000, -500], dtype=np.int64)
    with pytest.raises(FamsaError, match="not uploaded"):
        engine.prof_merge_batch([(PROF_LEAF | 0, PROF_LEAF | 9)], g, [(50, 50)])
    with pytest.raises(FamsaError, match="not a resident profile"):
        engine.prof_merge_batch([(PROF_LEAF | 0, 123456)], g, [(50, 50)])
    with pytest.raises(FamsaError, match="path_buf"):
        engine.prof_merge_batch([(PROF_LEAF | 0, PROF_LEAF | 1)], g, [(3, 3)])
    ids, _ = engine.prof_merge_batch([(PROF_LEAF | 0, PROF_LEAF | 1)], g, [(int(lens[0]), int(lens[1]))])
    w, _ = engine.prof_get(ids[0], tables=False)
    with pytest.raises(FamsaError, match="used twice"):
        engine.prof_merge_batch([(ids[0], ids[0])], g, [(w, w)])
    ids2, _ = engine.prof_merge_batch([(ids[0], PROF_LEAF | 2)], g, [(w, int(lens[2]))])
    with pytest.raises(FamsaError, match="not a resident profile"):      # consumed by the merge above
        engine.prof_get(ids[0])
    engine.prof_drop(ids2)
    with pytest.raises(FamsaError, match="not a resident profile"):
        engine.prof_drop(ids2)
    assert engine.prof_stats() == (0, 0)


@pytest.mark.parametrize("env", [{"FAMSA_PROF_FUSED": "0", "FAMSA_DP_MAX_CELLS": "60000"},
                                 {"FAMSA_PROF_FUSED": "0", "FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_CLUSTER_MIN": "40", "FAMSA_DP_TEAM_MIN": "32"},
                                 {"FAMSA_PROF_FUSED": "0", "FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_TEAM_MIN": "100000"},
                                 {"FAMSA_PROF_FUSED": "0", "FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_TEAM_WARPS": "2"},
                                 {"FAMSA_PROF_FUSED": "0", "FAMSA_DP_LATENCY_MODE": "1", "FAMSA_DP_MAX_CLUSTER": "2"},
                                 {"FAMSA_PROF_FUSED": "0", "FAMSA_DP_LATENCY_MODE": "1"},
                                 {"FAMSA_PROF_FUSED": "0", "FAMSA_DP_LATENCY_MODE": "1", "FAMSA_DP_DUO": "0"},
                                 {"FAMSA_PROF_FUSED": "0", "FAMSA_DP_LATENCY_MODE": "1", "FAMSA_DP_MAX_CLUSTER": "2", "FAMSA_DP_DUO": "0"},
                                 {"FAMSA_PROF_FUSED": "0", "FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_TEAM_MIN": "32", "FAMSA_DP_COMPACT": "2"},
                                 {"FAMSA_PROF_FUSED": "0", "FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_TEAM_MIN": "32", "FAMSA_DP_COMPACT": "2", "FAMSA_DP_TEAM_WARPS": "2"},
                                 {"FAMSA_PROF_FUSED": "0", "FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_TEAM_MIN": "32", "FAMSA_DP_COMPACT": "2", "FAMSA_DP_TEAM_WARPS": "4"},
                                 {"FAMSA_PROF_FUSED": "1"}])
def test_resident_launch_shapes(engine, monkeypatch, env):
    """The resident path through sub-batches of a few merges and through every launch shape of the fill kernel: the
    throughput-mode cluster (8 x 8 warps), one warp per merge, 2-warp teams, the compact 12-warps-per-SM kernel with 6, 2 and 4
    warps per merge, the latency-mode clusters of producer / consumer pairs and of plain 4-warp blocks, and the fused
    one-block-per-merge kernel (development knobs of dp.cu / prof.cu force each shape on an ordinary family)."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(41)
    codes, off, lens = seqio.synth_family(36, 150, 41, sort_desc=False)
    seqs = [seqio.decode(codes[int(o):int(o) + int(l)]) for o, l in zip(off, lens)]
    merges = random_tree(36, rng, caterpillar=0.4)
    g, recs = reference_merges(seqs, merges, threads=(1,), rng=rng, want_merged=True)
    _run_and_check(engine, seqs, merges, g, recs, _score_matrix(36))


def test_resident_golden_tables_without_reference(engine):
    """Needs only the committed fixture: the resident path over all 241 merges behind upgma.no_refine.fasta; totals,
    paths and the CRC32 of every merged profile's scores/counters equal the reference's (recorded at generation)."""
    import zlib
    z = np.load(os.path.join(GOLDEN, "adeno_upgma_merges.npz"))
    seqs = [str(s) for s in z["seqs"]]
    merges = [tuple(int(x) for x in m) for m in z["merges"]]
    crcs = {}

    def on_level(lvl, ids, res):
        for k, pid in zip(lvl, ids):
            s, c, _ = engine.prof_get(pid)
            crcs[k] = (zlib.crc32(s.tobytes()), zlib.crc32(c.tobytes()))
    rows, res, root = resident_progressive_alignment(engine, seqs, merges, z["gaps"], z["score_matrix"], on_level)
    engine.prof_drop([root])
    assert [r["total"] for r in res] == [int(t) for t in z["totals"]]
    assert np.array_equal(np.concatenate([r["path"] for r in res]), z["path"])
    assert [crcs[k] for k in range(len(merges))] == [tuple(int(x) for x in row) for row in z["merged_crc"]]
