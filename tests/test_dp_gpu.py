"""GPU parity tests for HP-2 (through the C ABI).  int64 scores -> bit-exact, paths byte-identical."""
import os
import zlib

import numpy as np
import pytest

from conftest import GOLDEN
from dp_cases import check_against_reference, random_tree, reference_merges
from famsa_b200 import seqio
from oracle import pyoracle

pytestmark = pytest.mark.gpu


def assert_same(got, want, dirs=True):
    assert got["variant"] == want["variant"] and got["swapped"] == want["swapped"]
    assert got["total"] == want["total"]
    assert np.array_equal(got["last"], want["last"])
    assert np.array_equal(got["path"], want["path"])
    if dirs:
        assert np.array_equal(got["dirs"], want["dirs"])


def test_pp_golden(engine):
    """The reference's profile-profile known answer (upgma.pp.fasta), incl. the whole direction matrix."""
    z = np.load(os.path.join(GOLDEN, "adeno_pp.npz"))
    job = (z["s1"], z["c1"], int(z["k1"]), z["s2"], z["c2"], int(z["k2"]))
    got = engine.dp_align_batch([job], z["gaps"], want_dirs=True)[0]
    assert got["total"] == int(z["total"]) and np.array_equal(got["path"], z["path"])
    assert_same(got, pyoracle.dp_align(*job, z["gaps"]))


def test_all_merges_of_golden_upgma_tree(engine):
    """241 merges behind upgma.no_refine.fasta in ONE batch: every variant, oracle + reference + fixture."""
    z = np.load(os.path.join(GOLDEN, "adeno_upgma_merges.npz"))
    seqs = [str(s) for s in z["seqs"]]
    merges = [tuple(int(x) for x in m) for m in z["merges"]]
    g, recs = reference_merges(seqs, merges, threads=(1,))
    got = engine.dp_align_batch([r["job"] for r in recs], g, want_dirs=True)
    check_against_reference(got, recs)
    assert [r["total"] for r in got] == [int(t) for t in z["totals"]]
    assert np.array_equal(np.concatenate([r["path"] for r in got]), z["path"])
    for r, rec in zip(got, recs):
        assert_same(r, pyoracle.dp_align(*rec["job"], g))


@pytest.mark.parametrize("want_dirs", [False, True])
def test_sub_batching(engine, monkeypatch, want_dirs):
    """Large batches are cut into sub-batches that bound the device scratch; force tiny ones."""
    z = np.load(os.path.join(GOLDEN, "adeno_upgma_merges.npz"))
    seqs = [str(s) for s in z["seqs"]]
    merges = [tuple(int(x) for x in m) for m in z["merges"]]
    g, recs = reference_merges(seqs, merges, threads=(1,))
    monkeypatch.setenv("FAMSA_DP_MAX_CELLS", "60000")
    got = engine.dp_align_batch([r["job"] for r in recs], g, want_dirs=want_dirs)
    check_against_reference(got, recs)
    if want_dirs:
        for r, rec in zip(got[::17], recs[::17]):
            assert np.array_equal(r["dirs"], pyoracle.dp_align(*rec["job"], g)["dirs"])


def test_hemopexin_all_merges(engine):
    """BASELINE config 4: all 4187 guide-tree merges of test/hemopexin (medoid-sl tree) on one B200, level by
    level the way a host scheduler would submit them; totals and path CRCs pinned by the fixture, which was
    generated from a reference run that reproduces medoid-sl.fasta byte for byte."""
    from treeutil import levels
    z = np.load(os.path.join(GOLDEN, "hemopexin_medoid_sl.npz"))
    seqs = [str(s) for s in z["seqs"]]
    merges = [tuple(int(x) for x in m) for m in z["merges"]]
    g, recs = reference_merges(seqs, merges, threads=(1,))
    assert np.array_equal(g, z["gaps"])
    n_checked = 0
    for lvl in levels(len(seqs), merges):
        got = engine.dp_align_batch([recs[k]["job"] for k in lvl], g)
        for k, r in zip(lvl, got):
            assert r["total"] == int(z["totals"][k]) == recs[k]["total"], f"merge {k}"
            assert zlib.crc32(r["path"].tobytes()) == int(z["path_crc"][k]), f"merge {k}"
            n_checked += 1
    assert n_checked == 4187
    check_against_reference(engine.dp_align_batch([recs[k]["job"] for k in range(4000, 4187)], g), recs[4000:])


@pytest.mark.parametrize("fixture", ["adeno_upgma_merges.npz", "hemopexin_medoid_sl.npz"])
def test_gpu_driven_progressive_alignment(engine, fixture):
    """Drop-in proof for HP-2: the GPU's direction matrices and corner scores feed the reference's UNMODIFIED
    ConstructProfile level by level (the loop INTEGRATION.md describes); the final multiple alignment is the
    reference's -- for adeno_fiber that is the golden upgma.no_refine.fasta, for hemopexin the golden
    medoid-sl.fasta (4188 sequences, 94 levels), both asserted equal to the reference run when the fixtures
    were generated."""
    from dp_cases import driven_progressive_alignment
    z = np.load(os.path.join(GOLDEN, fixture))
    seqs = [str(s) for s in z["seqs"]]
    merges = [tuple(int(x) for x in m) for m in z["merges"]]
    rows, total = driven_progressive_alignment(
        seqs, merges, lambda jobs, g: engine.dp_align_batch(jobs, g, want_dirs=True))
    _, recs = reference_merges(seqs, merges, threads=(1,))
    assert total == int(z["totals"][-1]) == recs[-1]["total"]
    assert rows == recs[-1]["rows"]


@pytest.mark.parametrize("seed,n,length,gaps", [(11, 70, 60, None), (12, 24, 500, None), (13, 40, 33, (-9000, -700, -300, -100)),
                                                (14, 12, 1300, None), (15, 30, 31, (-20000, -2000, -2500, -900))])
def test_random_families(engine, seed, n, length, gaps):
    """Ragged widths around the 32-row stripe size, > 1000 columns, non-default gap costs, X/B/Z residues."""
    rng = np.random.default_rng(seed)
    codes, off, lens = seqio.synth_family(n, length, seed, sort_desc=False)
    seqs = [seqio.decode(codes[int(o):int(o) + int(l)]) for o, l in zip(off, lens)]
    seqs[1] = seqs[1][:3] + "XBZ*" + seqs[1][7:]
    merges = random_tree(n, rng)
    g, recs = reference_merges(seqs, merges, threads=(1, 2), rng=rng, gaps=gaps)
    got = engine.dp_align_batch([r["job"] for r in recs], g, want_dirs=True)
    check_against_reference(got, recs)
    for r, rec in zip(got, recs):
        assert_same(r, pyoracle.dp_align(*rec["job"], g))


def test_cluster_path(engine, monkeypatch):
    """Very wide merges run on a thread-block cluster (8 blocks x 8 warps); force that path on ordinary sizes."""
    rng = np.random.default_rng(21)
    codes, off, lens = seqio.synth_family(48, 330, 21, sort_desc=False)
    seqs = [seqio.decode(codes[int(o):int(o) + int(l)]) for o, l in zip(off, lens)]
    merges = random_tree(48, rng)
    g, recs = reference_merges(seqs, merges, threads=(1,), rng=rng)
    monkeypatch.setenv("FAMSA_DP_CLUSTER_MIN", "200")
    got = engine.dp_align_batch([r["job"] for r in recs], g, want_dirs=True)
    check_against_reference(got, recs)
    for r, rec in zip(got, recs):
        assert_same(r, pyoracle.dp_align(*rec["job"], g))


def test_tiny_and_degenerate(engine):
    """Width-1 profiles, 1 x many, without the reference (oracle only)."""
    rng = np.random.default_rng(3)

    def prof(width, card):
        c = np.zeros((width + 1, 32), dtype=np.int32)
        for j in range(1, width + 1):
            for _ in range(card):
                c[j, int(rng.integers(0, 24))] += 1
        s = rng.integers(-5000, 5000, size=(width + 1, 32)).astype(np.int64) * card
        return s, c, card

    gaps = np.array([-14850, -1250, -660, -660], dtype=np.int64)
    jobs = []
    for w1, k1, w2, k2 in [(1, 1, 1, 1), (1, 1, 7, 1), (5, 1, 1, 3), (1, 4, 1, 2), (33, 2, 32, 5), (64, 3, 65, 3), (2, 1, 40, 9)]:
        a, b = prof(w1, k1), prof(w2, k2)
        jobs.append((a[0], a[1], a[2], b[0], b[1], b[2]))
    got = engine.dp_align_batch(jobs, gaps, want_dirs=True)
    for r, job in zip(got, jobs):
        assert_same(r, pyoracle.dp_align(*job, gaps))
    assert engine.dp_align_batch([], gaps) == []
    with pytest.raises(Exception):
        engine.dp_align_batch([(jobs[0][0][:1], jobs[0][1][:1], 1, jobs[0][3], jobs[0][4], 1)], gaps)


def test_inconsistent_profile_is_rejected(engine):
    """The cell loop multiplies scores with gap / residue counts as unsigned 32-bit values; a table whose counts are
    negative (more gaps than members -- nothing CProfile can build) must fail loudly instead of diverging silently."""
    from famsa_b200 import profiles
    from famsa_b200.binding import FamsaError
    rng = np.random.default_rng(2)
    sm = profiles.synth_score_matrix(rng)
    gaps = np.array([-14850, -1250, -660, -660], dtype=np.int64)
    a = profiles.tables_from_rows(profiles.synth_alignment(5, 40, rng), sm, gaps)
    b = profiles.tables_from_rows(profiles.synth_alignment(4, 35, rng), sm, gaps)
    engine.dp_align_batch([(a[0], a[1], a[2], b[0], b[1], b[2])], gaps)          # consistent: fine
    c = b[1].copy()
    c[7, 25] = 9                                                                  # 9 gap-opens in a 4-member profile
    with pytest.raises(FamsaError, match="negative"):
        engine.dp_align_batch([(a[0], a[1], a[2], b[0], c, b[2])], gaps)


@pytest.mark.parametrize("env", [{}, {"FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_TEAM_MIN": "32", "FAMSA_DP_COMPACT": "2"},
                                 {"FAMSA_DP_LATENCY_MODE": "1", "FAMSA_DP_DUO": "0"}])
def test_scores_beyond_32_bits(engine, monkeypatch, env):
    """The column-pair scores T have a tensor-core path for tables whose scores fit in int32 (every realistic profile) and a
    scalar 32 x 64 path otherwise, and the T ring holds 4- or 8-byte entries; substitution scores of ~1e9 push the tables
    past 2^31 and exercise the wide forms -- in the default launch shape, in the compact kernel (which must leave such merges
    to the full kernel launched behind it) and in plain clusters."""
    from famsa_b200 import profiles
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(9)
    sm = profiles.synth_score_matrix(rng) * 300_000
    gaps = np.array([-14850, -1250, -660, -660], dtype=np.int64) * 300_000
    jobs = []
    for _ in range(6):
        a = profiles.tables_from_rows(profiles.synth_alignment(int(rng.integers(3, 9)), int(rng.integers(40, 140)), rng), sm, gaps)
        b = profiles.tables_from_rows(profiles.synth_alignment(int(rng.integers(3, 9)), int(rng.integers(40, 140)), rng), sm, gaps)
        jobs.append((a[0], a[1], a[2], b[0], b[1], b[2]))
    assert max(int(np.abs(j[3]).max()) for j in jobs) > 2 ** 31
    got = engine.dp_align_batch(jobs, gaps, want_dirs=True)
    for r, j in zip(got, jobs):
        assert_same(r, pyoracle.dp_align(*j, gaps))
