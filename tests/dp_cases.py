"""Shared helpers for the HP-2 tests: drive the reference (oracle/_ref) through a guide tree, collecting
for every merge the inputs of CProfile::Align and the reference's outcome (path, total score)."""
from __future__ import annotations

import numpy as np

from oracle import pyoracle

import refgold


def random_tree(n: int, rng, caterpillar: float = 0.3) -> list[tuple[int, int]]:
    """Random binary merge order over n leaves (ids as in tree_structure)."""
    alive = list(range(n))
    merges = []
    while len(alive) > 1:
        if rng.random() < caterpillar and len(merges):
            a = alive.pop()                      # extend the newest node (deep, chain-like)
            b = alive.pop(int(rng.integers(len(alive))))
        else:
            a = alive.pop(int(rng.integers(len(alive))))
            b = alive.pop(int(rng.integers(len(alive))))
        merges.append((a, b))
        alive.append(n + len(merges) - 1)
    return merges


def reference_gaps(n_seqs_for_rescale: int, gaps=None) -> np.ndarray:
    """The reference's gap costs (CParams defaults or `gaps`, rescaled for n_seqs_for_rescale sequences)."""
    def run():
        dp = pyoracle.RefDp(n_seqs_for_rescale)
        if gaps is not None:
            dp.set_gaps(gaps)
        g = dp.gaps()
        dp.close()
        return g
    return refgold.answer("gaps/" + refgold.input_key(n_seqs_for_rescale, None if gaps is None else [int(x) for x in gaps]), run)


def reference_score_matrix(n_seqs_for_rescale: int = 0) -> np.ndarray:
    """The reference's substitution matrix (the same for every set size)."""
    def run():
        dp = pyoracle.RefDp(n_seqs_for_rescale)
        sm = dp.score_matrix()
        dp.close()
        return sm
    return refgold.answer("score_matrix", run)


def rows_crc(rows: dict[int, str]) -> int:
    return refgold.crc(np.frombuffer("\n".join(rows[k] for k in sorted(rows)).encode(), dtype=np.uint8))


def _job_crc(job) -> int:
    s1, c1, k1, s2, c2, k2 = job
    return refgold.crc(np.concatenate([s1.ravel(), c1.ravel().astype(np.int64), [k1], s2.ravel(), c2.ravel().astype(np.int64), [k2]]))


def _tables_crc(t) -> int:
    return refgold.crc(np.concatenate([t[0].ravel(), t[1].ravel().astype(np.int64), [t[2]]]))


def _path_crc(path, swapped: bool) -> int:
    """CRC of a path in the unswapped orientation (swapping the DP's roles exchanges H and V)."""
    p = np.asarray(path, dtype=np.uint8)
    return refgold.crc(np.where(p == 0, 0, 3 - p).astype(np.uint8) if swapped else p)


def _live_merges(seqs, merges, n_rescale, picks, gaps, want_merged):
    n = len(seqs)
    dp = pyoracle.RefDp(n_rescale)
    if gaps is not None:
        dp.set_gaps(gaps)
    g = dp.gaps()
    nodes = {i: (dp.leaf(seqs[i], i), {i}) for i in range(n)}
    recs = []
    for k, (a, b) in enumerate(merges):
        pa, ma = nodes.pop(a)
        pb, mb = nodes.pop(b)
        s1, c1, k1 = dp.tables(pa)
        s2, c2, k2 = dp.tables(pb)
        m, total = dp.align(pa, pb, picks[k])
        recs.append(dict(job=(s1, c1, k1, s2, c2, k2), m1=ma, m2=mb, total=total, rows=dp.rows(m)))
        merged = dp.tables(m)                    # the tables ConstructProfile built (profile.cpp:784-1002)
        recs[-1]["merged_crc"] = _tables_crc(merged)
        if want_merged:
            recs[-1]["merged"] = merged
        nodes[n + k] = (m, ma | mb)
    for p, _ in nodes.values():
        dp.free(p)
    dp.close()
    return g, recs


def _restated_merges(seqs, merges, g, sm):
    """The same progressive alignment from the host mirror of CalculateCountersScores (leaves) and the C restatement
    (DP, merged tables); the caller checks it against the reference's stored answers."""
    from famsa_b200 import profiles
    from famsa_b200 import seqio
    n = len(seqs)
    nodes = {i: (profiles.tables_from_rows(seqio.encode(seqs[i])[None, :], sm, g), {i}) for i in range(n)}
    recs, results = [], []
    for k, (a, b) in enumerate(merges):
        ta, ma = nodes.pop(a)
        tb, mb = nodes.pop(b)
        r = pyoracle.dp_align(*ta, *tb, g)
        rp, cp = (tb, ta) if r["swapped"] else (ta, tb)
        s, c, _, _ = pyoracle.dp_construct(rp, cp, r["path"], g)
        merged = (s, c, ta[2] + tb[2])
        recs.append(dict(job=(*ta, *tb), m1=ma, m2=mb, total=r["total"], merged=merged))
        results.append(r)
        nodes[n + k] = (merged, ma | mb)
    recs[-1]["rows"] = assemble_rows(seqs, merges, results)
    return recs, results


def reference_merges(seqs: list[str], merges, n_seqs_for_rescale: int | None = None, threads=(1, 2), rng=None,
                     gaps=None, want_merged: bool = False):
    """Runs the reference's progressive alignment.  Returns (gaps, records) where each record is a dict with
    the Align inputs (s1,c1,k1,s2,c2,k2), members, and the reference's result: total, path_crc (CRC of the path in
    the unswapped orientation), merged_crc (CRC of the merged tables), the merged tables with want_merged, and the rows
    of the merged profile.  Without oracle/_ref the inputs and tables come from the restatement, checked merge by merge
    against the reference's stored answers, and only the last record holds rows (the final alignment)."""
    rng = rng or np.random.default_rng(0)
    picks = [int(rng.choice(threads)) for _ in merges]
    n_rescale = len(seqs) if n_seqs_for_rescale is None else n_seqs_for_rescale
    key = "merges/" + refgold.input_key(seqs, [(int(a), int(b)) for a, b in merges], n_rescale,
                                        None if gaps is None else [int(x) for x in gaps])
    g, recs = _live_merges(seqs, merges, n_rescale, picks, gaps, want_merged) if refgold.live() else (None, None)
    g = refgold.answer(key + "/gaps", lambda: g)
    total = refgold.answer(key + "/total", lambda: np.array([r["total"] for r in recs], dtype=np.int64))
    path_crc = refgold.answer(key + "/path_crc", lambda: np.array(
        [refgold.crc(pyoracle.path_from_rows(r["rows"], r["m1"], r["m2"], False)) for r in recs], dtype=np.uint32))
    job_crc = refgold.answer(key + "/job_crc", lambda: np.array([_job_crc(r["job"]) for r in recs], dtype=np.uint32))
    merged_crc = refgold.answer(key + "/merged_crc", lambda: np.array([r["merged_crc"] for r in recs], dtype=np.uint32))
    final_crc = refgold.answer(key + "/rows_crc", lambda: np.array([rows_crc(recs[-1]["rows"])], dtype=np.uint32))
    if recs is None:
        recs, results = _restated_merges(seqs, merges, g, reference_score_matrix())
        for k, (rec, r) in enumerate(zip(recs, results)):
            assert _job_crc(rec["job"]) == job_crc[k], f"merge {k}: restated Align inputs differ from the reference's"
            assert rec["total"] == total[k] and _path_crc(r["path"], r["swapped"]) == path_crc[k], f"merge {k}"
            assert _tables_crc(rec["merged"]) == merged_crc[k], f"merge {k}: restated merged tables differ"
            rec["merged_crc"] = int(merged_crc[k])
            if not want_merged:
                del rec["merged"]
        assert rows_crc(recs[-1]["rows"]) == final_crc[0]
    for k, rec in enumerate(recs):
        rec["path_crc"] = int(path_crc[k])
    return g, recs


def check_against_reference(results, recs):
    """results: list of dicts with path/total/swapped (oracle or GPU), in the order of recs."""
    for k, (r, rec) in enumerate(zip(results, recs)):
        assert r["total"] == rec["total"], f"merge {k}: total {r['total']} != {rec['total']}"
        if "rows" in rec:
            want = pyoracle.path_from_rows(rec["rows"], rec["m1"], rec["m2"], r["swapped"])
            assert np.array_equal(r["path"], want[:len(r["path"])]) and len(want) == len(r["path"]), f"merge {k}: path differs"
        assert _path_crc(r["path"], r["swapped"]) == rec["path_crc"], f"merge {k}: path differs"


def driven_progressive_alignment(seqs, merges, align_level, n_seqs_for_rescale=None):
    """Level-synchronous progressive alignment in which the DP (direction matrices + corner scores) comes from
    `align_level(jobs, gaps) -> [dict(dirs, last, swapped, path), ...]` and everything else -- leaf profiles, the merged
    profile construction -- is the reference's own host code (ConstructProfile, profile.cpp:694-1002, through
    oracle/ref_harness.cpp); without oracle/_ref, the host mirror and the restatement, which reference_merges pins to
    the reference.  Returns the final alignment rows {seq_no: gapped string} and the root total score."""
    from famsa_b200.schedule import ready_levels
    n = len(seqs)
    n_rescale = n if n_seqs_for_rescale is None else n_seqs_for_rescale
    if not refgold.live():
        return _restated_driven(seqs, merges, align_level, reference_gaps(n_rescale))
    dp = pyoracle.RefDp(n_rescale)
    g = dp.gaps()
    assert np.array_equal(g, reference_gaps(n_rescale))
    nodes = {i: dp.leaf(seqs[i], i) for i in range(n)}
    for lvl in ready_levels(n, merges):
        jobs = []
        for k in lvl:
            a, b = merges[k]
            s1, c1, k1 = dp.tables(nodes[a])
            s2, c2, k2 = dp.tables(nodes[b])
            jobs.append((s1, c1, k1, s2, c2, k2))
        res = align_level(jobs, g)
        for k, r in zip(lvl, res):
            a, b = merges[k]
            nodes[n + k] = dp.construct(nodes.pop(a), nodes.pop(b), r["dirs"], r["last"], r["swapped"])
    root = nodes[n + len(merges) - 1]
    rows = dp.rows(root)
    total = int(dp.lib.ref_profile_total_score(root))
    dp.free(root)
    dp.close()
    return rows, total


def _restated_driven(seqs, merges, align_level, g):
    from famsa_b200 import profiles
    from famsa_b200 import seqio
    from famsa_b200.schedule import ready_levels
    n = len(seqs)
    sm = reference_score_matrix()
    nodes = {i: profiles.tables_from_rows(seqio.encode(seqs[i])[None, :], sm, g) for i in range(n)}
    results = [None] * len(merges)
    for lvl in ready_levels(n, merges):
        res = align_level([(*nodes[merges[k][0]], *nodes[merges[k][1]]) for k in lvl], g)
        for k, r in zip(lvl, res):
            ta, tb = nodes.pop(merges[k][0]), nodes.pop(merges[k][1])
            rp, cp = (tb, ta) if r["swapped"] else (ta, tb)
            s, c, _, _ = pyoracle.dp_construct(rp, cp, r["path"], g)
            nodes[n + k] = (s, c, ta[2] + tb[2])
            results[k] = r
    return assemble_rows(seqs, merges, results), int(results[-1]["total"])


def resident_progressive_alignment(engine, seqs, merges, gaps, score_matrix, on_level=None):
    """Level-synchronous progressive alignment with every profile resident on the GPU (famsa_prof_merge_batch):
    leaves come from the uploaded sequences, merged tables never leave HBM, the host receives one path per merge
    and applies its gap runs to the member rows (what FinalizeGaps does, profile.cpp:1053-1104).
    on_level(level_merge_indices, merged_ids, results) is called after each level, before the next consumes them.
    Returns ({seq_no: gapped string}, results per merge, root id)."""
    from famsa_b200 import seqio
    from famsa_b200.binding import PROF_LEAF
    from famsa_b200.schedule import ready_levels
    n = len(seqs)
    codes, off, lens = seqio.pack([seqio.encode(s) for s in seqs])
    engine.upload(codes, off, lens)
    engine.prof_set_scoring(score_matrix)
    node = {i: PROF_LEAF | i for i in range(n)}
    width = {i: len(seqs[i]) for i in range(n)}
    rows = {i: {i: np.frombuffer(seqs[i].encode(), dtype=np.uint8)} for i in range(n)}
    results = [None] * len(merges)
    for lvl in ready_levels(n, merges):
        pairs = [(node.pop(merges[k][0]), node.pop(merges[k][1])) for k in lvl]
        ids, res = engine.prof_merge_batch(pairs, gaps, [(width[merges[k][0]], width[merges[k][1]]) for k in lvl])
        for k, pid, r in zip(lvl, ids, res):
            a, b = merges[k]
            node[n + k] = pid
            width[n + k] = len(r["path"])
            ra, rb = rows.pop(a), rows.pop(b)
            rrows, crows = (rb, ra) if r["swapped"] else (ra, rb)
            out = {}
            for members, gapdir in ((rrows, 1), (crows, 2)):
                keep = r["path"] != gapdir
                for no, row in members.items():
                    g = np.full(len(r["path"]), ord("-"), dtype=np.uint8)
                    g[keep] = row
                    out[no] = g
            rows[n + k] = out
            results[k] = r
        if on_level:
            on_level(lvl, ids, res)
    root = n + len(merges) - 1
    return {no: row.tobytes().decode() for no, row in rows[root].items()}, results, node[root]


def assemble_rows(seqs, merges, results):
    """Final alignment {seq_no: gapped string} from the per-merge paths (what FinalizeGaps does on the host):
    H steps are gap columns in the members of the DP's row profile, V steps in those of the column profile."""
    n = len(seqs)
    rows = {i: {i: np.frombuffer(seqs[i].encode(), dtype=np.uint8)} for i in range(n)}
    for k, (a, b) in enumerate(merges):
        r = results[k]
        ra, rb = rows.pop(a), rows.pop(b)
        rrows, crows = (rb, ra) if r["swapped"] else (ra, rb)
        out = {}
        for members, gapdir in ((rrows, 1), (crows, 2)):
            keep = r["path"] != gapdir
            for no, row in members.items():
                g = np.full(len(r["path"]), ord("-"), dtype=np.uint8)
                g[keep] = row
                out[no] = g
        rows[n + k] = out
    return {no: row.tobytes().decode() for no, row in rows[n + len(merges) - 1].items()}


class OracleEngine:
    """CPU stand-in for Engine's resident-profile calls, built on the oracle (tests of the multi-rank host logic run
    without a GPU): same ids / leaf handles / consume-on-merge semantics as famsa_prof_*."""
    def __init__(self):
        self.tab = {}
        self.next = 0

    def upload(self, codes, off, lens):
        self.seqs = [np.asarray(codes[int(o):int(o) + int(l)]) for o, l in zip(off, lens)]

    def prof_set_scoring(self, sm):
        self.sm = np.asarray(sm, dtype=np.int64)

    def _tables(self, h, gaps):
        from famsa_b200 import profiles
        from famsa_b200.binding import PROF_LEAF
        if h & PROF_LEAF:
            return profiles.tables_from_rows(self.seqs[h & ~PROF_LEAF][None, :], self.sm, gaps)
        return self.tab.pop(h)

    def prof_merge_batch(self, pairs, gaps, widths):
        ids, out = [], []
        for a, b in pairs:
            ta, tb = self._tables(a, gaps), self._tables(b, gaps)
            r = pyoracle.dp_align(*ta, *tb, gaps)
            rp, cp = (tb, ta) if r["swapped"] else (ta, tb)
            s, c, _, _ = pyoracle.dp_construct(rp, cp, r["path"], gaps)
            self.tab[self.next] = (s, c, ta[2] + tb[2])
            ids.append(self.next); self.next += 1
            out.append(dict(path=r["path"], total=r["total"], last=r["last"], swapped=r["swapped"], variant=r["variant"]))
        return ids, out

    def prof_get(self, pid, tables=True):
        s, c, k = self.tab[pid]
        return (s, c, k) if tables else (s.shape[0] - 1, k)

    def prof_put(self, profs):
        ids = []
        for p in profs:
            self.tab[self.next] = p
            ids.append(self.next); self.next += 1
        return ids

    def prof_drop(self, ids):
        for i in ids:
            del self.tab[int(i)]
