"""Boundary tests of HP-2 (through the C ABI): every arithmetic mode of the column-pair scores T, every launch shape of the
fill and the traceback far from the diagonal, each against the int64 C restatement (oracle/) and, where the tables come
from real gapped rows under the reference's scoring, against the reference's own Align (stored answers without oracle/_ref).

k_dp_prep picks per merge (dp.cu, DpMeta::tmode / t32):
  tmode 0  IMMA with 1-byte counter digits   ProfProf, scores in int32, row profile <= 127 members
  tmode 1  IMMA with 2-byte counter digits   ProfProf, scores in int32, row profile <= 32767 members
  tmode 2  scalar 32 x 64 multiply-adds      ProfProf with wider scores or more members; always for Seq*
  t32      4-byte T ring: max|column score| < 2^31 / (7 nR) for ProfProf, < 2^31 for Seq*
The case builder restates that rule on the host, asserts that every case lands in the cell it was built for and that the
set covers every reachable (variant, tmode, t32) cell, both orientations and the stripe / chunk / ring edges."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from dp_cases import reference_gaps, reference_score_matrix
from famsa_b200 import profiles, seqio
from oracle import pyoracle

import refgold

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
I32_MAX, I32_MIN = 2 ** 31 - 1, -2 ** 31
CARDS = (2, 127, 128, 129, 32767, 32768, 40000)           # row-profile cards around the digit-width limits of IMMA
ROW_EDGES = (1, 31, 32, 33, 63, 64, 65)                    # 32-row stripes
COL_EDGES = (1, 7, 8, 9, 39, 40, 41, 63, 64, 65, 127, 128, 129, 1500)   # 8-column chunks, steady state at chunk 5, 64-entry rings
WIDE = 300_000                                             # scales PFASUM-like scores past int32

# fill-kernel launch shapes: development knobs of dp.cu force each on ordinary merges
LAUNCH_ENVS = [{},
               {"FAMSA_DP_MAX_CELLS": "60000"},
               {"FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_CLUSTER_MIN": "40", "FAMSA_DP_TEAM_MIN": "32"},
               {"FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_TEAM_MIN": "100000"},
               {"FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_TEAM_WARPS": "2"},
               {"FAMSA_DP_LATENCY_MODE": "1", "FAMSA_DP_MAX_CLUSTER": "2"},
               {"FAMSA_DP_LATENCY_MODE": "1"},
               {"FAMSA_DP_LATENCY_MODE": "1", "FAMSA_DP_DUO": "0"},
               {"FAMSA_DP_LATENCY_MODE": "1", "FAMSA_DP_MAX_CLUSTER": "2", "FAMSA_DP_DUO": "0"},
               {"FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_TEAM_MIN": "32", "FAMSA_DP_COMPACT": "2"},
               {"FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_TEAM_MIN": "32", "FAMSA_DP_COMPACT": "2", "FAMSA_DP_TEAM_WARPS": "2"},
               {"FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_TEAM_MIN": "32", "FAMSA_DP_COMPACT": "2", "FAMSA_DP_TEAM_WARPS": "4"},
               {"FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_TEAM_MIN": "32", "FAMSA_DP_COMPACT": "2", "FAMSA_DP_TEAM_WARPS": "6"}]
KNOBS = sorted({k for e in LAUNCH_ENVS for k in e})


# ---------------------------------------------------------------------------------------------------- host rule
def expected_cell(job):
    """(variant, swapped, nR, tmode, t32) as k_dp_prep decides them (CProfile::Align's variant and orientation)."""
    s1, c1, k1, s2, c2, k2 = job
    w1, w2 = s1.shape[0] - 1, s2.shape[0] - 1
    if k1 == 1 and k2 == 1:
        var, sw = 0, False
    elif k1 == 1:
        var, sw = 1, False
    elif k2 == 1:
        var, sw = 1, True
    else:
        var = 2
        sw = not (int(np.count_nonzero(c1)) * w2 < int(np.count_nonzero(c2)) * w1)
    sc, nR = (s1, k2) if sw else (s2, k1)
    v = sc[1:, :30]
    smax = int(np.abs(v).max())
    wide = bool(((v < I32_MIN) | (v > I32_MAX)).any())
    if var != 2:
        return var, sw, nR, 2, smax < 2 ** 31
    tmode = 2 if wide else (0 if nR <= 127 else 1 if nR <= 32767 else 2)
    return var, sw, nR, tmode, smax < 2 ** 31 // (7 * nR)


def t32_bound(nR: int) -> int:
    """The smallest max|column score| whose ProfProf T no longer goes to the 4-byte ring."""
    return 2 ** 31 // (7 * nR)


REACHABLE = {(0, 2, True), (0, 2, False), (1, 2, True), (1, 2, False),
             (2, 0, True), (2, 0, False), (2, 1, True), (2, 1, False), (2, 2, True), (2, 2, False)}


# ---------------------------------------------------------------------------------------------------- inputs
def block(rng, card, width, diverse=False):
    """An aligned block (card, width + 1) int8, gaps < 0.  Low-diversity blocks (one alternative residue per column) have
    few non-zero counters per column, so that k_dp_prep makes them the row profile against a diverse one.  The extra last
    column is the one the reference's string constructor drops (profile width = gapped length - 1): its tables are cut
    to `width` columns, and the reference builds the same profile from the same strings."""
    cons = rng.integers(0, 20, width)
    if diverse:
        rows = np.where(rng.random((card, width)) < 0.6, rng.integers(0, 20, (card, width)), cons)
    else:
        rows = np.where(rng.random((card, width)) < 0.05, (cons + rng.integers(1, 20, width)) % 20, cons)
    rows = rows.astype(np.int8)
    if width >= 8:
        start, ln = rng.integers(0, width, card), rng.integers(1, 6, card)
        j = np.arange(width)
        gap = (j >= start[:, None]) & (j < (start + ln)[:, None]) & (rng.random(card) < 0.3)[:, None]
        rows[gap] = profiles.GAP
        empty = (rows < 0).all(axis=0)
        rows[0, empty] = cons[empty]
    last = np.where(rows[:, -1] < 0, profiles.GAP, 0).astype(np.int8)[:, None]
    last[0, 0] = 0
    return np.concatenate([rows, last], axis=1)


def seq(rng, length):
    return rng.integers(0, 20, length).astype(np.int8)


_tables = {}


def tables(x, sm, g):
    """Tables of a block (see block()) or of a sequence (1-D codes: a leaf); the 40 000-member blocks recur, so cached."""
    key = (id(x), id(sm), id(g))
    if key not in _tables:
        if x.ndim == 1:
            t = profiles.tables_from_rows(x[None, :], sm, g)
        else:
            s, c, k = profiles.tables_from_rows(x, sm, g)
            t = (s[:-1].copy(), c[:-1].copy(), k)
        _tables[key] = (x, sm, g, t)                        # (the keys' objects stay alive with the entry)
    return _tables[key][3]


def tables_crc(t) -> int:
    return refgold.crc(np.concatenate([t[0].ravel(), t[1].ravel().astype(np.int64), [t[2]]]))


def adversarial(s, pool):
    """Column scores (rows 0..29 of columns 1..W) drawn from `pool`; the counters stay those of a real alignment."""
    rng = np.random.default_rng(len(pool) * 7919 + s.shape[0])
    s = s.copy()
    s[1:, :30] = rng.choice(np.asarray(pool, dtype=np.int64), size=(s.shape[0] - 1, 30))
    return s


def edge_pool(nR, rng):
    """int32 edges, both sides of the 4-byte-ring bound of nR, and byte patterns that set every digit plane and the sign
    of the top digit (as signed int32)."""
    q = t32_bound(nR)
    pats = [0x7f7f7f7f, 0x80808080, 0x00ff00ff, 0xff00ff00, 0x01020304, 0xfffefdfc, 0x80000001, 0x7fffff80,
            0x000000ff, 0x0000ff00, 0x00ff0000, 0xff000000, 0xffffffff, 0x00000080, 0x00008000, 0x00800000]
    pats = [p - 2 ** 32 if p >= 2 ** 31 else p for p in pats]
    return [I32_MAX, I32_MIN, q, -q, q - 1, 1 - q, q + 1, -q - 1, 0, 1, -1] + pats + list(rng.integers(I32_MIN, I32_MAX, 16))


def under_pool(nR, rng):
    """Values strictly inside the 4-byte-ring bound of nR, including its edge and every byte below it."""
    q = t32_bound(nR) - 1
    b = [v for v in (0x7f, 0xff, 0x7fff, 0xffff, 0x7fffff, 0xffffff, 0x7f7f7f, 0x808080) if v <= q]
    return [q, -q, 0, 1, -1] + b + [-v for v in b] + list(rng.integers(-q, q + 1, 16))


class Case:
    def __init__(self, name, a, b, sm, g, want=None, pin=False, adv=None):
        """a, b: block or sequence of the two sides; want: the (variant, swapped, tmode, t32) the case is built for (None:
        any); pin: compare with the reference's own Align; adv = (side, pool): that side's scores drawn from pool."""
        t = [tables(a, sm, g), tables(b, sm, g)]
        if adv is not None:
            side, pool = adv
            t[side] = (adversarial(t[side][0], pool), t[side][1], t[side][2])
        self.name, self.src, self.pin = name, (a, b), pin
        self.job = (*t[0], *t[1])
        self.cell = expected_cell(self.job)
        if want is not None:
            got = (self.cell[0], self.cell[1], self.cell[3], self.cell[4])
            assert all(w is None or w == x for w, x in zip(want, got)), f"{name}: lands in {self.cell}, built for {want}"


def _letters(x):
    return "".join("-" if c < 0 else seqio.ALPHABET[c] for c in x)


def reference_answer(case, g):
    """The reference's Align on the case's inputs: [total, CRC of both input tables, path (row / column profile = side
    1 / side 2) as the merged rows give it].  Blocks go through the string constructor, sequences through the leaf
    constructor, as in CFAMSA."""
    def run():
        dp = pyoracle.RefDp(0)
        dp.set_gaps(g)
        ps, members, no = [], [], 0
        for x in case.src:
            if x.ndim == 1:
                ps.append(dp.leaf(_letters(x), no)); members.append({no}); no += 1
            else:
                ids = list(range(no, no + x.shape[0])); no += x.shape[0]
                ps.append(dp.profile([_letters(r) for r in x], ids)); members.append(set(ids))
        crcs = [tables_crc(dp.tables(p)) for p in ps]
        m, total = dp.align(ps[0], ps[1], 1)
        rows = dp.rows(m)
        dp.free(m)
        dp.close()
        # the rows of string-built members keep the dropped column at their end: cut it off (it pairs up as one last
        # D step when both sides are blocks)
        n = min(len(r) for r in rows.values()) - all(x.ndim == 2 for x in case.src)
        path = pyoracle.path_from_rows({k: r[:n] for k, r in rows.items()}, members[0], members[1], False)
        return np.concatenate([[total, *crcs], path]).astype(np.int64)
    return refgold.answer("dp_regimes/" + case.name + "/" + refgold.input_key(*case.src, [int(x) for x in g]), run)


def build_groups():
    """{group: (gaps, [Case])}.  One batch per group (the gap costs are per batch): "ref" mixes every variant, size class
    and 4- / 8-byte T under the reference's scoring; "wide", "tiny" and "loose" (near-zero gap costs) are the other
    score regimes."""
    rng = np.random.default_rng(2026)
    sm, g = reference_score_matrix(), reference_gaps(0)
    smw, gw = sm * WIDE, g * WIDE
    smt = rng.integers(-2, 2, size=(24, 24)); smt = (smt + smt.T) // 2; smt[np.arange(24), np.arange(24)] = 3
    gt = np.array([-3, -1, -2, -1], dtype=np.int64)
    gl = np.array([-40, -10, -5, -5], dtype=np.int64)
    big = block(rng, max(CARDS), 48)
    low = {k: big[:k] if k > 1000 else block(rng, k, int(rng.integers(40, 200))) for k in CARDS}
    div = block(rng, 12, 60, diverse=True)
    s_short, s_long = seq(rng, 45), seq(rng, 170)
    ref, wide, tiny, loose = [], [], [], []

    # score regimes x cards x variants / orientations
    for k in CARDS:
        tm = 0 if k <= 127 else 1 if k <= 32767 else 2
        q = t32_bound(k)
        ref.append(Case(f"pp{k}", low[k], div, sm, g, want=(2, False, tm, None), pin=True))
        ref.append(Case(f"pp{k}sw", div, low[k], sm, g, want=(2, True, tm, None), pin=True))
        wide.append(Case(f"pp{k}", low[k], div, smw, gw, want=(2, False, 2, False)))
        wide.append(Case(f"pp{k}sw", div, low[k], smw, gw, want=(2, True, 2, False)))
        tiny.append(Case(f"pp{k}", low[k], div, smt, gt, want=(2, False, tm, True)))
        tiny.append(Case(f"pp{k}sw", div, low[k], smt, gt, want=(2, True, tm, True)))
        ref.append(Case(f"pp{k}edge", low[k], div, sm, g, want=(2, False, tm, False), adv=(1, edge_pool(k, rng))))
        ref.append(Case(f"pp{k}under", low[k], div, sm, g, want=(2, False, tm, True), adv=(1, under_pool(k, rng))))
        ref.append(Case(f"pp{k}at", low[k], div, sm, g, want=(2, False, tm, False), adv=(1, under_pool(k, rng)[1:] + [q])))
        ref.append(Case(f"pp{k}edgesw", div, low[k], sm, g, want=(2, True, tm, False), adv=(0, edge_pool(k, rng))))
    for k in (2, 128, 40000):
        for lst, m_, g_, pin in ((ref, sm, g, True), (wide, smw, gw, False), (tiny, smt, gt, False)):
            lst.append(Case(f"sp{k}", s_short, low[k], m_, g_, want=(1, False, 2, None), pin=pin))
            lst.append(Case(f"sp{k}sw", low[k], s_short, m_, g_, want=(1, True, 2, None), pin=pin))
    for lst, m_, g_, pin in ((ref, sm, g, True), (wide, smw, gw, False), (tiny, smt, gt, False)):
        lst.append(Case("ss", s_short, s_long, m_, g_, want=(0, False, 2, None), pin=pin))
    # Seq* on the two sides of the 4-byte test: column scores of exactly 2^31 - 1 and -2^31
    for nm, pool, t in (("max", [I32_MAX, 0, -5, I32_MAX - 1], True), ("min", [I32_MIN, 7, I32_MAX], False)):
        ref.append(Case(f"seq_{nm}_1", s_short, low[129], sm, g, want=(1, False, 2, t), adv=(1, pool)))
        ref.append(Case(f"seq_{nm}_1sw", low[129], s_short, sm, g, want=(1, True, 2, t), adv=(0, pool)))
        ref.append(Case(f"seq_{nm}_0", s_short, s_long, sm, g, want=(0, False, 2, t), adv=(1, pool)))

    # stripe / chunk / ring edges (row profile = the low-diversity side), ProfProf in full, Seq* on a subset
    for r in ROW_EDGES:
        a = block(rng, 2, r)
        for c in COL_EDGES:
            ref.append(Case(f"shape_pp_{r}x{c}", a, block(rng, 6, c, diverse=True), sm, g, want=(2, False, 0, True), pin=True))
    for r in (1, 32, 33, 65):
        a = seq(rng, r)
        for c in (1, 8, 9, 40, 64, 129):
            ref.append(Case(f"shape_sp_{r}x{c}", a, block(rng, 3, c, diverse=True), sm, g, want=(1, False, 2, True), pin=True))
            ref.append(Case(f"shape_ss_{r}x{c}", a, seq(rng, c), sm, g, want=(0, False, 2, True), pin=True))
    ref.append(Case("shape_pp_700x5", block(rng, 2, 700), block(rng, 6, 5, diverse=True), sm, g, want=(2, False, 0, True), pin=True))
    ref.append(Case("shape_pp_20x3000", block(rng, 2, 20), block(rng, 6, 3000, diverse=True), sm, g, want=(2, False, 0, True), pin=True))

    # traceback far from the diagonal: long H / V runs across several stripes
    s = seq(rng, 400)
    pre = np.concatenate([seq(rng, 300), s])
    ref.append(Case("tb_prefix_rows", pre, s, sm, g, pin=True))
    ref.append(Case("tb_prefix_cols", s, pre, sm, g, pin=True))
    ref.append(Case("tb_ratio_rows", seq(rng, 600), seq(rng, 60), sm, g, pin=True))
    ref.append(Case("tb_ratio_cols", seq(rng, 60), seq(rng, 600), sm, g, pin=True))
    ref.append(Case("tb_ratio_pp", block(rng, 2, 500), block(rng, 5, 50, diverse=True), sm, g, pin=True))
    ref.append(Case("tb_ratio_pp_cols", block(rng, 2, 50), block(rng, 5, 500, diverse=True), sm, g, pin=True))
    loose.append(Case("tb_loose_ss", seq(rng, 200), seq(rng, 230), sm, gl))
    loose.append(Case("tb_loose_pp", block(rng, 3, 150), block(rng, 5, 170, diverse=True), sm, gl))
    loose.append(Case("tb_loose_prefix", pre, s, sm, gl))
    return {"ref": (g, ref), "wide": (gw, wide), "tiny": (gt, tiny), "loose": (gl, loose)}


@pytest.fixture(scope="module")
def groups():
    gr = build_groups()
    want = {}
    for name, (g, cases) in gr.items():
        for c in cases:
            o = pyoracle.dp_align(*c.job, g)
            assert (o["variant"], o["swapped"]) == c.cell[:2], f"{name}/{c.name}: the restatement orients it differently"
            ra = reference_answer(c, g) if c.pin else None
            if ra is not None:
                assert ra[1] == tables_crc(c.job[:3]) and ra[2] == tables_crc(c.job[3:]), f"{c.name}: tables differ from the reference's"
                assert o["total"] == ra[0], f"{name}/{c.name}: restatement total differs from the reference's"
                p = np.where(o["path"] == 0, 0, 3 - o["path"]) if o["swapped"] else o["path"]
                assert np.array_equal(p, ra[3:]), f"{name}/{c.name}: restatement path differs from the reference's"
            want[name, c.name] = (o, ra)
    return gr, want


def test_case_set_covers_every_regime(groups):
    """The matrix the generator has to cover: every reachable (variant, tmode, t32) cell, both orientations, every
    row-profile card, every stripe / chunk / ring edge."""
    gr, _ = groups
    cases = [c for _, cs in gr.values() for c in cs]
    assert {(c.cell[0], c.cell[3], c.cell[4]) for c in cases} == REACHABLE
    assert {(c.cell[0], c.cell[1]) for c in cases} == {(0, False), (1, False), (1, True), (2, False), (2, True)}
    assert {c.cell[2] for c in cases if c.cell[0] == 2} >= set(CARDS)
    assert {(c.cell[2], c.cell[1]) for c in cases if c.cell[0] == 2 and c.cell[3] == 2 and c.cell[4]} >= {(40000, False), (40000, True)}
    dims = {(c.job[3].shape[0] - 1, c.job[0].shape[0] - 1) if c.cell[1] else (c.job[0].shape[0] - 1, c.job[3].shape[0] - 1) for c in cases}
    assert {r for r, _ in dims} >= set(ROW_EDGES) | {700} and {w for _, w in dims} >= set(COL_EDGES) | {3000}
    ref_cells = {(c.cell[0], c.cell[3], c.cell[4]) for c in gr["ref"][1]}
    assert (2, 0, True) in ref_cells and (2, 0, False) in ref_cells, "the mixed batch must hold 4- and 8-byte T merges"
    assert sum(c.pin for c in cases) > 100


def _check(got, want, name, env, dirs=True):
    o, ra = want
    where = f"{name} under {env}"
    assert got["variant"] == o["variant"] and got["swapped"] == o["swapped"], where
    assert got["total"] == o["total"], where
    assert np.array_equal(got["last"], o["last"]), where
    assert np.array_equal(got["path"], o["path"]), where
    if dirs:
        assert np.array_equal(got["dirs"], o["dirs"]), where
    if ra is not None:
        p = np.asarray(got["path"], dtype=np.uint8)
        p = np.where(p == 0, 0, 3 - p).astype(np.uint8) if got["swapped"] else p
        assert got["total"] == ra[0] and np.array_equal(p, ra[3:]), f"{where}: differs from the reference's Align"


@pytest.mark.parametrize("env", LAUNCH_ENVS, ids=lambda e: ",".join(f"{k[9:]}={v}" for k, v in e.items()) or "default")
def test_regimes_in_every_launch_shape(engine, groups, monkeypatch, env):
    """All cases, one batch per score regime, with CDPMatrix output (k_dp_unskew), in every fill shape."""
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    gr, want = groups
    for name, (g, cases) in gr.items():
        got = engine.dp_align_batch([c.job for c in cases], g, want_dirs=True)
        for c, r in zip(cases, got):
            assert (r["variant"], r["swapped"]) == c.cell[:2], f"{name}/{c.name} did not land where it was built for"
            _check(r, want[name, c.name], f"{name}/{c.name}", env)


@pytest.mark.parametrize("team_warps", ["2", "4", "6"])
def test_mixed_batch_compact(engine, groups, monkeypatch, team_warps):
    """k_dp_fill_compact over a batch of 4- and 8-byte T merges: it must skip the 8-byte ones and the wide_only k_dp_fill
    launched behind it must do exactly those; Seq* / ProfProf merges of other classes run on the aux streams beside it."""
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    for k, v in {"FAMSA_DP_LATENCY_MODE": "0", "FAMSA_DP_TEAM_MIN": "32", "FAMSA_DP_COMPACT": "2", "FAMSA_DP_TEAM_WARPS": team_warps}.items():
        monkeypatch.setenv(k, v)
    gr, want = groups
    g, cases = gr["ref"]
    mixed = [c for c in cases if c.cell[0] == 2 and min(c.job[0].shape[0], c.job[3].shape[0]) > 33]
    assert {c.cell[4] for c in mixed} == {True, False}
    rng = np.random.default_rng(int(team_warps))
    order = list(rng.permutation(len(cases)))                # interleave 4- and 8-byte merges and the other variants
    got = engine.dp_align_batch([cases[i].job for i in order], g)
    for i, r in zip(order, got):
        _check(r, want["ref", cases[i].name], cases[i].name, team_warps, dirs=False)


@pytest.mark.parametrize("fused", ["0", "1"])
def test_resident_large_cards(engine, groups, monkeypatch, fused):
    """famsa_prof_put + famsa_prof_merge_batch on large cards with wide and adversarial scores (k_merge_fused with "1":
    every merge has <= 512 DP rows); totals, paths and the merged tables k_prof_construct builds against the restatement."""
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("FAMSA_PROF_FUSED", fused)
    gr, want = groups
    engine.prof_set_scoring(reference_score_matrix())
    picked = {"wide": ("pp32768", "pp40000sw", "pp129", "sp40000", "ss"),
              "ref": ("pp40000edge", "pp32767under", "pp128at", "pp40000", "pp32768sw", "seq_min_1", "sp128sw")}
    for name, names in picked.items():
        g, cases = gr[name]
        sel = [c for c in cases if c.name in names]
        assert len(sel) == len(names)
        ids = engine.prof_put([p for c in sel for p in (c.job[:3], c.job[3:])])
        merged, res = engine.prof_merge_batch([(ids[2 * i], ids[2 * i + 1]) for i in range(len(sel))], g,
                                              [(c.job[0].shape[0] - 1, c.job[3].shape[0] - 1) for c in sel])
        for c, mid, r in zip(sel, merged, res):
            o, ra = want[name, c.name]
            assert r["variant"] == o["variant"] and r["swapped"] == o["swapped"] and r["total"] == o["total"], c.name
            assert np.array_equal(r["path"], o["path"]), c.name
            rp, cp = (c.job[3:], c.job[:3]) if r["swapped"] else (c.job[:3], c.job[3:])
            ws, wc, _, _ = pyoracle.dp_construct(rp, cp, r["path"], g)
            s, cn, k = engine.prof_get(mid)
            assert k == c.job[2] + c.job[5] and np.array_equal(cn, wc) and np.array_equal(s, ws), f"{name}/{c.name}: merged tables"
        engine.prof_drop(merged)
    assert engine.prof_stats() == (0, 0)


_DEBUG_CHILD = r"""
import os, sys
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
import json
import numpy as np
import famsa_b200
from famsa_b200 import profiles
from test_dp_regimes_gpu import block, tables, LAUNCH_ENVS, KNOBS
rng = np.random.default_rng(5)
sm = profiles.synth_score_matrix(rng)
g = np.array([-14850, -1250, -660, -660], dtype=np.int64)
job = (*tables(block(rng, 3, 200), sm, g), *tables(block(rng, 8, 210, diverse=True), sm, g))
eng = famsa_b200.Engine(0)
for k, env in enumerate(LAUNCH_ENVS):
    for n in KNOBS:
        os.environ.pop(n, None)
    os.environ.update(env)
    print(f"@@env {k}", file=sys.stderr, flush=True)
    eng.dp_align_batch([job], g)
eng.close()
"""


def test_forced_shapes_really_run():
    """FAMSA_DP_DEBUG is latched once per process: one child with it set runs a 200 x 210 ProfProf merge (7 stripes) under
    every knob set, and its stderr names the fill class each launch used -- 0 one warp, 1 team (compact with
    FAMSA_DP_COMPACT=2), 2 throughput cluster, 10 + cl latency cluster, 100 + cl producer / consumer pairs."""
    env = {k: v for k, v in os.environ.items() if k not in KNOBS}
    env["FAMSA_DP_DEBUG"] = "1"
    p = subprocess.run([sys.executable, "-c", _DEBUG_CHILD, ROOT], env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    classes, cur = {}, None
    for line in p.stderr.splitlines():
        m = re.match(r"@@env (\d+)", line)
        if m:
            cur = int(m.group(1)); classes[cur] = []
        m = re.search(r"\[dp\] batch of \d+: class (\d+)", line)
        if m and cur is not None:
            classes[cur].append(int(m.group(1)))
    want = [[102], [102], [2], [0], [1], [102], [102], [12], [12], [1], [1], [1], [1]]
    assert [classes.get(k) for k in range(len(LAUNCH_ENVS))] == want, p.stderr[-3000:]
