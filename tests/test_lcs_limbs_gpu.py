"""Boundary tests of HP-1 (through the C ABI): every limb count the tile kernel k_lcs_tile<NL> is instantiated for, the
dropped-carry detector k_quirky and the limits of the exact kernels, against the integer restatement (oracle/) and, for
the dropped-carry corner, against the reference's own rows (stored answers without oracle/_ref).

A mask group is 32 sequences of the length-descending order; it runs with the limb class of its first (longest) member,
nl_for_len(len) in lcs.cu: ceil(len / 32) limbs up to 32, then rounded up to a multiple of 4 up to 64 (2048 aa); longer
groups leave every pair of theirs to the exact kernels."""
import numpy as np
import pytest

from famsa_b200 import seqio
from oracle import pyoracle

import refgold

pytestmark = pytest.mark.gpu

CLASSES = list(range(1, 33)) + list(range(36, 65, 4))      # the instantiated k_lcs_tile<NL>
RUN = 3                                                    # residue of the dropped-carry runs (D)


def nl_for_len(n: int) -> int:
    req = max(1, (n + 31) // 32)
    if req <= 32:
        return req
    return (req + 3) // 4 * 4 if req <= 64 else 0


def group_classes(lens) -> list[int]:
    s = sorted((int(x) for x in lens), reverse=True)
    return [nl_for_len(s[g]) for g in range(0, len(s), 32)]


def low_complexity(rng, length):
    """2-4 letters, ~3 % codes >= 20 (B Z X *, which never match): long carry chains across limbs and limb groups."""
    alpha = rng.choice(20, size=int(rng.integers(2, 5)), replace=False)
    c = alpha[rng.integers(0, len(alpha), length)].astype(np.int8)
    k = rng.random(length) < 0.03
    c[k] = rng.integers(20, 24, int(k.sum()))
    return c


def class_set(nl, rng):
    """39 sequences whose two mask-group heads sit at the two edges of class nl: 32 nl and 32 (previous class) + 1."""
    prev = CLASSES[CLASSES.index(nl) - 1] if nl > 1 else 0
    hi, lo = 32 * nl, 32 * prev + 1
    lens = [hi] + [int(x) for x in rng.integers(lo, hi + 1, 31)] + [lo] + [int(x) for x in rng.integers(1, lo + 1, 6)]
    cl = [low_complexity(rng, n) for n in lens]
    return [cl[i] for i in rng.permutation(len(cl))]


def test_class_sets_launch_every_limb_count():
    rng = np.random.default_rng(64)
    got = set()
    for nl in CLASSES:
        heads = group_classes([len(c) for c in class_set(nl, rng)])
        assert heads == [nl, nl], f"class {nl}: group heads land in {heads}"
        got |= set(heads)
    assert got == set(CLASSES) and len(CLASSES) == 40


def test_every_limb_class(engine):
    """For each of the 40 classes: triangle (2- and 4-byte output) and rows against the restatement."""
    rng = np.random.default_rng(64)
    for nl in CLASSES:
        cl = class_set(nl, rng)
        codes, off, lens = seqio.pack(cl)
        engine.upload(codes, off, lens)
        want = pyoracle.lcs_triangle(codes, off, lens)
        assert np.array_equal(engine.triangle(dtype=np.uint32), want), f"NL {nl}: triangle"
        assert np.array_equal(engine.triangle(dtype=np.uint16), want), f"NL {nl}: 16-bit triangle"
        refs = [int(np.argmax(lens)), int(np.argmin(lens)), 0, len(cl) - 1]
        assert np.array_equal(engine.rows(refs), pyoracle.lcs_rows(codes, off, lens, refs)), f"NL {nl}: rows"


def _run(rng, length, start, n, code=RUN):
    c = rng.integers(0, 20, length).astype(np.int8)
    c[c == code] = (code + 1) % 20                            # no stray RUN residues next to the run
    c[start:start + n] = code
    return c


def quirk_set():
    """{name: codes}: runs of 64 identical residues at word starts 0 / 64 / 128 (a dropped-carry word), the near misses
    (a 64-run at 65, a 63-run), a run that fills the last word exactly and one a residue short, 64-runs of non-matching
    codes (X, B), and partners rich in the run's residue."""
    rng = np.random.default_rng(127)
    s = {"run0": _run(rng, 200, 0, 64), "run64": _run(rng, 260, 64, 64), "run128": _run(rng, 300, 128, 64),
         "run65": _run(rng, 260, 65, 64), "run63": _run(rng, 260, 64, 63), "end128": _run(rng, 128, 64, 64),
         "end127": _run(rng, 127, 64, 63), "x64": _run(rng, 200, 0, 64, code=22), "b64": _run(rng, 200, 64, 64, code=20),
         "two": _run(rng, 330, 192, 64)}
    s["two"][0:64] = RUN
    s["all192"] = np.full(192, RUN, dtype=np.int8)
    s["all128"] = np.full(128, RUN, dtype=np.int8)
    s["all70"] = np.full(70, RUN, dtype=np.int8)
    s["mix"] = np.where(rng.random(300) < 0.5, RUN, rng.integers(0, 20, 300)).astype(np.int8)
    s["short"] = np.array([RUN], dtype=np.int8)
    s["plain"] = rng.integers(0, 20, 150).astype(np.int8)
    return s


QUIRKY = {"run0", "run64", "run128", "end128", "two", "all192", "all128", "all70"}


def _reference_rows(cl, rows):
    letters = [seqio.decode(c) for c in cl]
    rs = pyoracle.RefSeqSet(letters)
    out = np.stack([rs.row_ids(i, np.arange(len(cl))) for i in rows])
    rs.close()
    return out.astype(np.uint32)


def test_dropped_carry_detector(engine):
    """Every run shape as row (seq0) and as column of the reference's recurrence: rows of the full square and the
    triangle, against the restatement and the reference's own rows."""
    s = quirk_set()
    names = list(s)
    cl = [s[k] for k in names]
    codes, off, lens = seqio.pack(cl)
    n = len(cl)
    sq = pyoracle.lcs_rows(codes, off, lens, np.arange(n))
    ref = refgold.answer("lcs_limbs/quirk_square/" + refgold.input_key(*cl), lambda: _reference_rows(cl, range(n)))
    assert np.array_equal(sq, ref), "the restatement misreads the dropped-carry corner"
    # the corner is reached (a dropped carry makes the square asymmetric) and only from the rows that own such a word
    plain = [i for i, k in enumerate(names) if k not in QUIRKY]
    assert not np.array_equal(sq, sq.T)
    assert np.array_equal(sq[np.ix_(plain, plain)], sq[np.ix_(plain, plain)].T)
    engine.upload(codes, off, lens)
    assert np.array_equal(engine.rows(np.arange(n)), ref)
    i, j = np.tril_indices(n, -1)
    assert np.array_equal(engine.triangle(dtype=np.uint32), ref[i, j])
    for k in ("run64", "end128", "b64", "run65"):               # one row against a column list with repeats
        cols = np.array([names.index(x) for x in ("all192", "all128", k, "mix", "all192")], dtype=np.uint32)
        assert np.array_equal(engine.rows([names.index(k)], cols)[0], ref[names.index(k), cols])


def test_exact_kernel_boundaries(engine):
    """Quirky rows of 4096 aa (the batched register-form exact kernel) and 4097 aa (the global-memory one), 32 over-long
    sequences (2049 aa and up: exact kernels only, 2049 x 2049 among them) and a 2048-aa mask group head (NL 64) that the
    over-long ones stream against in the tile kernel."""
    rng = np.random.default_rng(4097)
    q4096, q4097 = low_complexity(rng, 4096), low_complexity(rng, 4097)
    q4096[1024:1088] = RUN
    q4097[4032:4096] = RUN
    long_ = [low_complexity(rng, n) for n in [2049, 2049] + [int(x) for x in rng.integers(2050, 2200, 28)]]
    rest = [low_complexity(rng, n) for n in (2048, 1500, 700, 64)]
    rest[0][:64] = RUN
    cl = [q4096, q4097] + long_ + rest
    cl = [cl[i] for i in rng.permutation(len(cl))]
    codes, off, lens = seqio.pack(cl)
    assert group_classes(lens) == [0, 64]
    n = len(cl)
    engine.upload(codes, off, lens)
    want = pyoracle.lcs_triangle(codes, off, lens)
    assert np.array_equal(engine.triangle(dtype=np.uint32), want)
    assert np.array_equal(engine.triangle(dtype=np.uint16), want)
    qi = [k for k in range(n) if len(cl[k]) in (4096, 4097, 2048)] + [int(np.argmin(lens))]
    got = engine.rows(qi)
    assert np.array_equal(got, pyoracle.lcs_rows(codes, off, lens, qi))
    ref = refgold.answer("lcs_limbs/exact_rows/" + refgold.input_key(*cl), lambda: _reference_rows(cl, qi))
    assert np.array_equal(got, ref)
