"""CPU tests: the oracle (oracle/lcs_oracle.c) against the reference's golden vectors and against
the reference itself (oracle/_ref), so that the GPU parity tests stand on a pinned checker."""
import numpy as np
import pytest

from conftest import QUIRK_LCS, QUIRK_SEQS, random_set
from famsa_b200 import seqio
from oracle import pyoracle

import refgold


def test_oracle_matches_golden_pid_sq(adeno):
    """Every one of the 242 x 242 exact LCS lengths pinned by test/adeno_fiber/pid_sq.csv."""
    n = len(adeno["lens"])
    got = pyoracle.lcs_rows(adeno["codes"], adeno["offsets"], adeno["lens"], np.arange(n))
    assert np.array_equal(got, adeno["lcs"])


def test_oracle_triangle_layout(adeno):
    n = len(adeno["lens"])
    tri = pyoracle.lcs_triangle(adeno["codes"], adeno["offsets"], adeno["lens"])
    i, j = np.tril_indices(n, -1)
    assert np.array_equal(tri[i * (i - 1) // 2 + j], adeno["lcs"][i, j])
    part = pyoracle.lcs_triangle(adeno["codes"], adeno["offsets"], adeno["lens"], 100, 150)
    base = 100 * 99 // 2
    assert np.array_equal(part, tri[base:150 * 149 // 2])


def test_oracle_carry_quirk_vector():
    """SURVEY.md section 7 known-answer vector: the reference drops a carry when tB == ~0 and a
    carry arrives, so LCS is NOT symmetric here (row 1 reports 2 where the true LCS is 1)."""
    codes, offsets, lens = seqio.pack([seqio.encode(s) for s in QUIRK_SEQS])
    got = pyoracle.lcs_rows(codes, offsets, lens, np.arange(4))
    assert np.array_equal(got, QUIRK_LCS)


def test_oracle_distance_golden(adeno):
    """dist_sq.csv = LCS -> indel075_div_lcs in float -> 6-decimal print."""
    n = len(adeno["lens"])
    lens = adeno["lens"]
    for i in range(0, n, 7):
        for j in range(0, n, 5):
            if i == j:
                continue
            d = pyoracle.transform(0, int(adeno["lcs"][i, j]), int(lens[i]), int(lens[j]), double=False)
            assert abs(d - adeno["dist"][i, j]) < 1e-6 * max(1.0, abs(d)) + 6e-7


@pytest.mark.parametrize("isa", [0, 2])
def test_oracle_vs_reference_random(isa):
    rng = np.random.default_rng(5)
    code_list = random_set(rng, 70, 0, 300)
    code_list += random_set(rng, 10, 1, 40, alphabet=2)              # low complexity
    code_list.append(np.zeros(200, np.int8))                          # quirky: 'A' * 200
    code_list.append(np.concatenate([np.zeros(64, np.int8), np.ones(70, np.int8)]))
    letters = [seqio.decode(c) for c in code_list]
    rs = pyoracle.RefSeqSet(letters) if refgold.live() else None
    key = f"lcs_random/{isa}/" + refgold.input_key(letters)
    codes, offsets, lens = seqio.pack(code_list)
    assert refgold.crc(codes) == refgold.answer_crc(key + "/codes", lambda: np.concatenate(rs.codes()))
    n = len(code_list)
    want = refgold.answer(key + "/rows", lambda: np.stack([rs.row_prefix(r, n, isa) for r in range(n)]).astype(np.uint16))
    for r in range(n):
        got = pyoracle.lcs_rows(codes, offsets, lens, [r])[0]
        assert np.array_equal(got, want[r]), f"row {r}"
    ids = rng.permutation(n)[:37]
    want = refgold.answer(key + "/ids", lambda: rs.row_ids(3, ids, isa).astype(np.uint16))
    assert np.array_equal(want, pyoracle.lcs_rows(codes, offsets, lens, [3], ids)[0])


def test_reference_reproduces_golden(adeno):
    """The compiled reference (AVX2 path) reproduces its own pid_sq.csv through the harness (without oracle/_ref: the
    reference's stored answers do)."""
    rs = pyoracle.RefSeqSet(adeno["seqs"]) if refgold.live() else None
    n = len(adeno["lens"])
    rows = refgold.answer("adeno/rows_every_9th", lambda: np.stack([rs.row_prefix(r, n, 2) for r in range(0, n, 9)]).astype(np.uint16))
    assert np.array_equal(rows, adeno["lcs"][0:n:9])
    i, j = np.tril_indices(n, -1)
    want = adeno["lcs"][i, j].astype(np.uint32)

    def triangle():
        sec, pairs, tri = rs.triangle_mt(0, n, 4, 2, want_lcs=True)
        assert pairs == n * (n - 1) // 2
        return tri
    assert refgold.crc(want) == refgold.answer_crc("adeno/triangle", triangle)


def test_transform_vs_reference():
    rng = np.random.default_rng(1)
    args = []
    for _ in range(300):
        l1, l2 = (int(x) for x in rng.integers(1, 600, size=2))
        lcs = int(rng.integers(0, min(l1, l2) + 1))
        args += [(kind, lcs, l1, l2) for kind in (0, 1, 2)]

    def reference(f64):
        lib = pyoracle.ref()
        f = lib.ref_transform_f64 if f64 else lib.ref_transform_f32
        return np.array([f(*a) for a in args], dtype=np.float64 if f64 else np.float32)
    want64 = refgold.answer("transform/f64", lambda: reference(True))
    want32 = refgold.answer("transform/f32", lambda: reference(False))
    for a, w64, w32 in zip(args, want64, want32):
        assert pyoracle.transform(*a, True) == w64
        assert pyoracle.transform(*a, False) == w32
