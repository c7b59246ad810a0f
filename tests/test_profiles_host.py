"""famsa_b200.profiles (host mirror of CProfile::CalculateCounters/Scores) against the reference's tables."""
import numpy as np
import pytest

from famsa_b200 import profiles, seqio
from oracle import pyoracle

import refgold
from dp_cases import reference_gaps, reference_score_matrix


@pytest.mark.parametrize("card,width,seed", [(1, 30, 0), (6, 30, 1), (25, 60, 2), (40, 133, 3)])
def test_tables_match_reference(card, width, seed):
    rng = np.random.default_rng(seed)
    sm, g = reference_score_matrix(100), reference_gaps(100)
    rows = profiles.synth_alignment(card, width, rng, 0.4)
    if card > 3:
        rows[1, -7:] = -1
        rows[2, -1:] = -1
        rows[3, :5] = -1
    # CFAMSA::alignProfiles builds profiles through the string constructor, whose width is gapped_size - 1
    # (profile.cpp:334-337): add one trailing column and compare the first `width` ones.
    last = np.where(rows[:, -1] < 0, -1, 0).astype(np.int8)[:, None]
    last[0, 0] = 0
    rows2 = np.concatenate([rows, last], axis=1)
    strs = ["".join("-" if c < 0 else seqio.ALPHABET[c] for c in r) for r in rows2]
    s2, c2, k2 = profiles.tables_from_rows(rows2, sm, g)
    want = refgold.answer(f"profile_tables/{card}/{width}/{seed}/" + refgold.input_key(strs), lambda: _reference_tables(strs, card, width))
    assert want[0] == k2 == card
    assert want[1] == refgold.crc(c2[:width + 1]) and want[2] == refgold.crc(s2[:width + 1])


def _reference_tables(strs, card, width):
    """(card, CRC of the counters, CRC of the scores) of the first `width` columns of the reference's profile."""
    dp = pyoracle.RefDp(100)
    p = dp.profile(strs, list(range(card)))
    sc, cn, k = dp.tables(p)
    dp.free(p)
    dp.close()
    return np.array([k, refgold.crc(cn[:width + 1]), refgold.crc(sc[:width + 1])], dtype=np.int64)
