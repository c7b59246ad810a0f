"""The reference's answers that tests compare against, kept in tests/golden/reference_answers.npz.

Where oracle/_ref (the compiled, unmodified reference) is present, every answer is computed live and must equal the
stored copy; with FAMSA_RECORD_REFERENCE=<file.npz> set, the live answers are written there instead (copy the file to
tests/golden/reference_answers.npz to update the store).  Without oracle/_ref the stored answers are used, so each
comparison with the reference also runs on a machine that holds nothing but this repository.

Large answers are stored as CRC32 digests (crc()) rather than in full."""
from __future__ import annotations

import atexit
import os
import zlib

import numpy as np

from oracle import pyoracle

STORE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_answers.npz")
RECORD = os.environ.get("FAMSA_RECORD_REFERENCE")

_stored = None
_recorded: dict[str, np.ndarray] = {}


def crc(a) -> int:
    """CRC32 of an array's bytes (C order)."""
    return zlib.crc32(np.ascontiguousarray(a).tobytes())


def _store() -> dict:
    global _stored
    if _stored is None:
        _stored = dict(np.load(STORE)) if os.path.exists(STORE) else {}
    return _stored


def live() -> bool:
    return pyoracle.have_ref()


def answer(key: str, compute) -> np.ndarray:
    """The reference's answer for `key`: compute() where the reference is built (checked against the stored copy,
    or recorded), else the stored copy."""
    if live():
        v = np.asarray(compute())
        if RECORD:
            _recorded[key] = v
        elif key in _store():
            s = _store()[key]
            assert s.dtype == v.dtype and np.array_equal(s, v), f"stored reference answer {key!r} differs from the live reference"
        return v
    if key not in _store():
        raise AssertionError(f"no stored reference answer {key!r} in {STORE} and oracle/_ref is not built")
    return _store()[key]


def answer_crc(key: str, compute) -> int:
    """answer() for a large array, held as its CRC32."""
    return int(answer(key, lambda: np.array([crc(compute())], dtype=np.uint32))[0])


def input_key(*parts) -> str:
    """A stable key for a test input built from sequences, trees and parameters."""
    h = 0
    for p in parts:
        b = p.encode() if isinstance(p, str) else repr(p).encode() if not isinstance(p, np.ndarray) else p.tobytes()
        h = zlib.crc32(b, h)
    return f"{h:08x}"


@atexit.register
def _write():
    if RECORD and _recorded:
        old = dict(np.load(RECORD)) if os.path.exists(RECORD) else {}
        old.update(_recorded)
        np.savez_compressed(RECORD, **old)
