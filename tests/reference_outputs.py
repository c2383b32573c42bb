"""The reference's own outputs, kept in the repository as digests.

The *_vs_ref tests pin the restatement (oracle/) against the reference's own code, compiled from the original
sources into oracle/_ref by oracle/Makefile.  Those sources are not part of this repository, so every comparison
also goes through tests/golden/reference_digests.npz: for each reference call, a digest of its inputs maps to a
digest of what it returned.

  oracle/_ref built    the reference is called, its outputs must equal the restatement's bit for bit, and their
                       digest must equal the stored one (RPL_RECORD_REFERENCE=1 stores it instead)
  oracle/_ref absent   the restatement's outputs must have the stored digest

Digests are the first 8 bytes of SHA-256 over the shapes and raw bytes of the values.
"""
from __future__ import annotations

import hashlib
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.npz")


def _digest(kind: str, values) -> int:
    h = hashlib.sha256(kind.encode())
    for v in values:
        a = np.ascontiguousarray(np.asarray(v))
        h.update(repr(a.shape).encode())
        h.update(a.tobytes())
    return int.from_bytes(h.digest()[:8], "little")


class Reference:
    def __init__(self, oracle):
        self.live = oracle.have_ref() and oracle.have_ref_node() and oracle.have_ref_clock() and oracle.have_ref_holder()
        self.record = self.live and os.environ.get("RPL_RECORD_REFERENCE") == "1"
        self.stored = {}
        if os.path.exists(PATH):
            d = np.load(PATH)
            self.stored = dict(zip(d["inputs"].tolist(), d["outputs"].tolist()))

    def check(self, call: str, inputs, ours, live):
        """Asserts that the reference's `call` on `inputs` returns `ours` (a tuple of arrays and scalars, compared by
        shape and raw bytes).  `live()` makes the call itself; it runs only where oracle/_ref is built."""
        key = _digest(call, inputs)
        got = _digest("out", ours)
        if self.live:
            theirs = live()
            assert len(theirs) == len(ours), call
            for i, (a, b) in enumerate(zip(ours, theirs)):
                a, b = np.asarray(a), np.asarray(b)
                assert a.shape == b.shape and a.tobytes() == b.tobytes(), (call, i)
            if self.record:
                self.stored[key] = _digest("out", theirs)
                return
        assert key in self.stored, f"no stored output of the reference's {call} for these inputs"
        assert got == self.stored[key], f"differs from what the reference's {call} returned"

    def save(self):
        if self.record:
            keys = sorted(self.stored)
            np.savez_compressed(PATH, inputs=np.array(keys, np.uint64),
                                outputs=np.array([self.stored[k] for k in keys], np.uint64))
