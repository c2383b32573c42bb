"""Byte-level framing (the SDK's hunt for the capsule sync nibbles, reference
src/sdk/src/dataunpacker/unpacker/handler_capsules.cpp:107-135, 324-353, 639-668, 852-880) pinned against the
SDK's own unpacker: raw, DAMAGED byte streams (dropped, inserted and flipped bytes, false markers inside payloads,
truncated tails) -> oracle framing -> oracle capsule decoder must give the node stream LIDARSampleDataUnpacker
produces from the same bytes (the SDK's outputs are also stored as digests, see tests/reference_outputs.py).
tests/test_gpu_framing.py then holds the CUDA framer to the oracle framing."""
import numpy as np
import pytest

from test_capsule_oracle_vs_ref import unpacked_nodes
from test_decode_oracle_vs_ref import ref  # noqa: F401  (the fixture)

FORMATS = [0x82, 0x84, 0x85, 0x86]


def damaged_stream(O, ans, rng, ncap=160, max_edits=6):
    cb, per = O.capsule_bytes(ans), O.capsule_nodes(ans)
    payload = rng.integers(0, 256, (ncap, cb), dtype=np.uint8)
    step = 360.0 * per / 3200.0
    ang = (rng.uniform(0, 360) + np.arange(ncap) * step) % 360
    q6 = np.round(ang * 64).astype(np.uint32) % (360 * 64)
    sync = np.zeros(ncap, bool)
    sync[:: int(rng.integers(20, 60))] = True
    raw = bytearray(O.seal_capsules(ans, payload, q6, sync).reshape(-1).tobytes())
    for _ in range(int(rng.integers(0, max_edits + 1))):
        p = int(rng.integers(0, len(raw)))
        kind = int(rng.integers(0, 4))
        if kind == 0:
            del raw[p: p + int(rng.integers(1, 5))]
        elif kind == 1:
            raw[p:p] = bytes(rng.integers(0, 256, int(rng.integers(1, 200)), dtype=np.uint8))
        elif kind == 2:
            raw[p] ^= int(rng.integers(1, 256))
        else:  # a false marker pair in the middle of the stream
            raw[p:p] = bytes([0xA0 | int(rng.integers(0, 16)), 0x50 | int(rng.integers(0, 16))])
    if rng.random() < 0.5:
        del raw[len(raw) - int(rng.integers(0, cb)):]
    return np.frombuffer(bytes(raw), np.uint8)


@pytest.mark.parametrize("ans", FORMATS)
def test_framing_plus_decode_equals_the_sdk_unpacker_on_damaged_streams(ref, ans):
    oracle = ref
    rng = np.random.default_rng(ans)
    damaged = 0
    for trial in range(60):
        raw = damaged_stream(oracle, ans, rng)
        framed, left = oracle.frame_capsules(ans, raw)
        en, es, _, _ = oracle.decode_capsules(ans, framed, 31)
        unpacked_nodes(oracle, ans, raw, 31, 0, en)
        damaged += int(((es & oracle.CAPSULE_BAD_FRAME) != 0).any())
        assert left < oracle.capsule_bytes(ans)
    assert damaged > 10  # the resynchronisation was exercised


@pytest.mark.parametrize("ans", FORMATS)
def test_framing_of_a_clean_stream_is_the_identity(oracle, ans):
    rng = np.random.default_rng(1)
    raw = damaged_stream(oracle, ans, rng, ncap=50, max_edits=0)
    cb = oracle.capsule_bytes(ans)
    framed, left = oracle.frame_capsules(ans, raw)
    whole = len(raw) // cb
    assert framed.shape[0] == whole and left == len(raw) - whole * cb
    assert (framed.reshape(-1) == raw[: whole * cb]).all()


def test_garbage_only_and_empty_streams(oracle):
    for ans in FORMATS:
        f, left = oracle.frame_capsules(ans, np.zeros(0, np.uint8))
        assert f.shape[0] == 0 and left == 0
        f, left = oracle.frame_capsules(ans, np.full(1000, 0x11, np.uint8))
        assert f.shape[0] == 0 and left == 0
        f, left = oracle.frame_capsules(ans, np.array([0xA3], np.uint8))
        assert f.shape[0] == 0 and left == 1
