"""SURVEY.md 8(f) rank 1 -- dense-capsule decode.  Pins the restatement (oracle/decode_oracle.cpp)
against the SDK's OWN LIDARSampleDataUnpacker compiled in place (oracle/_ref; its outputs are also stored as
digests, see tests/reference_outputs.py): node for node and event for event (scan resets, checksum errors,
encoder-reset errors), including byte streams fed in odd chunk sizes.  CPU only."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def ref(oracle, reference):
    # the helpers here and in the other *_vs_ref modules are handed the oracle module and reach the reference
    # outputs through it
    oracle.reference = reference
    return oracle


class RefState:
    """The reference keeps lastNodeSyncBit in a function-static: it survives across streams in
    one process.  Track it so the restatement can be started from the same state."""
    value = 0


def make_stream(O, n_caps, caps_per_rev=80.0, seed=0, start_deg=0.0, p_zero=0.05, sync_every=None):
    rng = np.random.default_rng(seed)
    ang = (start_deg + np.arange(n_caps) * 360.0 / caps_per_rev + rng.normal(0, 0.03, n_caps)) % 360.0
    q6 = np.round(ang * 64).astype(np.uint32) % (360 * 64)
    sync = np.zeros(n_caps, bool)
    if sync_every:
        sync[::sync_every] = True
    dist = rng.integers(1, 65536, (n_caps, 40))
    dist[rng.random((n_caps, 40)) < p_zero] = 0
    return O.make_dense_capsules(q6, sync, dist)


def expected_events(O, status, offs):
    ev = []
    for st, off in zip(status.tolist(), offs.tolist()):
        if st & O.CAPSULE_CHECKSUM_ERR:
            ev.append((2, off, 0x8002))
        if st & O.CAPSULE_SYNC:
            if st & O.CAPSULE_ENCODER_RESET_ERR:
                ev.append((2, off, 0x8001))
            ev.append((1, off, 0))
    return np.array(ev, dtype=np.uint32).reshape(-1, 3)


def check(O, caps, sample_us=31, chunk=84):
    state = RefState.value
    nodes, status, offs, RefState.value = O.dense_decode(caps, sample_us, state)
    O.reference.check("dense capsule unpacker", (caps, sample_us, chunk, state), (nodes, expected_events(O, status, offs)),
                      lambda: O.ref_dense_decode(caps.reshape(-1), sample_us, chunk))
    return nodes, status


@pytest.mark.parametrize("caps_per_rev", [80.0, 20.0, 81.3, 7.0])
def test_clean_revolutions(ref, caps_per_rev):
    nodes, status = check(ref, make_stream(ref, 400, caps_per_rev, seed=int(caps_per_rev)))
    assert (status[1:] & ref.CAPSULE_EMIT).all() or caps_per_rev < 10  # big angular steps get discarded
    # every revolution raises exactly one scan-start flag
    if caps_per_rev >= 20:
        assert abs(int((nodes["flag"] & 1).sum()) - int(400 / caps_per_rev)) <= 1


def test_sync_capsules_checksum_errors_and_jumps(ref):
    rng = np.random.default_rng(5)
    caps = make_stream(ref, 600, 80.0, seed=1, sync_every=80)
    bad = rng.choice(600, 25, replace=False)
    caps[bad, 10] ^= 0x40  # payload corruption -> checksum error
    caps[200:204, 2] ^= 0xFF  # start-angle corruption is a checksum error too
    jump = make_stream(ref, 50, 80.0, seed=2, start_deg=123.0)  # angular jump in the middle
    allc = np.concatenate([caps[:300], jump, caps[300:]])
    nodes, status = check(ref, allc)
    assert ((status & ref.CAPSULE_CHECKSUM_ERR) != 0).sum() >= 25
    assert ((status & ref.CAPSULE_SYNC) != 0).sum() >= 4
    assert ((status & ref.CAPSULE_DISCARD) != 0).sum() >= 1


@pytest.mark.parametrize("chunk", [1, 7, 83, 84, 85, 1000])
def test_byte_stream_chunking_does_not_matter(ref, chunk):
    check(ref, make_stream(ref, 120, 80.0, seed=chunk, sync_every=40), chunk=chunk)


@pytest.mark.parametrize("sample_us", [31, 63, 125, 476])
def test_sample_duration_sets_the_jump_threshold(ref, sample_us):
    # slower sampling -> larger allowed angular step per capsule
    for cpr in (80.0, 12.0, 5.0):
        check(ref, make_stream(ref, 200, cpr, seed=sample_us), sample_us=sample_us)


def test_sync_bit_alternation_state_carries_over(ref):
    """Tiny angular increments make the raw sync test fire on many consecutive nodes; the
    reference's `(sync ^ last) & sync` then alternates, and the last value leaks into the next
    stream through the function-static."""
    q6 = (np.arange(300) % 3).astype(np.uint32)  # start angles 0, 1/64, 2/64 deg, ... wrapping
    caps = ref.make_dense_capsules(q6, np.zeros(300, bool), np.full((300, 40), 1234))
    nodes, _ = check(ref, caps)
    assert 0 < int((nodes["flag"] & 1).sum()) < len(nodes)
    check(ref, make_stream(ref, 100, 80.0, seed=9))  # starts from whatever state was left


def test_random_streams(ref):
    rng = np.random.default_rng(77)
    for t in range(40):
        n = int(rng.integers(1, 300))
        caps = make_stream(ref, n, float(rng.uniform(4, 200)), seed=1000 + t,
                           sync_every=int(rng.integers(5, 100)) if t % 2 else None)
        for j in rng.choice(n, max(1, n // 20), replace=False):
            caps[j, int(rng.integers(2, 84))] ^= int(rng.integers(1, 256))
        check(ref, caps, sample_us=int(rng.choice([31, 63, 125])))


# ---- scan assembly (8(f) rank 2): restatement vs the reference's real ScanDataHolder ----------------
def _scans(res):
    s, lens, k = res
    return (k, lens) + tuple(s[i, : lens[i]] for i in range(min(k, len(lens))))


def _same_scans(O, nodes, resets, max_nodes, max_scans):
    O.reference.check("ScanDataHolder", (nodes, resets, max_nodes, max_scans),
                      _scans(O.assemble_scans(nodes, resets, max_nodes, max_scans)),
                      lambda: _scans(O.ref_assemble_scans(nodes, resets, max_nodes, max_scans)))


def test_scan_assembly_matches_reference_holder(ref):
    rng = np.random.default_rng(3)
    for t in range(30):
        caps = make_stream(ref, int(rng.integers(50, 900)), float(rng.uniform(20, 200)), seed=500 + t,
                           sync_every=(int(rng.integers(30, 300)) if t % 3 == 0 else None))
        nodes, status, offs, _ = ref.dense_decode(caps, 31, 0)
        resets = ref.resets_from_capsules(status, offs)
        for max_nodes in (8192, 500):
            _same_scans(ref, nodes, resets, max_nodes, 64)
    # hand-made corner cases: nothing before the first scan start, resets at and between starts, cap
    mk = ref.make_nodes
    flags = np.array([2, 2, 1, 2, 2, 1, 2, 1, 1, 2, 2, 2, 1, 2], np.uint8)
    nodes = mk(np.arange(len(flags)) * 100, np.arange(len(flags)) + 5, 7, flags)
    for resets in ([], [0], [2], [3], [5], [6, 7], [8], [12], [13], [3, 9, 12]):
        r = np.array(resets, np.uint32)
        for max_nodes in (8192, 2, 1):
            _same_scans(ref, nodes, r, max_nodes, 16)
