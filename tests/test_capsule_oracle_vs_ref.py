"""SURVEY.md 8(f) rank 1, the other answer formats -- pins oracle/capsule_oracle.cpp against the SDK's
OWN LIDARSampleDataUnpacker compiled in place (oracle/_ref; its outputs are also stored as digests, see
tests/reference_outputs.py): express (0x82), HQ (0x83), ultra (0x84) and ultra-dense (0x86) capsules and the
5-byte standard nodes (0x81), node for node and event for event, with random payload bits so that every field is
exercised.  CPU only."""
import numpy as np
import pytest

from test_decode_oracle_vs_ref import expected_events, ref  # noqa: F401  (ref: the fixture)


def unpacked_nodes(O, ans, stream, sample_us, chunk, ours):
    """The nodes the SDK's unpacker makes of a raw byte stream must be `ours`."""
    O.reference.check("unpacker nodes", (ans, stream, sample_us, chunk), (ours,),
                      lambda: (O.ref_unpack(ans, stream, sample_us, chunk)[0],))


def make_capsules(O, ans, n, caps_per_rev=60.0, seed=0, sync_every=None, near=False):
    """Random payload, plausible start angles (so that the angle interpolation sees normal steps)."""
    rng = np.random.default_rng(seed)
    cb = O.capsule_bytes(ans)
    payload = rng.integers(0, 256, (n, cb), dtype=np.uint8)
    if ans == O.ANS_ULTRA_DENSE and near:
        # scale-0 samples a few counts apart: exercises the _last_dist_q2 smoothing chain
        base = rng.integers(50, 900, n)[:, None] * 4 + rng.integers(-2, 3, (n, 64)) * 4
        v = (base.astype(np.uint32) & 0xFFC) | (rng.integers(0, 16, (n, 64)).astype(np.uint32) << 12)
        v[rng.random((n, 64)) < 0.1] |= np.uint32(rng.integers(1, 4))  # some other scales in between
        cab = payload[:, 10:].reshape(n, 32, 5)
        cab[:, :, 0] = v[:, 0::2] & 0xFF
        cab[:, :, 1] = v[:, 0::2] >> 8
        cab[:, :, 2] = v[:, 1::2] & 0xFF
        cab[:, :, 3] = v[:, 1::2] >> 8
        payload[:, 10:] = cab.reshape(n, 160)
    if ans == O.ANS_HQ:
        return O.seal_capsules(ans, payload)
    ang = (np.arange(n) * 360.0 / caps_per_rev + rng.normal(0, 0.05, n)) % 360.0
    q6 = np.round(ang * 64).astype(np.uint32) % (360 * 64)
    sync = np.zeros(n, bool)
    if sync_every:
        sync[::sync_every] = True
    return O.seal_capsules(ans, payload, q6, sync)


def check(O, ans, caps, sample_us=31, chunk=0, state=(0, 0)):
    nodes, status, offs, out_state = O.decode_capsules(ans, caps, sample_us, state)
    O.reference.check("unpacker", (ans, caps, sample_us, chunk, state), (nodes, expected_events(O, status, offs)),
                      lambda: O.ref_unpack(ans, caps.reshape(-1), sample_us, chunk))
    return nodes, status


CAPSULE_FORMATS = [0x82, 0x83, 0x84, 0x86]


@pytest.mark.parametrize("ans", CAPSULE_FORMATS)
@pytest.mark.parametrize("caps_per_rev", [60.0, 11.3, 200.0])
def test_clean_streams(ref, ans, caps_per_rev):
    nodes, status = check(ref, ans, make_capsules(ref, ans, 300, caps_per_rev, seed=ans))
    assert len(nodes) > 0 and ((status & ref.CAPSULE_OK) != 0).all()


@pytest.mark.parametrize("ans", CAPSULE_FORMATS)
def test_errors_scan_starts_and_chunked_feeding(ref, ans):
    rng = np.random.default_rng(ans)
    caps = make_capsules(ref, ans, 500, 45.0, seed=100 + ans, sync_every=45)
    bad = rng.choice(500, 30, replace=False)
    caps[bad, 20] ^= 0x08  # payload bit flips: checksum / CRC errors
    for chunk in (0, 1, 7, 1000):
        _, status = check(ref, ans, caps, chunk=chunk)
    assert ((status & ref.CAPSULE_CHECKSUM_ERR) != 0).sum() == 30
    if ans != 0x83:
        assert ((status & ref.CAPSULE_SYNC) != 0).sum() >= 8
        assert ((status & ref.CAPSULE_ENCODER_RESET_ERR) != 0).sum() >= 4


def test_ultra_dense_smoothing_chain_and_jump_threshold(ref):
    for seed in range(6):
        caps = make_capsules(ref, 0x86, 300, 50.0, seed=seed, near=True)
        nodes, _ = check(ref, 0x86, caps)
        assert len(nodes) > 0
    for sample_us in (15, 31, 63, 125):
        for cpr in (50.0, 9.0, 4.0):
            check(ref, 0x86, make_capsules(ref, 0x86, 200, cpr, seed=sample_us), sample_us=sample_us)


def test_ultra_special_predict_codes_and_zero_majors(ref):
    """predict fields 0x200 / 0x1FF mean "no sample"; a zero major borrows the next cabin's base."""
    O = ref
    rng = np.random.default_rng(4)
    n = 200
    caps = make_capsules(O, 0x84, n, 60.0, seed=9)
    words = caps[:, 4:].copy().view("<u4").reshape(n, 32)
    pick = rng.random((n, 32))
    words[pick < 0.15] &= ~np.uint32(0xFFF)  # major = 0
    words[(pick > 0.2) & (pick < 0.3)] = (words[(pick > 0.2) & (pick < 0.3)] & ~np.uint32(0x3FF << 12)) | (0x200 << 12)
    words[(pick > 0.3) & (pick < 0.4)] = (words[(pick > 0.3) & (pick < 0.4)] & ~np.uint32(0x3FF << 22)) | (0x1FF << 22)
    small = (pick > 0.5) & (pick < 0.7)  # short distances: the angle-offset polynomial branch
    words[small] = (words[small] & ~np.uint32(0xFFF)) | rng.integers(1, 200, small.sum()).astype(np.uint32)
    caps[:, 4:] = words.view(np.uint8).reshape(n, 128)
    caps = O.seal_capsules(0x84, caps)
    nodes, _ = check(O, 0x84, caps)
    assert (nodes["dist_mm_q2"] == 0).any()


def test_standard_nodes_with_byte_level_resync(ref):
    O = ref
    rng = np.random.default_rng(11)
    n = 4000
    rec = np.zeros((n, 5), np.uint8)
    s = (rng.random(n) < 0.01).astype(np.uint8)
    rec[:, 0] = (rng.integers(0, 64, n).astype(np.uint8) << 2) | ((1 - s) << 1) | s
    ang = rng.integers(0, 360 * 64, n).astype(np.uint16)
    w = (ang << 1) | 1
    rec[:, 1], rec[:, 2] = w & 0xFF, w >> 8
    rec[:, 3:] = rng.integers(0, 256, (n, 2))
    clean = rec.reshape(-1)
    nodes, ends, pos = O.decode_normal(clean)
    unpacked_nodes(O, 0x81, clean, 476, 0, nodes)
    assert len(nodes) == n and pos == 0 and (ends == np.arange(n) * 5 + 4).all()
    # garbage: inserted / dropped / corrupted bytes make the state machine hunt for the next record
    for seed in range(8):
        r = np.random.default_rng(seed)
        b = clean.copy()
        b[r.choice(len(b), 200, replace=False)] = r.integers(0, 256, 200)
        b = np.delete(b, r.choice(len(b), 50, replace=False))
        b = np.insert(b, np.sort(r.choice(len(b), 50, replace=False)), r.integers(0, 256, 50).astype(np.uint8))
        nodes, _, _ = O.decode_normal(b)
        unpacked_nodes(O, 0x81, b, 476, int(r.integers(0, 9)), nodes)
        assert 0 < len(nodes) < n
    # pure noise
    b = rng.integers(0, 256, 20000, dtype=np.uint8)
    nodes, _, _ = O.decode_normal(b)
    unpacked_nodes(O, 0x81, b, 476, 0, nodes)
