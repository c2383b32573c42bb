"""SURVEY.md 8(f) rank 4 -- per-sample timestamps.  Pins oracle/timestamp_oracle.cpp against the SDK's own
unpackers running on a settable clock (oracle/_ref/libref_clock.so: the SDK compiled without its
timer.cpp) and the scan-begin timestamp against the real ScanDataHolder; their outputs are also stored as
digests, see tests/reference_outputs.py.  CPU only."""
import numpy as np
import pytest

from test_capsule_oracle_vs_ref import make_capsules
from test_decode_oracle_vs_ref import make_stream, ref  # noqa: F401  (ref: the fixture)

TIMINGS = [(31, 0, 0, 0), (63, 256000, 17, 0), (125, 1000000, 0, 2), (476, 115200, 250, 0), (31, 460800, 5, 1)]


def timestamped_nodes(O, ans, stream, chunk, rx, t4, nodes, ts):
    """The SDK's unpacker on its settable clock must give `nodes` stamped `ts`."""
    O.reference.check("unpacker on a clock", (ans, stream, chunk, rx, t4), (nodes, ts),
                      lambda: O.ref_unpack_ts(ans, stream, chunk, rx, t4))


def rx_times(n, seed):
    rng = np.random.default_rng(seed)
    return (10_000_000 + np.cumsum(rng.integers(200, 3000, n))).astype(np.uint64)


@pytest.mark.parametrize("ans", [0x82, 0x83, 0x84, 0x85, 0x86])
@pytest.mark.parametrize("timing", TIMINGS)
def test_capsule_node_timestamps(ref, ans, timing):
    O = ref
    n = 160
    if ans == 0x85:
        caps = make_stream(O, n, 80.0, seed=3, sync_every=50)
    else:
        caps = make_capsules(O, ans, n, 45.0, seed=3, sync_every=50)
    caps[[20, 77], 30] ^= 0x04  # two checksum errors: the capsule after each releases nothing
    t4 = O.timing4(*timing)
    rx = rx_times(n, ans)
    nodes, status, offs, _ = O.decode_capsules(ans, caps, timing[0])
    ts = O.node_timestamps(ans, t4, rx, status, offs, len(nodes))
    timestamped_nodes(O, ans, caps.reshape(-1), O.capsule_bytes(ans), rx, t4, nodes, ts)
    assert len(nodes) > 0


@pytest.mark.parametrize("timing", TIMINGS)
def test_standard_node_timestamps(ref, timing):
    O = ref
    rng = np.random.default_rng(5)
    n = 900
    rec = np.zeros((n, 5), np.uint8)
    s = (np.arange(n) % 360 == 0).astype(np.uint8)
    rec[:, 0] = (rng.integers(0, 64, n).astype(np.uint8) << 2) | ((1 - s) << 1) | s
    w = (rng.integers(0, 360 * 64, n).astype(np.uint16) << 1) | 1
    rec[:, 1], rec[:, 2] = w & 0xFF, w >> 8
    rec[:, 3:] = rng.integers(0, 256, (n, 2))
    b = rec.reshape(-1).copy()
    b[rng.choice(len(b), 40, replace=False)] ^= 0xFF
    t4 = O.timing4(*timing)
    for chunk in (5, 64, 333):
        rx = rx_times((len(b) + chunk - 1) // chunk, chunk)
        nodes, ends, _ = O.decode_normal(b)
        ts = O.normal_timestamps(t4, ends, chunk, rx)
        timestamped_nodes(O, 0x81, b, chunk, rx, t4, nodes, ts)
        assert len(nodes) > 0


def test_scan_begin_timestamp_matches_the_reference_holder(ref):
    O = ref
    caps = make_stream(O, 700, 80.0, seed=8, sync_every=260)
    t4 = O.timing4(31, 0, 0, 0)
    rx = rx_times(700, 1)
    nodes, status, offs, _ = O.dense_decode(caps, 31, 0)
    ts = O.node_timestamps(0x85, t4, rx, status, offs, len(nodes))
    resets = O.resets_from_capsules(status, offs)
    e, elen, ek, ets = O.assemble_scans_ts(nodes, ts, resets, 8192, 16)

    def begins(scans, lens, k, sts):
        return k, lens[:k], sts[:k]

    O.reference.check("ScanDataHolder timestamps", (nodes, ts, resets, 8192, 16), begins(e, elen, ek, ets),
                      lambda: begins(*O.ref_assemble_scans_ts(nodes, ts, resets, 8192, 16)))
    assert ek >= 4
    starts = np.flatnonzero(nodes["flag"] & 1)
    assert set(ets[:ek].tolist()) <= set(ts[starts].tolist())
