"""GPU tests of the byte-level framer (csrc/frame.cu, rpl_frame_capsules_dev) against the oracle framing, which
tests/test_framing_vs_ref.py pins against the SDK's own unpacker on damaged streams."""
import numpy as np
import pytest

from test_capsule_oracle_vs_ref import unpacked_nodes
from test_decode_oracle_vs_ref import ref  # noqa: F401  (the fixture)
from test_framing_vs_ref import FORMATS, damaged_stream

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def R():
    import rplidar_ros2_driver_b200 as R

    return R


def run_framer(R, ctx, ans, streams):
    import torch

    dev = torch.device("cuda")
    cb = R.lib().rpl_capsule_bytes(ans)
    n_streams = len(streams)
    stride_bytes = max(max(len(s) for s in streams), 1)
    host = np.zeros((n_streams, stride_bytes), np.uint8)
    for i, s in enumerate(streams):
        host[i, : len(s)] = s
    counts_h = np.array([len(s) for s in streams], np.uint32)
    stride_caps = 2 * (stride_bytes // cb) + 2
    raw = torch.from_numpy(host).to(dev)
    counts = torch.from_numpy(counts_h.view(np.int32)).to(dev)
    caps = torch.full((n_streams, stride_caps, cb), 0xEE, dtype=torch.uint8, device=dev)
    ccount = torch.zeros(n_streams, dtype=torch.int32, device=dev)
    left = torch.zeros(n_streams, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()  # buffers were filled on torch's stream; the library runs on its own
    ctx.frame_capsules_dev(ans, raw.data_ptr(), counts.data_ptr(), n_streams, stride_bytes, caps.data_ptr(), stride_caps,
                           ccount.data_ptr(), bytes_left_out=left.data_ptr())
    ctx.synchronize()
    torch.cuda.synchronize()
    return caps, ccount, left, stride_caps


@pytest.mark.parametrize("ans", FORMATS)
def test_framer_matches_the_oracle_on_damaged_and_long_streams(R, oracle, ans):
    ctx = R.Context(0, 8192, 1)
    rng = np.random.default_rng(100 + ans)
    cb = oracle.capsule_bytes(ans)
    streams = [damaged_stream(oracle, ans, rng) for _ in range(40)]
    # several tiles, clean and damaged; damage exactly at tile boundaries (16384 bytes); degenerate streams
    long_clean = damaged_stream(oracle, ans, rng, ncap=900, max_edits=0)
    streams.append(long_clean)
    streams.append(damaged_stream(oracle, ans, rng, ncap=900, max_edits=25))
    for cut in (16384 - 1, 16384, 16384 + 1, 2 * 16384 - cb // 2):
        s = bytearray(long_clean.tobytes())
        del s[cut: cut + 3]
        streams.append(np.frombuffer(bytes(s), np.uint8))
    streams += [np.zeros(0, np.uint8), np.array([0xA1], np.uint8), np.full(40000, 0x33, np.uint8),
                np.tile(np.array([0xA0, 0x11], np.uint8), 9000), long_clean[: cb - 1], long_clean[: cb], long_clean[1:]]
    caps, ccount, left, stride_caps = run_framer(R, ctx, ans, streams)
    hc, hn, hl = caps.cpu().numpy(), ccount.cpu().numpy(), left.cpu().numpy()
    for i, s in enumerate(streams):
        exp, eleft = oracle.frame_capsules(ans, s)
        assert hn[i] == exp.shape[0], (hex(ans), i, hn[i], exp.shape[0])
        assert hl[i] == eleft, (hex(ans), i)
        assert (hc[i, : hn[i]] == exp).all(), (hex(ans), i)
        assert (hc[i, hn[i]:] == 0xEE).all()  # nothing written past the frames
    ctx.close()


@pytest.mark.parametrize("ans", FORMATS)
def test_raw_bytes_to_nodes_on_the_device_equals_the_sdk(R, ref, ans):
    """raw damaged bytes -> rpl_frame_capsules_dev -> rpl_decode_capsules_batch_dev, no host round trip, against the
    SDK's own unpacker fed the same bytes."""
    import torch

    oracle = ref
    ctx = R.Context(0, 8192, 1)
    rng = np.random.default_rng(500 + ans)
    streams = [damaged_stream(oracle, ans, rng, ncap=300, max_edits=8) for _ in range(16)]
    caps, ccount, left, stride_caps = run_framer(R, ctx, ans, streams)
    dev = torch.device("cuda")
    per = oracle.capsule_nodes(ans)
    nodes = torch.zeros((len(streams), stride_caps * per, 8), dtype=torch.uint8, device=dev)
    ncount = torch.zeros(len(streams), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()  # buffers were filled on torch's stream; the library runs on its own
    ctx.decode_capsules_batch_dev(ans, caps.data_ptr(), ccount.data_ptr(), len(streams), stride_caps, 31, nodes.data_ptr(),
                                  ncount.data_ptr())
    ctx.synchronize()
    torch.cuda.synchronize()
    hn, hc = nodes.cpu().numpy(), ncount.cpu().numpy()
    for i, s in enumerate(streams):
        unpacked_nodes(oracle, ans, s, 31, 0, np.ascontiguousarray(hn[i, : hc[i]]).view(oracle.NODE_DTYPE).reshape(-1))
    ctx.close()
