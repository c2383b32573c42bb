"""GPU tests (-m gpu) of the entry points the chain, the exchange and the ROS overlay call, at their edges:
rpl_scan_views_dev over hand-made views, the single-scan calls (rpl_scan / rpl_laserscan / rpl_ascend_scan) across the
context sizes that switch their staging, the host-buffer batch wrappers, the chain's context limit, and empty or
overflowing batches in the cloud fuse, the peer push and the exchange.  The reference is the CPU oracle
(oracle.pipeline_batch with the stable tie rule, oracle.cloud); ranges, intensities, angle increments and nodes are
compared bit for bit.

Every device buffer here is a slice of a larger allocation whose padding, like every output, starts out as a sentinel
(node buffers carry n_scans * stride + 16 nodes of it past what nodes_total declares): a call that reads outside its
input or writes outside its output shows up as a mismatch, not as a fault."""
import ctypes as C

import numpy as np
import pytest

from helpers import bits
from test_decode_oracle_vs_ref import make_stream
from test_gpu_scan_parity import ALL_MODES, oracle_batch

pytestmark = pytest.mark.gpu

SENT_NODE = 0xA5A5A5A5A5A5A5A5  # a measured node (key 0xA5A5): read by mistake, it changes the result
SENT_OUT_NODE = 0x5A5A5A5A5A5A5A5A
SENT_F = 0x7FBADBAD  # a NaN no kernel produces
SENT_U = 0xDEADBEEF
INVALID = 0x80008000
FOUR_MODES = [(0, 0, 0), (1, 1, 0), (0, 1, 1), (1, 0, 1)]


@pytest.fixture(scope="module")
def R():
    import rplidar_ros2_driver_b200 as R

    return R


class Dev:
    """A device copy of `host` (uint32 or uint64 elements) followed by `pad` elements of `fill`."""

    def __init__(self, host, fill, pad):
        import torch

        flat = np.ascontiguousarray(host).reshape(-1)
        self.fill = flat.dtype.type(fill)
        whole = np.concatenate([flat, np.full(pad, self.fill, flat.dtype)])
        self.t = torch.from_numpy(whole.view(np.uint8)).to("cuda")
        self.t0 = self.t.clone()
        self.n, self.shape, self.dtype = flat.size, np.shape(host), flat.dtype

    @property
    def ptr(self):
        return self.t.data_ptr()

    def reset(self):
        self.t.copy_(self.t0)

    def get(self):
        """The live part; asserts that the padding behind it kept its sentinel."""
        w = self.t.cpu().numpy().view(self.dtype)
        assert (w[self.n:] == self.fill).all(), "written past the end of the buffer"
        return w[: self.n].reshape(self.shape)


def out(shape, fill, pad=64):
    dt = np.uint64 if fill in (SENT_NODE, SENT_OUT_NODE) else np.uint32
    return Dev(np.full(shape, fill, dt), fill, pad)


def on_device(ctx, fn):
    """The library works on its own stream: torch's copies must be done before, its work after."""
    import torch

    torch.cuda.synchronize()
    fn()
    ctx.synchronize()


def assert_rows(got, exp, what, views=None):
    bad = np.flatnonzero((np.asarray(got) != np.asarray(exp)).reshape(len(got), -1).any(axis=1))
    where = views[bad[:4]].tolist() if views is not None else ""
    assert bad.size == 0, f"{what}: {bad.size} rows differ, first {bad[:4].tolist()} {where}"


# ---- A. rpl_scan_views_dev ------------------------------------------------------------------------------------------
VS = 1000  # stride of the view batches: every count <= VS is a valid scan


@pytest.fixture(scope="module")
def vctx(R):
    c = R.Context(0, 8192, 4096)
    yield c
    c.close()


@pytest.fixture(scope="module")
def n_views():
    """More views than either kernel has CTAs: at most max_threads_per_SM / 256 shared-memory CTAs per SM."""
    import torch

    p = torch.cuda.get_device_properties(0)
    return getattr(p, "max_threads_per_multi_processor", 2048) // 256 * p.multi_processor_count + 40


def view_layout(oracle, content, total_parity, n_views, seed):
    """A node buffer of 12 revolutions of VS nodes (nodes_total = 12 * VS - total_parity) and n_views views into it:
    hand-made edges first, then random ones.  content: synth variant, or "wrap" (variant 0 with the last node of
    every revolution on its first node's key)."""
    rng = np.random.default_rng(seed)
    revs = oracle.synth_batch(seed, 12, VS, 0 if content == "wrap" else content)
    if content == "wrap":
        revs["dist_mm_q2"][:, [0, -1]] = np.maximum(revs["dist_mm_q2"][:, [0, -1]], 4000)
        revs["angle_z_q14"][:, -1] = revs["angle_z_q14"][:, 0]
    flat = revs.reshape(-1)
    hole = 5 * VS + 100
    flat["dist_mm_q2"][hole: hole + 10] = 0  # nothing measured here
    T = 12 * VS - total_parity
    S = VS
    hand = [
        (0, 0), (T, 0),                             # empty views, one at the very end of the buffer
        (2, 1), (3, 1), (hole, 1),                  # one node: even / odd first, unmeasured
        (10, 333), (11, 333), (12, 334), (13, 334),  # odd and even counts from even and odd firsts
        (4, S), (5, S), (S, S), (S, S),             # count == stride; two identical views
        (S + 500, S),                               # overlapping the previous two
        (2 * S, S), (6 * S, S),                     # whole revolutions ("wrap": first and last node share a key)
        (8 * S + 7, 640), (3 * S + 1, 640),         # reverse order, with a gap between
        (hole, 10), (hole + 1, 9),                  # nothing measured: ascend fails, buffer passes through
        (0, S + 1), (7, S + 1),                     # count above the stride: INVALID_DATA
        (T - 333, 333), (T - 999, 999),             # odd count ending exactly at nodes_total: an even first (odd T)
        (T - S, S), (T - 1, 1), (T - 334, 334),     # is staged with loads, an odd first (even T) by a bulk copy
        (T - 332, 333), (T, 1),                     # one node past nodes_total: INVALID_DATA
    ]
    views = np.zeros((n_views, 2), np.uint32)
    views[: len(hand)] = hand
    k = n_views - len(hand)
    counts = rng.integers(0, S + 1, k)
    counts[::7] = rng.integers(0, 8, len(counts[::7]))
    views[len(hand):, 1] = counts
    views[len(hand):, 0] = rng.integers(0, T - counts + 1)
    return flat.view(np.uint64).copy(), views, T


def view_runs(R, ctx, nodes_d, T, views_d, views, g_d, cb_d, prm, kind, ov, ob):
    n = len(views)
    for o in list(ov.values()) + list(ob.values()):
        o.reset()
    emit, scan = kind == "emit", kind in ("emit", "ranges")

    def args(o):
        return dict(nodes_out=o["nodes"].ptr if emit else None, ranges=o["ranges"].ptr if scan else None,
                    intensities=o["intens"].ptr if scan else None, beam_counts=o["beams"].ptr,
                    angle_increment=o["inc"].ptr, status=o["status"].ptr, path=o["path"].ptr)

    on_device(ctx, lambda: ctx.scan_views_dev(nodes_d.ptr, T, views_d.ptr, n, VS, prm, **args(ov)))
    on_device(ctx, lambda: ctx.scan_batch_dev(g_d.ptr, cb_d.ptr, n, VS, prm, **args(ob)))
    return {k: v.get() for k, v in ov.items()}, {k: v.get() for k, v in ob.items()}


@pytest.mark.parametrize("total_parity", [1, 0])
@pytest.mark.parametrize("content", [0, 2, 3, "wrap"])
def test_scan_views_against_the_oracle_and_the_batch_call(R, oracle, vctx, n_views, content, total_parity):
    """Every output of a view batch equals the oracle on the gathered [n_scans][stride] copy and equals
    rpl_scan_batch_dev on that copy; nothing past a scan's live part changes.  Views with a count above the stride or
    past nodes_total are INVALID_DATA rows with nothing else written."""
    seed = 4000 + 10 * total_parity + (7 if content == "wrap" else content)
    nodes, views, T = view_layout(oracle, content, total_parity, n_views, seed)
    n = len(views)
    first, cnt = views[:, 0].astype(np.int64), views[:, 1].astype(np.int64)
    valid = (cnt <= VS) & (first + cnt <= T)
    past = (cnt <= VS) & (first + cnt > T)
    assert past.sum() == 2 and (cnt > VS).sum() == 2
    g = np.full((n, VS), SENT_NODE, np.uint64)
    for s in np.flatnonzero(valid):
        g[s, : cnt[s]] = nodes[first[s]: first[s] + cnt[s]]
    cb = np.where(past, 0, cnt).astype(np.uint32)      # the batch call reports count > stride the same way
    c_or = np.where(valid, cnt, 0).astype(np.uint32)
    pad = n * VS + 16
    nodes_d = Dev(nodes[:T], SENT_NODE, len(nodes) - T + pad)
    views_d, g_d, cb_d = Dev(views, SENT_U, 64), Dev(g, SENT_NODE, pad), Dev(cb, SENT_U, 64)

    def outputs():
        return dict(nodes=out((n, VS), SENT_OUT_NODE, VS + 16), ranges=out((n, VS), SENT_F, VS + 16),
                    intens=out((n, VS), SENT_F, VS + 16), beams=out(n, SENT_U), inc=out(n, SENT_F),
                    status=out(n, SENT_U), path=out(n, SENT_U))

    ov, ob = outputs(), outputs()
    lane = np.arange(VS)[None, :]
    cache = {}
    for flags in (0, R.FLAG_FORCE_GENERAL):
        for mode in ALL_MODES:
            for kind, ascend in (("emit", 1), ("ranges", 0), ("status", 1)):
                if (mode, ascend) not in cache:
                    cache[mode, ascend] = oracle_batch(oracle, g.view(oracle.NODE_DTYPE), c_or, *mode, ascend)
                exp = cache[mode, ascend]
                tag = (content, total_parity, flags, mode, kind)
                got, ref = view_runs(R, vctx, nodes_d, T, views_d, views, g_d, cb_d,
                                     R.scan_params(*mode, ascend, flags), kind, ov, ob)
                m = np.where(valid, exp["beam_counts"], 0)
                assert_rows(got["beams"], m, ("beam counts", tag), views)
                assert_rows(got["inc"], np.where(valid, bits(exp["angle_increment"]), 0), ("angle increment", tag), views)
                assert_rows(got["status"], np.where(valid, exp["status"], INVALID), ("status", tag), views)
                if kind != "status":
                    live = lane < m[:, None]
                    assert_rows(got["ranges"], np.where(live, bits(exp["ranges"]), SENT_F), ("ranges", tag), views)
                    assert_rows(got["intens"], np.where(live, bits(exp["intensities"]), SENT_F), ("intensities", tag),
                                views)
                else:
                    assert (got["ranges"] == SENT_F).all() and (got["intens"] == SENT_F).all(), tag
                if kind == "emit":
                    live = lane < np.where(valid, cnt, 0)[:, None]
                    assert_rows(got["nodes"], np.where(live, exp["nodes"].view(np.uint64), SENT_OUT_NODE),
                                ("ascended nodes", tag), views)
                else:
                    assert (got["nodes"] == SENT_OUT_NODE).all(), tag
                for k in got:
                    assert_rows(got[k][~past], ref[k][~past], (k, "view batch vs batch call", tag), views[~past])


def test_scan_views_rejects_bad_calls_without_writing(R, oracle, vctx):
    """nodes_out without apply_ascend (the pass-through would copy [n_scans][stride] nodes from the buffer's start
    instead of the views), stride above 8192, RPL_FLAG_NO_SMALL and a node buffer that is not 16-byte aligned are
    rejected with RplError before anything is enqueued."""
    n, S = 40, VS
    nodes = oracle.synth_batch(77, n, S, 0).view(np.uint64).reshape(-1)
    T = n * S - 3
    wide = 8193
    nodes_d = Dev(nodes[:T], SENT_NODE, 3 + n * wide + 16)
    views = np.stack([np.arange(n) * (S - 3), np.full(n, S - 40)], axis=1).astype(np.uint32)
    views_d = Dev(views, SENT_U, 64)
    o = dict(nodes=out((n, wide), SENT_OUT_NODE), ranges=out((n, wide), SENT_F), intens=out((n, wide), SENT_F),
             beams=out(n, SENT_U), inc=out(n, SENT_F), status=out(n, SENT_U), path=out(n, SENT_U))
    cases = [
        ("nodes_out without apply_ascend", nodes_d.ptr, S, R.scan_params(0, 0, 0, 0), True),
        ("stride above 8192", nodes_d.ptr, wide, R.scan_params(0, 0, 0, 1), True),
        ("RPL_FLAG_NO_SMALL", nodes_d.ptr, S, R.scan_params(0, 1, 0, 1, R.FLAG_NO_SMALL), False),
        ("node buffer not 16-byte aligned", nodes_d.ptr + 8, S, R.scan_params(0, 1, 0, 1), True),
    ]
    for what, base, stride, prm, emit in cases:
        for v in o.values():
            v.reset()
        with pytest.raises(R.RplError):
            on_device(vctx, lambda: vctx.scan_views_dev(
                base, T - 1, views_d.ptr, n, stride, prm, nodes_out=o["nodes"].ptr if emit else None,
                ranges=o["ranges"].ptr, intensities=o["intens"].ptr, beam_counts=o["beams"].ptr,
                angle_increment=o["inc"].ptr, status=o["status"].ptr, path=o["path"].ptr))
        vctx.synchronize()
        for k, v in o.items():
            assert (v.get() == v.fill).all(), (what, k)


# ---- B. the single-scan calls ---------------------------------------------------------------------------------------
SIZES = [1, 2, 3, 359, 360, 4095, 8191, 8192, 32767, 32768, 65536, 70000]


def _ptr(a, t=None):
    return a.ctypes.data_as(C.POINTER(t)) if t is not None else C.c_void_p(a.ctypes.data)


def single(ctx, fn, nodes, prm=None):
    """One rpl_scan / rpl_laserscan / rpl_ascend_scan on a copy of `nodes` (uint64) with sentinel outputs."""
    L, h = ctx._L, ctx._h
    buf = nodes.copy()
    n = len(buf)
    r, it = np.full(n + 16, SENT_F, np.uint32), np.full(n + 16, SENT_F, np.uint32)
    b, inc, st = np.full(1, SENT_U, np.uint32), np.full(1, SENT_F, np.uint32), np.full(1, SENT_U, np.uint32)
    fb, fi = _ptr(b, C.c_uint32), _ptr(inc.view(np.float32), C.c_float)
    if fn == "scan":
        rc = L.rpl_scan(h, _ptr(buf), n, C.byref(prm), _ptr(r), _ptr(it), fb, fi, _ptr(st, C.c_uint32))
    elif fn == "laserscan":
        rc = L.rpl_laserscan(h, _ptr(buf), n, C.byref(prm), _ptr(r), _ptr(it), fb, fi)
    else:
        rc = L.rpl_ascend_scan(h, _ptr(buf), n)
    return dict(rc=int(rc), nodes=buf, ranges=r, intens=it, beams=int(b[0]), inc=int(inc[0]), status=int(st[0]))


def check_single(R, oracle, ctx, nodes, mode, ascend, tag):
    """rpl_scan with (mode, ascend), rpl_laserscan with mode and, when ascend, rpl_ascend_scan: against a [1, n] oracle
    batch.  Returns the raw results (for comparisons between contexts)."""
    n = len(nodes)
    expect = {a: oracle_batch(oracle, nodes.view(oracle.NODE_DTYPE)[None], np.array([n], np.uint32), *mode, a)
              for a in {0, ascend}}
    res = []
    for fn in ("scan", "laserscan") + (("ascend",) if ascend else ()):
        got = single(ctx, fn, nodes, R.scan_params(*mode, ascend))
        res.append(got)
        t = (fn,) + tag
        exp = expect[0 if fn == "laserscan" else ascend]  # rpl_laserscan: the LaserScan of the nodes as they are
        if fn == "ascend":
            assert got["rc"] == int(exp["status"][0]), t
            assert (got["nodes"] == exp["nodes"][0].view(np.uint64)).all(), t
            continue
        m = int(exp["beam_counts"][0])
        tail = np.full(n + 16 - m, SENT_F, np.uint32)
        assert got["rc"] == R.RESULT_OK, (t, hex(got["rc"]))
        assert got["beams"] == m, t
        assert got["inc"] == int(bits(exp["angle_increment"])[0]), t
        assert (got["ranges"][:m] == bits(exp["ranges"][0, :m])).all(), t
        assert (got["intens"][:m] == bits(exp["intensities"][0, :m])).all(), t
        assert (got["ranges"][m:] == tail).all() and (got["intens"][m:] == tail).all(), t
        if fn == "scan":
            assert got["status"] == (int(exp["status"][0]) if ascend else R.RESULT_OK), t
            assert (got["nodes"] == exp["nodes"][0].view(np.uint64)).all(), t
        else:
            assert (got["nodes"] == nodes).all(), t
    return res


@pytest.mark.parametrize("variant", [0, 2, 3])
@pytest.mark.parametrize("max_nodes", [360, 8192, 70000])
def test_single_scan_calls_across_context_sizes(R, oracle, max_nodes, variant):
    """Both H2D stagings (one copy when the scan nearly fills the context, else two), both D2H copies (one piece or
    split), the TMA / fast kernel on one CTA and the fallback to the general kernel (ties: variant 2).  Then a scan one
    node longer than the context: INVALID_DATA, and the caller's arrays untouched."""
    ctx = R.Context(0, max_nodes, 4)
    try:
        for n in [s for s in SIZES if s <= max_nodes]:
            nodes = oracle.synth_batch(6000 + 7 * n + variant, 1, n, variant)[0].view(np.uint64)
            for mode in (ALL_MODES if n in (360, 8192) else FOUR_MODES):
                for ascend in (0, 1):
                    check_single(R, oracle, ctx, nodes, mode, ascend, (max_nodes, variant, n, mode))
        big = oracle.synth_batch(99, 1, max_nodes + 1, variant)[0].view(np.uint64)
        for fn in ("scan", "laserscan", "ascend"):
            got = single(ctx, fn, big, R.scan_params(0, 1, 0, 1))
            assert got["rc"] == INVALID, (fn, hex(got["rc"]))
            assert (got["nodes"] == big).all(), fn
            assert (got["ranges"] == SENT_F).all() and (got["intens"] == SENT_F).all(), fn
    finally:
        ctx.close()


def test_single_scan_calls_ignore_the_previous_call(R, oracle):
    """One context, sizes shrinking and growing across odd and even: the staging keeps the previous revolution's nodes
    (rotated copies of one revolution: their keys collide with the current ones) and its outputs.  Every result
    equals the result of a fresh context and the oracle."""
    base = oracle.synth_batch(31337, 1, 8192, 0)[0].view(np.uint64)
    ctx = R.Context(0, 8192, 4)
    try:
        for k, n in enumerate((8191, 7, 8192, 1, 4097, 2, 8191, 3, 6000)):
            nodes = np.roll(base, 997 * k)[:n].copy()
            mode, ascend = ALL_MODES[k % 8], (k + 1) % 2
            tag = ("stale", k, n)
            got = check_single(R, oracle, ctx, nodes, mode, ascend, tag)
            fresh = R.Context(0, 8192, 4)
            try:
                again = check_single(R, oracle, fresh, nodes, mode, ascend, tag)
            finally:
                fresh.close()
            for a, b in zip(got, again):
                for key in a:
                    assert np.array_equal(a[key], b[key]), (tag, key)
    finally:
        ctx.close()


def test_host_batch_wrappers_over_both_lanes(R, oracle):
    """rpl_ascend_scan_batch (in place: nodes_out == nodes) and rpl_laserscan_batch on a batch of three staging
    chunks (about 32 MiB of nodes each), ragged counts with live nodes behind them, against the oracle."""
    n_scans, S = 2100, 4096
    ctx = R.Context(0, S, n_scans)
    try:
        rng = np.random.default_rng(8)
        nodes = np.concatenate([oracle.synth_batch(800 + v, n_scans // 3, S, v) for v in (0, 2, 3)])
        counts = rng.integers(0, S + 1, n_scans).astype(np.uint32)
        counts[:4] = (0, 1, S, S - 1)
        nodes[5]["dist_mm_q2"][:] = 0
        L, h = ctx._L, ctx._h
        buf = nodes.copy()
        st = np.full(n_scans, SENT_U, np.uint32)
        assert L.rpl_ascend_scan_batch(h, _ptr(buf), _ptr(counts), n_scans, S, _ptr(st)) == R.RESULT_OK
        exp = oracle_batch(oracle, nodes, counts, 0, 0, 0, 1)
        assert (st == exp["status"]).all()
        assert_rows(buf.view(np.uint64), exp["nodes"].view(np.uint64), "ascended in place")
        for mode in ((0, 1, 0), (1, 0, 1)):
            r, it = np.full((n_scans, S), SENT_F, np.uint32), np.full((n_scans, S), SENT_F, np.uint32)
            b, inc = np.full(n_scans, SENT_U, np.uint32), np.full(n_scans, SENT_F, np.uint32)
            before = nodes.copy()
            assert L.rpl_laserscan_batch(h, _ptr(nodes), _ptr(counts), n_scans, S, C.byref(R.scan_params(*mode, 1)),
                                         _ptr(r), _ptr(it), _ptr(b), _ptr(inc)) == R.RESULT_OK
            assert (nodes.view(np.uint64) == before.view(np.uint64)).all()
            exp = oracle_batch(oracle, nodes, counts, *mode, 0)
            assert (b == exp["beam_counts"]).all() and (inc == bits(exp["angle_increment"])).all(), mode
            live = np.arange(S)[None, :] < exp["beam_counts"][:, None]
            assert_rows(np.where(live, r, 0), np.where(live, bits(exp["ranges"]), 0), ("ranges", mode))
            assert_rows(np.where(live, it, 0), np.where(live, bits(exp["intensities"]), 0), ("intensities", mode))
    finally:
        ctx.close()


# ---- C. the chain's context limit -----------------------------------------------------------------------------------
def test_chain_rejects_max_nodes_above_the_context(R, oracle):
    """Revolutions of about 3200 nodes, the chain asked for max_nodes 4096 on a context made for 2048: the scan
    kernels would mark every revolution INVALID_DATA in a status the chain does not return, so the call must fail
    and leave the outputs alone."""
    ctx = R.Context(0, 2048, 64)
    try:
        n_streams, n_caps, max_nodes, max_scans = 4, 400, 4096, 8
        host = np.stack([make_stream(oracle, n_caps, 80.0, seed=700 + s) for s in range(n_streams)])
        ns = n_streams * max_scans
        o = dict(ranges=np.full((ns, max_nodes), SENT_F, np.uint32).view(np.float32),
                 intensities=np.full((ns, max_nodes), SENT_F, np.uint32).view(np.float32),
                 beam_counts=np.full(ns, SENT_U, np.uint32), angle_increment=np.full(ns, SENT_F, np.uint32).view(np.float32),
                 scans_per_stream=np.full(n_streams, SENT_U, np.uint32))
        with pytest.raises(R.RplError):
            ctx.chain_dense_laserscan(host, np.full(n_streams, n_caps, np.uint32), R.scan_params(1, 0, 0, 1), max_nodes,
                                      max_scans, out=o)
        for k, v in o.items():
            assert (v.view(np.uint32) == (SENT_F if v.dtype == np.float32 else SENT_U)).all(), k
    finally:
        ctx.close()


# ---- D. empty and overflowing batches in fuse, push and exchange (one GPU) ------------------------------------------
CS = 3200
CLOUD_KW = dict(range_min=0.15, range_max=40.0, voxel_size=0.05)


@pytest.fixture(scope="module")
def cctx(R):
    c = R.Context(0, CS, 64)
    yield c
    c.close()


def clouds(R, oracle, ctx, nodes, counts):
    """Per-scan clouds on the device (padded buffers) and the oracle's concatenation of them."""
    n = len(counts)
    nodes_d = Dev(nodes.view(np.uint64), SENT_NODE, n * CS + 16)
    counts_d = Dev(np.asarray(counts, np.uint32), SENT_U, 64)
    xyzi, pc = out((n, CS, 4), SENT_F, CS * 4), out(n, SENT_U)
    on_device(ctx, lambda: ctx.cloud_batch_dev(nodes_d.ptr, counts_d.ptr, n, CS, R.cloud_params(**CLOUD_KW), xyzi.ptr,
                                               pc.ptr))
    per = [oracle.cloud(nodes[s, : counts[s]], oracle.cloud_params(**CLOUD_KW)) for s in range(n)]
    assert (pc.get() == [len(p) for p in per]).all()
    exp = np.concatenate(per) if per else np.zeros((0, 4), np.float32)
    return xyzi, pc, per, exp


class _View:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2}


def read_device(ptr, shape, typestr):
    import torch

    return torch.as_tensor(_View(ptr, shape, typestr), device="cuda").cpu().numpy()


def test_cloud_fuse_empty_batch_and_empty_scans(R, oracle, cctx):
    """n_scans == 0 sets total to 0 (it was 0xDEADBEEF) and writes nothing else; a batch whose scans have no points
    (count 0, nothing measured, everything outside the window) packs the concatenation of the oracle's clouds."""
    xyzi0, pc0 = out((1, CS, 4), SENT_F), out(1, SENT_U)
    fused, offs, total = out((CS, 4), SENT_F), out(4, SENT_U), out(1, SENT_U)
    on_device(cctx, lambda: cctx.cloud_fuse_dev(xyzi0.ptr, pc0.ptr, 0, CS, fused.ptr, offs.ptr, total.ptr))
    assert int(total.get()[0]) == 0
    assert (offs.get() == SENT_U).all() and (fused.get() == SENT_F).all()

    nodes = oracle.synth_batch(4242, 7, CS, 4)
    counts = np.array([CS, 0, CS, 1, CS, 17, CS], np.uint32)
    nodes[2]["dist_mm_q2"][:] = 0                  # nothing measured
    nodes[4]["dist_mm_q2"][:] = 200000             # everything beyond range_max
    nodes[5]["dist_mm_q2"][:] = 0
    xyzi, pc, per, exp = clouds(R, oracle, cctx, nodes, counts)
    n_pts = np.array([len(p) for p in per])
    assert (n_pts[[1, 2, 4, 5]] == 0).all() and (n_pts[[0, 6]] > 0).all()
    fused, offs, total = out((7 * CS, 4), SENT_F, 64), out(7, SENT_U), out(1, SENT_U)
    on_device(cctx, lambda: cctx.cloud_fuse_dev(xyzi.ptr, pc.ptr, 7, CS, fused.ptr, offs.ptr, total.ptr))
    assert int(total.get()[0]) == len(exp)
    assert (offs.get() == np.concatenate([[0], np.cumsum(n_pts)[:-1]])).all()
    f = fused.get()
    assert (f[: len(exp)] == exp.view(np.uint32)).all() and (f[len(exp):] == SENT_F).all()


def test_exchange_world_one_empty_step_and_overflow(R, oracle, cctx):
    """Exchange(ctx, None, 1, 0, slot_points): steps of 4, 4 and 0 scans; the third reuses the first one's buffer and
    must publish 0 points, not the first step's count.  A slot smaller than the cloud holds its first slot_points points
    and the true total in its header."""
    steps = [oracle.synth_batch(500 + k, 4, CS, 4) for k in range(3)]
    ex = R.Exchange(cctx, None, 1, 0, 4 * CS)
    try:
        for k, (nodes, n) in enumerate(zip(steps, (4, 4, 0))):
            xyzi, pc, _, exp = clouds(R, oracle, cctx, nodes[:n] if n else nodes[:1], np.full(max(n, 1), CS, np.uint32))
            if n == 0:
                exp = exp[:0]
            idx = ex.allgather(xyzi.ptr, pc.ptr, n, CS)
            ex.synchronize()
            cctx.synchronize()
            assert idx == k % 2
            p_pts, p_cnt = ex.slot(idx, 0)
            c = int(read_device(p_cnt, (1,), "<u4")[0])
            assert c == len(exp), (k, c, len(exp))
            assert (read_device(p_pts, (max(c, 1), 4), "<f4")[:c].view(np.uint32) == exp.view(np.uint32)).all(), k
    finally:
        ex.close()
    xyzi, pc, _, exp = clouds(R, oracle, cctx, steps[0], np.full(4, CS, np.uint32))
    small = len(exp) // 2 + 3
    ex = R.Exchange(cctx, None, 1, 0, small)
    try:
        idx = ex.allgather(xyzi.ptr, pc.ptr, 4, CS)
        ex.synchronize()
        cctx.synchronize()
        p_pts, p_cnt = ex.slot(idx, 0)
        assert int(read_device(p_cnt, (1,), "<u4")[0]) == len(exp)
        assert (read_device(p_pts, (small, 4), "<f4").view(np.uint32) == exp[:small].view(np.uint32)).all()
    finally:
        ex.close()


def test_fuse_push_world_one_empty_batch_clears_the_header(R, oracle, cctx):
    """rpl_cloud_fuse_push_dev into a world-1 gather buffer from rpl_peer_alloc: a batch of 4 scans publishes its
    count and points, the empty batch after it publishes 0."""
    slot_points = 4 * CS
    base, _ = cctx.peer_alloc(R.lib().rpl_peer_gather_bytes(1, slot_points))
    try:
        xyzi, pc, _, exp = clouds(R, oracle, cctx, oracle.synth_batch(61, 4, CS, 4), np.full(4, CS, np.uint32))
        offs, total = out(4, SENT_U), out(1, SENT_U)
        on_device(cctx, lambda: cctx.cloud_fuse_push_dev(xyzi.ptr, pc.ptr, 4, CS, [base], 0, slot_points, offs.ptr,
                                                         total.ptr))
        assert int(read_device(base, (1,), "<u4")[0]) == len(exp) == int(total.get()[0])
        assert (read_device(base + 256, (len(exp), 4), "<f4").view(np.uint32) == exp.view(np.uint32)).all()
        on_device(cctx, lambda: cctx.cloud_fuse_push_dev(xyzi.ptr, pc.ptr, 0, CS, [base], 0, slot_points, offs.ptr,
                                                         total.ptr))
        assert int(read_device(base, (1,), "<u4")[0]) == 0
        assert int(total.get()[0]) == 0
    finally:
        cctx.peer_free(base)
