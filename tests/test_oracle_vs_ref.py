"""Checks the restatement against the reference's OWN compiled ascendScanData
(oracle/_ref, built from the reference sources by oracle/Makefile; its outputs are also stored as digests, see
tests/reference_outputs.py) on seeded random scans, tie-heavy ones included (same libstdc++ std::sort =>
identical permutation).  CPU only."""
import numpy as np
import pytest


def _same_ascend(O, reference, nodes):
    reference.check("ascendScanData", (nodes,), O.ascend(nodes, stable=False), lambda: O.ref_ascend(nodes))


@pytest.mark.parametrize("variant", [0, 1, 2, 3])
@pytest.mark.parametrize("n", [1, 2, 17, 360, 3200, 8192, 32768])
def test_ascend_synthetic_equals_reference(oracle, reference, n, variant):
    scans = oracle.synth_batch(1000 * variant + n, 3, n, variant)
    for s in scans:
        _same_ascend(oracle, reference, s)


def test_ascend_random_structures_equal_reference(oracle, reference):
    ref = oracle
    rng = np.random.default_rng(20260922)
    for trial in range(300):
        n = int(rng.integers(1, 600))
        keys = rng.integers(0, 65536, size=n) if trial % 3 else rng.integers(0, 64, size=n)
        dist = rng.integers(1, 1 << 20, size=n)
        p_inv = rng.choice([0.0, 0.05, 0.5, 0.95, 1.0])
        dist[rng.random(n) < p_inv] = 0
        nodes = ref.make_nodes(keys, dist, rng.integers(0, 256, size=n), rng.integers(0, 4, size=n))
        _same_ascend(ref, reference, nodes)


def test_stable_rule_is_a_valid_reference_outcome(oracle, reference):
    """On ties the CUDA path follows the stable rule; it must agree with the reference
    as a multiset per key and exactly wherever keys are unique."""
    ref = oracle
    scans = ref.synth_batch(77, 4, 2048, 2)
    for s in scans:
        _same_ascend(ref, reference, s)  # so the restatement's unstable order below is the reference's
        _, out_r = ref.ascend(s, stable=False)
        _, out_s = ref.ascend(s, stable=True)
        assert (out_r["angle_z_q14"] == out_s["angle_z_q14"]).all()
        a = np.sort(out_r.view(np.uint64))
        b = np.sort(out_s.view(np.uint64))
        assert (a == b).all()
        keys, cnt = np.unique(out_r["angle_z_q14"], return_counts=True)
        uniq = np.isin(out_r["angle_z_q14"], keys[cnt == 1])
        assert (out_r.view(np.uint64)[uniq] == out_s.view(np.uint64)[uniq]).all()


# ---- publish_scan: the restatement against the reference's REAL RPlidarNode::publish_scan -----------------------
# (src/rplidar_node.cpp compiled in place against the ROS API stubs in oracle/ros_stubs/, oracle/ref_shim_node.cpp)
def _published(pub, h7, ranges, intens):
    """What a LaserScan comparison looks at: nothing but the flag when no message goes out."""
    return (bool(pub), np.asarray(h7, np.float32), ranges, intens) if pub else (False,)


def _same_laserscan(O, reference, nodes, prm):
    hdr, r, it = O.publish(nodes, prm)
    mine = np.array([hdr.angle_min, hdr.angle_max, hdr.angle_increment, hdr.time_increment, hdr.scan_time,
                     hdr.range_min, hdr.range_max], np.float32)
    ours = _published(hdr.published, mine, r, it)
    fields = (prm.is_new_protocol, prm.scan_processing, prm.inverted, prm.range_max, prm.scan_duration)
    reference.check("publish_scan", (nodes,) + fields, ours, lambda: _published(*O.ref_publish(nodes, prm)))
    return len(r) if hdr.published else 0


CONFIGS = [(newp, mode_a, inv) for newp in (0, 1) for mode_a in (0, 1) for inv in (0, 1)]


@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("n", [1, 2, 17, 360, 3200, 8192, 32768])
def test_publish_scan_equals_the_real_node(oracle, reference, n, variant):
    O = oracle
    raw = O.synth_batch(4000 + n, 1, n, variant)[0]
    _same_ascend(O, reference, raw)
    rc, asc = O.ascend(raw)
    for newp, mode_a, inv in CONFIGS:
        for nodes in (raw, asc):
            _same_laserscan(O, reference, nodes, O.scan_params(newp, mode_a, inv, 0, 25.0, 0.0731))


def test_publish_scan_edge_cases_equal_the_real_node(oracle, reference):
    O = oracle
    mk = O.make_nodes
    cases = [mk([], []), mk([100], [0]), mk([0, 0, 0], [0, 0, 0]), mk([100], [4000], [40]),
             mk([5, 3], [4000, 8000], [1, 2]), mk([65535, 0, 1], [1, 2, 3], [255, 254, 253]),
             mk([7, 7, 7, 7], [400, 300, 200, 100], [4, 8, 12, 16])]  # four points on one angle
    rng = np.random.default_rng(12)
    for _ in range(40):
        n = int(rng.integers(1, 60))
        keys = rng.integers(0, 65536, n) if rng.random() < 0.5 else rng.integers(0, 64, n)  # dense ties
        dist = rng.integers(0, 1 << 20, n)
        dist[rng.random(n) < 0.3] = 0
        cases.append(mk(keys, dist, rng.integers(0, 256, n)))
    published = 0
    for c in cases:
        for newp, mode_a, inv in CONFIGS:
            published += 1 if _same_laserscan(O, reference, c, O.scan_params(newp, mode_a, inv, 0, 12.0, 0.1)) else 0
    assert published > 100


def test_laserscan_golden_fixture_is_what_the_real_node_produces(oracle, reference, golden_dir):
    """tests/golden/laserscan_golden.npz (generated through the restatement when the node could not be built)
    against the real publish_scan: every stored LaserScan, bit for bit."""
    O = oracle
    d = np.load(f"{golden_dir}/dummy_scans.npz")
    ls = np.load(f"{golden_dir}/laserscan_golden.npz")
    var = d["variants"].reshape(-1, 360, 8).copy().view(O.NODE_DTYPE).reshape(-1, 360)
    asc = d["variants_ascended"].reshape(-1, 360, 8).copy().view(O.NODE_DTYPE).reshape(-1, 360)
    for k in range(int(ls["n"])):
        vi, use_asc, newp, mode_a, inv = ls[f"cfg_{k}"].tolist()
        nodes = asc[vi] if use_asc else var[vi]
        prm = O.scan_params(newp, mode_a, inv, use_asc, 12.0, 0.1)
        assert len(ls[f"ranges_{k}"]) == int(ls[f"beams_{k}"])
        stored = _published(True, ls[f"hdr_{k}"], ls[f"ranges_{k}"], ls[f"intens_{k}"])
        reference.check("publish_scan", (nodes, newp, mode_a, inv, 12.0, 0.1), stored,
                        lambda: _published(*O.ref_publish(nodes, prm)))


@pytest.mark.parametrize("mode_a", [0, 1])
def test_batched_reference_path_equals_the_port(oracle, reference, mode_a):
    """ref_pipeline_batch (the reference's ascend glue + real publish_scan, 4 worker threads) against the oracle
    port on the same batch: what `bench.py --impl reference` times is the code the parity tests pin."""
    O = oracle
    S, N = 24, 3200
    batch = O.synth_batch(555, S, N, variant=0)
    counts = np.full(S, N, np.uint32)
    counts[3], counts[5] = 0, 17
    prm = O.scan_params(0, mode_a, 0, 1, 40.0, 0.1)

    def published(res):
        b = res["beam_counts"]
        return (b,) + tuple(res[k][s, : int(b[s])] for s in range(S) for k in ("ranges", "intensities"))

    port = O.pipeline_batch(batch.copy(), counts, prm, stable=False, threads=2)
    reference.check("ascend + publish_scan batch", (batch, counts, mode_a), published(port),
                    lambda: published(O.ref_pipeline_batch(batch, counts, prm, threads=4)))
    if reference.live:
        t = O.ref_pipeline_batch(batch, counts, prm, threads=4, outputs=False)
        assert t["seconds"] > 0 and t["ranges"] is None
