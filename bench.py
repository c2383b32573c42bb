#!/usr/bin/env python
"""bench.py -- the hot path on synthetic scan streams, one JSON line on stdout.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU loop

Workload (BASELINE.json configs[1], SURVEY.md 8(d) C2): S2 DenseBoost, 32768 nodes/scan x 4096
scans per GPU (1.07 GB of packed nodes in, 1.07 GB of LaserScan floats out per step -- both far
larger than the 126 MB L2, so no L2 flush is needed between iterations).  One step = one pass of
the fused path (ascendScanData status + filter + fixed-point unpack + angle rank + LaserScan
Mode B, the launch-file default `scan_processing: false`) over the whole batch.

  value     Mpoints/s (input nodes per second), buffers resident in HBM, CUDA events on the
            launching stream, max over ranks, whole-job aggregate over N GPUs (weak scaling:
            every rank owns its own 4096 scans; the LaserScan path has no data-path collective)
  e2e       the same metric through the host-buffer C-ABI call rpl_scan_batch: pinned host
            buffers in, H2D + kernels + D2H inside the timed region
  roofline  scan_fast_kernel: algorithmic bytes (16 B/node, SURVEY.md 8(d)) / kernel time from
            CUDA events recorded by the library around every launch, against the measured HBM
            copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline  the oracle (a port of the reference loop) on this box's host cores, same buffers

The oracle is used here ONLY as the cpu_baseline / --impl reference leg.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "Mpoints/s through unpack+filter+polar->xyz (LaserScan path: fused ascend+unpack+filter+angle-rank)"
UNIT = "Mpoints/s"
NODES_PER_SCAN = 32768
SCANS_PER_GPU = 4096
BYTES_PER_NODE_LASERSCAN = 16  # 8 B node read + 4 B ranges + 4 B intensities (SURVEY.md 8(d))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scans", type=int, default=SCANS_PER_GPU, help="scans per GPU")
    ap.add_argument("--nodes", type=int, default=NODES_PER_SCAN, help="nodes per scan")
    ap.add_argument("--mode", default="b", choices=["a", "b"], help="LaserScan mode of the headline")
    ap.add_argument("--variant", type=int, default=0, help="synthetic variant (SURVEY 8(d))")
    ap.add_argument("--workload", default="scan", choices=["scan", "cloud", "decode", "chain"],
                    help="scan: LaserScan path (headline, BASELINE configs[1]); cloud: PointCloud2 path "
                         "(configs[2]/[4]: 64 S3 streams per GPU, polar->xyz + 5 cm voxels, all-gather of the fused cloud)")
    ap.add_argument("--format", default="0x85",
                    help="decode workload: SDK answer type (0x81 standard nodes, 0x82 express, 0x83 HQ, 0x84 ultra, "
                         "0x85 dense, 0x86 ultra-dense)")
    ap.add_argument("--sor", type=int, default=0, help="cloud workload: SOR k (0 = off)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-wc", action="store_true",
                    help="e2e leg: the host INPUT buffer is write-combined pinned memory (cudaHostAllocWriteCombined): "
                         "the GPU's reads of it do not snoop the CPU caches")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--chain-copy", action="store_true",
                    help="chain workload: copy the revolutions out of the node stream (rpl_assemble_scans_dev) instead of "
                         "handing views to the scan kernel")
    ap.add_argument("--no-cloud", action="store_true", help="skip the PointCloud2 + exchange leg (extra.cloud)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="scan workload: after the timed steps, write what the last one returned (rank 0) as "
                         "DIR/<name>.npy, float32 or float64, for a fixed seeded sample of the scans")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "scan"):
        ap.error("--dump-outputs writes the outputs of the scan workload of this repo's path")
    return args


DUMP_BYTES = 60 << 20  # what --dump-outputs writes stays under 64 MB


def dump_scan_outputs(out_dir, ranges, intens, beams, inc, status):
    """The LaserScans of a fixed seeded sample of the batch, as a caller of rpl_scan_batch_dev receives them:
    ranges and intensities [k, nodes] (zero past each scan's beam count, where nothing is written), and per scan
    the beam count, angle increment and ascendScanData status.  scan_index holds the sampled scans' indices."""
    S, N = ranges.shape
    k = max(1, min(S, DUMP_BYTES // (8 * N + 32)))
    idx = np.sort(np.random.default_rng(0).choice(S, k, replace=False))
    sel = lambda t: t[idx].cpu().numpy()  # noqa: E731
    b = sel(beams)
    past = np.arange(N)[None, :] >= b[:, None]
    arrays = {"scan_index": idx.astype(np.float64), "beam_counts": b.astype(np.float64),
              "angle_increment": sel(inc).astype(np.float32), "status": sel(status).view(np.uint32).astype(np.float64),
              "ranges": np.where(past, np.float32(0), sel(ranges)), "intensities": np.where(past, np.float32(0), sel(intens))}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def workload_name(args):
    return (f"S2 DenseBoost {args.nodes} nodes/scan x {args.scans} scans per GPU, synthetic variant "
            f"{args.variant} (tie-free rotated revolution, 5% unmeasured), LaserScan Mode "
            f"{'A' if args.mode == 'a' else 'B'}, angle_compensate on")


def effective_cores():
    """(usable host threads, how it was derived): CPU affinity of this process capped by the cgroup CPU quota --
    os.cpu_count() reports the machine, not the lease."""
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota, src = None, None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:  # cgroup v2
            q, per = f.read().split()[:2]
        if q != "max":
            quota, src = int(q) / int(per), "cgroup v2 cpu.max"
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = int(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                per = int(f.read())
            if q > 0:
                quota, src = q / per, "cgroup v1 cfs quota"
        except Exception:
            pass
    n = aff
    how = f"sched_getaffinity={aff}, os.cpu_count()={os.cpu_count()}"
    if quota is not None:
        n = max(1, min(aff, int(quota + 0.999)))
        how += f", {src}={quota:.2f} CPUs"
    else:
        how += ", no cgroup CPU quota"
    return n, how


def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def numa_pin(dev_index):
    """Bind this process (and so the pinned host buffers it allocates from now on: first touch, local policy) to the
    CPUs of the NUMA node the GPU hangs off.  Returns a dict for the report; never raises.  (Keeps host traffic off
    the inter-socket link.  It is not what bounds the e2e figure at N >= 4 on the HGX box: four GPUs behind one
    socket share ~187 GB/s of DMA traffic however the buffers are placed -- DESIGN.md section 7.)"""
    info = {"pinned": False}
    try:
        import torch

        pr = torch.cuda.get_device_properties(dev_index)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read())
        info.update({"pci": bdf, "numa_node": node})
        if node < 0:
            info["note"] = "platform reports no NUMA node for this GPU"
            return info
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = _parse_cpulist(f.read())
        before = os.sched_getaffinity(0)
        want = cpus & before
        if not want:
            info["note"] = "no allowed CPU on the GPU's NUMA node"
            return info
        os.sched_setaffinity(0, want)
        info.update({"pinned": True, "cpus": len(want), "cpus_before": len(before)})
        info["_before"] = before
    except Exception as e:  # pragma: no cover - depends on the host
        info["note"] = f"not pinned: {e!r}"
    return info


def numa_unpin(info):
    before = info.pop("_before", None)
    if before:
        try:
            os.sched_setaffinity(0, before)
        except Exception:
            pass


def bench_config(args, world):
    """The `config` object -- the same keys and values in both arms (repo and --impl reference; the reference arm's
    bounded per-step sample is described in its cpu_baseline.sample, not here)."""
    return {"workload": workload_name(args), "scans_per_gpu": args.scans, "nodes_per_scan": args.nodes,
            "parallelism": f"{world} x independent stream shards (no data-path collective on the LaserScan path)",
            "l2": "inputs 1.07 GB + outputs 1.07 GB per step exceed the 126 MB L2; no flush needed"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


# ------------------------------------------------------------------------------------------------
# clocks: NVML polled from a thread DURING the timed regions
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting",
               0x10: "sync_boost"}

    def __init__(self, uuid: str | None, index: int):
        self.samples = []  # (t, sm_mhz, reasons_mask, power_w)
        self.windows = []
        self._stop = threading.Event()
        self._thr = None
        self.max_mhz = None
        self.ok = False
        try:
            import pynvml as nv

            nv.nvmlInit()
            self.nv = nv
            h = None
            if uuid:
                try:
                    h = nv.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
                except Exception:
                    h = None
            self.h = h if h is not None else nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def _reasons(self):
        nv = self.nv
        for name in ("nvmlDeviceGetCurrentClocksEventReasons", "nvmlDeviceGetCurrentClocksThrottleReasons"):
            fn = getattr(nv, name, None)
            if fn:
                try:
                    return int(fn(self.h))
                except Exception:
                    continue
        return 0

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                except Exception:
                    pw = 0.0
                self.samples.append((time.perf_counter(), mhz, self._reasons(), pw))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.ok:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=2)

    def window(self, t0, t1, name):
        self.windows.append((t0, t1, name))

    def summary_for(self, t0, t1):
        """Clocks over one window only (the per-leg `clocks` objects)."""
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "NVML unavailable"}
        w = [x for x in self.samples if t0 <= x[0] <= t1]
        if not w:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0,
                    "note": "window shorter than the 2 ms sampling period"}
        mask = 0
        for x in w:
            mask |= x[2]
        return {"sm_mhz": statistics.median([x[1] for x in w]), "sm_max_mhz": self.max_mhz,
                "reasons": [v for k, v in self.REASONS.items() if mask & k], "samples": len(w),
                "power_w_max": max(x[3] for x in w)}

    def summary(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "NVML unavailable"}
        used, names = [], []
        for t0, t1, name in self.windows:
            w = [s for s in self.samples if t0 <= s[0] <= t1]
            if w:
                used += w
                names.append(name)
            if len(used) >= 5:
                break
        if not used:
            used = self.samples[-5:]
            names = ["nearest samples"]
        mask = 0
        for s in used:
            mask |= s[2]
        reasons = [v for k, v in self.REASONS.items() if mask & k]
        return {"sm_mhz": statistics.median([s[1] for s in used]) if used else None,
                "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(used),
                "power_w_max": max([s[3] for s in used]) if used else None, "window": " + ".join(names)}


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU loop on the host cores
# ------------------------------------------------------------------------------------------------
def start_sampler(dev, local_rank):
    import torch

    uuid = None
    try:
        uuid = str(torch.cuda.get_device_properties(dev).uuid)
    except Exception:
        pass
    sp = ClockSampler(uuid, local_rank)
    sp.start()
    return sp


def cpu_kind(O):
    """("reference", text) when the reference's own code is available as oracle/_ref/libref_node.so (built in the
    authoring container from /root/reference: the SDK's ascendScanData + the node's real publish_scan, the latter
    compiled against ROS API stubs), else ("port", text): the line-by-line restatement in oracle/scan_oracle.cpp."""
    if O.have_ref_node():
        return "reference", ("the reference's own code: grab_scan_data's ascend glue + sl::ascendScanData + "
                             "RPlidarNode::publish_scan compiled from the reference sources (oracle/_ref/libref_node.so)")
    return "port", "oracle port of ascendScanData+publish_scan (validated against the compiled reference)"


def cpu_leg(O, nodes_host, counts, mode_a, threads, reps):
    """ascendScanData + publish_scan per scan (one scan per worker).  Returns (Mpoints/s, seconds)."""
    prm = O.scan_params(0, mode_a, 0, 1, 40.0, 0.1)
    total_pts = int(counts.sum())
    secs = 0.0
    use_ref = O.have_ref_node()
    if use_ref:  # untimed: every worker allocates (and first touches) its buffers once
        warm = min(nodes_host.shape[0], 2 * threads)
        O.ref_pipeline_batch(nodes_host[:warm], counts[:warm], prm, threads=threads, outputs=False)
    for _ in range(reps):
        if use_ref:  # copies every scan into its own buffer first, as the SDK delivers it
            res = O.ref_pipeline_batch(nodes_host, counts, prm, threads=threads, outputs=False)
        else:
            buf = nodes_host.copy()  # ascend works in place: start every rep from the raw buffers
            res = O.pipeline_batch(buf, counts, prm, stable=False, threads=threads)
        secs += res["seconds"]
    return total_pts * reps / secs / 1e6, secs


def run_reference(args, rank):
    if rank != 0:
        return  # rank 0 alone runs and prints the reference arm
    from oracle import pyoracle as O

    O.build(ref=False)
    cores, cores_how = effective_cores()
    mode_a = 1 if args.mode == "a" else 0
    # size the per-step sample: as much of the bench batch as fits ~90 s for the whole run, and never
    # so small that it sits in the CPUs' caches (the GPU arm streams a fresh 1 GB batch from host
    # memory every step; a 64 MB sample replayed from L3 would not be the same workload)
    probe = O.synth_batch(0, min(args.scans, 256), args.nodes, args.variant)
    pc = np.full(probe.shape[0], args.nodes, np.uint32)
    cpu_leg(O, probe, pc, mode_a, cores, 1)
    _, t_probe = cpu_leg(O, probe, pc, mode_a, cores, 1)
    per_scan = t_probe / probe.shape[0]
    budget_s = 90.0
    fit = int(budget_s / max(1, args.steps + max(args.warmup, 1)) / max(per_scan, 1e-9))
    sample_scans = int(min(args.scans, max(min(args.scans, 1024), fit)))
    nodes = O.synth_batch(0, sample_scans, args.nodes, args.variant)
    counts = np.full(sample_scans, args.nodes, np.uint32)
    for _ in range(max(args.warmup, 1)):
        cpu_leg(O, nodes, counts, mode_a, cores, 1)
    t_total, pts = 0.0, 0
    for _ in range(args.steps):
        _, s = cpu_leg(O, nodes, counts, mode_a, cores, 1)
        t_total += s
        pts += int(counts.sum())
    value = pts / t_total / 1e6
    one, _ = cpu_leg(O, nodes[:32].copy(), counts[:32], mode_a, 1, 1)
    kind, what = cpu_kind(O)
    sample = (f"{sample_scans} scans x {args.nodes} nodes per step ({sample_scans * args.nodes / 1e6:.1f} Mpoints), "
              f"{what}, one scan per worker thread, {cores} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_total / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(args, max(args.gpus, 1)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "cores_how": cores_how, "kind": kind,
                         "sample": sample, "value_1thread": one},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------
def run_b200(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    import rplidar_ros2_driver_b200 as R

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the CUDA library is the only implementation of this path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = numa_pin(local_rank)  # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    S, N = args.scans, args.nodes
    mode_a = 1 if args.mode == "a" else 0
    ctx = R.Context(local_rank, N, S)
    # a real (non-default) stream: the library treats a NULL stream as "use the context's own"
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sptr = stream.cuda_stream
    assert sptr != 0

    nodes = torch.empty((S, N, 8), dtype=torch.uint8, device=dev)
    counts = torch.empty(S, dtype=torch.int32, device=dev)
    ranges = torch.empty((S, N), dtype=torch.float32, device=dev)
    intens = torch.empty((S, N), dtype=torch.float32, device=dev)
    beams = torch.empty(S, dtype=torch.int32, device=dev)
    inc = torch.empty(S, dtype=torch.float32, device=dev)
    status = torch.empty(S, dtype=torch.int32, device=dev)
    path = torch.empty(S, dtype=torch.int32, device=dev)
    ctx.synth_batch_dev(rank * S, S, N, N, args.variant, nodes.data_ptr(), counts.data_ptr(), stream=sptr)
    torch.cuda.synchronize()

    def step(params, nodes_out=None):
        ctx.scan_batch_dev(nodes.data_ptr(), counts.data_ptr(), S, N, params, nodes_out=nodes_out,
                           ranges=ranges.data_ptr(), intensities=intens.data_ptr(), beam_counts=beams.data_ptr(),
                           angle_increment=inc.data_ptr(), status=status.data_ptr(), path=path.data_ptr(),
                           stream=sptr)

    uuid = None
    try:
        uuid = str(torch.cuda.get_device_properties(dev).uuid)
    except Exception:
        pass
    sampler = ClockSampler(uuid, local_rank)
    sampler.start()

    def timed(params, K, W, nodes_out=None, profile=False):
        for _ in range(W):
            step(params, nodes_out)
        torch.cuda.synchronize()
        ctx.profile_read()
        ctx.profile(profile)
        l0 = ctx.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(K):
            step(params, nodes_out)
        e1.record(stream)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1))
        prof = ctx.profile_read()
        ctx.profile(False)
        return ms, prof, ctx.launch_count - l0, (t0, t1)

    params = R.scan_params(0, mode_a, 0, 1)
    ms, prof, launches, win = timed(params, args.steps, max(args.warmup, 3), profile=True)
    sampler.window(win[0], win[1], "timed region")
    if args.dump_outputs and rank == 0:  # before the legs below reuse the buffers
        dump_scan_outputs(args.dump_outputs, ranges, intens, beams, inc, status)
    pts_step = S * N
    value = world * pts_step * args.steps / (ms * 1e-3) / 1e6
    n_fast = int((path == 0).sum().item())
    fast_ms = prof[0] / max(prof[1], 1)
    peak, peak_src = measured_peak()
    alg_bytes = BYTES_PER_NODE_LASERSCAN * pts_step
    achieved = alg_bytes / (fast_ms * 1e-3) / 1e9
    # DRAM bytes per launch from the committed ncu capture of THIS shape and mode (null when none exists)
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f).get(f"scan.mode_{args.mode}.{S}x{N}")
    except Exception:
        pass
    kname = ("scan_small_kernel<Mode %s> (revolution staged once into shared memory, scan_small.cu)" if N <= 8192 else
             "scan_tma_kernel<Mode %s> (TMA-ring fast kernel, scan_tma.cu)") % args.mode.upper()
    roofline = {"bound": "hbm", "kernel": kname,
                "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": fast_ms,
                "kernel_share_of_step": prof[0] / ms if ms > 0 else None,
                "general_kernel_ms": prof[2] / max(prof[3], 1)}

    extra = {"scans_on_fast_kernel": n_fast, "scans_total": S}
    if not args.no_extra:
        k2 = max(5, min(args.steps, 30))
        other = R.scan_params(0, 1 - mode_a, 0, 1)
        ms2, prof2, _, _ = timed(other, k2, 3, profile=True)
        extra[f"mode_{'b' if mode_a else 'a'}_mpoints_s"] = world * pts_step * k2 / (ms2 * 1e-3) / 1e6
        nodes_out = torch.empty((S, N, 8), dtype=torch.uint8, device=dev)
        ms3, prof3, _, _ = timed(params, k2, 3, nodes_out=nodes_out.data_ptr(), profile=True)
        f3 = prof3[0] / max(prof3[1], 1)
        extra["with_ascended_nodes_out"] = {
            "mpoints_s": world * pts_step * k2 / (ms3 * 1e-3) / 1e6, "bytes_per_node": 24,
            "achieved_gbs": 24 * pts_step / (f3 * 1e-3) / 1e9, "frac": 24 * pts_step / (f3 * 1e-3) / 1e9 / peak}
        del nodes_out

    # ---- the same kernels' work at the size a lidar delivers (S2/S3: ~3200 nodes per revolution), all three
    # LaserScan variants, device resident; the headline shape above is BASELINE.json's, this is the realistic one ----
    if not args.no_extra and N > 8192:
        S2, N2 = 40960, 3200
        c2 = R.Context(local_rank, N2, S2)
        n2 = torch.empty((S2, N2, 8), dtype=torch.uint8, device=dev)
        k2c = torch.empty(S2, dtype=torch.int32, device=dev)
        r2 = ranges.view(-1)[: S2 * N2].view(S2, N2)  # (the headline buffers are larger: reuse them)
        i2 = intens.view(-1)[: S2 * N2].view(S2, N2)
        o2 = torch.empty((S2, N2, 8), dtype=torch.uint8, device=dev)
        aux2 = torch.empty((4, S2), dtype=torch.int32, device=dev)  # beam counts, angle increments, status, path
        c2.synth_batch_dev(rank * S2 + 7, S2, N2, N2, args.variant, n2.data_ptr(), k2c.data_ptr(), stream=sptr)
        torch.cuda.synchronize()
        small = {"shape": f"{S2} scans x {N2} nodes per GPU", "kernel": "scan_small_kernel (scan_small.cu)"}
        for tag, ma, emit, bpn in (("mode_b", 0, False, 16), ("mode_a", 1, False, 16), ("mode_b_with_ascended_nodes_out", 0, True, 24)):
            prm2 = R.scan_params(0, ma, 0, 1)

            def step2():
                c2.scan_batch_dev(n2.data_ptr(), k2c.data_ptr(), S2, N2, prm2, nodes_out=o2.data_ptr() if emit else None,
                                  ranges=r2.data_ptr(), intensities=i2.data_ptr(), beam_counts=aux2[0].data_ptr(),
                                  angle_increment=aux2[1].data_ptr(), status=aux2[2].data_ptr(), path=aux2[3].data_ptr(),
                                  stream=sptr)

            for _ in range(3):
                step2()
            kk = max(5, min(args.steps, 30))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            torch.cuda.synchronize()
            e0.record(stream)
            for _ in range(kk):
                step2()
            e1.record(stream)
            torch.cuda.synchronize()
            msk = max_over_ranks(e0.elapsed_time(e1)) / kk
            gbs = bpn * S2 * N2 / (msk * 1e-3) / 1e9
            small[tag] = {"mpoints_s": world * S2 * N2 / (msk * 1e-3) / 1e6, "ms_per_step": msk, "bytes_per_node": bpn,
                          "achieved_gbs_per_gpu": gbs, "frac": gbs / peak,
                          "scans_on_this_kernel": int((aux2[3] == 0).sum().item())}
        extra["lidar_sized_revolutions"] = small
        del n2, o2
        c2.close()
        step(params)  # (the e2e leg compares against the headline buffers: refill them)
        torch.cuda.synchronize()

    # ---- single-scan latency through the reference-shaped call rpl_scan (host buffers) ------------
    if not args.no_extra and rank == 0:
        import ctypes as C

        L = R.lib()
        lat = {}
        lctx = R.Context(local_rank, 8192, 1)
        prm1 = R.scan_params(0, mode_a, 0, 1)
        for nn in (360, 3200, 8192):
            tmp = torch.empty((1, nn, 8), dtype=torch.uint8, device=dev)
            lctx.synth_batch_dev(rank * S, 1, nn, nn, args.variant, tmp.data_ptr(), None, stream=sptr)
            torch.cuda.synchronize()
            one = np.zeros(nn, dtype=R.NODE_DTYPE)
            one[:] = tmp[0].cpu().numpy().view(R.NODE_DTYPE).reshape(-1)
            r1, i1 = np.zeros(nn, np.float32), np.zeros(nn, np.float32)
            b1, a1, s1 = C.c_uint32(0), C.c_float(0), C.c_uint32(0)

            def call():
                L.rpl_scan(lctx._h, C.c_void_p(one.ctypes.data), nn, C.byref(prm1), C.c_void_p(r1.ctypes.data),
                           C.c_void_p(i1.ctypes.data), C.byref(b1), C.byref(a1), C.byref(s1))

            for _ in range(20):
                call()
            t0 = time.perf_counter()
            for _ in range(300):
                call()
            lat[str(nn)] = (time.perf_counter() - t0) / 300 * 1e6
        lctx.close()
        extra["single_scan_latency_us"] = lat
        extra["single_scan_latency_note"] = ("rpl_scan through the C-ABI (ascend + LaserScan, pageable host buffers): one "
                                             "lidar revolution at a time, the reference's actual operating point")

    # ---- e2e: host buffers through rpl_scan_batch ------------------------------------------------
    e2e = None
    h_nodes = None
    if not args.no_e2e:
        if args.e2e_wc:
            import ctypes as C

            rt = C.CDLL("libcudart.so.12")
            rt.cudaHostAlloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t, C.c_uint]
            wc_ptr = C.c_void_p()
            rc = rt.cudaHostAlloc(C.byref(wc_ptr), S * N * 8, 0x04)  # cudaHostAllocWriteCombined
            if rc != 0:
                raise SystemExit(f"cudaHostAlloc(write-combined) failed: {rc}")
            h_nodes_t = torch.from_numpy(np.ctypeslib.as_array((C.c_uint8 * (S * N * 8)).from_address(wc_ptr.value))).view(S, N, 8)
        else:
            h_nodes_t = torch.empty((S, N, 8), dtype=torch.uint8, pin_memory=True)
        h_nodes_t.copy_(nodes)
        h_counts = counts.cpu().numpy().astype(np.uint32)
        h_nodes = h_nodes_t.numpy().view(R.NODE_DTYPE).reshape(S, N)
        out_t = {"ranges": torch.empty((S, N), dtype=torch.float32, pin_memory=True),
                 "intensities": torch.empty((S, N), dtype=torch.float32, pin_memory=True)}
        out = {k: v.numpy() for k, v in out_t.items()}
        ke = max(3, min(args.steps, 10))
        # what the host link can do on this box (plain pinned copies of the same buffers)
        pc = []
        for src, dst in ((h_nodes_t, nodes), (ranges, out_t["ranges"])):
            if args.e2e_wc and src is h_nodes_t:  # (torch would stage a buffer it did not pin itself)
                pc.append(None)
                continue
            torch.cuda.synchronize()
            tp0 = time.perf_counter()
            dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize()
            pc.append(src.numel() * src.element_size() / (time.perf_counter() - tp0) / 1e9)
        for _ in range(2):
            res = ctx.scan_batch(h_nodes, h_counts, params, out=out)
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(ke):
            res = ctx.scan_batch(h_nodes, h_counts, params, out=out)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        barrier()
        sampler.window(t0, t1, "e2e leg")
        dt = max_over_ranks(t1 - t0)
        # the device-resident result and the host-path result must be the same bytes
        step(params)
        torch.cuda.synchronize()
        same = True
        for sidx in (0, S // 2, S - 1):
            m = int(res["beam_counts"][sidx])
            dev_r = ranges[sidx, :m].cpu().numpy().view(np.uint32)
            dev_i = intens[sidx, :m].cpu().numpy().view(np.uint32)
            same = same and m == int(beams[sidx].item()) and bool((dev_r == out["ranges"][sidx, :m].view(np.uint32)).all()) \
                and bool((dev_i == out["intensities"][sidx, :m].view(np.uint32)).all())
        e2e = {"value": world * pts_step * ke / dt / 1e6, "unit": UNIT,
               "h2d_bytes_per_step": S * N * 8 + S * 4, "d2h_bytes_per_step": 2 * S * N * 4 + 4 * S * 4,
               "steps": ke, "ms_per_step": dt / ke * 1e3, "api": "rpl_scan_batch (pinned host buffers)",
               "matches_device_path": same, "beam_count_scan0": int(res["beam_counts"][0]),
               "link_h2d_gbs": pc[0], "link_d2h_gbs": pc[1],
               "input_buffer": "write-combined pinned (cudaHostAllocWriteCombined)" if args.e2e_wc else "pinned"}
    # ---- BASELINE configs[2]/[4]: PointCloud2 path + the one exchange, at this world size --------
    if not args.no_cloud:
        try:
            extra["cloud"] = cloud_leg(args, ctx_factory=lambda mn, ms: R.Context(local_rank, mn, ms), rank=rank,
                                       world=world, dev=dev, stream=stream, sampler=sampler,
                                       steps=max(5, min(args.steps, 20)), barrier=barrier, max_over_ranks=max_over_ranks)
        except Exception as e:  # the headline line must still be printed
            import traceback

            extra["cloud"] = {"error": repr(e), "trace": traceback.format_exc()[-1500:]}
    sampler.stop()
    clocks = sampler.summary()
    numa_unpin(numa)  # the CPU baseline may use every core the lease has

    # ---- cpu baseline: rank 0, N=1 only -----------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import pyoracle as O

        O.build(ref=False)
        cores, cores_how = effective_cores()
        if h_nodes is None:
            h_nodes = nodes.cpu().numpy().view(R.NODE_DTYPE).reshape(S, N)
        hc = np.full(S, N, np.uint32)
        host = np.ascontiguousarray(h_nodes).view(O.NODE_DTYPE).reshape(S, N)
        v_all, secs = cpu_leg(O, host, hc, mode_a, cores, 2)
        sub = min(S, 128)
        v_one, _ = cpu_leg(O, host[:sub].copy(), hc[:sub], mode_a, 1, 1)
        per_scan = {}
        for nn in (360, 3200, 8192):
            sm_nodes = O.synth_batch(0, 64, nn, args.variant)
            if O.have_ref_node():
                rr = O.ref_pipeline_batch(sm_nodes, np.full(64, nn, np.uint32), O.scan_params(0, mode_a, 0, 1, 40.0, 0.1),
                                          threads=1, outputs=False)
            else:
                rr = O.pipeline_batch(sm_nodes, np.full(64, nn, np.uint32), O.scan_params(0, mode_a, 0, 1, 40.0, 0.1),
                                      stable=False, threads=1)
            per_scan[str(nn)] = rr["seconds"] / 64 * 1e6
        extra["single_scan_latency_cpu_1thread_us"] = per_scan
        kind, what = cpu_kind(O)
        cpu = {"value": v_all, "unit": UNIT, "cores": cores, "cores_how": cores_how, "kind": kind,
               "sample": (f"the bench batch itself, 2 passes x {S} scans x {N} nodes = {2 * S * N / 1e6:.0f} Mpoints "
                          f"({secs:.1f} s wall, {cores} worker threads, one scan per task); {what}"),
               "value_1thread": v_one, "sample_1thread": f"{sub} scans x {N} nodes"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(args, world),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "extra": extra,
        }
        line["extra"]["numa"] = {k: v for k, v in numa.items() if not k.startswith("_")}
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


CLOUD_STREAMS_PER_GPU, CLOUD_SCANS_PER_STREAM, CLOUD_NODES = 64, 256, 3200


def cloud_leg(args, ctx_factory, rank, world, dev, stream, sampler, steps, barrier, max_over_ranks, sor=0):
    """BASELINE configs[2] (N=1) / configs[4] (N>1): 64 synthetic S3 streams per GPU (256 revolutions x 3200 nodes
    each) -> window + polar->xyz + 5 cm voxel grid (+ SOR) per revolution -> fused per-GPU cloud -> ONE all-gather
    of the fused cloud per step.  Three exchanges, all behind the C-ABI:
      nccl  rpl_exchange (C++): pack on the compute stream, one ncclAllGather on the exchange stream, overlapped
            with the next batch's kernels
      copy  rpl_exchange (C++): pack on the compute stream, world-1 peer copies by the copy engines over NVLink
            (CUDA IPC mappings) + a 4-byte barrier on the exchange stream, overlapped likewise
      push  rpl_cloud_fuse_push_dev: pack AND all-gather in one kernel (stores straight into every peer's buffer),
            on the compute stream, not overlapped
    Before anything is timed the three must deliver identical bytes on every rank at this world size."""
    import torch
    import torch.distributed as dist

    import rplidar_ros2_driver_b200 as R
    from rplidar_ros2_driver_b200.multi_gpu import PeerCloudGather, shard_streams

    N = CLOUD_NODES
    streams_total = CLOUD_STREAMS_PER_GPU * world
    mine = shard_streams(streams_total, world, rank)
    S = len(mine) * CLOUD_SCANS_PER_STREAM
    ctx = ctx_factory(N, S)
    sp = stream.cuda_stream
    nodes = torch.empty((S, N, 8), dtype=torch.uint8, device=dev)
    counts = torch.empty(S, dtype=torch.int32, device=dev)
    xyzi = torch.empty((S, N, 4), dtype=torch.float32, device=dev)
    pc = torch.empty(S, dtype=torch.int32, device=dev)
    offs = torch.empty(S, dtype=torch.int32, device=dev)
    total = torch.zeros(1, dtype=torch.int32, device=dev)
    ctx.synth_batch_dev(mine.start * CLOUD_SCANS_PER_STREAM, S, N, N, 4, nodes.data_ptr(), counts.data_ptr(), stream=sp)
    prm = R.cloud_params(range_min=0.15, range_max=40.0, voxel_size=0.05, sor_k=sor, sor_alpha=1.0)

    def compute():
        ctx.cloud_batch_dev(nodes.data_ptr(), counts.data_ptr(), S, N, prm, xyzi.data_ptr(), pc.data_ptr(), stream=sp)

    compute()
    torch.cuda.synchronize()
    kept = int(pc.sum().item())
    cap = kept + 1024  # the synthetic batch is the same every step: the slot holds exactly this rank's cloud
    if world > 1:  # one slot size for every rank
        cap_t = torch.tensor([cap], device=dev)
        dist.all_reduce(cap_t, op=dist.ReduceOp.MAX)
        cap = int(cap_t.item())
    # the C++ exchange: rank 0 makes the NCCL id, the process group only carries its 128 bytes
    uid = None
    if world > 1:
        idt = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(R.exchange_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        uid = bytes(idt.cpu().numpy().tobytes())
    ex = R.Exchange(ctx, uid, world, rank, cap)
    g_push = PeerCloudGather(ctx, cap, dev)
    last = {"idx": 0, "half": 0}

    def exch(mode):
        def f():
            last["idx"] = ex.allgather(xyzi.data_ptr(), pc.data_ptr(), S, N, mode, stream=sp)
        return f

    def exch_push():
        last["half"] = g_push.push(xyzi.data_ptr(), pc.data_ptr(), S, N, offs.data_ptr(), total.data_ptr(), stream=sp)

    def drain():  # the compute stream catches up with the exchange stream
        ex.wait(0, stream=sp)
        ex.wait(1, stream=sp)

    def gathered_of_exchange(idx):
        outs, cnts = [], []
        for r in range(world):
            p_pts, p_cnt = ex.slot(idx, r)
            c = int(torch.as_tensor(_DevView(p_cnt, (1,), "<i4"), device=dev)[0].item())
            cnts.append(c)
            outs.append(torch.as_tensor(_DevView(p_pts, (cap, 4), "<f4"), device=dev)[:min(c, cap)].clone())
        return torch.cat(outs, dim=0), cnts

    # ---- on-box parity of the exchanges at THIS world size (driver-visible evidence) --------------------
    compute()
    exch(R.EXCHANGE_NCCL)()
    drain()
    torch.cuda.synchronize()
    a, c_n = gathered_of_exchange(last["idx"])
    exch(R.EXCHANGE_COPY)()
    drain()
    torch.cuda.synchronize()
    b, c_c = gathered_of_exchange(last["idx"])
    exch_push()
    torch.cuda.synchronize()
    c_p = [int(v) for v in g_push.counts(last["half"]).tolist()]
    gp = g_push.gathered(last["half"])
    d = torch.cat([gp[r, : c_p[r]] for r in range(world)], dim=0)
    # and what this rank itself produced sits in its own place
    own_lo = sum(c_n[:rank])
    own = torch.cat([xyzi[sidx, : int(k)] for sidx, k in enumerate(pc.tolist()) if k], dim=0) if kept else a[:0]
    ok = (c_n == c_c == c_p) and a.shape == b.shape == d.shape \
        and bool(torch.equal(a.view(torch.int32), b.view(torch.int32))) and bool(torch.equal(a.view(torch.int32), d.view(torch.int32))) \
        and c_n[rank] == kept and bool(torch.equal(a[own_lo: own_lo + kept].view(torch.int32), own.view(torch.int32)))
    ok_t = torch.tensor([1 if ok else 0], device=dev)
    sums = torch.tensor([float(a.double().sum().item())], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ok_t, op=dist.ReduceOp.MIN)
        smin, smax = sums.clone(), sums.clone()
        dist.all_reduce(smin, op=dist.ReduceOp.MIN)
        dist.all_reduce(smax, op=dist.ReduceOp.MAX)
        ok_t *= int(float(smin.item()) == float(smax.item()))  # every rank holds the same gathered cloud
    if int(ok_t.item()) != 1:
        raise RuntimeError("the exchanges disagree (NCCL all-gather / copy-engine push / fused push kernel), or ranks "
                           "hold different clouds")
    points_all = sum(c_n)
    del a, b, d, own

    def timed(fn, K, W=3, after=None):
        for _ in range(W):
            fn()
        if after:
            after()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(K):
            fn()
        if after:
            after()
        e1.record(stream)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / K, (t0, t1)

    l0 = ctx.launch_count
    ms_compute, w_c = timed(compute, steps)
    res = {}
    win = [w_c]
    slot_bytes = 16 + cap * 16
    variants = (("nccl", exch(R.EXCHANGE_NCCL), drain, True), ("copy", exch(R.EXCHANGE_COPY), drain, True),
                ("push", exch_push, None, False))
    for name, exf, after, overlapped in variants:
        ms_ex, w1 = timed(exf, steps, after=after)

        def full(exf=exf):
            compute()
            exf()

        ms_step, w2 = timed(full, steps, after=after)
        win += [w1, w2]
        recv_real = (points_all - kept) * 16
        recv_moved = recv_real if name == "push" else (world - 1) * slot_bytes
        res[name] = {"ms_per_step": ms_step, "exchange_ms": ms_ex, "overlapped_with_next_batch": overlapped,
                     "mpoints_s": world * S * N / (ms_step * 1e-3) / 1e6,
                     "payload_bytes_received_per_rank": recv_moved, "real_bytes_received_per_rank": recv_real,
                     "exchange_gbs_in_per_rank": (recv_moved / (ms_ex * 1e-3) / 1e9) if world > 1 else None,
                     "hidden_fraction_of_exchange": (max(0.0, min(1.0, (ms_compute + ms_ex - ms_step) / ms_ex))
                                                     if ms_ex > 0 else None)}
    launches = ctx.launch_count - l0
    t_lo, t_hi = min(w[0] for w in win), max(w[1] for w in win)
    sampler.window(t_lo, t_hi, "cloud leg")
    pts_step = S * N
    peak, peak_src = measured_peak()
    rho = kept / pts_step
    alg = (8 + 16 * rho) * pts_step
    best = min(res, key=lambda k: res[k]["ms_per_step"])
    out = {
        "workload": (f"PointCloud2 path: {CLOUD_STREAMS_PER_GPU} S3 streams per GPU x {CLOUD_SCANS_PER_STREAM} scans x {N} nodes "
                     f"(synthetic variant 4 'room'), window [0.15, 40] m, polar->xyz, 5 cm voxel grid"
                     f"{', SOR k=%d' % sor if sor else ''}, fused per-GPU cloud, one all-gather per step"),
        "n_gpus": world, "streams_total": streams_total, "steps": steps,
        "impl": best, "ms_per_step": res[best]["ms_per_step"], "mpoints_s": res[best]["mpoints_s"],
        "exchange_ms": res[best]["exchange_ms"], "payload_bytes": res[best]["payload_bytes_received_per_rank"],
        "compute_ms": ms_compute, "compute_mpoints_s_per_gpu": pts_step / (ms_compute * 1e-3) / 1e6,
        "rho_after_voxel": rho, "points_out_per_gpu": kept, "points_gathered": points_all,
        "exchanges_bit_identical": True, "by_exchange": res,
        "roofline": {"bound": "hbm", "kernels": "scan_small_kernel<cloud, post> (window + xyz + SOR + voxel in shared memory)",
                     "algorithmic_bytes_per_step": alg, "bytes_per_point": f"8 B read + 16 B x rho ({rho:.3f}) written",
                     "achieved": alg / (ms_compute * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": alg / (ms_compute * 1e-3) / 1e9 / peak, "peak_source": peak_src},
        "nvlink": ({"limiting_collective": "all-gather of the fused cloud: every rank receives the (world-1) other ranks' "
                                           "points, so bytes in per rank grow with N while the per-GPU compute does not",
                    "gbs_in_per_rank": res[best]["exchange_gbs_in_per_rank"], "peak_gbs_per_direction": 900.0,
                    "step_floor_ms_at_900gbs": (world - 1) * slot_bytes / 900e9 * 1e3}
                   if world > 1 else None),
        "gpu_launches": launches, "clocks": sampler.summary_for(t_lo, t_hi),
    }
    g_push.close()
    ex.close()
    ctx.close()
    return out


class _DevView:
    """A raw device address seen through __cuda_array_interface__ (zero-copy torch view)."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}


def cloud_cpu_baseline(sor):
    """The cloud definition (oracle/cloud_oracle.cpp, a self-authored port: the reference has no PointCloud2 code)
    on the host cores: a bounded sample of the same synthetic streams, one revolution per task."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import pyoracle as O

    O.build(ref=False)
    cores, cores_how = effective_cores()
    n_scans = max(256, 8 * cores)
    nodes = O.synth_batch(0, n_scans, CLOUD_NODES, 4)
    prm = O.cloud_params(range_min=0.15, range_max=40.0, voxel_size=0.05, sor_k=sor, sor_alpha=1.0)
    t0 = time.perf_counter()
    for i in range(16):
        O.cloud(nodes[i], prm)
    one = 16 * CLOUD_NODES / (time.perf_counter() - t0) / 1e6
    with ThreadPoolExecutor(cores) as ex:
        list(ex.map(lambda i: O.cloud(nodes[i], prm), range(min(n_scans, 2 * cores))))  # warm
        t0 = time.perf_counter()
        reps = 0
        while time.perf_counter() - t0 < 8.0:
            list(ex.map(lambda i: O.cloud(nodes[i], prm), range(n_scans)))
            reps += 1
        dt = time.perf_counter() - t0
    return {"value": reps * n_scans * CLOUD_NODES / dt / 1e6, "unit": UNIT, "cores": cores, "cores_how": cores_how,
            "kind": "port", "value_1thread": one,
            "sample": f"{reps} x {n_scans} revolutions x {CLOUD_NODES} nodes through oracle/cloud_oracle.cpp "
                      f"(window, sort, polar->xyz, voxel{', SOR' if sor else ''}), one revolution per task, {cores} threads"}


def run_cloud(args, rank, local_rank, world):
    """`--workload cloud [--sor k]`: the PointCloud2 leg on its own JSON line (the default run carries the same
    object under extra.cloud)."""
    import torch
    import torch.distributed as dist

    import rplidar_ros2_driver_b200 as R

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = numa_pin(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    uuid = None
    try:
        uuid = str(torch.cuda.get_device_properties(dev).uuid)
    except Exception:
        pass
    sampler = ClockSampler(uuid, local_rank)
    sampler.start()
    c = cloud_leg(args, lambda mn, ms: R.Context(local_rank, mn, ms), rank, world, dev, stream, sampler, args.steps,
                  barrier, max_over_ranks, sor=args.sor)
    sampler.stop()
    numa_unpin(numa)
    cpu = cloud_cpu_baseline(args.sor) if (rank == 0 and world == 1 and not args.no_cpu) else None
    if rank == 0:
        line = {
            "metric": METRIC, "value": c["mpoints_s"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": 3, "ms_per_step": c["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": c["workload"], "streams_total": c["streams_total"],
                       "parallelism": f"{world} ranks x {CLOUD_STREAMS_PER_GPU} streams, one all-gather of the fused cloud per step ({c['impl']})",
                       "l2": "inputs 419 MB + outputs per step exceed the 126 MB L2"},
            "roofline": dict(c["roofline"], traffic=None), "cpu_baseline": cpu, "e2e": None,
            "gpu_launches": c["gpu_launches"], "clocks": c["clocks"],
            "extra": {k: v for k, v in c.items() if k not in ("roofline", "clocks", "workload")},
        }
        line["extra"]["numa"] = {k: v for k, v in numa.items() if not k.startswith("_")}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ---- synthetic wire input for the decode / chain workloads (the oracle is only their CPU baseline) ----------
WIRE_CAPSULE = {0x82: (84, 32), 0x83: (781, 96), 0x84: (132, 96), 0x85: (84, 40), 0x86: (170, 64)}  # bytes, nodes


def wire_seal_capsules(fmt: int, payload: np.ndarray, start_q6=None, sync=None) -> np.ndarray:
    """Well-formed capsules from [n, capsule bytes] payload bytes: start angle / scan-start bit, sync markers and
    checksum (XOR of bytes 2.., split over the low nibbles of bytes 0 and 1; CRC-32 with the SDK's zero padding
    for 0x83)."""
    import zlib

    cb = WIRE_CAPSULE[fmt][0]
    caps = np.ascontiguousarray(payload, dtype=np.uint8).reshape(-1, cb).copy()
    if fmt == 0x83:
        caps[:, 0] = 0xA5
        pad = b"\0" * (4 - ((cb - 4) & 3))
        for j in range(caps.shape[0]):
            crc = zlib.crc32(caps[j, : cb - 4].tobytes() + pad) & 0xFFFFFFFF
            caps[j, cb - 4:] = np.frombuffer(np.uint32(crc).tobytes(), np.uint8)
        return caps
    off = 8 if fmt == 0x86 else 2
    if start_q6 is not None:
        word = (np.asarray(start_q6, dtype=np.uint32) & 0x7FFF) | (np.asarray(sync, dtype=np.uint32) << 15)
        caps[:, off] = word & 0xFF
        caps[:, off + 1] = word >> 8
    chk = np.bitwise_xor.reduce(caps[:, 2:], axis=1)
    caps[:, 0] = 0xA0 | (chk & 0xF)
    caps[:, 1] = 0x50 | (chk >> 4)
    return caps


def wire_dense_capsules(start_q6, sync, dist) -> np.ndarray:
    """Dense (0x85) capsules: start_q6 [n], sync [n] bool, dist [n, 40] u16."""
    n = len(start_q6)
    payload = np.zeros((n, 84), np.uint8)
    d = np.asarray(dist, dtype=np.uint16).reshape(n, 40)
    payload[:, 4::2] = d & 0xFF
    payload[:, 5::2] = d >> 8
    return wire_seal_capsules(0x85, payload, start_q6, sync)


def run_decode(args, rank, local_rank, world):
    """SURVEY.md 8(f) rank 1: dense-capsule decode, 512 streams x 4096 framed capsules per GPU."""
    import torch
    from concurrent.futures import ThreadPoolExecutor

    import rplidar_ros2_driver_b200 as R
    from oracle import pyoracle as O  # cpu_baseline leg only

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    n_streams, n_caps, distinct = 512, 4096, 16
    rng = np.random.default_rng(1 + rank)
    host = []
    for sidx in range(distinct):
        ang = (rng.uniform(0, 360) + np.arange(n_caps) * 4.5 + rng.normal(0, 0.03, n_caps)) % 360.0
        q6 = np.round(ang * 64).astype(np.uint32) % (360 * 64)
        dist = rng.integers(1, 40000, (n_caps, 40))
        dist[rng.random((n_caps, 40)) < 0.05] = 0
        sync = np.zeros(n_caps, bool)
        sync[::80] = True
        host.append(wire_dense_capsules(q6, sync, dist))
    host = np.stack(host)
    ctx = R.Context(local_rank, 8192, 1)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream
    caps = torch.from_numpy(np.tile(host, (n_streams // distinct, 1, 1))).to(dev)
    counts = torch.full((n_streams,), n_caps, dtype=torch.int32, device=dev)
    nodes = torch.empty((n_streams, n_caps * 40, 8), dtype=torch.uint8, device=dev)
    ncount = torch.zeros(n_streams, dtype=torch.int32, device=dev)

    def step():
        ctx.decode_dense_batch_dev(caps.data_ptr(), counts.data_ptr(), n_streams, n_caps, 31, nodes.data_ptr(),
                                   ncount.data_ptr(), stream=sp)

    W = max(args.warmup, 3)
    for _ in range(W):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ctx.launch_count
    sampler = start_sampler(dev, local_rank)
    tw0 = time.perf_counter()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    tw1 = time.perf_counter()
    sampler.stop()
    clocks = sampler.summary_for(tw0, tw1)
    ms = e0.elapsed_time(e1) / args.steps
    pts = int(ncount.sum().item())
    peak, peak_src = measured_peak()
    alg = n_streams * n_caps * 84 + pts * 8
    # CPU: the oracle's decode loop, one stream per task
    cores, _cores_how = effective_cores()
    t0 = time.perf_counter()
    O.dense_decode(host[0], 31, 0)
    t_one = time.perf_counter() - t0
    reps = max(cores, 32)
    with ThreadPoolExecutor(cores) as ex:
        t0 = time.perf_counter()
        list(ex.map(lambda i: O.dense_decode(host[i % distinct], 31, 0), range(reps)))
        t_all = time.perf_counter() - t0
    pts_stream = pts / n_streams
    line = {
        "metric": "Mpoints/s through dense-capsule decode (wire capsules -> HQ nodes)", "value": pts / (ms * 1e-3) / 1e6,
        "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": W, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": f"dense-capsule decode: {n_streams} streams x {n_caps} framed 84-byte capsules, scan start "
                               f"every 80 capsules (3200 points per revolution), 5% zero distances",
                   "l2": "176 MB of capsules in + 671 MB of nodes out per step exceed the 126 MB L2"},
        "roofline": {"bound": "hbm", "kernel": "decode_dense_kernel", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak,
                     "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg, "bytes_per_point": alg / pts},
        "cpu_baseline": {"value": reps * pts_stream / t_all / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{reps} streams x {n_caps} capsules through the oracle port of "
                                   f"UnpackerHandler_DenseCapsuleNode (validated against the compiled SDK unpacker)",
                         "value_1thread": pts_stream / t_one / 1e6},
        "e2e": None, "gpu_launches": ctx.launch_count - l0, "clocks": clocks,
    }
    print(json.dumps(line), flush=True)
    ctx.close()


def run_decode_format(args, rank, local_rank, world):
    """SURVEY.md 8(f) rank 1, the other answer formats: 512 streams per GPU, ~12 MB of wire bytes each
    in total; random payload bits, plausible start angles (see tests/test_capsule_oracle_vs_ref.py)."""
    import torch
    from concurrent.futures import ThreadPoolExecutor

    import rplidar_ros2_driver_b200 as R
    from oracle import pyoracle as O  # cpu_baseline leg only

    fmt = int(args.format, 0)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    names = {0x81: "standard nodes (UnpackerHandler_NormalNode)", 0x82: "express capsules (UnpackerHandler_CapsuleNode)",
             0x83: "HQ capsules (UnpackerHandler_HQNode)", 0x84: "ultra capsules (UnpackerHandler_UltraCapsuleNode)",
             0x86: "ultra-dense capsules (UnpackerHandler_UltraDenseCapsuleNode)"}
    kernels = {0x81: "decode_normal_kernel", 0x82: "decode_capsule_kernel<express>", 0x83: "decode_hq_kernel",
               0x84: "decode_capsule_kernel<ultra>", 0x86: "decode_capsule_kernel<ultra-dense>"}
    n_streams, distinct = 512, 16
    rng = np.random.default_rng(1 + rank)
    ctx = R.Context(local_rank, 8192, 1)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream
    if fmt == 0x81:
        n_rec = 65536
        host = []
        for _ in range(distinct):
            rec = np.zeros((n_rec, 5), np.uint8)
            s1 = (np.arange(n_rec) % 360 == 0).astype(np.uint8)
            rec[:, 0] = (rng.integers(0, 64, n_rec).astype(np.uint8) << 2) | ((1 - s1) << 1) | s1
            w = ((((np.arange(n_rec) % 360) * 64).astype(np.uint16)) << 1) | 1
            rec[:, 1], rec[:, 2] = w & 0xFF, w >> 8
            rec[:, 3:] = rng.integers(0, 256, (n_rec, 2))
            host.append(rec.reshape(-1))
        host = np.stack(host)
        stride = host.shape[1]
        wire = torch.from_numpy(np.tile(host, (n_streams // distinct, 1))).to(dev)
        counts = torch.full((n_streams,), stride, dtype=torch.int32, device=dev)
        nodes = torch.empty((n_streams, stride // 5, 8), dtype=torch.uint8, device=dev)
        ncount = torch.zeros(n_streams, dtype=torch.int32, device=dev)
        wire_bytes = n_streams * stride

        def step():
            ctx.decode_normal_batch_dev(wire.data_ptr(), counts.data_ptr(), n_streams, stride, nodes.data_ptr(),
                                        ncount.data_ptr(), stream=sp)

        cpu_one = lambda i: O.decode_normal(host[i % distinct])
        shape = f"{n_streams} streams x {n_rec} five-byte records"
    else:
        cb, per = WIRE_CAPSULE[fmt]
        n_caps = {0x82: 4096, 0x83: 512, 0x84: 2048, 0x86: 2048}[fmt]
        host = []
        for _ in range(distinct):
            payload = rng.integers(0, 256, (n_caps, cb), dtype=np.uint8)
            if fmt == 0x83:
                host.append(wire_seal_capsules(fmt, payload))
                continue
            step_deg = 360.0 * per / 3200.0  # 3200 points per revolution
            ang = (rng.uniform(0, 360) + np.arange(n_caps) * step_deg + rng.normal(0, 0.03, n_caps)) % 360.0
            q6 = np.round(ang * 64).astype(np.uint32) % (360 * 64)
            sync = np.zeros(n_caps, bool)
            sync[0] = True
            host.append(wire_seal_capsules(fmt, payload, q6, sync))
        host = np.stack(host)
        wire = torch.from_numpy(np.tile(host, (n_streams // distinct, 1, 1))).to(dev)
        counts = torch.full((n_streams,), n_caps, dtype=torch.int32, device=dev)
        nodes = torch.empty((n_streams, n_caps * per, 8), dtype=torch.uint8, device=dev)
        ncount = torch.zeros(n_streams, dtype=torch.int32, device=dev)
        wire_bytes = n_streams * n_caps * cb

        def step():
            ctx.decode_capsules_batch_dev(fmt, wire.data_ptr(), counts.data_ptr(), n_streams, n_caps, 31,
                                          nodes.data_ptr(), ncount.data_ptr(), stream=sp)

        cpu_one = lambda i: O.decode_capsules(fmt, host[i % distinct], 31)
        shape = f"{n_streams} streams x {n_caps} framed {cb}-byte capsules ({per} points each)"
    W = max(args.warmup, 3)
    for _ in range(W):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ctx.launch_count
    sampler = start_sampler(dev, local_rank)
    tw0 = time.perf_counter()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    tw1 = time.perf_counter()
    sampler.stop()
    clocks = sampler.summary_for(tw0, tw1)
    ms = e0.elapsed_time(e1) / args.steps
    pts = int(ncount.sum().item())
    peak, peak_src = measured_peak()
    alg = wire_bytes + pts * 8
    cores, _cores_how = effective_cores()
    t0 = time.perf_counter()
    cpu_one(0)
    t_one = time.perf_counter() - t0
    reps = max(cores, 32)
    with ThreadPoolExecutor(cores) as ex:
        t0 = time.perf_counter()
        list(ex.map(cpu_one, range(reps)))
        t_all = time.perf_counter() - t0
    pts_stream = pts / n_streams
    line = {
        "metric": f"Mpoints/s through answer-type {fmt:#x} decode (wire bytes -> HQ nodes)",
        "value": pts / (ms * 1e-3) / 1e6, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": W,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
        "data": "synthetic",
        "config": {"workload": f"{names[fmt]}: {shape}, random payload bits",
                   "l2": f"{wire_bytes / 1e6:.0f} MB in + {pts * 8 / 1e6:.0f} MB out per step exceed the 126 MB L2"},
        "roofline": {"bound": "hbm", "kernel": kernels[fmt], "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak,
                     "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg, "bytes_per_point": alg / max(pts, 1)},
        "cpu_baseline": {"value": reps * pts_stream / t_all / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{reps} streams through the oracle port (validated against the compiled SDK "
                                   f"unpacker)", "value_1thread": pts_stream / t_one / 1e6},
        "e2e": None, "gpu_launches": ctx.launch_count - l0, "clocks": clocks,
    }
    print(json.dumps(line), flush=True)
    ctx.close()


def run_chain(args, rank, local_rank, world):
    """Wire bytes -> LaserScan on the device: dense-capsule decode -> scan assembly -> scan kernel, three
    launches per step and no host round trip (SURVEY.md 8(f) rank 1 + 2 + the hot path)."""
    import torch

    import rplidar_ros2_driver_b200 as R
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    n_streams, n_caps, distinct, max_nodes, max_scans = 512, 4096, 16, 4096, 56
    rng = np.random.default_rng(1 + rank)
    host = []
    for sidx in range(distinct):
        ang = (rng.uniform(0, 360) + np.arange(n_caps) * 4.5 + rng.normal(0, 0.03, n_caps)) % 360.0
        q6 = np.round(ang * 64).astype(np.uint32) % (360 * 64)
        dist = rng.integers(1, 40000, (n_caps, 40))
        dist[rng.random((n_caps, 40)) < 0.05] = 0
        sync = np.zeros(n_caps, bool)
        sync[0] = True
        host.append(wire_dense_capsules(q6, sync, dist))
    host = np.stack(host)
    NS = n_streams * max_scans
    ctx = R.Context(local_rank, max_nodes, NS)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream
    caps = torch.from_numpy(np.tile(host, (n_streams // distinct, 1, 1))).to(dev)
    ccounts = torch.full((n_streams,), n_caps, dtype=torch.int32, device=dev)
    nodes = torch.empty((n_streams, n_caps * 40, 8), dtype=torch.uint8, device=dev)
    ncount = torch.zeros(n_streams, dtype=torch.int32, device=dev)
    status = torch.zeros((n_streams, n_caps), dtype=torch.int32, device=dev)
    offs = torch.zeros((n_streams, n_caps), dtype=torch.int32, device=dev)
    scans = torch.zeros((NS if args.chain_copy else 1, max_nodes, 8), dtype=torch.uint8, device=dev)
    views = torch.zeros((NS, 2), dtype=torch.int32, device=dev)
    starts = torch.zeros((n_streams, 128), dtype=torch.int32, device=dev)
    scnt = torch.zeros(n_streams, dtype=torch.int32, device=dev)
    slen = torch.zeros(NS, dtype=torch.int32, device=dev)
    sps = torch.zeros(n_streams, dtype=torch.int32, device=dev)
    ranges = torch.empty((NS, max_nodes), dtype=torch.float32, device=dev)
    intens = torch.empty((NS, max_nodes), dtype=torch.float32, device=dev)
    beams = torch.zeros(NS, dtype=torch.int32, device=dev)
    inc = torch.zeros(NS, dtype=torch.float32, device=dev)
    params = R.scan_params(1, 0, 0, 1)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]

    def step(timed=False):
        if timed:
            ev[0].record(stream)
        ctx.decode_dense_batch_dev(caps.data_ptr(), ccounts.data_ptr(), n_streams, n_caps, 31, nodes.data_ptr(),
                                   ncount.data_ptr(), capsule_status=status.data_ptr(),
                                   capsule_node_offset=offs.data_ptr(), stream=sp,
                                   scan_starts=None if args.chain_copy else starts.data_ptr(), starts_stride=128,
                                   scan_start_counts=None if args.chain_copy else scnt.data_ptr())
        if timed:
            ev[1].record(stream)
        if args.chain_copy:
            ctx.assemble_scans_dev(nodes.data_ptr(), ncount.data_ptr(), n_streams, n_caps * 40, max_nodes, max_scans,
                                   max_nodes, scans.data_ptr(), slen.data_ptr(), sps.data_ptr(),
                                   capsule_status=status.data_ptr(), capsule_node_offset=offs.data_ptr(),
                                   capsule_counts=ccounts.data_ptr(), stride_capsules=n_caps, stream=sp)
        else:  # no copy: the revolutions are handed on as views into the decoded stream
            ctx.assemble_scan_views_starts_dev(nodes.data_ptr(), ncount.data_ptr(), n_streams, n_caps * 40,
                                               starts.data_ptr(), 128, scnt.data_ptr(), max_nodes, max_scans,
                                               views.data_ptr(), slen.data_ptr(), sps.data_ptr(),
                                               capsule_status=status.data_ptr(), capsule_node_offset=offs.data_ptr(),
                                               capsule_counts=ccounts.data_ptr(), stride_capsules=n_caps, stream=sp)
        if timed:
            ev[2].record(stream)
        if args.chain_copy:
            ctx.scan_batch_dev(scans.data_ptr(), slen.data_ptr(), NS, max_nodes, params, ranges=ranges.data_ptr(),
                               intensities=intens.data_ptr(), beam_counts=beams.data_ptr(),
                               angle_increment=inc.data_ptr(), stream=sp)
        else:
            ctx.scan_views_dev(nodes.data_ptr(), n_streams * n_caps * 40, views.data_ptr(), NS, max_nodes, params,
                               ranges=ranges.data_ptr(), intensities=intens.data_ptr(), beam_counts=beams.data_ptr(),
                               angle_increment=inc.data_ptr(), stream=sp)
        if timed:
            ev[3].record(stream)

    W = max(args.warmup, 3)
    for _ in range(W):
        step()
    torch.cuda.synchronize()
    step(True)
    torch.cuda.synchronize()
    parts = [ev[i].elapsed_time(ev[i + 1]) for i in range(3)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ctx.launch_count
    sampler = start_sampler(dev, local_rank)
    tw0 = time.perf_counter()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    tw1 = time.perf_counter()
    sampler.stop()
    clocks = sampler.summary_for(tw0, tw1)
    ms = e0.elapsed_time(e1) / args.steps
    pts = int(slen.sum().item())      # nodes that reached a published scan
    n_scans = int(sps.sum().item())
    peak, peak_src = measured_peak()
    wire = n_streams * n_caps * 84
    # decode out; assemble: flag pass in (+ copy in+out in copy mode); scan in + out
    alg = wire + int(ncount.sum().item()) * (8 + (8 if args.chain_copy else 0)) + pts * ((8 + 8 if args.chain_copy else 0) + 8 + 8)
    # ---- e2e: the same chain through the host-buffer call rpl_chain_dense_laserscan (pinned buffers) ---------
    e2e = None
    if not args.no_e2e:
        out_nodes, out_scans = 3328, int(max(1, int(sps.max().item())))  # tight output slots: D2H is what the link carries
        ectx = R.Context(local_rank, out_nodes, 64 * out_scans)
        h_caps_t = torch.empty((n_streams, n_caps, 84), dtype=torch.uint8, pin_memory=True)
        h_caps_t.copy_(caps)
        ens = n_streams * out_scans
        outs_t = {"ranges": torch.empty((ens, out_nodes), dtype=torch.float32, pin_memory=True),
                  "intensities": torch.empty((ens, out_nodes), dtype=torch.float32, pin_memory=True)}
        outs = {k: v.numpy() for k, v in outs_t.items()}
        hcc = np.full(n_streams, n_caps, np.uint32)
        for _ in range(2):
            res = ectx.chain_dense_laserscan(h_caps_t.numpy(), hcc, params, out_nodes, out_scans, out=outs)
        ke = max(3, min(args.steps, 8))
        t0 = time.perf_counter()
        for _ in range(ke):
            res = ectx.chain_dense_laserscan(h_caps_t.numpy(), hcc, params, out_nodes, out_scans, out=outs)
        dt = time.perf_counter() - t0
        epts = int(res["beam_counts"].sum())  # measured points that reached a LaserScan
        same = int(res["scans_per_stream"].sum()) == n_scans
        e2e = {"value": pts * ke / dt / 1e6, "unit": UNIT, "h2d_bytes_per_step": n_streams * n_caps * 84 + n_streams * 4,
               "d2h_bytes_per_step": 2 * ens * out_nodes * 4 + 2 * ens * 4 + n_streams * 4, "steps": ke,
               "ms_per_step": dt / ke * 1e3, "api": "rpl_chain_dense_laserscan (pinned host buffers)",
               "scans_match_device_path": same, "beams_out": epts,
               "h2d_bytes_per_point": n_streams * n_caps * 84 / pts, "d2h_bytes_per_point": 2 * ens * out_nodes * 4 / pts}
        ectx.close()
    # ---- cpu baseline: the same chain with the oracle ports (decode, assembly) and the reference's own
    # ascendScanData + publish_scan, one stream per task ---------------------------------------------------------
    cpu = None
    if not args.no_cpu:
        from concurrent.futures import ThreadPoolExecutor

        from oracle import pyoracle as O

        O.build(ref=False)
        cores, cores_how = effective_cores()
        prm = O.scan_params(1, 0, 0, 1, 40.0, 0.1)

        def cut_stream(i):  # oracle ports: pure functions, safe to run side by side
            en, es, eo, _ = O.dense_decode(host[i % distinct], 31, 0)
            e, elen, ek = O.assemble_scans(en, O.resets_from_capsules(es, eo), max_nodes, max_scans)
            k = min(ek, max_scans)
            return np.ascontiguousarray(e[:k]), elen[:k].astype(np.uint32)

        def publish(parts, threads):  # the reference's own ascend + publish_scan over all revolutions (its worker pool)
            nodes_c = np.ascontiguousarray(np.concatenate([p_[0] for p_ in parts]))
            lens_c = np.concatenate([p_[1] for p_ in parts])
            if O.have_ref_node():
                O.ref_pipeline_batch(nodes_c, lens_c, prm, threads=threads, outputs=False)
            else:
                O.pipeline_batch(nodes_c.copy(), lens_c, prm, stable=False, threads=threads)
            return int(lens_c.sum())

        publish([cut_stream(0)], 1)
        t0 = time.perf_counter()
        p1 = publish([cut_stream(1)], 1)
        t_one = time.perf_counter() - t0
        reps = max(2 * cores, 32)
        with ThreadPoolExecutor(cores) as ex:
            t0 = time.perf_counter()
            cut = list(ex.map(cut_stream, range(reps)))
            ptsc = publish(cut, cores)
            t_all = time.perf_counter() - t0
        cpu = {"value": ptsc / t_all / 1e6, "unit": UNIT, "cores": cores, "cores_how": cores_how,
               "kind": "reference" if O.have_ref_node() else "port",
               "sample": f"{reps} streams x {n_caps} capsules: oracle ports of the dense decoder and the scan holder (validated "
                         f"against the compiled SDK), then the reference's own ascendScanData + publish_scan per revolution; "
                         f"one stream per task, {cores} threads", "value_1thread": p1 / t_one / 1e6}
    line = {
        "metric": "Mpoints/s wire capsules -> LaserScan (decode + scan assembly + scan kernel on the device)",
        "value": pts / (ms * 1e-3) / 1e6, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": W,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32+f32",
        "data": "synthetic",
        "config": {"workload": f"{n_streams} streams x {n_caps} dense capsules -> {n_scans} revolutions of ~3200 nodes, "
                               f"Mode B, angle_compensate on; "
                               + ("revolutions copied out by the assembler" if args.chain_copy else
                                  "revolutions read in place through views, scan starts handed over by the decoder (rpl_decode_dense_batch_starts_dev + rpl_assemble_scan_views_starts_dev + rpl_scan_views_dev)"),
                   "l2": "every stage streams > 126 MB"},
        "roofline": {"bound": "hbm", "kernel": "decode_dense + assemble + scan", "achieved": alg / (ms * 1e-3) / 1e9,
                     "peak": peak, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak, "traffic": None,
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": alg},
        "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": ctx.launch_count - l0, "clocks": clocks,
        "extra": {"ms_decode": parts[0], "ms_assemble": parts[1], "ms_scan": parts[2], "scans_published": n_scans,
                  "points_decoded": int(ncount.sum().item())},
    }
    print(json.dumps(line), flush=True)
    ctx.close()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # rank 0's stdout carries exactly one JSON line: NCCL prints its banner ("NCCL version ...") and its
    # diagnostics to stdout whenever NCCL_DEBUG is set (WARN included) -- send them to stderr instead
    # (NCCL honours NCCL_DEBUG_FILE only above the VERSION level, and prints the banner at WARN as well)
    if os.environ.get("NCCL_DEBUG"):
        if os.environ["NCCL_DEBUG"].upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.workload == "cloud":
        run_cloud(args, rank, local_rank, world)
        return
    if args.workload == "chain":
        if rank == 0:
            run_chain(args, rank, local_rank, world)
        return
    if args.workload == "decode":
        if rank == 0:
            if int(args.format, 0) == 0x85:
                run_decode(args, rank, local_rank, world)
            else:
                run_decode_format(args, rank, local_rank, world)
        return
    run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
