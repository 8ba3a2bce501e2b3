#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

  metric   : "compress+decompress MB/s on 1 GiB datagen, bit-exact vs reference"
  workload : configs[1] = level -10 compress + decompress, 1 GiB `datagen -P50`, 128 KiB independent blocks
             (--level 21 / 41 select configs[2] / [3] as the headline instead)
  step     : one pass of the hot path over the batch: compress all 8192 blocks, then decompress them.
  value    : uncompressed MB (10^6 B) per second of that round trip, inputs resident in HBM, CUDA-event timed,
             whole job over all ranks (weak scaling: every rank owns its own 1 GiB shard, no data-path collective).
             Statistic: MEAN over the K timed steps (the reference arm reports the mean of its K passes too).
  e2e      : same round trip through the reference-facing frame API on HOST buffers (LizardF_compressFrame +
             LizardF_decompress, 128 KiB independent blocks, pinned memory): H2D + kernels + D2H inside the timed
             region, wall clock; per-call split, the box's PCIe copy rates and the NUMA node the process was bound to
             are reported next to it; `e2e.with_content_checksum` is the same with contentChecksumFlag = 1 (the CLI default).
  legs     : the other BASELINE levels (configs[2] level -21, configs[3] level -41 decompress) timed kernel-only in the same
             run, each with its own roofline fractions, so that the driver records them.
  one_stream (N > 1, or --mode one-stream): BASELINE configs[4] as stated -- ONE N-GiB stream owned by rank 0, input block
             ranges scattered over NCCL (grouped send/recv), every rank runs the codec on its range, per-block sizes are
             all-gathered, the variable-length outputs are gathered into one concatenated stream on rank 0; then the way
             back.  Collective bytes, per-leg GB/s against NVLink and the limiter are reported.

`--impl reference` times the UNMODIFIED reference (oracle/_ref/liblizard_ref_speed.so, default flags) on the box's
host cores through the pthread harness in oracle/liboracle.so (worker pool created outside the timed passes), same
workload, on every hardware thread this process may use (sched_getaffinity and the cgroup cpu quota, not os.cpu_count()).

One JSON line on stdout (rank 0).
"""
import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BS = 1 << 17
METRIC = "compress+decompress MB/s on 1 GiB datagen, bit-exact vs reference"
# SURVEY.md section 8c: clean-state compressed totals of `datagen -g1G -P50` (seed 0), 8192 x 128 KiB, cap = BS-1
KNOWN_TOTALS_1G = {10: 670259129, 21: 616060194, 41: 385653946}
# dram__bytes_read.sum + dram__bytes_write.sum per launch come from committed `ncu --set full` captures: the newest
# profiles/r*_traffic.json (written by tools/ncu_traffic.py from the .ncu-rep of the build it names).  Never typed in here.
TRAFFIC_FILES = ["profiles/r02_traffic.json"]
NVLINK_GBPS_NOMINAL = 900.0       # per direction per GPU (B200_PROFILING.md)
NVLINK_GBPS_MEASURED = 770.0      # peer copy per direction measured on this pool (B200_PROFILING.md)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--level", type=int, default=10)
    ap.add_argument("--size-mib", type=int, default=1024)
    ap.add_argument("--cpu-sample-mib", type=int, default=64)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--legs", default="10,21,41", help="levels timed kernel-only next to the headline level ('' = none)")
    ap.add_argument("--mode", default="default", choices=["default", "one-stream"],
                    help="one-stream: run the NCCL scatter/gather form also at N = 1 (it always runs at N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy, to compare two builds")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------------------
def host_threads():
    """Hardware threads this process may really use: the scheduler affinity mask, capped by the cgroup CPU quota."""
    info = {"os_cpu_count": os.cpu_count()}
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    info["affinity"] = n
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:              # cgroup v2: "<quota|max> <period>"
            q, p = f.read().split()[:2]
            if q != "max":
                quota = float(q) / float(p)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = int(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                p = int(f.read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    info["cgroup_cpu_quota"] = quota
    if quota is not None:
        n = max(1, min(n, int(math.ceil(quota))))
    info["threads"] = n
    return n, info


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons with nvidia-smi while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                f = [x.strip() for x in line.split(",")]
                if len(f) < 6:
                    continue
                try:
                    self.samples.append(float(f[0]))
                    self.max_mhz = float(f[1])
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def load_checker_libs():
    ref = os.path.join(ROOT, "oracle", "_ref", "liblizard_ref_speed.so")
    orc = os.path.join(ROOT, "oracle", "liboracle.so")
    if not os.path.exists(orc):
        raise RuntimeError("oracle/liboracle.so missing: run __graft_entry__.build()")
    O = ctypes.CDLL(orc)
    O.oracle_time_compress.restype = ctypes.c_double
    O.oracle_time_compress.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int,
                                       ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    O.oracle_time_decompress.restype = ctypes.c_double
    O.oracle_time_decompress.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t,
                                         ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    O.oracle_time_last_mean.restype = ctypes.c_double
    if os.path.exists(ref):
        R = ctypes.CDLL(ref)
        cfn = ctypes.cast(R.Lizard_compress, ctypes.c_void_p)
        dfn = ctypes.cast(R.Lizard_decompress_safe, ctypes.c_void_p)
        kind = "reference"
    else:   # the reference did not travel: fall back to our restatement (level coverage is the same)
        cfn = ctypes.cast(O.oracle_Lizard_compress, ctypes.c_void_p)
        dfn = ctypes.cast(O.oracle_Lizard_decompress_safe, ctypes.c_void_p)
        kind = "port"
    return O, cfn, dfn, kind


def cpu_round_trip(O, cfn, dfn, src_ptr, nbytes, level, threads, iters):
    """Times compress and decompress of nbytes (128 KiB blocks) on `threads` host threads.
    Returns {"best": (tc, td), "mean": (tc, td)} seconds per pass, the compressed total and a round-trip check."""
    n = (nbytes + BS - 1) // BS
    stride = BS + 64
    comp = ctypes.create_string_buffer(n * stride)
    back = ctypes.create_string_buffer(n * BS)
    sizes = (ctypes.c_int * n)()
    ctypes.memset(comp, 1, n * stride)      # pre-touch, as programs/bench.c:195,225,260 does
    ctypes.memset(back, 1, n * BS)
    tc = O.oracle_time_compress(cfn, src_ptr, nbytes, BS, level, comp, stride, sizes, threads, iters)
    tc_mean = O.oracle_time_last_mean()
    td = O.oracle_time_decompress(dfn, comp, stride, sizes, n, back, BS, threads, iters)
    td_mean = O.oracle_time_last_mean()
    ok = ctypes.string_at(back, min(nbytes, 1 << 20)) == ctypes.string_at(src_ptr, min(nbytes, 1 << 20))
    return {"best": (tc, td), "mean": (tc_mean, td_mean)}, sum(sizes), ok


# ------------------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    if rank != 0:
        return
    import lizard_b200 as lz
    nbytes = args.size_mib << 20
    buf = ctypes.create_string_buffer(nbytes)
    lz.datagen_into(ctypes.addressof(buf), nbytes, 50.0, 0)
    O, cfn, dfn, kind = load_checker_libs()
    threads, tinfo = host_threads()
    K = max(args.steps, 1)
    for _ in range(max(args.warmup, 1) - 1):
        cpu_round_trip(O, cfn, dfn, ctypes.addressof(buf), min(nbytes, 256 << 20), args.level, threads, 1)
    t0 = time.time()
    t, csum, ok = cpu_round_trip(O, cfn, dfn, ctypes.addressof(buf), nbytes, args.level, threads, K)
    tc, td = t["mean"]
    # one thread on a bounded sample: shows how the box's cores scale (a CPU-starved slice is visible here)
    sample = min(nbytes, 32 << 20)
    t1, _, _ = cpu_round_trip(O, cfn, dfn, ctypes.addressof(buf), sample, args.level, 1, 1)
    one = sample / 1e6 / sum(t1["best"])
    mb = nbytes / 1e6
    value = mb / (tc + td)
    line = {
        "impl": "reference", "metric": METRIC,
        "value": round(value, 1), "unit": "MB/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round((tc + td) * 1e3, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": "level -%d compress + decompress, %d MiB datagen -P50, 128 KiB independent blocks"
                               % (args.level, args.size_mib), "level": args.level, "block": BS,
                   "where": "host CPU, unmodified reference" if kind == "reference" else "host CPU, oracle port",
                   "compress_MBps": round(mb / tc, 1), "decompress_MBps": round(mb / td, 1), "compressed_bytes": csum,
                   "round_trip_ok": bool(ok),
                   "statistic": "mean of %d passes (same statistic as the GPU arm); best pass: %.1f MB/s"
                                % (K, mb / sum(t["best"])),
                   "timing": "CLOCK_MONOTONIC around each pass, worker pool created outside the passes, pre-touched buffers",
                   "host_threads": tinfo,
                   "one_thread_MBps": round(one, 1), "scaling_vs_one_thread": round(value / one, 1)},
        "cpu_baseline": {"value": round(value, 1), "unit": "MB/s", "cores": threads, "kind": kind,
                         "sample": "whole %d MiB buffer, one Lizard_compress/Lizard_decompress_safe call per 128 KiB block, "
                                   "%d pthreads (affinity %s, cgroup quota %s, os.cpu_count %s)"
                                   % (args.size_mib, threads, tinfo["affinity"], tinfo["cgroup_cpu_quota"], tinfo["os_cpu_count"])},
        "e2e": {"value": round(value, 1), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": round(time.time() - t0, 2),
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
def bind_near_gpu(torch, local_rank):
    """Run this process (and therefore place its pinned host buffers, first touch) on the NUMA node the GPU's PCIe
    root hangs off.  Returns the node number or None when the topology cannot be read."""
    try:
        prop = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (prop.pci_domain_id, prop.pci_bus_id, prop.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            return node
    except Exception:
        pass
    return None


def pcie_probe(torch, dev, h_buf):
    """Pinned-memory copy rates of this box's link, GB/s: (H2D alone, D2H alone, both directions at once)."""
    n = min(h_buf.numel(), 256 << 20)
    h_a = h_buf[:n]
    h_b = torch.empty(n, dtype=torch.uint8).pin_memory()
    d_a = torch.empty(n, dtype=torch.uint8, device=dev)
    d_b = torch.zeros(n, dtype=torch.uint8, device=dev)
    s2 = torch.cuda.Stream(device=dev)

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t

    def both():
        with torch.cuda.stream(s2):
            h_b.copy_(d_b, non_blocking=True)
        d_a.copy_(h_a, non_blocking=True)

    t_h2d = timed(lambda: d_a.copy_(h_a, non_blocking=True))
    t_d2h = timed(lambda: h_b.copy_(d_b, non_blocking=True))
    t_both = timed(both)
    return round(n / t_h2d / 1e9, 1), round(n / t_d2h / 1e9, 1), round(2 * n / t_both / 1e9, 1)


def load_traffic():
    for rel in TRAFFIC_FILES:
        try:
            with open(os.path.join(ROOT, rel)) as f:
                return json.load(f), rel
        except Exception:
            continue
    return {}, None


def load_peaks():
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    return hbm_peak, src


DUMP_BLOCKS = 32            # blocks of the sample; with their compressed streams about 34 MB of float32


def dump_outputs(out_dir, torch, d_comp, d_csize, d_back, d_dsize, stride, n):
    """Writes what the last timed step handed a caller of LizardB200_compress_device / _decompress_device: every block's
    compressed and decompressed size, and for a fixed, seeded sample of blocks the compressed stream (zeros behind its
    size) and the decompressed bytes, byte values as float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    pick = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_BLOCKS), replace=False))
    idx = torch.from_numpy(pick).to(d_comp.device)
    csize = d_csize.cpu().numpy()
    comp = d_comp.view(n, stride).index_select(0, idx).cpu().numpy().astype(np.float32)
    comp[np.arange(stride)[None, :] >= np.maximum(csize[pick], 0)[:, None]] = 0.0
    back = d_back.view(n, BS).index_select(0, idx).cpu().numpy().astype(np.float32)
    for name, a in (("compressed_sizes", csize.astype(np.float64)), ("decompressed_sizes", d_dsize.cpu().numpy().astype(np.float64)),
                    ("sample_blocks", pick.astype(np.float64)), ("sample_compressed", comp), ("sample_decompressed", back)):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args, rank, world, local_rank):
    import torch
    import lizard_b200 as lz
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the codec has no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_node = bind_near_gpu(torch, local_rank)
    L = lz.lib()
    st = L.LizardB200_setDevice(local_rank)
    if st != 0:
        raise SystemExit("LizardB200_setDevice failed: %d %s" % (st, L.LizardB200_lastError().decode()))
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)

    nbytes = args.size_mib << 20
    n = nbytes // BS
    level = args.level
    K = args.steps
    W = max(args.warmup, 3)
    # ---- synthetic input: every rank owns one shard (seed = rank), generated straight into pinned memory ----
    h_src = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    lz.datagen_into(h_src.data_ptr(), nbytes, 50.0, rank)
    d_src = h_src.to(dev, non_blocking=True)
    stride = (L.Lizard_compressBound(BS) + 15) // 16 * 16
    d_comp = torch.empty(n * stride, dtype=torch.uint8, device=dev)
    d_back = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    idx = torch.arange(n, dtype=torch.int64, device=dev)
    d_src_off = idx * BS
    d_comp_off = idx * stride
    d_src_len = torch.full((n,), BS, dtype=torch.int32, device=dev)
    d_cap = torch.full((n,), BS - 1, dtype=torch.int32, device=dev)       # the frame layer's capacity (lizard_frame.c:459)
    d_back_cap = torch.full((n,), BS, dtype=torch.int32, device=dev)
    d_csize = torch.zeros(n, dtype=torch.int32, device=dev)
    d_dsize = torch.zeros(n, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)

    def compress(lv):
        s = L.LizardB200_compress_device(d_src.data_ptr(), d_src_off.data_ptr(), d_src_len.data_ptr(), d_comp.data_ptr(),
                                         d_comp_off.data_ptr(), d_cap.data_ptr(), d_csize.data_ptr(), n, lv, sp)
        if s != 0:
            raise SystemExit("compress_device failed: %d %s" % (s, L.LizardB200_lastError().decode()))

    def decompress():
        s = L.LizardB200_decompress_device(d_comp.data_ptr(), d_comp_off.data_ptr(), d_csize.data_ptr(), d_back.data_ptr(),
                                           d_src_off.data_ptr(), d_back_cap.data_ptr(), d_dsize.data_ptr(), n, sp)
        if s != 0:
            raise SystemExit("decompress_device failed: %d %s" % (s, L.LizardB200_lastError().decode()))

    def codec_leg(lv, steps, warm, barrier):
        """warm-up + correctness of what will be timed, then exactly `steps` steps between CUDA events."""
        for _ in range(warm):
            compress(lv)
            d_back.zero_()
            decompress()
        torch.cuda.synchronize()
        csize = d_csize.cpu()
        if int((csize <= 0).sum()) != 0:
            raise SystemExit("bench.py: level %d: %d blocks failed to compress" % (lv, int((csize <= 0).sum())))
        comp_total = int(csize.sum())
        if not torch.equal(d_back, d_src) or int((d_dsize != BS).sum()) != 0:
            raise SystemExit("bench.py: level %d: round trip mismatch" % lv)
        if rank == 0 and nbytes == (1 << 30) and lv in KNOWN_TOTALS_1G and comp_total != KNOWN_TOTALS_1G[lv]:
            raise SystemExit("bench.py: level %d compressed total %d != reference clean-state total %d"
                             % (lv, comp_total, KNOWN_TOTALS_1G[lv]))
        launches0 = L.LizardB200_launchCount()
        if barrier and dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
        for k in range(steps):
            ev[k][0].record(stream)
            compress(lv)
            ev[k][1].record(stream)
            decompress()
            ev[k][2].record(stream)
        torch.cuda.synchronize()
        if barrier and dist is not None:
            dist.barrier()
        t_c = sum(ev[k][0].elapsed_time(ev[k][1]) for k in range(steps)) / 1e3
        t_d = sum(ev[k][1].elapsed_time(ev[k][2]) for k in range(steps)) / 1e3
        return t_c, t_d, comp_total, L.LizardB200_launchCount() - launches0

    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    # ---- headline: timed region of exactly K steps, CUDA events on the launching stream, barrier + sync on both sides ----
    t_c, t_d, comp_total, launches = codec_leg(level, K, W, True)
    if args.dump_outputs and rank == 0:                 # before the other levels reuse the buffers
        dump_outputs(args.dump_outputs, torch, d_comp, d_csize, d_back, d_dsize, stride, n)

    # ---- the other BASELINE levels, kernel-only, same buffers (configs[2] level -21, configs[3] level -41) ----
    leg_levels = [int(x) for x in args.legs.split(",") if x.strip()] if args.legs else []
    legs_raw = {}
    for lv in leg_levels:
        if lv == level:
            continue
        ks = min(K, 5)
        c, d, tot, _ = codec_leg(lv, ks, 2, False)
        legs_raw[lv] = (c / ks, d / ks, tot)
    if legs_raw:                                     # leave the headline level's streams in d_comp
        compress(level)
        torch.cuda.synchronize()

    # ---- end to end through the host-buffer C-ABI (pinned host memory in, host memory out) ----
    e2e = None
    e2e_ck = None
    frame_size = 0
    split = [0.0, 0.0]
    if not args.no_e2e:
        # the reference-facing call a user makes: LizardF_compressFrame / LizardF_decompress on HOST buffers
        lz.bind_frame_api(L)
        h_back = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        dctx = ctypes.c_void_p()
        L.LizardF_createDecompressionContext(ctypes.byref(dctx), 100)
        h_frame = None

        def e2e_run(checksum, steps, warm):
            nonlocal h_frame
            prefs = lz.make_prefs(level, 1, True, checksum, 0)      # 128 KiB independent blocks
            cap = L.LizardF_compressFrameBound(nbytes, ctypes.byref(prefs))
            if h_frame is None or h_frame.numel() < cap:
                h_frame = torch.empty(cap, dtype=torch.uint8).pin_memory()
            sp_ = [0.0, 0.0]
            fs_box = [0]

            def step():
                t_a = time.perf_counter()
                fs = L.LizardF_compressFrame(h_frame.data_ptr(), cap, h_src.data_ptr(), nbytes, ctypes.byref(prefs))
                if L.LizardF_isError(fs):
                    raise SystemExit("LizardF_compressFrame: " + L.LizardF_getErrorName(fs).decode())
                so, si = ctypes.c_size_t(nbytes), ctypes.c_size_t(fs)
                t_b = time.perf_counter()
                r = L.LizardF_decompress(dctx, h_back.data_ptr(), ctypes.byref(so), h_frame.data_ptr(), ctypes.byref(si), None)
                sp_[0] += t_b - t_a
                sp_[1] += time.perf_counter() - t_b
                if r != 0 or so.value != nbytes or si.value != fs:
                    raise SystemExit("LizardF_decompress: result %d, out %d, in %d of %d" % (r, so.value, si.value, fs))
                fs_box[0] = fs

            # warm-up; the timed loop follows immediately (an idle gap lets the GPU drop to its idle clocks and the first
            # kernel afterwards runs ~10x slower for tens of ms); the result is verified after the timed loop
            for _ in range(warm):
                step()
            if dist is not None:
                dist.barrier()
            torch.cuda.synchronize()
            sp_[0] = sp_[1] = 0.0
            t0 = time.perf_counter()
            for _ in range(steps):
                step()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if not torch.equal(h_back, h_src):
                raise SystemExit("bench.py: e2e round trip mismatch")
            return dt, fs_box[0], sp_

        e2e, frame_size, split = e2e_run(False, K, W)
        ks = min(K, 5)
        t_ck, _, _ = e2e_run(True, ks, 1)
        e2e_ck = t_ck / ks
        L.LizardF_freeDecompressionContext(dctx)
    clocks = sampler.stop()
    # bare pinned-memory copies, all ranks at the same time: the ceiling the host side gives N concurrent e2e callers
    # (GPUs behind one socket share its DMA / memory bandwidth)
    if dist is not None:
        dist.barrier()
    link = pcie_probe(torch, dev, h_src) if e2e is not None else None

    # ---- BASELINE configs[4] as stated: one stream, NCCL scatter / gather around the codec ----
    one_stream = None
    if world > 1 or args.mode == "one-stream":
        one_stream = run_one_stream(args, torch, dist, lz, L, dev, rank, world, h_src, d_src, level, min(K, 5))

    # ---- max over ranks ----
    times = torch.tensor([t_c, t_d, e2e if e2e is not None else 0.0, e2e_ck if e2e_ck is not None else 0.0],
                         dtype=torch.float64, device=dev)
    totals = torch.tensor([float(comp_total)], dtype=torch.float64, device=dev)
    link_min = torch.tensor(list(link) if link else [0.0, 0.0, 0.0], dtype=torch.float64, device=dev)
    link_sum = link_min.clone()
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        dist.all_reduce(totals, op=dist.ReduceOp.SUM)
        dist.all_reduce(link_min, op=dist.ReduceOp.MIN)
        dist.all_reduce(link_sum, op=dist.ReduceOp.SUM)
    t_c, t_d, t_e, t_eck = [float(x) for x in times.cpu()]
    comp_all = float(totals.cpu()[0])
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    job_bytes = float(nbytes) * world
    mb = job_bytes / 1e6
    value = mb * K / (t_c + t_d)
    ratio = job_bytes / comp_all
    hbm_peak, peak_src = load_peaks()
    traffic_db, traffic_file = load_traffic()

    def roof(t_launch, kernel, lv, rat):
        algo = float(nbytes) * (1.0 + 1.0 / rat)        # one rank's launch: read 1 + write 1/ratio (and the reverse)
        ach = algo / t_launch / 1e9
        ent = traffic_db.get(str(lv), {}).get(kernel) if nbytes == (1 << 30) else None
        r = {"kernel": kernel, "bound": "hbm", "achieved": round(ach, 1), "peak": hbm_peak, "unit": "GB/s",
             "frac": round(ach / hbm_peak, 4), "traffic": ent["traffic"] if ent else None, "peak_source": peak_src,
             "algorithmic_bytes_per_launch": int(algo), "avg_launch_ms": round(t_launch * 1e3, 3)}
        if ent:
            r["traffic_source"] = "%s: %s, build %s" % (traffic_file, ent.get("report"), ent.get("build"))
        return r

    line = {
        "metric": METRIC,
        "value": round(value, 1), "unit": "MB/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": round((t_c + t_d) / K * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "level -%d compress + decompress, %d MiB datagen -P50, 128 KiB independent blocks"
                               % (level, args.size_mib), "level": level, "block": BS, "blocks_per_gpu": n,
                   "sharding": "every GPU owns one %d MiB shard (datagen seed = rank); no data-path collective in `value` "
                               "(see one_stream for the NCCL scatter/gather form)" % args.size_mib,
                   "dst_capacity": BS - 1, "l2": "inputs (1 GiB) larger than L2 (126 MB); no flush needed",
                   "statistic": "mean of %d timed steps" % K,
                   "compress_MBps": round(mb * K / t_c, 1), "decompress_MBps": round(mb * K / t_d, 1),
                   "compressed_bytes": int(comp_all), "ratio": round(ratio, 4),
                   "parity": "in-run check: round trip equal + compressed TOTAL == reference clean-state total (SURVEY 8c); "
                             "bit-exactness per block is pinned by tests/ (-m gpu)"
                             if (nbytes == (1 << 30) and level in KNOWN_TOTALS_1G) else "in-run check: round trip equal"},
        "roofline": roof(t_c / K, "lizard_encode_units_kernel", level, ratio),
        "roofline_decode": roof(t_d / K, "lizard_decode_units_kernel", level, ratio),
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    if legs_raw:
        legs = {}
        for lv, (c, d, tot) in legs_raw.items():
            rat = float(nbytes) / tot
            legs[str(lv)] = {"compress_ms": round(c * 1e3, 3), "decompress_ms": round(d * 1e3, 3),
                             "compress_MBps": round(nbytes / 1e6 / c, 1), "decompress_MBps": round(nbytes / 1e6 / d, 1),
                             "compressed_bytes": tot, "ratio": round(rat, 4),
                             "roofline": roof(c, "lizard_encode_units_kernel", lv, rat),
                             "roofline_decode": roof(d, "lizard_decode_units_kernel", lv, rat)}
        line["legs"] = legs
        line["config"]["legs"] = ("rank 0, kernel-only, same 1 GiB shard, mean of %d steps; level 41 decompress is BASELINE "
                                  "configs[3] (its input is bit-identical to the reference's clean-state stream)" % min(K, 5))
    if e2e is not None:
        line["e2e"] = {"value": round(mb * K / t_e, 1), "unit": "MB/s",
                       "h2d_bytes_per_step": int(nbytes + frame_size), "d2h_bytes_per_step": int(frame_size + nbytes),
                       "api": "LizardF_compressFrame + LizardF_decompress (128 KiB independent blocks), pinned host buffers, "
                              "wall clock, chunked H2D / kernels / D2H overlap", "frame_bytes": int(frame_size),
                       "compress_ms_rank0": round(split[0] / K * 1e3, 2), "decompress_ms_rank0": round(split[1] / K * 1e3, 2),
                       "with_content_checksum": {"value": round(mb / t_eck, 1) if t_eck > 0 else None, "unit": "MB/s",
                                                 "note": "contentChecksumFlag = 1 (XXH32 of all content, the CLI default)"},
                       "pcie_GBps_rank0": {"h2d": link[0], "d2h": link[1], "both_directions_total": link[2]},
                       "pcie_GBps_all_ranks_concurrently": {
                           "slowest_rank": {"h2d": round(float(link_min[0]), 1), "d2h": round(float(link_min[1]), 1),
                                            "both_directions_total": round(float(link_min[2]), 1)},
                           "sum_over_ranks_both_directions": round(float(link_sum[2]), 1)},
                       "host_numa_node_rank0": numa_node}
        # how close the codec calls come to moving their bytes at the bare-copy rate measured under the same concurrency
        moved = 2.0 * (nbytes + frame_size) * world * K
        ceiling = float(link_sum[2]) * 1e9
        if ceiling > 0:
            line["e2e"]["fraction_of_bare_copy_ceiling"] = round(moved / t_e / ceiling, 3)
            line["e2e"]["limiter"] = ("host link: each step moves %.2f GB per GPU across PCIe; bare pinned copies issued by all %d "
                                      "ranks at once reach %.0f GB/s in total (both directions)"
                                      % (2.0 * (nbytes + frame_size) / 1e9, world, float(link_sum[2])))
    if one_stream is not None:
        line["one_stream"] = one_stream
    # ---- CPU side by side (rank 0, N = 1 only): the reference's own code on one host thread, bounded sample ----
    if world == 1:
        try:
            O, cfn, dfn, kind = load_checker_libs()
            sample = min(nbytes, args.cpu_sample_mib << 20)
            t, _, ok = cpu_round_trip(O, cfn, dfn, h_src.data_ptr(), sample, level, 1, 2)
            tc, td = t["best"]
            line["cpu_baseline"] = {"value": round(sample / 1e6 / (tc + td), 1), "unit": "MB/s", "cores": 1, "kind": kind,
                                    "sample": "first %d MiB of the same buffer, per-128-KiB-block calls, best of 2 passes"
                                              % (sample >> 20),
                                    "compress_MBps": round(sample / 1e6 / tc, 1), "decompress_MBps": round(sample / 1e6 / td, 1),
                                    "round_trip_ok": bool(ok)}
        except Exception as ex:   # never lose the GPU line because the checker is missing
            line["cpu_baseline"] = {"value": None, "unit": "MB/s", "cores": 0, "kind": "unavailable", "sample": str(ex)}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------
def run_one_stream(args, torch, dist, lz, L, dev, rank, world, h_src, d_src, level, steps):
    """BASELINE configs[4]: rank 0 owns ONE stream of world x size bytes; scatter -> codec -> all_gather(sizes) -> gather,
    and back.  The stream is the concatenation of the shards the weak-scaling legs use (datagen seed 0 .. world-1, each
    --size-mib), so rank 0 generates it through its pinned buffer.  Times are CUDA events, max over ranks; one JSON object."""
    from lizard_b200 import dist as lzdist
    shard = h_src.numel()
    total = shard * world
    n_blocks = total // BS
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    single = dist is None
    if single:                                          # N = 1: the same code path over a 1-rank gloo/nccl group is pointless;
        import torch.distributed as dist                # run it over a local single-process group so the plumbing is identical
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", str(29400 + os.getpid() % 500))
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    whole = None
    if rank == 0:
        whole = torch.empty(total, dtype=torch.uint8, device=dev)
        whole[:shard].copy_(d_src)
        tmp = torch.empty(shard, dtype=torch.uint8).pin_memory()
        for r in range(1, world):
            lz.datagen_into(tmp.data_ptr(), shard, 50.0, r)
            whole[r * shard:(r + 1) * shard].copy_(tmp, non_blocking=False)
        del tmp
    lo, hi = lzdist.block_range(n_blocks, rank, world)
    n = hi - lo
    stride = (L.Lizard_compressBound(BS) + 15) // 16 * 16
    mine = torch.empty(n * BS, dtype=torch.uint8, device=dev)
    d_comp = torch.empty(n * stride, dtype=torch.uint8, device=dev)
    d_csize = torch.zeros(n, dtype=torch.int32, device=dev)
    idx = torch.arange(n, dtype=torch.int64, device=dev)
    src_off, comp_off = idx * BS, idx * stride
    src_len = torch.full((n,), BS, dtype=torch.int32, device=dev)
    cap = torch.full((n,), BS - 1, dtype=torch.int32, device=dev)
    blob = torch.empty(n * stride, dtype=torch.uint8, device=dev)
    part = torch.empty(n * stride, dtype=torch.uint8, device=dev)
    d_back = torch.empty(n * BS, dtype=torch.uint8, device=dev)
    back_cap = torch.full((n,), BS, dtype=torch.int32, device=dev)
    d_dsize = torch.zeros(n, dtype=torch.int32, device=dev)
    stream_buf = torch.empty(total, dtype=torch.uint8, device=dev) if rank == 0 else None      # concatenated compressed stream
    whole_back = torch.empty(total, dtype=torch.uint8, device=dev) if rank == 0 else None
    names = ["scatter_input", "compress", "pack", "allgather_sizes", "gather_stream", "scatter_stream", "decompress",
             "gather_blocks"]
    acc = {k: 0.0 for k in names}
    info = {}

    def one_pass(record):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
        ev[0].record(stream)
        lzdist.scatter_blocks(whole, total, BS, dev, out=mine)
        ev[1].record(stream)
        s = L.LizardB200_compress_device(mine.data_ptr(), src_off.data_ptr(), src_len.data_ptr(), d_comp.data_ptr(),
                                         comp_off.data_ptr(), cap.data_ptr(), d_csize.data_ptr(), n, level, sp)
        if s != 0:
            raise SystemExit("one_stream: compress_device failed: %d %s" % (s, L.LizardB200_lastError().decode()))
        ev[2].record(stream)
        sizes64 = d_csize.to(torch.int64)
        blob_off = torch.cumsum(sizes64, 0) - sizes64
        s = L.LizardB200_gather_device(d_comp.data_ptr(), comp_off.data_ptr(), d_csize.data_ptr(), blob.data_ptr(),
                                       blob_off.data_ptr(), n, sp)
        if s != 0:
            raise SystemExit("one_stream: gather_device failed: %d %s" % (s, L.LizardB200_lastError().decode()))
        ev[3].record(stream)
        all_sizes, _ = lzdist.exchange_sizes(sizes64, n_blocks)
        ev[4].record(stream)
        one = lzdist.gather_stream(blob, all_sizes, n_blocks, dev, out=stream_buf)
        ev[5].record(stream)
        my_part, my_sizes, lo2, hi2 = lzdist.scatter_stream(one, all_sizes if rank == 0 else None, n_blocks, dev, out=part)
        ev[6].record(stream)
        part_off = torch.cumsum(my_sizes, 0) - my_sizes
        part_len = my_sizes.to(torch.int32)
        s = L.LizardB200_decompress_device(my_part.data_ptr(), part_off.data_ptr(), part_len.data_ptr(), d_back.data_ptr(),
                                           src_off.data_ptr(), back_cap.data_ptr(), d_dsize.data_ptr(), n, sp)
        if s != 0:
            raise SystemExit("one_stream: decompress_device failed: %d %s" % (s, L.LizardB200_lastError().decode()))
        ev[7].record(stream)
        lzdist.gather_blocks(d_back, total, BS, dev, out=whole_back)
        ev[8].record(stream)
        torch.cuda.synchronize()
        if record:
            for i, k in enumerate(names):
                acc[k] += ev[i].elapsed_time(ev[i + 1])
            acc["_total"] = acc.get("_total", 0.0) + ev[0].elapsed_time(ev[8])
        info["compressed"] = int(all_sizes.sum())
        info["min_size"] = int(d_csize.min())
        info["ok_sizes"] = int((d_dsize != BS).sum()) == 0

    one_pass(False)                                     # warm-up (NCCL channels, workspaces)
    dist.barrier()
    torch.cuda.synchronize()
    for _ in range(steps):
        one_pass(True)
    dist.barrier()
    keys = names + ["_total"]
    t = torch.tensor([acc[k] / steps for k in keys], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = dict(zip(keys, [float(x) for x in t.cpu()]))
    ok = None
    if rank == 0:
        ok = bool(torch.equal(whole_back, whole)) and info["ok_sizes"] and info["min_size"] > 0
    if single:
        dist.destroy_process_group()
    if rank != 0:
        return None
    comp = info["compressed"]
    remote = (world - 1) / world                        # share of the bytes that leaves / enters rank 0 over NVLink
    legs = {"scatter_input": total * remote, "gather_stream": comp * remote, "scatter_stream": comp * remote,
            "gather_blocks": total * remote}
    gbps = {k: (round(v / 1e9 / (ms[k] / 1e3), 1) if ms[k] > 0 and v > 0 else None) for k, v in legs.items()}
    coll_ms = sum(ms[k] for k in legs) + ms["allgather_sizes"]
    codec_ms = ms["compress"] + ms["decompress"] + ms["pack"]
    return {
        "workload": "level -%d round trip of ONE %d MiB stream (datagen -P50 shards, seeds 0..%d) owned by rank 0, 128 KiB blocks: "
                    "scatter -> compress -> all_gather(sizes) -> gather stream; scatter stream -> decompress -> gather blocks"
                    % (level, total >> 20, world - 1),
        "n_gpus": world, "steps": steps, "round_trip_ok": ok, "compressed_bytes": comp,
        "value": round(total / 1e6 / (ms["_total"] / 1e3), 1), "unit": "MB/s",
        "ms_per_step": round(ms["_total"], 3), "phases_ms": {k: round(ms[k], 3) for k in names},
        "collective_bytes_per_step": int(sum(legs.values()) + 8 * n_blocks * (world - 1)),
        "leg_GBps_rank0_link": gbps,
        "nvlink_GBps_per_direction": {"nominal": NVLINK_GBPS_NOMINAL, "measured_peer_copy": NVLINK_GBPS_MEASURED},
        "codec_only_MBps": round(total / 1e6 / (codec_ms / 1e3), 1) if codec_ms > 0 else None,
        "limiter": (("rank 0's NVLink port: all {gib} GiB leave and re-enter one GPU ({coll:.1f} ms of {tot:.1f} ms per step in the "
                     "four scatter/gather legs, codec {codec:.1f} ms); the codec legs shrink with N, the rank-0 legs do not"
                     if coll_ms >= codec_ms else
                     "the codec ({codec:.1f} ms of {tot:.1f} ms per step; the scatter/gather legs through rank 0's NVLink port take "
                     "{coll:.1f} ms: all {gib} GiB leave and re-enter one GPU)")
                    .format(gib=total >> 30, coll=coll_ms, tot=ms["_total"], codec=codec_ms)) if world > 1 else
                   "single GPU: the scatter/gather legs are local copies",
        "transport": "torch.distributed NCCL, one batch_isend_irecv (ncclGroup of send/recv) per leg, receives land at "
                     "their final prefix-summed offsets",
    }


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
