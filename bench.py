#!/usr/bin/env python
"""bench.py — benchmark of the GPU I/O worker on the BASELINE.json configurations.

What a run does (both arms, `--impl b200` = this repo's worker, `--impl reference` = the CPU
LocalWorker of the reference, here its oracle port — the reference binary cannot be built in this
image, see DESIGN.md):

  --config c2 (default, BASELINE configs[1]): one file of --file-gib GiB (default 64) per GPU in
      --dir, 1 MiB blocks, sequential write phase + read phase with --verify. The file is
      worked through in W+K equal slices: step s = write phase + read phase over slice s of every
      file, expressed with the reference's own sharding (--rankoffset / numDataSetThreads:
      worker ranks [(r*S+s)*T, (r*S+s+1)*T) of N*S*T own exactly slice s of file r,
      LocalWorker.cpp:3576-3589). Over a whole run every file is written once and read once.
  --config c3 (configs[2]): 4 KiB random reads with --verify, iodepth 64, of a 64 GiB file per
      GPU; the K timed steps together issue file-size / 4 KiB I/Os (16.7 M at 64 GiB).
  --config c4 (configs[3]): one 32 GiB file per GPU written with --blockvarpct 100 (K3), then
      1 MiB sequential reads in slices like c2 (no --verify).
  --config c5 (configs[4]): directory tree of 2^20 files of 64 KiB over all GPUs (16 threads per
      GPU), write + read --verify; step s works on its own 1/(W+K) of the tree.
  The reference's --gds variants need nvidia-fs; on boxes without it (cuFileHandleRegister fails,
  see profiles/) the same workload runs through the staged engine and the line says so.

What is reported
  value / e2e.value : the BASELINE metric through the worker's public C ABI with host buffers and
      real files: storage I/O, host<->device transfers and the on-GPU fill / verify are all inside
      the timed region. (bytes written + bytes read) / (sum over timed steps of the phase times),
      phase time = max over all workers of all ranks. value == e2e.value by construction; the
      HBM-resident kernel numbers are under `roofline`.
  roofline : K1/K2/K3 over an HBM-resident window against the measured HBM peak (the dominant
      resident kernel), plus the PCIe roofline of the staging path measured in the same run and
      the storage roofline (raw pread/pwrite with the same threads).
  cpu_baseline : the CPU LocalWorker on a bounded sample of the same steps (rank 0, N=1).

Multi-GPU: one process per GPU under torchrun; no data-path collective; NCCL reduces the stats
only. scaling = weak (per-GPU work fixed). With N > 1 rank 0 afterwards also runs the in-process
worker pool (one process, --gpuids 0..N-1, grouped ncclReduce for the stats) on a sample and
reports it as extra.inprocess_pool.
"""
import argparse
import ctypes
import json
import os
import shutil
import statistics
import sys
import threading
import time

REPO_ROOT = os.path.dirname(os.path.abspath(__file__))
if REPO_ROOT not in sys.path:
    sys.path.insert(0, REPO_ROOT)

KiB = 1 << 10
MiB = 1 << 20
GiB = 1 << 30
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--config", default="c2", choices=["c2", "c3", "c4", "c5"])
    p.add_argument("--file-gib", type=float, default=0.0,
                   help="file size per GPU (GiB); 0 = the config's stated size")
    p.add_argument("--threads", type=int, default=int(os.environ.get("ELB_BENCH_THREADS", "0")),
                   help="worker threads per GPU (-t), both arms; 0 = min(16, usable CPUs / GPUs): "
                        "the boxes give the container a CPU quota (16 CPUs at 1 GPU, 96 at 8) and "
                        "more busy threads than that get throttled")
    p.add_argument("--dir", default=os.environ.get("ELB_BENCH_DIR", "/dev/shm"))
    p.add_argument("--salt", type=int, default=1)
    p.add_argument("--direct", action="store_true", help="O_DIRECT (--direct)")
    p.add_argument("--window-gib", type=float, default=4.0,
                   help="HBM-resident window of the kernel-level (roofline) measurement")
    p.add_argument("--cpu-sample-steps", type=int, default=4,
                   help="timed steps of the bounded cpu_baseline / storage roofline samples")
    p.add_argument("--skip-cpu", action="store_true")
    p.add_argument("--skip-kernels", action="store_true")
    p.add_argument("--skip-pool", action="store_true")
    p.add_argument("--only-kernels", action="store_true",
                   help="kernel-level measurement only (for ncu captures)")
    p.add_argument("--staging", default="auto", choices=["auto", "kernel", "copyengine"])
    p.add_argument("--batch-blocks", type=int, default=0)
    p.add_argument("--num-batches", type=int, default=0)
    p.add_argument("--write-gate", default="auto", choices=["auto", "on", "off"])
    p.add_argument("--no-gpu-numa", action="store_true")
    p.add_argument("--kernel-block-kib", type=int, default=0,
                   help="block size of the kernel-level window (0 = the config's block size)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last timed step computed to "
                        "DIR/<name>.npy (see dump_outputs)")
    args = p.parse_args()
    if args.steps < 1 or args.warmup < 0:
        p.error("--steps must be >= 1 and --warmup >= 0")
    if args.threads <= 0:
        args.threads = max(1, min(16, int(cpu_quota() // max(1, args.gpus))))
    return args


# ------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------

class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU while running (NVML, 10 ms period)."""

    REASONS = {
        0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
        0x4: "sw_power_cap", 0x80: "hw_power_brake", 0x2: "applications_clocks_setting",
    }

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(self.gpu_index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nvml = None
            return self
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        return self

    def _run(self):
        nv = self._nvml
        while not self._stop.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self._handle, nv.NVML_CLOCK_SM)
                util = nv.nvmlDeviceGetUtilizationRates(self._handle).gpu
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._handle)
                self.samples.append((mhz, util))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        loaded = [m for m, u in self.samples if u > 0] or [m for m, _ in self.samples]
        return {"sm_mhz": statistics.median(loaded), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples),
                "gpu_busy_mean_pct": round(statistics.mean(u for _, u in self.samples), 1)}


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------

def load_hbm_peak():
    path = os.path.join(REPO_ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_ncu_traffic(window_bytes, block_bytes, kernel_key):
    """DRAM bytes (read + write) of one launch of the given kernel from the committed
    `ncu --set full` captures (profiles/ncu_traffic.json): the capture with the same block size and
    window; a capture of the same block size with another window is scaled to this window (the
    kernels' traffic is proportional to the bytes they cover) and the source says so."""
    path = os.path.join(REPO_ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(path) as f:
            data = json.load(f)
        captures = data["captures"] if "captures" in data else [data]
        same_block = [c for c in captures if int(c.get("block_bytes", MiB)) == int(block_bytes)
                      and kernel_key in c["kernels"]]
        for entry in same_block:
            if int(entry["window_bytes"]) == int(window_bytes):
                kern = entry["kernels"][kernel_key]
                return kern["dram_bytes_read"] + kern["dram_bytes_write"], entry.get("source")
        if same_block:
            entry = same_block[0]
            kern = entry["kernels"][kernel_key]
            scale = float(window_bytes) / float(entry["window_bytes"])
            return (int((kern["dram_bytes_read"] + kern["dram_bytes_write"]) * scale),
                    "%s (captured over a %.0f GiB window, scaled x%.2f to this one)" % (
                        entry.get("source"), int(entry["window_bytes"]) / GiB, scale))
    except Exception:
        pass
    return None, None


def dist_env():
    return (int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")),
            int(os.environ.get("WORLD_SIZE", "1")))


def bench_dir(args):
    path = os.path.join(args.dir, "elb_bench_%d" % os.getuid())
    os.makedirs(path, exist_ok=True)
    return path


def cpu_quota():
    """CPUs this container may use: cgroup cpu.max quota, else the affinity mask."""
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            return round(int(quota) / int(period), 1)
    except Exception:
        pass
    try:
        return float(len(os.sched_getaffinity(0)))
    except Exception:
        return float(os.cpu_count() or 1)


def storage_free_gib(path):
    """free space of the (RAM backed) storage: statvfs and, for tmpfs, the cgroup memory limit"""
    stat = os.statvfs(path)
    free = stat.f_bavail * stat.f_frsize / GiB
    try:
        limit = open("/sys/fs/cgroup/memory.max").read().strip()
        if limit != "max":
            used = int(open("/sys/fs/cgroup/memory.current").read())
            free = min(free, (int(limit) - used) / GiB)
    except Exception:
        pass
    return free


_REAL_STDOUT = None


def protect_stdout():
    """The driver parses ONE JSON line from stdout; libraries (NCCL's version banner) also write
    there. Keep the real stdout aside and point fd 1 at stderr for everything else."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def log(msg):
    sys.stderr.write("[bench] %s\n" % msg)
    sys.stderr.flush()


def histo_summary(histo):
    """min / avg / max and percentiles of a latency histogram dict (LatencyHistogram.h rules:
    bucket index = floor(log2(usec) * 4), percentile = upper bound of the bucket)"""
    num = histo["num"]
    if not num:
        return None
    out = {"num": num, "min_usec": histo["min_usec"], "avg_usec": round(histo["sum_usec"] / num, 1),
           "max_usec": histo["max_usec"]}
    for pct in (50, 99, 99.9):
        want = num * pct / 100.0
        seen = 0
        for idx, count in enumerate(histo["buckets"]):
            seen += count
            if seen >= want:
                out["p%s_usec_le" % pct] = round(2 ** ((idx + 1) / 4.0), 1)
                break
    return out


# ------------------------------------------------------------------------------------------------
# workloads: what one step of a configuration is, identically for both arms
# ------------------------------------------------------------------------------------------------

class Workload:
    """One BASELINE configuration. plan(step, rank) -> (WorkerConfig kwargs, [phases]) of the step
    for the process that owns file / tree share `rank` (the GPU arm runs rank = its own rank, the
    CPU arm runs all ranks of the job concurrently in one process)."""

    def __init__(self, args, world):
        self.args = args
        self.world = world
        self.threads = args.threads
        self.num_slices = args.warmup + args.steps
        self.workdir = bench_dir(args)

    # -- to be provided by the configs
    name = ""
    metric = ""
    unit = "GiB/s"
    block = MiB

    def describe(self):
        raise NotImplementedError

    def prepare_plan(self, rank):
        """untimed preparation (e.g. the files a read-only config reads): like plan() or None"""
        return None

    def plan(self, step, rank):
        raise NotImplementedError

    def value_of(self, totals):
        """headline value from the summed timed steps"""
        return totals["bytes"] / GiB / (totals["usec"] / 1e6) if totals["usec"] else 0.0

    def cleanup_paths(self, rank):
        return []

    def written_regions(self, step, rank):
        """[(path, offset, length)] of the file data that step writes on behalf of `rank`"""
        return []

    def common_cfg(self):
        return dict(block_size=self.block, use_direct_io=self.args.direct)


class SeqFileWorkload(Workload):
    """c2 / c4: one file per GPU, sliced into W+K steps through the reference's rank sharding."""

    def __init__(self, args, world, file_gib, do_verify, blockvarpct, do_write_in_step):
        super().__init__(args, world)
        self.do_verify = do_verify
        self.blockvarpct = blockvarpct
        self.do_write_in_step = do_write_in_step
        blocks_per_slice_thread = int(file_gib * GiB) // self.block // (self.num_slices *
                                                                      self.threads)
        if blocks_per_slice_thread < 1:
            raise SystemExit("file too small for %d slices x %d threads" % (self.num_slices,
                                                                            self.threads))
        self.file_size = blocks_per_slice_thread * self.num_slices * self.threads * self.block
        self.slice_bytes = self.file_size // self.num_slices
        self.paths = [os.path.join(self.workdir, "%s_file_%d.bin" % (self.name, r))
                      for r in range(world)]

    def base_cfg(self):
        cfg = self.common_cfg()
        cfg.update(paths=self.paths, file_size=self.file_size, num_threads=self.threads,
                   integrity_check_salt=self.args.salt if self.do_verify else 0,
                   block_variance_percent=self.blockvarpct, block_variance_seed=4711)
        return cfg

    def plan(self, step, rank):
        from elbencho_b200 import BenchPhase
        cfg = self.base_cfg()
        cfg.update(rank_offset=(rank * self.num_slices + step) * self.threads,
                   num_dataset_threads=self.world * self.num_slices * self.threads)
        phases = ([BenchPhase.CREATEFILES] if self.do_write_in_step else []) + \
            [BenchPhase.READFILES]
        return cfg, phases

    def cleanup_paths(self, rank):
        return [self.paths[rank]]

    def written_regions(self, step, rank):
        if not self.do_write_in_step:
            return []
        return [(self.paths[rank], step * self.slice_bytes, self.slice_bytes)]


class C2(SeqFileWorkload):
    name = "c2"
    metric = "seq_write_read_verify_throughput"

    def __init__(self, args, world):
        super().__init__(args, world, args.file_gib or 64.0, True, 0, True)

    def describe(self):
        return ("BASELINE configs[1]: single %.2f GiB file per GPU, 1 MiB blocks, sequential write "
                "+ read with --verify %d, --gpuids <gpu>, pinned host ring staging"
                % (self.file_size / GiB, self.args.salt))


class C4(SeqFileWorkload):
    name = "c4"
    metric = "seq_read_throughput_blockvar_files"

    def __init__(self, args, world):
        super().__init__(args, world, args.file_gib or 32.0, False, 100, False)

    def describe(self):
        return ("BASELINE configs[3]: one %.2f GiB file per GPU written with --blockvarpct 100 "
                "(on-GPU random fill), then 1 MiB sequential reads into GPU memory; --gds is "
                "replaced by the staged engine where cuFile cannot register handles"
                % (self.file_size / GiB))

    def prepare_plan(self, rank):
        from elbencho_b200 import BenchPhase
        cfg = self.base_cfg()
        cfg.update(rank_offset=rank * self.threads, num_dataset_threads=self.world * self.threads)
        return cfg, [BenchPhase.CREATEFILES]

    def value_of(self, totals):
        """the read phase alone is the metric of this config (the write is its preparation)"""
        read = totals["phase"]["READFILES"]
        return read["bytes"] / GiB / (read["usec"] / 1e6) if read["usec"] else 0.0


class C3(Workload):
    name = "c3"
    metric = "rand_read_4k_verify_iops"
    unit = "IOPS"
    block = 4 * KiB

    def __init__(self, args, world):
        super().__init__(args, world)
        per_thread = int((args.file_gib or 64.0) * GiB) // self.block // (args.steps *
                                                                          self.threads)
        self.ios_per_step = per_thread * self.threads
        self.file_size = self.ios_per_step * args.steps * self.block
        self.paths = [os.path.join(self.workdir, "c3_file_%d.bin" % r) for r in range(world)]

    def describe(self):
        return ("BASELINE configs[2]: single %.2f GiB file per GPU, 4 KiB random reads with "
                "--verify %d, --iodepth 64, %d I/Os per GPU over the timed steps; --gds cuFile "
                "batch is replaced by the staged engine where cuFile cannot register handles"
                % (self.file_size / GiB, self.args.salt, self.ios_per_step * self.args.steps))

    def base_cfg(self, rank):
        cfg = self.common_cfg()
        cfg.update(paths=[self.paths[rank]], file_size=self.file_size, num_threads=self.threads,
                   integrity_check_salt=self.args.salt)
        return cfg

    def prepare_plan(self, rank):
        from elbencho_b200 import BenchPhase
        cfg = self.base_cfg(rank)
        cfg.update(block_size=MiB)
        return cfg, [BenchPhase.CREATEFILES]

    def plan(self, step, rank):
        from elbencho_b200 import BenchPhase, IOEngine
        cfg = self.base_cfg(rank)
        cfg.update(use_random_offsets=True, random_amount=self.ios_per_step * self.block,
                   rand_offset_seed=1000 + 97 * step + rank, io_depth=64,
                   io_engine=int(IOEngine.AIO))
        return cfg, [BenchPhase.READFILES]

    def value_of(self, totals):
        return totals["iops"] / (totals["usec"] / 1e6) if totals["usec"] else 0.0

    def cleanup_paths(self, rank):
        return [self.paths[rank]]


class C5(Workload):
    name = "c5"
    metric = "dir_tree_write_read_verify_throughput"
    block = 64 * KiB

    DIRS_PER_STEP = 4

    def __init__(self, args, world):
        super().__init__(args, world)
        total_files = int(args.file_gib * GiB) // self.block if args.file_gib else (1 << 20)
        self.files_per_dir = max(1, total_files // (world * self.threads * self.num_slices *
                                                    self.DIRS_PER_STEP))
        self.files_per_step_gpu = self.files_per_dir * self.DIRS_PER_STEP * self.threads
        self.total_files = self.files_per_step_gpu * world * self.num_slices

    def describe(self):
        return ("BASELINE configs[4]: directory tree of %d files x 64 KiB over all GPUs (2^20 "
                "asked, rounded down to whole steps), %d threads per GPU, create+write and read "
                "with --verify %d; step s works on its own 1/%d of the tree" % (
                    self.total_files, self.threads, self.args.salt, self.num_slices))

    def step_dir(self, step):
        return os.path.join(self.workdir, "c5_step_%d" % step)

    def plan(self, step, rank):
        from elbencho_b200 import BenchPhase, PathType
        path = self.step_dir(step)
        os.makedirs(path, exist_ok=True)
        cfg = self.common_cfg()
        cfg.update(paths=[path], path_type=int(PathType.DIR), file_size=self.block,
                   num_threads=self.threads, num_dirs=self.DIRS_PER_STEP,
                   num_files=self.files_per_dir, integrity_check_salt=self.args.salt,
                   rank_offset=rank * self.threads, num_dataset_threads=self.world * self.threads)
        return cfg, [BenchPhase.CREATEDIRS, BenchPhase.CREATEFILES, BenchPhase.READFILES]

    def cleanup_paths(self, rank):
        return [self.step_dir(s) for s in range(self.num_slices)] if rank == 0 else []

    def written_regions(self, step, rank):
        """every file of the step's tree (the ranks share it), in path order"""
        files = sorted(os.path.join(root, name) for root, _, names in os.walk(self.step_dir(step))
                       for name in names)
        return [(path, 0, os.path.getsize(path)) for path in files]


WORKLOADS = {"c2": C2, "c3": C3, "c4": C4, "c5": C5}
TIMED_PHASES = ("CREATEFILES", "READFILES")  # (mkdirs of c5 are preparation of the step)


def remove_paths(paths):
    for path in paths:
        if os.path.isdir(path):
            shutil.rmtree(path, ignore_errors=True)
        elif os.path.exists(path):
            os.unlink(path)


def new_totals():
    return {"bytes": 0, "iops": 0, "entries": 0, "usec": 0,
            "phase": {name: {"bytes": 0, "iops": 0, "entries": 0, "usec": 0}
                      for name in TIMED_PHASES}}


def add_phase(totals, name, num_bytes, iops, entries, usec):
    if name not in TIMED_PHASES:
        return
    for tgt in (totals, totals["phase"][name]):
        tgt["bytes"] += num_bytes
        tgt["iops"] += iops
        tgt["entries"] += entries
        tgt["usec"] += usec


def phase_rates(totals):
    out = {}
    for name, short in (("CREATEFILES", "write"), ("READFILES", "read")):
        ph = totals["phase"][name]
        if not ph["usec"]:
            continue
        secs = ph["usec"] / 1e6
        out[short + "_gib_s"] = round(ph["bytes"] / GiB / secs, 3)
        out[short + "_iops"] = int(ph["iops"] / secs)
        if ph["entries"]:
            out[short + "_files_s"] = int(ph["entries"] / secs)
    return out


DUMP_SEED = 20240531
DUMP_CHUNKS = 256
DUMP_CHUNK_BYTES = 4096


def dump_outputs(out_dir, workload, step, rank, step_results):
    """Write what timed step `step` computed, so that two builds can be compared output for
    output on the same arguments:
      <phase>_counters.npy      float64 [entries, bytes, iops, verified bytes, verify mismatch
                                bytes, filled bytes] of each timed phase (the job-wide results the
                                caller receives; times and latencies are left out, they differ
                                from run to run)
      written_sample.npy        float32 [DUMP_CHUNKS, chunk] bytes of the file data the step wrote,
                                at offsets drawn with a fixed seed (configs whose steps write)
      written_sample_where.npy  float64 [DUMP_CHUNKS, 2] (region index, offset in region) of each
                                row, regions in the order of workload.written_regions()
    At most 4 MiB in all."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, res in step_results.items():
        if name not in TIMED_PHASES:
            continue
        ops = res["ops_total"]
        counters = [ops["entries"], ops["bytes"], ops["iops"], res["verified_bytes"],
                    res["verify_mismatch_bytes"], res["filled_bytes"]]
        np.save(os.path.join(out_dir, name.lower() + "_counters.npy"),
                np.array(counters, dtype=np.float64))
    regions = workload.written_regions(step, rank)
    if not regions:
        return
    lengths = np.array([length for _, _, length in regions], dtype=np.int64)
    chunk = int(min(DUMP_CHUNK_BYTES, lengths.min()))
    rng = np.random.default_rng(DUMP_SEED)
    picks = rng.choice(len(regions), size=DUMP_CHUNKS, p=lengths / lengths.sum())
    offsets = rng.integers(0, lengths[picks] - chunk, endpoint=True)
    sample = np.empty((DUMP_CHUNKS, chunk), dtype=np.float32)
    for row, (idx, off) in enumerate(zip(picks, offsets)):
        path, start, _ = regions[idx]
        with open(path, "rb") as f:
            f.seek(start + int(off))
            data = f.read(chunk)
        if len(data) != chunk:
            raise RuntimeError("short read of %s at %d" % (path, start + int(off)))
        sample[row] = np.frombuffer(data, dtype=np.uint8)
    np.save(os.path.join(out_dir, "written_sample.npy"), sample)
    np.save(os.path.join(out_dir, "written_sample_where.npy"),
            np.stack([picks, offsets], axis=1).astype(np.float64))


# ------------------------------------------------------------------------------------------------
# the CPU LocalWorker arm (oracle port of the reference loop)
# ------------------------------------------------------------------------------------------------

def cpu_run_plan(plans):
    """Run one step's plan of every rank concurrently in this process (one oracle run per rank,
    like the GPU arm's one process per GPU). plans: [(cfg kwargs, phases)] -> per phase name:
    dict(bytes, iops, entries, usec = max over the ranks)"""
    from elbencho_b200 import WorkerConfig
    from tests import oracle_lib  # oracle: only used as the CPU baseline / reference arm here
    out = {}
    phases = plans[0][1]
    for phase in phases:
        results = [None] * len(plans)
        errors = []

        def run(idx):
            try:
                cfg = WorkerConfig(**plans[idx][0])
                rc, workers, pres = oracle_lib.run_oracle_phase(cfg, phase)
                if rc != 0:
                    raise RuntimeError("CPU LocalWorker failed: " + "; ".join(
                        w.errorMsg.decode() for w in workers if w.hadError))
                results[idx] = pres
            except Exception as err:  # noqa: BLE001
                errors.append(err)

        threads = [threading.Thread(target=run, args=(i,)) for i in range(len(plans))]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        out[phase.name] = {
            "bytes": sum(r.opsTotal.numBytesDone for r in results),
            "iops": sum(r.opsTotal.numIOPSDone for r in results),
            "entries": sum(r.opsTotal.numEntriesDone for r in results),
            "usec": max(r.lastFinishUSec for r in results)}
    return out


def cpu_arm(workload, steps, warmup, salt_override=None):
    """the CPU LocalWorker over `warmup` untimed + `steps` timed steps of the workload"""
    world = workload.world
    totals = new_totals()
    prep = [workload.prepare_plan(r) for r in range(world)]
    if prep[0] is not None:
        cpu_run_plan(prep)
    for step in range(warmup + steps):
        plans = [workload.plan(step, r) for r in range(world)]
        if salt_override is not None:
            for cfg, _ in plans:
                cfg["integrity_check_salt"] = salt_override
                cfg["block_variance_percent"] = 0
        res = cpu_run_plan(plans)
        if step >= warmup:
            for name, ph in res.items():
                add_phase(totals, name, ph["bytes"], ph["iops"], ph["entries"], ph["usec"])
    return totals


def cpu_kernels_per_core(block_size, salt, total_bytes=256 * MiB):
    """GB/s of ONE host core for the reference's per-block operators (the oracle restatement of
    preWriteIntegrityCheckFillBuf / postReadIntegrityCheckVerifyBuf, LocalWorker.cpp:2091-2179) on
    a block-sized buffer, as a CPU counterpart of the K1 / K2 numbers (SURVEY.md 8d)."""
    from tests import oracle_lib  # oracle: CPU baseline leg only
    lib = oracle_lib.load_oracle()
    buf = ctypes.create_string_buffer(block_size)
    nblocks = max(1, total_bytes // block_size)
    num, first = ctypes.c_uint64(), ctypes.c_uint64()
    exp, act = ctypes.c_uint(), ctypes.c_uint()
    msg = ctypes.create_string_buffer(256)
    out = {}
    t0 = time.perf_counter()
    for i in range(nblocks):
        lib.orc_fill_pattern(buf, block_size, i * block_size, salt)
    out["fill_pattern_gb_s"] = round(nblocks * block_size / (time.perf_counter() - t0) / 1e9, 2)
    t0 = time.perf_counter()
    bad = 0
    for i in range(nblocks):
        bad += lib.orc_verify_pattern(buf, block_size, (nblocks - 1) * block_size, salt,
                                      ctypes.byref(num), ctypes.byref(first), ctypes.byref(exp),
                                      ctypes.byref(act), msg, len(msg))
    out["verify_pattern_gb_s"] = round(nblocks * block_size / (time.perf_counter() - t0) / 1e9, 2)
    if bad:
        raise RuntimeError("CPU verify of a CPU-filled block failed")
    out["note"] = "one core, %d x %d KiB blocks, cache-resident buffer" % (nblocks,
                                                                            block_size // 1024)
    return out


def common_config(args, workload, world):
    """the `config` object: identical for both arms (same files, sizes, steps, threads)"""
    cfg = {
        "workload": workload.describe(),
        "baseline_config": workload.name,
        "num_files_or_trees": world,
        "block_kib": workload.block // KiB,
        "threads_per_gpu": workload.threads,
        "steps_layout": "%d warm-up + %d timed steps; step s = slice s of the per-GPU data set "
                        "(reference sharding by --rankoffset / numDataSetThreads)" % (
                            args.warmup, args.steps),
        "storage_dir": args.dir, "direct": args.direct,
        "l2": "every step works on fresh file data larger than L2 (>= %.2f GiB per GPU and step)" % (
            getattr(workload, "slice_bytes", 0) / GiB) if hasattr(workload, "slice_bytes")
        else "every step works on fresh data (files / random offsets not touched before)",
        "host_cpus_usable": cpu_quota(),
    }
    if hasattr(workload, "file_size"):
        cfg["file_gib"] = round(workload.file_size / GiB, 4)
    if hasattr(workload, "total_files"):
        cfg["total_files"] = workload.total_files
    return cfg


def reference_arm(args):
    """bench.py --impl reference: the reference's CPU path on the host cores, same metric, same
    files, same steps, same thread count."""
    rank, _, world_env = dist_env()
    if rank != 0:
        return 0  # other ranks exit without work
    world = max(1, args.gpus)
    workload = WORKLOADS[args.config](args, world)
    try:
        totals = cpu_arm(workload, args.steps, args.warmup)
    finally:
        for r in range(world):
            remove_paths(workload.cleanup_paths(r))
    value = workload.value_of(totals)
    cores = workload.threads * world
    sample = "%d timed steps of the workload (all of it), %d threads (%d per file/GPU share) in %s" % (
        args.steps, cores, workload.threads, args.dir)
    line = {
        "impl": "reference", "metric": workload.metric, "value": round(value, 3),
        "unit": workload.unit, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(totals["usec"] / 1e3 / max(1, args.steps), 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic",
        "config": common_config(args, workload, world),
        "cpu_baseline": {"value": round(value, 3), "unit": workload.unit, "cores": cores,
                         "kind": "port", "sample": sample,
                         "impl_note": "oracle port of LocalWorker.cpp:1669-1781 + 2091-2179 "
                                      "(the reference binary cannot be built here)",
                         **phase_rates(totals),
                         "operators_per_core": cpu_kernels_per_core(workload.block, args.salt)},
        "e2e": {"value": round(value, 3), "unit": workload.unit, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------------
# kernel-level measurement (HBM-resident window) -> roofline of K1 / K2 / K3
# ------------------------------------------------------------------------------------------------

def kernel_level(args, torch, device, block, steps=10, warmup=3):
    from elbencho_b200 import kernels
    nblocks = max(1, int(args.window_gib * GiB) // block)
    window = nblocks * block
    arena = torch.empty(window, dtype=torch.uint8, device=device)
    counters = torch.zeros(kernels.DEVCTR_NUM, dtype=torch.int64, device=device)
    results = torch.zeros(2 * nblocks, dtype=torch.int64, device=device)
    stream = torch.cuda.current_stream(device)
    handle = stream.cuda_stream

    desc_tensors = []
    for step in range(warmup + steps):
        base = step * window
        blocks = [(arena.data_ptr() + i * block, block, base + i * block, i) for i in range(nblocks)]
        raw = kernels.pack_block_descs(blocks)
        desc_tensors.append(torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(device))

    def ev():
        return torch.cuda.Event(enable_timing=True)

    launches_before = kernels.num_kernel_launches()
    timings = {"fill": [], "verify": [], "rand": []}
    for step in range(warmup + steps):
        descs = desc_tensors[step]
        events = [ev() for _ in range(4)]
        events[0].record(stream)
        kernels.fill_pattern_batch(descs.data_ptr(), nblocks, args.salt, counters.data_ptr(),
                                   handle, total_bytes=window, max_block_len=block)
        events[1].record(stream)
        kernels.verify_pattern_batch(descs.data_ptr(), nblocks, args.salt, results.data_ptr(),
                                     counters.data_ptr(), handle, total_bytes=window,
                                     max_block_len=block)
        events[2].record(stream)
        kernels.fill_random_batch(descs.data_ptr(), nblocks, 100, 12345, 0, handle,
                                  total_bytes=window, max_block_len=block)
        events[3].record(stream)
        if step >= warmup:
            timings["fill"].append((events[0], events[1]))
            timings["verify"].append((events[1], events[2]))
            timings["rand"].append((events[2], events[3]))
    torch.cuda.synchronize(device)
    launches = kernels.num_kernel_launches() - launches_before

    ctr = counters.cpu().tolist()
    if ctr[kernels.DEVCTR_VERIFY_MISMATCH_BYTES] or int(results.view(-1, 2)[:, 0].sum()) != 0:
        raise RuntimeError("verify kernel reported mismatches on freshly filled data")
    ms = {k: statistics.mean(a.elapsed_time(b) for a, b in v) for k, v in timings.items()}
    del arena
    return {"window_bytes": window, "block_bytes": block, "nblocks": nblocks, "ms": ms,
            "launches": launches}


def pcie_level(torch, device):
    """PCIe roofline of the staging path, measured in this run: pinned cudaMemcpyAsync in 16 MiB
    chunks (copy engine) and the worker's own stage-copy kernels at 1 MiB per launch."""
    from elbencho_b200 import kernels
    nbytes = 256 * MiB
    host = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    dev = torch.empty(nbytes, dtype=torch.uint8, device=device)
    stream = torch.cuda.current_stream(device)
    out = {}

    def timed(fn, total_bytes, reps=3):
        best = None
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            torch.cuda.synchronize(device)
            ms = a.elapsed_time(b)
            best = ms if best is None else min(best, ms)
        return round(total_bytes / GiB / (best / 1e3), 2)

    chunk = 64 * MiB

    def h2d():
        for off in range(0, nbytes, chunk):
            dev[off:off + chunk].copy_(host[off:off + chunk], non_blocking=True)

    def d2h():
        for off in range(0, nbytes, chunk):
            host[off:off + chunk].copy_(dev[off:off + chunk], non_blocking=True)

    out["copy_engine_h2d_gib_s"] = timed(h2d, nbytes)
    out["copy_engine_d2h_gib_s"] = timed(d2h, nbytes)

    delta = host.data_ptr() - dev.data_ptr()
    nblocks = nbytes // MiB
    raw = kernels.pack_block_descs([(dev.data_ptr() + i * MiB, MiB, 0, 0) for i in range(nblocks)])
    descs = torch.frombuffer(bytearray(raw), dtype=torch.uint8).pin_memory()
    desc_bytes = len(raw) // nblocks
    per_launch = 16  # blocks per launch (a launch of the worker carries 2..256 blocks)

    def staged(to_device):
        def run():
            for i in range(0, nblocks, per_launch):
                kernels.stage_copy(descs.data_ptr() + i * desc_bytes, per_launch, to_device, delta,
                                   stream.cuda_stream, total_bytes=per_launch * MiB,
                                   max_block_len=MiB)
        return run

    out["stage_kernel_h2d_gib_s"] = timed(staged(True), nbytes)
    out["stage_kernel_d2h_gib_s"] = timed(staged(False), nbytes)
    out["note"] = ("pinned host <-> HBM on this GPU, one stream: cudaMemcpyAsync in 64 MiB chunks; "
                   "stage-copy kernel, 16 blocks of 1 MiB per launch")
    return out


def barrier(torch, device):
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        dist.barrier(device_ids=[device.index] if device.type == "cuda" else None)
    torch.cuda.synchronize(device)


# ------------------------------------------------------------------------------------------------
# the GPU worker arm
# ------------------------------------------------------------------------------------------------

def tuning_kwargs(args, gpu_ids):
    return dict(gpu_ids=gpu_ids,
                staging_engine={"auto": 0, "kernel": 1, "copyengine": 2}[args.staging],
                pipeline_batch_blocks=args.batch_blocks, pipeline_num_batches=args.num_batches,
                serialize_buffered_writes={"auto": 0, "on": 1, "off": 2}[args.write_gate],
                no_gpu_numa_binding=args.no_gpu_numa)


def gpu_run_plan(args, torch, device, plan, gpu_ids, reduce_fn):
    """one step on this process: a manager for the step's config, its phases bracketed by
    barriers; -> {phase name: job-wide reduced results}"""
    from elbencho_b200 import WorkerConfig, WorkerManager
    cfg_kwargs, phases = plan
    cfg_kwargs = dict(cfg_kwargs)
    cfg_kwargs.update(tuning_kwargs(args, gpu_ids))
    out = {}
    with WorkerManager(WorkerConfig(**cfg_kwargs)) as mgr:
        for phase in phases:
            barrier(torch, device)
            local = mgr.run_phase(phase)
            barrier(torch, device)
            out[phase.name] = reduce_fn(local)
    return out


def gpu_arm(args, torch, device, workload, rank):
    from elbencho_b200 import distributed as elbdist

    def reduce_fn(local):
        return elbdist.reduce_phase_results(local, device)  # NCCL: stats only

    gpu_ids = [device.index]
    totals = new_totals()
    extra = {"h2d_bytes": 0, "d2h_bytes": 0, "launches": 0, "dev_kernel_usec": 0,
             "verified_bytes": 0, "filled_bytes": 0, "histos": {}}
    prep = workload.prepare_plan(rank)
    prep_info = None
    if prep is not None:
        res = gpu_run_plan(args, torch, device, prep, gpu_ids, reduce_fn)
        prep_info = {name: {"gib_s": round(r["ops_total"]["bytes"] / GiB /
                                           (r["last_finish_usec"] / 1e6), 3),
                            "filled_bytes": r["filled_bytes"]} for name, r in res.items()}
    for step in range(args.warmup + args.steps):
        res = gpu_run_plan(args, torch, device, workload.plan(step, rank), gpu_ids, reduce_fn)
        for name, r in res.items():
            if r["verify_mismatch_bytes"]:
                raise RuntimeError("step %d %s found integrity mismatches" % (step, name))
            if r["num_workers_done_with_error"]:
                raise RuntimeError("step %d %s had worker errors" % (step, name))
        if step < args.warmup:
            continue
        for name, r in res.items():
            add_phase(totals, name, r["ops_total"]["bytes"], r["ops_total"]["iops"],
                      r["ops_total"]["entries"], r["last_finish_usec"])
            if name not in TIMED_PHASES:
                continue
            extra["h2d_bytes"] += r["h2d_bytes"]
            extra["d2h_bytes"] += r["d2h_bytes"]
            extra["launches"] += r["num_kernel_launches"]
            extra["dev_kernel_usec"] += r["dev_kernel_usec"]
            extra["verified_bytes"] += r["verified_bytes"]
            extra["filled_bytes"] += r["filled_bytes"]
            histo = extra["histos"].setdefault(name, {"buckets": [0] * len(
                r["iops_lat_histo"]["buckets"]), "num": 0, "sum_usec": 0,
                "min_usec": 1 << 62, "max_usec": 0})
            src = r["iops_lat_histo"]
            histo["buckets"] = [a + b for a, b in zip(histo["buckets"], src["buckets"])]
            histo["num"] += src["num"]
            histo["sum_usec"] += src["sum_usec"]
            if src["num"]:
                histo["min_usec"] = min(histo["min_usec"], src["min_usec"])
                histo["max_usec"] = max(histo["max_usec"], src["max_usec"])
    return totals, extra, prep_info, res


def pool_steps(workload, world, warmup, steps):
    """The steps of the in-process pool sample: ONE manager config per step that covers all GPUs
    (worker rank g -> GPU g % N, LocalWorker.cpp:1420-1429). yields (cfg kwargs, phases, paths to
    remove after the step)."""
    from elbencho_b200 import BenchPhase
    threads = world * workload.threads
    if isinstance(workload, SeqFileWorkload):
        # N fresh files of one slice each per step, T consecutive ranks per file
        for step in range(warmup + steps):
            paths = [os.path.join(workload.workdir, "pool_s%d_f%d.bin" % (step, r))
                     for r in range(world)]
            cfg = workload.base_cfg()
            cfg.update(paths=paths, file_size=workload.slice_bytes, num_threads=threads,
                       rank_offset=0, num_dataset_threads=threads)
            yield cfg, [BenchPhase.CREATEFILES, BenchPhase.READFILES], paths
    elif isinstance(workload, C3):
        cfg = workload.base_cfg(0)
        cfg.update(paths=workload.paths, num_threads=threads, block_size=MiB)
        yield cfg, [BenchPhase.CREATEFILES], []  # (step 0 of the warm-up: the files to read)
        for step in range(1, warmup + steps):
            cfg, phases = workload.plan(step, 0)
            cfg.update(paths=workload.paths, num_threads=threads,
                       random_amount=workload.ios_per_step * workload.block * world)
            yield cfg, phases, (workload.paths if step == warmup + steps - 1 else [])
    else:
        for step in range(warmup + steps):
            cfg, phases = workload.plan(step, 0)
            cfg.update(num_threads=threads, rank_offset=0, num_dataset_threads=threads)
            yield cfg, phases, [workload.step_dir(step)]


def inprocess_pool(args, torch, workload_cls, world):
    """The single-process worker pool north_star describes: one manager, --gpuids 0..N-1, rank ->
    GPU round robin (LocalWorker.cpp:1420-1429), live and phase-end statistics through the grouped
    ncclReduce of the library (replaces the host loop of Statistics.cpp:1338-1344). Runs a sample
    of the same workload (2 warm-up + 4 timed steps of the main run's step size) on rank 0 while
    the other ranks wait."""
    import copy
    from elbencho_b200 import WorkerConfig, WorkerManager
    warmup, steps = 2, 4
    pool_args = copy.copy(args)
    workload = workload_cls(pool_args, world)  # same slicing as the main run
    workload.workdir = os.path.join(workload.workdir, "pool")
    os.makedirs(workload.workdir, exist_ok=True)
    if hasattr(workload, "paths"):
        workload.paths = [os.path.join(workload.workdir, os.path.basename(p))
                          for p in workload.paths]
    if isinstance(workload, C3):  # smaller files for the sample
        workload.file_size = min(workload.file_size, 8 * GiB)
    gpu_ids = list(range(world))
    totals = new_totals()
    info = {}
    try:
        for step, (cfg_kwargs, phases, stale) in enumerate(pool_steps(workload, world, warmup,
                                                                      steps)):
            cfg_kwargs = dict(cfg_kwargs)
            cfg_kwargs.update(tuning_kwargs(pool_args, gpu_ids))
            with WorkerManager(WorkerConfig(**cfg_kwargs)) as mgr:
                for phase in phases:
                    mgr.start_phase(phase)
                    while not mgr.wait_done(50):
                        snap = mgr.live_snapshot()
                        info["live_reduced_with_nccl"] = snap["reduced_with_nccl"]
                        info["live_num_gpus"] = snap["num_gpus"]
                    res = mgr.phase_results()
                    if res["verify_mismatch_bytes"] or res["num_workers_done_with_error"]:
                        raise RuntimeError("in-process pool: %s failed: %s" % (phase.name,
                                                                               mgr.last_error))
                    info["phase_stats_reduced_with_nccl"] = res["stats_reduced_with_nccl"]
                    info["live_reduce_info"] = mgr.live_reduce_info()
                    if step >= warmup:
                        add_phase(totals, phase.name, res["ops_total"]["bytes"],
                                  res["ops_total"]["iops"], res["ops_total"]["entries"],
                                  res["last_finish_usec"])
            remove_paths(stale)
    finally:
        shutil.rmtree(workload.workdir, ignore_errors=True)
    info.update(phase_rates(totals))
    info["value"] = round(workload.value_of(totals), 3)
    info["unit"] = workload.unit
    info["gpu_ids"] = gpu_ids
    info["threads"] = world * workload.threads
    info["sample"] = ("%d warm-up + %d timed steps of the main run's step size, one manager over "
                      "all GPUs; workload: %s" % (warmup, steps, workload.describe()))
    return info


def build_line(args, workload, world, value, totals, extra, prep_info, kern, pcie, storage, cpu,
               pool, clocks, requested_gib):
    """the ONE JSON line of the b200 arm from what was measured (pure: testable without a GPU)"""
    peak, peak_src = load_hbm_peak()
    rates = phase_rates(totals)
    timed_secs = totals["usec"] / 1e6

    line = {
        "metric": workload.metric, "value": round(value, 3), "unit": workload.unit,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(totals["usec"] / 1e3 / max(1, args.steps), 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic",
        "config": common_config(args, workload, world),
        "impl_config": {
            "staging": args.staging, "batch_blocks": args.batch_blocks,
            "num_batches": args.num_batches, "write_gate": args.write_gate,
            "gpu_numa_binding": not args.no_gpu_numa,
            "file_gib_requested": requested_gib or None,
            "parallelism": "%d process(es) x %d worker threads, rank r <-> file r <-> GPU r" % (
                world, workload.threads),
            "timing": "phase time = max over all workers of all ranks (host steady clock inside "
                      "the worker, as the reference measures phases), phases bracketed by barrier "
                      "+ cudaDeviceSynchronize; value = bytes of the timed steps / sum of phase times",
        },
        "gpu_launches": extra["launches"],
        "clocks": clocks,
        "parity": {
            "checked_in_this_run": "every read phase verified its blocks on the GPU (0 mismatching "
                                   "bytes, verified_bytes below) and byte / IOPS totals equal the "
                                   "expected ones" if workload.name != "c4" else
                                   "byte / IOPS totals equal the expected ones (no --verify in c4)",
            "bit_exact_vs_oracle": "tests/ -m gpu: file bytes, counters, verify outcome and "
                                   "exception text against the CPU oracle, which is pinned to the "
                                   "reference's own headers (oracle/_ref, tests/golden/)",
            "random_fill_content": "K3 (--blockvarpct) is bit-exact against its own CPU twin only: "
                                   "the reference's random fill is self-seeded, its content cannot "
                                   "be pinned (SURVEY 8c); the layout rule is the reference's",
        },
    }
    line["e2e"] = {
        "value": round(value, 3), "unit": workload.unit,
        "h2d_bytes_per_step": extra["h2d_bytes"] // max(1, args.steps),
        "d2h_bytes_per_step": extra["d2h_bytes"] // max(1, args.steps),
        "step": "the phases of one step through the worker's C ABI: storage I/O into / out of the "
                "pinned host ring, host<->device transfer and on-GPU fill / verify",
        **rates,
        "gpu_launches": extra["launches"],
        "dev_kernel_usec": extra["dev_kernel_usec"],
        "dev_kernel_share_of_timed": round(extra["dev_kernel_usec"] / 1e6 /
                                           (timed_secs * workload.threads * world), 4)
        if timed_secs else None,
        "verified_bytes": extra["verified_bytes"], "filled_bytes": extra["filled_bytes"],
        "total_usec": totals["usec"],
        "latency": {name: histo_summary(h) for name, h in extra["histos"].items()},
    }
    if prep_info:
        line["e2e"]["preparation"] = prep_info

    roofline = {}
    if kern:
        window = kern["window_bytes"]
        gbs = {k: window / (v * 1e-3) / 1e9 for k, v in kern["ms"].items()}
        # dominant resident kernel of the configuration
        if workload.name == "c4":
            dom_key, dom_name, dom = "K3_fill_random_pct100", \
                "elb_blocks_tiled_kernel<FILL_RANDOM> (K3)", gbs["rand"]
        elif workload.name == "c3" or kern["ms"]["verify"] >= kern["ms"]["fill"]:
            dom_key, dom_name, dom = "K2_verify_pattern", \
                "elb_blocks_tiled_kernel<VERIFY_PATTERN> (K2)", gbs["verify"]
        else:
            dom_key, dom_name, dom = "K1_fill_pattern", \
                "elb_blocks_tiled_kernel<FILL_PATTERN> (K1)", gbs["fill"]
        traffic, traffic_src = load_ncu_traffic(window, kern["block_bytes"], dom_key)
        roofline = {
            "bound": "hbm", "kernel": dom_name, "achieved": round(dom, 1), "peak": peak,
            "unit": "GB/s", "frac": round(dom / peak, 4), "traffic": traffic,
            "traffic_source": traffic_src, "peak_source": peak_src,
            "measured": "CUDA events around each launch over a %.1f GiB HBM-resident window of "
                        "%d KiB blocks (larger than L2), %d launches each" % (
                            window / GiB, kern["block_bytes"] // KiB, 10),
            "note": "peak is the driver-measured COPY bandwidth; one-directional streams exceed "
                    "it (copy-engine cudaMemset writes 7.35 TB/s), hence frac > 1",
            "algorithmic_bytes_per_launch": window,
            "all_kernels": {
                "K1_fill_pattern": {"achieved": round(gbs["fill"], 1),
                                    "frac": round(gbs["fill"] / peak, 4),
                                    "ms_per_launch": round(kern["ms"]["fill"], 4)},
                "K2_verify_pattern": {"achieved": round(gbs["verify"], 1),
                                      "frac": round(gbs["verify"] / peak, 4),
                                      "ms_per_launch": round(kern["ms"]["verify"], 4)},
                "K3_fill_random_pct100": {"achieved": round(gbs["rand"], 1),
                                          "frac": round(gbs["rand"] / peak, 4),
                                          "ms_per_launch": round(kern["ms"]["rand"], 4)},
            },
        }
    if pcie:
        roofline["pcie"] = pcie
        if "read_gib_s" in rates:
            best_h2d = max(pcie["copy_engine_h2d_gib_s"], pcie["stage_kernel_h2d_gib_s"])
            roofline["pcie"]["e2e_read_frac_of_pcie"] = round(
                rates["read_gib_s"] / (best_h2d * world), 3)
        if "write_gib_s" in rates:
            best_d2h = max(pcie["copy_engine_d2h_gib_s"], pcie["stage_kernel_d2h_gib_s"])
            roofline["pcie"]["e2e_write_frac_of_pcie"] = round(
                rates["write_gib_s"] / (best_d2h * world), 3)
    if storage:
        roofline["storage"] = storage
        for key in ("read_gib_s", "write_gib_s"):
            if key in rates and storage.get(key):
                roofline["storage"]["e2e_%s_frac" % key.split("_")[0]] = round(
                    rates[key] / storage[key], 3)
        if storage["value"]:
            roofline["storage"]["e2e_frac"] = round(value / storage["value"], 3)
    line["roofline"] = roofline
    if cpu:
        line["cpu_baseline"] = cpu
    extra_out = {}
    if pool:
        extra_out["inprocess_pool"] = pool
    if extra_out:
        line["extra"] = extra_out
    return line


# ------------------------------------------------------------------------------------------------
# main
# ------------------------------------------------------------------------------------------------

def main():
    args = parse_args()
    protect_stdout()

    if args.impl == "reference":
        return reference_arm(args)

    import torch
    import torch.distributed as dist
    from elbencho_b200 import _native

    _native.load()  # fails loudly if the CUDA library is missing

    rank, local_rank, world = dist_env()
    if world != args.gpus and world > 1:
        raise SystemExit("WORLD_SIZE=%d but --gpus %d" % (world, args.gpus))
    if args.gpus > 1 and world == 1:
        raise SystemExit("--gpus %d needs one process per GPU: launch with "
                         "python -m torch.distributed.run --nproc-per-node %d ..." % (
                             args.gpus, args.gpus))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA GPU (there is no CPU fallback for the product path)")

    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)

    workload_cls = WORKLOADS[args.config]

    # all files of the job must fit into the (RAM backed) storage next to the baseline samples
    requested_gib = args.file_gib
    if workload_cls is not C5:
        want = args.file_gib or {"c2": 64.0, "c3": 64.0, "c4": 32.0}[args.config]
        os.makedirs(args.dir, exist_ok=True)
        fit = torch.tensor([storage_free_gib(args.dir)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(fit, op=dist.ReduceOp.MIN)
        usable = float(fit.item()) * 0.7 / world
        if want > usable:
            args.file_gib = max(1.0, float(int(usable)))
            log("file size reduced to %.0f GiB per GPU (storage has %.0f GiB free)" % (
                args.file_gib, float(fit.item())))

    workload = workload_cls(args, world)
    block = args.kernel_block_kib * KiB if args.kernel_block_kib else workload.block

    kern = None
    if not args.skip_kernels:
        kern = kernel_level(args, torch, device, block)
    if args.only_kernels:
        emit({"kernel_level": {k: v for k, v in kern.items()}})
        return 0

    pcie = pcie_level(torch, device) if rank == 0 else None

    sampler = ClockSampler(local_rank).start() if rank == 0 else None
    try:
        totals, extra, prep_info, last_step = gpu_arm(args, torch, device, workload, rank)
        if args.dump_outputs and rank == 0:  # (before the cleanup removes the written files)
            dump_outputs(args.dump_outputs, workload, args.warmup + args.steps - 1, rank,
                         last_step)
    finally:
        barrier(torch, device)
        remove_paths(workload.cleanup_paths(rank))
    clocks = sampler.stop() if sampler else None

    value = workload.value_of(totals)

    cpu = None
    storage = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        import copy
        sample_args = copy.copy(args)
        sample_args.warmup, sample_args.steps = 1, args.cpu_sample_steps
        # same slice size as the main run: scale the file with the number of slices
        if hasattr(workload, "slice_bytes"):
            sample_args.file_gib = workload.slice_bytes * (1 + args.cpu_sample_steps) / GiB
        elif isinstance(workload, C3):
            sample_args.file_gib = min(workload.file_size / GiB, 16.0)
        sample = workload_cls(sample_args, 1)
        try:
            cpu_totals = cpu_arm(sample, sample_args.steps, sample_args.warmup)
            remove_paths(sample.cleanup_paths(0))  # (the raw pass must allocate its pages too)
            raw_totals = cpu_arm(sample, sample_args.steps, sample_args.warmup, salt_override=0)
        finally:
            remove_paths(sample.cleanup_paths(0))
        cpu_value = sample.value_of(cpu_totals)
        cpu = {"value": round(cpu_value, 3), "unit": workload.unit, "cores": workload.threads,
               "kind": "port",
               "sample": "1 warm-up + %d timed steps of the same step size (%s), -t %d, in %s "
                         "(oracle port of LocalWorker.cpp:1669-1781 + 2091-2179)" % (
                             sample_args.steps, sample.describe(), workload.threads, args.dir),
               **phase_rates(cpu_totals),
               "operators_per_core": cpu_kernels_per_core(workload.block, args.salt)}
        storage = {"value": round(sample.value_of(raw_totals), 3), "unit": workload.unit,
                   **phase_rates(raw_totals), "threads": workload.threads,
                   "note": "raw pread/pwrite of the CPU loop without fill/verify on the same "
                           "storage, steps and thread count (bounded sample, one cache-resident "
                           "buffer per thread): the storage roofline of value"}

    pool = None
    if world > 1 and not args.skip_pool:
        # the other ranks wait on the HOST (polling a flag file) while rank 0 drives all GPUs from
        # one process: a pending NCCL barrier would keep a spinning kernel on every GPU the pool
        # wants to use
        flag = os.path.join(bench_dir(args), "pool_done.flag")
        if rank == 0 and os.path.exists(flag):
            os.unlink(flag)
        barrier(torch, device)  # (everybody is done with its GPU; a stale flag is gone)
        if rank == 0:
            try:
                pool = inprocess_pool(args, torch, workload_cls, world)
            except Exception as err:  # noqa: BLE001 (an extra must not break the bench line)
                pool = {"error": str(err)}
            finally:
                with open(flag, "w") as f:
                    f.write("done\n")
        else:
            deadline = time.time() + 1800
            while not os.path.exists(flag) and time.time() < deadline:
                time.sleep(0.05)
        barrier(torch, device)
        if rank == 0 and os.path.exists(flag):
            os.unlink(flag)

    if world > 1:
        dist.barrier(device_ids=[device.index])
        dist.destroy_process_group()

    if rank != 0:
        return 0

    line = build_line(args, workload, world, value, totals, extra, prep_info, kern, pcie, storage, cpu,
                      pool, clocks, requested_gib)
    emit(line)
    return 0


if __name__ == "__main__":
    sys.exit(main())
