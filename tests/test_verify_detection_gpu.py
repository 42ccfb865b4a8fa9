"""End-to-end detection outcome of --verify: files are corrupted on purpose, read back through the
worker pipeline, and what the worker reports is compared with a plain numpy reference of the
pattern (no product code, no oracle code) and, for the stop-at-first message, with the CPU oracle.

Each corruption class targets a place where the verify code branches: the first byte, both sides
of a block boundary, every byte position within a u64 word, the byte-wise tail of odd-length
blocks, a run across a 32-byte vector and a block boundary, a zeroed 4 KiB region (pattern bytes
that are 0 anyway do not count), a byte rewritten with its own value (does not count), the last
partial block and the last block of every worker.

Two checks per case:
- collect-all: the device-side count equals the number of differing bytes, in the phase results
  and in the live snapshot, and a second read phase on the same manager counts the same again
  (the counters start from zero in each phase);
- stop at first: the error text names the first bad byte (the oracle's text with one thread, the
  first bad byte of each worker's own block range with several), and after the bytes are restored
  the same manager reads the file cleanly (in-flight batches and armed results were cleaned up).
"""
import dataclasses
import json
import os
import random
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

MOCK_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "mock_cufile")
MOCK_LIB = os.path.join(MOCK_DIR, "libmock_cufile.so")

# must be set before the native library binds cuFile for the first time in this process
os.environ.setdefault("ELB_CUFILE_LIB", MOCK_LIB)

from elbencho_b200 import BenchPhase, PathType, WorkerConfig, WorkerError, WorkerManager  # noqa: E402
from elbencho_b200.worker import IOEngine  # noqa: E402
from tests import oracle_lib  # noqa: E402

pytestmark = pytest.mark.gpu

KiB = 1 << 10
MiB = 1 << 20
SALT = 0x2A
DEVCTR_MISMATCH = 0
GOLDEN_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_vectors.json")


# ------------------------------------------------------------------------------------------------
# reference: the closed-form pattern in numpy
# ------------------------------------------------------------------------------------------------

def expected_pattern(file_offset, length, salt):
    """byte i = byte ((file_offset + i) % 8) of little-endian u64 (((file_offset + i) & ~7) + salt),
    arithmetic mod 2^64"""
    start = file_offset & ~7
    num_words = (file_offset + length - start + 7) // 8
    words = np.uint64(start) + np.arange(num_words, dtype=np.uint64) * np.uint64(8)
    words += np.uint64(salt)  # (wraps mod 2^64)
    skip = file_offset - start
    return words.astype("<u8").view(np.uint8)[skip:skip + length]


def mismatches(data, file_offset, salt):
    """-> (number of bytes that differ from the pattern, index of the first one or None)"""
    got = np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else data
    diff = got != expected_pattern(file_offset, len(got), salt)
    bad = np.flatnonzero(diff)
    return int(np.count_nonzero(diff)), (int(bad[0]) if bad.size else None)


def verify_error_text(offset, data, salt):
    return "Data verification failed. Offset: %d; Expected value: %d; Actual value: %d" % (
        offset, int(expected_pattern(offset, 1, salt)[0]), data[offset])


def test_reference_pattern_matches_golden_vectors():
    with open(GOLDEN_PATH) as f:
        golden = json.load(f)["pattern_closed_form"]
    assert golden
    for vec in golden:
        got = expected_pattern(vec["fileOffset"], vec["len"], vec["salt"]).tobytes()
        assert got.hex() == vec["hex"], vec


def rank_ranges(size, block, threads):
    """file mode, sequential: each rank gets a contiguous block range, the last rank also takes
    the remainder (LocalWorker.cpp:3576-3589) -> [(first byte, end byte)] by rank"""
    num_blocks = -(-size // block)
    std = num_blocks // threads
    out = []
    for rank in range(threads):
        first = rank * std
        end = num_blocks if rank == threads - 1 else first + std
        out.append((first * block, min(end * block, size)))
    return out


def corrupt(path, rng, block, worker_ends=()):
    """Write one corruption of every class into the file -> [(offset, bytes written)], in write
    order (later writes may overlap earlier ones; the count is taken from the file afterwards)."""
    size = os.path.getsize(path)
    assert size >= 4096 + 200
    num_blocks = -(-size // block)
    num_full = size // block
    writes = []
    with open(path, "r+b") as f:
        def cur(off):
            f.seek(off)
            return f.read(1)[0]

        def put(off, data):
            f.seek(off)
            f.write(bytes(data))
            writes.append((off, bytes(data)))

        def flip(off):
            put(off, [cur(off) ^ rng.randrange(1, 256)])

        flip(0)  # first byte of the file
        if num_blocks > 1:  # last byte of one block, first byte of the next
            boundary = block * rng.randrange(1, num_blocks)
            flip(boundary - 1)
            flip(boundary)
        for sub in range(1, 8):  # every byte position inside a pattern word
            flip((rng.randrange(8, size - 8) & ~7) | sub)
        if num_full:  # inside the < 32 byte tail of a block (the last vector if there is none)
            tail = block % 32 or 32
            flip(block * rng.randrange(num_full) + block - 1 - rng.randrange(tail))
        # 100 byte run across a block boundary (and so across a 32-byte vector boundary)
        boundary = block * rng.randrange(1, num_blocks) if num_blocks > 1 else size // 2
        start = min(max(boundary - 50, 0), size - 100)
        put(start, [rng.randrange(256) for _ in range(100)])
        # a zeroed 4 KiB region: pattern bytes that are 0 already do not count
        zero = rng.randrange(0, size - 4096) & ~4095
        assert 0 < mismatches(bytes(4096), zero, SALT)[0] < 4096
        put(zero, bytes(4096))
        own = rng.randrange(size)  # rewritten with its own value: not a mismatch
        put(own, [cur(own)])
        last_len = size - (num_blocks - 1) * block  # the last (maybe partial) block
        flip(size - 1 - rng.randrange(last_len))
        for end in worker_ends:  # the last block (so the last batch) of every worker
            flip(end - 1 - rng.randrange(min(block, end)))
    return writes


def corrupt_every_block(path, rng, block):
    """Random reads draw offsets with replacement: which blocks are read, and how often, is up to
    the generator. Flipping the same in-block positions of every full block keeps the expected
    count exact anyway: flips per block x blocks read. -> (writes, flips per block)"""
    size = os.path.getsize(path)
    # first and last byte, every position inside a pattern word, a run across a vector boundary
    rel = sorted({0, block - 1,
                  *[(rng.randrange(1, block // 8 - 1) * 8) | sub for sub in range(1, 8)],
                  *range(block // 2 - 20, block // 2 + 20)})
    writes = []
    with open(path, "r+b") as f:
        for base in range(0, size - block + 1, block):
            f.seek(base)
            data = bytearray(f.read(block))
            for pos in rel:
                data[pos] ^= rng.randrange(1, 256)
            f.seek(base)
            f.write(data)
            writes.append((base, bytes(data)))
    return writes, len(rel)


def restore(path, original, writes):
    with open(path, "r+b") as f:
        for off, data in writes:
            f.seek(off)
            f.write(original[off:off + len(data)])


def read_file(path):
    with open(path, "rb") as f:
        return f.read()


# ------------------------------------------------------------------------------------------------
# cases
# ------------------------------------------------------------------------------------------------

@dataclasses.dataclass
class Case:
    common: dict                       # WorkerConfig fields of the write and the read phase
    read: dict = dataclasses.field(default_factory=dict)   # read phase only
    write: dict = dataclasses.field(default_factory=dict)  # write phase only
    collect_all: bool = True           # the access pattern reads whole blocks
    several_threads: bool = False      # sequential with > 1 thread: per-rank first bad byte


CASES = {
    # tiled staged kernel, many batches per worker (BASELINE configs[1] shape, scaled down)
    "c2_like": Case(dict(num_threads=16, block_size=MiB, file_size=256 * MiB),
                    several_threads=True),
    # warp kernel (hint 4 KiB), aio with batches in flight (BASELINE configs[2] shape); random
    # reads, so collect-all counts flips that every block carries
    "c3_like": Case(dict(num_threads=2, block_size=4 * KiB, file_size=8 * MiB),
                    read=dict(use_random_offsets=True, rand_offset_seed=77,
                              io_engine=IOEngine.AIO, io_depth=64)),
    # warp kernel, partial last block
    "small_sync_4k": Case(dict(num_threads=2, block_size=4 * KiB, file_size=4 * MiB + 100,
                               io_engine=IOEngine.SYNC), several_threads=True),
    # warp kernel with its byte-wise tail (24 bytes per block)
    "small_sync_8k_minus_8": Case(dict(num_threads=2, block_size=8 * KiB - 8,
                                       file_size=(8 * KiB - 8) * 700 + 777,
                                       io_engine=IOEngine.SYNC), several_threads=True),
    # tile 0 byte-wise tails, partial last block of one byte
    "odd_block_1000": Case(dict(num_threads=2, block_size=1000, file_size=10001),
                           several_threads=True),
    "odd_block_64k_plus_3": Case(dict(num_threads=3, block_size=64 * KiB + 3,
                                      file_size=(64 * KiB + 3) * 40 + 12345),
                                 several_threads=True),
    # copy engine: per-batch graphs replayed (16 blocks a batch, 10 full batches per worker)
    "graph_replay": Case(dict(num_threads=2, block_size=64 * KiB, file_size=20 * MiB,
                              pipeline_batch_blocks=16), several_threads=True),
    # read block boundaries that are not write block boundaries
    "write_block_ne_read_block": Case(dict(num_threads=2, block_size=12 * KiB,
                                           file_size=6 * MiB + 5000),
                                      write=dict(block_size=MiB), several_threads=True),
    # unaligned random offsets: the funnel-shift pattern path; bytes may be read twice or never
    "unaligned_random": Case(dict(num_threads=1, block_size=12 * KiB, file_size=4 * MiB),
                             read=dict(use_random_offsets=True, use_random_unaligned=True,
                                       rand_offset_seed=9, random_amount=4 * MiB),
                             collect_all=False),
    # dir mode (BASELINE configs[4] shape): every file has its own offsets starting at 0
    "dir_mode": Case(dict(path_type=PathType.DIR, num_threads=3, num_dirs=2, num_files=3,
                          block_size=16 * KiB, file_size=64 * KiB)),
}


@pytest.fixture(params=[1, 2], ids=["kernel_staging", "copyengine_staging"])
def staging_engine(request):
    return request.param


@pytest.fixture()
def workdir(cuda_device):
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    path = tempfile.mkdtemp(prefix="elb_verify_det_", dir=base)
    yield path
    shutil.rmtree(path, ignore_errors=True)


def data_files(case, root):
    """the files a case reads, in a fixed order, with the file offset each starts at (0)"""
    if case.common.get("path_type") != PathType.DIR:
        return [root]
    return sorted(os.path.join(r, f) for r, _, fs in os.walk(root) for f in fs)


def config(case, path, phase_kwargs, **extra):
    kwargs = dict(case.common)
    kwargs.update(phase_kwargs)
    kwargs.update(extra)
    return WorkerConfig(paths=[path], integrity_check_salt=SALT, **kwargs)


def read_bytes_expected(case, cfg):
    if case.common.get("path_type") == PathType.DIR:
        return cfg.num_threads * cfg.num_dirs * cfg.num_files * cfg.file_size
    return cfg.random_amount or cfg.file_size


@pytest.mark.parametrize("name", list(CASES))
def test_corruption_is_reported_exactly(workdir, staging_engine, name):
    case = CASES[name]
    rng = random.Random(name)
    is_dir = case.common.get("path_type") == PathType.DIR
    root = os.path.join(workdir, "data")
    if is_dir:
        os.mkdir(root)
    eng = dict(staging_engine=staging_engine)

    with WorkerManager(config(case, root, case.write, **eng)) as mgr:
        if is_dir:
            mgr.run_phase(BenchPhase.CREATEDIRS)
        res = mgr.run_phase(BenchPhase.CREATEFILES)
        assert res["num_workers_done_with_error"] == 0

    files = data_files(case, root)
    originals = {}
    for path in files:
        originals[path] = read_file(path)
        assert mismatches(originals[path], 0, SALT)[0] == 0, path
    block = case.common["block_size"]
    threads = case.common["num_threads"]
    if is_dir:  # one corrupted file per rank
        victims = [os.path.join(root, "r%d" % r, "d%d" % (r % 2), "r%d-f%d" % (r, 1))
                   for r in range(threads)]
        ends = {p: () for p in victims}
    else:
        victims = files
        ends = {root: [end for _, end in rank_ranges(os.path.getsize(root), block, threads)]}

    def apply_corruption():
        return {p: corrupt(p, random.Random(rng.random()), block, ends[p]) for p in victims}

    def restore_all(writes):
        for p, w in writes.items():
            restore(p, originals[p], w)

    writes = apply_corruption()
    expected_count = sum(mismatches(read_file(p), 0, SALT)[0] for p in files)
    assert expected_count > 0

    # collect-all: the count of differing bytes, in every phase anew
    if case.collect_all:
        random_reads = case.read.get("use_random_offsets", False)
        if random_reads:
            restore_all(writes)
            every_block, per_block = corrupt_every_block(root, random.Random(name), block)
        cfg = config(case, root, case.read, verify_collect_all=True, **eng)
        with WorkerManager(cfg) as mgr:
            for rep in range(2):
                res = mgr.run_phase(BenchPhase.READFILES)
                assert res["num_workers_done_with_error"] == 0, rep
                assert res["verified_bytes"] == read_bytes_expected(case, cfg), rep
                count = per_block * (res["verified_bytes"] // block) if random_reads else \
                    expected_count
                assert res["verify_mismatch_bytes"] == count, rep
                snap = mgr.live_snapshot()
                assert snap["dev_counters"][DEVCTR_MISMATCH] == count, rep
        if random_reads:
            restore(root, originals[root], every_block)
            writes = apply_corruption()

    # stop at first, one thread: the oracle's text on a copy of the same corrupted data
    cfg1 = config(case, root, case.read, num_threads=1, **eng)
    oracle_root = os.path.join(workdir, "oracle_copy")
    (shutil.copytree if is_dir else shutil.copy)(root, oracle_root)
    ocfg = config(case, oracle_root, case.read, num_threads=1)
    rc, ow, _ = oracle_lib.run_oracle_phase(ocfg, BenchPhase.READFILES)
    assert rc != 0 and ow[0].hadError
    oracle_msg = ow[0].errorMsg.decode()
    if not is_dir and not case.read.get("use_random_offsets"):
        data = read_file(root)
        assert oracle_msg == verify_error_text(mismatches(data, 0, SALT)[1], data, SALT)
    with WorkerManager(cfg1) as mgr:
        with pytest.raises(WorkerError) as excinfo:
            mgr.run_phase(BenchPhase.READFILES)
        assert str(excinfo.value) == oracle_msg
        assert mgr.worker(0).last_error == oracle_msg
        restore_all(writes)
        res = mgr.run_phase(BenchPhase.READFILES)
        assert res["num_workers_done_with_error"] == 0
        assert res["verify_mismatch_bytes"] == 0
        assert res["verified_bytes"] == read_bytes_expected(case, cfg1)

    # stop at first, several threads: each worker that fails names the first bad byte of its own
    # block range
    if case.several_threads:
        writes = apply_corruption()
        data = read_file(root)
        ranges = rank_ranges(len(data), block, threads)
        cfgn = config(case, root, case.read, **eng)
        with WorkerManager(cfgn) as mgr:
            with pytest.raises(WorkerError) as excinfo:
                mgr.run_phase(BenchPhase.READFILES)
            reported = {}
            for worker in mgr.workers():
                if not worker.last_error:
                    continue  # stopped by the manager after another worker's error
                lo, hi = ranges[worker.rank]
                first = mismatches(data[lo:hi], lo, SALT)[1]
                assert first is not None, worker.rank
                assert worker.last_error == verify_error_text(lo + first, data, SALT), worker.rank
                reported[worker.rank] = worker.last_error
            assert reported
            assert str(excinfo.value) in reported.values()
            restore_all(writes)
            res = mgr.run_phase(BenchPhase.READFILES)
            assert res["num_workers_done_with_error"] == 0
            assert res["verify_mismatch_bytes"] == 0
            assert res["verified_bytes"] == len(data)


# ------------------------------------------------------------------------------------------------
# cuFile batch engine and several GPUs: collect-all count
# ------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def mock_cufile():
    if not os.path.exists(MOCK_LIB):
        subprocess.run(["make", "-s", "-C", MOCK_DIR], check=True)
    return MOCK_LIB


def _collect_all_count(path, size, block, cfg_kwargs):
    """write path sequentially, corrupt it, count with collect-all twice -> list of results"""
    with WorkerManager(WorkerConfig(paths=[path], block_size=MiB, file_size=size,
                                    integrity_check_salt=SALT)) as mgr:
        mgr.run_phase(BenchPhase.CREATEFILES)
    random_reads = cfg_kwargs.get("use_random_offsets", False)
    if random_reads:
        _, per_block = corrupt_every_block(path, random.Random(path), block)
    else:
        threads = cfg_kwargs.get("num_threads", 1)
        corrupt(path, random.Random(path), block,
                [end for _, end in rank_ranges(size, block, threads)])
        expected = mismatches(read_file(path), 0, SALT)[0]
        assert expected > 0
    cfg = WorkerConfig(paths=[path], block_size=block, file_size=size, integrity_check_salt=SALT,
                       verify_collect_all=True, **cfg_kwargs)
    with WorkerManager(cfg) as mgr:
        for rep in range(2):
            res = mgr.run_phase(BenchPhase.READFILES)
            assert res["num_workers_done_with_error"] == 0, rep
            assert res["verified_bytes"] == size, rep
            if random_reads:
                expected = per_block * (size // block)
            assert res["verify_mismatch_bytes"] == expected, rep
            assert mgr.live_snapshot()["dev_counters"][DEVCTR_MISMATCH] == expected, rep
        return res


def test_cufile_batch_collect_all_count(workdir, mock_cufile):
    """--gds with iodepth 16 (cuFile batch API): the blocks land in the device slots only and are
    verified there (no staging engine takes part)"""
    _collect_all_count(os.path.join(workdir, "g"), 4 * MiB, 4 * KiB,
                       dict(num_threads=2, use_cufile=True, use_gds_buf_reg=True, io_depth=16,
                            use_random_offsets=True, rand_offset_seed=31))


@pytest.mark.parametrize("staging_engine", [1, 2], ids=["kernel_staging", "copyengine_staging"])
def test_multi_gpu_collect_all_count_is_reduced(workdir, staging_engine):
    """workers on two GPUs: the phase-end reduce of the device counter blocks over NCCL carries
    the exact mismatch count"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    res = _collect_all_count(os.path.join(workdir, "mg"), 64 * MiB, MiB,
                             dict(num_threads=4, gpu_ids=(0, 1), staging_engine=staging_engine))
    assert res["stats_reduced_with_nccl"]
