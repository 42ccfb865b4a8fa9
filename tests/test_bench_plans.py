"""CPU tests of bench.py's step plans: the slices of all (rank, step) pairs tile every file exactly
once (the reference's --rankoffset sharding, LocalWorker.cpp:3576-3589), for one and two GPUs'
worth of files; run through the oracle (the reference arm's path)."""
import argparse
import os
import shutil
import tempfile

import pytest

import bench
from elbencho_b200 import BenchPhase, WorkerConfig
from tests import oracle_lib

MiB = 1 << 20


def make_args(workdir, **over):
    args = argparse.Namespace(gpus=1, steps=3, warmup=1, impl="reference", config="c2",
                              file_gib=24 / 1024, threads=2, dir=workdir, salt=5, direct=False)
    for key, val in over.items():
        setattr(args, key, val)
    return args


@pytest.fixture()
def workdir():
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    path = tempfile.mkdtemp(prefix="elb_benchplan_", dir=base)
    yield path
    shutil.rmtree(path, ignore_errors=True)


@pytest.mark.parametrize("world", [1, 2])
def test_c2_slices_tile_every_file_exactly_once(workdir, world):
    args = make_args(workdir, gpus=world)
    workload = bench.C2(args, world)
    assert workload.file_size % (workload.num_slices * workload.threads * MiB) == 0
    covered = [bytearray(workload.file_size // MiB) for _ in range(world)]
    block = workload.block
    for step in range(workload.num_slices):
        for rank in range(world):
            cfg, phases = workload.plan(step, rank)
            assert [p.name for p in phases] == ["CREATEFILES", "READFILES"]
            threads, total = cfg["num_threads"], cfg["num_dataset_threads"]
            blocks_total = world * workload.file_size // block
            per_rank = blocks_total // total
            for t in range(threads):
                g = cfg["rank_offset"] + t
                for blk in range(g * per_rank, (g + 1) * per_rank):
                    file_idx, in_file = divmod(blk, workload.file_size // block)
                    assert file_idx == rank  # a process only touches its own file
                    covered[file_idx][in_file] += 1
    assert all(set(c) == {1} for c in covered)

    # and through the oracle: all steps written -> every file verifies as a whole
    totals = bench.cpu_arm(workload, args.steps, args.warmup)
    assert totals["phase"]["CREATEFILES"]["bytes"] == args.steps * workload.slice_bytes * world
    assert totals["phase"]["READFILES"]["bytes"] == args.steps * workload.slice_bytes * world
    for path in workload.paths:
        assert os.path.getsize(path) == workload.file_size
        whole = WorkerConfig(paths=[path], num_threads=1, block_size=MiB,
                             file_size=workload.file_size, integrity_check_salt=args.salt)
        assert oracle_lib.run_oracle_phase(whole, BenchPhase.READFILES)[0] == 0


def test_config_objects_of_both_arms_are_equal(workdir):
    """what the driver compares for `same_config`"""
    for name in ("c2", "c3", "c4", "c5"):
        args = make_args(workdir, config=name, file_gib=32 / 1024)
        workload = bench.WORKLOADS[name](args, 1)
        assert bench.common_config(args, workload, 1) == bench.common_config(args, workload, 1)
        assert bench.common_config(args, workload, 1)["baseline_config"] == name


def test_c3_issues_the_file_worth_of_ios_over_the_timed_steps(workdir):
    args = make_args(workdir, config="c3", file_gib=16 / 1024, steps=4, warmup=1)
    workload = bench.C3(args, 1)
    assert workload.ios_per_step * args.steps * workload.block == workload.file_size
    totals = bench.cpu_arm(workload, args.steps, args.warmup)
    assert totals["iops"] == workload.ios_per_step * args.steps
    assert workload.value_of(totals) > 0


def test_c5_counts_files_and_reads_them_back(workdir):
    args = make_args(workdir, config="c5", file_gib=64 / 1024, steps=2, warmup=1)
    workload = bench.C5(args, 1)
    totals = bench.cpu_arm(workload, args.steps, args.warmup)
    files_per_step = workload.files_per_dir * workload.DIRS_PER_STEP * workload.threads
    assert totals["phase"]["CREATEFILES"]["entries"] == files_per_step * args.steps
    assert totals["phase"]["READFILES"]["entries"] == files_per_step * args.steps
    assert totals["phase"]["READFILES"]["bytes"] == files_per_step * args.steps * workload.block


@pytest.mark.parametrize("name", ["c2", "c5"])
def test_dump_outputs_samples_what_the_last_step_wrote(workdir, tmp_path, name):
    import numpy as np
    args = make_args(workdir, config=name, file_gib=(24 if name == "c2" else 64) / 1024)
    workload = bench.WORKLOADS[name](args, 1)
    bench.cpu_arm(workload, args.steps, args.warmup)
    last = args.warmup + args.steps - 1
    counters = {"ops_total": {"entries": 3, "bytes": 4 << 20, "iops": 4}, "verified_bytes": 7,
                "verify_mismatch_bytes": 0, "filled_bytes": 4 << 20}
    step_results = {"CREATEDIRS": counters, "CREATEFILES": counters, "READFILES": counters}
    dumps = [tmp_path / "a", tmp_path / "b"]
    for out in dumps:
        bench.dump_outputs(str(out), workload, last, 0, step_results)
    names = sorted(os.listdir(dumps[0]))
    assert names == ["createfiles_counters.npy", "readfiles_counters.npy", "written_sample.npy",
                     "written_sample_where.npy"]
    total = 0
    for fname in names:
        a, b = np.load(dumps[0] / fname), np.load(dumps[1] / fname)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b)  # seeded: repeatable
        total += a.nbytes
    assert total <= 64 << 20
    assert np.load(dumps[0] / "readfiles_counters.npy").tolist() == [3, 4 << 20, 4, 7, 0, 4 << 20]
    sample = np.load(dumps[0] / "written_sample.npy")
    where = np.load(dumps[0] / "written_sample_where.npy").astype(np.int64)
    regions = workload.written_regions(last, 0)
    assert sample.shape == (bench.DUMP_CHUNKS, min(bench.DUMP_CHUNK_BYTES,
                                                   min(r[2] for r in regions)))
    if name == "c2":
        assert regions == [(workload.paths[0], last * workload.slice_bytes, workload.slice_bytes)]
    for row, (idx, off) in zip(sample, where):
        path, start, length = regions[idx]
        assert 0 <= off <= length - sample.shape[1]
        want = oracle_lib.fill_pattern(sample.shape[1], start + off, args.salt)
        assert row.astype(np.uint8).tobytes() == want


@pytest.mark.parametrize("name", ["c2", "c3", "c4", "c5"])
@pytest.mark.parametrize("world", [1, 8])
def test_b200_arm_json_line_from_fake_measurements(workdir, name, world):
    """the line builder of the b200 arm is pure: feed it plausible measurements and check the
    contract keys (metric, value == e2e.value, roofline, cpu_baseline, config equality)"""
    import json
    args = make_args(workdir, config=name, gpus=world, file_gib=64 / 1024, steps=4, warmup=1,
                     staging="auto", batch_blocks=0, num_batches=0, write_gate="auto",
                     no_gpu_numa=False, window_gib=4.0)
    workload = bench.WORKLOADS[name](args, world)
    totals = bench.new_totals()
    if name != "c4":
        bench.add_phase(totals, "CREATEFILES", 4 << 30, 4096, 10, 1100000)
    bench.add_phase(totals, "READFILES", 4 << 30, 4096, 10, 130000)
    bench.add_phase(totals, "CREATEDIRS", 0, 0, 5, 1000)  # (not a timed phase)
    histo = {"buckets": [0] * 112, "num": 4096, "sum_usec": 4096 * 500, "min_usec": 100,
             "max_usec": 9000}
    histo["buckets"][36] = 4096
    extra = {"h2d_bytes": 4 << 30, "d2h_bytes": 4 << 30, "launches": 4096, "dev_kernel_usec": 300000,
             "verified_bytes": 4 << 30, "filled_bytes": 4 << 30, "histos": {"READFILES": histo}}
    kern = {"window_bytes": 4 << 30, "block_bytes": workload.block, "nblocks": 4096,
            "ms": {"fill": 0.57, "verify": 0.59, "rand": 0.62}, "launches": 39}
    pcie = {"copy_engine_h2d_gib_s": 50.0, "copy_engine_d2h_gib_s": 52.0,
            "stage_kernel_h2d_gib_s": 46.0, "stage_kernel_d2h_gib_s": 47.0, "note": "x"}
    value = workload.value_of(totals)
    storage = {"value": value * 1.05, "unit": workload.unit, "read_gib_s": 35.0,
               "write_gib_s": 3.9, "threads": 2, "note": "x"} if world == 1 else None
    cpu = {"value": value / 1.2, "unit": workload.unit, "cores": 2, "kind": "port",
           "sample": "x"} if world == 1 else None
    pool = {"value": 1.0, "unit": workload.unit} if world > 1 else None
    clocks = {"sm_mhz": 1965, "sm_max_mhz": 1965, "reasons": [], "samples": 10}
    line = bench.build_line(args, workload, world, value, totals, extra, {"CREATEFILES": {}} if
                            name in ("c3", "c4") else None, kern, pcie, storage, cpu, pool, clocks, 0.0)
    json.dumps(line)  # serialisable
    assert line["metric"] == workload.metric and line["unit"] == workload.unit
    assert line["value"] == line["e2e"]["value"] == round(value, 3) > 0
    assert line["n_gpus"] == world and line["steps"] == 4 and line["warmup"] == 1
    assert line["higher_is_better"] is True and line["scaling"] == "weak"
    assert line["vs_baseline"] is None and line["dtype"] == "u64"
    assert line["gpu_launches"] == 4096 and line["e2e"]["dev_kernel_usec"] == 300000
    assert line["e2e"]["h2d_bytes_per_step"] == (4 << 30) // 4
    assert line["roofline"]["bound"] == "hbm" and line["roofline"]["peak"] > 0
    assert 0 < line["roofline"]["frac"] == round(line["roofline"]["achieved"] /
                                                line["roofline"]["peak"], 4)
    assert set(line["roofline"]["all_kernels"]) == {"K1_fill_pattern", "K2_verify_pattern",
                                                    "K3_fill_random_pct100"}
    assert line["roofline"]["pcie"]["e2e_read_frac_of_pcie"] > 0
    assert line["config"] == bench.common_config(args, workload, world)  # == the reference arm's
    assert line["e2e"]["latency"]["READFILES"]["avg_usec"] == 500.0
    if world == 1:
        assert line["cpu_baseline"]["kind"] == "port" and "storage" in line["roofline"]
    else:
        assert line["extra"]["inprocess_pool"]["value"] == 1.0
    if name == "c4":
        assert line["roofline"]["kernel"].endswith("(K3)")
    if name == "c3":
        assert line["unit"] == "IOPS"
