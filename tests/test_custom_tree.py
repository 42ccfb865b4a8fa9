"""Custom tree mode (--treefile): tree file parsing and the per-worker partition of the product
against an independent Python restatement (tests/tree_model.py); CLI dry run totals; tree scan."""
import base64
import ctypes
import os
import random
import subprocess

import pytest

from elbencho_b200.build import CLI_PATH
from tests import tree_model

KiB = 1 << 10
MiB = 1 << 20


def product_list(native, tree_path, block, share, round_up, rank, nthreads, kind):
    buf = ctypes.create_string_buffer(1 << 20)
    res = native.elb_custom_tree_worker_list(str(tree_path).encode(), block, share, round_up, rank,
                                             nthreads, kind, buf, len(buf))
    assert res >= 0, native.elb_last_error()
    rows = []
    for line in buf.value.decode().splitlines():
        path, total, start, length = line.split("\t")
        rows.append((path, int(total), int(start), int(length)))
    return rows


def make_tree_text(rng, nfiles, ndirs, block):
    lines = ["# generated for the test"]
    dirs = set()
    for i in range(ndirs):
        depth = rng.randrange(1, 4)
        dirs.add("/".join("dir%d" % rng.randrange(6) for _ in range(depth)))
    for d in sorted(dirs):
        lines.append("d " + d)
    for i in range(nfiles):
        size = rng.choice([0, 1, 777, block - 1, block, block + 1, 5 * block, 31 * block,
                           32 * block, 33 * block + 5, 100 * block, rng.randrange(200 * block)])
        lines.append("f %d %s/file with space %d.bin" % (size, rng.choice(sorted(dirs)), i))
    lines.append("x ignored line")
    return "\n".join(lines) + "\n"


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_worker_sublists_match_python_restatement(native, tmp_path, seed):
    rng = random.Random(seed)
    block = rng.choice([4 * KiB, 64 * KiB])
    text = make_tree_text(rng, 40, 8, block)
    tree_path = tmp_path / "tree.txt"
    tree_path.write_text(text)
    dirs, files = tree_model.parse_tree(text)
    for nthreads in (1, 3, 7):
        for share, round_up in ((0, 0), (8 * block, 0), (0, 4096), (1 << 62, 0)):
            seen_bytes = 0
            for rank in range(nthreads):
                got = product_list(native, tree_path, block, share, round_up, rank, nthreads, 1)
                want = tree_model.worker_files(files, rank, nthreads, block, share, round_up)
                assert got == want, (nthreads, share, round_up, rank)
                seen_bytes += sum(row[3] for row in got)
                got_dirs = product_list(native, tree_path, block, share, round_up, rank,
                                        nthreads, 0)
                assert [row[0] for row in got_dirs] == tree_model.worker_dirs(dirs, rank, nthreads)
            # every byte of every file is handed out exactly once
            sizes = [s if not (round_up and s % round_up) else s - s % round_up + round_up
                     for _, s in files]
            assert seen_bytes == sum(sizes)


def test_base64_tree_file_and_scan_round_trip(native, tmp_path):
    """FileTk::scanCustomTree writes base64 paths behind a '# encoding=base64' header"""
    root = tmp_path / "data"
    (root / "a" / "b").mkdir(parents=True)
    (root / "c d").mkdir()
    (root / "a" / "one.bin").write_bytes(b"x" * 1000)
    (root / "a" / "b" / "two  spaces.bin").write_bytes(b"y" * 70000)
    (root / "c d" / "empty").write_bytes(b"")
    tree_path = tmp_path / "scan.txt"
    found = native.elb_custom_tree_scan(str(root).encode(), str(tree_path).encode())
    assert found == 6  # 3 dirs + 3 files
    lines = tree_path.read_text().splitlines()
    assert lines[0] == "# encoding=base64"
    decoded = sorted(base64.b64decode(line.split()[-1]).decode() for line in lines[1:])
    assert decoded == sorted(["a", "a/b", "c d", "a/one.bin", "a/b/two  spaces.bin",
                              "c d/empty"])
    files = product_list(native, tree_path, 4096, 0, 0, 0, 1, 1)
    assert sorted(files) == sorted([("a/one.bin", 1000, 0, 1000), ("c d/empty", 0, 0, 0),
                                    ("a/b/two  spaces.bin", 70000, 0, 70000)])
    dirs = product_list(native, tree_path, 4096, 0, 0, 0, 1, 0)
    assert [d[0] for d in dirs] == sorted(["a", "a/b", "c d"], key=lambda p: (len(p), p))


def test_tree_file_errors(native, tmp_path):
    bad = tmp_path / "bad.txt"
    bad.write_text("f notanumber some/path\n")
    buf = ctypes.create_string_buffer(64)
    assert native.elb_custom_tree_worker_list(str(bad).encode(), 4096, 0, 0, 0, 1, 1, buf, 64) == -1
    assert b"invalid file line without size" in native.elb_last_error()
    assert native.elb_custom_tree_worker_list(str(tmp_path / "none").encode(), 4096, 0, 0, 0, 1, 1,
                                              buf, 64) == -1
    assert b"Opening input file failed" in native.elb_last_error()


def test_cli_dryrun_totals_and_validation(tmp_path):
    tree_path = tmp_path / "tree.txt"
    tree_path.write_text("d sub\nf 1048576 sub/a\nf 3145728 sub/b\nf 100 c\n")
    bench_dir = tmp_path / "bench"
    bench_dir.mkdir()
    res = subprocess.run([CLI_PATH, "--dryrun", "-d", "-w", "-r", "-t", "2", "-b", "64K",
                          "--treefile", str(tree_path), "--gpuids", "0", str(bench_dir)],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    # (WorkerManager.cpp:406-450: entries and bytes per thread = totals / dataset threads)
    assert "* Entries per thread: 1 |" in res.stdout  # 3 files / 2
    assert "* Bytes per thread:   %d |" % ((1048576 + 3145728 + 100) // 2) in res.stdout
    res = subprocess.run([CLI_PATH, "-w", "--treefile", str(tree_path), "--gpuids", "0", "-s", "1M",
                          str(tmp_path / "afile.bin")], capture_output=True, text=True)
    assert res.returncode == 1
    assert "Custom tree mode requires benchmark path to be a directory." in res.stderr


def test_partition_matches_reference_pathstore_golden(native, tmp_path):
    """golden lists produced by the reference's own PathStore.cpp (compiled in place into
    oracle/_ref, oracle/ref_harness_tree.cpp): dirs and files per worker, byte for byte"""
    import json
    with open(os.path.join(os.path.dirname(__file__), "golden", "ref_vectors.json")) as f:
        golden = json.load(f)["custom_tree"]
    tree_path = tmp_path / "golden_tree.txt"
    tree_path.write_text(golden["tree_text"])
    buf = ctypes.create_string_buffer(1 << 20)
    for case in golden["cases"]:
        for rank, want in enumerate(case["per_rank"]):
            for kind, name in ((0, "dirs"), (1, "files")):
                res = native.elb_custom_tree_worker_list(
                    str(tree_path).encode(), case["blockSize"], case["fileShareSize"],
                    case["treeRoundUpSize"], rank, case["numDataSetThreads"], kind, buf, len(buf))
                assert res >= 0
                assert buf.value.decode() == want[name], (case["numDataSetThreads"], rank, name)


def test_partition_live_against_reference_pathstore(native, recorded, tmp_path):
    """random trees against the reference's own PathStore.cpp (digests of its dir and file lists
    per worker, recorded by tests/golden/make_golden.py)"""
    from tests.golden import make_golden
    cases = make_golden.custom_tree_cases()
    assert len(cases) == len(recorded["custom_trees"])
    buf = ctypes.create_string_buffer(1 << 20)
    for round_idx, ((block, tree_text, splits), want) in enumerate(
            zip(cases, recorded["custom_trees"])):
        tree_path = tmp_path / ("tree%d.txt" % round_idx)
        tree_path.write_text(tree_text)
        for (nthreads, share, round_up), digests in zip(splits, want):
            got = []
            for rank in range(nthreads):
                for kind in (0, 1):
                    args = (str(tree_path).encode(), block, share, round_up, rank, nthreads, kind)
                    assert native.elb_custom_tree_worker_list(*args, buf, len(buf)) >= 0
                    got.append(make_golden.tree_list_digest(buf.value.decode()))
            assert got == digests, (block, nthreads, share, round_up)
