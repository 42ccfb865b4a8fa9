"""CPU-only checks of the product library: it loads, exports every symbol include/*.h declares,
its struct layouts match the binding, and its host logic (offset plans, histogram, per-sec units)
equals the oracle / the reference golden vectors. No compute kernel is called here."""
import ctypes
import json
import os
import random
import re

import pytest

from elbencho_b200 import _native
from tests import oracle_lib

REPO_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(REPO_ROOT, "include", "elbencho_b200.h")
GOLDEN_PATH = os.path.join(os.path.dirname(__file__), "golden", "ref_vectors.json")


def declared_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(elb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(native):
    names = declared_functions()
    assert len(names) >= 40
    for name in names:
        assert hasattr(native, name), "declared in include/elbencho_b200.h but not exported: " + name


def test_binding_covers_every_declared_symbol():
    assert sorted(_native.SIGNATURES) == declared_functions()


def test_struct_layouts(native):
    assert native.elb_abi_version() == _native.ABI_VERSION
    assert native.elb_cfg_struct_size() == ctypes.sizeof(_native.Cfg)
    assert native.elb_phase_results_struct_size() == ctypes.sizeof(_native.PhaseResults)
    assert ctypes.sizeof(_native.BlockDesc) == 32
    assert ctypes.sizeof(_native.VerifyResult) == 16


def test_product_never_links_oracle():
    """the product path must not route through the oracle (no CPU fallback)"""
    import subprocess
    out = subprocess.run(["ldd", _native.lib_path()], capture_output=True, text=True).stdout
    assert "oracle" not in out and "elb_ref" not in out
    syms = subprocess.run(["nm", "-D", _native.lib_path()], capture_output=True, text=True).stdout
    assert "orc_" not in syms


def plan_sequence(native, kind, amount, range_len, range_offset, block, threads, state, lcg,
                  restarts=()):
    st = (ctypes.c_uint64 * 4)(*state)
    plan = native.elb_offset_plan_create(kind, amount, range_len, range_offset, block, threads, st,
                                         lcg, 1)
    assert plan
    out = []
    off = ctypes.c_uint64()
    length = ctypes.c_uint64()
    try:
        while native.elb_offset_plan_next(plan, ctypes.byref(off), ctypes.byref(length)):
            out.append((off.value, length.value))
            assert len(out) < 200000
        for restart in restarts:
            if restart is None:
                native.elb_offset_plan_restart(plan)
            else:
                native.elb_offset_plan_restart_range(plan, *restart)
            while native.elb_offset_plan_next(plan, ctypes.byref(off), ctypes.byref(length)):
                out.append((off.value, length.value))
    finally:
        native.elb_offset_plan_destroy(plan)
    return out


def test_offset_plans_match_reference_golden(native):
    with open(GOLDEN_PATH) as f:
        golden = json.load(f)
    for vec in golden["offsetgen"]:
        kind = vec["kind"]
        is_random = kind in (2, 3, 5)
        amount = vec["numBytesTotal"] if is_random else vec["len"]
        seq = plan_sequence(native, kind, amount, vec["len"], vec["offset"], vec["blockSize"],
                            vec["numDataSetThreads"], vec["randState"], vec["lcgSeed"])
        assert [list(x) for x in seq] == vec["sequence"], vec


def test_rand_algos_match_reference_golden(native):
    """--randalgo fast / balanced / balanced_single / strong: RandAlgoInterface::next() streams"""
    with open(GOLDEN_PATH) as f:
        golden = json.load(f)
    import hashlib
    for vec in golden["randalgo"]:
        st = (ctypes.c_uint64 * 4)(*vec["state"])
        algo = native.elb_rand_algo_create(vec["algo"], st)
        assert algo
        nexts = [native.elb_rand_algo_next(algo) for _ in range(700)]
        native.elb_rand_algo_destroy(algo)
        assert nexts[:8] == vec["next8"], vec["algo"]
        digest = hashlib.sha256(b"".join(v.to_bytes(8, "little") for v in nexts)).hexdigest()
        assert digest == vec["next700_sha256"], vec["algo"]
    assert not native.elb_rand_algo_create(9, (ctypes.c_uint64 * 4)(1, 2, 3, 4))


def test_offset_plans_with_rand_algos_match_reference_golden(native):
    with open(GOLDEN_PATH) as f:
        golden = json.load(f)
    for vec in golden["offsetgen_randalgo"]:
        st = (ctypes.c_uint64 * 4)(*vec["randState"])
        plan = native.elb_offset_plan_create_algo(
            vec["kind"], vec["numBytesTotal"], vec["len"], vec["offset"], vec["blockSize"],
            vec["numDataSetThreads"], vec["algo"], st, vec["lcgSeed"], 1)
        assert plan
        out = []
        off = ctypes.c_uint64()
        length = ctypes.c_uint64()
        while native.elb_offset_plan_next(plan, ctypes.byref(off), ctypes.byref(length)):
            out.append([off.value, length.value])
        native.elb_offset_plan_destroy(plan)
        assert out == vec["sequence"], (vec["algo"], vec["kind"])


def test_offset_plans_match_oracle_random_cases(native, oracle):
    rng = random.Random(4321)
    for _ in range(150):
        kind = rng.randrange(6)
        block = rng.choice([512, 4096, 65536, 1000, 1])
        nblocks = rng.randrange(1, 60)
        length = nblocks * block + (rng.randrange(block) if kind in (0, 1, 2, 3) else 0)
        offset = rng.randrange(0, 100) * block
        total = rng.randrange(1, 200) * block + rng.choice([0, 0, 17])
        threads = rng.randrange(1, 5)
        state = [rng.getrandbits(64) for _ in range(4)]
        lcg = rng.getrandbits(64)
        is_random = kind in (2, 3, 5)
        a = plan_sequence(native, kind, total if is_random else length, length, offset, block,
                          threads, state, lcg)
        b = oracle_lib.offsetgen_sequence(oracle, "orc", kind, total, length, offset, block,
                                          threads, state, lcg)
        assert a == b, (kind, total, length, offset, block)


def test_offset_plan_restarts_match_oracle(native, oracle):
    """reset() per file (dir mode) and reset(len, offset) per file piece (file mode)"""
    state = [11, 22, 33, 44]
    for kind in range(6):
        block, length, total = 4096, 10 * 4096, 6 * 4096
        restarts = [None, (5 * 4096 + 100 if kind < 4 else 5 * 4096, 3 * 4096), None]
        got = plan_sequence(native, kind, total if kind in (2, 3, 5) else length, length, 0,
                            block, 2, state, 77, restarts)
        gen = oracle.orc_offsetgen_create(kind, total, length, 0, block, 2,
                                          oracle_lib.u64x4(state), 77)
        exp = []

        def drain():
            while oracle.orc_offsetgen_bytes_left(gen):
                off = oracle.orc_offsetgen_next_offset(gen)
                blen = oracle.orc_offsetgen_next_block_size(gen)
                exp.append((off, blen))
                oracle.orc_offsetgen_add_bytes_submitted(gen, blen)
        drain()
        for restart in restarts:
            if restart is None:
                oracle.orc_offsetgen_reset(gen)
            else:
                oracle.orc_offsetgen_reset_range(gen, *restart)
            drain()
        oracle.orc_offsetgen_destroy(gen)
        assert got == exp, kind


def test_histogram_matches_oracle(native, oracle):
    rng = random.Random(7)
    a = _native.Histogram()
    b = _native.Histogram()
    native.elb_histogram_reset(ctypes.byref(a))
    oracle.orc_histogram_reset(ctypes.byref(b))
    for _ in range(5000):
        lat = rng.choice([0, 1, 2, 3, rng.randrange(1 << 10), rng.randrange(1 << 20),
                          rng.randrange(1 << 30), (1 << 28) - 1, 1 << 28])
        native.elb_histogram_add_latency(ctypes.byref(a), lat)
        oracle.orc_histogram_add_latency(ctypes.byref(b), lat)
    assert bytes(a) == bytes(b)
    for pct in (1, 50, 75, 99, 99.9):
        assert native.elb_histogram_percentile(ctypes.byref(a), pct) == \
            oracle.orc_histogram_percentile(ctypes.byref(b), pct)
    c = _native.Histogram()
    d = _native.Histogram()
    native.elb_histogram_reset(ctypes.byref(c))
    oracle.orc_histogram_reset(ctypes.byref(d))
    native.elb_histogram_merge(ctypes.byref(c), ctypes.byref(a))
    oracle.orc_histogram_merge(ctypes.byref(d), ctypes.byref(b))
    assert bytes(c) == bytes(d) == bytes(a)


def test_per_sec_matches_oracle(native, oracle):
    rng = random.Random(8)
    for _ in range(1000):
        total = rng.getrandbits(rng.randrange(1, 50))
        usec = rng.randrange(1, 1 << 36)
        assert native.elb_per_sec_from_usec(total, usec) == \
            oracle.orc_per_sec_from_usec(total, usec)


def test_seed_expansion_matches_oracle_convention(native):
    out = (ctypes.c_uint64 * 4)()
    native.elb_expand_offset_seed(1234, 3, out)
    # splitmix64 stream of (seed + rank*GOLDEN)
    mask = (1 << 64) - 1
    golden = 0x9E3779B97F4A7C15
    counter = (1234 + 3 * golden) & mask
    exp = []
    for _ in range(4):
        counter = (counter + golden) & mask
        z = counter
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & mask
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & mask
        exp.append(z ^ (z >> 31))
    assert list(out) == exp


def test_manager_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from elbencho_b200 import WorkerConfig, WorkerError, WorkerManager
    with pytest.raises(WorkerError):
        WorkerManager(WorkerConfig(paths=["/tmp/elb_nogpu_test.bin"], file_size=1 << 20))
    if os.path.exists("/tmp/elb_nogpu_test.bin"):
        os.unlink("/tmp/elb_nogpu_test.bin")


def test_config_validation_errors():
    from elbencho_b200 import WorkerConfig, WorkerError, WorkerManager
    with pytest.raises(WorkerError, match="No GPU IDs given"):
        WorkerManager(WorkerConfig(paths=["/tmp/x"], file_size=4096, gpu_ids=()))
    with pytest.raises(WorkerError, match="multiple of required size"):
        WorkerManager(WorkerConfig(paths=["/tmp/x"], file_size=4096 * 3, block_size=1000,
                                   use_direct_io=True))
    with pytest.raises(WorkerError, match="rwmixpct"):
        WorkerManager(WorkerConfig(paths=["/tmp/x"], file_size=4096, integrity_check_salt=1,
                                   rwmix_read_percent=10))


def test_nodiocheck_skips_the_direct_io_block_size_check(native):
    """ProgArgs.cpp:1566-1584: with --direct the block size has to be a multiple of 512 unless
    --nodiocheck is given (checked at configuration time, before any GPU is touched)"""
    from elbencho_b200 import WorkerConfig, WorkerError, WorkerManager
    common = dict(paths=["/tmp/elb_nodio.bin"], block_size=1000, file_size=8000,
                  use_direct_io=True, gpu_ids=[0])
    with pytest.raises(WorkerError, match="Block size for direct IO is not a multiple"):
        WorkerManager(WorkerConfig(**common))
    try:
        # gets past the check: the manager is created where there is a GPU, else fails on that
        WorkerManager(WorkerConfig(no_direct_io_check=True, **common)).close()
    except WorkerError as err:
        assert "Block size for direct IO" not in str(err)
    finally:
        if os.path.exists(common["paths"][0]):
            os.unlink(common["paths"][0])


@pytest.mark.parametrize("host_delta", [4, -8])
def test_staged_entry_points_reject_misaligned_host_delta(native, host_delta):
    """the staged kernels move 32-byte vectors to / from (devPtr + hostDelta): a hostDelta that is
    not a multiple of 32 is refused by the argument check, before anything reaches the GPU"""
    desc = _native.BlockDesc()  # never read: the check comes first
    ptr = ctypes.cast(ctypes.pointer(desc), ctypes.c_void_p)
    calls = {
        "elb_fill_pattern_staged": lambda: native.elb_fill_pattern_staged(
            ptr, 1, 1, host_delta, None, 4096, 4096, None),
        "elb_fill_random_staged": lambda: native.elb_fill_random_staged(
            ptr, 1, 50, 1, 0, host_delta, None, 4096, 4096, None),
        "elb_verify_pattern_staged": lambda: native.elb_verify_pattern_staged(
            ptr, 1, 1, host_delta, ptr, None, None, None, 4096, 4096, None),
        "elb_stage_copy": lambda: native.elb_stage_copy(ptr, 1, 1, host_delta, 4096, 4096, None),
    }
    for name, call in calls.items():
        assert call() == -1, name
        err = _native.last_error()
        assert err.startswith(name + ": hostDelta must be a multiple of 32"), err
        assert "Given: %d" % host_delta in err
