"""Pin the CPU oracle: against the committed golden vectors generated from the reference's own
headers (tests/golden/ref_vectors.json) and against those headers' answers to additional seeded
random cases (tests/golden/ref_recorded.json). No GPU needed."""
import ctypes
import hashlib
import json
import os
import random

import pytest

from tests import oracle_lib
from tests.golden import make_golden
from tests.golden.make_golden import pattern_closed_form

GOLDEN_PATH = os.path.join(os.path.dirname(__file__), "golden", "ref_vectors.json")


@pytest.fixture(scope="module")
def golden():
    with open(GOLDEN_PATH) as f:
        return json.load(f)


def test_pattern_matches_closed_form_golden(oracle, golden):
    for vec in golden["pattern_closed_form"]:
        got = oracle_lib.fill_pattern(vec["len"], vec["fileOffset"], vec["salt"])
        assert got.hex() == vec["hex"], vec


def test_pattern_survey_vector(oracle):
    # SURVEY.md §8c: salt 1 -> file bytes 0..15
    assert oracle_lib.fill_pattern(16, 0, 1) == bytes.fromhex("0100000000000000" "0900000000000000")


def test_pattern_random_offsets_vs_closed_form(oracle):
    rng = random.Random(1234)
    for _ in range(200):
        length = rng.choice([0, 1, 2, 7, 8, 9, 15, 16, 17, 31, 63, 64, 100, 4096, 5000])
        offset = rng.choice([0, 1, 5, 8, 4095, 1 << 20, (1 << 40) + 3, rng.getrandbits(48)])
        salt = rng.choice([1, 2, 0xFFFFFFFFFFFFFFFF, rng.getrandbits(64)])
        assert oracle_lib.fill_pattern(length, offset, salt) == \
            pattern_closed_form(length, offset, salt)


def test_pattern_block_size_independence(oracle):
    """tools/test-examples.sh:226,243: write -b 1m, read back -b 128k must verify."""
    salt = 1
    whole = oracle_lib.fill_pattern(3 * 4096 + 100, 0, salt)
    for block in (1, 7, 512, 1000, 4096):
        pieces = b"".join(oracle_lib.fill_pattern(min(block, len(whole) - off), off, salt)
                          for off in range(0, len(whole), block))
        assert pieces == whole


def test_verify_ok_and_error_text(oracle):
    data = bytearray(oracle_lib.fill_pattern(4096, 8192, 7))
    assert oracle_lib.verify_pattern(data, 8192, 7)[0] == 0
    data[100] ^= 0xFF
    data[3000] ^= 0x01
    rc, num, first, exp, act, msg = oracle_lib.verify_pattern(data, 8192, 7)
    assert (rc, num, first) == (1, 2, 100)
    assert exp == pattern_closed_form(1, 8192 + 100, 7)[0]
    assert act == data[100]
    # exact text of LocalWorker.cpp:2174-2177
    assert msg == "Data verification failed. Offset: %d; Expected value: %d; Actual value: %d" % (
        8192 + 100, exp, act)
    # wrong salt: every word differs somewhere
    rc, num, first, *_ = oracle_lib.verify_pattern(oracle_lib.fill_pattern(64, 0, 1), 0, 2)
    assert rc == 1 and first == 0 and num == 8


def test_verify_empty_buffer(oracle):
    assert oracle_lib.verify_pattern(b"", 0, 1)[0] == 0  # LocalWorker.cpp:2140-2141


def test_buf_fill(oracle):
    for length in (0, 1, 7, 8, 9, 16, 21):
        buf = ctypes.create_string_buffer(max(1, length))
        oracle.orc_buf_fill(buf, 0x1122334455667788, length)
        expected = (0x1122334455667788).to_bytes(8, "little") * 4
        assert buf.raw[:length] == expected[:length]


def test_xoshiro_golden(oracle, golden):
    for vec in golden["xoshiro256ss"]:
        st = oracle_lib.Xoshiro256ss()
        st.s[:] = vec["state"]
        assert [oracle.orc_xoshiro256ss_next(ctypes.byref(st)) for _ in range(16)] == vec["next16"]
        buf = ctypes.create_string_buffer(37)
        oracle.orc_xoshiro256ss_fill_buf(ctypes.byref(st), buf, 37)
        assert buf.raw.hex() == vec["then_fill37_hex"]


def test_goldenprime_golden(oracle, golden):
    for vec in golden["goldenprime"]:
        st = oracle_lib.GoldenPrime()
        oracle.orc_goldenprime_init(ctypes.byref(st), vec["seed"],
                                    oracle_lib.u64x4(vec["seeder_state"]))
        assert [oracle.orc_goldenprime_next(ctypes.byref(st)) for _ in range(8)] == vec["next8"]
        buf = ctypes.create_string_buffer(vec["fill_len"])
        oracle.orc_goldenprime_fill_buf(ctypes.byref(st), buf, vec["fill_len"])
        assert hashlib.sha256(buf.raw).hexdigest() == vec["fill_sha256"]
        assert buf.raw[:64].hex() == vec["fill_first64_hex"]
        assert buf.raw[-16:].hex() == vec["fill_last16_hex"]
        assert oracle.orc_goldenprime_next(ctypes.byref(st)) == vec["next_after_fill"]


def test_goldenprime_survey_known_answer(oracle):
    # SURVEY.md §8c: RandAlgoGoldenPrime(12345) -> first two next()
    st = oracle_lib.GoldenPrime()
    oracle.orc_goldenprime_init(ctypes.byref(st), 12345, oracle_lib.u64x4([1, 2, 3, 4]))
    assert oracle.orc_goldenprime_next(ctypes.byref(st)) == 0x14259c4569db3215
    assert oracle.orc_goldenprime_next(ctypes.byref(st)) == 0x099e3ccb3809e8f7


def test_randalgo_golden(oracle, golden):
    """the four --randalgo generators (RandAlgoSelectorTk.cpp:37-53) for injected states"""
    assert {vec["algo"] for vec in golden["randalgo"]} == {0, 1, 2, 3}
    for vec in golden["randalgo"]:
        algo = oracle.orc_randalgo_create(vec["algo"], oracle_lib.u64x4(vec["state"]))
        assert algo
        nexts = [oracle.orc_randalgo_next(algo) for _ in range(700)]
        oracle.orc_randalgo_destroy(algo)
        assert nexts[:8] == vec["next8"], vec["algo"]
        assert nexts[-1] == vec["last"]
        digest = hashlib.sha256(b"".join(v.to_bytes(8, "little") for v in nexts)).hexdigest()
        assert digest == vec["next700_sha256"], vec["algo"]


def test_randalgo_mt19937_64_known_answer(oracle):
    # C++ standard [rand.predef]: the 10000th invocation of a default-constructed mt19937_64
    # (seed 5489) produces 9981545732273789042
    algo = oracle.orc_randalgo_create(3, oracle_lib.u64x4([5489, 0, 0, 0]))
    val = 0
    for _ in range(10000):
        val = oracle.orc_randalgo_next(algo)
    oracle.orc_randalgo_destroy(algo)
    assert val == 9981545732273789042


def test_randalgo_invalid(oracle):
    assert not oracle.orc_randalgo_create(4, oracle_lib.u64x4([1, 2, 3, 4]))


def test_offsetgen_randalgo_golden(oracle, golden):
    assert golden["offsetgen_randalgo"]
    for vec in golden["offsetgen_randalgo"]:
        seq = oracle_lib.offsetgen_sequence(
            oracle, "orc", vec["kind"], vec["numBytesTotal"], vec["len"], vec["offset"],
            vec["blockSize"], vec["numDataSetThreads"], vec["randState"], vec["lcgSeed"],
            rand_algo=vec["algo"])
        assert [list(x) for x in seq] == vec["sequence"], (vec["algo"], vec["kind"])


def test_randalgo_live_vs_reference_headers(oracle, recorded):
    """random injected states against the answers of the reference's headers
    (recorded by tests/golden/make_golden.py)"""
    cases = make_golden.randalgo_cases()
    assert len(cases) == len(recorded["randalgo"])
    for (algo_id, state), want in zip(cases, recorded["randalgo"]):
        algo = oracle.orc_randalgo_create(algo_id, oracle_lib.u64x4(state))
        nexts = [oracle.orc_randalgo_next(algo) for _ in range(1000)]
        oracle.orc_randalgo_destroy(algo)
        assert nexts[:8] == want["next8"], algo_id
        assert make_golden.u64_digest(nexts) == want["next1000_sha256"], algo_id
        for args, seq in zip(make_golden.RANDALGO_OFFSETGEN_ARGS, want["offsetgen_sequences"]):
            got = oracle_lib.offsetgen_sequence(oracle, "orc", *args, state, 0, rand_algo=algo_id)
            assert [list(x) for x in got] == seq, (algo_id, args[0])


def test_offsetgen_golden(oracle, golden):
    for vec in golden["offsetgen"]:
        seq = oracle_lib.offsetgen_sequence(
            oracle, "orc", vec["kind"], vec["numBytesTotal"], vec["len"], vec["offset"],
            vec["blockSize"], vec["numDataSetThreads"], vec["randState"], vec["lcgSeed"])
        assert [list(x) for x in seq] == vec["sequence"], vec["kind"]


def test_offsetgen_fullcoverage_multi_cycle_is_permutation_per_cycle(oracle):
    block, nblocks = 512, 37
    seq = oracle_lib.offsetgen_sequence(oracle, "orc", oracle_lib.OFFGEN_FULLCOV,
                                        3 * nblocks * block, nblocks * block, 0, block, 1,
                                        [1, 2, 3, 4], 5)
    assert len(seq) == 3 * nblocks
    for cycle in range(3):
        offs = sorted(off for off, _ in seq[cycle * nblocks:(cycle + 1) * nblocks])
        assert offs == [i * block for i in range(nblocks)]


def test_offsetgen_fullcoverage_covers_every_block(oracle):
    """tools/test-examples.sh:373-387 pins full coverage of the default random-write generator."""
    block, nblocks, first = 4096, 1000, 17
    seq = oracle_lib.offsetgen_sequence(oracle, "orc", oracle_lib.OFFGEN_FULLCOV, nblocks * block,
                                        nblocks * block, first * block, block, 1, [1, 2, 3, 4], 99)
    assert sorted(off for off, _ in seq) == [(first + i) * block for i in range(nblocks)]


def test_offsetgen_live_vs_reference_headers(oracle, recorded):
    """random geometries, states and seeds of all six generators against the answers of the
    reference's headers (recorded by tests/golden/make_golden.py)"""
    cases = make_golden.offsetgen_cases()
    assert len(cases) == len(recorded["offsetgen"])
    for case, want in zip(cases, recorded["offsetgen"]):
        got = oracle_lib.offsetgen_sequence(oracle, "orc", *case)
        assert [list(x) for x in got] == want, case[:6]


def test_prngs_live_vs_reference_headers(oracle, recorded):
    """golden prime buffer fills against the answers of the reference's headers (recorded by
    tests/golden/make_golden.py)"""
    cases = make_golden.goldenprime_cases()
    assert len(cases) == len(recorded["goldenprime"])
    for (state, seed, length), want in zip(cases, recorded["goldenprime"]):
        st = oracle_lib.GoldenPrime()
        oracle.orc_goldenprime_init(ctypes.byref(st), seed, oracle_lib.u64x4(state))
        obuf = ctypes.create_string_buffer(max(1, length))
        oracle.orc_goldenprime_fill_buf(ctypes.byref(st), obuf, length)
        assert hashlib.sha256(obuf.raw[:length]).hexdigest() == want["fill_sha256"], length
        assert oracle.orc_goldenprime_next(ctypes.byref(st)) == want["next_after_fill"]


def test_rand_refill_layout(oracle):
    """LocalWorker.cpp:2209-2230: first len*pct/100 bytes random, rest one repeated u64."""
    st = oracle_lib.GoldenPrime()
    oracle.orc_goldenprime_init(ctypes.byref(st), 777, oracle_lib.u64x4([5, 6, 7, 8]))
    buf = ctypes.create_string_buffer(1000)
    oracle.orc_rand_refill_goldenprime(ctypes.byref(st), buf, 1000, 30)
    tail = buf.raw[300:]
    assert tail == (tail[:8] * 100)[:700]


def test_fill_random_ctr_layout(oracle):
    """GPU layout (LocalWorker.cpp:2236-2277): varFillLen rounded down to x4, remainder repeated."""
    data = oracle_lib.fill_random_ctr(1001, 33, 42, 7)
    var_len = (1001 * 33 // 100) & ~3
    tail = data[var_len:]
    assert tail == (tail[:8] * 200)[:len(tail)]
    assert oracle_lib.fill_random_ctr(1001, 33, 42, 7) == data          # deterministic
    assert oracle_lib.fill_random_ctr(1001, 33, 42, 8)[:8] != data[:8]  # counter keyed
    assert oracle_lib.fill_random_ctr(64, 0, 42, 7) == oracle_lib.fill_random_ctr(64, 0, 42, 7)[:8] * 8
    full = oracle_lib.fill_random_ctr(4096, 100, 1, 0)
    assert len(set(full[i:i + 8] for i in range(0, 4096, 8))) == 512


def test_histogram_and_units(oracle):
    from elbencho_b200._native import Histogram
    histo = Histogram()
    oracle.orc_histogram_reset(ctypes.byref(histo))
    for lat in (0, 1, 2, 3, 4, 100, 1 << 27, (1 << 28) + 5, 1 << 40):
        oracle.orc_histogram_add_latency(ctypes.byref(histo), lat)
    assert histo.buckets[0] == 2          # 0 and 1 usec (log2(1)*4 = 0)
    assert histo.buckets[4] == 1          # 2 usec
    assert histo.buckets[6] == 1          # 3 usec: floor(log2(3)*4) = 6
    assert histo.buckets[8] == 1          # 4 usec
    assert histo.buckets[26] == 1         # 100 usec: floor(6.64*4)
    assert histo.buckets[108] == 1        # 2^27
    assert histo.buckets[111] == 2        # clamped (LatencyHistogram.h:73-74)
    assert histo.numStoredValues == 9 and histo.minMicroSecLat == 0
    assert histo.maxMicroSecLat == 1 << 40
    # UnitTk.h:48-56: total * (1e6 / usec) in double, truncated
    assert oracle.orc_per_sec_from_usec(1 << 30, 1000000) == 1 << 30
    assert oracle.orc_per_sec_from_usec(1000, 3) == int(1000 * (1000000.0 / 3))
