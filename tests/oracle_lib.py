"""TEST INFRASTRUCTURE: ctypes loaders for the CPU oracle (oracle/libelb_oracle.so) and for the
reference's own headers behind a C ABI (oracle/_ref/libelb_ref.so).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
"""
import ctypes
import os
import subprocess

from elbencho_b200._native import Cfg, Histogram, LiveOps, PhaseResults

REPO_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(REPO_ROOT, "oracle")
ORACLE_LIB = os.path.join(ORACLE_DIR, "libelb_oracle.so")
REF_LIB = os.path.join(ORACLE_DIR, "_ref", "libelb_ref.so")

c_u64 = ctypes.c_uint64
_VP = ctypes.c_void_p

# enum orc_offsetgen_kind (== elb_offset_plan kinds)
OFFGEN_SEQUENTIAL, OFFGEN_REVERSE_SEQ, OFFGEN_RANDOM, OFFGEN_RANDOM_ALIGNED, OFFGEN_STRIDED, \
    OFFGEN_FULLCOV = range(6)


class Xoshiro256ss(ctypes.Structure):
    _fields_ = [("s", c_u64 * 4)]


class GoldenPrime(ctypes.Structure):
    _fields_ = [("stateSeeder", Xoshiro256ss), ("state", c_u64),
                ("currentGoldenPrimeIdx", ctypes.c_uint)]


class WorkerResult(ctypes.Structure):
    _fields_ = [
        ("liveOps", LiveOps),
        ("liveOpsReadMix", LiveOps),
        ("iopsLatHisto", Histogram),
        ("entriesLatHisto", Histogram),
        ("elapsedUSec", c_u64),
        ("gotPhaseWork", ctypes.c_int32),
        ("hadError", ctypes.c_int32),
        ("errorMsg", ctypes.c_char * 512),
    ]


_oracle = None
_ref = None
_ref_tried = False


def _build_oracle():
    subprocess.run(["make", "-s", "-C", ORACLE_DIR], check=True)


def load_oracle():
    global _oracle
    if _oracle is not None:
        return _oracle
    src_mtime = max(os.path.getmtime(os.path.join(ORACLE_DIR, f))
                    for f in ("elb_oracle.c", "elb_oracle.h"))
    if not os.path.exists(ORACLE_LIB) or os.path.getmtime(ORACLE_LIB) < src_mtime:
        _build_oracle()
    lib = ctypes.CDLL(ORACLE_LIB)
    u64p = ctypes.POINTER(c_u64)
    uip = ctypes.POINTER(ctypes.c_uint)
    sigs = {
        "orc_fill_pattern": (None, [_VP, ctypes.c_size_t, c_u64, c_u64]),
        "orc_verify_pattern": (ctypes.c_int, [_VP, ctypes.c_size_t, c_u64, c_u64, u64p, u64p,
                                               uip, uip, ctypes.c_char_p, ctypes.c_size_t]),
        "orc_buf_fill": (None, [_VP, c_u64, ctypes.c_size_t]),
        "orc_xoshiro256ss_next": (c_u64, [ctypes.POINTER(Xoshiro256ss)]),
        "orc_xoshiro256ss_fill_buf": (None, [ctypes.POINTER(Xoshiro256ss), _VP, c_u64]),
        "orc_goldenprime_init": (None, [ctypes.POINTER(GoldenPrime), c_u64, u64p]),
        "orc_goldenprime_next": (c_u64, [ctypes.POINTER(GoldenPrime)]),
        "orc_goldenprime_fill_buf": (None, [ctypes.POINTER(GoldenPrime), _VP, c_u64]),
        "orc_rand_refill_goldenprime": (None, [ctypes.POINTER(GoldenPrime), _VP, ctypes.c_size_t,
                                               ctypes.c_uint]),
        "orc_fill_random_ctr": (None, [_VP, c_u64, ctypes.c_uint, c_u64, c_u64]),
        "orc_offsetgen_create": (_VP, [ctypes.c_int, c_u64, c_u64, c_u64, c_u64, c_u64, u64p,
                                        c_u64]),
        "orc_offsetgen_create_algo": (_VP, [ctypes.c_int, c_u64, c_u64, c_u64, c_u64, c_u64,
                                             ctypes.c_int, u64p, c_u64]),
        "orc_randalgo_create": (_VP, [ctypes.c_int, u64p]),
        "orc_randalgo_next": (c_u64, [_VP]),
        "orc_randalgo_destroy": (None, [_VP]),
        "orc_offsetgen_destroy": (None, [_VP]),
        "orc_offsetgen_reset": (None, [_VP]),
        "orc_offsetgen_reset_range": (None, [_VP, c_u64, c_u64]),
        "orc_offsetgen_next_offset": (c_u64, [_VP]),
        "orc_offsetgen_next_block_size": (c_u64, [_VP]),
        "orc_offsetgen_bytes_total": (c_u64, [_VP]),
        "orc_offsetgen_bytes_left": (c_u64, [_VP]),
        "orc_offsetgen_add_bytes_submitted": (None, [_VP, c_u64]),
        "orc_histogram_reset": (None, [ctypes.POINTER(Histogram)]),
        "orc_histogram_add_latency": (None, [ctypes.POINTER(Histogram), c_u64]),
        "orc_histogram_merge": (None, [ctypes.POINTER(Histogram), ctypes.POINTER(Histogram)]),
        "orc_histogram_percentile": (ctypes.c_double, [ctypes.POINTER(Histogram),
                                                       ctypes.c_double]),
        "orc_per_sec_from_usec": (c_u64, [c_u64, c_u64]),
        "orc_run_phase": (ctypes.c_int, [ctypes.POINTER(Cfg), ctypes.c_int,
                                          ctypes.POINTER(WorkerResult),
                                          ctypes.POINTER(PhaseResults)]),
        "orc_expected_per_worker": (None, [ctypes.POINTER(Cfg), ctypes.c_int, u64p, u64p]),
        "orc_bench_fill_pattern": (ctypes.c_double, [ctypes.c_size_t, ctypes.c_size_t]),
        "orc_bench_verify_pattern": (ctypes.c_double, [ctypes.c_size_t, ctypes.c_size_t]),
    }
    for name, (restype, argtypes) in sigs.items():
        func = getattr(lib, name)
        func.restype = restype
        func.argtypes = argtypes
    _oracle = lib
    return lib


def load_ref():
    """oracle/_ref/libelb_ref.so (reference headers compiled where they lie), or None."""
    global _ref, _ref_tried
    if _ref_tried:
        return _ref
    _ref_tried = True
    if not os.path.exists(REF_LIB):
        return None
    lib = ctypes.CDLL(REF_LIB)
    u64p = ctypes.POINTER(c_u64)
    sigs = {
        "ref_xoshiro256ss_create": (_VP, [u64p]),
        "ref_goldenprime_create": (_VP, [c_u64, u64p]),
        "ref_randalgo_next": (c_u64, [_VP]),
        "ref_randalgo_fill_buf": (None, [_VP, _VP, c_u64]),
        "ref_randalgo_destroy": (None, [_VP]),
        "ref_offsetgen_create": (_VP, [ctypes.c_int, c_u64, c_u64, c_u64, c_u64, c_u64, u64p,
                                        c_u64]),
        "ref_offsetgen_create_algo": (_VP, [ctypes.c_int, c_u64, c_u64, c_u64, c_u64, c_u64,
                                             ctypes.c_int, u64p, c_u64]),
        "ref_randalgo_create": (_VP, [ctypes.c_int, u64p]),
        # the reference's LatencyHistogram.h and UnitTk (oracle/ref_harness_stats.cpp)
        "ref_histogram_create": (_VP, []),
        "ref_histogram_destroy": (None, [_VP]),
        "ref_histogram_add": (None, [_VP, c_u64]),
        "ref_histogram_merge": (None, [_VP, _VP]),
        "ref_histogram_num": (c_u64, [_VP]),
        "ref_histogram_min": (c_u64, [_VP]),
        "ref_histogram_max": (c_u64, [_VP]),
        "ref_histogram_avg": (c_u64, [_VP]),
        "ref_histogram_sum": (c_u64, [_VP]),
        "ref_histogram_exceeded": (ctypes.c_int, [_VP]),
        "ref_histogram_percentile": (ctypes.c_double, [_VP, ctypes.c_double]),
        "ref_histogram_num_buckets": (c_u64, [_VP]),
        "ref_histogram_buckets": (None, [_VP, u64p]),
        "ref_histogram_str": (ctypes.c_int64, [_VP, ctypes.c_char_p, c_u64]),
        "ref_histogram_percentile_str": (ctypes.c_int64, [_VP, ctypes.c_double, ctypes.c_char_p,
                                                          c_u64]),
        "ref_per_sec_from_usec": (c_u64, [c_u64, c_u64]),
        "ref_simple128": (ctypes.c_int64, [ctypes.c_char_p, ctypes.c_char_p, c_u64]),
        # the reference's PathStore (oracle/ref_harness_tree.cpp)
        "ref_custom_tree_worker_list": (ctypes.c_int64, [ctypes.c_char_p, c_u64, c_u64, c_u64, c_u64,
                                                         c_u64, ctypes.c_int, ctypes.c_char_p,
                                                         c_u64]),
        "ref_unit_str": (ctypes.c_int64, [ctypes.c_int, c_u64, ctypes.c_char_p, c_u64]),
        "ref_num_human_to_bytes": (ctypes.c_int, [ctypes.c_char_p, u64p, ctypes.c_char_p, c_u64]),
        "ref_offsetgen_destroy": (None, [_VP]),
        "ref_offsetgen_reset": (None, [_VP]),
        "ref_offsetgen_reset_range": (None, [_VP, c_u64, c_u64]),
        "ref_offsetgen_next_offset": (c_u64, [_VP]),
        "ref_offsetgen_next_block_size": (c_u64, [_VP]),
        "ref_offsetgen_bytes_total": (c_u64, [_VP]),
        "ref_offsetgen_bytes_left": (c_u64, [_VP]),
        "ref_offsetgen_add_bytes_submitted": (None, [_VP, c_u64]),
        "ref_offsetgen_fullcov_set_state": (None, [_VP, c_u64]),
        "ref_offsetgen_fullcov_modulus": (c_u64, [_VP]),
    }
    for name, (restype, argtypes) in sigs.items():
        func = getattr(lib, name)
        func.restype = restype
        func.argtypes = argtypes
    _ref = lib
    return lib


# ---- convenience wrappers used by several tests -------------------------------------------------

def u64x4(values):
    return (c_u64 * 4)(*values)


def fill_pattern(length, file_offset, salt):
    buf = ctypes.create_string_buffer(max(1, length))
    load_oracle().orc_fill_pattern(buf, length, file_offset, salt)
    return buf.raw[:length]


def verify_pattern(data, file_offset, salt):
    """-> (rc, num_mismatch, first_idx, expected, actual, message)"""
    lib = load_oracle()
    buf = ctypes.create_string_buffer(bytes(data), max(1, len(data)))
    num = c_u64()
    first = c_u64()
    exp = ctypes.c_uint()
    act = ctypes.c_uint()
    msg = ctypes.create_string_buffer(512)
    rc = lib.orc_verify_pattern(buf, len(data), file_offset, salt, ctypes.byref(num),
                                ctypes.byref(first), ctypes.byref(exp), ctypes.byref(act), msg,
                                512)
    return rc, num.value, first.value, exp.value, act.value, msg.value.decode()


def fill_random_ctr(length, pct, seed, block_counter):
    buf = ctypes.create_string_buffer(max(1, length))
    load_oracle().orc_fill_random_ctr(buf, length, pct, seed, block_counter)
    return buf.raw[:length]


def offsetgen_sequence(lib, prefix, kind, num_bytes_total, length, offset, block_size,
                       num_dataset_threads, rand_state, lcg_seed, max_steps=100000, rand_algo=0):
    """Drive an offset generator the way rwBlockSized does (getNextOffset, getNextBlockSize,
    addBytesSubmitted(blockSize)) -> list of (offset, len). rand_algo: enum elb_offset_rand_algo."""
    create = getattr(lib, prefix + "_offsetgen_create_algo")
    state = u64x4(rand_state) if rand_state is not None else None
    gen = create(kind, num_bytes_total, length, offset, block_size, num_dataset_threads,
                 rand_algo, state, lcg_seed)
    assert gen
    if prefix == "ref" and kind == OFFGEN_FULLCOV:
        # the reference takes random_device()() (32 bit) % m as start state
        lib.ref_offsetgen_fullcov_set_state(gen, lcg_seed & 0xFFFFFFFF)
    out = []
    try:
        while getattr(lib, prefix + "_offsetgen_bytes_left")(gen) and len(out) < max_steps:
            off = getattr(lib, prefix + "_offsetgen_next_offset")(gen)
            blen = getattr(lib, prefix + "_offsetgen_next_block_size")(gen)
            out.append((off, blen))
            getattr(lib, prefix + "_offsetgen_add_bytes_submitted")(gen, blen)
    finally:
        getattr(lib, prefix + "_offsetgen_destroy")(gen)
    return out


def run_oracle_phase(config, phase):
    """Run one phase on the CPU oracle worker. config: elbencho_b200.WorkerConfig.
    -> (rc, [WorkerResult...], PhaseResults)"""
    lib = load_oracle()
    cfg, keepalive = config.to_abi()
    results = (WorkerResult * config.num_threads)()
    phase_results = PhaseResults()
    rc = lib.orc_run_phase(ctypes.byref(cfg), int(phase), results, ctypes.byref(phase_results))
    del keepalive
    return rc, list(results), phase_results
