"""Histogram arithmetic, percentile rule, per-second rule and the human-readable number formats of
the result table, pinned to the REFERENCE's own LatencyHistogram.h and toolkits/UnitTk.{h,cpp}
through golden vectors (tests/golden/make_golden.py, oracle/ref_harness_stats.cpp): the oracle's
restatement and the product's C ABI must both reproduce them."""
import ctypes
import json
import os

import pytest

from elbencho_b200._native import Histogram
from tests.golden import make_golden

GOLDEN_PATH = os.path.join(os.path.dirname(__file__), "golden", "ref_vectors.json")


@pytest.fixture(scope="module")
def golden():
    with open(GOLDEN_PATH) as f:
        return json.load(f)


def fmt(native, kind, value=0, pct=0.0, histo=None):
    buf = ctypes.create_string_buffer(8192)
    res = native.elb_format_value(kind, value, pct, ctypes.byref(histo) if histo else None, buf,
                                  len(buf))
    assert res >= 0, native.elb_last_error()
    return buf.value.decode()


def test_product_histogram_matches_reference(native, golden):
    for vec in golden["latency_histogram"]:
        histo = Histogram()
        native.elb_histogram_reset(ctypes.byref(histo))
        for lat in vec["latencies"]:
            native.elb_histogram_add_latency(ctypes.byref(histo), lat)
        assert len(histo.buckets) == vec["num_buckets"]
        assert list(histo.buckets) == vec["buckets"]
        assert histo.numStoredValues == vec["num"]
        assert histo.numMicroSecTotal == vec["sum"]
        assert histo.minMicroSecLat == vec["min"] and histo.maxMicroSecLat == vec["max"]
        assert fmt(native, 3, histo=histo) == vec["histogram_str"]
        for pct, want in vec["percentiles"].items():
            got = native.elb_histogram_percentile(ctypes.byref(histo), float(pct))
            assert got == pytest.approx(want["value"], rel=1e-12), pct
            assert fmt(native, 4, pct=float(pct), histo=histo) == want["str"], pct


def test_oracle_histogram_matches_reference(oracle, golden):
    for vec in golden["latency_histogram"]:
        histo = Histogram()
        oracle.orc_histogram_reset(ctypes.byref(histo))
        for lat in vec["latencies"]:
            oracle.orc_histogram_add_latency(ctypes.byref(histo), lat)
        assert list(histo.buckets) == vec["buckets"]
        assert (histo.numStoredValues, histo.numMicroSecTotal, histo.minMicroSecLat,
                histo.maxMicroSecLat) == (vec["num"], vec["sum"], vec["min"], vec["max"])
        for pct, want in vec["percentiles"].items():
            got = oracle.orc_histogram_percentile(ctypes.byref(histo), float(pct))
            assert got == pytest.approx(want["value"], rel=1e-12), pct


def test_product_unit_formats_match_reference(native, golden):
    units = golden["units"]
    for val, want in units["latency_us"].items():
        assert fmt(native, 0, int(val)) == want, val
    for val, want in units["elapsed_ms"].items():
        assert fmt(native, 1, int(val)) == want, val
    for val, want in units["elapsed_sec"].items():
        assert fmt(native, 2, int(val)) == want, val
    for total, usec, want in units["per_sec"]:
        assert native.elb_per_sec_from_usec(total, usec) == want, (total, usec)
    out = ctypes.c_uint64()
    for text, want in units["human_to_bytes"].items():
        rc = native.elb_num_human_to_bytes(text.encode(), ctypes.byref(out))
        if isinstance(want, dict):
            assert rc == -1, text
            assert native.elb_last_error().decode() == want["error"], text
        else:
            assert rc == 0 and out.value == want, text


def test_oracle_per_sec_matches_reference(oracle, golden):
    for total, usec, want in golden["units"]["per_sec"]:
        assert oracle.orc_per_sec_from_usec(total, usec) == want


def test_live_against_reference_headers(native, oracle, recorded):
    """random latency sets, merged pairwise: product == oracle == the reference's class (its
    answers recorded by tests/golden/make_golden.py)"""
    cases = make_golden.histogram_merge_cases()
    assert len(cases) == len(recorded["histogram_merges"])
    for parts, want in zip(cases, recorded["histogram_merges"]):
        histos = []
        for lats in parts:
            mine, orc = Histogram(), Histogram()
            native.elb_histogram_reset(ctypes.byref(mine))
            oracle.orc_histogram_reset(ctypes.byref(orc))
            for lat in lats:
                native.elb_histogram_add_latency(ctypes.byref(mine), lat)
                oracle.orc_histogram_add_latency(ctypes.byref(orc), lat)
            histos.append((mine, orc))
        native.elb_histogram_merge(ctypes.byref(histos[0][0]), ctypes.byref(histos[1][0]))
        oracle.orc_histogram_merge(ctypes.byref(histos[0][1]), ctypes.byref(histos[1][1]))
        mine, orc = histos[0]
        assert list(mine.buckets) == list(orc.buckets) == want["buckets"]
        for histo in (mine, orc):
            assert histo.numStoredValues == want["num"]
            assert histo.numMicroSecTotal == want["sum"]
            if histo.numStoredValues:
                assert histo.minMicroSecLat == want["min"]
                assert histo.maxMicroSecLat == want["max"]
        if mine.numStoredValues:
            for pct, value in want["percentiles"].items():
                assert native.elb_histogram_percentile(ctypes.byref(mine), float(pct)) == \
                    pytest.approx(value, rel=1e-12)


def test_service_password_hash_matches_reference(native, golden):
    """HashTk::simple128 (toolkits/HashTk.cpp), incl. sign extension of non-ASCII bytes"""
    out = ctypes.create_string_buffer(33)
    for text, want in golden["units"]["simple128"].items():
        native.elb_simple128_hash(text.encode(), out)
        assert out.value.decode() == want, text
