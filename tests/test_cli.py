"""CPU-only tests of the command line front end: option parsing, the reference's validation
messages, dry-run counters of the BASELINE configs (SURVEY.md §8d), the result table / CSV / JSON
formats (checked against strings derived by hand from the reference's format code) and the JSON /
HTTP plumbing of service mode as far as it works without a GPU."""
import ctypes
import http.client
import json
import os
import socket
import subprocess
import sys
import time

import pytest

from elbencho_b200 import _native
from elbencho_b200.build import CLI_PATH
from elbencho_b200._native import PhaseResults

GiB = 1 << 30
MiB = 1 << 20


def run_cli(*args, timeout=60):
    return subprocess.run([CLI_PATH] + list(args), capture_output=True, text=True, timeout=timeout)


def test_cli_binary_exists_and_reports_version():
    res = run_cli("--version")
    assert res.returncode == 0 and "protocol 3.1.1" in res.stdout
    res = run_cli("--help")
    assert res.returncode == 0
    for opt in ("--gpuids", "--verify", "--blockvarpct", "--iodepth", "--gds", "--hosts",
                "--service", "-t [ --threads ]", "--rwmixpct", "--csvfile"):
        assert opt in res.stdout, opt


@pytest.mark.parametrize("args,entries,total_bytes", [
    # SURVEY.md §8d: C1/C2/C4/C5 expected counters per phase
    (["-w", "-r", "-t", "1", "-b", "1M", "-s", "1G", "--verify", "1", "--gpuids", "0", "/tmp/elb_dry"],
     1, 1073741824),
    (["-w", "-r", "-t", "1", "-b", "1M", "-s", "64G", "--verify", "1", "--gpuids", "0", "/tmp/elb_dry"],
     1, 64 * GiB),
    (["-r", "-t", "8", "-b", "1M", "-s", "32G", "--gpuids", "0-7", "--gds"] +
     ["/tmp/elb_dry%d" % i for i in range(8)], 8 * 8, 8 * 32 * GiB),
    (["-w", "-r", "-t", "128", "-n", "64", "-N", "128", "-s", "64K", "-b", "64K", "--verify", "1",
      "--gpuids", "[0-7]", "/tmp"], 1048576, 68719476736),
])
def test_dryrun_counters_of_baseline_configs(args, entries, total_bytes):
    res = run_cli("--dryrun", *args)
    assert res.returncode == 0, res.stderr
    phases = res.stdout.split("Phase: ")[1:]
    assert phases
    for phase in phases:
        lines = phase.splitlines()
        assert lines[2].startswith("* Entries total:      %d |" % entries)
        if lines[0] in ("WRITE", "READ"):
            assert lines[4].startswith("* Bytes total:        %d |" % total_bytes)


@pytest.mark.parametrize("algo", ["fast", "balanced", "balanced_single", "strong"])
def test_rand_algo_names_of_the_reference_are_accepted(algo):
    # RandAlgoSelectorTk.h:10-13
    res = run_cli("--dryrun", "-r", "-b", "4K", "-s", "1G", "--rand", "--randalgo", algo,
                  "--blockvaralgo", algo, "--gpuids", "0", "/tmp/elb_dry")
    assert res.returncode == 0, res.stderr


def test_config_file_options_and_paths(tmp_path):
    """--configfile: OPTIONNAME=VALUE lines, command line wins, path= lines (ProgArgs.cpp:1012-1030)"""
    cfg = tmp_path / "bench.conf"
    cfg.write_text("# comment\nwrite=1\nread = true\nblock=4K\nsize=1M\nthreads=2\n"
                   "gpuids=0\nverify=0\npath=/tmp/elb_dry_cfg\n")
    res = run_cli("--dryrun", "-c", str(cfg), "-t", "4")
    assert res.returncode == 0, res.stderr
    assert "WRITE" in res.stdout and "READ" in res.stdout
    # 1 MiB file / 4 threads (command line wins over threads=2)
    assert "* Bytes per thread:   %d |" % (MiB // 4) in res.stdout
    cfg.write_text("nosuchoption=1\n")
    res = run_cli("--dryrun", "-c", str(cfg), "-w", "--gpuids", "0", "/tmp/x")
    assert res.returncode == 1 and "unrecognised option 'nosuchoption'" in res.stderr
    res = run_cli("--dryrun", "-c", str(tmp_path / "missing.conf"), "-w", "--gpuids", "0", "/tmp/x")
    assert res.returncode == 1 and "Unable to read config file" in res.stderr


def test_hosts_file_numhosts_and_duplicates(tmp_path):
    """ProgArgs::parseHosts (ProgArgs.cpp:2221-2340)"""
    hosts = tmp_path / "hosts.txt"
    hosts.write_text("# services\nnode1:1611\nnode2\n")
    # --numhosts 0: ignore all hosts and run locally (here: dry run)
    res = run_cli("--dryrun", "-w", "-s", "1M", "--gpuids", "0", "--hostsfile", str(hosts),
                  "--numhosts", "0", "/tmp/elb_dry")
    assert res.returncode == 0, res.stderr
    res = run_cli("-w", "-s", "1M", "--gpuids", "0", "--hosts", "node1,node1", "/tmp/elb_dry")
    assert res.returncode == 1 and "List of hosts contains duplicates" in res.stderr
    res = run_cli("-w", "-s", "1M", "--gpuids", "0", "--hostsfile", str(tmp_path / "none"),
                  "/tmp/elb_dry")
    assert res.returncode == 1 and "Unable to read hosts file" in res.stderr
    # unreachable services: --svcwait bounds the wait (Coordinator.cpp:160-230)
    res = run_cli("-w", "-s", "1M", "--gpuids", "0", "--hosts", "127.0.0.1:1", "--svcwait", "1",
                  "/tmp/elb_dry", timeout=30)
    assert res.returncode == 1
    assert "Timed out waiting for services to become ready. Unreachable service: 127.0.0.1:1" \
        in res.stderr


def test_dryrun_detects_size_of_existing_file(tmp_path):
    path = tmp_path / "existing.bin"
    path.write_bytes(b"\0" * (3 * MiB))
    res = run_cli("--dryrun", "-r", "-t", "3", "-b", "1M", "--gpuids", "0", str(path))
    assert res.returncode == 0, res.stderr
    assert "* Bytes total:        %d |" % (3 * MiB) in res.stdout


def test_new_run_control_options_parse():
    res = run_cli("--dryrun", "-w", "-r", "-s", "1M", "--gpuids", "0", "--infloop", "--timelimit",
                  "1", "--limitread", "10M", "--limitwrite", "1G", "--live1", "--live1n",
                  "--cuhostbufreg", "--nodiocheck", "--nopathexp", "--datasetthreads", "4",
                  "--rankoffset", "1", "--start", "0", "--livecsv", "/tmp/elb_live.csv",
                  "--cores", "0-1,3", "--zones", "0", "--flock", "range", "--fadv",
                  "seq,willneed", "--statinline",
                  "/tmp/elb_dry")
    assert res.returncode == 0, res.stderr


def test_config3_random_read_iops_via_dryrun():
    # C3: 64 GiB / 4 KiB random reads -> randamount defaults to the file size (ProgArgs.cpp:1558)
    res = run_cli("--dryrun", "-r", "-b", "4K", "-s", "64G", "--rand", "--iodepth", "64",
                  "--gpuids", "0", "--gds", "/tmp/elb_dry")
    assert "* Bytes total:        %d |" % (64 * GiB) in res.stdout


@pytest.mark.parametrize("args,message", [
    (["-w", "-s", "1g", "/tmp/x"], '"--gpuids" is mandatory'),
    (["-w", "-s", "1g", "--gpuids", "0", "--rand", "--verify", "1", "/tmp/x"],
     "Integrity check writes are not supported in combination with random offsets."),
    (["-w", "-s", "1g", "--gpuids", "0", "--verify", "1", "--rwmixpct", "10", "/tmp/x"],
     'Option --rwmixpct cannot be used together with option "--verify"'),
    (["-w", "-s", "1g", "--gpuids", "0", "--rwmixpct", "10", "--rwmixthr", "1", "/tmp/x"],
     'Option "--rwmixpct" cannot be used together with "--rwmixthr"'),
    (["-r", "-s", "1g", "--gpuids", "0", "--verify", "1", "--verifydirect", "/tmp/x"],
     "Direct verification requires --verify and --write"),
    (["-w", "-s", "1g", "--gpuids", "0", "--readinline", "--iodepth", "4", "/tmp/x"],
     "Inline read cannot be used together with --iodepth"),
    (["-w", "-s", "1.5g", "--gpuids", "0", "/tmp/x"], "containing '.' character"),
    (["-w", "-s", "1g", "--gpuids", "0", "--nosuchoption", "/tmp/x"], "unrecognised option"),
    (["-s", "1g", "--gpuids", "0", "/tmp/x"], "No benchmark phase selected"),
    (["-w", "-d", "-s", "1g", "--gpuids", "0", "/tmp/elb_not_a_dir.bin"],
     "only allowed if benchmark path is a directory"),
    (["-w", "-s", "1g", "--gpuids", "0"], "Benchmark path missing."),
    (["-w", "-s", "1g", "-t", "2", "--gpuids", "0", "--rwmixthr", "1", "--rwmixthrpct", "40",
      "--limitwrite", "1M", "/tmp/x"],
     'Option "--rwmixthrpct" cannot be used together with "--limitread" or "--limitwrite"'),
    (["-r", "-s", "1g", "--gpuids", "0", "--flock", "maybe", "/tmp/x"],
     "Invalid file lock type: maybe"),
    (["-r", "-s", "1g", "--gpuids", "0", "--fadv", "seq,fast", "/tmp/x"], "Invalid fadvise: fast"),
    (["-r", "-s", "1g", "--gpuids", "0", "--rand", "--randalgo", "quick", "/tmp/x"],
     "Invalid random algo: quick"),
    (["-w", "-s", "1g", "--gpuids", "0", "--blockvarpct", "50", "--blockvaralgo", "best",
      "/tmp/x"], "Invalid random algo: best"),
])
def test_validation_messages(args, message):
    res = run_cli(*args)
    assert res.returncode == 1
    assert message in res.stderr, res.stderr


def make_results():
    res = PhaseResults()
    res.firstFinishUSec = 512345
    res.lastFinishUSec = 61 * 1000000 + 7000
    res.opsTotal.numBytesDone = 64 * GiB
    res.opsTotal.numIOPSDone = 65536
    res.opsStoneWallTotal.numBytesDone = 32 * GiB
    res.opsStoneWallTotal.numIOPSDone = 32768
    res.opsPerSec.numBytesDone = 1100 << 20
    res.opsPerSec.numIOPSDone = 1100
    res.opsStoneWallPerSec.numBytesDone = (2000 << 20) + 5
    res.opsStoneWallPerSec.numIOPSDone = 2000
    res.iopsLatHisto.numStoredValues = 3
    res.iopsLatHisto.numMicroSecTotal = 300 + 1500 + 25000
    res.iopsLatHisto.minMicroSecLat = 300
    res.iopsLatHisto.maxMicroSecLat = 25000
    res.iopsLatHisto.buckets[32] = 1   # 300 us
    res.iopsLatHisto.buckets[42] = 1   # 1500 us
    res.iopsLatHisto.buckets[58] = 1   # 25000 us
    res.entriesLatHisto.minMicroSecLat = (1 << 64) - 1
    res.iopsLatHistoReadMix.minMicroSecLat = (1 << 64) - 1
    res.entriesLatHistoReadMix.minMicroSecLat = (1 << 64) - 1
    res.cpuUtilStoneWallPercent = 7
    res.cpuUtilPercent = 9
    return res


def format_results(argv, phase, res, fmt):
    lib = _native.load()
    args = (ctypes.c_char_p * len(argv))(*[a.encode() for a in argv])
    buf = ctypes.create_string_buffer(1 << 16)
    n = lib.elb_format_phase_results(len(argv), args, phase, ctypes.byref(res), fmt, buf, 1 << 16)
    assert n >= 0, _native.last_error()
    return buf.value.decode()


ARGV = ["elbencho-b200", "-w", "-t", "4", "-b", "1M", "-s", "16G", "--gpuids", "0", "--lat",
        "--latpercent", "--lathisto", "--cpu", "--label", "my,label", "/tmp/elb_fmt.bin"]


def row(operation, result_type, colon, first, last):
    """boost::format("%|-11| %|-17|%|1| %|11| %|11|") of Statistics.h:138, written independently"""
    return "%-11s %-17s%-1s %11s %11s" % (operation, result_type, colon, first, last)


def row_left(operation, result_type, colon):
    """boost::format("%|-11| %|-17|%|1| ") of Statistics.h:139"""
    return "%-11s %-17s%-1s " % (operation, result_type, colon)


def test_console_table_format():
    """row layout and row order of Statistics::printPhaseResultsToStream (:1771-2140)"""
    text = format_results(ARGV, 4, make_results(), 0)
    lines = text.splitlines()
    assert lines[0] == row("OPERATION", "RESULT TYPE", "", "FIRST DONE", "LAST DONE")
    assert lines[1] == row("===========", "================", "", "==========", "=========")
    assert lines[2] == row("WRITE", "Elapsed time", ":", "512ms", "1m1.007s")
    assert lines[3] == row("", "IOPS", ":", 2000, 1100)
    assert lines[4] == row("", "Throughput MiB/s", ":", 2000, 1100)
    assert lines[5] == row("", "Total MiB", ":", 32768, 65536)
    assert lines[6] == row("", "CPU util %", ":", 7, 9)
    assert lines[7] == row_left("", "IO latency", ":") + "[ min=300us avg=8.93ms max=25.0ms ]"
    # percentile = upper bound of the bucket: 2^((idx+1)/4) (LatencyHistogram.h:140-159)
    assert lines[8] == row_left("", "IO lat % us", ":") + \
        "[ 1%<=304 50%<=1722 75%<=27554 99%<=27554 ]"
    assert lines[9] == row_left("", "IO lat hist", ":") + "[ 304: 1, 1722: 1, 27554: 1 ]"
    assert lines[10] == "---"
    assert lines[2] == "WRITE       Elapsed time     :       512ms    1m1.007s"


def test_console_table_rwmix_rows():
    res = make_results()
    res.opsReadMixTotal.numBytesDone = 8 * GiB
    res.opsReadMixTotal.numIOPSDone = 8192
    res.opsReadMixPerSec.numBytesDone = 100 << 20
    res.opsReadMixPerSec.numIOPSDone = 100
    res.opsStoneWallReadMixPerSec.numBytesDone = 200 << 20
    res.opsStoneWallReadMixPerSec.numIOPSDone = 200
    res.opsStoneWallReadMixTotal.numBytesDone = 4 * GiB
    argv = ["elbencho-b200", "-w", "-s", "16G", "--gpuids", "0", "--rwmixpct", "30", "--cufile",
            "/tmp/elb_fmt.bin"]
    lines = format_results(argv, 4, res, 0).splitlines()
    assert lines[2] == row("RWMIX30", "Elapsed time", ":", "512ms", "1m1.007s")
    assert lines[3] == row("", "IOPS write", ":", 2000, 1100)
    assert lines[4] == row("", "IOPS read", ":", 200, 100)
    assert lines[5] == row("", "IOPS total", ":", 2200, 1200)
    assert lines[6] == row("", "MiB/s write", ":", 2000, 1100)
    assert lines[7] == row("", "MiB/s read", ":", 200, 100)
    assert lines[8] == row("", "MiB/s total", ":", 2200, 1200)
    assert lines[9] == row("", "MiB write", ":", 32768, 65536)
    assert lines[10] == row("", "MiB read", ":", 4096, 8192)


def test_csv_columns_match_reference_docs():
    text = format_results(ARGV, 4, make_results(), 1)
    labels, values = [line.split(",") for line in text.splitlines()]
    # docs/csv-docs.md:9-43 + Statistics.cpp:2151-2323 (order matters for existing tooling)
    assert labels[:17] == ["ISO date", "label", "path type", "paths", "hosts", "threads", "dirs",
                           "files", "file size", "block size", "direct IO", "random",
                           "random aligned", "IO depth", "shared paths", "truncate", "operation"]
    assert labels[17:33] == ["time ms [first]", "time ms [last]", "entries/s [first]",
                             "entries/s [last]", "IOPS [first]", "IOPS [last]", "MiB/s [first]",
                             "MiB/s [last]", "CPU% [first]", "CPU% [last]", "entries [first]",
                             "entries [last]", "MiB [first]", "MiB [last]", "Ent lat us [min]",
                             "Ent lat us [avg]"]
    assert labels[-2:] == ["version", "command"] and len(labels) == len(values) == 55
    row = dict(zip(labels, values))
    assert row["label"] == "my label" and row["operation"] == "WRITE"
    assert row["threads"] == "4" and row["file size"] == str(16 * GiB)
    assert row["block size"] == "1048576" and row["dirs"] == "" and row["random aligned"] == ""
    assert row["time ms [first]"] == "512" and row["time ms [last]"] == "61007"
    assert row["IOPS [last]"] == "1100" and row["MiB/s [first]"] == "2000"
    assert row["entries/s [first]"] == "" and row["MiB [last]"] == "65536"
    assert row["IO lat us [min]"] == "300" and row["IO lat us [avg]"] == "8933"
    assert row["Ent lat us [min]"] == "" and row["rwmix read IOPS [last]"] == ""


def test_json_results_format():
    doc = json.loads(format_results(ARGV, 6, make_results(), 2))
    assert doc["phase_type"] == "READ" and doc["label"] == "my,label"
    # boost::property_tree writes every leaf as a string
    assert doc["config"]["threads"] == "4" and doc["config"]["file_size"] == str(16 * GiB)
    assert doc["config"]["direct_io"] == "false" and doc["config"]["path_type"] == "file"
    assert doc["first_done"] == {"elapsed_time_ms": "512", "iops": "2000",
                                 "bytes/s": str((2000 << 20) + 5), "bytes": str(32 * GiB),
                                 "cpu%": "7"}
    assert doc["last_done"]["latency"]["IO"] == {"min_us": "300", "avg_us": "8933",
                                                 "max_us": "25000"}
    assert "entries" not in doc["last_done"]["latency"]


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_service_http_endpoints_without_gpu():
    """service mode plumbing that needs no GPU: /protocolversion, /info, /status (idle), a failing
    /preparephase with the error text, unknown paths, and --quit from a master"""
    port = free_port()
    proc = subprocess.Popen([CLI_PATH, "--service", "--foreground", "--port", str(port)],
                            stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    try:
        for _ in range(100):
            try:
                conn = http.client.HTTPConnection("127.0.0.1", port, timeout=5)
                conn.request("GET", "/protocolversion")
                resp = conn.getresponse()
                break
            except OSError:
                time.sleep(0.1)
        assert resp.status == 200 and resp.read() == b"3.1.1"

        def call(method, path, body=None):
            conn.request(method, path, body=body)  # same connection: keep-alive
            response = conn.getresponse()
            return response.status, response.read()

        status, body = call("GET", "/info")
        assert status == 200 and b"elbencho-b200" in body
        status, body = call("GET", "/status")
        tree = json.loads(body)
        assert status == 200 and tree["PhaseName"] == "IDLE" and tree["NumWorkersDone"] == "0"
        assert tree["NumBytesDone"] == "0" and "ErrorHistory" in tree
        assert call("GET", "/nosuchpath")[0] == 404
        status, body = call("POST", "/preparephase?ProtocolVersion=1.0.0&PwHash=", "{}")
        assert status == 400 and b"Protocol version mismatch" in body
        prep = json.dumps({"path": "/tmp/elb_svc_test.bin", "block": "4096", "size": "8192",
                           "threads": "1", "write": "true", "gpuids": ""})
        status, body = call("POST", "/preparephase?ProtocolVersion=3.1.1&PwHash=", prep)
        assert status == 400 and b"--gpuids" in body
        # tree file upload for custom tree mode (HTTPServiceSWS.cpp:262-350)
        tree_text = "d up\nf 1000 up/a.bin\n"
        status, body = call("POST", "/preparefile?ProtocolVersion=3.1.1&PwHash=&FileName="
                            "..%2F..%2Ftreefile.txt", tree_text)
        assert status == 200 and body == b""
        import getpass
        upload_path = "/var/tmp/elbencho-b200_%s_p%d/treefile.txt" % (getpass.getuser(), port)
        with open(upload_path) as f:
            assert f.read() == tree_text  # (stored under its base name only)
        os.unlink(upload_path)
        os.rmdir(os.path.dirname(upload_path))
        status, body = call("POST", "/preparefile?ProtocolVersion=3.1.1&PwHash=", "x")
        assert status == 400 and b"Missing parameter: FileName" in body
        conn.close()
        res = run_cli("--hosts", "127.0.0.1:%d" % port, "--quit")
        assert res.returncode == 0, res.stderr
        proc.wait(timeout=20)
        assert proc.returncode == 0
        assert "Shutting down as requested by client" in proc.stdout.read()
    finally:
        if proc.poll() is None:
            proc.kill()


def test_options_md_is_in_sync_with_the_cli_table():
    """OPTIONS.md (coverage of the reference's ProgArgs) is generated"""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                    "scripts"))
    import gen_options_md
    with open(os.path.join(gen_options_md.REPO, "OPTIONS.md")) as f:
        assert f.read() == gen_options_md.generate()
