"""GPU parity tests of the sm_100a kernels against the CPU oracle, through the C ABI.

Bit-exact bar (integer/byte work): K1 fill_pattern and K3 fill_random produce the oracle's bytes,
K2 verify_pattern produces the oracle's mismatch count / first index. Sizes here are what the
oracle finishes in seconds; full-size checks use size-independent properties."""
import ctypes
import random

import pytest
import torch

from elbencho_b200 import kernels
from tests import oracle_lib
from tests.golden.make_golden import pattern_closed_form

pytestmark = pytest.mark.gpu


def dev_bytes(n, device, fill=0xA5):
    return torch.full((max(1, n),), fill, dtype=torch.uint8, device=device)


def stream_handle():
    return torch.cuda.current_stream().cuda_stream


def read_result(res_tensor):
    vals = res_tensor.cpu().tolist()
    return [(vals[i] & 0xFFFFFFFFFFFFFFFF, vals[i + 1] & 0xFFFFFFFFFFFFFFFF)
            for i in range(0, len(vals), 2)]


def to_bytes(t, n=None):
    data = t.cpu().numpy().tobytes()
    return data if n is None else data[:n]


EDGE_LENS = [1, 2, 7, 8, 9, 31, 32, 33, 63, 64, 65, 255, 4096, 4097, 32768, 32769, 65536 + 17,
             (1 << 20), (1 << 20) + 5]


@pytest.mark.parametrize("misalign", [0, 1, 8, 13, 16, 31])
def test_fill_pattern_matches_oracle_edge_grid(cuda_device, misalign):
    rng = random.Random(misalign)
    for length in EDGE_LENS:
        file_offset = rng.choice([0, 1, 3, 8, 4096, (1 << 33) + 5, rng.getrandbits(50)])
        salt = rng.choice([1, 0xFFFFFFFFFFFFFFFF, rng.getrandbits(64)])
        buf = dev_bytes(length + 64 + misalign, cuda_device)
        kernels.fill_pattern(buf.data_ptr() + misalign, length, file_offset, salt, stream_handle())
        torch.cuda.synchronize()
        host = to_bytes(buf)
        assert host[misalign:misalign + length] == oracle_lib.fill_pattern(length, file_offset, salt)
        # nothing outside the block was touched
        assert host[:misalign] == b"\xa5" * misalign
        assert host[misalign + length:] == b"\xa5" * (len(host) - misalign - length)


def test_fill_pattern_golden_vectors(cuda_device):
    import json
    import os
    with open(os.path.join(os.path.dirname(__file__), "golden", "ref_vectors.json")) as f:
        golden = json.load(f)
    for vec in golden["pattern_closed_form"]:
        buf = dev_bytes(vec["len"] + 32, cuda_device)
        kernels.fill_pattern(buf.data_ptr(), vec["len"], vec["fileOffset"], vec["salt"],
                             stream_handle())
        torch.cuda.synchronize()
        assert to_bytes(buf, vec["len"]).hex() == vec["hex"]


def test_fill_pattern_salt_wraparound(cuda_device):
    length, off, salt = 4096, 0xFFFFFFFFFFFFF000, 0xFFF0
    buf = dev_bytes(length, cuda_device)
    kernels.fill_pattern(buf.data_ptr(), length, off, salt, stream_handle())
    torch.cuda.synchronize()
    assert to_bytes(buf, length) == pattern_closed_form(length, off, salt)


def test_fill_zero_length_is_noop(cuda_device):
    buf = dev_bytes(64, cuda_device)
    kernels.fill_pattern(buf.data_ptr(), 0, 0, 1, stream_handle())
    kernels.fill_random(buf.data_ptr(), 0, 50, 1, 1, stream_handle())
    torch.cuda.synchronize()
    assert to_bytes(buf) == b"\xa5" * 64


@pytest.mark.parametrize("misalign", [0, 5, 16])
def test_verify_pattern_clean_and_corrupt(cuda_device, misalign):
    rng = random.Random(100 + misalign)
    res = torch.zeros(2, dtype=torch.int64, device=cuda_device)
    for length in EDGE_LENS:
        file_offset = rng.choice([0, 7, 4096, rng.getrandbits(45)])
        salt = rng.getrandbits(64) | 1
        good = oracle_lib.fill_pattern(length, file_offset, salt)
        data = bytearray(good)
        # clean
        buf = torch.frombuffer(bytearray(b"\0" * misalign + bytes(data)), dtype=torch.uint8).to(
            cuda_device)
        kernels.verify_pattern(buf.data_ptr() + misalign, length, file_offset, salt,
                               res.data_ptr(), stream_handle())
        torch.cuda.synchronize()
        assert read_result(res) == [(0, 0xFFFFFFFFFFFFFFFF)], length
        # corrupt a few bytes (including first/last positions)
        bad_positions = sorted({0, length - 1, rng.randrange(length), rng.randrange(length)})
        keep = rng.sample(bad_positions, rng.randrange(1, len(bad_positions) + 1))
        for pos in keep:
            data[pos] ^= rng.randrange(1, 256)
        buf = torch.frombuffer(bytearray(b"\0" * misalign + bytes(data)), dtype=torch.uint8).to(
            cuda_device)
        kernels.verify_pattern(buf.data_ptr() + misalign, length, file_offset, salt,
                               res.data_ptr(), stream_handle())
        torch.cuda.synchronize()
        rc, num, first, _, _, _ = oracle_lib.verify_pattern(data, file_offset, salt)
        assert rc == 1
        assert read_result(res) == [(num, first)], (length, keep)


def test_verify_wrong_salt_counts_all_differences(cuda_device):
    length = (1 << 20) + 3
    buf = dev_bytes(length, cuda_device)
    res = torch.zeros(2, dtype=torch.int64, device=cuda_device)
    kernels.fill_pattern(buf.data_ptr(), length, 0, 1, stream_handle())
    kernels.verify_pattern(buf.data_ptr(), length, 0, 0x0101010101010102, res.data_ptr(),
                           stream_handle())
    torch.cuda.synchronize()
    _, num, first, _, _, _ = oracle_lib.verify_pattern(to_bytes(buf, length), 0,
                                                       0x0101010101010102)
    assert read_result(res) == [(num, first)]
    assert first == 0 and num == length  # every byte differs for this salt pair


def test_verify_empty_buffer(cuda_device):
    res = torch.full((2,), 5, dtype=torch.int64, device=cuda_device)
    kernels.verify_pattern(0, 0, 0, 1, res.data_ptr(), stream_handle())
    torch.cuda.synchronize()
    assert read_result(res) == [(0, 0xFFFFFFFFFFFFFFFF)]


@pytest.mark.parametrize("pct", [0, 1, 33, 50, 99, 100])
def test_fill_random_matches_cpu_twin(cuda_device, pct):
    rng = random.Random(pct)
    for length in EDGE_LENS:
        for misalign in (0, 8, 3):
            seed = rng.getrandbits(64)
            ctr = rng.getrandbits(48)
            buf = dev_bytes(length + 64, cuda_device)
            kernels.fill_random(buf.data_ptr() + misalign, length, pct, seed, ctr, stream_handle())
            torch.cuda.synchronize()
            host = to_bytes(buf)
            assert host[misalign:misalign + length] == \
                oracle_lib.fill_random_ctr(length, pct, seed, ctr), (length, misalign)
            assert host[misalign + length:] == b"\xa5" * (len(host) - misalign - length)


def test_fill_random_rejects_bad_args(cuda_device):
    buf = dev_bytes(64, cuda_device)
    with pytest.raises(kernels.KernelError):
        kernels.fill_random(buf.data_ptr(), 64, 101, 1, 1, stream_handle())
    with pytest.raises(kernels.KernelError):
        kernels.fill_random(buf.data_ptr(), 64, 50, 1, 1, stream_handle(), algo=99)


def make_batch(cuda_device, blocks):
    """blocks: list of (ptr, len, off, ctr) -> device descriptor tensor"""
    raw = kernels.pack_block_descs(blocks)
    return torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(cuda_device)


@pytest.mark.parametrize("max_block_len", [0, 1 << 20, 1 << 26])
def test_batched_window_ragged_blocks(cuda_device, max_block_len):
    """one launch over a ragged window: different lengths, offsets, alignments, empty blocks.
    max_block_len 0: persistent grid with static tile partition; 1 MiB: hardware-scheduled tiles
    (CTAs past the end of shorter blocks exit); 64 MiB: bound so loose that the launcher falls
    back to the persistent grid"""
    rng = random.Random(77)
    lens = [1 << 20, 4096, 0, 65536 + 3, 1, (1 << 20) - 32, 777, 32768 * 3, 5, 1 << 16]
    arena = dev_bytes(sum(lens) + 64 * len(lens), cuda_device)
    blocks = []
    pos = 0
    for i, length in enumerate(lens):
        pos += rng.choice([0, 1, 8, 31])
        blocks.append((arena.data_ptr() + pos, length, rng.getrandbits(44), rng.getrandbits(40)))
        pos += length + 16
    descs = make_batch(cuda_device, blocks)
    counters = torch.zeros(kernels.DEVCTR_NUM, dtype=torch.int64, device=cuda_device)
    results = torch.zeros(2 * len(blocks), dtype=torch.int64, device=cuda_device)
    salt = 0xABCDEF0123456789

    kernels.fill_pattern_batch(descs.data_ptr(), len(blocks), salt, counters.data_ptr(),
                               stream_handle(), total_bytes=sum(lens), max_block_len=max_block_len)
    torch.cuda.synchronize()
    host = to_bytes(arena)
    base = arena.data_ptr()
    for ptr, length, off, _ in blocks:
        assert host[ptr - base:ptr - base + length] == oracle_lib.fill_pattern(length, off, salt)
    assert counters.cpu().tolist()[kernels.DEVCTR_FILLED_BYTES] == sum(lens)

    # verify: clean
    kernels.verify_pattern_batch(descs.data_ptr(), len(blocks), salt, results.data_ptr(),
                                 counters.data_ptr(), stream_handle(), total_bytes=sum(lens),
                                 max_block_len=max_block_len)
    torch.cuda.synchronize()
    assert read_result(results) == [(0, 0xFFFFFFFFFFFFFFFF)] * len(blocks)
    ctr = counters.cpu().tolist()
    assert ctr[kernels.DEVCTR_VERIFIED_BYTES] == sum(lens)
    assert ctr[kernels.DEVCTR_VERIFY_MISMATCH_BYTES] == 0

    # corrupt blocks 3 and 7, verify again: per-block results + device counter
    corrupt = {3: [0, 65536 + 2, 40000], 7: [32768 * 3 - 1]}
    for idx, positions in corrupt.items():
        ptr = blocks[idx][0]
        for p in positions:
            arena[ptr - base + p] ^= 0x5A
    kernels.verify_pattern_batch(descs.data_ptr(), len(blocks), salt, results.data_ptr(),
                                 counters.data_ptr(), stream_handle(), total_bytes=sum(lens),
                                 max_block_len=max_block_len)
    torch.cuda.synchronize()
    got = read_result(results)
    for idx in range(len(blocks)):
        if idx in corrupt:
            assert got[idx] == (len(corrupt[idx]), min(corrupt[idx]))
        else:
            assert got[idx] == (0, 0xFFFFFFFFFFFFFFFF)
    assert counters.cpu().tolist()[kernels.DEVCTR_VERIFY_MISMATCH_BYTES] == 4

    # random fill over the same ragged window
    kernels.fill_random_batch(descs.data_ptr(), len(blocks), 60, 999, 0, stream_handle(),
                              total_bytes=sum(lens), max_block_len=max_block_len)
    torch.cuda.synchronize()
    host = to_bytes(arena)
    for ptr, length, _, ctr_val in blocks:
        assert host[ptr - base:ptr - base + length] == \
            oracle_lib.fill_random_ctr(length, 60, 999, ctr_val)


def test_block_longer_than_size_hint_is_fully_processed(cuda_device):
    """max_block_len is a HINT for the launch shape: a descriptor that is longer than the hint
    must still be filled / verified completely (no silently skipped tail tiles)."""
    block, hint, salt = (1 << 20) + 4096 + 7, 64 << 10, 0x77
    nblocks = 6
    arena = dev_bytes(block * nblocks, cuda_device, fill=0)
    blocks = [(arena.data_ptr() + i * block, block, i * block, i) for i in range(nblocks)]
    descs = make_batch(cuda_device, blocks)
    results = torch.zeros(2 * nblocks, dtype=torch.int64, device=cuda_device)
    kernels.fill_pattern_batch(descs.data_ptr(), nblocks, salt, 0, stream_handle(),
                               total_bytes=hint * nblocks, max_block_len=hint)
    torch.cuda.synchronize()
    assert to_bytes(arena, block * nblocks) == oracle_lib.fill_pattern(block * nblocks, 0, salt)
    # a flipped byte in the part of each block that lies beyond the hint must be found
    for i in range(nblocks):
        arena[i * block + hint + 12345 + i] ^= 0x40
    kernels.verify_pattern_batch(descs.data_ptr(), nblocks, salt, results.data_ptr(), 0,
                                 stream_handle(), total_bytes=hint * nblocks, max_block_len=hint)
    torch.cuda.synchronize()
    assert read_result(results) == [(1, hint + 12345 + i) for i in range(nblocks)]
    kernels.fill_random_batch(descs.data_ptr(), nblocks, 100, 42, 0, stream_handle(),
                              total_bytes=hint * nblocks, max_block_len=hint)
    torch.cuda.synchronize()
    host = to_bytes(arena)
    for i in range(nblocks):
        assert host[i * block:(i + 1) * block] == oracle_lib.fill_random_ctr(block, 100, 42, i)


def test_large_window_round_trip_properties(cuda_device):
    """BASELINE-sized blocks (1 MiB x 1024 = 1 GiB window), checked through size-independent
    properties: fill -> verify is clean; one flipped byte anywhere is found at exactly that
    offset; write-block-size != read-block-size still verifies (tools/test-examples.sh:226,243)."""
    block = 1 << 20
    nblocks = 1024
    arena = torch.empty(block * nblocks, dtype=torch.uint8, device=cuda_device)
    salt = 1
    wblocks = [(arena.data_ptr() + i * block, block, i * block, i) for i in range(nblocks)]
    wdescs = make_batch(cuda_device, wblocks)
    kernels.fill_pattern_batch(wdescs.data_ptr(), nblocks, salt, 0, stream_handle(),
                               total_bytes=block * nblocks, max_block_len=block)
    # read back with 128 KiB blocks
    rblock = 128 << 10
    rn = block * nblocks // rblock
    rblocks = [(arena.data_ptr() + i * rblock, rblock, i * rblock, 0) for i in range(rn)]
    rdescs = make_batch(cuda_device, rblocks)
    results = torch.zeros(2 * rn, dtype=torch.int64, device=cuda_device)
    counters = torch.zeros(kernels.DEVCTR_NUM, dtype=torch.int64, device=cuda_device)
    kernels.verify_pattern_batch(rdescs.data_ptr(), rn, salt, results.data_ptr(),
                                 counters.data_ptr(), stream_handle(), total_bytes=block * nblocks,
                                 max_block_len=rblock)
    torch.cuda.synchronize()
    assert int(results.view(-1, 2)[:, 0].sum()) == 0
    assert counters.cpu().tolist()[kernels.DEVCTR_VERIFIED_BYTES] == block * nblocks
    # spot check the bytes against the oracle at a few places
    for i in (0, 1, 511, 1023):
        assert to_bytes(arena[i * block:i * block + 4096]) == \
            oracle_lib.fill_pattern(4096, i * block, salt)
    # flip single bytes
    rng = random.Random(3)
    flips = sorted(rng.sample(range(block * nblocks), 5))
    for pos in flips:
        arena[pos] ^= 0x80
    kernels.verify_pattern_batch(rdescs.data_ptr(), rn, salt, results.data_ptr(),
                                 counters.data_ptr(), stream_handle())
    torch.cuda.synchronize()
    res = results.view(-1, 2).cpu()
    bad = [(i, int(res[i, 0]), int(res[i, 1])) for i in range(rn) if int(res[i, 0])]
    expected = {}
    for pos in flips:
        blk = pos // rblock
        cnt, first = expected.get(blk, (0, 1 << 62))
        expected[blk] = (cnt + 1, min(first, pos % rblock))
    assert bad == [(blk, cnt, first) for blk, (cnt, first) in sorted(expected.items())]


def test_random_fill_large_window_checksum_of_blocks(cuda_device):
    """full-size blocks: identical (seed, counter) -> identical block; different counter ->
    different block; remainder is one repeated word"""
    block = 1 << 20
    arena = torch.empty(block * 4, dtype=torch.uint8, device=cuda_device)
    blocks = [(arena.data_ptr() + i * block, block, 0, ctr) for i, ctr in enumerate([5, 6, 5, 7])]
    descs = make_batch(cuda_device, blocks)
    kernels.fill_random_batch(descs.data_ptr(), 4, 75, 31337, 0, stream_handle())
    torch.cuda.synchronize()
    b = [arena[i * block:(i + 1) * block] for i in range(4)]
    assert torch.equal(b[0], b[2])
    assert not torch.equal(b[0], b[1])
    var_len = (block * 75 // 100) & ~3
    tail = b[0][var_len:].cpu().numpy().tobytes()
    assert tail == (tail[:8] * (len(tail) // 8 + 1))[:len(tail)]
    assert to_bytes(b[3]) == oracle_lib.fill_random_ctr(block, 75, 31337, 7)


def test_kernel_launch_counter(cuda_device):
    before = kernels.num_kernel_launches()
    buf = dev_bytes(4096, cuda_device)
    kernels.fill_pattern(buf.data_ptr(), 4096, 0, 1, stream_handle())
    torch.cuda.synchronize()
    assert kernels.num_kernel_launches() == before + 1


# ------------------------------------------------------------------------------------------------
# staged forms: the kernels move the block between a pinned host buffer and the device buffer
# ------------------------------------------------------------------------------------------------

def _staged_arena(cuda_device, nbytes):
    """device arena + pinned host arena of the same layout -> (dev, host, host_delta)"""
    dev = torch.full((nbytes,), 0xA5, dtype=torch.uint8, device=cuda_device)
    host = torch.full((nbytes,), 0x5A, dtype=torch.uint8).pin_memory()
    return dev, host, host.data_ptr() - dev.data_ptr()


def _pinned_descs(blocks):
    raw = kernels.pack_block_descs(blocks)
    return torch.frombuffer(bytearray(raw), dtype=torch.uint8).pin_memory()


@pytest.mark.parametrize("misalign", [0, 7, 16])
@pytest.mark.parametrize("hinted", [True, False])
def test_staged_fill_writes_both_rings(cuda_device, misalign, hinted):
    """fill + stage-out: device slot and host slot both hold the oracle's bytes, nothing else is
    touched; descriptors are read from pinned host memory (ragged lengths, both launch shapes)."""
    lens = [1 << 20, (1 << 20) - 13, 4096, 33, 0, 65536 + 5]
    stride = (1 << 20) + 4096
    dev, host, delta = _staged_arena(cuda_device, stride * len(lens) + 64)
    salt = 0xABCDEF0102
    blocks = [(dev.data_ptr() + i * stride + misalign, n, (i << 21) + 3 * i, i)
              for i, n in enumerate(lens)]
    descs = _pinned_descs(blocks)
    hints = dict(total_bytes=sum(lens), max_block_len=max(lens)) if hinted else {}
    kernels.fill_pattern_staged(descs.data_ptr(), len(blocks), salt, delta, 0, stream_handle(),
                                **hints)
    torch.cuda.synchronize()
    dev_bytes_, host_bytes = to_bytes(dev), host.numpy().tobytes()
    for i, (ptr, n, off, _) in enumerate(blocks):
        lo = ptr - dev.data_ptr()
        expected = oracle_lib.fill_pattern(n, off, salt) if n else b""
        assert dev_bytes_[lo:lo + n] == expected, i
        assert host_bytes[lo:lo + n] == expected, i
        gap_end = (i + 1) * stride + misalign if i + 1 < len(blocks) else len(dev_bytes_)
        assert dev_bytes_[lo + n:gap_end] == b"\xa5" * (gap_end - lo - n)
        assert host_bytes[lo + n:gap_end] == b"\x5a" * (gap_end - lo - n)
    # random fill through the same path
    kernels.fill_random_staged(descs.data_ptr(), len(blocks), 70, 4242, delta, 0, stream_handle(),
                               **hints)
    torch.cuda.synchronize()
    dev_bytes_, host_bytes = to_bytes(dev), host.numpy().tobytes()
    for ptr, n, _, ctr in blocks:
        lo = ptr - dev.data_ptr()
        expected = oracle_lib.fill_random_ctr(n, 70, 4242, ctr) if n else b""
        assert dev_bytes_[lo:lo + n] == expected and host_bytes[lo:lo + n] == expected


@pytest.mark.parametrize("misalign", [0, 5])
def test_staged_verify_reads_host_ring_and_publishes_results(cuda_device, misalign):
    """stage-in + verify: data comes from the pinned host slot, lands in the device slot, the
    last CTA publishes per-block results to pinned host memory and re-arms the device results."""
    lens = [1 << 20, 70000, 4096, 0, (1 << 20) + 31]
    stride = (1 << 20) + 4096
    dev, host, delta = _staged_arena(cuda_device, stride * len(lens) + 64)
    salt = 99
    blocks = [(dev.data_ptr() + i * stride + misalign, n, i * (1 << 24) + 8 * i, 0)
              for i, n in enumerate(lens)]
    descs = _pinned_descs(blocks)
    host_np = host.numpy()
    for ptr, n, off, _ in blocks:
        lo = ptr - dev.data_ptr()
        if n:
            host_np[lo:lo + n] = list(oracle_lib.fill_pattern(n, off, salt))
    bad = {0: [5, 70001, (1 << 20) - 1], 2: [4095], 4: [(1 << 20) + 30]}
    for idx, positions in bad.items():
        lo = blocks[idx][0] - dev.data_ptr()
        for pos in positions:
            host_np[lo + pos] ^= 0x11
    dev_results = torch.zeros(2 * len(blocks), dtype=torch.int64, device=cuda_device)
    host_results = torch.full((2 * len(blocks),), 7, dtype=torch.int64).pin_memory()
    ticket = torch.zeros(1, dtype=torch.int32, device=cuda_device)
    counters = torch.zeros(kernels.DEVCTR_NUM, dtype=torch.int64, device=cuda_device)
    kernels.verify_results_init(dev_results.data_ptr(), len(blocks), stream_handle())
    for rep in range(2):  # second launch: device results were re-armed by the first
        kernels.verify_pattern_staged(descs.data_ptr(), len(blocks), salt, delta,
                                      dev_results.data_ptr(), host_results.data_ptr(),
                                      ticket.data_ptr(), counters.data_ptr(), stream_handle(),
                                      total_bytes=sum(lens), max_block_len=max(lens))
        torch.cuda.synchronize()
        got = [(int(host_results[2 * i]) & (2 ** 64 - 1), int(host_results[2 * i + 1]) & (2 ** 64 - 1))
               for i in range(len(blocks))]
        for i in range(len(blocks)):
            exp = (len(bad[i]), min(bad[i])) if i in bad else (0, 2 ** 64 - 1)
            assert got[i] == exp, (rep, i)
        assert read_result(dev_results) == [(0, 2 ** 64 - 1)] * len(blocks)  # re-armed
        assert int(ticket.item()) == 0
    assert counters.cpu().tolist()[kernels.DEVCTR_VERIFY_MISMATCH_BYTES] == 2 * 5
    # the device slots now hold what was in the host slots
    dev_bytes_ = to_bytes(dev)
    for ptr, n, _, _ in blocks:
        lo = ptr - dev.data_ptr()
        assert dev_bytes_[lo:lo + n] == host_np[lo:lo + n].tobytes()


def test_verify_publishes_results_without_staging(cuda_device):
    """host_delta 0: verify on the device slot (copy-engine staging / cuFile), results still
    published by the last CTA"""
    n, salt = (1 << 20) + 17, 3
    dev = dev_bytes(n, cuda_device)
    kernels.fill_pattern(dev.data_ptr(), n, 4096, salt, stream_handle())
    dev[123456] ^= 1
    descs = _pinned_descs([(dev.data_ptr(), n, 4096, 0)])
    dev_results = torch.zeros(2, dtype=torch.int64, device=cuda_device)
    host_results = torch.zeros(2, dtype=torch.int64).pin_memory()
    ticket = torch.zeros(1, dtype=torch.int32, device=cuda_device)
    kernels.verify_results_init(dev_results.data_ptr(), 1, stream_handle())
    kernels.verify_pattern_staged(descs.data_ptr(), 1, salt, 0, dev_results.data_ptr(),
                                  host_results.data_ptr(), ticket.data_ptr(), 0, stream_handle(),
                                  total_bytes=n, max_block_len=n)
    torch.cuda.synchronize()
    assert host_results.tolist() == [1, 123456]


@pytest.mark.parametrize("to_device", [True, False])
def test_stage_copy_kernels(cuda_device, to_device):
    lens = [1 << 20, 12345, 0, 4096]
    stride = (1 << 20) + 4096
    dev, host, delta = _staged_arena(cuda_device, stride * len(lens))
    blocks = [(dev.data_ptr() + i * stride + 3, n, 0, 0) for i, n in enumerate(lens)]
    descs = _pinned_descs(blocks)
    rnd = torch.randint(0, 256, (stride * len(lens),), dtype=torch.uint8)
    if to_device:
        host.copy_(rnd)
    else:
        dev.copy_(rnd.to(cuda_device))
    kernels.stage_copy(descs.data_ptr(), len(blocks), to_device, delta, stream_handle(),
                       total_bytes=sum(lens), max_block_len=max(lens))
    torch.cuda.synchronize()
    dev_bytes_, host_bytes, src = to_bytes(dev), host.numpy().tobytes(), rnd.numpy().tobytes()
    for ptr, n, _, _ in blocks:
        lo = ptr - dev.data_ptr()
        assert dev_bytes_[lo:lo + n] == src[lo:lo + n]
        assert host_bytes[lo:lo + n] == src[lo:lo + n]
    dst_bytes, fill = (dev_bytes_, b"\xa5") if to_device else (host_bytes, b"\x5a")
    assert dst_bytes[:3] == fill * 3  # nothing outside the blocks was written


# ------------------------------------------------------------------------------------------------
# small blocks: warp-per-block kernels (block size hint <= 8 KiB)
# ------------------------------------------------------------------------------------------------

SMALL_LENS = [4096, 4096, 1, 31, 32, 33, 0, 1000, 4095, 4097, 8192, 8191, 4096, 20000, 64, 4096]


@pytest.mark.parametrize("misalign", [0, 3, 16])
def test_small_block_kernels_match_oracle(cuda_device, misalign):
    """hint <= 8 KiB -> one warp per block: ragged lengths, unaligned addresses and file offsets,
    a block longer than the hint, more blocks than one CTA takes; fill / verify / random fill"""
    hint = 4096
    stride = 24 * 1024
    nblocks = len(SMALL_LENS) * 3 + 1  # (not a multiple of the 8 blocks a CTA takes)
    lens = (SMALL_LENS * 4)[:nblocks]
    arena = dev_bytes(stride * nblocks + 64, cuda_device)
    base = arena.data_ptr()
    salt = 0x5151
    blocks = [(base + i * stride + (misalign if i % 2 else 0), n, 4096 * i + (5 if i % 3 == 0 else 0),
               100 + i) for i, n in enumerate(lens)]
    descs = make_batch(cuda_device, blocks)
    results = torch.zeros(2 * nblocks, dtype=torch.int64, device=cuda_device)
    counters = torch.zeros(kernels.DEVCTR_NUM, dtype=torch.int64, device=cuda_device)
    kernels.fill_pattern_batch(descs.data_ptr(), nblocks, salt, counters.data_ptr(),
                               stream_handle(), total_bytes=sum(lens), max_block_len=hint)
    torch.cuda.synchronize()
    host = to_bytes(arena)
    covered = bytearray(len(host))
    for ptr, n, off, _ in blocks:
        lo = ptr - base
        assert host[lo:lo + n] == (oracle_lib.fill_pattern(n, off, salt) if n else b""), (lo, n)
        covered[lo:lo + n] = b"\x01" * n
    assert all(host[i] == 0xA5 for i in range(len(host)) if not covered[i])
    assert counters.cpu().tolist()[kernels.DEVCTR_FILLED_BYTES] == sum(lens)

    # verify: clean, then corrupted
    kernels.verify_pattern_batch(descs.data_ptr(), nblocks, salt, results.data_ptr(),
                                 counters.data_ptr(), stream_handle(), total_bytes=sum(lens),
                                 max_block_len=hint)
    torch.cuda.synchronize()
    assert read_result(results) == [(0, 0xFFFFFFFFFFFFFFFF)] * nblocks
    assert counters.cpu().tolist()[kernels.DEVCTR_VERIFIED_BYTES] == sum(lens)
    bad = {}
    rng = random.Random(misalign)
    for idx in (0, 3, 9, 13, nblocks - 1):
        n = blocks[idx][1]
        if not n:
            continue
        positions = sorted({0, n - 1, rng.randrange(n)})
        bad[idx] = positions
        for pos in positions:
            arena[blocks[idx][0] - base + pos] ^= 0x3C
    kernels.verify_pattern_batch(descs.data_ptr(), nblocks, salt, results.data_ptr(), 0,
                                 stream_handle(), total_bytes=sum(lens), max_block_len=hint)
    torch.cuda.synchronize()
    got = read_result(results)
    for idx in range(nblocks):
        exp = (len(bad[idx]), bad[idx][0]) if idx in bad else (0, 0xFFFFFFFFFFFFFFFF)
        assert got[idx] == exp, idx

    kernels.fill_random_batch(descs.data_ptr(), nblocks, 50, 777, 0, stream_handle(),
                              total_bytes=sum(lens), max_block_len=hint)
    torch.cuda.synchronize()
    host = to_bytes(arena)
    for ptr, n, _, ctr in blocks:
        lo = ptr - base
        assert host[lo:lo + n] == (oracle_lib.fill_random_ctr(n, 50, 777, ctr) if n else b"")


def test_small_block_staged_kernels(cuda_device):
    """the staged forms of the warp-per-block kernels: fill + stage-out, stage-in + verify with
    published results, stage copies"""
    hint, stride = 4096, 8192
    lens = [4096] * 21 + [100, 0, 4095, 8192 - 64]
    nblocks = len(lens)
    dev, host, delta = _staged_arena(cuda_device, stride * nblocks + 64)
    salt = 12
    blocks = [(dev.data_ptr() + i * stride + (8 if i % 4 == 1 else 0), n, 1 << 30 | (i * 4096), i)
              for i, n in enumerate(lens)]
    descs = _pinned_descs(blocks)
    hints = dict(total_bytes=sum(lens), max_block_len=hint)
    kernels.fill_pattern_staged(descs.data_ptr(), nblocks, salt, delta, 0, stream_handle(), **hints)
    torch.cuda.synchronize()
    dev_b, host_b = to_bytes(dev), host.numpy().tobytes()
    for ptr, n, off, _ in blocks:
        lo = ptr - dev.data_ptr()
        expected = oracle_lib.fill_pattern(n, off, salt) if n else b""
        assert dev_b[lo:lo + n] == expected and host_b[lo:lo + n] == expected
    # corrupt the HOST copy of two blocks; stage-in + verify must see it and repair nothing
    host_np = host.numpy()
    host_np[blocks[2][0] - dev.data_ptr() + 77] ^= 1
    host_np[blocks[20][0] - dev.data_ptr() + 4095] ^= 0x80
    dev.fill_(0)
    dev_results = torch.zeros(2 * nblocks, dtype=torch.int64, device=cuda_device)
    host_results = torch.zeros(2 * nblocks, dtype=torch.int64).pin_memory()
    ticket = torch.zeros(1, dtype=torch.int32, device=cuda_device)
    kernels.verify_results_init(dev_results.data_ptr(), nblocks, stream_handle())
    kernels.verify_pattern_staged(descs.data_ptr(), nblocks, salt, delta, dev_results.data_ptr(),
                                  host_results.data_ptr(), ticket.data_ptr(), 0, stream_handle(),
                                  **hints)
    torch.cuda.synchronize()
    got = host_results.view(-1, 2).tolist()
    for i in range(nblocks):
        exp = [1, 77] if i == 2 else ([1, 4095] if i == 20 else [0, -1])
        assert got[i] == exp, i
    dev_b = to_bytes(dev)
    for ptr, n, _, _ in blocks:
        lo = ptr - dev.data_ptr()
        assert dev_b[lo:lo + n] == host_np[lo:lo + n].tobytes()
    # stage copy out of a changed device ring
    dev.copy_(torch.randint(0, 256, (dev.numel(),), dtype=torch.uint8).to(cuda_device))
    kernels.stage_copy(descs.data_ptr(), nblocks, False, delta, stream_handle(), **hints)
    torch.cuda.synchronize()
    dev_b, host_b = to_bytes(dev), host.numpy().tobytes()
    for ptr, n, _, _ in blocks:
        lo = ptr - dev.data_ptr()
        assert host_b[lo:lo + n] == dev_b[lo:lo + n]


# ------------------------------------------------------------------------------------------------
# 64-bit edges: one block longer than 2^32 bytes
# ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("shape", ["warp", "tiled", "persistent"])
def test_block_longer_than_4gib_counts_and_locates_in_64_bits(cuda_device, shape):
    """a single block of 4 GiB + 16 KiB + 5 through each launch shape (picked by the size hints;
    the warp kernel walks a block longer than its hint completely): a count of every byte must not
    wrap at 2^32, and a first mismatch beyond 2^32 takes the high word of the 64-bit minimum"""
    length = 2 ** 32 + 16 * 1024 + 5
    salt = 0x1122334455667788
    other_salt = (salt + 0x0101010101010101) % 2 ** 64  # differs from salt in every byte
    hints = {"warp": dict(total_bytes=length, max_block_len=4096),
             "tiled": dict(total_bytes=length, max_block_len=length),
             "persistent": {}}[shape]
    buf = torch.empty(length, dtype=torch.uint8, device=cuda_device)
    try:
        descs = make_batch(cuda_device, [(buf.data_ptr(), length, 0, 0)])
        results = torch.zeros(2, dtype=torch.int64, device=cuda_device)
        counters = torch.zeros(kernels.DEVCTR_NUM, dtype=torch.int64, device=cuda_device)
        kernels.fill_pattern_batch(descs.data_ptr(), 1, salt, 0, stream_handle(),
                                   total_bytes=length, max_block_len=length)
        kernels.verify_pattern_batch(descs.data_ptr(), 1, other_salt, results.data_ptr(),
                                     counters.data_ptr(), stream_handle(), **hints)
        torch.cuda.synchronize()
        assert read_result(results) == [(length, 0)]
        ctr = counters.cpu().tolist()
        assert ctr[kernels.DEVCTR_VERIFY_MISMATCH_BYTES] == length
        assert ctr[kernels.DEVCTR_VERIFIED_BYTES] == length

        bad = 2 ** 32 + 12345
        buf[bad] ^= 0x10
        kernels.verify_pattern_batch(descs.data_ptr(), 1, salt, results.data_ptr(), 0,
                                     stream_handle(), **hints)
        torch.cuda.synchronize()
        assert read_result(results) == [(1, bad)]
    finally:
        del buf
        torch.cuda.empty_cache()
