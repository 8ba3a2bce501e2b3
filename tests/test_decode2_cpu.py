"""CPU tests of the second-generation decoder (lizard_b200/csrc/decode2.cuh: parser -> records -> destination-first
copier with an output tile) through the TEST-ONLY host build: one lane and the 32-lane warp emulator, batches handed to
the copier through the in-line sink.  The checker is the unmodified reference (tests/refs.py): same return codes on valid
and damaged streams, same bytes whenever the reference's own output is well defined, nothing written outside
[dst, dst + result).  The device-only plumbing (mbarrier pipeline, TMA ring) is covered by the -m gpu tests."""
import ctypes
import os
import random

import pytest

import lizard_b200 as lz
from tests import refs
from tests.test_oracle import _inputs, stored_optimal_parser_cases

BS = lz.BLOCK_SIZE


@pytest.fixture(scope="module")
def shim():
    p = os.path.join(refs.ROOT, "lizard_b200", "libhostshim.so")
    if not os.path.exists(p):
        pytest.skip("libhostshim.so not built")
    L = ctypes.CDLL(p)
    L.lzb_host_decompress2.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_uint]
    return L


@pytest.fixture(scope="module")
def ref():
    return refs.reference()


def dec2(shim, comp, cap, mode, span, mis=0):
    """Decode into a buffer whose start is `mis` bytes off a 16-byte boundary, guarded on both sides."""
    guard = 64
    raw = ctypes.create_string_buffer(bytes([0xEE]) * (cap + 2 * guard + 32), cap + 2 * guard + 32)
    base = ctypes.addressof(raw) + guard
    base += (-base) % 16 + mis
    r = shim.lzb_host_decompress2(comp, len(comp), ctypes.c_void_p(base), cap, mode, span)
    before = ctypes.string_at(base - guard // 2, guard // 2)
    n = max(r, 0)
    after = ctypes.string_at(base + n, 16)
    return r, ctypes.string_at(base, n), before == bytes([0xEE]) * (guard // 2), after


@pytest.mark.parametrize("mode,span,count", [(0, 4032, 60), (0, 64, 30), (0, 700, 30), (1, 4032, 10), (1, 300, 8)])
def test_decode2_matches_reference_valid_and_damaged(ref, shim, mode, span, count):
    rnd = random.Random(77 + span + mode)
    compared = 0
    for data in _inputs(31 + span, count):
        level = rnd.choice([10, 21, 41, 30, 17, 22, 42])
        comp = ref.compress(data, level)
        cases = [(comp, len(data)), (comp, max(len(data) - 1, 0)), (comp, len(data) + 77)]
        for _ in range(5):
            bad = bytearray(comp)
            if not bad:
                break
            k = rnd.randrange(3)
            if k == 0:
                bad[rnd.randrange(len(bad))] ^= 1 << rnd.randrange(8)
            elif k == 1:
                bad = bad[: rnd.randrange(0, len(bad) + 1)]
            else:
                bad[rnd.randrange(min(40, len(bad)))] = rnd.randrange(256)
            cases.append((bytes(bad), rnd.choice([len(data), max(len(data) - 1, 0), len(data) + 100])))
        for c, cap in cases:
            rr, ro = ref.decompress(c, cap)
            r, o, clean_before, after = dec2(shim, c, cap, mode, span, rnd.randrange(16))
            assert r == rr, (mode, span, level, len(data), len(c), cap)
            assert clean_before, "wrote in front of the destination"
            if rr > 0 and refs.stream_obeys_min_offset(c, cap):
                compared += 1
                assert o == ro, (mode, span, level, len(data), cap)
                assert after == bytes([0xEE]) * 16, "wrote past the decoded size"
    assert compared > 0


@pytest.mark.parametrize("level", [10, 21, 41])
@pytest.mark.parametrize("mode", [0, 1])
def test_decode2_full_blocks_every_alignment_class(ref, shim, level, mode):
    """Whole 128 KiB datagen blocks, a unit of two inner blocks and repetitive input (self-overlapping and near matches:
    the copier's late-match path) at odd destination alignments and several batch spans."""
    data = lz.datagen(3 * BS)
    rep = b"abcdefghij" * 3000 + bytes(range(256)) * 40 + b"\0" * 5000 + b"xyzw" * 4000 + data[:3000] + b"q" * 70000
    cases = [data[:BS], data[BS:2 * BS + 4321], rep, bytes(BS), data[:20], data[:21], b""]
    for i, c in enumerate(cases):
        comp = ref.compress(c, level)
        for span in ((4032, 96) if mode == 0 else (4032, 900)):
            # the emulator runs the lanes between two collectives forward, reversed or shuffled: a missing barrier between a
            # write by one lane and a read by another only fails under some orders
            shim.lzb_emu_lane_order((i + span) % 3 if mode else 0)
            mis = (5 * i + level + span) % 16
            r, o, clean_before, after = dec2(shim, comp, len(c), mode, span, mis)
            assert r == len(c) and o == c, (level, mode, i, span, r)
            assert clean_before and after == bytes([0xEE]) * 16
    shim.lzb_emu_lane_order(0)


def test_decode2_long_literal_runs_are_split(ref, shim):
    """A block whose tokens carry literal runs far longer than one batch span (incompressible stretches between
    repeats): the parser hands them on through its one-token path and the literal-only records of the last literals."""
    rnd = random.Random(5)
    noise = bytes(rnd.randrange(256) for _ in range(40000))
    data = noise[:30000] + b"0123456789abcdef" * 64 + noise[30000:] + b"0123456789abcdef" * 64 + noise[:9000]
    for level in (10, 21):
        comp = ref.compress(data, level)
        for mode, span in ((0, 4032), (0, 128), (1, 4032)):
            r, o, ok, after = dec2(shim, comp, len(data), mode, span, 3)
            assert r == len(data) and o == data and ok and after == bytes([0xEE]) * 16, (level, mode, span, r)


def test_decode2_stored_optimal_parser_streams(ref, shim):
    """Streams of the reference's lowest-price and optimal parsers (levels 24 and 45), valid and damaged, through both
    copier modes: same codes and bytes as the reference, nothing written outside the destination."""
    compared = 0
    for i, (level, data, comp, cap, intact) in enumerate(stored_optimal_parser_cases()):
        rr, ro = ref.decompress(comp, cap)
        for mode, span in ((0, 4032), (0, 96), (1, 4032)):
            r, o, clean_before, after = dec2(shim, comp, cap, mode, span, (i + span) % 16)
            assert r == rr, (level, len(data), len(comp), cap, mode, span, r, rr)
            assert clean_before, "wrote in front of the destination"
            if intact:
                assert o == data
            if rr > 0 and refs.stream_obeys_min_offset(comp, cap):
                compared += 1
                assert o == ro and after == bytes([0xEE]) * 16, (level, len(data), cap, mode, span)
    assert compared > 0
