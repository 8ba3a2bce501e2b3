"""CPU tests that PIN the oracle (oracle/lizard_oracle.c, our plain-C restatement) and the host build of the
lane-generic codec code (lizard_b200/libhostshim.so, TEST-ONLY) against the unmodified reference: its recorded
answers (tests/refs.py) and the committed golden fixtures generated from its build."""
import ctypes
import hashlib
import json
import os
import random

import numpy as np
import pytest

import lizard_b200 as lz
from tests import refs

BS = lz.BLOCK_SIZE
LEVELS = [10, 11, 13, 16, 20, 21, 22, 30, 31, 34, 40, 41, 42]      # fastSmall, fast, hashChain (13-17/34-38), fastBig, priceFast
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _oracle():
    p = os.path.join(refs.ROOT, "oracle", "liboracle.so")
    if not os.path.exists(p):
        pytest.skip("oracle/liboracle.so not built (run __graft_entry__.build())")
    L = ctypes.CDLL(p)
    L.oracle_Lizard_compress.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    L.oracle_Lizard_decompress_safe.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_int]
    L.oracle_HUF_compress.restype = ctypes.c_size_t
    L.oracle_HUF_compress.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t]
    L.oracle_HUF_decompress.restype = ctypes.c_size_t
    L.oracle_HUF_decompress.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t]
    return L


def _shim():
    p = os.path.join(refs.ROOT, "lizard_b200", "libhostshim.so")
    if not os.path.exists(p):
        pytest.skip("libhostshim.so not built")
    L = ctypes.CDLL(p)
    L.lzb_host_compress.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_int, ctypes.c_int]
    L.lzb_host_huf_decompress.argtypes = [ctypes.c_char_p, ctypes.c_uint, ctypes.c_char_p, ctypes.c_uint]
    L.lzb_emu_compress.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_int, ctypes.c_int]
    for f in ("lzb_host_decompress", "lzb_emu_decompress"):
        getattr(L, f).argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_int]
    return L


@pytest.fixture(scope="module")
def oracle():
    return _oracle()


@pytest.fixture(scope="module")
def shim():
    return _shim()


@pytest.fixture(scope="module")
def ref():
    return refs.reference()


def o_compress(L, data, level, cap=None):
    cap = lz_bound(len(data)) if cap is None else cap
    dst = ctypes.create_string_buffer(max(cap, 1) + 64)
    n = L.oracle_Lizard_compress(data, dst, len(data), cap, level)
    return dst.raw[:n]


def shim_compress(L, data, level, cap=None):
    cap = lz_bound(len(data)) if cap is None else cap
    dst = ctypes.create_string_buffer(max(cap, 1) + 64)
    n = L.lzb_host_compress(data, len(data), dst, cap, level)
    return dst.raw[:n]


def emu_compress(L, data, level, cap=None):
    """The device code path (ballot / shuffle / match_any, 32 lanes) run on the coroutine warp emulator."""
    cap = lz_bound(len(data)) if cap is None else cap
    dst = ctypes.create_string_buffer(max(cap, 1) + 64)
    n = L.lzb_emu_compress(data, len(data), dst, cap, level)
    return dst.raw[:n]


def o_decompress(L, comp, cap):
    dst = ctypes.create_string_buffer(max(cap, 1) + 64)
    r = L.oracle_Lizard_decompress_safe(comp, dst, len(comp), cap)
    return r, (dst.raw[:r] if r > 0 else b"")


def lz_bound(n):
    return n + 2 + (n // BS + 1) * 4


def far_match_input(seed=3, n=BS):
    """Matches 65536 or more bytes back, short and long: exercises the LIZv1 parsers' rule that a far candidate is only taken
    when the match is at least MM_LONGOFF + MINMATCH long (lizard_parser_fastbig.h:99,142; lizard_parser_pricefast.h:69) and
    the 24-bit-offset codewords."""
    rnd = random.Random(seed)
    head = bytes(rnd.randrange(256) for _ in range(70000))
    out = bytearray(head)
    while len(out) < n:
        k = rnd.choice([5, 8, 12, 17, 19, 20, 21, 24, 40, 100])
        at = rnd.randrange(0, 4000)                      # source near the start: offsets >= 65536
        out += head[at:at + k]
        out += bytes(rnd.randrange(256) for _ in range(rnd.randrange(1, 30)))
    return bytes(out[:n])


def _inputs(seed, count):
    rnd = random.Random(seed)
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        kind = rnd.randrange(7)
        n = rnd.choice([0, 1, 5, 19, 20, 21, 22, 40, 100, 1000, 1025, 2000, 4096, 30000, 65536, 131071, 131072,
                        131073, 200000])
        if kind == 0:
            out.append(lz.datagen(n, rnd.choice([10, 30, 50, 70, 90, 100]), rnd.randrange(1000)))
        elif kind == 1:
            out.append(bytes(n))
        elif kind == 2:
            out.append(rng.integers(0, 256, n, dtype=np.uint8).tobytes())
        elif kind == 3:
            out.append(rng.integers(0, 4, n, dtype=np.uint8).tobytes())
        elif kind == 4:
            out.append((b"abcdefgh" * (n // 8 + 1))[:n])
        elif kind == 5:
            out.append(rng.choice(np.array([65, 66, 67, 200], dtype=np.uint8), size=n, p=[0.9, 0.05, 0.04, 0.01]).tobytes())
        else:
            p = rng.dirichlet(np.ones(256) * 0.05)
            out.append(rng.choice(256, size=n, p=p).astype(np.uint8).tobytes())
    return out


# ---------------------------------------------------------------------------------------------------------
# golden fixtures (generated from the compiled reference by tests/golden/make_golden.py)
# ---------------------------------------------------------------------------------------------------------
def _golden():
    with open(os.path.join(GOLDEN, "golden.json")) as f:
        return json.load(f)


def _golden_input(spec):
    if spec["kind"] == "datagen":
        return lz.datagen(spec["size"], spec["pct"], spec["seed"])
    if spec["kind"] == "zeros":
        return bytes(spec["size"])
    if spec["kind"] == "pattern":
        return (b"abcdefgh" * (spec["size"] // 8 + 1))[: spec["size"]]
    raise ValueError(spec)


def test_datagen_matches_reference_md5():
    g = _golden()
    for spec in g["datagen_md5"]:
        assert hashlib.md5(lz.datagen(spec["size"], spec["pct"], spec["seed"])).hexdigest() == spec["md5"]


def test_oracle_and_shim_compress_match_golden(oracle, shim):
    for case in _golden()["compress"]:
        data = _golden_input(case["input"])
        for impl, fn in (("oracle", o_compress), ("shim", shim_compress)):
            L = oracle if impl == "oracle" else shim
            if case["mode"] == "single":
                got = fn(L, data, case["level"])
            else:
                got = b"".join(fn(L, data[i:i + BS], case["level"], case.get("cap")) for i in range(0, len(data), BS))
            assert len(got) == case["size"], (impl, case)
            assert hashlib.sha256(got).hexdigest() == case["sha256"], (impl, case)


def test_oracle_decompress_matches_golden_vectors(oracle):
    for case in _golden()["vectors"]:
        comp = bytes.fromhex(case["compressed_hex"])
        r, out = o_decompress(oracle, comp, case["cap"])
        assert r == case["result"], case["name"]
        if r > 0:
            assert hashlib.sha256(out).hexdigest() == case["sha256"], case["name"]


# ---------------------------------------------------------------------------------------------------------
# comparison with the reference's answers
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("level", LEVELS)
def test_compress_parity_datagen_blocks(ref, oracle, shim, level):
    data = lz.datagen(1 << 20)
    for i in range(0, len(data), BS):
        blk = data[i:i + BS]
        want = ref.compress(blk, level, BS - 1)
        assert o_compress(oracle, blk, level, BS - 1) == want, (level, i)
        assert shim_compress(shim, blk, level, BS - 1) == want, (level, i)


@pytest.mark.parametrize("level", [10, 21, 41])
def test_compress_parity_multi_inner_block(ref, oracle, shim, level):
    data = lz.datagen((1 << 20) + 4321, 50, 2)
    want = ref.compress(data, level)
    assert o_compress(oracle, data, level) == want
    assert shim_compress(shim, data, level) == want


def test_compress_parity_fuzz(ref, oracle, shim):
    rnd = random.Random(3)
    for data in _inputs(3, 250):
        level = rnd.choice(LEVELS)
        bound = lz_bound(len(data))
        cap = rnd.choice([bound, bound, max(len(data) - 1, 1), len(data) // 2 + 1, rnd.randrange(1, bound + 1)])
        want = ref.compress(data, level, cap)
        assert o_compress(oracle, data, level, cap) == want, (level, len(data), cap)
        assert shim_compress(shim, data, level, cap) == want, (level, len(data), cap)


@pytest.mark.parametrize("level", LEVELS)
def test_warp_emulated_device_path_bit_exact(ref, shim, level):
    """32-lane lane-parallel parsers + Huffman packer (the code the GPU runs) vs the reference."""
    rnd = random.Random(level)
    chain = level in (13, 16, 34)            # the chain walk is slow under the coroutine emulator: smaller inputs
    data = lz.datagen(BS + 3000, 50, level)
    if chain:
        assert emu_compress(shim, data[:40000], level, 39999) == ref.compress(data[:40000], level, 39999)
        tail = data[BS - 9000:]                 # 12000 bytes
        assert emu_compress(shim, tail, level) == ref.compress(tail, level)
    else:
        assert emu_compress(shim, data[:BS], level, BS - 1) == ref.compress(data[:BS], level, BS - 1)
        assert emu_compress(shim, data, level) == ref.compress(data, level)      # two inner blocks
    for d in _inputs(100 + level, 14):
        if chain and len(d) > 30000:
            d = d[:30000]
        cap = rnd.choice([lz_bound(len(d)), max(len(d) - 1, 1), len(d) // 2 + 1])
        assert emu_compress(shim, d, level, cap) == ref.compress(d, level, cap), (level, len(d), cap)


@pytest.mark.parametrize("level", [20, 40, 21, 41, 22])
def test_far_matches_bit_exact(ref, oracle, shim, level):
    """LIZv1 levels on input whose matches lie 65536 or more bytes back, shorter and longer than MM_LONGOFF + MINMATCH: the
    far-candidate rule of fastBig / priceFast and the 24-bit-offset codewords; oracle, one lane, 32 emulated lanes, packed and
    plain (tagged) table, a two-inner-block unit."""
    for seed, n in ((3, BS), (4, BS), (5, 100000), (6, BS + 50000)):
        data = far_match_input(seed, n)
        want = ref.compress(data, level)
        assert 0 < len(want) < len(data)
        assert o_compress(oracle, data, level) == want, (level, seed)
        assert shim_compress(shim, data, level) == want, (level, seed)
        assert emu_compress(shim, data, level) == want, (level, seed)
        shim.lzb_force_plain_table(1)
        try:
            assert shim_compress(shim, data, level) == want, (level, seed)
            assert emu_compress(shim, data, level) == want, (level, seed)
        finally:
            shim.lzb_force_plain_table(0)
        r, out = o_decompress(oracle, want, len(data))
        assert r == len(data) and out == data


@pytest.mark.parametrize("level", [10, 30, 21, 41, 22, 20])
def test_plain_table_with_entry_tags_bit_exact(ref, shim, level):
    """On the device the warps of a CTA that have no shared-memory table run these levels on the plain 32-bit table,
    whose entries carry a 7-bit candidate tag while every position of the unit is below 2^17.  Same bytes as the
    reference, one lane and 32 emulated lanes, single-block units (tagged) and a two-block unit (untagged)."""
    rnd = random.Random(1000 + level)
    shim.lzb_force_plain_table(1)
    try:
        data = lz.datagen(2 * BS + 777, 50, level)
        for blk in (data[:BS], data[BS:2 * BS], data[:70000]):
            want = ref.compress(blk, level, BS - 1)
            assert shim_compress(shim, blk, level, BS - 1) == want, (level, len(blk))
            assert emu_compress(shim, blk, level, BS - 1) == want, (level, len(blk))
        want = ref.compress(data, level)
        assert shim_compress(shim, data, level) == want
        assert emu_compress(shim, data, level) == want
        for d in _inputs(200 + level, 12):
            cap = rnd.choice([lz_bound(len(d)), max(len(d) - 1, 1)])
            want = ref.compress(d, level, cap)
            assert shim_compress(shim, d, level, cap) == want, (level, len(d), cap)
            assert emu_compress(shim, d, level, cap) == want, (level, len(d), cap)
    finally:
        shim.lzb_force_plain_table(0)


def test_decompress_parity_valid_and_corrupt(ref, oracle):
    rnd = random.Random(9)
    for data in _inputs(9, 120):
        level = rnd.choice([10, 21, 41, 30, 17, 22])
        comp = ref.compress(data, level)
        r, out = o_decompress(oracle, comp, len(data))
        assert r == len(data) and out == data
        for _ in range(8):
            bad = bytearray(comp)
            mode = rnd.randrange(3)
            if mode == 0 and bad:
                bad[rnd.randrange(len(bad))] ^= 1 << rnd.randrange(8)
            elif mode == 1:
                bad = bad[: rnd.randrange(0, len(bad) + 1)]
            elif bad:
                bad[rnd.randrange(min(len(bad), 30))] = rnd.randrange(256)
            bad = bytes(bad)
            cap = rnd.choice([len(data), len(data), max(len(data) - 1, 0), len(data) + 50])
            rr, ro = ref.decompress(bad, cap)
            r, out = o_decompress(oracle, bad, cap)
            assert r == rr, (level, len(data), len(bad), cap)
            if rr > 0:
                assert out == ro


def _shim_decompress(L, fn, comp, cap):
    dst = ctypes.create_string_buffer(max(cap, 1) + 64)
    r = getattr(L, fn)(comp, len(comp), dst, cap)
    return r, (dst.raw[:r] if r > 0 else b"")


@pytest.mark.parametrize("level", [10, 21, 41, 30, 17])
def test_compress_into_exact_and_short_capacity(ref, oracle, shim, level):
    """tests/fuzzer.c:442-481 of the reference: compressing into exactly `compressedSize` bytes succeeds with the same
    bytes, one byte less returns what the reference returns (0), and nothing is written behind the capacity."""
    for blk in (lz.datagen(BS, 50, level), lz.datagen(70000, 30, level + 1), lz.datagen(3000, 50, 7), bytes(5000)):
        full = ref.compress(blk, level)
        for cap in (len(full), len(full) - 1, len(full) // 2):
            want = ref.compress(blk, level, cap)
            assert (want == full) == (cap == len(full))
            assert o_compress(oracle, blk, level, cap) == want, (level, len(blk), cap)
            for fn in (shim.lzb_host_compress, shim.lzb_emu_compress):
                dst = ctypes.create_string_buffer(b"\xA5" * (cap + 64), cap + 64)
                n = fn(blk, len(blk), dst, cap, level)
                assert dst.raw[:n] == want, (level, len(blk), cap, n, len(want))
                assert dst.raw[cap:] == b"\xA5" * 64, "wrote behind the capacity"


def test_reference_overrun_behind_a_raw_inner_block_is_refused(ref, oracle, shim):
    """Found by tools/fuzz_parity.py.  A unit whose first inner block is stored raw and whose second is compressed, decoded
    with maxDecompressedSize one byte (or 100) short: the reference does not charge the raw block against the capacity
    (lib/lizard_decompress.c:164-180), decodes the second block past the end of `dst` and reports success.  The oracle
    restates that; the device decoder (host build, one lane and 32 emulated lanes) refuses and writes nothing behind the
    capacity.  Everything agrees again as soon as the capacity is the real size."""
    rng = np.random.default_rng(1)
    data = rng.integers(0, 256, BS, dtype=np.uint8).tobytes() + lz.datagen(40000)
    shim.lzb_host_decompress.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_int]
    shim.lzb_emu_decompress.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_int]
    for level in (10, 21, 41):
        comp = ref.compress(data, level)
        assert comp[1] == 0x80                                   # first inner block raw
        for cap in (len(data), len(data) - 1, len(data) - 100):
            rr, _ = ref.decompress(comp, cap)
            assert rr == len(data)                                  # the reference "succeeds" in all three cases
            assert o_decompress(oracle, comp, cap)[0] == rr if cap == len(data) else True
            for fn in (shim.lzb_host_decompress, shim.lzb_emu_decompress):
                dst = ctypes.create_string_buffer(b"\xA5" * (len(data) + 64), len(data) + 64)
                r = fn(comp, len(comp), dst, cap)
                assert dst.raw[cap:] == b"\xA5" * (len(data) + 64 - cap), "wrote behind the capacity"
                if cap == len(data):
                    assert r == len(data) and dst.raw[:r] == data
                else:
                    assert r < 0, (level, cap, r)


def test_input_one_byte_short_or_long_matches_reference(ref, oracle, shim):
    """tests/fuzzer.c:417-427 of the reference: compressed input with one byte missing / extra bytes appended.  Oracle
    restatement and the host build of the device decoder return what the reference returns."""
    rnd = random.Random(9)
    shim.lzb_host_decompress.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_int]
    for level in (10, 21, 41, 30, 17):
        for blk in (lz.datagen(BS, 50, level), lz.datagen(5000, 50, level), lz.datagen(BS + 777, 50, level), b"", b"a" * 100):
            comp = ref.compress(blk, level)
            for c in (comp[:-1], comp + b"\x00", comp + b"\x80", comp + b"\xff", comp + bytes([rnd.randrange(256)]),
                      comp + bytes(4)):
                for cap in (len(blk), len(blk) + 64):
                    rr, _ = ref.decompress(c, cap)
                    assert o_decompress(oracle, c, cap)[0] == rr, (level, len(blk), len(c), cap)
                    buf = ctypes.create_string_buffer(max(cap, 1) + 64)
                    assert shim.lzb_host_decompress(c, len(c), buf, cap) == rr, (level, len(blk), len(c), cap)


@pytest.mark.parametrize("fn,count,variant,order", [("lzb_host_decompress", 90, 3, 0), ("lzb_host_decompress", 40, 0, 0),
                                                    ("lzb_emu_decompress", 14, 3, 0), ("lzb_emu_decompress", 14, 3, 2),
                                                    ("lzb_emu_decompress", 10, 3, 1), ("lzb_emu_decompress", 8, 0, 2),
                                                    ("lzb_emu_decompress", 6, 1, 1), ("lzb_emu_decompress", 6, 2, 2)])
def test_device_decoder_code_on_host_matches_reference(ref, shim, fn, count, variant, order):
    """The batch token loops (1 lane, and 32 emulated lanes = what the GPU runs): same return codes as the
    reference on valid and damaged streams, same bytes whenever the reference's own output is well defined.
    `variant` = schedule of the token loops (bit 0 pooled copy sweeps, bit 1 compact extension chain; the device
    default is 3), `order` = order in which the emulator runs the lanes between two collectives (forward, reverse,
    shuffled): a missing barrier only shows under some orders."""
    shim.lzb_set_decode_variant(variant)
    shim.lzb_emu_lane_order(order)
    rnd = random.Random(21)
    compared = 0
    for data in _inputs(21, count):
        level = rnd.choice([10, 21, 41, 30, 17, 22, 42])
        comp = ref.compress(data, level)
        cases = [(comp, len(data)), (comp, max(len(data) - 1, 0)), (comp, len(data) + 77)]
        for _ in range(5):
            bad = bytearray(comp)
            if not bad:
                break
            mode = rnd.randrange(3)
            if mode == 0:
                bad[rnd.randrange(len(bad))] ^= 1 << rnd.randrange(8)
            elif mode == 1:
                bad = bad[: rnd.randrange(0, len(bad) + 1)]
            else:
                bad[rnd.randrange(min(40, len(bad)))] = rnd.randrange(256)
            cases.append((bytes(bad), rnd.choice([len(data), max(len(data) - 1, 0), len(data) + 100])))
        for c, cap in cases:
            rr, ro = ref.decompress(c, cap)
            r, o = _shim_decompress(shim, fn, c, cap)
            assert r == rr, (fn, level, len(data), len(c), cap)
            if rr > 0 and refs.stream_obeys_min_offset(c, cap):
                compared += 1
                assert o == ro, (fn, level, len(data), cap)
    shim.lzb_set_decode_variant(3)
    shim.lzb_emu_lane_order(0)
    assert compared > 0


def stored_optimal_parser_cases():
    """(level, input, stream, cap, intact) of the reference's lowest-price (24) and optimal (45) parsers, which the oracle
    does not restate: the stored streams (tests/golden/make_golden.py) with room for all and for one byte less, and damaged
    copies."""
    rnd = random.Random(2445)
    out = []
    with np.load(os.path.join(GOLDEN, "optimal_parser_streams.npz")) as z:
        for name in sorted(z.files):
            level, size, pct, seed = (int(f[1:]) for f in name.split("_"))
            data, comp = lz.datagen(size, pct, seed), z[name].tobytes()
            out += [(level, data, comp, size, True), (level, data, comp, size - 1, False)]
            for _ in range(6):
                bad = bytearray(comp)
                if rnd.randrange(2):
                    bad = bad[:rnd.randrange(len(bad))]
                else:
                    bad[rnd.randrange(len(bad))] ^= 1 << rnd.randrange(8)
                out.append((level, data, bytes(bad), size, False))
    return out


def test_decoders_on_stored_optimal_parser_streams(ref, oracle, shim):
    """The random-input decode tests use levels the oracle can compress; the reference's lowest-price and optimal parsers
    write the same two stream formats with other token choices.  Their stored streams, valid and damaged: the oracle, the
    one-lane and the 32-lane token decoder return what the reference returns."""
    compared = 0
    for level, data, comp, cap, intact in stored_optimal_parser_cases():
        rr, ro = ref.decompress(comp, cap)
        if intact:
            assert rr == len(data) and ro == data
        results = [o_decompress(oracle, comp, cap)] + [_shim_decompress(shim, fn, comp, cap)
                                                        for fn in ("lzb_host_decompress", "lzb_emu_decompress")]
        for i, (r, o) in enumerate(results):
            assert r == rr, (i, level, len(data), len(comp), cap, r, rr)
            if rr > 0 and refs.stream_obeys_min_offset(comp, cap):
                compared += 1
                assert o == ro, (i, level, len(data), cap)
    assert compared > 0


@pytest.mark.parametrize("level", [10, 21, 41])
def test_emulated_decoder_full_blocks_all_schedules(ref, shim, level):
    """Whole 128 KiB datagen blocks (long literal runs and matches, multi-byte length extensions), a two-inner-block
    unit and highly repetitive input (overlapping and near matches) through every schedule of the 32-lane decoder, at
    odd destination alignments (the pooled sweeps cut runs at the 16-byte boundaries of the destination)."""
    data = lz.datagen(3 * BS)
    rep = b"abcdefghij" * 3000 + bytes(range(256)) * 40 + b"\0" * 5000 + b"xyzw" * 4000 + data[:3000]
    cases = [data[:BS], data[BS:2 * BS + 4321], rep]
    for variant, order in ((3, 0), (3, 2), (1, 1), (2, 2)):
        shim.lzb_set_decode_variant(variant)
        shim.lzb_emu_lane_order(order)
        for i, c in enumerate(cases):
            comp = ref.compress(c, level)
            buf = ctypes.create_string_buffer(len(c) + 96)
            mis = (5 * i + variant + order) % 16
            base = ctypes.addressof(buf) + mis
            r = shim.lzb_emu_decompress(comp, len(comp), ctypes.cast(base, ctypes.c_char_p), len(c))
            assert r == len(c) and ctypes.string_at(base, len(c)) == c, (level, variant, order, i, r)
            assert ctypes.string_at(base + len(c), 16) == bytes(16), "wrote past the end of the destination"
    shim.lzb_set_decode_variant(3)
    shim.lzb_emu_lane_order(0)


def test_emulated_decoder_chain_window_source_alignments(ref, shim):
    """The compact extension chain walks a 1 KiB window of the literals stream that starts at the 16-byte aligned ADDRESS at
    or below the chain's position (decode.cuh: ext_chain_win), so its behaviour depends on where the compressed stream lies in
    memory.  Every source alignment mod 16, both codeword flavours, inputs with long literal runs (multi-byte extension
    fields, several windows per batch) and with only short ones, plus damaged copies of one stream: same code (and bytes)
    as the reference."""
    rnd = random.Random(17)
    data = lz.datagen(BS + 64, 30, 5)
    runs = bytearray()
    while len(runs) < 70000:                      # literal runs of 300-5000 bytes between short matches
        runs += bytes(rnd.randrange(256) for _ in range(rnd.choice([300, 700, 1021, 1024, 1030, 5000]))) + runs[-40:-8] * 2
    cases = [data[:BS], bytes(runs[:70000]), lz.datagen(40000, 90, 3)]
    shim.lzb_set_decode_variant(3)
    for level in (10, 21):
        for ci, c in enumerate(cases):
            comp = ref.compress(c, level)
            for mis in range(16):
                raw = ctypes.create_string_buffer(len(comp) + 32)
                ctypes.memmove(ctypes.addressof(raw) + mis, comp, len(comp))
                buf = ctypes.create_string_buffer(len(c) + 64)
                r = shim.lzb_emu_decompress(ctypes.cast(ctypes.addressof(raw) + mis, ctypes.c_char_p), len(comp), buf, len(c))
                assert r == len(c) and buf.raw[:len(c)] == c, (level, ci, mis, r)
        comp = ref.compress(cases[1], level)
        for t in range(60):
            bad = bytearray(comp)
            if t % 3 == 0:
                bad = bad[:rnd.randrange(len(bad) // 2, len(bad))]
            else:
                for _ in range(rnd.randrange(1, 4)):
                    bad[rnd.randrange(16, len(bad))] = rnd.randrange(256)
            bad = bytes(bad)
            mis = t % 16
            raw = ctypes.create_string_buffer(len(bad) + 32)
            ctypes.memmove(ctypes.addressof(raw) + mis, bad, len(bad))
            buf = ctypes.create_string_buffer(len(cases[1]) + 64)
            rr, ro = ref.decompress(bad, len(cases[1]))
            r = shim.lzb_emu_decompress(ctypes.cast(ctypes.addressof(raw) + mis, ctypes.c_char_p), len(bad), buf, len(cases[1]))
            assert r == rr, (level, t, r, rr)
            if rr > 0 and refs.stream_obeys_min_offset(bad, len(cases[1])):
                assert buf.raw[:rr] == ro


def test_prepasses_match_reference(ref, shim):
    """The decoder's two pre-passes run serially on the host -- Huffman pre-pass (plan the first inner block, expand the
    planned streams segment by segment) and token pre-pass (one-lane parse of the block into sequence records, mode bit
    4) -- feeding the 1-lane and the 32-lane token decoder: same return codes and bytes as the reference on valid and
    damaged streams, and the token decoder really consumes the pre-expanded bytes (negative control)."""
    shim.lzb_decompress_with_prepass.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_int, ctypes.c_int,
                                                 ctypes.POINTER(ctypes.c_int)]

    def dec(comp, cap, mode):
        buf = ctypes.create_string_buffer(cap + 64)
        jd = ctypes.c_int(0)
        r = shim.lzb_decompress_with_prepass(comp, len(comp), buf, cap, mode, ctypes.byref(jd))
        return r, buf.raw[:max(r, 0)], jd.value

    rnd = random.Random(3)
    data = lz.datagen(3 * BS)
    expanded = 0
    for level in (41, 30, 42, 10, 37):
        for blk in (data[:BS], data[BS:2 * BS + 999], data[:20000]):
            comp = ref.compress(blk, level)
            for mode in (0, 1, 4, 5):                             # one lane / 32 emulated lanes, without / with token pre-pass
                r, out, jd = dec(comp, len(blk), mode)
                assert r == len(blk) and out == blk, (level, len(blk), mode, r)
                if mode & 4:
                    assert jd & 16, (level, len(blk), mode)           # the block was parsed into records
            expanded += jd & 15
            if level >= 30 and len(blk) >= BS:
                assert (jd & 15) >= 1, (level, jd)
                assert dec(comp, len(blk), 2)[1] != blk           # expanded streams overwritten -> output must change
            for _ in range(25):
                bad = bytearray(comp)
                m = rnd.randrange(3)
                if m == 0:
                    bad[rnd.randrange(len(bad))] ^= 1 << rnd.randrange(8)
                elif m == 1:
                    bad = bad[: rnd.randrange(0, len(bad) + 1)]
                else:
                    bad[rnd.randrange(min(60, len(bad)))] = rnd.randrange(256)
                bad = bytes(bad)
                cap = rnd.choice([len(blk), len(blk) - 1, len(blk) + 50])
                rr, ro = ref.decompress(bad, cap)
                r, out, _ = dec(bad, cap, rnd.choice([0, 4, 5]))
                assert r == rr, (level, len(blk), len(bad), cap, r, rr)
                if rr > 0 and refs.stream_obeys_min_offset(bad, cap):
                    assert out == ro
    assert expanded > 0


def test_huffman_ring_window_misaligned_sources_and_long_codes(ref, shim):
    """The expand pre-pass's sixteen-symbol rounds read the bitstream through an address-mapped 64-byte ring refilled once
    per round (decode.cuh: huf_lane_segment_t<true>); the CPU shim runs the same loop with an abort on any reload that
    would miss the ring.  Sources at every alignment mod 16, and streams whose tail is made of 10/11-bit codes (a round
    then consumes more than 16 bytes: two refills in one round)."""
    shim.lzb_decompress_with_prepass.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_int, ctypes.c_int,
                                                 ctypes.POINTER(ctypes.c_int)]
    rnd = random.Random(11)

    def check(blk, level, mis):
        comp = ref.compress(blk, level)
        raw = ctypes.create_string_buffer(len(comp) + 32)
        ctypes.memmove(ctypes.addressof(raw) + mis, comp, len(comp))
        buf = ctypes.create_string_buffer(len(blk) + 64)
        jd = ctypes.c_int(0)
        r = shim.lzb_decompress_with_prepass(ctypes.cast(ctypes.addressof(raw) + mis, ctypes.c_char_p), len(comp), buf, len(blk),
                                             0, ctypes.byref(jd))
        assert r == len(blk) and buf.raw[:len(blk)] == blk, (level, len(blk), mis, r)
        return jd.value & 15

    data = lz.datagen(BS + 16)
    jobs = 0
    for mis in range(16):
        jobs += check(data[mis:mis + BS], 41 if mis & 1 else 30, mis)

    def skewed(n, nrare, tail):
        common = [rnd.randrange(256) for _ in range(3)]
        rare = rnd.sample(range(256), nrare)
        out = bytearray()
        cut = int(n * (1 - tail))
        while len(out) < cut:
            out.append(rnd.choice(common) if rnd.random() < 0.97 else rnd.choice(rare))
        while len(out) < n:
            out.append(rnd.choice(rare) if rnd.random() < 0.9 else rnd.choice(common))
        return bytes(out)

    for trial in range(10):
        blk = skewed(rnd.choice([BS, 70000, 40000]), rnd.choice([60, 120, 200, 250]), rnd.choice([0.05, 0.1, 0.25]))
        for level in (30, 41):
            jobs += check(blk, level, trial % 16)
    assert jobs >= 30


def test_huffman_two_level_table_equals_reference_layout(shim):
    """The pre-pass's two-level decode table (HufCompact) answers every lookup like the 1 << tableLog table of
    HUF_readDTableX2 (huf_decompress.c:87-133), for random complete codes of every table log."""
    rnd = random.Random(5)
    shim.lzb_huf_compact_check.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int]
    seen = set()
    for trial in range(400):
        max_depth = rnd.randrange(1, 12)
        leaves = [1, 1]
        want = rnd.randrange(2, 257)
        while len(leaves) < want:
            cand = [i for i, d in enumerate(leaves) if d < max_depth]
            if not cand:
                break
            # prefer deep leaves now and then so that long codes (the second level) are well populated
            i = max(cand, key=lambda k: leaves[k]) if rnd.random() < 0.3 else rnd.choice(cand)
            d = leaves.pop(i)
            leaves += [d + 1, d + 1]
        tl = max(leaves)
        syms = rnd.sample(range(256), len(leaves))
        weights = bytearray(256)
        for s, d in zip(syms, leaves):
            weights[s] = tl + 1 - d
        nsym = max(syms) + 1
        assert shim.lzb_huf_compact_check(bytes(weights), nsym, tl) == 0, (trial, tl, len(leaves))
        seen.add(tl)
    assert seen >= set(range(2, 12))


def test_huffman_stage_parity(ref, oracle, shim):
    rnd = random.Random(4)
    rng = np.random.default_rng(4)
    for _ in range(300):
        n = rnd.choice([13, 50, 300, 1025, 5000, 20000, 70000, 131072])
        k = rnd.choice([2, 3, 16, 100, 256])
        p = rng.dirichlet(np.ones(k) * rnd.choice([0.1, 0.5, 2.0]))
        data = rng.choice(k, size=n, p=p).astype(np.uint8).tobytes()
        cap = n + n // 256 + 8 + 129
        b = ctypes.create_string_buffer(cap + 16)
        want = ref.huf_compress(data, cap)
        cb = oracle.oracle_HUF_compress(b, cap, data, n)
        if want is None:
            assert cb == ctypes.c_size_t(-1).value
            continue
        ca = len(want)
        assert ca == cb and (ca <= 1 or want == b.raw[:cb]), (n, k)
        if ca <= 1:
            continue
        comp = bytearray(want)
        for trial in range(5):
            bad = bytes(comp) if trial == 0 else bytes(_damage(comp, rnd))
            nn = n if trial < 3 else n + rnd.choice([-1, 1])
            d2 = ctypes.create_string_buffer(nn + 16)
            d3 = ctypes.create_string_buffer(nn + 16)
            r1, o1 = ref.huf_decompress(bad, nn)
            r2 = oracle.oracle_HUF_decompress(d2, nn, bad, len(bad))
            r3 = shim.lzb_host_huf_decompress(d3, nn, bad, len(bad))
            e1 = r1 < 0
            assert e1 == (r2 == ctypes.c_size_t(-1).value) == (r3 < 0), (n, k, trial)
            if not e1:
                assert o1 == d2.raw[:nn] == d3.raw[:nn]


def _damage(comp, rnd):
    bad = bytearray(comp)
    mode = rnd.randrange(3)
    if mode == 0:
        bad[rnd.randrange(len(bad))] ^= 1 << rnd.randrange(8)
    elif mode == 1:
        bad = bad[: rnd.randrange(1, len(bad) + 1)]
    else:
        bad[-1] = rnd.randrange(256)
    return bad


def test_reference_facts_from_survey(ref):
    """SURVEY.md section 8c regression facts, reproduced with the reference's answers."""
    data = lz.datagen(4 << 20)
    assert hashlib.md5(data).hexdigest() == "b4ac2db04e3844e152d1c9987ed8a711"
    for level, single, blocks in ((10, 2475712, 2647396), (21, 2239670, 2431837), (41, 1413150, 1521776)):
        assert len(ref.compress(data, level)) == single
        assert sum(len(ref.compress(data[i:i + BS], level)) for i in range(0, len(data), BS)) == blocks
