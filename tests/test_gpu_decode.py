"""GPU parity: Lizard_decompress_safe / LizardB200_decompress_batch vs the compiled reference."""
import ctypes
import random

import pytest

import lizard_b200 as lz
from tests import refs

pytestmark = pytest.mark.gpu
BS = lz.BLOCK_SIZE
DEFAULT_VARIANT = 7          # the library's default (api.cu Context::dec_variant)


@pytest.fixture(scope="module")
def ref():
    return refs.reference()


@pytest.fixture(scope="module")
def data4m():
    return lz.datagen(4 << 20)


@pytest.fixture(params=[7, 23], autouse=True, ids=["gen1", "gen2"])
def decode_generation(request):
    """Every test of this file runs on both decode kernels: 7 = first generation (one warp per unit, Huffman pre-pass on),
    23 = second generation (parser + copier warp per unit, TMA-staged literals ring; decode2.cuh)."""
    L = lz.lib()
    L.LizardB200_setDecodeVariant.argtypes = [ctypes.c_int]
    assert L.LizardB200_setDecodeVariant(request.param) == 0
    yield request.param
    L.LizardB200_setDecodeVariant(DEFAULT_VARIANT)


@pytest.mark.parametrize("level", [10, 21, 41, 30, 11, 17, 22, 42])
def test_decode_blocks_match_original(ref, data4m, level):
    n = 32 if level in (10, 21, 41) else 6
    blocks = [data4m[i * BS:(i + 1) * BS] for i in range(n)]
    comp = [ref.compress(b, level) for b in blocks]
    out = lz.decompress_batch(comp, [BS] * len(comp))
    for i, (r, o) in enumerate(out):
        assert r == BS, (level, i, r)
        assert o == blocks[i], (level, i)


@pytest.mark.parametrize("level", [10, 21, 41])
def test_decode_multi_inner_block_unit(ref, data4m, level):
    data = data4m[: 5 * BS + 12345]
    comp = ref.compress(data, level)
    r, o = lz.decompress(comp, len(data))
    assert r == len(data) and o == data


def test_decode_edge_sizes(ref):
    rnd = random.Random(7)
    cases = [b"", b"a", b"ab" * 10, bytes(100), bytes(BS), bytes(rnd.randrange(256) for _ in range(5000)),
             lz.datagen(1000), lz.datagen(BS + 1), lz.datagen(70000, 90.0, 3)]
    for level in (10, 21, 41):
        comp = [ref.compress(c, level) for c in cases]
        out = lz.decompress_batch(comp, [len(c) for c in cases])
        for c, (r, o) in zip(cases, out):
            assert r == len(c) and o == c, (level, len(c), r)
        # one byte short must fail exactly like the reference (fuzzer property, tests/fuzzer.c:400-404)
        out = lz.decompress_batch(comp, [max(len(c) - 1, 0) for c in cases])
        for c, k, (r, o) in zip(cases, comp, out):
            rr, _ = ref.decompress(k, max(len(c) - 1, 0))
            assert r == rr, (level, len(c), r, rr)


def test_input_one_byte_short_or_long_matches_reference(ref):
    """Fuzzer property of the reference (tests/fuzzer.c:417-427): a compressed block with one byte missing or one byte
    (or a few) appended must not decode like the original; whatever the reference returns, we return."""
    rnd = random.Random(9)
    units, caps = [], []
    for level in (10, 21, 41, 30, 17):
        for blk in (lz.datagen(BS, 50, level), lz.datagen(5000, 50, level), lz.datagen(BS + 777, 50, level), b"", b"a" * 100):
            comp = ref.compress(blk, level)
            for c in (comp[:-1], comp + b"\x00", comp + b"\x80", comp + b"\xff", comp + bytes([rnd.randrange(256)]),
                      comp + bytes(4)):
                for cap in (len(blk), len(blk) + 64):
                    units.append(c); caps.append(cap)
    got = lz.decompress_batch(units, caps)
    for i, ((r, _), u, cap) in enumerate(zip(got, units, caps)):
        rr, _ = ref.decompress(u, cap)
        assert r == rr, (i, len(u), cap, r, rr)


@pytest.mark.parametrize("level", [10, 21, 41])
def test_decode_corrupt_matches_reference(ref, data4m, level):
    """Return codes (and bytes when accepted) equal the reference on damaged streams."""
    rnd = random.Random(level)
    blocks = [data4m[i * BS:(i + 1) * BS] for i in range(8)]
    comp = [ref.compress(b, level) for b in blocks]
    bad, caps = [], []
    for k in comp:
        for _ in range(40):
            b = bytearray(k)
            mode = rnd.randrange(4)
            if mode == 0:
                b[rnd.randrange(len(b))] ^= 1 << rnd.randrange(8)
            elif mode == 1:
                b = b[: rnd.randrange(1, len(b))]
            elif mode == 2:
                b[rnd.randrange(min(40, len(b)))] = rnd.randrange(256)
            else:
                for _ in range(3):
                    b[rnd.randrange(len(b))] = rnd.randrange(256)
            bad.append(bytes(b))
            caps.append(rnd.choice([BS, BS, BS - 1, BS + 100]))
    out = lz.decompress_batch(bad, caps)
    n_cmp = 0
    mism = []
    for idx, (b, cap, (r, o)) in enumerate(zip(bad, caps, out)):
        rr, ro = ref.decompress(b, cap)
        if r != rr:
            mism.append((idx, len(b), cap, r, rr))
        elif rr > 0 and refs.stream_obeys_min_offset(b, cap):
            n_cmp += 1
            if o != ro:
                mism.append((idx, len(b), cap, "content"))
    assert not mism, (level, len(mism), mism[:10])
    assert n_cmp > 0


def test_decode_stored_optimal_parser_streams(ref):
    """Streams of the reference's lowest-price and optimal parsers (levels 24 and 45; the other tests draw their streams
    from levels our restatement can compress), valid and damaged, in one batch: same codes and bytes as the reference."""
    from tests.test_oracle import stored_optimal_parser_cases
    cases = stored_optimal_parser_cases()
    got = lz.decompress_batch([c[2] for c in cases], [c[3] for c in cases])
    compared = 0
    for (level, data, comp, cap, intact), (r, o) in zip(cases, got):
        rr, ro = ref.decompress(comp, cap)
        assert r == rr, (level, len(data), len(comp), cap, r, rr)
        if intact:
            assert o == data
        if rr > 0 and refs.stream_obeys_min_offset(comp, cap):
            compared += 1
            assert o == ro, (level, len(data), cap)
    assert compared > 0


def test_decode_schedules_and_prepass_agree(ref, data4m):
    """Every decode configuration (token-loop schedules, with and without the Huffman pre-pass) returns the same
    codes and bytes on a mixed batch: all levels side by side, damaged streams in between, a multi-inner-block unit."""
    rnd = random.Random(77)
    L = lz.lib()
    L.LizardB200_setDecodeVariant.argtypes = [ctypes.c_int]
    units, caps = [], []
    for i in range(48):
        level = [41, 30, 10, 21, 42, 37][i % 6]
        blk = data4m[i * BS:(i + 1) * BS] if i % 5 else data4m[i * BS:i * BS + rnd.randrange(1, BS)]
        k = ref.compress(blk, level)
        units.append(k); caps.append(len(blk))
        b = bytearray(k)
        for _ in range(rnd.randrange(1, 4)):
            b[rnd.randrange(len(b))] ^= 1 << rnd.randrange(8)
        units.append(bytes(b)); caps.append(len(blk))
    big = data4m[: 3 * BS + 555]
    units.append(ref.compress(big, 41)); caps.append(len(big))
    want = [ref.decompress(u, c) for u, c in zip(units, caps)]
    try:
        for variant in (15, 7, 11, 3, 12, 0, 5, 6, 23, 19, 16):
            assert L.LizardB200_setDecodeVariant(variant) == 0
            got = lz.decompress_batch(units, caps)
            for i, ((r, o), (rr, ro)) in enumerate(zip(got, want)):
                assert r == rr, (variant, i, r, rr)
                if rr > 0 and refs.stream_obeys_min_offset(units[i], caps[i]):
                    assert o == ro, (variant, i)
    finally:
        L.LizardB200_setDecodeVariant(DEFAULT_VARIANT)


def test_device_api_unaligned_destinations(ref, data4m):
    """LizardB200_decompress_device with units decoding to arbitrary byte offsets of a device buffer (the second-generation
    copier works in the 16-byte aligned space of each destination and must not touch a byte outside [dst, dst + size))."""
    import torch
    L = lz.lib()
    rnd = random.Random(3)
    dev = torch.device("cuda", 0)
    for level in (10, 21, 41):
        blocks, comp = [], []
        for i in range(24):
            n = BS if i % 3 else rnd.randrange(1, BS)
            blocks.append(data4m[i * BS:i * BS + n])
            comp.append(ref.compress(blocks[-1], level))
        src_off, dst_off, pos_s, pos_d = [], [], 0, 0
        for b, c in zip(blocks, comp):
            pos_s += rnd.randrange(0, 9)
            pos_d += rnd.randrange(1, 40)
            src_off.append(pos_s); dst_off.append(pos_d)
            pos_s += len(c); pos_d += len(b)
        h_src = bytearray(pos_s + 64)
        for o, c in zip(src_off, comp):
            h_src[o:o + len(c)] = c
        d_src = torch.frombuffer(h_src, dtype=torch.uint8).to(dev)
        d_dst = torch.full((pos_d + 64,), 0xEE, dtype=torch.uint8, device=dev)
        t_so = torch.tensor(src_off, dtype=torch.int64, device=dev)
        t_sl = torch.tensor([len(c) for c in comp], dtype=torch.int32, device=dev)
        t_do = torch.tensor(dst_off, dtype=torch.int64, device=dev)
        t_dc = torch.tensor([len(b) for b in blocks], dtype=torch.int32, device=dev)
        t_res = torch.zeros(len(blocks), dtype=torch.int32, device=dev)
        st = L.LizardB200_decompress_device(d_src.data_ptr(), t_so.data_ptr(), t_sl.data_ptr(), d_dst.data_ptr(), t_do.data_ptr(),
                                            t_dc.data_ptr(), t_res.data_ptr(), len(blocks), None)
        assert st == 0, L.LizardB200_lastError()
        torch.cuda.synchronize()
        out = bytes(d_dst.cpu().numpy())
        res = t_res.cpu().tolist()
        want = bytearray(b"\xEE" * len(out))
        for o, b in zip(dst_off, blocks):
            want[o:o + len(b)] = b
        assert res == [len(b) for b in blocks], (level, res)
        assert out == bytes(want), level
