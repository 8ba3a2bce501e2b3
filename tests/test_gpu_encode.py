"""GPU parity: Lizard_compress / LizardB200_compress_batch output must be byte-identical to the reference
built with -DLIZARD_RESET_MEM (clean hash table per call; SURVEY.md section 0.5)."""
import random

import numpy as np
import pytest

import lizard_b200 as lz
from tests import refs

pytestmark = pytest.mark.gpu
BS = lz.BLOCK_SIZE
LEVELS = [10, 11, 13, 15, 17, 20, 21, 22, 30, 31, 34, 38, 40, 41, 42]


@pytest.fixture(scope="module")
def ref():
    return refs.reference()


@pytest.fixture(scope="module")
def data4m():
    return lz.datagen(4 << 20)


@pytest.mark.parametrize("level", LEVELS)
def test_blocks_bit_exact(ref, data4m, level):
    blocks = [data4m[i * BS:(i + 1) * BS] for i in range(32)]
    out = lz.compress_batch(blocks, level, [BS - 1] * 32)      # frame layer's capacity (lizard_frame.c:459)
    for i, (r, o) in enumerate(out):
        want = ref.compress(blocks[i], level, BS - 1)
        assert r == len(want) and o == want, (level, i, r, len(want))


@pytest.mark.parametrize("level", [10, 21, 41])
def test_multi_inner_block_call_bit_exact(ref, data4m, level):
    """Config 1 of BASELINE.json: one Lizard_compress call over 4 MiB = 32 dependent inner blocks."""
    got = lz.compress(data4m, level)
    want = ref.compress(data4m, level)
    assert got == want
    r, back = lz.decompress(got, len(data4m))
    assert r == len(data4m) and back == data4m


def _cases():
    rnd = random.Random(11)
    rng = np.random.default_rng(11)
    out = []
    for n in [0, 1, 5, 19, 20, 21, 22, 40, 100, 1000, 1025, 4096, 65536, 131071, 131072, 131073, 200000]:
        out.append(lz.datagen(n, rnd.choice([10, 50, 90]), rnd.randrange(99)))
        out.append(bytes(n))
        out.append(rng.integers(0, 256, n, dtype=np.uint8).tobytes())
        out.append(rng.integers(0, 3, n, dtype=np.uint8).tobytes())
        out.append((b"abcdefgh" * (n // 8 + 1))[:n])
    return out


@pytest.mark.parametrize("level", LEVELS)
def test_edge_inputs_and_capacities(ref, level):
    rnd = random.Random(level)
    cases = _cases()
    caps = []
    for c in cases:
        bound = ref.Lizard_compressBound(len(c))
        caps.append(rnd.choice([bound, bound, max(len(c) - 1, 1), len(c) // 2 + 1, rnd.randrange(1, bound + 1)]))
    out = lz.compress_batch(cases, level, caps)
    for c, cap, (r, o) in zip(cases, caps, out):
        want = ref.compress(c, level, cap)
        assert r == len(want) and o == want, (level, len(c), cap, r, len(want))


@pytest.mark.parametrize("level", [10, 21, 41, 30, 17])
def test_compress_into_exact_and_short_capacity(ref, level):
    """tests/fuzzer.c:442-481 of the reference: exactly `compressedSize` bytes of room give the same bytes, one byte less
    gives what the reference gives (0)."""
    units, caps = [], []
    for blk in (lz.datagen(BS, 50, level), lz.datagen(70000, 30, level + 1), lz.datagen(3000, 50, 7), bytes(5000)):
        full = ref.compress(blk, level)
        for cap in (len(full), len(full) - 1, len(full) // 2):
            units.append(blk); caps.append(cap)
    out = lz.compress_batch(units, level, caps)
    for blk, cap, (r, o) in zip(units, caps, out):
        want = ref.compress(blk, level, cap)
        assert r == len(want) and o == want, (level, len(blk), cap, r, len(want))


def test_unsupported_level_fails_loudly():
    with pytest.raises(lz.LizardB200Error):
        lz.compress_batch([b"x" * 1000], 12)
    assert lz.compress(b"x" * 1000, 12) == b""      # drop-in symbol: 0 = failed, never a CPU fallback


@pytest.mark.parametrize("level", LEVELS)
def test_round_trip_through_both_gpu_paths(level):
    data = lz.datagen(3 * BS + 777, 60, level)
    blocks = [data[i:i + BS] for i in range(0, len(data), BS)]
    comp = lz.compress_batch(blocks, level)
    back = lz.decompress_batch([c for _, c in comp], [len(b) for b in blocks])
    assert [o for _, o in back] == blocks
