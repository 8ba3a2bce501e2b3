"""GPU parity at BASELINE.json's full size (configs 1-3: 1 GiB `datagen -P50`, 8192 independent 128 KiB blocks).

The compiled reference needs minutes for 1 GiB per level, so the check goes through reference-generated facts instead --
a checksum of checksums: the input's md5, the total compressed size and the SHA-256 of the 8192 compressed blocks
concatenated, all taken from the reference built with -DLIZARD_RESET_MEM (`Lizard_compress(block, cap = srcSize-1)` per
block; the sizes and the XXH64 of the same streams are SURVEY.md section 8c's facts) -- plus the round trip."""
import ctypes
import hashlib

import numpy as np
import pytest

import lizard_b200 as lz

pytestmark = pytest.mark.gpu
BS = lz.BLOCK_SIZE
N = 1 << 30
# level -> (compressed bytes, SHA-256 of the concatenated blocks)
FACTS_1G = {10: (670259129, "ed6159bb08e1509bc0d585195f1d1d6fc589724749c90b358ab8cc589a89f023"),
            21: (616060194, "e19093ae2fdfc7f595fb3670323b1d7b535fd9d0abf4e058c6146c1ff9cfc8e4"),
            41: (385653946, "b564134e421d99fd4687da6fa90e29a30fc60e58f5f410b395e25a05c04b4d90")}
MD5_1G = "b98d56d2653b6ab1b74ebe6c827ec231"


@pytest.fixture(scope="module")
def data1g():
    a = np.empty(N, dtype=np.uint8)
    lz.datagen_into(a.ctypes.data, N, 50.0, 0)
    assert hashlib.md5(a).hexdigest() == MD5_1G          # == `datagen -g1G -P50` of the reference (programs/datagen.c)
    return a


@pytest.mark.parametrize("level", [10, 21, 41])
def test_one_gib_matches_reference_facts(data1g, level):
    L = lz.lib()
    L.LizardB200_compress_blocks.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t,
                                             ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    L.LizardB200_decompress_blocks.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t,
                                               ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    n = N // BS
    comp = np.empty(n * BS, dtype=np.uint8)              # unit i at i * BS, capacity BS - 1 (lizard_frame.c:459)
    sizes = np.zeros(n, dtype=np.int32)
    st = L.LizardB200_compress_blocks(data1g.ctypes.data, N, BS, comp.ctypes.data, BS, BS - 1, sizes.ctypes.data, level)
    assert st == 0, L.LizardB200_lastError()
    assert int(sizes.min()) > 0
    total, sha = FACTS_1G[level]
    assert int(sizes.sum(dtype=np.int64)) == total
    packed = np.empty(total, dtype=np.uint8)
    at = 0
    for i in range(n):
        k = int(sizes[i])
        packed[at:at + k] = comp[i * BS:i * BS + k]
        at += k
    assert hashlib.sha256(packed).hexdigest() == sha
    del packed
    back = np.zeros(N, dtype=np.uint8)
    res = np.zeros(n, dtype=np.int32)
    st = L.LizardB200_decompress_blocks(comp.ctypes.data, BS, sizes.ctypes.data, n, back.ctypes.data, BS, res.ctypes.data)
    assert st == 0, L.LizardB200_lastError()
    assert int(res.min()) == BS and int(res.max()) == BS
    assert np.array_equal(back, data1g)
