"""GPU parity of the frame layer: LizardF_compressFrame bytes == compiled reference (-DLIZARD_RESET_MEM),
LizardF_decompress of reference frames == original, incl. checksum, content size, raw blocks, chunked feeding."""
import ctypes
import random

import numpy as np
import pytest

import lizard_b200 as lz
from tests import refs

pytestmark = pytest.mark.gpu
BS = lz.BLOCK_SIZE


@pytest.fixture(scope="module")
def ref():
    return refs.reference()


@pytest.fixture(scope="module")
def ours():
    return lz.bind_frame_api(lz.lib())


def _mixed(n, seed):
    rng = np.random.default_rng(seed)
    a = bytearray(lz.datagen(n, 50, seed))
    # one incompressible stretch so that some blocks are stored raw (bit 31 of the size word)
    lo = min(len(a), 3 * BS + 100)
    hi = min(len(a), lo + BS + 5000)
    a[lo:hi] = rng.integers(0, 256, hi - lo, dtype=np.uint8).tobytes()
    return bytes(a)


@pytest.mark.parametrize("level", [10, 21, 41])
@pytest.mark.parametrize("checksum,csize", [(False, 0), (True, 1)])
def test_compress_frame_bit_exact(ref, ours, level, checksum, csize):
    data = _mixed(9 * BS + 12345, level)
    p = lz.make_prefs(level, 1, True, checksum, csize)
    want = ref.frame_compress(data, p)
    got = lz.frame_compress(ours, data, p)
    assert got == want
    r, back = lz.frame_decompress(ours, got, len(data))
    assert r == 0 and back == data
    r, back = ref.frame_decompress(got, len(data))
    assert r == 0 and back == data


def test_compress_frame_small_and_empty(ref, ours):
    for n in (0, 1, 100, 5000, BS - 1, BS, BS + 1):
        data = lz.datagen(n, 50, 3)
        for level in (10, 41):
            p = lz.make_prefs(level, 1, True, True, 0)
            assert lz.frame_compress(ours, data, p) == ref.frame_compress(data, p), (n, level)


def test_larger_frame_blocks_bit_exact(ref, ours):
    data = lz.datagen(600000, 50, 9)
    p = lz.make_prefs(10, 2, True, False, 0)          # 256 KiB frame blocks = units of two dependent inner blocks
    assert lz.frame_compress(ours, data, p) == ref.frame_compress(data, p)


def test_streaming_compress_matches_one_shot(ref, ours):
    rnd = random.Random(5)
    data = _mixed(6 * BS + 777, 5)
    p = lz.make_prefs(10, 1, True, True, 0)
    want = ref.frame_compress(data, p)
    ctx = ctypes.c_void_p()
    assert ours.LizardF_createCompressionContext(ctypes.byref(ctx), 100) == 0
    out = bytearray()
    buf = ctypes.create_string_buffer(len(data) + (len(data) // BS + 2) * 8 + 64)
    n = ours.LizardF_compressBegin(ctx, buf, len(buf), ctypes.byref(p))
    assert not ours.LizardF_isError(n)
    out += buf.raw[:n]
    pos = 0
    while pos < len(data):
        k = min(rnd.choice([1000, 70000, BS, 2 * BS + 5, 300000]), len(data) - pos)
        n = ours.LizardF_compressUpdate(ctx, buf, len(buf), data[pos:pos + k], k, None)
        assert not ours.LizardF_isError(n), ours.LizardF_getErrorName(n)
        out += buf.raw[:n]
        pos += k
    n = ours.LizardF_compressEnd(ctx, buf, len(buf), None)
    assert not ours.LizardF_isError(n)
    out += buf.raw[:n]
    ours.LizardF_freeCompressionContext(ctx)
    assert bytes(out) == want


@pytest.mark.parametrize("level", [10, 21, 41, 17])
def test_decompress_reference_frames(ref, ours, level):
    data = _mixed(7 * BS + 4321, level + 1)
    p = lz.make_prefs(level, 1, True, True, 1)
    frame = ref.frame_compress(data, p)
    for chunk, dchunk in ((0, 0), (1 << 20, 0), (65536, 0), (777, 0), (0, BS // 2), (100000, 200000)):
        r, back = lz.frame_decompress(ours, frame, len(data), chunk, dchunk)
        assert r == 0 and back == data, (level, chunk, dchunk, r, len(back))


def test_frame_errors_match_reference(ref, ours):
    data = lz.datagen(3 * BS, 50, 2)
    p = lz.make_prefs(10, 1, True, True, 0)
    frame = bytearray(ref.frame_compress(data, p))
    cases = []
    for pos, val in ((0, 0x05), (4, 0xFF), (5, 0x80), (6, 0x00), (7, 0xFF), (len(frame) - 1, frame[-1] ^ 1), (20, frame[20] ^ 0x40)):
        b = bytearray(frame)
        b[pos] = val
        cases.append(bytes(b))
    for b in cases:
        r1, o1 = ref.frame_decompress(b, len(data))
        r2, o2 = lz.frame_decompress(ours, b, len(data))
        assert (r1 < 0) == bool(ours.LizardF_isError(r2))
        if r1 < 0:
            assert ours.LizardF_getErrorName(r2) == o1           # the reference's error name


def test_linked_blocks_are_refused(ours):
    p = lz.make_prefs(10, 1, False, False, 0)
    with pytest.raises(lz.LizardB200Error, match="blockMode"):
        lz.frame_compress(ours, lz.datagen(3 * BS), p)


def test_decoder_chunk_ramp_small_chunks_subprocess():
    """The decoder's host pipeline starts with a doubling ramp of small chunks when a call has at least two full chunks
    (frame.inl: FrameChunks).  With LIZARDB200_FRAME_CHUNK_MIB=2 (16 blocks per chunk, ramp 1 / 2 / 4 / 8 blocks) a 6 MiB
    frame exercises the ramp, full chunks and a ragged last chunk; the variable is read once per process, hence the
    subprocess.  Frames from the reference, checksummed, levels 10 and 41, decoded whole and in pieces."""
    import os
    import subprocess
    import sys
    code = r'''
import sys
import lizard_b200 as lz
from tests import refs
BS = lz.BLOCK_SIZE
ref = refs.reference()
ours = lz.bind_frame_api(lz.lib())
L = lz.lib()
import ctypes
L.LizardB200_chunkPlan.argtypes = [ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_uint] + [ctypes.POINTER(ctypes.c_uint)] * 3
assert L.LizardB200_chunkPlan(50, 16, 1, 0, None, None, None) == 4 + 3          # ramp of four chunks, then 16 + 16 + 3 units
for level in (10, 41):
    for nblk, extra in ((50, 777), (32, 0), (47, 1)):
        data = lz.datagen(nblk * BS + extra, 50, level + nblk)
        p = lz.make_prefs(level, 1, True, True, 1)
        frame = ref.frame_compress(data, p)
        assert lz.frame_compress(ours, data, p) == frame
        for chunk, dchunk in ((0, 0), (3 << 20, 0)):
            r, back = lz.frame_decompress(ours, frame, len(data), chunk, dchunk)
            assert r == 0 and back == data, (level, nblk, chunk, r, len(back))
print("ramp ok")
'''
    env = dict(os.environ, LIZARDB200_FRAME_CHUNK_MIB="2")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ramp ok" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]
