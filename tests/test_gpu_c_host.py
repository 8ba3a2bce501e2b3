"""GPU: the plain-C host programs -- examples/frame_roundtrip.c (LizardF_compressFrame / LizardF_decompress) and
examples/block_bench.c (the batch form of programs/bench.c: LizardB200_compress_blocks / _decompress_blocks)."""
import subprocess

import pytest

from tests.test_abi_cpu import build_c_host

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("level", [10, 41])
def test_c_host_frame_round_trip(tmp_path, level):
    exe = build_c_host(tmp_path)
    r = subprocess.run([exe, "32", str(level)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    assert "round trip ok" in r.stdout


@pytest.mark.parametrize("level", [10, 41])
def test_c_host_block_bench(tmp_path, level):
    exe = build_c_host(tmp_path, "block_bench")
    r = subprocess.run([exe, str(level), "64", "1"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    assert "512 blocks of 128 KiB" in r.stdout and "MB/s" in r.stdout


@pytest.mark.parametrize("level,checksum", [(10, 1), (41, 0)])
def test_c_host_whole_file_batching(tmp_path, level, checksum):
    """examples/lizard_file.c: the CLI's file loop (programs/lizardio.c:397-441, 617-677) with whole-file batches.  The .liz it
    writes is byte-identical to the reference's own LizardF_compressFrame of the same bytes (parity build) and the reference's
    frame decoder reads it; decoding through the tool with a small input chunk (blocks straddle reads) gives the file back."""
    import ctypes
    import lizard_b200 as lz
    from tests import refs
    exe = build_c_host(tmp_path, "lizard_file")
    data = lz.datagen(5 * (1 << 20) + 12345, 50, level)
    src, liz, back = [str(tmp_path / n) for n in ("in.bin", "out.liz", "back.bin")]
    open(src, "wb").write(data)
    r = subprocess.run([exe, "c", str(level), src, liz, "2", str(checksum)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.stdout, r.stderr)
    frame = open(liz, "rb").read()
    ref = refs.reference()
    want = ref.frame_compress(data, lz.make_prefs(level, 1, True, bool(checksum), 0))
    assert frame == want
    res, out = ref.frame_decompress(frame, len(data))
    assert res == 0 and out == data
    r = subprocess.run([exe, "d", liz, back, "1"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.stdout, r.stderr)
    assert open(back, "rb").read() == data
