"""The C-ABI boundary without a GPU: liblizard_b200.so loads, exports every function include/lizard_b200.h declares, and
every entry point of the product path FAILS (no CPU fallback) when there is no B200 -- loudly through the batch API
(negative status + message), with the reference's own failure value through the drop-in symbols.  Pure host helpers
(Lizard_compressBound, LizardF_compressFrameBound, error names) answer like the reference's."""
import ctypes
import os
import re

import pytest

import lizard_b200 as lz
from tests import refs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "lizard_b200.h")


def _declared_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)              # the header's comments cite symbols it replaces
    text = re.sub(r"//[^\n]*", " ", text)
    names = set(re.findall(r"\b((?:Lizard|LizardF|LizardB200)_\w+)\s*\(", text))
    names -= {n for n in names if re.search(r"typedef[^;]*\b%s\b" % re.escape(n), text)}
    return sorted(names)


def _no_gpu():
    try:
        import torch
        return not torch.cuda.is_available()
    except Exception:
        return True


def test_header_declares_the_reference_surface():
    names = _declared_functions()
    for must in ("Lizard_compress", "Lizard_compress_extState", "Lizard_compressBound", "Lizard_sizeofState",
                 "Lizard_decompress_safe", "LizardF_compressFrame", "LizardF_compressFrameBound", "LizardF_compressBegin",
                 "LizardF_compressUpdate", "LizardF_flush", "LizardF_compressEnd", "LizardF_decompress",
                 "LizardF_getFrameInfo", "LizardF_isError", "LizardF_getErrorName", "LizardB200_compress_batch",
                 "LizardB200_decompress_batch", "LizardB200_compress_device", "LizardB200_decompress_device"):
        assert must in names, must


def test_library_exports_every_declared_symbol():
    L = lz.lib()
    missing = [n for n in _declared_functions() if not hasattr(L, n)]
    assert not missing, missing


def test_host_only_helpers_match_the_reference():
    L = lz.lib()
    ref = refs.reference()
    for n in (0, 1, 20, 131071, 131072, 131073, 1 << 20, 0x7E000000, 0x7E000001):
        assert L.Lizard_compressBound(n) == ref.Lizard_compressBound(n), n
    assert L.Lizard_versionNumber() > 0


def test_sizeof_state_equals_the_reference_for_every_level():
    """Lizard_sizeofState (lib/lizard_compress.c:311-323): callers malloc this many bytes for Lizard_compress_extState; the
    device keeps its own state, but the figure must be the reference's (SURVEY 8 a2: 806045 at level 10, 17632409 at 21/41)."""
    L = lz.lib()
    ref = refs.reference()
    for level in list(range(10, 50)) + [0, 5, 9, 50, 99, -3]:
        assert L.Lizard_sizeofState(level) == ref.Lizard_sizeofState(level), level
    assert L.Lizard_sizeofState(10) == 806045 and L.Lizard_sizeofState(21) == 17632409 == L.Lizard_sizeofState(41)


@pytest.mark.skipif(not _no_gpu(), reason="checks the behaviour of a box WITHOUT a GPU")
def test_product_path_fails_without_a_gpu_instead_of_falling_back():
    L = lz.lib()
    assert L.LizardB200_available() == 0
    src = b"abcdefgh" * 4096
    dst = ctypes.create_string_buffer(len(src) + 64)
    # drop-in symbols: the reference's own failure values (0 = compression failed, negative = decode error)
    assert L.Lizard_compress(src, dst, len(src), len(dst), 10) == 0
    assert L.Lizard_decompress_safe(b"\x0a\x80\x01\x00\x00a", dst, 6, 64) < 0
    # batch API: negative status and a message
    with pytest.raises(lz.LizardB200Error):
        lz.compress_batch([src], 10)
    with pytest.raises(lz.LizardB200Error):
        lz.decompress_batch([b"\x0a\x80\x01\x00\x00a"], [64])
    assert L.LizardB200_lastError()


def build_c_host(tmp_path, name="frame_roundtrip"):
    """Compile examples/<name>.c as strict C99 against include/lizard_b200.h and link it to the library."""
    import subprocess
    exe = os.path.join(str(tmp_path), name)
    cmd = ["gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-O2", "-I" + os.path.join(ROOT, "include"),
           os.path.join(ROOT, "examples", name + ".c"), os.path.join(ROOT, "tools", "datagen.c"),
           "-L" + os.path.join(ROOT, "lizard_b200"), "-llizard_b200", "-Wl,-rpath," + os.path.join(ROOT, "lizard_b200"),
           "-lm", "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_c_host_compiles_as_c99_and_fails_loudly_without_a_gpu(tmp_path):
    """The north_star keeps the host side in C: the header must be valid C (not only C++), and a C program written like
    the reference's own callers links against the library with nothing but that header."""
    import subprocess
    lz.lib()                                              # built
    exe = build_c_host(tmp_path)
    bench = build_c_host(tmp_path, "block_bench")
    build_c_host(tmp_path, "lizard_file")
    if _no_gpu():
        r = subprocess.run([exe, "1", "10"], capture_output=True, text=True, timeout=120)
        assert r.returncode == 1 and "LizardF_compressFrame" in r.stderr, (r.returncode, r.stderr)
        r = subprocess.run([bench, "10", "1", "1"], capture_output=True, text=True, timeout=120)
        assert r.returncode == 1 and "LizardB200_compress_blocks" in r.stderr, (r.returncode, r.stderr)


def test_reference_frame_layer_relinks_against_the_library(tmp_path):
    """INTEGRATION.md section 1: the reference's unmodified lizard_frame.c links against the library (every symbol of
    lib/dll/liblizard.def it references is exported) and runs.  Without a GPU our block codec reports failure (0), which
    the reference's frame layer answers by storing every block raw (lizard_frame.c:462-466): a valid frame that the pure
    reference decodes -- still no CPU codec behind the drop-in symbols."""
    import subprocess
    exe = os.path.join(refs.REF_DIR, "relinked_frame")
    ref = refs.ref_parity()
    if ref is None or not os.path.exists(exe):
        pytest.skip("oracle/_ref not built")
    out = os.path.join(str(tmp_path), "f.liz")
    r = subprocess.run([exe, "10", "1", out, "1"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    frame = open(out, "rb").read()
    lz.bind_frame_api(ref)
    res, back = lz.frame_decompress(ref, frame, 1 << 20)
    assert res == 0 and back == lz.datagen(1 << 20)
    if _no_gpu():
        assert "8 blocks, 8 stored raw" in r.stdout, r.stdout


def test_encoder_launch_shapes_are_the_measured_ones():
    """The per-level launch shapes were picked from sweeps on the B200 (profiles/r01_SUMMARY.md section 8); a refactoring of
    encode_shape() must not move them silently.  (warps per CTA, shared-memory tables per CTA, CTAs per SM)"""
    L = lz.lib()
    want = {10: (14, 3, 2), 30: (14, 3, 2), 11: (14, 0, 2), 31: (14, 0, 2), 21: (14, 2, 2), 22: (14, 0, 2), 41: (14, 0, 2), 20: (14, 2, 2), 40: (14, 0, 2),
            13: (14, 0, 2), 17: (14, 0, 2), 34: (14, 0, 2)}
    for level, shape in want.items():
        w, t, k, b = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        assert L.LizardB200_encodeShape(level, ctypes.byref(w), ctypes.byref(t), ctypes.byref(k), ctypes.byref(b)) == 0
        assert (w.value, t.value, k.value) == shape, (level, w.value, t.value, k.value)
        assert 2 * (b.value + 1024) <= 196 * 1024          # two CTAs inside the 196 KB carve-out step
    assert L.LizardB200_encodeShape(12, None, None, None, None) < 0


def test_pipeline_chunk_plan_host_and_kernel_arithmetic_agree():
    """The host-buffer calls cut their units into pipeline chunks (frame.inl: FrameChunks; the decoder's calls start with a
    doubling ramp of small chunks); the kernels find a unit's chunk with their own arithmetic (decode.cuh: progress_chunk).
    Every unit of a range of shapes must get the same chunk, first unit and size from both, and the chunks must tile the
    units exactly."""
    L = lz.lib()
    L.LizardB200_chunkPlan.argtypes = [ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_uint] + [ctypes.POINTER(ctypes.c_uint)] * 3
    for n, per, ramp in [(8192, 512, 1), (8192, 512, 0), (1025, 512, 1), (1024, 512, 1), (1023, 512, 1), (100, 512, 1), (5000, 48, 1),
                         (5000, 40, 1), (1, 512, 1), (33, 16, 1), (7, 1, 1), (4097, 2048, 1)]:
        c, f, k = ctypes.c_uint(), ctypes.c_uint(), ctypes.c_uint()
        seen = {}
        nch = None
        for u in range(n):
            r = L.LizardB200_chunkPlan(n, per, ramp, u, ctypes.byref(c), ctypes.byref(f), ctypes.byref(k))
            assert r > 0, (n, per, ramp, u, r)
            nch = r
            seen.setdefault(c.value, (f.value, k.value))
            assert seen[c.value] == (f.value, k.value)
        assert sorted(seen) == list(range(nch)), (n, per, ramp, sorted(seen)[:8], nch)
        pos = 0
        for ci in range(nch):
            assert seen[ci][0] == pos and seen[ci][1] >= 1
            pos += seen[ci][1]
        assert pos == n
        if ramp and per % 16 == 0 and n >= 2 * per:
            assert seen[0][1] == per // 16 and seen[4][1] == per          # 1/16, 1/8, 1/4, 1/2, then full chunks
