"""Test-only access to the checkers: the reference's recorded answers (tests/golden/reference_calls.bin), the compiled
reference itself (oracle/_ref, built only where the reference's sources are present) and our C restatement
(oracle/liboracle.so).

The tests compare against `reference()`, which answers every call from the recorded file, so the suite needs nothing
outside the repository.  Each entry holds the result code and a 32-bit SHA-256 prefix of the output of one call of the
unmodified reference (-DLIZARD_RESET_MEM build), keyed by a hash of the call's arguments.  Where a test needs the
reference's output bytes themselves (to feed them to a decoder), they are produced by our own implementation (the oracle
for blocks and Huffman streams, the library for frames) and checked against the recorded digest first.

To add or refresh entries, build oracle/_ref and run the suite with LIZARD_RECORD_REFERENCE=<file> (the GPU tests on a
B200): every call is then answered by the compiled reference and merged into <file>."""
import atexit
import ctypes
import hashlib
import os
import struct

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
CALLS = os.path.join(ROOT, "tests", "golden", "reference_calls.bin")
_ENTRY = struct.Struct("<QiI")          # key, result, digest of the output


def _bind(L):
    L.Lizard_compressBound.argtypes = [ctypes.c_int]
    L.Lizard_sizeofState.argtypes = [ctypes.c_int]
    L.Lizard_compress.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    L.Lizard_decompress_safe.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_int]
    return L


def ref_parity():
    """Reference compiled with -DLIZARD_RESET_MEM: the bit-exact target for compression."""
    p = os.path.join(REF_DIR, "liblizard_ref_parity.so")
    return _bind(ctypes.CDLL(p)) if os.path.exists(p) else None


def ref_speed():
    p = os.path.join(REF_DIR, "liblizard_ref_speed.so")
    return _bind(ctypes.CDLL(p)) if os.path.exists(p) else None


def ref_compress(L, data: bytes, level: int, cap: int = None) -> bytes:
    cap = L.Lizard_compressBound(len(data)) if cap is None else cap
    dst = ctypes.create_string_buffer(max(cap, 1))
    n = L.Lizard_compress(data, dst, len(data), cap, level)
    return dst.raw[:n]


def ref_decompress(L, comp: bytes, cap: int):
    # twice the capacity: the reference does not charge a raw inner block against maxDecompressedSize
    # (lib/lizard_decompress.c:164-180 never reduces outputSize), so a compressed inner block behind a raw one may write up
    # to the raw block's size past the capacity (DESIGN.md 3.5); a result > cap tells the caller that this happened
    dst = ctypes.create_string_buffer(2 * max(cap, 1) + 64)
    r = L.Lizard_decompress_safe(comp, dst, len(comp), cap)
    return r, (dst.raw[:r] if r > 0 else b"")


def digest(b: bytes) -> int:
    return int.from_bytes(hashlib.sha256(b).digest()[:4], "little")


class Digest:
    """Stands for output bytes of the reference that were recorded as a digest: equal to bytes with the same digest."""

    def __init__(self, d):
        self.d = d

    def __eq__(self, other):
        if isinstance(other, Digest):
            return self.d == other.d
        return isinstance(other, (bytes, bytearray)) and digest(bytes(other)) == self.d

    def __hash__(self):
        return self.d

    def __repr__(self):
        return "Digest(%08x)" % self.d


def _key(name, ints, blob=b""):
    h = hashlib.sha256(("%s|%s|" % (name, ",".join(str(int(i)) for i in ints))).encode())
    h.update(blob)
    return int.from_bytes(h.digest()[:8], "little")


def _load(path):
    table = {}
    if os.path.exists(path):
        with open(path, "rb") as f:
            for k, r, d in _ENTRY.iter_unpack(f.read()):
                table[k] = (r, d)
    return table


def _store(path, new):
    table = _load(path)
    table.update(new)
    with open(path, "wb") as f:
        for k in sorted(table):
            f.write(_ENTRY.pack(k, *table[k]))


class Reference:
    """The unmodified reference's answers: recorded (default) or live from oracle/_ref while recording."""

    def __init__(self):
        self.record_path = os.environ.get("LIZARD_RECORD_REFERENCE")
        if self.record_path:
            self.live = ref_parity()
            self.live_speed = ref_speed()
            assert self.live is not None and self.live_speed is not None, "recording needs oracle/_ref"
            self.new = {}
            atexit.register(lambda: _store(self.record_path, self.new))
        else:
            self.table = _load(CALLS)

    def _answer(self, name, ints, blob, live):
        k = _key(name, ints, blob)
        if self.record_path:
            res, out = live()
            self.new[k] = (max(min(res, 2 ** 31 - 1), -2 ** 31), digest(out))
            return res, out
        if k not in self.table:
            raise LookupError("no recorded answer of the reference for %s%s (%d input bytes): record it, see tests/refs.py"
                              % (name, tuple(ints), len(blob)))
        return self.table[k]

    @staticmethod
    def _checked(name, got, res, dig):
        assert len(got) == res and digest(got) == dig, \
            "%s: our output (%d bytes) differs from the reference's recorded one (%d bytes)" % (name, len(got), res)
        return got

    # ---- block format -------------------------------------------------------------------------------------------------
    def Lizard_compressBound(self, n):
        return self._answer("compressBound", (n,), b"", lambda: (self.live.Lizard_compressBound(n), b""))[0]

    def Lizard_sizeofState(self, level):
        return self._answer("sizeofState", (level,), b"", lambda: (self.live.Lizard_sizeofState(level), b""))[0]

    def compress(self, data: bytes, level: int, cap: int = None) -> bytes:
        """Lizard_compress(data, cap (default: compressBound), level): the reference's bytes."""
        cap = self.Lizard_compressBound(len(data)) if cap is None else cap

        def live():
            out = ref_compress(self.live, data, level, cap)
            assert _oracle_compress(data, level, cap) == out, "oracle/liboracle.so differs from the reference"
            return len(out), out
        r = self._answer("compress", (level, cap), data, live)
        if self.record_path:
            return r[1]
        return self._checked("compress", _oracle_compress(data, level, cap), *r)

    def decompress(self, comp: bytes, cap: int):
        """Lizard_decompress_safe(comp, cap): (return code, bytes or their Digest)."""
        def live():
            r, out = ref_decompress(self.live, comp, cap)
            return r, out
        r, d = self._answer("decompress", (cap,), comp, live)
        if self.record_path:
            return r, d
        return r, (Digest(d) if r > 0 else b"")

    # ---- Huffman stage (entropy/huf_*.c) -----------------------------------------------------------------------------
    def huf_compress(self, data: bytes, cap: int):
        """HUF_compress(cap): None when the reference reports an error, else its output bytes."""
        def live():
            L = self.live_speed
            _bind_huf(L)
            a = ctypes.create_string_buffer(cap + 16)
            ca = L.HUF_compress(a, cap, data, len(data))
            if L.HUF_isError(ca):
                return -1, b""
            out = a.raw[:ca]
            assert _oracle_huf_compress(data, cap) == out, "oracle/liboracle.so differs from the reference"
            return ca, out
        r = self._answer("huf_compress", (cap,), data, live)
        if self.record_path:
            return None if r[0] < 0 else r[1]
        if r[0] < 0:
            return None
        return self._checked("huf_compress", _oracle_huf_compress(data, cap), *r)

    def huf_decompress(self, comp: bytes, n: int):
        """HUF_decompress into n bytes: (-1 on error else the result, the n output bytes or their Digest)."""
        def live():
            L = self.live_speed
            _bind_huf(L)
            d = ctypes.create_string_buffer(n + 16)
            r = L.HUF_decompress(d, n, comp, len(comp))
            return (-1, b"") if L.HUF_isError(r) else (r, d.raw[:n])
        r, d = self._answer("huf_decompress", (n,), comp, live)
        if self.record_path:
            return r, d
        return r, (Digest(d) if r >= 0 else b"")

    # ---- frame format (lizard_frame.c) -------------------------------------------------------------------------------
    def frame_compress(self, data: bytes, prefs) -> bytes:
        """LizardF_compressFrame: the reference's frame (produced by the library and checked against the record)."""
        import lizard_b200 as lz
        fi = prefs.frameInfo
        ints = (prefs.compressionLevel, fi.blockSizeID, fi.blockMode, fi.contentChecksumFlag, fi.contentSize)

        def live():
            out = lz.frame_compress(lz.bind_frame_api(self.live), data, prefs)
            return len(out), out
        r = self._answer("frame_compress", ints, data, live)
        if self.record_path:
            return r[1]
        return self._checked("frame_compress", lz.frame_compress(lz.bind_frame_api(lz.lib()), data, prefs), *r)

    def frame_decompress(self, frame: bytes, cap: int):
        """LizardF_decompress of a whole frame: (-1 on error else the last result, the output or on error the error
        name, as bytes or their Digest)."""
        import lizard_b200 as lz

        def live():
            L = lz.bind_frame_api(self.live)
            r, out = lz.frame_decompress(L, frame, cap)
            return (-1, L.LizardF_getErrorName(r)) if L.LizardF_isError(r) else (r, out)
        r, d = self._answer("frame_decompress", (cap,), frame, live)
        if self.record_path:
            return r, d
        return r, Digest(d)


_REFERENCE = None


def reference():
    global _REFERENCE
    if _REFERENCE is None:
        _REFERENCE = Reference()
    return _REFERENCE


def _bind_huf(L):
    L.HUF_compress.restype = ctypes.c_size_t
    L.HUF_compress.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t]
    L.HUF_decompress.restype = ctypes.c_size_t
    L.HUF_decompress.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t]
    L.HUF_isError.argtypes = [ctypes.c_size_t]


def _oracle_compress(data, level, cap):
    dst = ctypes.create_string_buffer(max(cap, 1) + 64)
    n = oracle().oracle_Lizard_compress(data, dst, len(data), cap, level)
    return dst.raw[:n]


def _oracle_huf_compress(data, cap):
    b = ctypes.create_string_buffer(cap + 16)
    n = oracle().oracle_HUF_compress(b, cap, data, len(data))
    return b.raw[:n]


_ORACLE = None


def oracle():
    """Our plain-C restatement (oracle/liboracle.so); None if not built."""
    global _ORACLE
    p = os.path.join(ROOT, "oracle", "liboracle.so")
    if _ORACLE is None and os.path.exists(p):
        L = ctypes.CDLL(p)
        L.oracle_Lizard_compress.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
        L.oracle_Lizard_decompress_safe.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_int]
        L.oracle_last_min_offset.restype = ctypes.c_uint
        L.oracle_HUF_compress.restype = ctypes.c_size_t
        L.oracle_HUF_compress.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t]
        _ORACLE = L
    return _ORACLE


def stream_obeys_min_offset(comp: bytes, cap: int) -> bool:
    """True when every match of a (successfully decoded) stream has offset >= 8, the rule all Lizard parsers
    enforce (LIZARD_*_MIN_OFFSET).  Below that the reference's 8-byte granule copies make ITS output depend on
    stale bytes beyond the write cursor, so byte parity is only defined for streams that obey the rule."""
    L = oracle()
    dst = ctypes.create_string_buffer(max(cap, 1) + 64)
    r = L.oracle_Lizard_decompress_safe(comp, dst, len(comp), cap)
    return r > 0 and L.oracle_last_min_offset() >= 8
