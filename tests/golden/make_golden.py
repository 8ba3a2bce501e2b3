"""Generate tests/golden/golden.json and tests/golden/optimal_parser_streams.npz from the UNMODIFIED reference compiled
at oracle/_ref (`make -C oracle ref REF=<reference checkout>`, -DLIZARD_RESET_MEM build):
    python tests/golden/make_golden.py
The fixtures let any machine check the oracle and the CUDA path against reference outputs without the reference
being present.  The recorded answers of tests/golden/reference_calls.bin are made by the suite itself (tests/refs.py)."""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import lizard_b200 as lz  # noqa: E402
from tests import refs  # noqa: E402

BS = 1 << 17
ref = refs.ref_parity()
assert ref is not None, "build oracle/_ref first"


def make_input(spec):
    if spec["kind"] == "datagen":
        return lz.datagen(spec["size"], spec["pct"], spec["seed"])
    if spec["kind"] == "zeros":
        return bytes(spec["size"])
    return (b"abcdefgh" * (spec["size"] // 8 + 1))[: spec["size"]]


out = {"generator": "oracle/_ref/liblizard_ref_parity.so (inikep/lizard af8518cc, gcc -O3 -DLIZARD_RESET_MEM)",
       "datagen_md5": [], "compress": [], "vectors": []}
for size, pct, seed in ((4 << 20, 50, 0), (1 << 20, 50, 0), (100000, 90, 3), (1000, 10, 7)):
    out["datagen_md5"].append({"size": size, "pct": pct, "seed": seed,
                               "md5": hashlib.md5(lz.datagen(size, pct, seed)).hexdigest()})

inputs = [{"kind": "datagen", "size": 4 << 20, "pct": 50, "seed": 0},
          {"kind": "datagen", "size": 300000, "pct": 80, "seed": 5},
          {"kind": "zeros", "size": BS},
          {"kind": "pattern", "size": 70001}]
for spec in inputs:
    data = make_input(spec)
    for level in (10, 11, 13, 16, 21, 22, 30, 31, 34, 41, 42):
        c = refs.ref_compress(ref, data, level)
        out["compress"].append({"input": spec, "level": level, "mode": "single", "size": len(c),
                                "sha256": hashlib.sha256(c).hexdigest()})
        parts = [refs.ref_compress(ref, data[i:i + BS], level, BS - 1) for i in range(0, len(data), BS)]
        cc = b"".join(parts)
        out["compress"].append({"input": spec, "level": level, "mode": "blocks", "cap": BS - 1, "size": len(cc),
                                "sha256": hashlib.sha256(cc).hexdigest()})

# small compressed vectors incl. every level family and a few damaged streams with the reference's verdict
small = [("dg2000_p50", lz.datagen(2000, 50, 1)), ("dg5000_p90", lz.datagen(5000, 90, 2)), ("zeros3000", bytes(3000)),
         ("pattern1500", (b"abcdefgh" * 200)[:1500]), ("tiny20", bytes(range(20))), ("empty", b"")]
for name, data in small:
    for level in (10, 17, 21, 24, 30, 41, 45):
        c = refs.ref_compress(ref, data, level)
        for tag, comp, cap in (("ok", c, len(data)), ("short_dst", c, max(len(data) - 1, 0)),
                               ("truncated", c[: max(len(c) - 3, 0)], len(data)),
                               ("flip", bytes(b ^ (0x10 if i == len(c) // 2 else 0) for i, b in enumerate(c)), len(data))):
            r, o = refs.ref_decompress(ref, comp, cap)
            out["vectors"].append({"name": "%s_L%d_%s" % (name, level, tag), "compressed_hex": comp.hex(), "cap": cap,
                                   "result": r, "sha256": hashlib.sha256(o).hexdigest() if r > 0 else None})

with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden.json"), "w") as f:
    json.dump(out, f, indent=0)
print("wrote golden.json:", len(out["compress"]), "compress facts,", len(out["vectors"]), "vectors")

# streams of the lowest-price (24) and optimal (45) parsers, which the oracle does not restate: decoder inputs for
# test_*::*stored_optimal_parser_streams, named L<level>_n<size>_p<match pct>_s<seed> after their datagen input
streams = {}
for level in (24, 45):
    for size, pct, seed in ((BS, 90, 1), (BS + 3000, 90, 3), (40000, 50, 4)):
        c = refs.ref_compress(ref, lz.datagen(size, pct, seed), level)
        streams["L%d_n%d_p%d_s%d" % (level, size, pct, seed)] = np.frombuffer(c, dtype=np.uint8)
np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "optimal_parser_streams.npz"), **streams)
print("wrote optimal_parser_streams.npz:", sum(len(v) for v in streams.values()), "bytes of streams")
