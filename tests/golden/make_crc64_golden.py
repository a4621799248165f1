"""Regenerates tests/golden/crc64_reference.json: crc64 of seeded random buffers (lengths around the 8- and 16-byte
strides of table-driven implementations) under two initial values, as computed by the reference's own
src/utils/crc.cpp.  `make -C oracle` compiles that file into oracle/_ref/ when the reference tree is present; the JSON is
committed so that the test needs neither.  Run from the repo root after the build:
    python tests/golden/make_crc64_golden.py"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import oracle_py  # noqa: E402

LENGTHS = [0, 1, 2, 7, 15, 16, 17, 31, 64, 1000, 4097]
INITS = [0, 0x1234567890ABCDEF]

if __name__ == "__main__":
    ref = oracle_py.ref_crc()
    if ref is None:
        sys.exit("oracle/_ref/libref_crc.so is missing: build with the reference tree present (make -C oracle)")
    rng = np.random.default_rng(1)
    rows = []
    for n in LENGTHS:
        b = bytes(rng.integers(0, 256, n, dtype=np.uint8))
        for init in INITS:
            rows.append({"data": b.hex(), "init": "0x%016x" % init, "crc64": "0x%016x" % ref.ref_crc64(b, n, init)})
    with open(os.path.join(ROOT, "tests", "golden", "crc64_reference.json"), "w") as f:
        json.dump({"source": "reference src/utils/crc.cpp (dsn::utils::crc64_calc) through oracle/ref_crc_shim.cpp",
                   "rows": rows}, f, indent=1)
        f.write("\n")
    print(len(rows), "rows")
