"""Regenerates tests/golden/frames.npz from libzstd (oracle/ref.py).  The committed file was made by the reference's
vendored libzstd 1.5.6; tests/test_oracle.py checks that the libzstd in use still writes the same bytes.

    python tools/make_golden.py
Each entry: name -> compressed frame; `<name>.raw` -> expected bytes.  Small on purpose (a few KB each).
sample_dict.raw is the reference's inst/sample_dict.raw (binary fixture used by R/dictionaries.R:20-24).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref  # noqa: E402
from zstdlite_b200 import corpus  # noqa: E402

out = {}
sd = open(os.path.join(ROOT, "tests", "golden", "sample_dict.raw"), "rb").read()
for fam in ("text", "rdf", "lowent", "rand", "rle"):
    for size in (0, 1, 300, 5000, 20000):
        d = corpus.make(fam, size, 21).tobytes()
        for lvl in (1, 3, 9):
            for ck in (0, 1):
                name = f"{fam}_{size}_l{lvl}_c{ck}"
                out[name] = np.frombuffer(ref.compress(d, lvl, bool(ck)), dtype=np.uint8)
        out[f"{fam}_{size}.raw"] = np.frombuffer(d, dtype=np.uint8)
    d = corpus.make(fam, 3000, 22).tobytes()
    out[f"{fam}_dict"] = np.frombuffer(ref.compress(d, 3, True, dict=sd), dtype=np.uint8)
    out[f"{fam}_dict.raw"] = np.frombuffer(d, dtype=np.uint8)
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "frames.npz"), **out)
print(len(out), "entries")
