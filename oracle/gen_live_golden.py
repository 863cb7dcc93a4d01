"""TEST INFRASTRUCTURE ONLY -- write tests/golden/inference_live.npz: this package's record of the seeded random cases of
oracle/inference_cases.py (14 rendering scenarios, 16 messenger settings, tokenizer decodes on random metres).

    python oracle/gen_live_golden.py

The tests that compare these cases with the original project live (tests/test_inference_host.py, `*_live`) found this package
identical to it, bit for bit, when its inference code last changed; the record pins that state so the comparison holds without a
copy of the original.  Regenerate only for a change that those live tests, run against the original, accept.
"""
from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests.test_inference_host import GOLDEN, live_records  # noqa: E402

if __name__ == "__main__":
    out = {f"{part}/{k}": v for part, rec in live_records(native=True).items() for k, v in rec.items()}
    path = os.path.join(GOLDEN, "inference_live.npz")
    np.savez_compressed(path, **out)
    print(path, len(out), "arrays,", os.path.getsize(path), "bytes")
