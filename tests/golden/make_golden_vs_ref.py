#!/usr/bin/env python
"""Generate tests/golden/vs_ref.json and vs_ref.npz from the UNMODIFIED reference (oracle/_ref/ref_harness
and ref_harness_rawheap, built by `make -C oracle ref REF=<hacktv source tree>`).

Runs tests/test_oracle_vs_ref.py with its comparisons pointed at the reference binaries: every stream the
reference emits there is checked against the oracle, as the tests check it, and then stored as its sha256,
its size and an evenly spaced sample of its values (short streams whole).

    python tests/golden/make_golden_vs_ref.py
"""
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import orc  # noqa: E402
import test_oracle_vs_ref as T  # noqa: E402


def main():
    assert orc.have_ref(), "build the reference first: make -C oracle ref REF=<hacktv source tree>"
    T.RECORD = {}
    rc = pytest.main(["-q", "-p", "no:cacheprovider", T.__file__])
    assert rc == 0, "the oracle and the reference disagree: nothing written"
    with open(T.GOLD_JSON, "w") as f:
        json.dump({k: {"sha256": v["sha256"], "size": v["size"]} for k, v in sorted(T.RECORD.items())}, f, indent=1)
    np.savez_compressed(T.GOLD_NPZ, **{k: v["sample"] for k, v in sorted(T.RECORD.items())})
    print(len(T.RECORD), "reference streams")


if __name__ == "__main__":
    main()
