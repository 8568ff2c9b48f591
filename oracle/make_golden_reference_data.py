#!/usr/bin/env python
"""TEST INFRASTRUCTURE ONLY -- data taken from the reference tree for the tests that check against it:
  tests/golden/latency_lookup_table.json   the shipped latency lookup table (train/latency_lookup_table.npy, identical in
                                           search/ and latency/): operator key -> measured latency in ms
  tests/golden/reference_line_counts.json  the line count of every reference .py file, so that the `dir/file.py:LINE` citations
                                           in our sources can be checked (tools/check_citations.py)
Run where the reference tree is available:  python oracle/make_golden_reference_data.py"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from oracle import ref_harness  # noqa: E402
import check_citations  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def main():
    if not ref_harness.reference_available():
        raise SystemExit("reference tree not present at %s" % ref_harness.REFERENCE_ROOT)
    table = np.load(os.path.join(ref_harness.REFERENCE_ROOT, "train", "latency_lookup_table.npy"), allow_pickle=True).item()
    with open(os.path.join(GOLDEN, "latency_lookup_table.json"), "w") as f:
        json.dump({k: float(v) for k, v in sorted(table.items())}, f, indent=0)
    with open(os.path.join(GOLDEN, "reference_line_counts.json"), "w") as f:
        json.dump(check_citations.line_counts(ref_harness.REFERENCE_ROOT), f, indent=0, sort_keys=True)
    print("wrote latency_lookup_table.json (%d keys) and reference_line_counts.json" % len(table))


if __name__ == "__main__":
    main()
