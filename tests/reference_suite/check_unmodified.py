#!/usr/bin/env python
"""Check that the vendored reference tests are the reference's files byte for byte: their SHA-256
against tests/golden/reference_suite_sha256.json and, given the root of an oxli checkout as the
argument, against that checkout's src/python/tests too (exit 0 if all match)."""
import filecmp
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
MINE = os.path.join(HERE, "src", "python", "tests")
DIGESTS = os.path.join(os.path.dirname(HERE), "golden", "reference_suite_sha256.json")


def main(ref_root: str | None = None) -> int:
    want = json.load(open(DIGESTS))["files"]
    mine = sorted(f for f in os.listdir(MINE) if f.endswith(".py"))
    bad = [n for n in want if n not in mine or hashlib.sha256(open(os.path.join(MINE, n), "rb").read()).hexdigest() != want[n]]
    bad += [n for n in mine if n not in want]
    if ref_root:
        ref = os.path.join(ref_root, "src", "python", "tests")
        names = sorted(f for f in os.listdir(ref) if f.endswith(".py"))
        bad += [n for n in names if n not in mine or not filecmp.cmp(os.path.join(ref, n), os.path.join(MINE, n), shallow=False)]
        bad += [n for n in mine if n not in names]
    bad = sorted(set(bad))
    print(f"{len(want)} reference test files, {len(bad)} differing: {bad}")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1] if len(sys.argv) > 1 else None))
