"""Writes tests/golden/anchor_lists.json: what libcpecan.so's filterToRemoveOverlap and
convertPairwiseForwardStrandAlignmentToAnchorPairs return on the seeded inputs of tests/test_anchors.py and
tests/test_realign_host.py.  The reference build (oracle/_ref) could not be run when the fixture was recorded, so these are the
library's own outputs: they pin its current behaviour, and the live tests still compare it with the reference wherever
oracle/_ref is built.  Usage (after build()): python tools/make_anchor_golden.py"""
import json
import os
import sys

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)

import test_anchors as ta  # noqa: E402
import test_realign_host as tr  # noqa: E402


def main():
    ours, host = ta.Lists(ta.LIB), tr.Host()
    out = {"source": "libcpecan.so via tools/make_anchor_golden.py (the library's own outputs, not the reference's)",
           "filterToRemoveOverlap": [[list(p) for p in ta.filtered(ours, t)] for t in ta.overlap_cases()],
           "cigarAnchors": [tr.host_cigar_anchors(host, *c).tolist() for c in tr.cigar_cases()]}
    with open(ta.GOLDEN, "w") as f:
        json.dump(out, f)
    print("wrote", ta.GOLDEN, os.path.getsize(ta.GOLDEN), "bytes")


if __name__ == "__main__":
    main()
