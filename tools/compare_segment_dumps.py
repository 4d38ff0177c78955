"""Compare two segment dumps of bench.py --dump-outputs (two builds, same seeded inputs).

    python tools/compare_segment_dumps.py DIR_A DIR_B [--prefix rank0_] [--show 20]

A record is keyed by (hapA, hapB, posStart, posEnd, level).  Prints one JSON line: the record count of each dump, the
records found in one dump only, and, over the records found in both, the largest relative difference of prob, postMean
and mapTime (and of mapState as an exact count).  Records found in one dump only are grouped by pair and listed: in the
fast mode they are expected only where a site's IBD posterior lies within the mode's tolerance of a level threshold, which
moves a segment boundary or splits a segment.  Exit code 0 when the keyed records match and every score is within --rtol.
"""
import argparse
import collections
import json
import os
import sys

import numpy as np

FIELDS = ("hapA", "hapB", "posStart", "posEnd", "mapState", "level", "prob", "postMean", "mapTime")
KEY = ("hapA", "hapB", "posStart", "posEnd", "level")


def load(directory, prefix):
    return {f: np.load(os.path.join(directory, f"{prefix}segment_{f}.npy")) for f in FIELDS}


def index(d):
    keys = list(zip(*(d[f].astype(np.int64).tolist() for f in KEY)))
    out = {}
    for i, k in enumerate(keys):
        out.setdefault(k, i)
    return out, len(keys) - len(set(keys))


def rel(a, b):
    a = a.astype(np.float64)
    b = b.astype(np.float64)
    den = np.maximum(np.abs(a), np.abs(b))
    with np.errstate(invalid="ignore", divide="ignore"):
        r = np.where(den > 0, np.abs(a - b) / den, 0.0)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("a")
    ap.add_argument("b")
    ap.add_argument("--prefix", default="")
    ap.add_argument("--rtol", type=float, default=1e-4)
    ap.add_argument("--show", type=int, default=20, help="pairs with unmatched records to list")
    args = ap.parse_args()
    A, B = load(args.a, args.prefix), load(args.b, args.prefix)
    ia, dupA = index(A)
    ib, dupB = index(B)
    common = [k for k in ia if k in ib]
    onlyA = [k for k in ia if k not in ib]
    onlyB = [k for k in ib if k not in ia]
    sa = np.array([ia[k] for k in common], dtype=np.int64)
    sb = np.array([ib[k] for k in common], dtype=np.int64)
    result = {"records_a": int(len(A["hapA"])), "records_b": int(len(B["hapA"])), "duplicate_keys": [dupA, dupB],
              "matched": len(common), "only_a": len(onlyA), "only_b": len(onlyB)}
    ok = not onlyA and not onlyB
    for f in ("prob", "postMean", "mapTime"):
        r = rel(A[f][sa], B[f][sb]) if len(common) else np.zeros(1)
        result[f"max_rel_{f}"] = float(r.max())
        ok = ok and float(r.max()) <= args.rtol
    result["mapState_differs"] = int(np.count_nonzero(A["mapState"][sa] != B["mapState"][sb])) if len(common) else 0
    byPair = collections.defaultdict(lambda: ([], []))
    for k in onlyA:
        byPair[k[:2]][0].append(k[2:])
    for k in onlyB:
        byPair[k[:2]][1].append(k[2:])
    result["pairs_with_unmatched"] = len(byPair)
    print(json.dumps(result), flush=True)
    for pair, (ra, rb) in list(byPair.items())[:args.show]:
        print(f"  pair {pair}: only in A (start, end, level) {sorted(ra)}; only in B {sorted(rb)}")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
