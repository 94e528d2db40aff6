"""What the UNMODIFIED reference (oracle/_ref/libracon_ref.so: spoa through Window::generate_consensus, and edlib) returns
for the seeded inputs of tests/test_oracle.py and tests/test_myers_oracle.py, stored as CRC-32s so that those tests compare
the restated oracle with the reference without needing the reference itself:
  poa/<case>/<m>_<x>_<g>  per window: CRC-32 of the consensus, its length, the polished flag
  poa_no_trim             the same for test_oracle_equals_reference_no_trim_and_tiny
  edlib/<test>/<params>   per pair: CRC-32 of the CIGAR string, the edit distance
Stored in tests/golden/ref_outputs.npz.  Run where the reference is built:  python tests/golden/make_ref_outputs.py"""
import os
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import bindings as ob  # noqa: E402
from tests import test_myers_oracle as tm, test_oracle as to  # noqa: E402


def poa_rows(cons, pol):
    return np.asarray([[zlib.crc32(c), len(c), int(p)] for c, p in zip(cons, pol)], np.uint32).reshape(-1, 3)


def cigar_rows(pairs):
    rows = []
    for q, t in pairs:
        cigar, dist = ob.ref_edlib_cigar(q, t)
        rows.append([zlib.crc32(cigar.encode()), dist])
    return np.asarray(rows, np.uint32).reshape(-1, 2)


def main():
    assert ob.have_ref(), "oracle/_ref/libracon_ref.so is not built"
    out = {}
    for name in sorted(to.CASES):
        for scores in to.SCORES:
            ws, wl = to.case_windows(name, scores)
            ref, pol, _ = ob.ref_consensus(ws, *scores, window_length=wl, threads=8)
            out[to.poa_key(name, scores)] = poa_rows(ref, pol)
    ref, pol, _ = ob.ref_consensus(to._mk("partial", seed=7), trim=False, threads=4)
    out["poa_no_trim"] = poa_rows(ref, pol)
    for test, params in (("traceback", tm.TRACEBACK), ("hirschberg", tm.HIRSCHBERG)):
        for p in params:
            out[tm.edlib_key(test, p)] = cigar_rows(getattr(tm, test + "_pairs")(*p))
    out[tm.edlib_key("degenerate", ())] = cigar_rows(tm.DEGENERATE)
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_outputs.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
