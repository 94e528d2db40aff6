"""Pins the restated oracle (oracle/poa_oracle.cpp).

(a) known-answer checksums of the reference (SURVEY.md §8d) — run everywhere;
(b) window-by-window equality with the unmodified reference (oracle/_ref, compiled by oracle/Makefile) on full-span,
    partial-span (Subgraph path), quality-weighted, NGS and non-default-score windows — against the reference's results
    for these seeded windows as stored in tests/golden/ref_outputs.npz (tests/golden/make_ref_outputs.py), so it runs
    everywhere;
(c) committed golden fixtures (tests/golden/, generated from oracle/_ref by tests/golden/make_golden.py).
"""
import json
import zlib
import os

import numpy as np
import pytest

from oracle import bindings as ob
from racon_b200 import windows
from tests import util

KAT = [(0.12, 200, "50f18d884e3254d2"), (0.06, 100, "f64dfc685e9591b6"), (0.15, 100, "3beef354919c0528")]


@pytest.mark.parametrize("err,n,expect", KAT)
def test_oracle_known_answer_checksums(err, n, expect):
    ws, _ = windows.synth_windows(n, err=err)
    cons, pol, _ = ob.oracle_consensus(ws, threads=8)
    assert "%016x" % windows.fnv1a64(cons) == expect
    assert pol.all()


needs_ref = pytest.mark.skipif(not ob.have_ref(), reason="oracle/_ref not built")


@needs_ref
@pytest.mark.parametrize("err,n,expect", KAT[:1])
def test_ref_known_answer_checksum(err, n, expect):
    ws, _ = windows.synth_windows(n, err=err)
    cons, pol, _ = ob.ref_consensus(ws, threads=8)
    assert "%016x" % windows.fnv1a64(cons) == expect


CASES = {
    "fullspan": dict(n=24, wlen=500, depth=32, err=0.12),
    "partial": dict(n=24, wlen=500, depth=30, err=0.10, partial_frac=0.5),
    "partial_qual": dict(n=24, wlen=500, depth=24, err=0.12, partial_frac=0.3, with_qual=True, backbone_qual=True),
    "ngs_short": dict(n=40, wlen=200, depth=40, err=0.01, partial_frac=0.9, with_qual=True, types=0),
    "acgtn": dict(n=16, wlen=300, depth=20, err=0.15, partial_frac=0.2, alphabet=b"ACGTN"),
    "shallow": dict(n=30, wlen=120, depth=3, err=0.2, partial_frac=0.3),
    "w1000": dict(n=6, wlen=1000, depth=20, err=0.12, partial_frac=0.2),
}


def _mk(name, seed):
    kw = dict(CASES[name])
    n = kw.pop("n")
    t = kw.pop("types", None)
    ws = util.make_set(seed, n, **kw)
    if t is not None:
        ws.win_type[:] = t
    return ws


SCORES = [(3, -5, -4), (5, -4, -8), (1, -1, -1)]
REF_OUTPUTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_outputs.npz")


def case_windows(name, scores):
    """The seeded windows of a (case, scores) pair and their window length."""
    return _mk(name, seed=zlib.crc32(name.encode()) % 1000 + scores[0]), 1000 if name == "w1000" else 500


def poa_key(name, scores):
    return "poa/%s/%d_%d_%d" % ((name,) + tuple(scores))


def _assert_equals_reference(key, cons, pol):
    """Per window (CRC-32 of the consensus, its length, polished) against what the reference returned."""
    ref = np.load(REF_OUTPUTS)[key]
    got = np.asarray([[zlib.crc32(c), len(c), int(p)] for c, p in zip(cons, pol)], np.uint32).reshape(-1, 3)
    assert got.shape == ref.shape
    assert (got[:, 2] == ref[:, 2]).all()
    bad = np.flatnonzero((got != ref).any(axis=1))
    assert not len(bad), "oracle != reference on windows %s" % bad[:5].tolist()


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("scores", SCORES)
def test_oracle_equals_reference(name, scores):
    ws, wl = case_windows(name, scores)
    ora, opol, _ = ob.oracle_consensus(ws, *scores, window_length=wl, threads=8)
    _assert_equals_reference(poa_key(name, scores), ora, opol)


def test_oracle_equals_reference_no_trim_and_tiny():
    ora, opol, _ = ob.oracle_consensus(_mk("partial", seed=7), trim=False, threads=4)
    _assert_equals_reference("poa_no_trim", ora, opol)
    # < 3 sequences: backbone copied, polished = False (window.cpp:68-71)
    tiny = windows.from_lists([[(b"ACGTACGT", None, 0, 0), (b"ACGTTCGT", None, 0, 7)], [(b"AC", None, 0, 0)]])
    ora, opol, _ = ob.oracle_consensus(tiny)
    assert ora == [b"ACGTACGT", b"AC"] and not opol.any()
    if ob.have_ref():
        ref, rpol, _ = ob.ref_consensus(tiny)
        assert ref == ora and not rpol.any()


def test_oracle_matches_golden_fixtures():
    path = os.path.join(os.path.dirname(__file__), "golden", "poa_golden.json")
    with open(path) as f:
        gold = json.load(f)
    assert gold["cases"], "empty golden file"
    for case in gold["cases"]:
        ws = windows.from_lists([[(s[0].encode(), s[1].encode() if s[1] else None, s[2], s[3]) for s in win]
                                 for win in case["windows"]], case["types"])
        m, x, g = case["scores"]
        ora, opol, _ = ob.oracle_consensus(ws, m, x, g, trim=case["trim"], threads=4)
        assert [c.decode() for c in ora] == case["consensus"], case["name"]
        assert [bool(p) for p in opol] == case["polished"], case["name"]
