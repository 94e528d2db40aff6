"""Pins oracle/myers_oracle.cpp (the plain-DP restatement of what racon asks of edlib, SURVEY.md §8 a10) against
the UNMODIFIED edlib compiled into oracle/_ref: identical CIGAR strings and edit distances on random pairs in both
of edlib's regimes (stored-matrix traceback below 1 MiB of alignment data, Hirschberg above).  What edlib returned for
these seeded pairs is stored in tests/golden/ref_outputs.npz (tests/golden/make_ref_outputs.py), so this runs everywhere."""
import os
import zlib

import numpy as np
import pytest

from oracle import bindings as ob
from tests import util

REF_OUTPUTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_outputs.npz")
TRACEBACK = [(1, 0.5, 20), (7, 0.3, 60), (64, 0.2, 60), (65, 0.1, 40), (300, 0.15, 40), (1500, 0.12, 12), (1900, 0.25, 8)]
HIRSCHBERG = [(2500, 0.12, 6), (4000, 0.05, 4), (6000, 0.15, 3), (3000, 0.35, 4)]
DEGENERATE = [(b"A", b"A"), (b"A", b"C"), (b"ACGT", b"A"), (b"A", b"ACGT"), (b"AAAA", b"TTTT"), (b"ACGTACGT", b"ACGT"),
              (b"ACGT" * 700, b"ACGT" * 100), (b"A" * 3000, b"A" * 2990 + b"C" * 500)]


def _pair(rng, n, err, skew=0.0):
    t = bytes(util.BASES[i] for i in rng.integers(4, size=n))
    q = util.mutate(rng, t, err)
    if skew:  # drop a prefix/suffix of the query so the lengths differ markedly
        k = int(len(q) * skew)
        q = q[k // 2:len(q) - k // 2]
    return q, t


def traceback_pairs(n, err, count):
    rng = np.random.default_rng(n)
    pairs = [_pair(rng, n, err, skew=rng.choice([0.0, 0.0, 0.2])) for _ in range(count)]
    return [(q, t) for q, t in pairs if q]


def hirschberg_pairs(n, err, count):
    rng = np.random.default_rng(n + 1)
    return [_pair(rng, n, err, skew=rng.choice([0.0, 0.1, 0.3])) for _ in range(count)]


def edlib_key(test, params):
    return "edlib/%s/%s" % (test, "_".join(str(p) for p in params))


def _assert_equals_edlib(key, pairs):
    """Per pair (CRC-32 of the CIGAR string, edit distance) against what edlib returned."""
    ref = np.load(REF_OUTPUTS)[key]
    assert len(ref) == len(pairs)
    for k, (q, t) in enumerate(pairs):
        cigar, dist = ob.oracle_myers_cigar(q, t)
        assert (zlib.crc32(cigar.encode()), dist) == tuple(int(v) for v in ref[k]), (k, len(q), len(t))


@pytest.mark.parametrize("n,err,count", TRACEBACK)
def test_traceback_regime(n, err, count):
    _assert_equals_edlib(edlib_key("traceback", (n, err, count)), traceback_pairs(n, err, count))


@pytest.mark.parametrize("n,err,count", HIRSCHBERG)
def test_hirschberg_regime(n, err, count):
    _assert_equals_edlib(edlib_key("hirschberg", (n, err, count)), hirschberg_pairs(n, err, count))


def test_degenerate_pairs():
    _assert_equals_edlib(edlib_key("degenerate", ()), DEGENERATE)
