"""Input layer of the C++ host layer (racon_b200/csrc/reads_io.*; SURVEY §8 f4): FASTA / FASTQ / PAF / MHAP / SAM files ->
the state racon::Polisher::initialize holds before it looks for breaking points, against what the UNMODIFIED reference
held for the same files (tests/golden/sample/input_cases.npz, made by tests/golden/make_input_cases.py from
oracle/_ref/refpol_dump).
Host code only: runs without a GPU.  The files are a cut of the reference's lambda sample, tests/golden/sample/
(tests/golden/make_sample_data.py)."""
import gzip
import os
import zlib

import numpy as np
import pytest

from racon_b200 import api
from tests import util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DATA = os.path.join(ROOT, "tests", "golden", "sample")
GOLD = os.path.join(DATA, "input_cases.npz")

CASES = {
    "fastq_paf": ("sample_reads.fastq.gz", "sample_overlaps.paf.gz", "sample_layout.fasta.gz", False, 0.3),
    "fasta_paf": ("sample_reads.fasta.gz", "sample_overlaps.paf.gz", "sample_layout.fasta.gz", False, 0.3),
    "fastq_sam": ("sample_reads.fastq.gz", "sample_overlaps.sam.gz", "sample_layout.fasta.gz", False, 0.3),
    "fastq_mhap": ("sample_reads.fastq.gz", "sample_ava_overlaps.mhap.gz", "sample_reads.fastq.gz", False, 0.3),
    "frag_fastq_paf": ("sample_reads.fastq.gz", "sample_ava_overlaps.paf.gz", "sample_reads.fastq.gz", True, 0.3),
    "frag_fasta_mhap": ("sample_reads.fasta.gz", "sample_ava_overlaps.mhap.gz", "sample_reads.fasta.gz", True, 0.3),
    "fastq_paf_strict": ("sample_reads.fastq.gz", "sample_overlaps.paf.gz", "sample_layout.fasta.gz", False, 0.05),
}


def _open(case):
    reads, overlaps, target, frag, e = CASES[case]
    return api.InputFiles(os.path.join(DATA, reads), os.path.join(DATA, overlaps), os.path.join(DATA, target),
                          fragment_correction=frag, error_threshold=e)


@pytest.mark.parametrize("case", sorted(CASES))
def test_loaded_input_equals_the_reference_state(case):
    g = np.load(GOLD)
    f = _open(case)
    length = np.diff(f.seq_off.astype(np.int64))
    ref_len = g[case + "/length"].astype(np.int64)
    assert len(length) == len(ref_len)
    kept = ref_len > 0                       # the reference frees the data of reads no overlap points at
    assert (length[kept] == ref_len[kept]).all()
    assert (f.seq_has_qual[kept] == g[case + "/has_qual"][kept]).all()
    for i in np.flatnonzero(kept):
        a, b = int(f.seq_off[i]), int(f.seq_off[i + 1])
        assert zlib.crc32(f.bases[a:b].tobytes()) == int(g[case + "/crc_data"][i]), "bases of sequence %d" % i
        if f.seq_has_qual[i]:
            assert zlib.crc32(f.quals[a:b].tobytes()) == int(g[case + "/crc_qual"][i]), "qualities of sequence %d" % i
    ref_names = g[case + "/names"].tobytes().split(b"\0")
    assert f.names[:f.n_targets] == ref_names[:f.n_targets]   # the reference drops the names of non-target reads
    assert f.overlaps.shape == g[case + "/overlaps"].shape
    ref_ov = g[case + "/overlaps"].copy()
    ref_ov[:, 2] = ref_ov[:, 2] != 0         # the reference keeps `flag & 0x10` of a SAM record as its strand
    assert (f.overlaps == ref_ov).all()
    # every overlap points at sequences the reference kept
    assert kept[f.overlaps[:, 0]].all() and kept[f.overlaps[:, 1]].all()
    assert f.window_type_tgs        # the sample's reads average ~7 kb


def test_sam_alignments_give_the_reference_breaking_points():
    g = np.load(GOLD)
    f = _open("fastq_sam")
    off, bp = g["fastq_sam/bp_off"], g["fastq_sam/bp"]
    assert all(c for c in f.cigars)
    for i in range(len(f.overlaps)):
        mine = f.cigar_breaking_points(i, 500)
        assert (mine == bp[int(off[i]):int(off[i + 1])]).all(), "overlap %d" % i
    # another window length: against a base-by-base walk of the same CIGAR (the definition, overlap.cpp:226-292)
    for i in (0, 7, len(f.overlaps) - 1):
        assert (f.cigar_breaking_points(i, 137) == _walk(f.cigars[i].decode(), f.overlaps[i], 137)).all()


def test_sam_files_to_windows_equal_the_reference_windows():
    """SAM input carries its alignments, so files -> windows needs no device: createPolisher + initialize of the host layer
    against the windows the unmodified reference built from the same three files (layers, qualities, positions)."""
    g = np.load(GOLD)
    reads, overlaps, target, _, _ = CASES["fastq_sam"]
    pol = api.MirrorPolisher.from_files(os.path.join(DATA, reads), os.path.join(DATA, overlaps), os.path.join(DATA, target))
    try:
        r = pol.export()
        assert (np.diff(r["win_first"].astype(np.int64)) == g["fastq_sam/window_layers"]).all()
        assert (util.window_crcs(r) == g["fastq_sam/window_crc"]).all()
    finally:
        pol.close()


def _walk(cigar, o, w):
    _, _, strand, qb, qe, ql, tb, te, _ = (int(x) for x in o)
    ends = [i - 1 for i in range(0, te, w) if i > tb] + [te - 1]
    q, t, k, found, first, last, out, num = (ql - qe if strand else qb) - 1, tb - 1, 0, False, None, None, [], ""
    for c in cigar:
        if c.isdigit():
            num += c
            continue
        n, num = int(num), ""
        for _ in range(n if c in "M=XDN" else 0):
            t += 1
            if c in "M=X":
                q += 1
                if not found:
                    found, first = True, (t, q)
                last = (t + 1, q + 1)
            if k < len(ends) and t == ends[k]:
                if found:
                    out += [first, last]
                found, k = False, k + 1
        if c == "I":
            q += n
    return np.asarray(out, np.uint32).reshape(-1, 2)


def _write(path, text):
    with (gzip.open if path.endswith(".gz") else open)(path, "wb") as fh:
        fh.write(text.encode())


def test_record_rules_on_handwritten_files(tmp_path):
    """Multi-line FASTA/FASTQ, names cut at the first blank, lower case -> upper case, an all-'!' quality dropped, a read
    that is also a target kept once, MHAP ordinals, one overlap per read (the longest; first of equals), -e and
    self-overlaps filtered, unknown names skipped, CRLF line ends, no newline at the end of the file."""
    d = str(tmp_path)
    t1, t2 = "ACGTACGTAAACCCGGGTTT" * 3, "TTGACCAGTA" * 5
    _write(d + "/t.fasta", ">ctg1 some description\n%s\n%s\n>ctg2\r\n%s\r\n" % (t1[:25], t1[25:].lower(), t2))
    r1, r2, r3 = "ACGTACGTAAACCCGGGTTTACGT", "GGGTTTACGTACGTAAACCC", "ACGTTGCA" * 4
    _write(d + "/r.fastq.gz", "@r1 x\n%s\n+\n%s\n@r2\n%s\n%s\n+r2\n%s\n%s\n@ctg2\n%s\n+\n%s\n@r3\n%s\n+\n%s" % (
        r1, "I" * len(r1), r2[:7], r2[7:], "5" * 7, "6" * (len(r2) - 7), t2, "!" * len(t2), r3, "!" * len(r3)))
    paf = [("r1", len(r1), 0, 20, "+", "ctg1", 60, 0, 20), ("r1", len(r1), 0, 24, "+", "ctg1", 60, 20, 44),
           ("r1", len(r1), 2, 24, "-", "ctg2", 50, 3, 27),      # shorter than the second: dropped
           ("r2", len(r2), 0, 10, "+", "ctg1", 60, 0, 20),      # error 0.5 > 0.3: dropped
           ("r2", len(r2), 0, 20, "-", "ctg2", 50, 1, 21), ("nobody", 10, 0, 10, "+", "ctg1", 60, 0, 10),
           ("ctg2", 50, 0, 50, "+", "ctg2", 50, 0, 50),         # a sequence against itself: dropped
           ("r3", len(r3), 0, 32, "+", "ctg2", 50, 0, 32), ("r3", len(r3), 0, 32, "+", "ctg1", 60, 4, 36)]
    _write(d + "/o.paf", "".join("\t".join(str(x) for x in row) + "\t10\t20\t255\ttp:A:P\n" for row in paf))
    f = api.InputFiles(d + "/r.fastq.gz", d + "/o.paf", d + "/t.fasta")
    assert f.n_targets == 2 and f.names == [b"ctg1", b"ctg2", b"r1", b"r2", b"r3"]
    seq = [f.bases[int(a):int(b)].tobytes().decode() for a, b in zip(f.seq_off[:-1], f.seq_off[1:])]
    assert seq == [t1, t2, r1, r2, r3]
    assert list(f.seq_has_qual) == [0, 0, 1, 1, 0]
    assert f.quals[int(f.seq_off[3]):int(f.seq_off[4])].tobytes() == b"5" * 7 + b"6" * (len(r2) - 7)
    assert not f.window_type_tgs                     # reads average <= 1000 bases -> kNGS
    assert f.overlaps.tolist() == [[2, 0, 0, 0, 24, 24, 20, 44, 60], [3, 1, 1, 0, 20, 20, 1, 21, 50],
                                   [4, 1, 0, 0, 32, 32, 0, 32, 50]]
    # -f keeps every overlap that passes -e and is not a self-overlap
    ff = api.InputFiles(d + "/r.fastq.gz", d + "/o.paf", d + "/t.fasta", fragment_correction=True)
    assert len(ff.overlaps) == 6
    # MHAP: 1-based ordinals of the reads file / the target file; strand = a_rc xor b_rc
    _write(d + "/o.mhap", "1 1 0.1 10 0 0 24 24 0 20 44 60\n2 2 0.1 10 0 0 20 20 1 1 21 50\n9 1 0.1 10 0 0 5 5 0 0 5 60\n"
                          "3 2 0.1 10 1 0 50 50 1 0 50 50\n")
    fm = api.InputFiles(d + "/r.fastq.gz", d + "/o.mhap", d + "/t.fasta")
    assert fm.overlaps.tolist() == [[2, 0, 0, 0, 24, 24, 20, 44, 60], [3, 1, 1, 0, 20, 20, 1, 21, 50]]


def test_input_errors_are_reported_like_the_reference(tmp_path):
    d = str(tmp_path)
    _write(d + "/t.fasta", ">c\nACGTACGTAC\n")
    _write(d + "/r.fasta", ">r\nACGTAC\n")
    _write(d + "/o.paf", "r\t6\t0\t6\t+\tc\t10\t0\t6\t6\t6\t255\n")
    api.InputFiles(d + "/r.fasta", d + "/o.paf", d + "/t.fasta")
    with pytest.raises(RuntimeError, match="unsupported format extension"):
        api.InputFiles(d + "/r.txt", d + "/o.paf", d + "/t.fasta")
    with pytest.raises(RuntimeError, match="unsupported format extension"):
        api.InputFiles(d + "/r.fasta", d + "/o.bed", d + "/t.fasta")
    with pytest.raises(RuntimeError, match="unable to open"):
        api.InputFiles(d + "/missing.fasta", d + "/o.paf", d + "/t.fasta")
    _write(d + "/bad.paf", "r\t7\t0\t6\t+\tc\t10\t0\t6\t6\t6\t255\n")         # read length disagrees with the file
    with pytest.raises(RuntimeError, match="unequal lengths in sequence and overlap file"):
        api.InputFiles(d + "/r.fasta", d + "/bad.paf", d + "/t.fasta")
    _write(d + "/bad2.paf", "r\t6\t0\t6\t+\tc\t11\t0\t6\t6\t6\t255\n")
    with pytest.raises(RuntimeError, match="unequal lengths in target and overlap file"):
        api.InputFiles(d + "/r.fasta", d + "/bad2.paf", d + "/t.fasta")
    _write(d + "/none.paf", "x\t6\t0\t6\t+\tc\t10\t0\t6\t6\t6\t255\n")
    with pytest.raises(RuntimeError, match="empty overlap set"):
        api.InputFiles(d + "/r.fasta", d + "/none.paf", d + "/t.fasta")
    _write(d + "/short.paf", "r\t6\t0\t6\t+\tc\t10\n")
    with pytest.raises(RuntimeError, match="invalid PAF record"):
        api.InputFiles(d + "/r.fasta", d + "/short.paf", d + "/t.fasta")
    _write(d + "/trunc.fastq", "@r\nACGTAC\n+\nIII\n")
    with pytest.raises(RuntimeError, match="invalid FASTQ record"):
        api.InputFiles(d + "/trunc.fastq", d + "/o.paf", d + "/t.fasta")
    _write(d + "/dup.fasta", ">c\nACGT\n")                                      # same name as a target, other length
    with pytest.raises(RuntimeError, match="duplicate sequence c with unequal data"):
        api.InputFiles(d + "/dup.fasta", d + "/o.paf", d + "/t.fasta")
