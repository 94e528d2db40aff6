"""Files in, polished FASTA out through the C++ host layer (reads_io -> Polisher::initialize -> polish_streaming): every
file-format combination of the reference's own tests (test/racon_test.cpp:86-295), against what the UNMODIFIED reference
built and polished from the same files on the CPU (tests/golden/sample/input_cases.npz, made by
tests/golden/make_input_cases.py).
Alignment, breaking points and consensus run on the device; parsing, filtering, window assembly and stitching on the host.
(The file name sorts after the parity tests of the kernels on purpose: this is the widest test, it runs last.)"""
import hashlib
import os

import numpy as np
import pytest

from racon_b200 import api
from tests import util
from tests.test_reads_io import CASES, DATA, GOLD

pytestmark = pytest.mark.gpu


def _records(path):
    names, seqs = [], []
    for line in open(path, "rb").read().split(b"\n"):
        if line.startswith(b">"):
            names.append(line[1:].decode())
        elif line:
            seqs.append(line)
    return names, seqs


@pytest.mark.parametrize("case", sorted(CASES))
def test_files_to_polished_fasta_equals_the_reference(case, tmp_path):
    g = np.load(GOLD)
    reads, overlaps, target, frag, e = CASES[case]
    pol = api.MirrorPolisher.from_files(os.path.join(DATA, reads), os.path.join(DATA, overlaps), os.path.join(DATA, target),
                                        fragment_correction=frag, error_threshold=e)
    try:
        r = pol.export()
        assert (np.diff(r["win_first"].astype(np.int64)) == g[case + "/window_layers"]).all()
        assert (util.window_crcs(r) == g[case + "/window_crc"]).all(), "windows differ from the reference's"
        out = str(tmp_path / "polished.fasta")
        n = pol.stream_fasta(out, None, drop_unpolished=False)
        assert pol.failed() == (0, 0)
    finally:
        pol.close()
    names, seqs = _records(out)
    count, bases = (int(x) for x in g[case + "/polished"])
    assert n == count == len(seqs)
    assert sum(len(s) for s in seqs) == bases
    assert hashlib.md5(b"".join(seqs)).hexdigest() == g[case + "/polished_md5"].tobytes().decode()
    assert names == g[case + "/polished_names"].tobytes().decode().split("\n")


@pytest.mark.parametrize("case", ["fastq_sam", "fasta_paf", "frag_fastq_paf"])
def test_files_to_polished_fasta_with_resident_reads(case, tmp_path):
    """The same run with every sequence uploaded once, the aligner's spans and the windows' pieces named by reference
    (SURVEY §8 f2: extracted on the device, reverse complements and weights included): the reference's bytes again."""
    g = np.load(GOLD)
    reads, overlaps, target, frag, e = CASES[case]
    pol = api.MirrorPolisher.from_files(os.path.join(DATA, reads), os.path.join(DATA, overlaps), os.path.join(DATA, target),
                                        fragment_correction=frag, error_threshold=e, resident_reads=True)
    try:
        out = str(tmp_path / "polished.fasta")
        n = pol.stream_fasta(out, None, drop_unpolished=False, resident_reads=True, mem_bytes=256 << 20)
        assert pol.failed() == (0, 0)
    finally:
        pol.close()
    names, seqs = _records(out)
    count, bases = (int(x) for x in g[case + "/polished"])
    assert n == count == len(seqs) and sum(len(s) for s in seqs) == bases
    assert hashlib.md5(b"".join(seqs)).hexdigest() == g[case + "/polished_md5"].tobytes().decode()
    assert names == g[case + "/polished_names"].tobytes().decode().split("\n")


def test_polish_files_drops_unpolished_like_the_cli(tmp_path):
    """api.polish_files = the racon command line's default (unpolished sequences dropped): the lambda sample gives the
    one polished contig of the reference's CPU run, byte for byte (md5 of the reference's `racon` stdout on the same files)."""
    g = np.load(GOLD)
    out = str(tmp_path / "o.fasta")
    n, fo, fw = api.polish_files(os.path.join(DATA, "sample_reads.fastq.gz"), os.path.join(DATA, "sample_overlaps.paf.gz"),
                                 os.path.join(DATA, "sample_layout.fasta.gz"), out)
    assert (n, fo, fw) == (1, 0, 0)
    assert hashlib.md5(open(out, "rb").read()).hexdigest() == g["cli_md5"].tobytes().decode()
