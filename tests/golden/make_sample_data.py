"""A small cut of the reference's lambda-phage sample (test/data/sample_*.gz of the reference), stored under
tests/golden/sample/ with the original file names, for the tests that read input files (tests/test_reads_io.py,
tests/test_zz_files_pipeline.py):
  * the reads (FASTQ and FASTA) whose alignment to the contig ends before CUT_BASES, plus the two shortest reads that no
    overlap to the contig points at, in the original order and with the original records;
  * every overlap / SAM record between sequences that were kept (PAF, SAM), MHAP ordinals renumbered to the cut reads file;
  * the contig (sample_layout.fasta.gz) unchanged.
What the reference makes of these files is then tests/golden/sample/input_cases.npz (tests/golden/make_input_cases.py).
Run with the reference's source tree:  python tests/golden/make_sample_data.py REFERENCE_DIR"""
import gzip
import os
import sys

SRC = os.path.join(sys.argv[1], "test", "data")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "sample")
CUT_BASES = 13000


def read(name):
    return gzip.open(os.path.join(SRC, name)).read().decode()


def write(name, text):
    with open(os.path.join(OUT, name), "wb") as raw, gzip.GzipFile(fileobj=raw, mode="wb", mtime=0) as fh:
        fh.write(text.encode())


def records(text, marker):
    """(name, record text) of a FASTA or FASTQ file; sequences and qualities may span several lines."""
    out, lines, i = [], text.split("\n"), 0
    while i < len(lines):
        if not lines[i]:
            i += 1
            continue
        assert lines[i][0] == marker, lines[i][:40]
        j = i + 1
        if marker == ">":
            while j < len(lines) and not lines[j].startswith(">"):
                j += 1
        else:
            n = 0
            while not lines[j].startswith("+"):
                n += len(lines[j])
                j += 1
            j, q = j + 1, 0
            while q < n:
                q += len(lines[j])
                j += 1
        out.append((lines[i][1:].split()[0], "\n".join(lines[i:j]) + "\n"))
        i = j
    return out


def main():
    os.makedirs(OUT, exist_ok=True)
    fastq, fasta = records(read("sample_reads.fastq.gz"), "@"), records(read("sample_reads.fasta.gz"), ">")
    assert [n for n, _ in fastq] == [n for n, _ in fasta]
    paf = [l for l in read("sample_overlaps.paf.gz").split("\n") if l]
    mapped = {l.split("\t")[0]: int(l.split("\t")[8]) for l in paf}
    keep = {n for n, end in mapped.items() if end <= CUT_BASES}
    keep |= set(sorted((n for n, r in fastq if n not in mapped), key=lambda n: len(dict(fastq)[n]))[:2])
    write("sample_reads.fastq.gz", "".join(r for n, r in fastq if n in keep))
    write("sample_reads.fasta.gz", "".join(r for n, r in fasta if n in keep))
    write("sample_layout.fasta.gz", read("sample_layout.fasta.gz"))
    write("sample_overlaps.paf.gz", "".join(l + "\n" for l in paf if l.split("\t")[0] in keep))
    write("sample_ava_overlaps.paf.gz", "".join(l + "\n" for l in read("sample_ava_overlaps.paf.gz").split("\n")
                                                 if l and l.split("\t")[0] in keep and l.split("\t")[5] in keep))
    write("sample_overlaps.sam.gz", "".join(l + "\n" for l in read("sample_overlaps.sam.gz").split("\n")
                                             if l and (l[0] == "@" or l.split("\t")[0] in keep)))
    ordinal = {}   # MHAP names reads by their 1-based position in the reads file
    for i, (n, _) in enumerate(fastq):
        if n in keep:
            ordinal[str(i + 1)] = str(len(ordinal) + 1)
    mhap = []
    for l in read("sample_ava_overlaps.mhap.gz").split("\n"):
        f = l.split(" ")
        if l and f[0] in ordinal and f[1] in ordinal:
            mhap.append(" ".join([ordinal[f[0]], ordinal[f[1]]] + f[2:]) + "\n")
    write("sample_ava_overlaps.mhap.gz", "".join(mhap))
    print("kept %d of %d reads" % (len(keep), len(fastq)))
    for name in sorted(os.listdir(OUT)):
        print(name, os.path.getsize(os.path.join(OUT, name)), "bytes")


if __name__ == "__main__":
    main()
