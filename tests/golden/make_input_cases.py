"""Fixture for the input layer (SURVEY §8 f4; racon_b200/csrc/reads_io.*): what the UNMODIFIED reference Polisher holds
after parsing + filtering — oracle/_ref/refpol_dump with $REFPOL_OVERLAP_DUMP (oracle/ref_polisher_harness.cpp) — for every
file-format combination the reference's own tests use (test/racon_test.cpp:86-295):
  per case: sequence lengths, quality flags and CRC-32 of the bases / qualities of every sequence the reference kept the
  data of (it frees reads no overlap points at), the target names, the filtered overlap table (ids, strand, coordinates)
  and — SAM input, where the alignment comes from the file — the breaking points of every overlap; one CRC-32 per window
  the reference built (layers with qualities and positions), and count / bases / md5 / names+tags of what it polished
  (scores 3 -5 -4, w 500, q 10, trimming on, unpolished sequences kept); and the md5 of what the reference's command
  line (integration/_build/racon, CPU path, default options) prints for the fastq_paf files.
The input files are the cut of the reference's sample under tests/golden/sample/ (tests/golden/make_sample_data.py).
Stored in tests/golden/sample/input_cases.npz.  Run where the reference is built:  python tests/golden/make_input_cases.py"""
import hashlib
import os
import struct
import subprocess
import sys
import tempfile
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests.util import window_crcs  # noqa: E402
DATA = os.path.join(ROOT, "tests", "golden", "sample") + os.sep

# name: reads, overlaps, target, fragment correction, error threshold
CASES = {
    "fastq_paf": ("sample_reads.fastq.gz", "sample_overlaps.paf.gz", "sample_layout.fasta.gz", 0, 0.3),
    "fasta_paf": ("sample_reads.fasta.gz", "sample_overlaps.paf.gz", "sample_layout.fasta.gz", 0, 0.3),
    "fastq_sam": ("sample_reads.fastq.gz", "sample_overlaps.sam.gz", "sample_layout.fasta.gz", 0, 0.3),
    "fastq_mhap": ("sample_reads.fastq.gz", "sample_ava_overlaps.mhap.gz", "sample_reads.fastq.gz", 0, 0.3),
    "frag_fastq_paf": ("sample_reads.fastq.gz", "sample_ava_overlaps.paf.gz", "sample_reads.fastq.gz", 1, 0.3),
    "frag_fasta_mhap": ("sample_reads.fasta.gz", "sample_ava_overlaps.mhap.gz", "sample_reads.fasta.gz", 1, 0.3),
    "fastq_paf_strict": ("sample_reads.fastq.gz", "sample_overlaps.paf.gz", "sample_layout.fasta.gz", 0, 0.05),
}


def reference_state(reads, overlaps, target, fragment, error_threshold, window_length=500):
    exe = os.path.join(ROOT, "oracle", "_ref", "refpol_dump")
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "refpol"], stdout=subprocess.DEVNULL)
    with tempfile.TemporaryDirectory() as tmp:
        dump = os.path.join(tmp, "ov.bin")
        env = dict(os.environ, REFPOL_OVERLAP_DUMP=dump)
        subprocess.check_call([exe, DATA + reads, DATA + overlaps, DATA + target, str(fragment), str(window_length),
                               "10.0", str(error_threshold), "1", "3", "-5", "-4", "8", os.path.join(tmp, "w.bin")],
                              env=env, stderr=subprocess.DEVNULL)
        raw = open(dump, "rb").read()
        wraw = open(os.path.join(tmp, "w.bin"), "rb").read()
    pos = 0

    def take(fmt):
        nonlocal pos
        (v,) = struct.unpack_from(fmt, raw, pos)
        pos += struct.calcsize(fmt)
        return v

    def blob(n):
        nonlocal pos
        b = raw[pos:pos + n]
        pos += n
        return b

    seqs = []
    for _ in range(take("<Q")):
        name = blob(take("<I"))
        data = blob(take("<Q"))
        qual = blob(take("<Q"))
        seqs.append((name, data, qual))
    nov = take("<Q")
    ov = np.zeros((nov, 9), np.uint32)
    bp_off, bps = [0], []
    for i in range(nov):
        ov[i] = [take("<I") for _ in range(9)]
        n = take("<I")
        bps.append(np.frombuffer(blob(8 * n), np.uint32).reshape(n, 2).copy())
        bp_off.append(bp_off[-1] + n)
    assert pos == len(raw)
    return (seqs, ov, np.asarray(bp_off, np.uint64), (np.concatenate(bps) if bps else np.zeros((0, 2), np.uint32)),
            windows_and_polished(wraw))


def windows_and_polished(raw):
    import hashlib
    nw, ns, nb, npol = struct.unpack_from("<4Q", raw, 0)
    pos = 32
    r = {}
    for key, dt, n in (("bases", np.uint8, nb), ("quals", np.uint8, nb), ("seq_off", np.uint64, ns + 1),
                       ("seq_has_qual", np.uint8, ns), ("seq_begin", np.uint32, ns), ("seq_end", np.uint32, ns),
                       ("win_first", np.uint32, nw + 1), ("win_type", np.uint8, nw), ("win_target", np.uint64, nw),
                       ("win_rank", np.uint32, nw)):
        r[key] = np.frombuffer(raw, dt, n, pos)
        pos += n * np.dtype(dt).itemsize
    for _ in range(nw):
        (n,) = struct.unpack_from("<I", raw, pos)
        pos += 4 + n
    h = hashlib.md5()
    total, tags = 0, []
    for _ in range(npol):
        (nl,) = struct.unpack_from("<I", raw, pos)
        pos += 4
        name = raw[pos:pos + nl].decode()
        pos += nl
        (n,) = struct.unpack_from("<Q", raw, pos)
        pos += 8
        h.update(raw[pos:pos + n])
        total += n
        pos += n
        tags.append(name)
    return dict(window_crc=window_crcs(r), layers=np.diff(r["win_first"].astype(np.int64)).astype(np.uint32),
                polished_count=npol, polished_bases=total, polished_md5=h.hexdigest(), polished_names="\n".join(tags))


def main():
    out = {}
    for name, (reads, overlaps, target, fragment, e) in CASES.items():
        seqs, ov, bp_off, bp, wp = reference_state(reads, overlaps, target, fragment, e)
        out[name + "/window_crc"], out[name + "/window_layers"] = wp["window_crc"], wp["layers"]
        out[name + "/polished"] = np.asarray([wp["polished_count"], wp["polished_bases"]], np.uint64)
        out[name + "/polished_md5"] = np.frombuffer(wp["polished_md5"].encode(), np.uint8)
        out[name + "/polished_names"] = np.frombuffer(wp["polished_names"].encode(), np.uint8)
        out[name + "/length"] = np.asarray([len(d) for _, d, _ in seqs], np.uint64)
        out[name + "/has_qual"] = np.asarray([1 if q else 0 for _, _, q in seqs], np.uint8)
        out[name + "/crc_data"] = np.asarray([zlib.crc32(d) for _, d, _ in seqs], np.uint32)
        out[name + "/crc_qual"] = np.asarray([zlib.crc32(q) for _, _, q in seqs], np.uint32)
        out[name + "/names"] = np.frombuffer(b"\0".join(n for n, _, _ in seqs), np.uint8)
        out[name + "/overlaps"] = ov
        if overlaps.endswith(".sam.gz"):
            out[name + "/bp_off"], out[name + "/bp"] = bp_off, bp
        print(name, "sequences", len(seqs), "with data", sum(1 for _, d, _ in seqs if d), "overlaps", len(ov), "windows",
              len(wp["window_crc"]), "polished", wp["polished_count"], wp["polished_bases"], wp["polished_md5"])
    racon = os.path.join(ROOT, "integration", "_build", "racon")
    reads, overlaps, target, _, _ = CASES["fastq_paf"]
    cli = subprocess.run([racon, "-t", "4", DATA + reads, DATA + overlaps, DATA + target], stdout=subprocess.PIPE,
                         stderr=subprocess.DEVNULL, check=True).stdout
    out["cli_md5"] = np.frombuffer(hashlib.md5(cli).hexdigest().encode(), np.uint8)
    print("racon stdout", len(cli), "bytes, md5", hashlib.md5(cli).hexdigest())
    path = DATA + "input_cases.npz"
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
