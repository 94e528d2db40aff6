"""The UNMODIFIED reference host (src/main.cpp, src/polisher.cpp, src/cuda/cudapolisher.cpp, ... compiled where they lie
by integration/Makefile with -DCUDA_ENABLED) linked against libracon_b200.so through integration/cudabatch.cpp and
integration/cudaaligner.cpp, run on the reference's own sample files.

  * `racon -c 1 [-b] [--cudaaligner-batches 1]` prints exactly what the reference's CPU build prints (md5 of stdout);
  * the reference's CUDA test cases (test/racon_test.cpp:297-507) reach the CPU goldens of test/racon_test.cpp:86-295 —
    the reference's own CUDA build does not (it carries separate goldens: 1385, 1607, 1541, 1661, 4168, 1361, 397185 ...).

`make -C oracle integration` compiles the reference's part and copies the sample files into oracle/_ref/integration/
(where the reference's sources exist); `make -C integration` (run by build()) links them with integration/'s own sources
into integration/_build/.  The tests skip where the reference's part was not built."""
import hashlib
import json
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "integration", "_build")
RACON = os.path.join(BUILD, "racon")
GOLDENS = os.path.join(BUILD, "racon_goldens")
DATA = os.path.join(ROOT, "oracle", "_ref", "integration", "data")

# racon's stdout on the sample with default scores (SURVEY.md §8c: identical for 1/4/8 threads, SISD and AVX2 builds)
MD5_DEFAULT = "b0e2a2788440a4982e544e2e9b3bf378"

# test/racon_test.cpp CPU goldens: edit distance to sample_reference (:104,:128,:151,:174,:197,:220) and
# sequences / total length of the fragment-correction runs (:234-240, :252-258, :270-276, :288-294)
CPU_GOLDENS = {
    "ConsensusWithQualitiesCUDA": dict(sequences=1, edit_distance=1312),
    "ConsensusWithoutQualitiesCUDA": dict(sequences=1, edit_distance=1566),
    "ConsensusWithQualitiesAndAlignmentsCUDA": dict(sequences=1, edit_distance=1317),
    "ConsensusWithoutQualitiesAndWithAlignmentsCUDA": dict(sequences=1, edit_distance=1770),
    "ConsensusWithQualitiesLargerWindowCUDA": dict(sequences=1, edit_distance=1289),
    "ConsensusWithQualitiesEditDistanceCUDA": dict(sequences=1, edit_distance=1321),
    "FragmentCorrectionWithQualitiesCUDA": dict(sequences=40, total_length=401246),
    "FragmentCorrectionWithQualitiesFullCUDA": dict(sequences=236, total_length=1658216),
    "FragmentCorrectionWithoutQualitiesFullCUDA": dict(sequences=236, total_length=1663982),
    "FragmentCorrectionWithQualitiesFullMhapCUDA": dict(sequences=236, total_length=1658216),
}


def _need_build():
    if not (os.path.exists(RACON) and os.path.exists(GOLDENS) and os.path.isdir(DATA)):
        pytest.skip("integration/_build missing: needs oracle/_ref/integration, built from the reference's sources")


def test_integration_binaries_are_the_reference_host_linked_to_the_product_library():
    """CPU side: the build exists, is dynamically linked to libracon_b200.so, and its CPU path still prints the golden
    output (so what the GPU test compares against is the unmodified reference behaviour)."""
    _need_build()
    ldd = subprocess.run(["ldd", RACON], stdout=subprocess.PIPE, text=True).stdout
    assert "libracon_b200.so" in ldd
    out = subprocess.run([RACON, "--version"], stdout=subprocess.PIPE, text=True).stdout
    assert out.startswith("1.5.0")
    cpu = subprocess.run([RACON, "-t", "4", os.path.join(DATA, "sample_reads.fastq.gz"),
                          os.path.join(DATA, "sample_overlaps.paf.gz"), os.path.join(DATA, "sample_layout.fasta.gz")],
                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL).stdout
    assert hashlib.md5(cpu).hexdigest() == MD5_DEFAULT


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [["-c", "1"], ["-c", "2", "-b"], ["-c", "1", "--cudaaligner-batches", "1"],
                                   ["-c", "1", "-b", "--cudaaligner-batches", "2"]],
                         ids=["c1", "c2_banded", "c1_aligner", "c1_banded_aligner2"])
def test_racon_cli_with_cuda_flags_prints_the_cpu_output(flags):
    _need_build()
    r = subprocess.run([RACON, "-t", "8"] + flags + [os.path.join(DATA, "sample_reads.fastq.gz"),
                                                      os.path.join(DATA, "sample_overlaps.paf.gz"),
                                                      os.path.join(DATA, "sample_layout.fasta.gz")],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    assert hashlib.md5(r.stdout).hexdigest() == MD5_DEFAULT, r.stderr.decode()[-1500:]
    err = r.stderr.decode()
    assert "[racon::CUDAPolisher::polish] polished windows on GPU" in err
    if "--cudaaligner-batches" in flags:
        assert "Alignment skipped by GPU: 0 /" in err


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [[], ["--banded"], ["--aligner-batches", "1"]], ids=["poa", "poa_banded", "poa_aligner"])
def test_reference_cuda_test_cases_reach_the_cpu_goldens(extra):
    _need_build()
    env = dict(os.environ)
    if "--banded" in extra:
        # -b only uses the band layout for windows of >= 768 bases (where it is the faster kernel); these goldens are
        # about the band itself, so ask for it explicitly on the 500-base cases too (256 columns)
        env["RP_POA_BAND_K"] = "8"
    r = subprocess.run([GOLDENS, DATA] + extra, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=1500, env=env)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    got = {}
    for line in r.stdout.decode().splitlines():
        if line.startswith("{"):
            d = json.loads(line)
            got[d["case"]] = d
    assert set(got) == set(CPU_GOLDENS)
    for name, want in CPU_GOLDENS.items():
        for k, v in want.items():
            assert got[name][k] == v, (name, k, got[name], want)
