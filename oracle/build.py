"""Builds the checkers (TEST INFRASTRUCTURE): oracle/_build/libpoa_oracle.so and, where /root/reference
exists, oracle/_ref/libracon_ref.so — both via oracle/Makefile."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))


def _make(target):
    r = subprocess.run(["make", "-C", HERE, target], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("oracle build failed (%s):\n%s" % (target, r.stdout))


def build_oracle():
    _make("oracle")
    return os.path.join(HERE, "_build", "libpoa_oracle.so")


def build_ref():
    out = os.path.join(HERE, "_ref", "libracon_ref.so")
    if os.path.isdir("/root/reference/src"):
        _make("ref")
    return out if os.path.exists(out) else None


def build_ref_cudapoa():
    """The reference's own GPU path (GenomeWorks cudapoa) compiled unmodified for sm_100 — timing baseline only."""
    out = os.path.join(HERE, "_ref", "libref_cudapoa.so")
    if os.path.isdir("/root/reference/vendor/GenomeWorks/cudapoa/src"):
        try:
            _make("refcuda")
        except RuntimeError as e:  # a baseline, not a checker: its absence is reported by bench.py, not fatal
            print("[oracle] reference cudapoa not built: %s" % str(e)[:500])
    return out if os.path.exists(out) else None


def build_integration():
    """The reference's host program compiled for integration/ (objects, the headers integration/ includes, the sample
    files) -> oracle/_ref/integration."""
    _make("integration")
    out = os.path.join(HERE, "_ref", "integration")
    return out if os.path.isdir(out) else None


def build_refpol():
    out = os.path.join(HERE, "_ref", "refpol_dump")
    if os.path.isdir("/root/reference/src"):
        _make("refpol")
    return out if os.path.exists(out) else None
