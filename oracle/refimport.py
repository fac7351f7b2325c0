"""Import the REAL reference (pfnet/pfrl).

TEST INFRASTRUCTURE ONLY.  The reference tree (PFRL_REFERENCE_ROOT) is read-only
and only present where fixtures are generated, so this is used by the
oracle/gen_golden*.py generators and by bench.py's CPU baseline, never by the
tests: they compare against what the generators recorded under tests/golden/.
"""
import os
import sys

REFERENCE_ROOT = os.environ.get("PFRL_REFERENCE_ROOT", "/root/reference")
_HERE = os.path.dirname(os.path.abspath(__file__))
_SHIM = os.path.join(_HERE, "gym_shim")
# the unmodified reference package zipped by oracle/build_ref.py (travels to the GPU box)
REF_ARCHIVE = os.path.join(_HERE, "_ref", "pfrl_ref.zip")


def tree_available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "pfrl"))


def available():
    return tree_available() or os.path.exists(REF_ARCHIVE)


def import_reference():
    """Return the reference's top-level ``pfrl`` module (or raise ImportError):
    from the reference tree when present (build container), else from the
    archive oracle/build_ref.py made of it."""
    if not available():
        raise ImportError("reference neither at %s nor in %s" % (REFERENCE_ROOT, REF_ARCHIVE))
    sys.dont_write_bytecode = True  # the mount is read-only
    src = REFERENCE_ROOT if tree_available() else REF_ARCHIVE
    for p in (_SHIM, src):
        if p not in sys.path:
            sys.path.insert(0, p)
    import pfrl  # noqa: E402

    return pfrl
