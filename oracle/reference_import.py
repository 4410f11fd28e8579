"""Make the UNMODIFIED Python reference (the rl-colosseum 1.2 package) importable.

TEST INFRASTRUCTURE ONLY.  Used by tests/golden/make_*.py (to generate the committed golden vectors) and by the
cross-checks against live reference objects, which skip when the package is not staged.  Nothing in colosseum_b200/
imports this.

What it does (SURVEY.md section 8c): puts oracle/ref_shim (stand-ins for dm_env, gin, toolz, pydtmc, sparse, gym) and
REFERENCE_ROOT on sys.path, and restores two names the reference needs that numpy-2 / py3.12 dropped
(`numpy.core._exceptions`, `collections.Container`).
"""
import collections
import collections.abc
import os
import sys
import types

# where the UNMODIFIED package is looked for: $COLOSSEUM_REFERENCE_ROOT, else a copy staged inside the tree (both
# git-ignored), e.g. by `pip install --no-index --no-deps --target oracle/_ref <source of rl-colosseum 1.2>`
_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_CANDIDATES = [os.path.join(_REPO, "oracle", "_ref"), os.path.join(_REPO, "baseline", "_ref")]
REFERENCE_ROOT = os.environ.get("COLOSSEUM_REFERENCE_ROOT") or next(
    (c for c in _CANDIDATES if os.path.isdir(os.path.join(c, "colosseum"))), _CANDIDATES[0])
_SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_shim")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "colosseum"))


def import_reference():
    """Returns the imported `colosseum` reference package (raises if it is not staged)."""
    if not reference_available():
        raise ImportError(f"reference not present at {REFERENCE_ROOT}")
    for p in (_SHIM, REFERENCE_ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)
    if not hasattr(collections, "Container"):
        collections.Container = collections.abc.Container
    import numpy as np

    if "numpy.core._exceptions" not in sys.modules:
        try:
            import numpy._core._exceptions as _exc
        except Exception:  # pragma: no cover
            _exc = types.ModuleType("numpy.core._exceptions")
            _exc._ArrayMemoryError = MemoryError
        sys.modules["numpy.core._exceptions"] = _exc
    # importing the reference copies its hardness cache (3,007 files) and creates `tmp/` in the CURRENT directory
    # (colosseum/config.py:255-270): do the import from a scratch directory so nothing lands in the repository
    import tempfile

    cwd = os.getcwd()
    os.chdir(tempfile.mkdtemp(prefix="colosseum_ref_"))
    try:
        import colosseum  # noqa: E402
    finally:
        os.chdir(cwd)

    colosseum.config.disable_multiprocessing()
    colosseum.config.VERBOSE_LEVEL = 0
    return colosseum
