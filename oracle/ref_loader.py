"""Load the UNMODIFIED reference modules from a checkout of the reference (directory
ECW_REFERENCE_DIR) behind the pyscf stub.  Used by the oracle/make_golden*.py
scripts that write the fixtures under tests/golden/ (and by __graft_entry__.build()
as an import check when a checkout is present); the tests read those fixtures and
need no reference checkout.
"""
import importlib
import os
import sys

REF_DIR = os.environ.get("ECW_REFERENCE_DIR", "/root/reference/ECW_CC")
_STUB = os.path.join(os.path.dirname(os.path.abspath(__file__)), "pyscf_stub")


def available():
    return os.path.isfile(os.path.join(REF_DIR, "CCSD.py"))


def load(*names):
    """Return the requested reference modules (e.g. load('CCSD','CCS'))."""
    if not available():
        raise ImportError("reference tree not present at %s" % REF_DIR)
    try:
        import pyscf  # noqa: F401  (a real PySCF wins if it ever exists)
    except ImportError:
        if _STUB not in sys.path:
            sys.path.insert(0, _STUB)
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)  # the reference uses flat imports (CCSD.py:23)
    mods = [importlib.import_module(n) for n in names]
    return mods[0] if len(mods) == 1 else mods
