"""Locate the host framework.  PyTensor itself is NOT part of this repo: it is the host whose Linker plugin surface
the backend implements.  Search order: an installed `pytensor`, then the reference build in `oracle/_ref` (produced by
oracle/build_ref.sh from `__graft_entry__.build()`; git-ignored).
"""

from __future__ import annotations

import importlib.util
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CANDIDATES = [os.path.join(REPO, "oracle", "_ref")]


def ensure_pytensor() -> str:
    """Make `import pytensor` work; returns the directory it comes from. Raises ImportError with a recipe otherwise."""
    if "pytensor" in sys.modules:
        return os.path.dirname(os.path.dirname(sys.modules["pytensor"].__file__))
    if importlib.util.find_spec("pytensor") is None:
        for c in CANDIDATES:
            if os.path.isdir(os.path.join(c, "pytensor")):
                sys.path.insert(0, c)
                break
        else:
            raise ImportError(
                "pytensor (the host framework) is not importable; run `bash oracle/build_ref.sh <pytensor checkout>` "
                "to build oracle/_ref"
            )
    # a writable compile dir for the host's C linker (used by the oracle; the CUDA backend does not need it)
    if "PYTENSOR_FLAGS" not in os.environ or "base_compiledir" not in os.environ.get("PYTENSOR_FLAGS", ""):
        cdir = os.environ.get("PTK_COMPILEDIR", os.path.join("/tmp", f"ptk_compiledir_{os.getuid()}"))
        flags = os.environ.get("PYTENSOR_FLAGS", "")
        os.environ["PYTENSOR_FLAGS"] = (flags + "," if flags else "") + f"base_compiledir={cdir}"
    import pytensor  # noqa: F401

    return os.path.dirname(os.path.dirname(pytensor.__file__))
