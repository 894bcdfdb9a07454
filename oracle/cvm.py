"""Reference oracle: the reference's own C linker (`mode="CVM"`, pytensor/compile/mode.py:511) on the host CPU.

TEST INFRASTRUCTURE — see oracle/__init__.py.  The reference is imported from oracle/_ref (built by
oracle/build_ref.sh from a pytensor checkout); nothing here reads the checkout itself at run time.
"""

from __future__ import annotations

import glob
import os
import sys
import time

_HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(_HERE)
_configured = False


def _find_blas():
    """A linkable BLAS with standard (un-prefixed) symbols: the OpenBLAS inside the opencv wheel (SURVEY.md §8c.2)."""
    for sp in sys.path:
        d = os.path.join(sp, "opencv_python_headless.libs")
        libs = glob.glob(os.path.join(d, "libopenblas*.so"))
        if libs:
            return d, os.path.basename(libs[0])
    return None, None


def configure(floatX=None):
    """Set PYTENSOR_FLAGS (compile dir, BLAS) BEFORE pytensor is imported; import it from oracle/_ref."""
    global _configured
    if not _configured:
        flags = [f for f in os.environ.get("PYTENSOR_FLAGS", "").split(",") if f]
        keys = {f.split("=")[0] for f in flags}
        if "base_compiledir" not in keys:
            flags.append("base_compiledir=" + os.environ.get("PTK_COMPILEDIR", f"/tmp/ptk_compiledir_{os.getuid()}"))
        if "pytensor" not in sys.modules:
            d, lib = _find_blas()
            if d:
                # the wheel's OpenBLAS needs its sibling libgfortran/libquadmath: preload them by path so that the
                # C linker's modules resolve them by SONAME without LD_LIBRARY_PATH (also when the flag was inherited)
                import ctypes

                ok = True
                for pat in ("libquadmath*", "libgfortran*", lib):
                    for so in sorted(glob.glob(os.path.join(d, pat))):
                        try:
                            ctypes.CDLL(so, mode=ctypes.RTLD_GLOBAL)
                        except OSError:
                            ok = False
                if ok and "blas__ldflags" not in keys:
                    flags.append(f"blas__ldflags=-L{d} -l:{lib}")
        os.environ["PYTENSOR_FLAGS"] = ",".join(flags)
        ref = os.path.join(_HERE, "_ref")
        if "pytensor" not in sys.modules and os.path.isdir(os.path.join(ref, "pytensor")) and ref not in sys.path:
            sys.path.insert(0, ref)
        _configured = True
    import pytensor

    if floatX is not None:
        pytensor.config.floatX = floatX
    return pytensor


def describe():
    """Environment line recorded next to every CPU-baseline number (BASELINE.md §3)."""
    pytensor = configure()
    try:
        from pytensor.scan import scan_perform_ext  # noqa: F401

        cython_scan = True
    except Exception:
        cython_scan = False
    return {
        "cores": os.cpu_count(),
        "blas__ldflags": pytensor.config.blas__ldflags,
        "openmp": bool(pytensor.config.openmp),
        "cxx": pytensor.config.cxx,
        "cython_scan": cython_scan,
        "OMP_NUM_THREADS": os.environ.get("OMP_NUM_THREADS"),
        "OPENBLAS_NUM_THREADS": os.environ.get("OPENBLAS_NUM_THREADS"),
    }


def cvm_function(inputs, outputs, **kw):
    pytensor = configure()
    return pytensor.function(inputs, outputs, mode="CVM", **kw)


def time_function(f, args, min_seconds=3.0, min_calls=3, max_calls=1000):
    """Warm (1 call, includes the g++ compile) then wall-clock timing; returns (evals/s, n_calls)."""
    f(*args)
    n = 0
    t0 = time.perf_counter()
    while True:
        f(*args)
        n += 1
        dt = time.perf_counter() - t0
        if (dt >= min_seconds and n >= min_calls) or n >= max_calls:
            break
    return n / dt, n
