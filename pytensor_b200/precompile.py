"""Build-time kernel cache warm-up: trace the BASELINE workloads in trace-only mode (runtime/lib.py TRACE_ONLY) so that
every NVRTC kernel they launch is compiled for sm_100a, without a GPU, into the cache `__graft_entry__.build()` points
PTK_KCACHE at (`pytensor_b200/_kcache/`)."""

from __future__ import annotations

import numpy as np


def trace_function(f, args):
    """Run `f` once in trace-only mode (no device, no results); returns the number of kernels it would launch."""
    from pytensor_b200.runtime import jit
    from pytensor_b200.runtime import lib as _lib

    prev = _lib.TRACE_ONLY
    _lib.set_trace_only(True)
    try:
        n0 = jit.stats["launches"]
        f(*args)
        return jit.stats["launches"] - n0
    finally:
        _lib.set_trace_only(prev)


def precompile_workloads(verbose=True):
    from pytensor_b200._host import ensure_pytensor

    ensure_pytensor()
    import pytensor

    import pytensor_b200  # noqa: F401
    from pytensor_b200 import workloads as W
    from pytensor_b200.runtime import jit

    old = pytensor.config.floatX
    pytensor.config.floatX = "float32"
    try:
        jobs = [("cfg2", W.cfg2_fused_elemwise(4096), "CUDA"), ("cfg2-smoke", W.cfg2_fused_elemwise(512), "CUDA"),
                ("cfg1", W.cfg1_readme(1024), "CUDA")]
        for name, (ins, outs, make_args, meta), mode in jobs:
            f = pytensor.function(ins, outs, mode=mode)
            args = [np.empty_like(a) for a in make_args()]
            n = trace_function(f, args)
            if verbose:
                print(f"[precompile] {name}: {n} launches traced; cache stats {jit.stats}")
    finally:
        pytensor.config.floatX = old
