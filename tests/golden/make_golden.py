#!/usr/bin/env python
"""Generate tests/golden/<case>.npz: inputs + the outputs of the UNMODIFIED reference executing the graph through its C
linker (mode="CVM").  Run after `__graft_entry__.build()` (it builds the reference into oracle/_ref):
    python tests/golden/make_golden.py
The fixtures pin (a) the CUDA backend on the GPU box without needing the reference there, and (b) oracle/numpy_port.py.
"""

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)

from cases import CASES  # noqa: E402
from oracle import cvm  # noqa: E402


def main():
    for name, build in CASES.items():
        ins, outs, args, floatX = build()
        pytensor = cvm.configure(floatX)
        f = pytensor.function(ins, outs, mode="CVM")
        res = f(*[np.array(a, copy=True) for a in args])
        payload = {f"in{k}": np.asarray(a) for k, a in enumerate(args)}
        payload.update({f"out{k}": np.asarray(r) for k, r in enumerate(res)})
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **payload)
        print(name, [np.asarray(r).shape for r in res])


if __name__ == "__main__":
    main()
