#!/usr/bin/env python
"""from_device_csc right after the generator (no host work in between): the bound must equal the
one of a run that waited (checks the producer-stream synchronisation in Engine.from_device_csc)."""
import ctypes as C, os, sys
sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import numpy as np, torch
import bench
from ccfindr_b200 import _lib, synth
from ccfindr_b200.engine import Engine
wl = bench.WORKLOADS["c3"]; n, r = wl["n"], wl["rank"]; m = int(sys.argv[1]) if len(sys.argv) > 1 else 400000
dev = torch.device("cuda", 0)
w0, h0 = bench.init_factors(n, m, r, seed=1000 * r + 1)
for wait in ("nosync", True, False, "nosync"):
    colptr, rowidx, values, _ = synth.tenx_like_device(n, m, wl["r_true"], wl["density"], wl["seed"], dev)
    if wait is True:
        torch.cuda.synchronize()
    if wait == "nosync":   # the constructor as it was before the fix: no wait for torch's stream
        eng = Engine._create(lambda out: _lib.load().vbnmf_create_from_device(
            out, n, m, int(rowidx.numel()), C.c_void_p(colptr.data_ptr()),
            C.c_void_p(rowidx.data_ptr()), C.c_void_p(values.data_ptr()), 0),
            0, keep=(colptr, rowidx, values))
    else:
        eng = Engine.from_device_csc(n, m, int(rowidx.numel()), colptr, rowidx, values)
    eng.set_state(w0, h0)
    out = eng.run(bench.HYPER, Itmax=2, Tol=0.0)
    eng.close()
    print({True: "waited", False: "immediate", "nosync": "no sync (old)"}[wait], [float(v) for v in out["lkh_trace"]], flush=True)
    del colptr, rowidx, values
