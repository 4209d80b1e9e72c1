#!/usr/bin/env python
"""Records tests/golden/reference_shaders/shading_matrix.npz: what the reference's own tracer.fs (compiled for the CPU,
oracle/reference_shaders.py) computes on the crafted shading cases of tests/test_gpu_shading_matrix.py -- the
accumulator after every tick, no NaN sanitising, no refraction cap.  The oracle must give the same bits on every case
(asserted before anything is written).  Records are stored as make_reference_outputs.py stores them (digest + sample).

Only tracer.fs is needed, so the library may be built without the atlas blit shader; pass such a build with --lib, so
that it never lands in oracle/_ref/ (where reference_shaders.available() would take it for a complete build):
    python tests/golden/make_shading_matrix.py [--lib path/to/libfspt_ref.so]
"""
import ctypes
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def make(out, oracle_mod, R):
    import test_gpu_shading_matrix as M
    from fspt_b200 import scenes
    for name, res in M.IDS:
        sa, cam, _ = M.build_case(name, res)
        Rf = R.Reference(sa)
        rc, rt = scenes.rand_bases(M.TICKS, M.SEED)
        fbs, _, _ = M.oracle_case(name, res)
        fr = None
        for k in range(M.TICKS):
            pos, d = M.primary(oracle_mod, cam, rc[k])
            fr = Rf.trace(pos, d, M.W, M.H, k, rt[k], cam["env_theta"], fb_prev=fr)
            assert golden.beq(fr, fbs[k]), (name, res, k)
            golden.record(out, M.record_key(name, res, k), fr)
    return M.PATH


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    sys.path.insert(0, os.path.dirname(HERE))
    sys.path.insert(0, HERE)
    import make_reference_outputs as golden  # noqa: E402
    import oracle  # noqa: E402
    from oracle import reference_shaders as R  # noqa: E402
    if "--lib" in sys.argv:
        R._lib = ctypes.CDLL(os.path.abspath(sys.argv[sys.argv.index("--lib") + 1]))
    elif not R.available():
        sys.exit("the reference's shaders are not built: `make -C oracle ref REFERENCE=<reference tree>` or --lib")
    out = {}
    path = make(out, oracle, R)
    np.savez_compressed(path, **out)
    print("%s: %d outputs" % (path, len([k for k in out if k.endswith(":sha256")])))
