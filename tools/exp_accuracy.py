#!/usr/bin/env python
"""Wavefield accuracy of the complex64 engines at a benchmark grid size against the complex128 oracle, under a set of
environment toggles (one subprocess each): which kernel variant / constant moves the error.

    python tools/exp_accuracy.py [n] [nrhs]
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHILD = r"""
import os, sys
import numpy as np
sys.path.insert(0, %r); sys.path.insert(0, os.path.join(%r, "tests"))
import waveforminversionust_b200 as w
from waveforminversionust_b200 import geometry as G
n, nrhs, engine = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3]
d = np.load(sys.argv[4])
geom = G.ring_geometry(n, 256)
f = G.frequency_for_grid(n)
vel, src, bde = d["vel"], d["src"], tuple(d["bde"])
inner = (slice(1, -1), slice(1, -1))
out = []
for adjoint in (False, True):
    truth = d["adj" if adjoint else "fwd"]
    got = w.solve_helmholtz(geom.xi, geom.yi, vel, src, f, geom.a0, geom.L_PML, adjoint, dtype="c64", bde=bde, engine=engine)
    e = np.linalg.norm((got[inner] - truth[inner]).ravel()) / np.linalg.norm(truth[inner].ravel())
    out.append("%%.3e" %% e)
print(" ".join(out))
""" % (ROOT, ROOT)


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 512
    nrhs = int(sys.argv[2]) if len(sys.argv) > 2 else 8
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    from common import bde_for
    from oracle import helmholtz as oh
    from waveforminversionust_b200 import geometry as G
    geom = G.ring_geometry(n, 256)
    f = G.frequency_for_grid(n)
    vel = G.blob_model(geom).astype(np.float32)
    bde = bde_for(geom, vel, f)
    src = geom.dense_src(np.complex64)[:, :, ::256 // nrhs]
    fac = oh.HelmholtzFactor(geom.xi, geom.yi, vel.astype(np.float64), f, geom.a0, geom.L_PML, "c128", bde=bde)
    path = "/tmp/exp_accuracy_truth.npz"
    np.savez(path, vel=vel, src=src, bde=np.array(bde), fwd=fac.solve(src.astype(np.complex128), False),
             adj=fac.solve(src.astype(np.complex128), True))
    cases = [("simt", {}), ("tc2", {}), ("tc2", {"UST_NO_LOOKAHEAD": "1"}), ("tc2", {"UST_TC2_BIAS_FIX": "0"}),
             ("tc2", {"UST_TC2_BIAS_FIX": "2.0e-8"}), ("tc2", {"UST_TC2_BIAS_FIX": "3.0e-8"})]
    for engine, env in cases:
        r = subprocess.run([sys.executable, "-c", CHILD, str(n), str(nrhs), engine, path], env=dict(os.environ, **env),
                           capture_output=True, text=True)
        print(f"n={n} {engine:5s} {env}: forward / adjoint interior error {r.stdout.strip() or r.stderr[-300:]}", flush=True)


if __name__ == "__main__":
    main()
