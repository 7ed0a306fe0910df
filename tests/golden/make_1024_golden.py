"""Known answers at the cfg4 grid size (BASELINE configs[3]: 1024 x 1024 grid, 1024-element ring) from the complex128 oracle.
    python tests/golden/make_1024_golden.py          # ~12 min, 12 GB: one SuperLU factorisation of the 1 M-unknown operator
The oracle is too slow at this size to run inside the GPU test suite, so its wavefields for 8 of the 1024 sources (forward and
adjoint) are sampled -- every ring-element node, three full grid rows, the field norms -- and committed; tests/test_gpu_parity.py
holds the CUDA path (complex64 and complex128) to them."""
import io
import os
import sys
import time
import zipfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from common import bde_for  # noqa: E402
from oracle import helmholtz as oh  # noqa: E402
from waveforminversionust_b200 import geometry as G  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
ROWS = (100, 512, 900)

if __name__ == "__main__":
    n, nelem, stride = 1024, 1024, 128
    geom = G.ring_geometry(n, nelem)
    f = G.frequency_for_grid(n)
    vel = G.blob_model(geom).astype(np.float32)  # the float32 map both precisions of the CUDA path receive
    bde = bde_for(geom, vel, f)
    t0 = time.time()
    fac = oh.HelmholtzFactor(geom.xi, geom.yi, vel.astype(np.float64), f, geom.a0, geom.L_PML, "c128", bde=bde)
    print("factor %.0f s" % (time.time() - t0), flush=True)
    src = geom.dense_src(np.complex128)[:, :, ::stride]
    out = {}
    for adj, key in ((False, "fwd"), (True, "adj")):
        u = fac.solve(src, adj, threads=8)
        out["at_elements_" + key] = u[geom.y_idx, geom.x_idx, :]
        out["rows_" + key] = u[list(ROWS), :, :]
        out["norm_" + key] = np.linalg.norm(u.reshape(-1, u.shape[2]), axis=0)
        out["norm_interior_" + key] = np.linalg.norm(u[1:-1, 1:-1].reshape(-1, u.shape[2]), axis=0)
        print(key, out["norm_" + key], flush=True)
    out.update(n=n, nelem=nelem, stride=stride, f=f, bde=np.array(bde), rows=np.array(ROWS))
    # an .npz with LZMA members (np.load reads them): deflate leaves the complex128 samples just over 1 MB
    with zipfile.ZipFile(os.path.join(HERE, "cfg4_1024_wavefields.npz"), "w", compression=zipfile.ZIP_LZMA) as zf:
        for k, v in out.items():
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(v))
            zf.writestr(k + ".npy", buf.getvalue())
    print("done %.0f s" % (time.time() - t0))
