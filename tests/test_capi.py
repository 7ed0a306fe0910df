"""CPU tests of the boundary: libustfwi.so loads and exports every symbol include/ustfwi.h declares
(no compute calls without a GPU), and the host-side conversions of the reference's arrays."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    txt = open(os.path.join(ROOT, "include", "ustfwi.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(ust_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as ge
    ge.build()
    from waveforminversionust_b200 import _lib
    L = _lib.lib()
    syms = _header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/ustfwi.h but not exported"
    assert sorted(_lib.EXPORTS) == syms
    assert b"sm_100a" in L.ust_version()


def test_library_is_built_for_sm100a_only():
    from waveforminversionust_b200 import build
    import subprocess
    cuobjdump = os.path.join(os.path.dirname(os.path.realpath(build._nvcc())), "cuobjdump")  # the toolkit that built the library, on PATH or not
    out = subprocess.run([cuobjdump, "-lelf", build.LIBPATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_calls_fail_loudly_without_a_device_or_with_bad_arguments():
    import torch
    from waveforminversionust_b200 import _lib
    L = _lib.lib()
    h = ctypes.c_void_p()
    desc = _lib.PlanDesc(3, 3, 0, 1, 1, 0, 0, 0, 0)
    assert L.ust_plan_create(ctypes.byref(desc), ctypes.byref(h)) != 0
    assert b"5x5" in L.ust_last_error()
    if not torch.cuda.is_available():
        desc = _lib.PlanDesc(32, 32, 0, 1, 1, 0, 0, 0, 0)
        assert L.ust_plan_create(ctypes.byref(desc), ctypes.byref(h)) != 0  # no CPU fallback
        assert len(L.ust_last_error()) > 0
        from waveforminversionust_b200 import HelmholtzPlan
        with pytest.raises(_lib.UstError):
            HelmholtzPlan(32, 32)
    assert L.ust_solve(None, 0, None, 1, 0, None) != 0
    assert L.ust_plan_destroy(None) == 0
    # ust_idtft validates its arguments before touching the device
    one = (ctypes.c_double * 1)(1.0)
    assert L.ust_idtft(0, None, 1, 1, one, one, 1.0, one, 1, None, None) != 0 and b"null" in L.ust_last_error()
    buf = ctypes.create_string_buffer(16)
    assert L.ust_idtft(0, buf, 0, 1, one, one, 1.0, one, 1, buf, None) != 0 and b"empty" in L.ust_last_error()
    assert L.ust_idtft(7, buf, 1, 1, one, one, 1.0, one, 1, buf, None) != 0 and b"dtype" in L.ust_last_error()


def test_acquisition_conversion_matches_reference_indexing():
    """ind_matlab (fwi_script.py:68) indexes the order='F' flattening; the C ABI takes row-major nodes."""
    from waveforminversionust_b200 import api, geometry as G
    geom = G.ring_geometry(37, 16)
    src_lin, rx_lin, mask = api._acquisition(geom.dense_src(), geom.ind_matlab, geom.mask_indices, 37, 37)
    assert np.array_equal(src_lin, geom.src_lin)
    W = np.arange(37 * 37, dtype=np.float64).reshape(37, 37)  # W[y, x] = row-major node id
    assert np.array_equal(W.ravel(order="F")[geom.ind_matlab], rx_lin)
    assert np.array_equal(mask, geom.mask_indices)
    src_lin2, _, _ = api._acquisition(api.OneHotSources(geom.src_lin, (37, 37, 16)), geom.ind_matlab, geom.mask_indices, 37, 37)
    assert np.array_equal(src_lin2, src_lin)
    bad = geom.dense_src()
    bad[5, 5, 0] = 2.0
    with pytest.raises(NotImplementedError):
        api._acquisition(bad, geom.ind_matlab, geom.mask_indices, 37, 37)


def test_geometry_follows_fwi_script():
    from waveforminversionust_b200 import geometry as G
    geom = G.ring_geometry(301, 256)
    assert geom.mask_indices.shape == (256, 193)  # 256 - 63 excluded (fwi_script.py:39-44)
    assert 0 not in geom.mask_indices[0] and 31 not in geom.mask_indices[0] and 32 in geom.mask_indices[0]
    assert 225 not in geom.mask_indices[0] and 224 in geom.mask_indices[0]
    r = np.hypot(geom.xi[geom.x_idx], geom.yi[geom.y_idx])
    assert np.all(np.abs(r - 0.110) < 1e-3)
    S = geom.dense_src()
    assert S.shape == (301, 301, 256) and S.sum() == 256
    assert np.all(geom.x_idx > 0) and np.all(geom.x_idx < 300)
    sub = G.ring_geometry(64, 32, dwnsmp=2)
    assert sub.tx_include.size == 16 and sub.mask_indices.shape[0] == 16
