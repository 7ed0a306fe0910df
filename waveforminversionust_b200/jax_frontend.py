"""JAX front end: the XLA FFI custom calls that replace the reference's ``jax.pure_callback(scipy_solve, ...)`` seam
(``Final_python/solve_helmholtz.py:85-93``) so that ``solve_helmholtz`` / ``fwi_loss_function`` stay traceable inside
``jax.jit`` / ``lax.scan`` (``nonlinearcg.py:172-174, 305-307``) / ``jaxopt.LBFGS``.

Reference gradient only: the handlers' plans keep the default ``UST_GRAD_REFERENCE`` linearisation; the ``gradient="discrete"``
mode of ``api`` (DESIGN.md section 7f) is not exposed through XLA.

STATUS: ``csrc/xla_ffi_shim.cc`` binds the C ABI of libustfwi.so as two XLA FFI handlers.  JAX / jaxlib are not installable
in the build image (no network), so here the shim is compiled against a test double of ``xla/ffi/api/ffi.h``
(``build_ffi(stub=True)``, ``tests/xla_ffi_stub/``) and its handlers are driven on the GPU by ``tests/test_ffi_shim.py``;
the registration and the traceable wrappers below need a real JAX and are UNTESTED.  Where JAX is installed:

    from waveforminversionust_b200 import jax_frontend
    jax_frontend.register()                                   # builds libustfwi_xla.so against jax.ffi.include_dir()
    from waveforminversionust_b200.jax_frontend import solve_helmholtz, fwi_loss_function
"""
from __future__ import annotations

import os
import subprocess

from . import build as _build

HERE = os.path.dirname(os.path.abspath(__file__))
SHIM = os.path.join(HERE, "csrc", "xla_ffi_shim.cc")
STUB_DIR = os.path.join(os.path.dirname(HERE), "tests", "xla_ffi_stub")
XLA_LIB = os.path.join(_build.LIBDIR, "libustfwi_xla.so")
STUB_LIB = os.path.join(_build.LIBDIR, "libustfwi_xla_stub.so")
CUDA_HOME = os.environ.get("CUDA_HOME", "/usr/local/cuda")


class FfiUnavailable(RuntimeError):
    pass


def xla_include_dir():
    """``jax.ffi.include_dir()`` (jax >= 0.4.38; ``jax.extend.ffi`` before that), or None when JAX is absent."""
    try:
        import jax
    except Exception:
        return None
    for mod in ("jax.ffi", "jax.extend.ffi"):
        try:
            m = __import__(mod, fromlist=["include_dir"])
            return m.include_dir()
        except Exception:
            continue
    return None


def build_ffi(include_dir=None, stub=False, force=False):
    """Compile csrc/xla_ffi_shim.cc into a shared library next to libustfwi.so and return its path.

    ``include_dir`` defaults to ``jax.ffi.include_dir()``.  ``stub=True`` compiles against the repo's test double of the XLA
    header instead (plus the frame helpers a test needs); that library exercises the shim's logic but cannot be registered
    with JAX.  Raises ``FfiUnavailable`` when neither real headers nor ``stub`` are available -- there is no silent fallback.
    """
    _build.build_library()
    if stub:
        inc, out, extra = STUB_DIR, STUB_LIB, [os.path.join(STUB_DIR, "stub_frame.cc")]
    else:
        inc = include_dir or xla_include_dir()
        if not inc or not os.path.exists(os.path.join(inc, "xla", "ffi", "api", "ffi.h")):
            raise FfiUnavailable("XLA FFI headers not found: JAX / jaxlib are not installed (jax.ffi.include_dir() is what ships "
                                 "xla/ffi/api/ffi.h); pass include_dir=..., or build_ffi(stub=True) for the test double")
        out, extra = XLA_LIB, []
    deps = [SHIM, os.path.join(HERE, "..", "include", "ustfwi.h")] + extra
    if not force and os.path.exists(out) and all(os.path.getmtime(d) <= os.path.getmtime(out) for d in deps):
        return out
    cmd = ["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-I", inc, "-I", os.path.join(CUDA_HOME, "include"), SHIM, *extra,
           "-o", out, "-L", _build.LIBDIR, "-lustfwi", "-Wl,-rpath,$ORIGIN", "-L", os.path.join(CUDA_HOME, "lib64"), "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("building the XLA FFI shim failed:\n" + r.stdout + r.stderr)
    return out


_REGISTERED = False


def register():
    """Build the shim against the real XLA headers and register both handlers as CUDA FFI targets."""
    global _REGISTERED
    if _REGISTERED:
        return
    import ctypes
    import jax
    lib = ctypes.CDLL(build_ffi())
    jax.ffi.register_ffi_target("ust_solve_helmholtz", jax.ffi.pycapsule(lib.ust_solve_helmholtz_ffi), platform="CUDA")
    jax.ffi.register_ffi_target("ust_fwi_loss_grad", jax.ffi.pycapsule(lib.ust_fwi_loss_grad_ffi), platform="CUDA")
    _REGISTERED = True


def solve_helmholtz(x, y, vel, src, f, a0, L_PML, adjoint):
    """Traceable drop-in for ``solve_helmholtz.py:21-101`` (same positional arguments, ``adjoint`` may be traced)."""
    import jax
    import jax.numpy as jnp
    register()
    Ny, Nx = vel.shape
    rhs = jnp.reshape(src, (Nx * Ny, -1)).astype(jnp.complex64)  # :78-79
    out = jax.ffi.ffi_call("ust_solve_helmholtz", jax.ShapeDtypeStruct(rhs.shape, jnp.complex64))(
        jnp.asarray(x, jnp.float32), jnp.asarray(y, jnp.float32), jnp.asarray(vel, jnp.float32), rhs,
        jnp.asarray(f, jnp.float32).reshape(1), jnp.asarray(adjoint, jnp.int32).reshape(1), a0=float(a0), L_PML=float(L_PML))
    return out.reshape(Ny, Nx, -1)  # :101


def fwi_loss_function(params, xi, yi, REC_DATA, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices, num_elements):
    """Traceable ``fwi_loss_function(...) -> (loss, grad)`` with the reference's 12 parameters
    (``fwi_loss_function.py:29-42``); ``grad`` has ``params``' shape.  ``SRC`` must be one-hot (``fwi_script.py:72-74``):
    the acquisition arrays are converted on the host once, at trace time, exactly as ``api._acquisition`` does."""
    import jax
    import jax.numpy as jnp
    import numpy as np
    from .api import _acquisition
    register()
    Ny, Nx = int(np.asarray(yi).size), int(np.asarray(xi).size)
    src_lin, rx_lin, mask = _acquisition(np.asarray(SRC), np.asarray(ind_matlab), np.asarray(mask_indices), Nx, Ny)
    fr = jnp.atleast_1d(jnp.asarray(f, jnp.float32))
    rec = jnp.asarray(REC_DATA, jnp.complex64).reshape(fr.shape[0], src_lin.size, rx_lin.size)
    loss2, grad = jax.ffi.ffi_call("ust_fwi_loss_grad", (jax.ShapeDtypeStruct((2,), jnp.float32),
                                                          jax.ShapeDtypeStruct((Ny, Nx), jnp.float32)))(
        jnp.asarray(params, jnp.float32).reshape(Ny, Nx), rec, jnp.asarray(src_lin), jnp.asarray(rx_lin), jnp.asarray(mask),
        jnp.asarray(xi, jnp.float32), jnp.asarray(yi, jnp.float32), fr, a0=float(a0), L_PML=float(L_PML))
    return loss2[0] + loss2[1], grad.reshape(jnp.shape(params))
