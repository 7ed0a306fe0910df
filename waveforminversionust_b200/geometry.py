"""Ring-array acquisition geometry and synthetic sound-speed models.

Host-side input construction mirroring ``fwi_script.py:31-85`` (mask of excluded
receivers, grid, nearest-node element snapping, ``ind_matlab``, one-hot ``SRC``,
``mask_indices``) and the synthetic-benchmark recipe of SURVEY.md section 8(d)
(``SimulateData.m:7-62``: ring of radius 110 mm, elements at theta_k = -pi + 2 pi k/E).
Pure NumPy; no device work happens here.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np


@dataclass
class RingGeometry:
    xi: np.ndarray  # (Nx,) grid x coordinates
    yi: np.ndarray  # (Ny,) grid y coordinates
    x_idx: np.ndarray  # (E,) grid column of each element
    y_idx: np.ndarray  # (E,) grid row of each element
    # (E,) x_idx*Ny + y_idx: the column-major (order='F') index of a (Ny, Nx) field, which api._acquisition decodes.  The
    # reference writes x_idx*Nxi + y_idx (fwi_script.py:68), which is the same only on square grids.
    ind_matlab: np.ndarray
    tx_include: np.ndarray  # (Nt,) transmitting elements               fwi_script.py:35
    mask_indices: np.ndarray  # (Nt, Nm) receivers kept per transmitter fwi_script.py:79-85
    num_elements: int
    a0: float
    L_PML: float

    @property
    def Nx(self):
        return self.xi.size

    @property
    def Ny(self):
        return self.yi.size

    @property
    def src_lin(self):
        """Row-major node index y*Nx + x of each transmitter's one-hot source."""
        t = self.tx_include
        return (self.y_idx[t] * self.Nx + self.x_idx[t]).astype(np.int32)

    def dense_src(self, dtype=np.complex64):
        """(Ny, Nx, Nt) one-hot source array, ``fwi_script.py:72-74``."""
        S = np.zeros((self.Ny, self.Nx, self.tx_include.size), dtype=dtype)
        for i, t in enumerate(self.tx_include):
            S[self.y_idx[t], self.x_idx[t], i] = 1.0
        return S


def build_masks(num_elements, tx_include, num_elem_lr):
    """Receivers kept per transmitter: all but tx +- num_elem_lr (``fwi_script.py:39-44, 79-85``)."""
    ar = np.arange(-num_elem_lr, num_elem_lr + 1)
    inc = np.ones((num_elements, num_elements), dtype=bool)
    for tx in range(num_elements):
        inc[tx, (ar + tx) % num_elements] = False
    return np.stack([np.nonzero(inc[t])[0] for t in tx_include], axis=0).astype(np.int64)


def snap_elements(xi, yi, x_circ, y_circ):
    """Nearest grid node of each element by argmin (``fwi_script.py:65-66``)."""
    x_idx = np.argmin(np.abs(xi[None, :] - np.asarray(x_circ).ravel()[:, None]), axis=1)
    y_idx = np.argmin(np.abs(yi[None, :] - np.asarray(y_circ).ravel()[:, None]), axis=1)
    return x_idx, y_idx


def ring_geometry(n, num_elements=256, dwnsmp=1, xmax=0.12, radius=0.110, a0=10.0, pml_cells=11.25,
                  num_elem_lr=None, dtype=np.float32):
    """Synthetic n x n configuration of SURVEY.md 8(d): domain [-xmax, xmax]^2, ring of
    ``num_elements`` at ``radius``, L_PML = pml_cells*h, exclusion +-floor(31*E/256)."""
    xi = np.linspace(-xmax, xmax, n).astype(dtype)
    yi = xi.copy()
    h = 2 * xmax / (n - 1)
    theta = -np.pi + 2 * np.pi * np.arange(num_elements) / num_elements  # SimulateData.m:15-19
    x_circ, y_circ = radius * np.cos(theta), radius * np.sin(theta)
    x_idx, y_idx = snap_elements(xi.astype(np.float64), yi.astype(np.float64), x_circ, y_circ)
    if num_elem_lr is None:
        num_elem_lr = (31 * num_elements) // 256
    tx_include = np.arange(0, num_elements, dwnsmp)
    mask_indices = build_masks(num_elements, tx_include, num_elem_lr)
    return RingGeometry(xi=xi, yi=yi, x_idx=x_idx, y_idx=y_idx, ind_matlab=x_idx * n + y_idx,
                        tx_include=tx_include, mask_indices=mask_indices, num_elements=num_elements,
                        a0=float(a0), L_PML=float(pml_cells * h))


def blob_model(geom, c0=1500.0, dc=60.0, nblobs=5, seed=1234, r_max=0.09):
    """Smooth synthetic sound-speed map: background c0 plus ``nblobs`` Gaussian inclusions of
    amplitude up to +-dc inside radius r_max (SURVEY.md 8(d))."""
    rng = np.random.default_rng(seed)
    X, Y = np.meshgrid(geom.xi.astype(np.float64), geom.yi.astype(np.float64), indexing="xy")
    c = np.full(X.shape, c0)
    for _ in range(nblobs):
        r = 0.6 * r_max * np.sqrt(rng.uniform())
        th = rng.uniform(0, 2 * np.pi)
        sig = rng.uniform(5e-3, 15e-3)
        amp = dc * rng.uniform(-1, 1)
        c += amp * np.exp(-((X - r * np.cos(th)) ** 2 + (Y - r * np.sin(th)) ** 2) / (2 * sig**2))
    return c


# alpha0 [dB/(cm MHz)] of the attenuation slowness kappa [s/m]: the amplitude attenuation is alpha(f) = 2 pi f kappa Np/m
# (complex slowness s - i kappa), and 1 Np = 20/ln(10) dB, 1 m = 100 cm, f in MHz = f / 1e6
DB_CM_MHZ_PER_KAPPA = 2.0 * np.pi * 1e6 * (20.0 / np.log(10.0)) / 100.0  # ~5.458e5


def db_cm_mhz_to_kappa(alpha0):
    """Attenuation slowness kappa (s/m) of an attenuation coefficient ``alpha0`` in dB/(cm MHz) (linear in frequency)."""
    return np.asarray(alpha0, dtype=np.float64) / DB_CM_MHZ_PER_KAPPA


def kappa_to_db_cm_mhz(kappa):
    """Inverse of ``db_cm_mhz_to_kappa``."""
    return np.asarray(kappa, dtype=np.float64) * DB_CM_MHZ_PER_KAPPA


def attenuation_blob_model(geom, alpha0=0.0, dalpha=0.5, nblobs=5, seed=4321, r_max=0.09):
    """Smooth synthetic attenuation map, built like ``blob_model``: attenuation slowness kappa (s/m) of a background
    ``alpha0`` dB/(cm MHz) plus ``nblobs`` Gaussian inclusions of ``dalpha`` times U(0.5, 1) dB/(cm MHz) (non-negative, so
    kappa >= 0 everywhere) inside radius r_max."""
    rng = np.random.default_rng(seed)
    X, Y = np.meshgrid(geom.xi.astype(np.float64), geom.yi.astype(np.float64), indexing="xy")
    a = np.full(X.shape, float(alpha0))
    for _ in range(nblobs):
        r = 0.6 * r_max * np.sqrt(rng.uniform())
        th = rng.uniform(0, 2 * np.pi)
        sig = rng.uniform(5e-3, 15e-3)
        amp = dalpha * rng.uniform(0.5, 1.0)
        a += amp * np.exp(-((X - r * np.cos(th)) ** 2 + (Y - r * np.sin(th)) ** 2) / (2 * sig**2))
    return db_cm_mhz_to_kappa(a)


def source_amplitudes(nt, seed=1234):
    """Per-source random complex amplitude (``SimulateData.m:26``)."""
    rng = np.random.default_rng(seed)
    return rng.standard_normal(nt) + 1j * rng.standard_normal(nt)


def frequency_for_grid(n, xmax=0.12, c_ref=1480.0, ppw=5.29):
    """Frequency keeping ``ppw`` grid points per wavelength at c_ref (cfg1 has 5.29)."""
    h = 2 * xmax / (n - 1)
    return c_ref / (ppw * h)
