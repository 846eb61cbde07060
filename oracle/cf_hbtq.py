"""ctypes binding of oracle/cf_hbtq.c, the CPU restatement of the HBT Fourier sums of the emission function -- TEST INFRASTRUCTURE ONLY.

May be imported by tests/ and tools, never by the product package (is3d_b200/).  The library is compiled on first use into the system
temporary directory (named after a hash of the sources), so that a read-only tree works and a changed source is never stale.  It also
exports cfo_hbt_moments (the same translation unit), bound by hbt_moments() here.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import cf_hbt
from oracle import cf_oracle as cfo

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = ("cf_hbtq.c", "cf_hbt.c", "cf_oracle.c", "cf_oracle.h")
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        h = hashlib.sha256()
        for f in _SOURCES:
            with open(os.path.join(_HERE, f), "rb") as fh:
                h.update(fh.read())
        path = os.path.join(tempfile.gettempdir(), "is3d_cf_hbtq_%s_%d.so" % (h.hexdigest()[:16], os.getuid()))
        if not os.path.exists(path):
            fd, tmp = tempfile.mkstemp(suffix=".so", dir=tempfile.gettempdir())
            os.close(fd)
            # the flags of libcf_oracle.so (oracle/Makefile): Re[d][0] must round exactly like cfo_smooth_vh
            subprocess.check_call([cf_hbt._compiler(), "-O2", "-std=gnu11", "-fPIC", "-shared", "-ffp-contract=off", "-fopenmp", "-I", _HERE,
                                   "-o", tmp, os.path.join(_HERE, "cf_hbtq.c"), "-lm"])
            os.replace(tmp, path)
        L = C.CDLL(path)
        L.cfo_hbt_fourier.restype = C.c_int64
        L.cfo_hbt_moments.restype = C.c_int64
        _LIB = L
    return _LIB


def hbt_fourier(flags, cells, species, grid, tables, qrays):
    """cfo_hbt_fourier: returns (dict Re, Im of raw sums, shape (n_dir, n_q, n_bins), bins flat [y][phi][pT][species]; skipped cells;
    per-bin sum of the weight's |terms| magnitude, shape (n_bins,)).  cells must carry "x" and "y"; qrays: dict dir (n_dir x 3), dq, n_q."""
    keep = cfo._Keep()
    nb = cfo.n_bins(species, grid)
    d = np.ascontiguousarray(np.asarray(qrays["dir"], dtype=np.float64).reshape(-1, 3))
    n_dir, n_q = d.shape[0], int(qrays["n_q"])
    Re = np.zeros((n_dir, n_q, nb)); Im = np.zeros_like(Re); A = np.zeros(nb)
    fl = cfo._flags(flags); c = cfo._cells(keep, cells); sp = cfo._species(keep, species); g = cfo._grid(keep, grid)
    t = cfo._tables(keep, tables)
    rc = lib().cfo_hbt_fourier(C.byref(fl), C.byref(c), keep.arr(cells["x"]), keep.arr(cells["y"]), C.byref(sp), C.byref(g), C.byref(t),
                               C.c_int(n_dir), C.c_int(n_q), C.c_double(float(qrays["dq"])), cfo._p(d), cfo._p(Re), cfo._p(Im), cfo._p(A))
    if rc < 0:
        raise RuntimeError("cf_hbtq oracle error %d" % rc)
    return dict(Re=Re, Im=Im), int(rc), A


def hbt_moments(flags, cells, species, grid, tables):
    """cfo_hbt_moments of this library (the translation unit of cfo_hbt_fourier): dict S0 .. Ssl of raw sums."""
    keep = cfo._Keep()
    S = np.zeros((10, cfo.n_bins(species, grid)))
    fl = cfo._flags(flags); c = cfo._cells(keep, cells); sp = cfo._species(keep, species); g = cfo._grid(keep, grid)
    t = cfo._tables(keep, tables)
    rc = lib().cfo_hbt_moments(C.byref(fl), C.byref(c), keep.arr(cells["x"]), keep.arr(cells["y"]), C.byref(sp), C.byref(g), C.byref(t),
                               cfo._p(S), None)
    if rc < 0:
        raise RuntimeError("cf_hbt oracle error %d" % rc)
    return {k: S[q] for q, k in enumerate(cf_hbt.HBT_FIELDS)}
