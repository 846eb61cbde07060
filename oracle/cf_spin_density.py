"""ctypes binding of oracle/cf_spin_density.c, the CPU restatement of the spin density matrix from thermal vorticity -- TEST
INFRASTRUCTURE ONLY.

May be imported by tests/ and tools, never by the product package (is3d_b200/).  The library is compiled on first use into the system
temporary directory (named after a hash of the sources), so that a read-only tree works and a changed source is never stale.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import cf_oracle as cfo
from oracle.cf_polzn import VORTICITY_FIELDS, Vorticity, _compiler

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = ("cf_spin_density.c", "cf_polzn.c", "cf_oracle.h")
_LIB = None

SPIN_DENSITY_FIELDS = ("Snorm", "Px", "Py", "Pz", "Qxx", "Qxy", "Qxz", "Qyy", "Qyz")


def lib():
    global _LIB
    if _LIB is None:
        h = hashlib.sha256()
        for f in _SOURCES:
            with open(os.path.join(_HERE, f), "rb") as fh:
                h.update(fh.read())
        path = os.path.join(tempfile.gettempdir(), "is3d_cf_spin_density_%s_%d.so" % (h.hexdigest()[:16], os.getuid()))
        if not os.path.exists(path):
            fd, tmp = tempfile.mkstemp(suffix=".so", dir=tempfile.gettempdir())
            os.close(fd)
            subprocess.check_call([_compiler(), "-O2", "-std=gnu11", "-fPIC", "-shared", "-ffp-contract=off", "-fopenmp", "-I", _HERE,
                                   "-o", tmp, os.path.join(_HERE, "cf_spin_density.c"), "-lm"])
            os.replace(tmp, path)
        L = C.CDLL(path)
        L.cfo_spin_density.restype = C.c_int64
        L.cfo_spin_polarization.restype = C.c_int64
        _LIB = L
    return _LIB


def spin_density(flags, cells, vorticity, species, grid, conditioning=False):
    """cfo_spin_density: returns (dict of the nine raw sums Snorm, Px, Py, Pz, Qxx, Qxy, Qxz, Qyy, Qyz, flat [y][phi][pT][species];
    skipped cells) and, with conditioning=True, a third item: dict of the per-bin sums of |terms| of the nine arrays.  Raises
    RuntimeError with the oracle's code on an error (-5: a boson evaluation without a valid top-level occupation)."""
    keep = cfo._Keep()
    nb = cfo.n_bins(species, grid)
    out = np.zeros((9, nb)); A = np.zeros((9, nb)) if conditioning else None
    w = Vorticity()
    for k in VORTICITY_FIELDS:
        setattr(w, k, keep.arr(vorticity[k]))
    fl = cfo._flags(flags); c = cfo._cells(keep, cells); sp = cfo._species(keep, species); g = cfo._grid(keep, grid)
    rc = lib().cfo_spin_density(C.byref(fl), C.byref(c), C.byref(w), C.byref(sp), C.byref(g), cfo._p(out), cfo._p(A) if A is not None else None)
    if rc < 0:
        raise RuntimeError("cf_spin_density oracle error %d" % rc)
    res = {k: out[j] for j, k in enumerate(SPIN_DENSITY_FIELDS)}
    if conditioning:
        return res, int(rc), {k: A[j] for j, k in enumerate(SPIN_DENSITY_FIELDS)}
    return res, int(rc)
