"""ctypes binding of oracle/cf_polzn_she.c, the CPU restatement of the spin Hall spin polarization -- TEST INFRASTRUCTURE ONLY.

May be imported by tests/ and tools, never by the product package (is3d_b200/).  The library is compiled on first use into the system
temporary directory (named after a hash of the sources), so that a read-only tree works and a changed source is never stale.
"""
import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle import cf_oracle as cfo

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = ("cf_polzn_she.c", "cf_polzn.c", "cf_oracle.h")
_LIB = None
_D = C.POINTER(C.c_double)

BARYON_GRADIENT_FIELDS = ("dt", "dx", "dy", "dn")


class BaryonGradient(C.Structure):
    _fields_ = [("d", _D * 4)]


def _compiler():
    # the distro compiler: it has libgomp (oracle/Makefile uses the same rule)
    return "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else (shutil.which("gcc") or "cc")


def lib():
    global _LIB
    if _LIB is None:
        h = hashlib.sha256()
        for f in _SOURCES:
            with open(os.path.join(_HERE, f), "rb") as fh:
                h.update(fh.read())
        path = os.path.join(tempfile.gettempdir(), "is3d_cf_polzn_she_%s_%d.so" % (h.hexdigest()[:16], os.getuid()))
        if not os.path.exists(path):
            fd, tmp = tempfile.mkstemp(suffix=".so", dir=tempfile.gettempdir())
            os.close(fd)
            # the flags of oracle/cf_polzn.py: Snorm must round exactly like cfo_spin_polarization
            subprocess.check_call([_compiler(), "-O2", "-std=gnu11", "-fPIC", "-shared", "-ffp-contract=off", "-fopenmp", "-I", _HERE,
                                   "-o", tmp, os.path.join(_HERE, "cf_polzn_she.c"), "-lm"])
            os.replace(tmp, path)
        L = C.CDLL(path)
        L.cfo_spin_polarization_spin_hall.restype = C.c_int64
        L.cfo_cart_gradient.restype = None
        L.cfo_cart_gradient.argtypes = [_D, C.c_double, C.c_double, _D]
        _LIB = L
    return _LIB


def cart_gradient(d, tau, eta):
    """cfo_cart_gradient: the four covariant Milne components (d_tau, d_x, d_y, d_eta) -> Cartesian (d_t, d_x, d_y, d_z)."""
    din = np.ascontiguousarray(d, dtype=np.float64)
    out = np.zeros(4)
    lib().cfo_cart_gradient(din.ctypes.data_as(_D), float(tau), float(eta), out.ctypes.data_as(_D))
    return out


def spin_polarization_spin_hall(flags, cells, gradient, species, grid, conditioning=False):
    """cfo_spin_polarization_spin_hall: returns (dict St, Sx, Sy, Sz, Snorm of raw sums, flat [y][phi][pT][species]; skipped cells) and,
    with conditioning=True, a third item: dict of the per-bin sums of |terms| of St, Sx, Sy, Sz.  species needs 'baryon'."""
    keep = cfo._Keep()
    nb = cfo.n_bins(species, grid)
    N = np.zeros((4, nb)); Sn = np.zeros(nb); A = np.zeros((4, nb)) if conditioning else None
    gb = BaryonGradient()
    for j, k in enumerate(BARYON_GRADIENT_FIELDS):
        gb.d[j] = keep.arr(gradient[k])
    fl = cfo._flags(flags); c = cfo._cells(keep, cells); sp = cfo._species(keep, species); g = cfo._grid(keep, grid)
    rc = lib().cfo_spin_polarization_spin_hall(C.byref(fl), C.byref(c), C.byref(gb), C.byref(sp), C.byref(g), cfo._p(N), cfo._p(Sn),
                                               cfo._p(A) if A is not None else None)
    if rc < 0:
        raise RuntimeError("cf_polzn_she oracle error %d" % rc)
    out = dict(St=N[0], Sx=N[1], Sy=N[2], Sz=N[3], Snorm=Sn)
    if conditioning:
        return out, int(rc), dict(St=A[0], Sx=A[1], Sy=A[2], Sz=A[3])
    return out, int(rc)
