"""ctypes binding of oracle/cf_polzn_xi.c, the CPU restatement of the thermal-shear spin polarization -- TEST INFRASTRUCTURE ONLY.

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
_SOURCES = ("cf_polzn_xi.c", "cf_polzn.c", "cf_oracle.h")
_LIB = None
_D = C.POINTER(C.c_double)

THERMAL_SHEAR_FIELDS = ("xtt", "xtx", "xty", "xtn", "xxx", "xxy", "xxn", "xyy", "xyn", "xnn")


class ThermalShear(C.Structure):
    _fields_ = [("x", _D * 10)]


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
        path = os.path.join(tempfile.gettempdir(), "is3d_cf_polzn_xi_%s_%d.so" % (h.hexdigest()[:16], os.getuid()))
        if not os.path.exists(path):
            fd, tmp = tempfile.mkstemp(suffix=".so", dir=tempfile.gettempdir())
            os.close(fd)
            # the flags of oracle/cf_polzn.py: Snorm must round exactly like cfo_spin_polarization
            subprocess.check_call([_compiler(), "-O2", "-std=gnu11", "-fPIC", "-shared", "-ffp-contract=off", "-fopenmp", "-I", _HERE,
                                   "-o", tmp, os.path.join(_HERE, "cf_polzn_xi.c"), "-lm"])
            os.replace(tmp, path)
        L = C.CDLL(path)
        L.cfo_spin_polarization_shear.restype = C.c_int64
        L.cfo_cart_shear.restype = None
        L.cfo_cart_shear.argtypes = [_D, C.c_double, C.c_double, _D]
        _LIB = L
    return _LIB


def cart_shear(x, tau, eta):
    """cfo_cart_shear: the ten covariant Milne components -> (xi_tt, xi_tx, xi_ty, xi_tz, xi_xx, xi_xy, xi_xz, xi_yy, xi_yz, xi_zz)."""
    xin = np.ascontiguousarray(x, dtype=np.float64)
    out = np.zeros(10)
    lib().cfo_cart_shear(xin.ctypes.data_as(_D), float(tau), float(eta), out.ctypes.data_as(_D))
    return out


def spin_polarization_shear(flags, cells, shear, species, grid, conditioning=False):
    """cfo_spin_polarization_shear: returns (dict St, Sx, Sy, Sz, Snorm of raw sums, flat [y][phi][pT][species]; skipped cells) and,
    with conditioning=True, a third item: dict of the per-bin sums of |terms| of St, Sx, Sy, Sz."""
    keep = cfo._Keep()
    nb = cfo.n_bins(species, grid)
    N = np.zeros((4, nb)); Sn = np.zeros(nb); A = np.zeros((4, nb)) if conditioning else None
    xs = ThermalShear()
    for j, k in enumerate(THERMAL_SHEAR_FIELDS):
        xs.x[j] = keep.arr(shear[k])
    fl = cfo._flags(flags); c = cfo._cells(keep, cells); sp = cfo._species(keep, species); g = cfo._grid(keep, grid)
    rc = lib().cfo_spin_polarization_shear(C.byref(fl), C.byref(c), C.byref(xs), C.byref(sp), C.byref(g), cfo._p(N), cfo._p(Sn),
                                           cfo._p(A) if A is not None else None)
    if rc < 0:
        raise RuntimeError("cf_polzn_xi oracle error %d" % rc)
    out = dict(St=N[0], Sx=N[1], Sy=N[2], Sz=N[3], Snorm=Sn)
    if conditioning:
        return out, int(rc), dict(St=A[0], Sx=A[1], Sy=A[2], Sz=A[3])
    return out, int(rc)
