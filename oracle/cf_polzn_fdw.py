"""ctypes binding of oracle/cf_polzn_fdw.c, the CPU restatement of the feed-down of the spin-polarization sums through weak 2-body decays
-- TEST INFRASTRUCTURE ONLY.

May be imported by tests/ and tools, never by the product package (is3d_b200/).  The library is compiled on first use into the system
temporary directory, named after a hash of the sources, so that a read-only tree works and a changed source is never stale.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import cf_oracle as cfo
from oracle import cf_polzn_fd as fdo

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = ("cf_polzn_fdw.c", "cf_polzn_fd.c", "cf_decays.c", "cf_oracle.h")
_LIB = None
_D = C.POINTER(C.c_double)
_I = C.POINTER(C.c_int32)
FIELDS = fdo.FIELDS
WEAK_COLUMNS = ("parent", "daughter", "partner", "branching", "alpha", "phi")


def lib():
    global _LIB
    if _LIB is None:
        h = hashlib.sha256()
        for f in _SOURCES:
            with open(os.path.join(_HERE, f), "rb") as fh:
                h.update(fh.read())
        path = os.path.join(tempfile.gettempdir(), "is3d_cf_polzn_fdw_%s_%d.so" % (h.hexdigest()[:16], os.getuid()))
        if not os.path.exists(path):
            fd, tmp = tempfile.mkstemp(suffix=".so", dir=tempfile.gettempdir())
            os.close(fd)
            subprocess.check_call([fdo._compiler(), "-O2", "-std=gnu11", "-fPIC", "-shared", "-ffp-contract=off", "-fopenmp", "-I", _HERE,
                                   "-o", tmp, os.path.join(_HERE, "cf_polzn_fdw.c"), "-lm"])
            os.replace(tmp, path)
        L = C.CDLL(path)
        L.cfo_polarization_weak_decays.restype = C.c_int
        L.cfo_fdw_chain.restype = None
        L.cfo_fdw_chain.argtypes = [_D, C.c_double, _D, C.c_int, _D, C.c_double, C.c_double, C.c_double, C.c_double, _D, _D]
        _LIB = L
    return _LIB


def chain(P, M, Sp, dim2, p, mD, alpha, beta, gamma):
    """cfo_fdw_chain: (the daughter's lab spin numerator four-vector, the yield 1 + 2 alpha S.n) at one integrand point."""
    P = np.ascontiguousarray(P, dtype=np.float64); Sp = np.ascontiguousarray(Sp, dtype=np.float64)
    p = np.ascontiguousarray(p, dtype=np.float64); out = np.zeros(4); y = C.c_double(0.0)
    lib().cfo_fdw_chain(P.ctypes.data_as(_D), float(M), Sp.ctypes.data_as(_D), int(bool(dim2)), p.ctypes.data_as(_D), float(mD), float(alpha),
                        float(beta), float(gamma), out.ctypes.data_as(_D), C.byref(y))
    return out, y.value


def _particles(pdg, ia, da):
    p = cfo.Particles()
    p.n_particles = len(pdg["mcid"])
    p.mcid = ia(pdg["mcid"]); p.mass = da(pdg["mass"]); p.width = da(pdg["width"]); p.stable = ia(pdg["stable"]); p.decays = ia(pdg["decays"])
    p.dec_first = ia(pdg["dec_first"]); p.dec_npart = ia(pdg["dec_npart"]); p.dec_br = da(pdg["dec_br"]); p.dec_part = ia(np.asarray(pdg["dec_part"]).ravel())
    return p


def polarization_weak_decays(pdg, spin_parity, weak, chosen_pdg_index, grid, dimension, sums, conditioning=False):
    """cfo_polarization_weak_decays: returns the amended copy of sums (dict St, Sx, Sy, Sz, Snorm) and, with conditioning=True, a second
    item: dict of the five per-bin sums of |point contribution| x (1 + |log dN|) of the feed-down.  weak: dict of the six columns."""
    keep = []

    def ia(x):
        a = np.ascontiguousarray(x, dtype=np.int32); keep.append(a)
        return a.ctypes.data_as(_I)

    def da(x):
        a = np.ascontiguousarray(x, dtype=np.float64); keep.append(a)
        return a.ctypes.data_as(_D)

    p = _particles(pdg, ia, da)
    k = cfo._Keep(); g = cfo._grid(k, grid)
    n = len(np.asarray(sums["Snorm"]))
    S = np.concatenate([np.asarray(sums[f], dtype=np.float64) for f in FIELDS])
    A = np.zeros(5 * n)
    rows = len(np.atleast_1d(weak["parent"]))
    rc = lib().cfo_polarization_weak_decays(C.byref(p), ia(spin_parity["spin2"]), C.c_int32(rows), ia(weak["parent"]), ia(weak["daughter"]),
                                            ia(weak["partner"]), da(weak["branching"]), da(weak["alpha"]), da(weak["phi"]),
                                            C.c_int32(len(chosen_pdg_index)), ia(chosen_pdg_index), C.byref(g), C.c_int32(dimension),
                                            S.ctypes.data_as(_D), A.ctypes.data_as(_D))
    if rc:
        raise RuntimeError("cf_polzn_fdw oracle error %d" % rc)
    out = {f: S[i * n:(i + 1) * n].copy() for i, f in enumerate(FIELDS)}
    if conditioning:
        return out, {f: A[i * n:(i + 1) * n].copy() for i, f in enumerate(FIELDS)}
    return out

