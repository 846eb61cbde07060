"""ctypes binding of oracle/cf_polzn_fd.c, the CPU restatement of the feed-down of the spin-polarization sums through 2-body decays --
TEST INFRASTRUCTURE ONLY.

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
_SOURCES = ("cf_polzn_fd.c", "cf_decays.c", "cf_oracle.h")
_LIB = None
_D = C.POINTER(C.c_double)
_I = C.POINTER(C.c_int32)
FIELDS = ("St", "Sx", "Sy", "Sz", "Snorm")


def _compiler():
    return "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else (shutil.which("gcc") or "cc")


def lib():
    global _LIB
    if _LIB is None:
        h = hashlib.sha256()
        for f in _SOURCES:
            with open(os.path.join(_HERE, f), "rb") as fh:
                h.update(fh.read())
        path = os.path.join(tempfile.gettempdir(), "is3d_cf_polzn_fd_%s_%d.so" % (h.hexdigest()[:16], os.getuid()))
        if not os.path.exists(path):
            fd, tmp = tempfile.mkstemp(suffix=".so", dir=tempfile.gettempdir())
            os.close(fd)
            # the flags of oracle/Makefile's libcf_oracle.so: Snorm must round exactly like cfo_resonance_decays
            subprocess.check_call([_compiler(), "-O2", "-std=gnu11", "-fPIC", "-shared", "-ffp-contract=off", "-fopenmp", "-I", _HERE,
                                   "-o", tmp, os.path.join(_HERE, "cf_polzn_fd.c"), "-lm"])
            os.replace(tmp, path)
        L = C.CDLL(path)
        L.cfo_polarization_decays.restype = C.c_int
        L.cfo_fd_chain.restype = None
        L.cfo_fd_chain.argtypes = [_D, C.c_double, _D, C.c_int, _D, C.c_double, C.c_double, C.c_double, _D]
        _LIB = L
    return _LIB


def chain(P, M, Sp, dim2, p, mD, a, b):
    """cfo_fd_chain: the daughter's lab spin four-vector at one integrand point."""
    P = np.ascontiguousarray(P, dtype=np.float64); Sp = np.ascontiguousarray(Sp, dtype=np.float64)
    p = np.ascontiguousarray(p, dtype=np.float64); out = np.zeros(4)
    lib().cfo_fd_chain(P.ctypes.data_as(_D), float(M), Sp.ctypes.data_as(_D), int(bool(dim2)), p.ctypes.data_as(_D), float(mD), float(a), float(b),
                       out.ctypes.data_as(_D))
    return out


def polarization_decays(pdg, spin_parity, chosen_pdg_index, grid, dimension, sums, conditioning=False):
    """cfo_polarization_decays: returns the amended copy of sums (dict St, Sx, Sy, Sz, Snorm) and, with conditioning=True, a second item:
    dict St, Sx, Sy, Sz of the per-bin sums of |point contribution| x (1 + |log dN|) of the feed-down (each point's weight is exp of an
    interpolated log spectrum, so an ulp of log dN is |log dN| ulps of the contribution)."""
    keep = []

    def ia(x):
        a = np.ascontiguousarray(x, dtype=np.int32); keep.append(a)
        return a.ctypes.data_as(_I)

    def da(x):
        a = np.ascontiguousarray(x, dtype=np.float64); keep.append(a)
        return a.ctypes.data_as(_D)

    p = cfo.Particles()
    p.n_particles = len(pdg["mcid"])
    p.mcid = ia(pdg["mcid"]); p.mass = da(pdg["mass"]); p.width = da(pdg["width"]); p.stable = ia(pdg["stable"]); p.decays = ia(pdg["decays"])
    p.dec_first = ia(pdg["dec_first"]); p.dec_npart = ia(pdg["dec_npart"]); p.dec_br = da(pdg["dec_br"]); p.dec_part = ia(np.asarray(pdg["dec_part"]).ravel())
    k = cfo._Keep(); g = cfo._grid(k, grid)
    n = len(np.asarray(sums["Snorm"]))
    S = np.concatenate([np.asarray(sums[f], dtype=np.float64) for f in FIELDS])
    A = np.zeros(4 * n)
    rc = lib().cfo_polarization_decays(C.byref(p), ia(spin_parity["spin2"]), ia(spin_parity["parity"]), C.c_int32(len(chosen_pdg_index)),
                                       ia(chosen_pdg_index), C.byref(g), C.c_int32(dimension), S.ctypes.data_as(_D),
                                       A.ctypes.data_as(_D))
    if rc:
        raise RuntimeError("cf_polzn_fd oracle error %d" % rc)
    out = {f: S[i * n:(i + 1) * n].copy() for i, f in enumerate(FIELDS)}
    if conditioning:
        return out, {f: A[i * n:(i + 1) * n].copy() for i, f in enumerate(FIELDS[:4])}
    return out
