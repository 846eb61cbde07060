"""ctypes binding of oracle/cf_hbt.c, the CPU restatement of the HBT moments of the emission function -- TEST INFRASTRUCTURE ONLY.

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
_SOURCES = ("cf_hbt.c", "cf_oracle.c", "cf_oracle.h")
_LIB = None

HBT_FIELDS = ("S0", "So", "Ss", "Sl", "Soo", "Sss", "Sll", "Sos", "Sol", "Ssl")


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
        path = os.path.join(tempfile.gettempdir(), "is3d_cf_hbt_%s_%d.so" % (h.hexdigest()[:16], os.getuid()))
        if not os.path.exists(path):
            fd, tmp = tempfile.mkstemp(suffix=".so", dir=tempfile.gettempdir())
            os.close(fd)
            # the flags of libcf_oracle.so (oracle/Makefile): S0 must round exactly like cfo_smooth_vh
            subprocess.check_call([_compiler(), "-O2", "-std=gnu11", "-fPIC", "-shared", "-ffp-contract=off", "-fopenmp", "-I", _HERE,
                                   "-o", tmp, os.path.join(_HERE, "cf_hbt.c"), "-lm"])
            os.replace(tmp, path)
        L = C.CDLL(path)
        L.cfo_hbt_moments.restype = C.c_int64
        _LIB = L
    return _LIB


def hbt_moments(flags, cells, species, grid, tables, conditioning=False):
    """cfo_hbt_moments: returns (dict S0 .. Ssl of raw sums, flat [y][phi][pT][species]; skipped cells) and, with conditioning=True,
    a third item: dict of the per-bin sums of |terms| of every array.  cells must carry "x" and "y"."""
    keep = cfo._Keep()
    nb = cfo.n_bins(species, grid)
    S = np.zeros((10, nb)); A = np.zeros((10, nb)) if conditioning else None
    fl = cfo._flags(flags); c = cfo._cells(keep, cells); sp = cfo._species(keep, species); g = cfo._grid(keep, grid)
    t = cfo._tables(keep, tables)
    rc = lib().cfo_hbt_moments(C.byref(fl), C.byref(c), keep.arr(cells["x"]), keep.arr(cells["y"]), C.byref(sp), C.byref(g), C.byref(t),
                               cfo._p(S), cfo._p(A) if A is not None else None)
    if rc < 0:
        raise RuntimeError("cf_hbt oracle error %d" % rc)
    out = {k: S[q] for q, k in enumerate(HBT_FIELDS)}
    if conditioning:
        return out, int(rc), {k: A[q] for q, k in enumerate(HBT_FIELDS)}
    return out, int(rc)
