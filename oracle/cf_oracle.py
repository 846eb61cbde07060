"""ctypes binding of oracle/libcf_oracle.so -- TEST INFRASTRUCTURE ONLY.

May be imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs, never by the
product package (is3d_b200/).  Also drives the compiled reference (oracle/_ref/is3d_ref) inside a materialised
working directory.
"""
import ctypes as C
import json
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_D = C.POINTER(C.c_double)

CELL_FIELDS = ("tau", "eta", "dat", "dax", "day", "dan", "ux", "uy", "un", "T", "P", "E",
               "pixx", "pixy", "pixn", "piyy", "piyn", "bulkPi", "muB", "nB", "Vx", "Vy", "Vn",
               "pitt", "pitx", "pity", "pitn", "pinn", "Wx", "Wy", "Lambda", "aL", "c0", "c1", "c2", "c3", "c4")


class Cells(C.Structure):
    _fields_ = [("n_cells", C.c_int64)] + [(k, _D) for k in CELL_FIELDS]


class Species(C.Structure):
    _fields_ = [("n", C.c_int32), ("mass", _D), ("sign", _D), ("degeneracy", _D), ("baryon", _D)]


class Grid(C.Structure):
    _fields_ = [("n_pT", C.c_int32), ("n_phi", C.c_int32), ("n_y", C.c_int32), ("n_eta", C.c_int32),
                ("pT", _D), ("phi", _D), ("phi_weight", _D), ("y", _D), ("eta", _D), ("eta_weight", _D)]


class Flags(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("df_mode", "dimension", "include_baryon", "include_bulk", "include_shear",
                                         "include_diff", "regulate_deltaf", "outflow")] + \
               [("deta_min", C.c_double), ("mass_pion0", C.c_double)]


class DfTables(C.Structure):
    _fields_ = [("n_T", C.c_int32)] + [(k, _D) for k in ("T", "c0", "c1", "c2", "c3", "c4", "F", "G", "betabulk", "betaV", "betapi")] + \
               [("n_jonah", C.c_int32), ("jonah_x", _D), ("jonah_lambda2", _D), ("jonah_z", _D), ("bulkPi_over_Peq_max", C.c_double)]


class SpacetimeSpec(C.Structure):
    _fields_ = [("tau_min", C.c_double), ("tau_max", C.c_double), ("r_min", C.c_double), ("r_max", C.c_double),
                ("tau_bins", C.c_int32), ("r_bins", C.c_int32), ("x", _D), ("y", _D), ("pT_weight", _D)]


class Laguerre(C.Structure):
    _fields_ = [("n_points", C.c_int32), ("root1", _D), ("weight1", _D), ("root2", _D), ("weight2", _D)]


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE, "oracle"])


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "libcf_oracle.so")
        if not os.path.exists(path):
            build()
        L = C.CDLL(path)
        L.cfo_smooth_vh.restype = C.c_int64
        L.cfo_smooth_feqmod.restype = C.c_int64
        L.cfo_smooth_vah.restype = C.c_int64
        L.cfo_spacetime_vh.restype = C.c_int64
        L.cfo_spacetime_feqmod.restype = C.c_int64
        L.cfo_total_yield.restype = C.c_int64
        L.cfo_jonah_tables.restype = C.c_double
        L.cfo_aL_fit.restype = C.c_double; L.cfo_aL_fit.argtypes = [C.c_double]
        L.cfo_R200.restype = C.c_double; L.cfo_R200.argtypes = [C.c_double]
        L.cfo_spline_eval.restype = C.c_double
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(_D)


class _Keep(list):
    """keeps numpy arrays alive for the duration of a call"""

    def arr(self, x):
        a = np.ascontiguousarray(x, dtype=np.float64)
        self.append(a)
        return _p(a)


def _cells(keep, cells):
    st = Cells()
    n = len(cells["tau"])
    st.n_cells = n
    for k in CELL_FIELDS:
        if k in cells and cells[k] is not None:
            setattr(st, k, keep.arr(cells[k]))
    return st


def _species(keep, sp):
    st = Species()
    st.n = len(sp["mass"])
    for k in ("mass", "sign", "degeneracy", "baryon"):
        setattr(st, k, keep.arr(sp[k]))
    return st


def _grid(keep, g):
    st = Grid()
    st.n_pT, st.n_phi, st.n_y, st.n_eta = len(g["pT"]), len(g["phi"]), len(g["y"]), len(g["eta"])
    for k in ("pT", "phi", "phi_weight", "y", "eta", "eta_weight"):
        setattr(st, k, keep.arr(g[k]))
    return st


def _flags(fl):
    st = Flags()
    for k, _ in Flags._fields_:
        setattr(st, k, fl[k])
    return st


def _tables(keep, tab):
    st = DfTables()
    st.n_T = len(tab["T"])
    for k in ("T", "c0", "c1", "c2", "c3", "c4", "F", "G", "betabulk", "betaV", "betapi"):
        setattr(st, k, keep.arr(tab[k]))
    if tab.get("jonah_x") is not None:
        st.n_jonah = len(tab["jonah_x"])
        st.jonah_x = keep.arr(tab["jonah_x"]); st.jonah_lambda2 = keep.arr(tab["jonah_lambda2"]); st.jonah_z = keep.arr(tab["jonah_z"])
        st.bulkPi_over_Peq_max = tab["bulkPi_over_Peq_max"]
    return st


def _laguerre(keep, gla):
    st = Laguerre()
    st.n_points = len(gla["root1"])
    for k in ("root1", "weight1", "root2", "weight2"):
        setattr(st, k, keep.arr(gla[k]))
    return st


def n_bins(sp, g):
    return len(sp["mass"]) * len(g["pT"]) * len(g["phi"]) * len(g["y"])


def surface_averages(cells):
    keep = _Keep(); out = np.zeros(5)
    st = _cells(keep, cells)
    lib().cfo_surface_averages(C.byref(st), _p(out))
    return out


def jonah_tables(mass, degeneracy, sign, T_avg, gla):
    keep = _Keep()
    x = np.zeros(301); l2 = np.zeros(301); z = np.zeros(301)
    g = _laguerre(keep, gla)
    mx = lib().cfo_jonah_tables(C.c_int(len(mass)), keep.arr(mass), keep.arr(degeneracy), keep.arr(sign), C.c_double(T_avg),
                                C.byref(g), _p(x), _p(l2), _p(z))
    return dict(jonah_x=x, jonah_lambda2=l2, jonah_z=z, bulkPi_over_Peq_max=mx)


def smooth(flags, cells, species, grid, tables=None, laguerre=None, vah=False, conditioning=None):
    """Run the matching oracle kernel; returns (dN flat [y][phi][pT][species], skipped, breakdown).

    conditioning: optional zero-initialised array (df_mode 1, 2 only) that receives the per-bin magnitude sum dN_abs."""
    keep = _Keep()
    dN = np.zeros(n_bins(species, grid))
    fl = _flags(flags); c = _cells(keep, cells); sp = _species(keep, species); g = _grid(keep, grid)
    bd = C.c_int64(0)
    if vah:
        rc = lib().cfo_smooth_vah(C.byref(fl), C.byref(c), C.byref(sp), C.byref(g), _p(dN))
    elif flags["df_mode"] in (1, 2):
        t = _tables(keep, tables)
        rc = lib().cfo_smooth_vh(C.byref(fl), C.byref(c), C.byref(sp), C.byref(g), C.byref(t), _p(dN), _p(conditioning) if conditioning is not None else None)
    else:
        t = _tables(keep, tables); la = _laguerre(keep, laguerre)
        rc = lib().cfo_smooth_feqmod(C.byref(fl), C.byref(c), C.byref(sp), C.byref(g), C.byref(t), C.byref(la), _p(dN), C.byref(bd))
    if rc < 0:
        raise RuntimeError("cf_oracle error %d" % rc)
    return dN, int(rc), int(bd.value)


def spacetime(flags, cells, species, grid, tables, bins, laguerre=None):
    """operation = 0 oracle.  cells must carry "x" and "y"; bins = dict(tau_min, tau_max, tau_bins, r_min, r_max, r_bins).

    Returns (dict of raw sums dN_tau [s][tau], dN_r [s][r], dN_taur [s][tau][r], dN_dydeta [s][eta_pts], dN_dy [s]), skipped."""
    keep = _Keep()
    ns = len(species["mass"]); nt = int(bins["tau_bins"]); nr = int(bins["r_bins"])
    eta_pts = len(grid["eta"]) if flags["dimension"] == 2 else 1
    out = dict(dN_tau=np.zeros((ns, nt)), dN_r=np.zeros((ns, nr)), dN_taur=np.zeros((ns, nt, nr)),
               dN_dydeta=np.zeros((ns, eta_pts)), dN_dy=np.zeros(ns))
    spec = SpacetimeSpec()
    spec.tau_min, spec.tau_max, spec.r_min, spec.r_max = (float(bins[k]) for k in ("tau_min", "tau_max", "r_min", "r_max"))
    spec.tau_bins, spec.r_bins = nt, nr
    spec.x = keep.arr(cells["x"]); spec.y = keep.arr(cells["y"]); spec.pT_weight = keep.arr(grid["pT_weight"])
    fl = _flags(flags); c = _cells(keep, cells); sp = _species(keep, species); g = _grid(keep, grid)
    t = _tables(keep, tables)
    if flags["df_mode"] in (1, 2):
        rc = lib().cfo_spacetime_vh(C.byref(fl), C.byref(c), C.byref(sp), C.byref(g), C.byref(t), C.byref(spec),
                                    _p(out["dN_tau"]), _p(out["dN_r"]), _p(out["dN_taur"]), _p(out["dN_dydeta"]), _p(out["dN_dy"]))
    else:
        la = _laguerre(keep, laguerre); bd = C.c_int64(0)
        rc = lib().cfo_spacetime_feqmod(C.byref(fl), C.byref(c), C.byref(sp), C.byref(g), C.byref(t), C.byref(la), C.byref(spec),
                                        _p(out["dN_tau"]), _p(out["dN_r"]), _p(out["dN_taur"]), _p(out["dN_dydeta"]), _p(out["dN_dy"]),
                                        C.byref(bd))
        out["breakdown"] = int(bd.value)
    if rc < 0:
        raise RuntimeError("cf_oracle error %d" % rc)
    return out, int(rc)


def read_spacetime_files(workdir, mcid, bins, eta_pts):
    """Parse results/spacetime_distribution/*_<mcid>.dat as the reference writes them (smooth_kernels.cpp:1404-1435) and undo
    the bin-width normalisation -> the same raw sums as spacetime() (7 significant digits)."""
    nt = int(bins["tau_bins"]); nr = int(bins["r_bins"])
    tw = (bins["tau_max"] - bins["tau_min"]) / nt; rw = (bins["r_max"] - bins["r_min"]) / nr
    d = os.path.join(workdir, "results", "spacetime_distribution")
    a = np.loadtxt(os.path.join(d, "dN_taudtaudy_%d.dat" % mcid), ndmin=2)
    b = np.loadtxt(os.path.join(d, "dN_twopirdrdy_%d.dat" % mcid), ndmin=2)
    c = np.loadtxt(os.path.join(d, "dN_twopitaurdtaudrdy_%d.dat" % mcid), ndmin=2)
    e = np.loadtxt(os.path.join(d, "dN_dydeta_%d_%dpt.dat" % (mcid, eta_pts)), ndmin=2)
    tau_mid = bins["tau_min"] + tw * (np.arange(nt) + 0.5); r_mid = bins["r_min"] + rw * (np.arange(nr) + 0.5)
    out = dict(dN_tau=a[:, 1] * tau_mid * tw, dN_r=b[:, 1] * 2.0 * np.pi * r_mid * rw,
               dN_taur=(c[:, 2].reshape(nr, nt) * (2.0 * np.pi * tw * rw) * r_mid[:, None] * tau_mid[None, :]).T,
               dN_dydeta=e[:, 1], eta_column=e[:, 0], tau_mid=a[:, 0], r_mid=b[:, 0])
    return out


def particle_densities(species, avg5, df_mode, tables, gla, root3, weight3):
    """(n_eq, dn_bulk, dn_diff) per species at the surface averages avg5 = (T, E, P, muB, nB)"""
    keep = _Keep()
    n = len(species["mass"])
    neq = np.zeros(n); bulk = np.zeros(n); diff = np.zeros(n)
    t = _tables(keep, tables); la = _laguerre(keep, gla)
    rc = lib().cfo_particle_densities(C.c_int(n), keep.arr(species["mass"]), keep.arr(species["degeneracy"]), keep.arr(species["baryon"]),
                                      keep.arr(species["sign"]), keep.arr(avg5), C.c_int(df_mode), C.byref(t), C.byref(la),
                                      keep.arr(root3), keep.arr(weight3), _p(neq), _p(bulk), _p(diff))
    if rc:
        raise RuntimeError("cf_oracle error %d" % rc)
    return neq, bulk, diff


def total_yield(flags, cells, neq, bulk, tables, y_cut):
    """sampler mean yield; returns (Ntot, skipped cells)"""
    keep = _Keep()
    fl = _flags(flags); c = _cells(keep, cells); t = _tables(keep, tables)
    out = C.c_double(0.0)
    rc = lib().cfo_total_yield(C.byref(fl), C.byref(c), C.c_int(len(neq)), keep.arr(neq), keep.arr(bulk), C.byref(t), C.c_double(y_cut), C.byref(out))
    if rc < 0:
        raise RuntimeError("cf_oracle error %d" % rc)
    return out.value, int(rc)


# --------------------------------------------------------------------------- compiled reference (oracle/_ref)
def ref_binary(omp=False):
    p = os.path.join(_HERE, "_ref", "is3d_ref_omp" if omp else "is3d_ref")
    return p if os.path.exists(p) else None


def run_reference(workdir, what="kernel", omp=False, threads=None, timeout=3600):
    """Run oracle/_ref/is3d_ref inside `workdir`; returns (dN flat, info dict incl. seconds, mcid, breakdown)."""
    exe = ref_binary(omp)
    if exe is None:
        raise FileNotFoundError("oracle/_ref not built (run `make -C oracle ref` with REF or IS3D_REFERENCE naming an iS3D checkout)")
    env = dict(os.environ)
    if threads:
        env["OMP_NUM_THREADS"] = str(threads)
    out = os.path.join(workdir, "results", "dN_raw.bin")
    r = subprocess.run([exe, what, out], cwd=workdir, capture_output=True, text=True, env=env, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError("reference failed (%d): %s\n%s" % (r.returncode, r.stdout[-2000:], r.stderr[-2000:]))
    info = None
    for line in r.stdout.splitlines():
        if line.startswith("REF_JSON "):
            info = json.loads(line[len("REF_JSON "):])
        if "feqmod breaks down for" in line:
            bd = int(line.split("feqmod breaks down for")[1].split()[0])
    if info is None:
        raise RuntimeError("reference printed no REF_JSON line:\n" + r.stdout[-2000:])
    info["breakdown"] = locals().get("bd", 0)
    info["stdout"] = r.stdout
    return np.fromfile(out), info


def run_vah_reference(aL, Lambda_GeV, fixture=None):
    """c0..c4 per cell from the reference's own reader (oracle/_ref/vah_ref = DeltafReader::load_coefficients of
    src/cuda/deltafReader.cu, unmodified): returns an (n, 5) array in GeV units; cells outside the table keep the driver's
    sentinel -12345 (the reference leaves them untouched)."""
    import tempfile
    from is3d_b200 import workdir
    exe = os.path.join(_HERE, "_ref", "vah_ref")
    if not os.path.exists(exe):
        raise FileNotFoundError("oracle/_ref/vah_ref not built (run `make -C oracle ref` with REF or IS3D_REFERENCE naming an iS3D checkout)")
    aL = np.ascontiguousarray(aL, dtype=np.float64); Lam = np.ascontiguousarray(Lambda_GeV, dtype=np.float64)
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, fixture=fixture, vah=True, operation=1, mode=2, hrg_eos=1, dimension=3, df_mode=1)
        with open(os.path.join(wd, "in.bin"), "wb") as f:
            f.write(aL.tobytes()); f.write(Lam.tobytes())
        r = subprocess.run([exe, "in.bin", "out.bin"], cwd=wd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("vah_ref failed: %s" % r.stderr[-1000:])
        return np.fromfile(os.path.join(wd, "out.bin")).reshape(len(aL), 5)


# --------------------------------------------------------------------------- resonance decays (SURVEY 8f, row N3)
class Particles(C.Structure):
    _I = C.POINTER(C.c_int32)
    _fields_ = [("n_particles", C.c_int32), ("mcid", _I), ("mass", _D), ("width", _D), ("stable", _I), ("decays", _I), ("dec_first", _I),
                ("dec_npart", _I), ("dec_br", _D), ("dec_part", _I)]


def resonance_decays(pdg, chosen_pdg_index, grid, dimension, dN):
    """cfo_resonance_decays: pdg = dict from is3d_b200.tables.pdg_decay_table(); returns the amended copy of dN."""
    keep = []

    def ia(x):
        a = np.ascontiguousarray(x, dtype=np.int32); keep.append(a)
        return a.ctypes.data_as(C.POINTER(C.c_int32))

    def da(x):
        a = np.ascontiguousarray(x, dtype=np.float64); keep.append(a)
        return a.ctypes.data_as(_D)

    p = Particles()
    p.n_particles = len(pdg["mcid"])
    p.mcid = ia(pdg["mcid"]); p.mass = da(pdg["mass"]); p.width = da(pdg["width"]); p.stable = ia(pdg["stable"]); p.decays = ia(pdg["decays"])
    p.dec_first = ia(pdg["dec_first"]); p.dec_npart = ia(pdg["dec_npart"]); p.dec_br = da(pdg["dec_br"]); p.dec_part = ia(np.asarray(pdg["dec_part"]).ravel())
    k = _Keep(); g = _grid(k, grid)
    out = np.array(dN, dtype=np.float64, copy=True)
    f = lib().cfo_resonance_decays
    f.restype = C.c_int
    rc = f(C.byref(p), C.c_int32(len(chosen_pdg_index)), ia(chosen_pdg_index), C.byref(g), C.c_int32(dimension), _p(out))
    if rc:
        raise RuntimeError("cf_oracle resonance decays error %d" % rc)
    return out


def run_reference_decays(workdir_path, dN_in, timeout=3600):
    """oracle/_ref/is3d_ref_decays (the reference's do_resonance_decays behind oracle/ref_decays_prefix.h) on the spectra dN_in inside a
    materialised working directory; returns (amended spectra, info)."""
    exe = os.path.join(_HERE, "_ref", "is3d_ref_decays")
    if not os.path.exists(exe):
        raise FileNotFoundError("oracle/_ref/is3d_ref_decays not built (run `make -C oracle ref` with REF or IS3D_REFERENCE naming an iS3D checkout)")
    np.ascontiguousarray(dN_in, dtype=np.float64).tofile(os.path.join(workdir_path, "input", "spectra_in.bin"))
    out = os.path.join(workdir_path, "results", "dN_decays.bin")
    r = subprocess.run([exe, "decays", out], cwd=workdir_path, capture_output=True, text=True, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError("reference decays failed (%d): %s\n%s" % (r.returncode, r.stdout[-2000:], r.stderr[-2000:]))
    info = None
    for line in r.stdout.splitlines():
        if line.startswith("REF_JSON "):
            info = json.loads(line[len("REF_JSON "):])
    return np.fromfile(out), info
