"""ctypes binding of the C ABI in include/is3d_b200.h (is3d_b200/libis3d_b200.so).

This is the host-side mirror used by tests, bench.py and the torch.distributed driver: it only marshals pointers.
The library is built in-tree by `is3d_b200.build`; if it is missing, or no CUDA device is present, calls fail loudly
-- there is no CPU fallback anywhere in this package.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libis3d_b200.so")
_D = C.POINTER(C.c_double)

SURFACE_FIELDS = ("tau", "eta", "dat", "dax", "day", "dan", "ux", "uy", "un", "T", "P", "E",
                  "pixx", "pixy", "pixn", "piyy", "piyn", "bulkPi", "muB", "nB", "Vx", "Vy", "Vn",
                  "pitt", "pitx", "pity", "pitn", "pinn", "Wx", "Wy", "Lambda", "aL", "c0", "c1", "c2", "c3", "c4", "x", "y")
DF_FIELDS = ("T", "c0", "c1", "c2", "c3", "c4", "F", "G", "betabulk", "betaV", "betapi")

ERRORS = {0: "IS3D_OK", 1: "IS3D_ERR_ARGUMENT", 2: "IS3D_ERR_UNSUPPORTED", 3: "IS3D_ERR_TABLE_RANGE", 4: "IS3D_ERR_CUDA",
          5: "IS3D_ERR_NO_DEVICE", 6: "IS3D_ERR_IO", 7: "IS3D_ERR_NCCL"}


class Surface(C.Structure):
    _fields_ = [("n_cells", C.c_int64)] + [(k, _D) for k in SURFACE_FIELDS]


class Species(C.Structure):
    _fields_ = [("n", C.c_int32), ("mass", _D), ("sign", _D), ("degeneracy", _D), ("baryon", _D)]


class Grid(C.Structure):
    _fields_ = [("n_pT", C.c_int32), ("n_phi", C.c_int32), ("n_y", C.c_int32), ("n_eta", C.c_int32),
                ("pT", _D), ("phi", _D), ("y", _D), ("eta", _D), ("eta_weight", _D)]


class Flags(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("mode", "df_mode", "dimension", "include_baryon", "include_bulk_deltaf",
                                         "include_shear_deltaf", "include_baryondiff_deltaf", "regulate_deltaf", "outflow")] + \
               [("deta_min", C.c_double), ("mass_pion0", C.c_double)]


class DfTables(C.Structure):
    _fields_ = [("n_T", C.c_int32)] + [(k, _D) for k in DF_FIELDS] + \
               [("n_jonah", C.c_int32), ("jonah_x", _D), ("jonah_lambda2", _D), ("jonah_z", _D),
                ("bulkPi_over_Peq_max", C.c_double)]


class Laguerre(C.Structure):
    _fields_ = [("n_points", C.c_int32), ("root1", _D), ("weight1", _D), ("root2", _D), ("weight2", _D)]


class Options(C.Structure):
    _fields_ = [("memory", C.c_int32), ("stream", C.c_void_p), ("n_chunks", C.c_int32), ("tile_variant", C.c_int32),
                ("reserved", C.c_int32 * 4)]


class Stats(C.Structure):
    _fields_ = [("cells_skipped_udsigma", C.c_int64), ("cells_feqmod_breakdown", C.c_int64), ("evaluations", C.c_int64),
                ("h2d_ms", C.c_double), ("prepare_ms", C.c_double), ("kernel_ms", C.c_double), ("reduce_ms", C.c_double),
                ("d2h_ms", C.c_double), ("total_ms", C.c_double), ("gpu_launches", C.c_int32), ("n_chunks", C.c_int32),
                ("tile_variant", C.c_int32), ("n_gpus", C.c_int32), ("allreduce_ms", C.c_double),
                ("n_chunks_wanted", C.c_int32), ("reserved", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class Is3dError(RuntimeError):
    def __init__(self, code, text):
        super().__init__("%s (%d): %s" % (ERRORS.get(code, "?"), code, text))
        self.code = code


_LIB = None


def lib():
    """Load libis3d_b200.so; raises if it has not been built (no fallback)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError("%s is missing: run `python -m is3d_b200.build` (needs nvcc)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.is3d_b200_strerror.restype = C.c_char_p
        L.is3d_b200_last_error.restype = C.c_char_p
        L.is3d_b200_smooth_spectra.restype = C.c_int
        L.is3d_b200_smooth_spectra.argtypes = [C.POINTER(Flags), C.POINTER(Surface), C.POINTER(Species), C.POINTER(Grid),
                                               C.POINTER(DfTables), C.POINTER(Laguerre), C.POINTER(Options), C.c_void_p,
                                               C.POINTER(Stats)]
        L.is3d_b200_measure_fp64_peak.argtypes = [_D, _D]
        _LIB = L
    return _LIB


def _check(rc):
    if rc != 0:
        raise Is3dError(rc, lib().is3d_b200_last_error().decode() or lib().is3d_b200_strerror(rc).decode())


def init():
    _check(lib().is3d_b200_init())


def shutdown():
    _check(lib().is3d_b200_shutdown())


def init_devices(n_gpus=0):
    """One process, several GPUs: select the first n_gpus visible devices (0: all / IS3D_B200_GPUS) for the *_multi entry points."""
    _check(lib().is3d_b200_init_devices(int(n_gpus)))
    return lib().is3d_b200_device_count()


def measure_fp64_peak():
    t = C.c_double(0); ms = C.c_double(0)
    _check(lib().is3d_b200_measure_fp64_peak(C.byref(t), C.byref(ms)))
    return t.value, ms.value


def measure_fp64_sustained(seconds=3.0):
    t = C.c_double(0)
    _check(lib().is3d_b200_measure_fp64_sustained(C.c_double(seconds), C.byref(t)))
    return t.value


def surface_averages(cells):
    """T, E, P, muB, nB surface averages after the reference's 15-digit text round trip (host arrays)."""
    m = _Marshal(False)
    sf = Surface(); sf.n_cells = len(cells["tau"])
    for k in SURFACE_FIELDS:
        if k in cells and cells[k] is not None:
            setattr(sf, k, m.cells(cells[k]))
    out = np.zeros(5)
    _check(lib().is3d_b200_surface_averages(C.byref(sf), out.ctypes.data_as(_D)))
    return out


def jonah_tables(pdg_mass, pdg_degeneracy, pdg_sign, T_avg, laguerre):
    """lambda^2(Pi/P), z(Pi/P) tables for df_mode 4 (host computation in the C++ layer)."""
    m = _Marshal(False)
    x = np.zeros(301); l2 = np.zeros(301); z = np.zeros(301); mx = C.c_double(0)
    f = lib().is3d_b200_jonah_tables
    f.argtypes = [C.c_int32, _D, _D, _D, C.c_double, C.c_int32, _D, _D, _D, _D, _D, C.POINTER(C.c_double)]
    _check(f(len(pdg_mass), m.host(pdg_mass), m.host(pdg_degeneracy), m.host(pdg_sign), float(T_avg), len(laguerre["root2"]),
             m.host(laguerre["root2"]), m.host(laguerre["weight2"]), x.ctypes.data_as(_D), l2.ctypes.data_as(_D),
             z.ctypes.data_as(_D), C.byref(mx)))
    return dict(jonah_x=x, jonah_lambda2=l2, jonah_z=z, bulkPi_over_Peq_max=mx.value)


def vah_cells(columns, fx):
    """Mode-2 (31 column) surface -> SoA dict incl. alpha_L, Lambda and per-cell c0..c4 (C++ host layer, in memory)."""
    from . import synthetic
    cells = synthetic.columns_to_cells(columns, 2)
    a = np.ascontiguousarray(columns, dtype=np.float64)
    n = len(a)
    m = _Marshal(False)
    aL = np.zeros(n); Lam = np.zeros(n)
    f = lib().is3d_b200_vah_anisotropy
    f.argtypes = [C.c_int64, _D, _D, _D, _D, _D]
    _check(f(n, m.host(a[:, 13]), m.host(a[:, 14]), m.host(a[:, 15]), aL.ctypes.data_as(_D), Lam.ctypes.data_as(_D)))
    out = vah_coefficients(fx, Lam, aL)
    cells["aL"] = aL; cells["Lambda"] = Lam
    for k in range(5):
        cells["c%d" % k] = out[k]
    return cells


def vah_coefficients(fx, Lambda_GeV, aL):
    """Per-cell c0..c4 [GeV units] of the anisotropic model from the (Lambda [fm^-1], alpha_L) tables: is3d_b200_vah_coefficients
    (C++ host layer).  Raises Is3dError(IS3D_ERR_TABLE_RANGE) if a cell lies outside the table (the reference leaves garbage)."""
    m = _Marshal(False)
    n = len(aL)
    nL, naL = int(fx["df_vah/nL"]), int(fx["df_vah/naL"])
    Lg = fx["df_vah/L_col"][:nL]; ag = fx["df_vah/aL_col"][::nL]
    tabs = [np.ascontiguousarray(fx["df_vah/c%d" % k].reshape(naL, nL).T) for k in range(5)]      # -> [iL][iaL]
    out = [np.zeros(n) for _ in range(5)]
    g = lib().is3d_b200_vah_coefficients
    g.argtypes = [C.c_int32, C.c_int32, _D, _D, _D, _D, _D, _D, _D, C.c_int64, _D, _D, _D, _D, _D, _D, _D]
    rc = g(nL, naL, m.host(Lg), m.host(ag), *[m.host(t) for t in tabs], n, m.host(Lambda_GeV), m.host(aL), *[o.ctypes.data_as(_D) for o in out])
    if rc:
        raise Is3dError(rc, lib().is3d_b200_host_error().decode() or lib().is3d_b200_strerror(rc).decode())
    return out


def _is_torch(x):
    return type(x).__module__.startswith("torch")


class _Marshal:
    """Turns numpy arrays / torch tensors into double* and keeps them alive."""

    def __init__(self, device):
        self.keep = []
        self.device = device

    def host(self, x):
        a = np.ascontiguousarray(x, dtype=np.float64)
        self.keep.append(a)
        return a.ctypes.data_as(_D)

    def cells(self, x):
        if self.device:
            if not _is_torch(x) or not x.is_cuda:
                raise TypeError("memory='device' needs CUDA tensors for the surface arrays")
            import torch
            t = x.contiguous()
            if t.dtype != torch.float64:
                raise TypeError("surface tensors must be float64")
            self.keep.append(t)
            return C.cast(C.c_void_p(t.data_ptr()), _D)
        if _is_torch(x):
            x = x.detach().cpu().numpy()
        return self.host(x)


def make_flags(flags, mode=1):
    f = Flags()
    f.mode = flags.get("mode", mode)
    f.df_mode = flags["df_mode"]; f.dimension = flags["dimension"]
    f.include_baryon = flags.get("include_baryon", 0)
    f.include_bulk_deltaf = flags.get("include_bulk", flags.get("include_bulk_deltaf", 1))
    f.include_shear_deltaf = flags.get("include_shear", flags.get("include_shear_deltaf", 1))
    f.include_baryondiff_deltaf = flags.get("include_diff", flags.get("include_baryondiff_deltaf", 0))
    f.regulate_deltaf = flags.get("regulate_deltaf", 1); f.outflow = flags.get("outflow", 1)
    f.deta_min = flags.get("deta_min", 1.0e-5); f.mass_pion0 = flags.get("mass_pion0", 0.138)
    return f


def _marshal_problem(m, cells, species, grid, df_tables, laguerre):
    sf = Surface()
    n = len(cells["tau"]) if not _is_torch(cells["tau"]) else int(cells["tau"].numel())
    sf.n_cells = n
    for k in SURFACE_FIELDS:
        if k in cells and cells[k] is not None:
            setattr(sf, k, m.cells(cells[k]))
    sp = Species(); sp.n = len(species["mass"])
    for k in ("mass", "sign", "degeneracy", "baryon"):
        setattr(sp, k, m.host(species[k]))
    g = Grid()
    g.n_pT, g.n_phi, g.n_y, g.n_eta = len(grid["pT"]), len(grid["phi"]), len(grid["y"]), len(grid["eta"])
    for k in ("pT", "phi", "y", "eta", "eta_weight"):
        setattr(g, k, m.host(grid[k]))
    dft = DfTables()
    if df_tables is not None:
        dft.n_T = len(df_tables["T"])
        for k in DF_FIELDS:
            if df_tables.get(k) is not None:
                setattr(dft, k, m.host(df_tables[k]))
        if df_tables.get("jonah_x") is not None:
            dft.n_jonah = len(df_tables["jonah_x"])
            dft.jonah_x = m.host(df_tables["jonah_x"]); dft.jonah_lambda2 = m.host(df_tables["jonah_lambda2"])
            dft.jonah_z = m.host(df_tables["jonah_z"]); dft.bulkPi_over_Peq_max = float(df_tables["bulkPi_over_Peq_max"])
    la = Laguerre()
    if laguerre is not None:
        la.n_points = len(laguerre["root1"])
        for k in ("root1", "weight1", "root2", "weight2"):
            setattr(la, k, m.host(laguerre[k]))
    return sf, sp, g, dft, la


def smooth_spectra(flags, cells, species, grid, df_tables=None, laguerre=None, out=None, memory="host",
                   stream=None, n_chunks=0, tile_variant=0, multi=False):
    """Call is3d_b200_smooth_spectra.

    cells: dict of per-cell arrays (numpy for memory='host', float64 CUDA tensors for memory='device').
    Returns (dN, stats dict); dN is flat [y][phi][pT][species] (species fastest), numpy or the CUDA tensor `out`.
    The result is ADDED into `out` when given.
    """
    device = (memory == "device")
    m = _Marshal(device)
    sf, sp, g, dft, la = _marshal_problem(m, cells, species, grid, df_tables, laguerre)
    n_bins = sp.n * g.n_pT * g.n_phi * g.n_y
    if device:
        import torch
        if out is None:
            out = torch.zeros(n_bins, dtype=torch.float64, device=cells["tau"].device)
        out_ptr = C.c_void_p(out.data_ptr())
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
    else:
        if out is None:
            out = np.zeros(n_bins)
        assert out.dtype == np.float64 and out.flags["C_CONTIGUOUS"] and out.size == n_bins
        out_ptr = C.c_void_p(out.ctypes.data)
    opt = Options(); opt.memory = 1 if device else 0
    opt.stream = C.c_void_p(stream or 0); opt.n_chunks = n_chunks; opt.tile_variant = tile_variant
    st = Stats()
    fl = make_flags(flags)
    fn = lib().is3d_b200_smooth_spectra_multi if multi else lib().is3d_b200_smooth_spectra      # multi: host arrays, all devices of init_devices()
    fn.restype = C.c_int
    fn.argtypes = lib().is3d_b200_smooth_spectra.argtypes
    rc = fn(C.byref(fl), C.byref(sf), C.byref(sp), C.byref(g), C.byref(dft), C.byref(la), C.byref(opt), out_ptr, C.byref(st))
    _check(rc)
    return out, st.as_dict()


class SpacetimeBins(C.Structure):
    _fields_ = [("tau_min", C.c_double), ("tau_max", C.c_double), ("r_min", C.c_double), ("r_max", C.c_double),
                ("tau_bins", C.c_int32), ("r_bins", C.c_int32), ("pT_weight", _D), ("phi_weight", _D)]


class SpacetimeResult(C.Structure):
    _fields_ = [(k, _D) for k in ("dN_tau", "dN_r", "dN_taur", "dN_dydeta", "dN_dy")]


def spacetime_distributions(flags, cells, species, grid, df_tables, laguerre, bins, memory="host", stream=None,
                            n_chunks=0, tile_variant=0, multi=False):
    """Call is3d_b200_spacetime_distributions (operation = 0).

    cells must also carry the transverse positions "x", "y"; grid the quadrature weights "pT_weight", "phi_weight";
    bins = dict(tau_min, tau_max, tau_bins, r_min, r_max, r_bins).  Returns (dict of raw sums as numpy arrays:
    dN_tau [species][tau], dN_r [species][r], dN_taur [species][tau][r], dN_dydeta [species][eta_pts], dN_dy [species]; stats)."""
    device = (memory == "device")
    m = _Marshal(device)
    sf, sp, g, dft, la = _marshal_problem(m, cells, species, grid, df_tables, laguerre)
    b = SpacetimeBins()
    b.tau_min, b.tau_max, b.r_min, b.r_max = (float(bins[k]) for k in ("tau_min", "tau_max", "r_min", "r_max"))
    b.tau_bins, b.r_bins = int(bins["tau_bins"]), int(bins["r_bins"])
    if cells.get("x") is None or cells.get("y") is None:
        raise KeyError("spacetime_distributions needs the transverse cell positions cells['x'], cells['y']")
    b.pT_weight = m.host(grid["pT_weight"]); b.phi_weight = m.host(grid["phi_weight"])
    ns = sp.n; eta_pts = g.n_eta if flags["dimension"] == 2 else 1
    out = dict(dN_tau=np.zeros((ns, b.tau_bins)), dN_r=np.zeros((ns, b.r_bins)), dN_taur=np.zeros((ns, b.tau_bins, b.r_bins)),
               dN_dydeta=np.zeros((ns, eta_pts)), dN_dy=np.zeros(ns))
    res = SpacetimeResult()
    for k in out:
        setattr(res, k, out[k].ctypes.data_as(_D))
    if device and stream is None:
        import torch
        stream = torch.cuda.current_stream().cuda_stream
    opt = Options(); opt.memory = 1 if device else 0
    opt.stream = C.c_void_p(stream or 0); opt.n_chunks = n_chunks; opt.tile_variant = tile_variant
    st = Stats()
    fl = make_flags(flags)
    f = lib().is3d_b200_spacetime_distributions_multi if multi else lib().is3d_b200_spacetime_distributions
    f.restype = C.c_int
    f.argtypes = [C.POINTER(Flags), C.POINTER(Surface), C.POINTER(Species), C.POINTER(Grid), C.POINTER(DfTables),
                  C.POINTER(Laguerre), C.POINTER(SpacetimeBins), C.POINTER(Options), C.POINTER(SpacetimeResult), C.POINTER(Stats)]
    _check(f(C.byref(fl), C.byref(sf), C.byref(sp), C.byref(g), C.byref(dft), C.byref(la), C.byref(b), C.byref(opt),
             C.byref(res), C.byref(st)))
    return out, st.as_dict()


def particle_densities(species, avg5, df_mode, df_tables, laguerre3):
    """(n_eq, dn_bulk, dn_diff) per species at the surface averages avg5 = (T, E, P, muB, nB) (host computation in the C++ layer).

    laguerre3: dict root1, weight1, root2, weight2, root3, weight3 (alpha = 1, 2, 3 rows of the Gauss-Laguerre table)."""
    m = _Marshal(False)
    n = len(species["mass"])
    dft = DfTables(); dft.n_T = len(df_tables["T"])
    for k in DF_FIELDS:
        if df_tables.get(k) is not None:
            setattr(dft, k, m.host(df_tables[k]))
    neq = np.zeros(n); bulk = np.zeros(n); diff = np.zeros(n)
    f = lib().is3d_b200_particle_densities
    f.restype = C.c_int
    f.argtypes = [C.c_int32, _D, _D, _D, _D, _D, C.c_int32, C.POINTER(DfTables), C.c_int32, _D, _D, _D, _D, _D, _D, _D, _D, _D]
    rc = f(n, m.host(species["mass"]), m.host(species["degeneracy"]), m.host(species["baryon"]), m.host(species["sign"]), m.host(avg5),
           int(df_mode), C.byref(dft), len(laguerre3["root1"]), m.host(laguerre3["root1"]), m.host(laguerre3["weight1"]),
           m.host(laguerre3["root2"]), m.host(laguerre3["weight2"]), m.host(laguerre3["root3"]), m.host(laguerre3["weight3"]),
           neq.ctypes.data_as(_D), bulk.ctypes.data_as(_D), diff.ctypes.data_as(_D))
    if rc:
        raise Is3dError(rc, lib().is3d_b200_host_error().decode() or lib().is3d_b200_strerror(rc).decode())
    return neq, bulk, diff


def mean_yield(flags, cells, neq, dn_bulk, df_tables=None, y_cut=5.0, memory="host", stream=None):
    """Call is3d_b200_mean_yield (the sampler's total-yield estimate); returns (Ntot, stats dict)."""
    device = (memory == "device")
    m = _Marshal(device)
    sf = Surface()
    sf.n_cells = len(cells["tau"]) if not _is_torch(cells["tau"]) else int(cells["tau"].numel())
    for k in ("tau", "ux", "uy", "un", "dat", "dax", "day", "dan", "bulkPi", "P"):
        if k in cells and cells[k] is not None:
            setattr(sf, k, m.cells(cells[k]))
    dft = DfTables()
    if df_tables is not None and df_tables.get("jonah_x") is not None:
        dft.n_jonah = len(df_tables["jonah_x"])
        dft.jonah_x = m.host(df_tables["jonah_x"]); dft.jonah_lambda2 = m.host(df_tables["jonah_lambda2"])
        dft.jonah_z = m.host(df_tables["jonah_z"]); dft.bulkPi_over_Peq_max = float(df_tables["bulkPi_over_Peq_max"])
    if device and stream is None:
        import torch
        stream = torch.cuda.current_stream().cuda_stream
    opt = Options(); opt.memory = 1 if device else 0; opt.stream = C.c_void_p(stream or 0)
    st = Stats(); out = C.c_double(0.0)
    f = lib().is3d_b200_mean_yield
    f.restype = C.c_int
    f.argtypes = [C.POINTER(Flags), C.POINTER(Surface), C.c_int32, _D, _D, C.POINTER(DfTables), C.c_double, C.POINTER(Options),
                  C.POINTER(C.c_double), C.POINTER(Stats)]
    fl = make_flags(flags)
    _check(f(C.byref(fl), C.byref(sf), len(neq), m.host(neq), m.host(dn_bulk) if dn_bulk is not None else None, C.byref(dft),
             float(y_cut), C.byref(opt), C.byref(out), C.byref(st)))
    return out.value, st.as_dict()


class ParticleList(C.Structure):
    _I = C.POINTER(C.c_int32)
    _fields_ = [("n_particles", C.c_int32), ("mcid", _I), ("mass", _D), ("width", _D), ("stable", _I), ("decays", _I), ("dec_first", _I),
                ("dec_npart", _I), ("dec_br", _D), ("dec_part", _I)]


def _decay_problem(pdg, grid, keep):
    """ParticleList and Grid structures for the decay entry points; the arrays they point to are appended to keep."""
    def ia(x):
        a = np.ascontiguousarray(x, dtype=np.int32); keep.append(a)
        return a.ctypes.data_as(C.POINTER(C.c_int32))

    m = _Marshal(False)
    keep.append(m)
    p = ParticleList()
    p.n_particles = len(pdg["mcid"])
    p.mcid = ia(pdg["mcid"]); p.mass = m.host(pdg["mass"]); p.width = m.host(pdg["width"]); p.stable = ia(pdg["stable"])
    p.decays = ia(pdg["decays"]); p.dec_first = ia(pdg["dec_first"]); p.dec_npart = ia(pdg["dec_npart"]); p.dec_br = m.host(pdg["dec_br"])
    p.dec_part = ia(np.asarray(pdg["dec_part"]).ravel())
    g = Grid()
    g.n_pT, g.n_phi, g.n_y, g.n_eta = len(grid["pT"]), len(grid["phi"]), len(grid["y"]), len(grid["eta"])
    for k in ("pT", "phi", "y", "eta", "eta_weight"):
        setattr(g, k, m.host(grid[k]))
    return p, g, ia


def resonance_decays(pdg, chosen_pdg_index, grid, dimension, dN, memory="host", stream=None):
    """Call is3d_b200_resonance_decays (SURVEY 8f, row N3): feed-down of the unstable chosen species into their chosen daughters.

    pdg: dict of arrays mcid, mass, width, stable, decays, dec_first, dec_npart, dec_br, dec_part[rows, 5] (tables.pdg_decay_table);
    dN: numpy array (memory='host'; a copy is amended and returned) or float64 CUDA tensor (memory='device'; amended in place)."""
    keep = []
    p, g, ia = _decay_problem(pdg, grid, keep)
    device = (memory == "device")
    if device:
        import torch
        out = dN
        ptr = C.c_void_p(out.data_ptr())
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
    else:
        out = np.array(dN, dtype=np.float64, copy=True)
        ptr = C.c_void_p(out.ctypes.data)
    opt = Options(); opt.memory = 1 if device else 0; opt.stream = C.c_void_p(stream or 0)
    st = Stats()
    f = lib().is3d_b200_resonance_decays
    f.restype = C.c_int
    f.argtypes = [C.POINTER(ParticleList), C.c_int32, C.POINTER(C.c_int32), C.POINTER(Grid), C.c_int32, C.POINTER(Options), C.c_void_p, C.POINTER(Stats)]
    _check(f(C.byref(p), len(chosen_pdg_index), ia(chosen_pdg_index), C.byref(g), int(dimension), C.byref(opt), ptr, C.byref(st)))
    return out, st.as_dict()


class SpinParity(C.Structure):
    _fields_ = [("spin2", C.POINTER(C.c_int32)), ("parity", C.POINTER(C.c_int32))]


def polarization_decays(pdg, spin_parity, chosen_pdg_index, grid, dimension, sums, memory="host", stream=None):
    """Call is3d_b200_polarization_decays: feed-down of the spin-polarization raw sums through the decay tables.

    pdg as for resonance_decays; spin_parity: dict spin2 (2J), parity (+1 / -1, 0 unknown) per particle-list entry
    (tables.spin_parity); sums: dict St, Sx, Sy, Sz, Snorm as spin_polarization returns them (or vorticity + shear sums added).
    memory='host': numpy arrays, an amended copy is returned; memory='device': float64 CUDA tensors, amended in place.  Returns
    (sums, stats dict); mean_spin() forms S and S* from the result.  spin_parity=None passes a NULL table (the library rejects it)."""
    keep = []
    p, g, ia = _decay_problem(pdg, grid, keep)
    sp = None
    if spin_parity is not None:
        sp = SpinParity()
        sp.spin2 = ia(spin_parity["spin2"]); sp.parity = ia(spin_parity["parity"])
    device = (memory == "device")
    res = PolarizationResult()
    if device:
        import torch
        out = sums
        for k in POLARIZATION_FIELDS:
            setattr(res, k, C.cast(C.c_void_p(out[k].data_ptr()), _D))
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
    else:
        out = {k: np.array(sums[k], dtype=np.float64, copy=True) for k in POLARIZATION_FIELDS}
        for k in POLARIZATION_FIELDS:
            setattr(res, k, out[k].ctypes.data_as(_D))
    opt = Options(); opt.memory = 1 if device else 0; opt.stream = C.c_void_p(stream or 0)
    st = Stats()
    f = lib().is3d_b200_polarization_decays
    f.restype = C.c_int
    f.argtypes = [C.POINTER(ParticleList), C.POINTER(SpinParity), C.c_int32, C.POINTER(C.c_int32), C.POINTER(Grid), C.c_int32,
                  C.POINTER(Options), C.POINTER(PolarizationResult), C.POINTER(Stats)]
    _check(f(C.byref(p), C.byref(sp) if sp is not None else None, len(chosen_pdg_index), ia(chosen_pdg_index), C.byref(g), int(dimension),
             C.byref(opt), C.byref(res), C.byref(st)))
    return out, st.as_dict()


WEAK_DECAY_COLUMNS = ("parent", "daughter", "partner", "branching", "alpha", "phi")


class WeakDecays(C.Structure):
    _fields_ = [("n", C.c_int32), ("parent", C.POINTER(C.c_int32)), ("daughter", C.POINTER(C.c_int32)), ("partner", C.POINTER(C.c_int32)),
                ("branching", _D), ("alpha", _D), ("phi", _D)]


def polarization_weak_decays(pdg, spin_parity, weak, chosen_pdg_index, grid, dimension, sums, memory="host", stream=None):
    """Call is3d_b200_polarization_weak_decays: feed-down of the spin-polarization raw sums through weak 2-body decays (Lee-Yang law), meant
    for the output of polarization_decays.

    weak: dict of the six columns parent, daughter, partner (MC ids), branching, alpha, phi (radians), as tables.weak_decays reads them;
    None passes a NULL table (the library rejects it).  Other arguments, memory and the return value as for polarization_decays."""
    keep = []
    p, g, ia = _decay_problem(pdg, grid, keep)
    sp = None
    if spin_parity is not None:
        sp = SpinParity()
        sp.spin2 = ia(spin_parity["spin2"]); sp.parity = ia(spin_parity["parity"])
    wd = None
    if weak is not None:
        wd = WeakDecays()
        wd.n = len(np.atleast_1d(weak["parent"]))
        for k in ("parent", "daughter", "partner"):
            setattr(wd, k, ia(np.atleast_1d(weak[k])))
        for k in ("branching", "alpha", "phi"):
            a = np.ascontiguousarray(np.atleast_1d(weak[k]), dtype=np.float64); keep.append(a)
            setattr(wd, k, a.ctypes.data_as(_D))
    device = (memory == "device")
    res = PolarizationResult()
    if device:
        import torch
        out = sums
        for k in POLARIZATION_FIELDS:
            setattr(res, k, C.cast(C.c_void_p(out[k].data_ptr()), _D))
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
    else:
        out = {k: np.array(sums[k], dtype=np.float64, copy=True) for k in POLARIZATION_FIELDS}
        for k in POLARIZATION_FIELDS:
            setattr(res, k, out[k].ctypes.data_as(_D))
    opt = Options(); opt.memory = 1 if device else 0; opt.stream = C.c_void_p(stream or 0)
    st = Stats()
    f = lib().is3d_b200_polarization_weak_decays
    f.restype = C.c_int
    f.argtypes = [C.POINTER(ParticleList), C.POINTER(SpinParity), C.POINTER(WeakDecays), C.c_int32, C.POINTER(C.c_int32), C.POINTER(Grid),
                  C.c_int32, C.POINTER(Options), C.POINTER(PolarizationResult), C.POINTER(Stats)]
    _check(f(C.byref(p), C.byref(sp) if sp is not None else None, C.byref(wd) if wd is not None else None, len(chosen_pdg_index),
             ia(chosen_pdg_index), C.byref(g), int(dimension), C.byref(opt), C.byref(res), C.byref(st)))
    return out, st.as_dict()


VORTICITY_FIELDS = ("wtx", "wty", "wtn", "wxy", "wxn", "wyn")
POLARIZATION_FIELDS = ("St", "Sx", "Sy", "Sz", "Snorm")


class Vorticity(C.Structure):
    _fields_ = [(k, _D) for k in VORTICITY_FIELDS]


class PolarizationResult(C.Structure):
    _fields_ = [(k, _D) for k in POLARIZATION_FIELDS]


def spin_polarization(flags, cells, vorticity, species, grid, memory="host", stream=None, multi=False):
    """Call is3d_b200_spin_polarization (or the _multi entry point over the devices of init_devices(), host arrays only).

    vorticity: dict wtx, wty, wtn, wxy, wxn, wyn -- the six thermal-vorticity columns of a mode-5 surface (covariant Milne components,
    dimensionless), numpy for memory='host', float64 CUDA tensors for memory='device'.  Returns (dict St, Sx, Sy, Sz, Snorm of RAW sums,
    flat [y][phi][pT][species], numpy or CUDA tensors; stats dict).  mean_spin() turns them into the mean spin vector."""
    device = (memory == "device")
    m = _Marshal(device)
    sf, sp, g, _, _ = _marshal_problem(m, cells, species, grid, None, None)
    vo = None
    if vorticity is not None:
        vo = Vorticity()
        for k in VORTICITY_FIELDS:
            setattr(vo, k, m.cells(vorticity[k]))
    n = sp.n * g.n_pT * g.n_phi * g.n_y
    res = PolarizationResult()
    if device:
        import torch
        out = {k: torch.zeros(n, dtype=torch.float64, device=cells["tau"].device) for k in POLARIZATION_FIELDS}
        for k in POLARIZATION_FIELDS:
            setattr(res, k, C.cast(C.c_void_p(out[k].data_ptr()), _D))
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
    else:
        out = {k: np.zeros(n) for k in POLARIZATION_FIELDS}
        for k in POLARIZATION_FIELDS:
            setattr(res, k, out[k].ctypes.data_as(_D))
    opt = Options(); opt.memory = 1 if device else 0; opt.stream = C.c_void_p(stream or 0)
    st = Stats()
    fl = make_flags(flags)
    f = lib().is3d_b200_spin_polarization_multi if multi else lib().is3d_b200_spin_polarization
    f.restype = C.c_int
    f.argtypes = [C.POINTER(Flags), C.POINTER(Surface), C.POINTER(Vorticity), C.POINTER(Species), C.POINTER(Grid), C.POINTER(Options),
                  C.POINTER(PolarizationResult), C.POINTER(Stats)]
    _check(f(C.byref(fl), C.byref(sf), C.byref(vo) if vo is not None else None, C.byref(sp), C.byref(g), C.byref(opt), C.byref(res),
             C.byref(st)))
    return out, st.as_dict()


THERMAL_SHEAR_FIELDS = ("xtt", "xtx", "xty", "xtn", "xxx", "xxy", "xxn", "xyy", "xyn", "xnn")


class ThermalShear(C.Structure):
    _fields_ = [(k, _D) for k in THERMAL_SHEAR_FIELDS]


def spin_polarization_shear(flags, cells, shear, species, grid, memory="host", stream=None, multi=False):
    """Call is3d_b200_spin_polarization_shear (or the _multi entry point over the devices of init_devices(), host arrays only).

    shear: dict xtt, xtx, xty, xtn, xxx, xxy, xxn, xyy, xyn, xnn -- the ten covariant Milne components of the thermal shear
    (dimensionless), numpy for memory='host', float64 CUDA tensors for memory='device'.  Returns (dict St, Sx, Sy, Sz, Snorm of RAW sums,
    flat [y][phi][pT][species]: St = 0, Sx, Sy, Sz = N_xi, Snorm the ideal spectrum; stats dict).  mean_spin(vorticity_sums, ...,
    shear=these) forms the total mean spin vector."""
    device = (memory == "device")
    m = _Marshal(device)
    sf, sp, g, _, _ = _marshal_problem(m, cells, species, grid, None, None)
    xi = None
    if shear is not None:
        xi = ThermalShear()
        for k in THERMAL_SHEAR_FIELDS:
            if shear.get(k) is not None:                      # a missing column stays NULL (the library rejects it)
                setattr(xi, k, m.cells(shear[k]))
    n = sp.n * g.n_pT * g.n_phi * g.n_y
    res = PolarizationResult()
    if device:
        import torch
        out = {k: torch.zeros(n, dtype=torch.float64, device=cells["tau"].device) for k in POLARIZATION_FIELDS}
        for k in POLARIZATION_FIELDS:
            setattr(res, k, C.cast(C.c_void_p(out[k].data_ptr()), _D))
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
    else:
        out = {k: np.zeros(n) for k in POLARIZATION_FIELDS}
        for k in POLARIZATION_FIELDS:
            setattr(res, k, out[k].ctypes.data_as(_D))
    opt = Options(); opt.memory = 1 if device else 0; opt.stream = C.c_void_p(stream or 0)
    st = Stats()
    fl = make_flags(flags)
    f = lib().is3d_b200_spin_polarization_shear_multi if multi else lib().is3d_b200_spin_polarization_shear
    f.restype = C.c_int
    f.argtypes = [C.POINTER(Flags), C.POINTER(Surface), C.POINTER(ThermalShear), C.POINTER(Species), C.POINTER(Grid), C.POINTER(Options),
                  C.POINTER(PolarizationResult), C.POINTER(Stats)]
    _check(f(C.byref(fl), C.byref(sf), C.byref(xi) if xi is not None else None, C.byref(sp), C.byref(g), C.byref(opt), C.byref(res),
             C.byref(st)))
    return out, st.as_dict()


BARYON_GRADIENT_FIELDS = ("dt", "dx", "dy", "dn")


class BaryonGradient(C.Structure):
    _fields_ = [(k, _D) for k in BARYON_GRADIENT_FIELDS]


def spin_polarization_spin_hall(flags, cells, gradient, species, grid, memory="host", stream=None, multi=False):
    """Call is3d_b200_spin_polarization_spin_hall (or the _multi entry point over the devices of init_devices(), host arrays only).

    gradient: dict dt, dx, dy, dn -- the covariant Milne components of the gradient of alpha_B = muB/T (d_tau, d_x, d_y in 1/fm, d_eta
    dimensionless), numpy for memory='host', float64 CUDA tensors for memory='device'.  species needs 'baryon' (q_B).  Returns (dict St,
    Sx, Sy, Sz, Snorm of RAW sums, flat [y][phi][pT][species]: St = 0, Sx, Sy, Sz = N_she, Snorm the ideal spectrum; stats dict).
    mean_spin(vorticity_sums, ..., spin_hall=these) forms the total mean spin vector."""
    device = (memory == "device")
    m = _Marshal(device)
    sf, sp, g, _, _ = _marshal_problem(m, cells, species, grid, None, None)
    gd = None
    if gradient is not None:
        gd = BaryonGradient()
        for k in BARYON_GRADIENT_FIELDS:
            if gradient.get(k) is not None:                   # a missing column stays NULL (the library rejects it)
                setattr(gd, k, m.cells(gradient[k]))
    n = sp.n * g.n_pT * g.n_phi * g.n_y
    res = PolarizationResult()
    if device:
        import torch
        out = {k: torch.zeros(n, dtype=torch.float64, device=cells["tau"].device) for k in POLARIZATION_FIELDS}
        for k in POLARIZATION_FIELDS:
            setattr(res, k, C.cast(C.c_void_p(out[k].data_ptr()), _D))
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
    else:
        out = {k: np.zeros(n) for k in POLARIZATION_FIELDS}
        for k in POLARIZATION_FIELDS:
            setattr(res, k, out[k].ctypes.data_as(_D))
    opt = Options(); opt.memory = 1 if device else 0; opt.stream = C.c_void_p(stream or 0)
    st = Stats()
    fl = make_flags(flags)
    f = lib().is3d_b200_spin_polarization_spin_hall_multi if multi else lib().is3d_b200_spin_polarization_spin_hall
    f.restype = C.c_int
    f.argtypes = [C.POINTER(Flags), C.POINTER(Surface), C.POINTER(BaryonGradient), C.POINTER(Species), C.POINTER(Grid), C.POINTER(Options),
                  C.POINTER(PolarizationResult), C.POINTER(Stats)]
    _check(f(C.byref(fl), C.byref(sf), C.byref(gd) if gd is not None else None, C.byref(sp), C.byref(g), C.byref(opt), C.byref(res),
             C.byref(st)))
    return out, st.as_dict()


def mean_spin(result, species, grid, dimension, shear=None, spin_hall=None):
    """Mean spin vector from the raw sums of spin_polarization(): returns (S [4][n_bins] = N^mu / Snorm in lab components t, x, y, z,
    0 where Snorm = 0; S* [3][n_bins] = S^i - S^t p^i / (E + m), the rest-frame spin, P* = 2 S* for spin 1/2).  The same numbers
    results/polarization/S_<mcid>.dat holds.  shear (optional): the raw sums of spin_polarization_shear() on the same problem; S is then
    the total (N^mu + N_xi^mu) / Snorm and S* its rest-frame part, the totals of results/polarization/S_xi_<mcid>.dat.  spin_hall
    (optional): the raw sums of spin_polarization_spin_hall() on the same problem, added the same way (after shear), the totals of
    results/polarization/S_she_<mcid>.dat."""
    r = {k: np.asarray(result[k].cpu() if _is_torch(result[k]) else result[k], dtype=np.float64) for k in POLARIZATION_FIELDS}
    for extra in (shear, spin_hall):
        if extra is not None:
            for k in ("St", "Sx", "Sy", "Sz"):
                r[k] = r[k] + np.asarray(extra[k].cpu() if _is_torch(extra[k]) else extra[k], dtype=np.float64)
    m = np.asarray(species["mass"], dtype=np.float64)
    pT = np.asarray(grid["pT"], dtype=np.float64); phi = np.asarray(grid["phi"], dtype=np.float64)
    y = np.asarray(grid["y"], dtype=np.float64)
    if dimension == 2:
        y = np.zeros_like(y)
    yy, ff, pp, mm = np.meshgrid(y, phi, pT, m, indexing="ij")          # [y][phi][pT][species] = the flat bin order
    mT = np.sqrt(mm * mm + pp * pp)
    E = (mT * np.cosh(yy)).ravel()
    p = np.stack([(pp * np.cos(ff)).ravel(), (pp * np.sin(ff)).ravel(), (mT * np.sinh(yy)).ravel()])
    sn = r["Snorm"]
    nz = sn != 0
    S = np.zeros((4, sn.size))
    for i, k in enumerate(("St", "Sx", "Sy", "Sz")):
        S[i, nz] = r[k][nz] / sn[nz]
    rest = S[1:] - S[0] * p / (E + mm.ravel())
    return S, rest


SPIN_DENSITY_FIELDS = ("Snorm", "Px", "Py", "Pz", "Qxx", "Qxy", "Qxz", "Qyy", "Qyz")
SPIN_TENSOR_FIELDS = ("xx", "xy", "xz", "yy", "yz", "zz")


class SpinDensityResult(C.Structure):
    _fields_ = [(k, _D) for k in SPIN_DENSITY_FIELDS]


def spin_density(flags, cells, vorticity, species, grid, memory="host", stream=None, multi=False):
    """Call is3d_b200_spin_density (or the _multi entry point over the devices of init_devices(), host arrays only): the spin density
    matrix of every species (spin J = (degeneracy - 1)/2) with the thermal-vorticity term exponentiated, on a mode-5 surface.

    vorticity: as for spin_polarization().  Returns (dict Snorm, Px, Py, Pz, Qxx, Qxy, Qxz, Qyy, Qyz of RAW sums, flat
    [y][phi][pT][species], numpy or CUDA tensors; stats dict).  spin_moments() and spin_alignment() form the ratios."""
    device = (memory == "device")
    m = _Marshal(device)
    sf, sp, g, _, _ = _marshal_problem(m, cells, species, grid, None, None)
    vo = None
    if vorticity is not None:
        vo = Vorticity()
        for k in VORTICITY_FIELDS:
            setattr(vo, k, m.cells(vorticity[k]))
    n = sp.n * g.n_pT * g.n_phi * g.n_y
    res = SpinDensityResult()
    if device:
        import torch
        out = {k: torch.zeros(n, dtype=torch.float64, device=cells["tau"].device) for k in SPIN_DENSITY_FIELDS}
        for k in SPIN_DENSITY_FIELDS:
            setattr(res, k, C.cast(C.c_void_p(out[k].data_ptr()), _D))
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
    else:
        out = {k: np.zeros(n) for k in SPIN_DENSITY_FIELDS}
        for k in SPIN_DENSITY_FIELDS:
            setattr(res, k, out[k].ctypes.data_as(_D))
    opt = Options(); opt.memory = 1 if device else 0; opt.stream = C.c_void_p(stream or 0)
    st = Stats()
    fl = make_flags(flags)
    f = lib().is3d_b200_spin_density_multi if multi else lib().is3d_b200_spin_density
    f.restype = C.c_int
    f.argtypes = [C.POINTER(Flags), C.POINTER(Surface), C.POINTER(Vorticity), C.POINTER(Species), C.POINTER(Grid), C.POINTER(Options),
                  C.POINTER(SpinDensityResult), C.POINTER(Stats)]
    _check(f(C.byref(fl), C.byref(sf), C.byref(vo) if vo is not None else None, C.byref(sp), C.byref(g), C.byref(opt), C.byref(res),
             C.byref(st)))
    return out, st.as_dict()


def spin_moments(result, species):
    """Ratios of the raw sums of spin_density(): returns (S* [3][n_bins] = <S*_i> = P_i / Snorm, the all-order rest-frame mean spin;
    T [6][n_bins] = <S*_i S*_j> - J(J+1) delta_ij / 3 = Q_ij / Snorm in the order xx, xy, xz, yy, yz, zz), 0 where Snorm = 0.  The
    numbers results/polarization/spin_<mcid>.dat holds.  species is accepted for symmetry with mean_spin(); the ratios need only the sums."""
    r = {k: np.asarray(result[k].cpu() if _is_torch(result[k]) else result[k], dtype=np.float64) for k in SPIN_DENSITY_FIELDS}
    sn = r["Snorm"]
    nz = sn != 0
    S = np.zeros((3, sn.size)); T = np.zeros((6, sn.size))
    for i, k in enumerate(("Px", "Py", "Pz")):
        S[i, nz] = r[k][nz] / sn[nz]
    for i, k in enumerate(("Qxx", "Qxy", "Qxz", "Qyy", "Qyz")):
        T[i, nz] = r[k][nz] / sn[nz]
    T[5, nz] = -(r["Qxx"][nz] + r["Qyy"][nz]) / sn[nz]
    return S, T


def spin_alignment(result, species, grid, dimension, axis):
    """Vector-meson spin alignment rho00 = 1/3 - n.T.n from the raw sums of spin_density(), [n_bins], for the species with J = 1
    (degeneracy 3); NaN for every other species.  axis: "x", "y", "z" (a fixed rest-frame axis) or "helicity" (n = p / |p|, the bin's
    momentum direction; 2+1D bins have y = 0)."""
    _, T = spin_moments(result, species)
    m = np.asarray(species["mass"], dtype=np.float64)
    deg = np.asarray(species["degeneracy"], dtype=np.float64)
    pT = np.asarray(grid["pT"], dtype=np.float64); phi = np.asarray(grid["phi"], dtype=np.float64)
    y = np.asarray(grid["y"], dtype=np.float64)
    if dimension == 2:
        y = np.zeros_like(y)
    yy, ff, pp, mm = np.meshgrid(y, phi, pT, m, indexing="ij")          # [y][phi][pT][species] = the flat bin order
    _, _, _, gg = np.meshgrid(y, phi, pT, deg, indexing="ij")
    if axis == "helicity":
        mT = np.sqrt(mm * mm + pp * pp)
        p = np.stack([(pp * np.cos(ff)).ravel(), (pp * np.sin(ff)).ravel(), (mT * np.sinh(yy)).ravel()])
        n = p / np.linalg.norm(p, axis=0)
    elif axis in ("x", "y", "z"):
        n = np.zeros((3, T.shape[1]))
        n["xyz".index(axis)] = 1.0
    else:
        raise ValueError("axis must be 'x', 'y', 'z' or 'helicity'")
    Tm = {k: T[i] for i, k in enumerate(SPIN_TENSOR_FIELDS)}
    nTn = (n[0] * n[0] * Tm["xx"] + n[1] * n[1] * Tm["yy"] + n[2] * n[2] * Tm["zz"]
           + 2.0 * (n[0] * n[1] * Tm["xy"] + n[0] * n[2] * Tm["xz"] + n[1] * n[2] * Tm["yz"]))
    return np.where(gg.ravel() == 3, 1.0 / 3.0 - nTn, np.nan)


HBT_FIELDS = ("S0", "So", "Ss", "Sl", "Soo", "Sss", "Sll", "Sos", "Sol", "Ssl")
HBT_RADII = ("out", "side", "long", "outside", "outlong", "sidelong")


class HbtResult(C.Structure):
    _fields_ = [(k, _D) for k in HBT_FIELDS]


def hbt_moments(flags, cells, species, grid, df_tables, memory="host", stream=None, multi=False):
    """Call is3d_b200_hbt_moments (or the _multi entry point over the devices of init_devices(), host arrays only).

    cells must carry the transverse positions "x" and "y" [fm] besides the spectra's arrays (numpy for memory='host', float64 CUDA
    tensors for memory='device').  Returns (dict S0, So, Ss, Sl, Soo, Sss, Sll, Sos, Sol, Ssl of RAW sums, flat [y][phi][pT][species],
    numpy or CUDA tensors; stats dict).  S0 is the spectrum; hbt_radii() turns the sums into the radii."""
    device = (memory == "device")
    m = _Marshal(device)
    sf, sp, g, dft, _ = _marshal_problem(m, cells, species, grid, df_tables, None)
    n = sp.n * g.n_pT * g.n_phi * g.n_y
    res = HbtResult()
    if device:
        import torch
        out = {k: torch.zeros(n, dtype=torch.float64, device=cells["tau"].device) for k in HBT_FIELDS}
        for k in HBT_FIELDS:
            setattr(res, k, C.cast(C.c_void_p(out[k].data_ptr()), _D))
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
    else:
        out = {k: np.zeros(n) for k in HBT_FIELDS}
        for k in HBT_FIELDS:
            setattr(res, k, out[k].ctypes.data_as(_D))
    opt = Options(); opt.memory = 1 if device else 0; opt.stream = C.c_void_p(stream or 0)
    st = Stats()
    fl = make_flags(flags)
    f = lib().is3d_b200_hbt_moments_multi if multi else lib().is3d_b200_hbt_moments
    f.restype = C.c_int
    f.argtypes = [C.POINTER(Flags), C.POINTER(Surface), C.POINTER(Species), C.POINTER(Grid), C.POINTER(DfTables), C.POINTER(Options),
                  C.POINTER(HbtResult), C.POINTER(Stats)]
    _check(f(C.byref(fl), C.byref(sf), C.byref(sp), C.byref(g), C.byref(dft), C.byref(opt), C.byref(res), C.byref(st)))
    return out, st.as_dict()


def hbt_radii(sums):
    """HBT radii [fm^2] from the raw sums of hbt_moments(): dict out, side, long, outside, outlong, sidelong of
    R^2_ij = S_ij / S0 - (S_i / S0)(S_j / S0), 0 where S0 = 0 -- the numbers results/hbt/R2_<mcid>.dat holds."""
    r = {k: np.asarray(sums[k].cpu() if _is_torch(sums[k]) else sums[k], dtype=np.float64) for k in HBT_FIELDS}
    s0 = r["S0"]
    nz = s0 != 0
    first = {i: np.where(nz, r["S" + i], 0.0) / np.where(nz, s0, 1.0) for i in "osl"}
    out = {}
    for name, (i, j) in zip(HBT_RADII, (("o", "o"), ("s", "s"), ("l", "l"), ("o", "s"), ("o", "l"), ("s", "l"))):
        v = np.where(nz, r["S" + i + j], 0.0) / np.where(nz, s0, 1.0) - first[i] * first[j]
        out[name] = np.where(nz, v, 0.0)
    return out


HBARC = 0.197327053          # GeV fm


class HbtQrays(C.Structure):
    _fields_ = [("n_dir", C.c_int32), ("n_q", C.c_int32), ("dq", C.c_double), ("dir", _D)]


class HbtFourierResult(C.Structure):
    _fields_ = [("Re", _D), ("Im", _D)]


def hbt_fourier(flags, cells, species, grid, df_tables, qrays, memory="host", stream=None, multi=False):
    """Call is3d_b200_hbt_fourier (or the _multi entry point over the devices of init_devices(), host arrays only).

    qrays: dict dir (n_dir x 3 directions (o, s, l), not normalised), dq [GeV] and n_q; the q points are q_k = k dq dir, k < n_q.
    cells must carry "x" and "y" [fm] as for hbt_moments().  Returns (dict Re, Im of RAW sums sum w cos(q.r / hbar c), sum w sin(...),
    shape (n_dir, n_q, n_bins) with the spectra bin layout inside, numpy or CUDA tensors; stats dict).  Re[d, 0] is the spectrum;
    hbt_correlation() turns the sums into C."""
    device = (memory == "device")
    m = _Marshal(device)
    sf, sp, g, dft, _ = _marshal_problem(m, cells, species, grid, df_tables, None)
    d = np.ascontiguousarray(np.asarray(qrays["dir"], dtype=np.float64).reshape(-1, 3))
    n_dir, n_q = d.shape[0], int(qrays["n_q"])
    qr = HbtQrays(n_dir, n_q, float(qrays["dq"]), d.ctypes.data_as(_D))
    shape = (n_dir, max(n_q, 0), sp.n * g.n_pT * g.n_phi * g.n_y)
    res = HbtFourierResult()
    if device:
        import torch
        out = {k: torch.zeros(shape, dtype=torch.float64, device=cells["tau"].device) for k in ("Re", "Im")}
        for k in out:
            setattr(res, k, C.cast(C.c_void_p(out[k].data_ptr()), _D))
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
    else:
        out = {k: np.zeros(shape) for k in ("Re", "Im")}
        for k in out:
            setattr(res, k, out[k].ctypes.data_as(_D))
    opt = Options(); opt.memory = 1 if device else 0; opt.stream = C.c_void_p(stream or 0)
    st = Stats()
    fl = make_flags(flags)
    f = lib().is3d_b200_hbt_fourier_multi if multi else lib().is3d_b200_hbt_fourier
    f.restype = C.c_int
    f.argtypes = [C.POINTER(Flags), C.POINTER(Surface), C.POINTER(Species), C.POINTER(Grid), C.POINTER(DfTables), C.POINTER(HbtQrays),
                  C.POINTER(Options), C.POINTER(HbtFourierResult), C.POINTER(Stats)]
    _check(f(C.byref(fl), C.byref(sf), C.byref(sp), C.byref(g), C.byref(dft), C.byref(qr), C.byref(opt), C.byref(res), C.byref(st)))
    return out, st.as_dict()


def hbt_correlation(sums, species):
    """Correlation functions of identical particles from the raw sums of hbt_fourier(): C = 1 - sign (Re^2 + Im^2) / (g S0^2) with
    S0 = Re[d, 0], sign = -1 (bosons) / +1 (fermions) and g the degeneracy of each bin's species; 1 where S0 = 0.  Shape (n_dir, n_q,
    n_bins) -- the numbers results/hbt/C_<mcid>.dat holds."""
    re, im = (np.asarray(sums[k].cpu() if _is_torch(sums[k]) else sums[k], dtype=np.float64) for k in ("Re", "Im"))
    ns = len(species["sign"])
    sign = np.resize(np.asarray(species["sign"], dtype=np.float64), re.shape[-1])        # bin = species + n_species * (...)
    g = np.resize(np.asarray(species["degeneracy"], dtype=np.float64), re.shape[-1])
    assert re.shape[-1] % ns == 0
    s0 = re[:, :1, :]
    nz = s0 != 0
    r, m = re / np.where(nz, s0, 1.0), im / np.where(nz, s0, 1.0)          # ratios first: S0^2 underflows in the far tails
    return np.where(nz, 1.0 - sign * (r * r + m * m) / g, 1.0)
