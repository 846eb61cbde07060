"""Re-create an iS3D-style working directory from the committed numeric fixture.

iS3D (and this drop-in) read every input from CWD-relative paths (reference src/cpp/iS3D.cpp:83,156-167;
deltafReader.h:27-29; readindata.h:217-219).  `materialize()` writes those files -- parameter file, particle
lists, quadrature tables, delta-f coefficient tables, surface -- into a directory, using the same text formats the
reference's readers expect, from `is3d_b200/data/is3d_tables.npz` (numeric content extracted once by
tests/golden/make_tables_fixture.py).  Numbers are written with repr(), which round-trips every double exactly.

This is tooling for tests / benchmarks / the smoke test; the product's C++ host layer (csrc/host_*.cpp) only ever
sees the resulting files, exactly as it would see a user's own iS3D checkout.
"""
import os

import numpy as np

from is3d_b200.synthetic import BARYON_GRADIENT_COLUMNS, THERMAL_SHEAR_COLUMNS

_FIXTURE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "is3d_tables.npz")

# every key the reference constructor getVal()s (emissionfunction.cpp:170-222, readindata.cpp:111-118,
# deltafReader.cpp:24-27, iS3D.cpp:164); a missing key is fatal there, so the template carries all of them.
DEFAULT_PARAMETERS = [
    ("operation", 1), ("mode", 1), ("hrg_eos", 1), ("set_FO_temperature", 0), ("T_switch", 0.151),
    ("dimension", 3), ("df_mode", 1), ("include_baryon", 0), ("include_bulk_deltaf", 1),
    ("include_shear_deltaf", 1), ("include_baryondiff_deltaf", 0), ("regulate_deltaf", 1), ("outflow", 1),
    ("deta_min", 1.0e-5), ("group_particles", 0), ("particle_diff_tolerance", 0.01), ("mass_pion0", 0.138),
    ("do_resonance_decays", 0), ("lightest_particle", 111), ("oversample", 0), ("min_num_hadrons", 1.0e8),
    ("max_num_samples", 500), ("fast", 1), ("y_cut", 5.0), ("sampler_seed", 1), ("test_sampler", 0),
    ("pT_lower_cut", 0.0), ("pT_upper_cut", 3.0), ("pT_bins", 100), ("y_bins", 50), ("eta_cut", 7),
    ("eta_bins", 70), ("tau_min", 0.0), ("tau_max", 12.0), ("tau_bins", 120), ("r_min", 0.0),
    ("r_max", 12.0), ("r_bins", 60),
]

# keys of this drop-in that the reference does not read: written only when a caller sets them (absent: 0, or the default of the host layer)
OPTIONAL_PARAMETERS = ("spin_polarization", "thermal_shear_polarization", "spin_hall_polarization", "polarization_feed_down", "polarization_weak_decays", "spin_density", "hbt_radii", "hbt_correlation", "hbt_dq",
                       "hbt_q_points")

_EOS_DIR = {1: "urqmd", 2: "smash", 3: "smash_box"}
_EOS_PDG = {1: ("pdg_urqmd", "pdg-urqmd_v3.3+.dat"), 2: ("pdg_smash", "pdg_smash.dat"), 3: ("pdg_box", "pdg_box.dat")}
_DF_NAMES = ("c0", "c1", "c2", "c3", "c4", "F", "G", "betabulk", "betaV", "betapi")


def load_fixture(path=None):
    return np.load(path or _FIXTURE)


def _r(x):
    return repr(float(x))


def write_parameters(path, **overrides):
    """Write iS3D_parameters.dat (`name = value # comment`, ParameterReader.cpp:38-98)."""
    low = {k.lower(): v for k, v in overrides.items()}
    known = {k.lower() for k, _ in DEFAULT_PARAMETERS} | set(OPTIONAL_PARAMETERS)
    unknown = set(low) - known
    if unknown:
        raise KeyError("unknown iS3D parameter(s): %s" % sorted(unknown))
    with open(path, "w") as f:
        for k, v in DEFAULT_PARAMETERS + [(k, low[k]) for k in OPTIONAL_PARAMETERS if k in low]:
            v = low.get(k.lower(), v)
            f.write("%-28s = %s\t# written by is3d_b200.workdir\n" % (k, repr(v) if isinstance(v, float) else v))


def write_table(path, cols):
    """Whitespace block file, one newline-terminated row per line (arsenal.cpp:406-453)."""
    a = np.atleast_2d(np.asarray(cols, dtype=np.float64))
    with open(path, "w") as f:
        for row in a:
            f.write("\t".join(_r(v) for v in row) + "\n")


def write_surface(path, columns):
    """columns: (n_cells, n_cols) array already in the file's units (fm^-n for E,T,P,pi,Pi; see readindata.cpp:343-420)."""
    a = np.ascontiguousarray(columns, dtype=np.float64)
    with open(path, "w") as f:
        # '%.17g' round-trips a double; one text row per cell, newline-terminated (row count rule)
        np.savetxt(f, a, fmt="%.17g", delimiter=" ")


def write_chosen(path, mcids):
    with open(path, "w") as f:
        for m in mcids:
            f.write("\t%d\n" % int(m))


def _write_pdg_conventional(path, fx, key):
    g = lambda k: fx["%s/%s" % (key, k)]
    owner = g("dec_owner"); dn = g("dec_n"); br = g("dec_br"); parts = g("dec_parts")
    first = np.searchsorted(owner, np.arange(len(g("mcid"))))
    with open(path, "w") as f:
        for i in range(len(g("mcid"))):
            f.write("%9d  %-20s %s %s %d %d %d %d %d %d %d %d\n" % (
                g("mcid")[i], g("name")[i], _r(g("mass")[i]), _r(g("width")[i]), g("gspin")[i], g("baryon")[i],
                g("strange")[i], g("charm")[i], g("bottom")[i], g("gisospin")[i], g("charge")[i], g("decays")[i]))
            for j in range(first[i], first[i] + g("decays")[i]):
                f.write("%9d %d %s %d %d %d %d %d\n" % (g("mcid")[i], dn[j], _r(br[j]), *parts[j]))


def write_weak_decays(path, weak):
    """PDG/weak_decays.dat: `parent daughter partner branching alpha phi` per line, after a comment line naming the columns."""
    with open(path, "w") as f:
        f.write("# parent_mcid daughter_mcid partner_mcid branching alpha phi[rad]\n")
        for row in zip(*(np.atleast_1d(weak[k]) for k in ("parent", "daughter", "partner", "branching", "alpha", "phi"))):
            f.write("%d %d %d %s %s %s\n" % (int(row[0]), int(row[1]), int(row[2]), _r(row[3]), _r(row[4]), _r(row[5])))


def _write_pdg_box(path, fx):
    with open(path, "w", encoding="utf-8") as f:
        f.write("# NAME MASS[GEV] WIDTH[GEV] PARITY PDG\n\n")
        for i in range(len(fx["pdg_box/name"])):
            ids = " ".join(str(int(v)) for v in fx["pdg_box/mcid"][i] if v != 0)
            f.write("%s %s %s %s %s\n" % (fx["pdg_box/name"][i], _r(fx["pdg_box/mass"][i]), _r(fx["pdg_box/width"][i]),
                                          fx["pdg_box/parity"][i], ids))


def _write_df_vh(dirname, fx, eos):
    os.makedirs(dirname, exist_ok=True)
    T = fx["df_%s/T" % eos]; mu = fx["df_%s/muB0" % eos]
    for name in _DF_NAMES:
        v = fx["df_%s/%s" % (eos, name)]
        with open(os.path.join(dirname, name + ".dat"), "w") as f:
            # header: points_T, points_muB, one text line (deltafReader.cpp:121-146); only the muB = 0 block is
            # materialised, which is all the reader touches when include_baryon = 0 (points_muB forced to 1).
            f.write("%d\n%d\nT [GeV]\t\tmuB [GeV]\t\t%s\n" % (len(T), 1, name))
            for t, m, c in zip(T, mu, v):
                f.write("%s\t\t%s\t\t%s\n" % (_r(t), _r(m), _r(c)))


def _write_df_vah(dirname, fx):
    os.makedirs(dirname, exist_ok=True)
    L = fx["df_vah/L_col"]; aL = fx["df_vah/aL_col"]
    for k in range(5):
        with open(os.path.join(dirname, "c%d_vah1.dat" % k), "w") as f:
            f.write("%d\n%d\nL [fm^-1]\t\taL\t\tc%d_vah1\n" % (int(fx["df_vah/nL"]), int(fx["df_vah/naL"]), k))
            for a, b, c in zip(L, aL, fx["df_vah/c%d" % k]):
                f.write("%s\t\t%s\t\t%s\n" % (_r(a), _r(b), _r(c)))


def materialize(root, surface_columns=None, chosen=None, fixture=None, tables=None, vah=False, thermal_shear=None, baryon_gradient=None,
                weak_decays=None, **params):
    """Create `root` as an iS3D working directory.

    surface_columns : (n_cells, n_cols) array in file units, or None for the shipped one-cell toy surface.
    chosen          : iterable of MC ids, or the name of a fixture list ("chosen_pikp", "chosen_urqmd", ...).
    tables          : optional dict overriding quadrature tables: keys pT, phi, y, eta -> (n, 2) arrays.
    thermal_shear   : optional (n_cells, 10) array or dict of the ten columns of synthetic.THERMAL_SHEAR_COLUMNS, written to
                      input/thermal_shear.dat (read when thermal_shear_polarization = 1).
    baryon_gradient : optional (n_cells, 4) array or dict of the four columns of synthetic.BARYON_GRADIENT_COLUMNS, written to
                      input/muB_over_T_gradient.dat (read when spin_hall_polarization = 1).
    weak_decays     : optional dict of the six columns of tables.weak_decays (parent, daughter, partner, branching, alpha, phi), written
                      to PDG/weak_decays.dat (read when polarization_weak_decays = 1).
    params          : iS3D_parameters.dat overrides (operation, mode, df_mode, dimension, ...).
    """
    fx = fixture if fixture is not None else load_fixture()
    p = {k.lower(): v for k, v in params.items()}
    hrg_eos = int(p.get("hrg_eos", dict(DEFAULT_PARAMETERS)["hrg_eos"]))
    for d in ("input", "PDG", "tables/eta", "results/vn_continuous", "results/continuous", "results/sampled", "results/spacetime_distribution", "results/polarization",
              "results/hbt",
              "deltaf_coefficients/vh", "deltaf_coefficients/vah"):
        os.makedirs(os.path.join(root, d), exist_ok=True)
    write_parameters(os.path.join(root, "iS3D_parameters.dat"), **params)
    if surface_columns is None:
        surface_columns = fx["toy_surface"]
    write_surface(os.path.join(root, "input", "surface.dat"), surface_columns)
    if thermal_shear is not None:
        if isinstance(thermal_shear, dict):
            thermal_shear = np.column_stack([thermal_shear[k] for k in THERMAL_SHEAR_COLUMNS])
        write_surface(os.path.join(root, "input", "thermal_shear.dat"), thermal_shear)
    if baryon_gradient is not None:
        if isinstance(baryon_gradient, dict):
            baryon_gradient = np.column_stack([baryon_gradient[k] for k in BARYON_GRADIENT_COLUMNS])
        write_surface(os.path.join(root, "input", "muB_over_T_gradient.dat"), baryon_gradient)
    key, fname = _EOS_PDG[hrg_eos]
    if hrg_eos == 3:
        _write_pdg_box(os.path.join(root, "PDG", fname), fx)
    else:
        _write_pdg_conventional(os.path.join(root, "PDG", fname), fx, key)
        if int(p.get("polarization_feed_down", 0)):
            _write_pdg_box(os.path.join(root, "PDG", "pdg_box.dat"), fx)     # the parities the polarization feed-down reads
    if weak_decays is not None:
        write_weak_decays(os.path.join(root, "PDG", "weak_decays.dat"), weak_decays)
    if chosen is None:
        chosen = "chosen_pikp"
    if isinstance(chosen, str):
        chosen = fx[chosen]
    write_chosen(os.path.join(root, "PDG", "chosen_particles.dat"), chosen)
    t = tables or {}
    write_table(os.path.join(root, "tables", "pT_gauss_legendre_table.dat"), t.get("pT", fx["pT_tab"]))
    write_table(os.path.join(root, "tables", "phi_gauss_legendre_table.dat"), t.get("phi", fx["phi_tab"]))
    write_table(os.path.join(root, "tables", "y_trapezoid_table_21pt.dat"), t.get("y", fx["y_tab"]))
    write_table(os.path.join(root, "tables", "eta", "eta_trapezoid_table_241pt.dat"), t.get("eta", fx["eta_tab"]))
    with open(os.path.join(root, "tables", "gla_roots_weights_32_points.txt"), "w") as f:
        na, npts = fx["gla_root"].shape
        f.write("%d\t%d\n" % (na, npts))
        for a in range(na):
            for j in range(npts):
                f.write("%d\t%s\t%s\n" % (a, _r(fx["gla_root"][a, j]), _r(fx["gla_weight"][a, j])))
    with open(os.path.join(root, "tables", "gauss_legendre_48pts.dat"), "w") as f:
        f.write("%d\n" % len(fx["legendre48"]))
        for a, b in fx["legendre48"]:
            f.write("%s\t%s\n" % (_r(a), _r(b)))
    _write_df_vh(os.path.join(root, "deltaf_coefficients", "vh", _EOS_DIR[hrg_eos]), fx, _EOS_DIR[hrg_eos])
    if vah:
        _write_df_vah(os.path.join(root, "deltaf_coefficients", "vah"), fx)
    return root
