"""Seeded synthetic freeze-out surfaces for the BASELINE.json configurations (SURVEY.md section 8d).

Every generator returns the surface as the *text-file columns* of the reference's formats
(mode 1: 20 columns, readindata.cpp:320-420; mode 2: 31 columns, readindata.cpp:813-928), i.e. E, T, P, pi^{mu nu}
and Pi in fm^-n.  `columns_to_cells()` applies the same unit conversion the readers apply (x hbarC, one multiply
per value) and returns the structure-of-arrays dict the C ABI takes.  All cells satisfy u.dsigma > 0 (SURVEY R4).
"""
import numpy as np

HBARC = 0.197327053  # GeV fm, reference src/cpp/iS3D.h:9

SEEDS = {"cfg1": 1001, "cfg2": 1002, "cfg3": 1003, "cfg4": 1004, "cfg5": 1005}

MODE1_COLUMNS = ("tau", "x", "y", "eta", "dat", "dax", "day", "dan", "ux", "uy", "un", "E", "T", "P",
                 "pixx", "pixy", "pixn", "piyy", "piyn", "bulkPi")
MODE2_COLUMNS = ("tau", "x", "y", "eta", "dat", "dax", "day", "dan", "ut", "ux", "uy", "un", "E", "T", "P", "PL",
                 "pitt", "pitx", "pity", "pitn", "pixx", "pixy", "pixn", "piyy", "piyn", "pinn",
                 "Wt", "Wx", "Wy", "Wn", "bulkPi")
_GEV_FIELDS = {"E", "T", "P", "PL", "pitt", "pitx", "pity", "pitn", "pixx", "pixy", "pixn", "piyy", "piyn", "pinn",
               "Wt", "Wx", "Wy", "Wn", "bulkPi"}


def _flow_and_normal(rng, n, three_d):
    tau = rng.uniform(0.6, 12.0, n)
    x = rng.uniform(-10.0, 10.0, n)
    y = rng.uniform(-10.0, 10.0, n)
    eta = rng.uniform(-3.5, 3.5, n) if three_d else np.zeros(n)
    rho = rng.uniform(0.0, 1.1, n)
    psi = rng.uniform(0.0, 2.0 * np.pi, n)
    ux = np.sinh(rho) * np.cos(psi)
    uy = np.sinh(rho) * np.sin(psi)
    un = rng.normal(0.0, 0.15, n) / tau if three_d else np.zeros(n)
    v0 = 0.02
    dat = tau * rng.uniform(0.5, 2.0, n) * v0
    dax = tau * rng.normal(0.0, 0.2, n) * v0
    day = tau * rng.normal(0.0, 0.2, n) * v0
    dan = tau * rng.normal(0.0, 0.2, n) * v0 if three_d else np.zeros(n)
    # resample the spatial normal until u.dsigma > 0 everywhere
    for _ in range(100):
        ut = np.sqrt(1.0 + ux * ux + uy * uy + tau * tau * un * un)
        bad = (ut * dat + ux * dax + uy * day + un * dan) <= 0.0
        if not bad.any():
            break
        k = int(bad.sum())
        dax[bad] = tau[bad] * rng.normal(0.0, 0.2, k) * v0
        day[bad] = tau[bad] * rng.normal(0.0, 0.2, k) * v0
        if three_d:
            dan[bad] = tau[bad] * rng.normal(0.0, 0.2, k) * v0
    else:
        raise RuntimeError("could not make u.dsigma > 0")
    return tau, x, y, eta, dat, dax, day, dan, ux, uy, un


def surface_vh(n_cells, seed, three_d=True, viscous=True, stress=False):
    """Mode-1 (20 column) viscous-hydro surface: cfg2 (three_d=False, viscous=False) / cfg3 / cfg4."""
    rng = np.random.default_rng(seed)
    tau, x, y, eta, dat, dax, day, dan, ux, uy, un = _flow_and_normal(rng, n_cells, three_d)
    T = 0.150 * (1.0 + rng.uniform(-0.02, 0.02, n_cells))
    E = np.full(n_cells, 0.30)
    P = np.full(n_cells, 0.05)
    s_pi, s_bulk = (0.03, 0.01) if stress else (0.002, 0.002)   # stress: ~27 % of cells take the feqmod breakdown branch
    if viscous:
        pixx = rng.normal(0.0, s_pi, n_cells)
        pixy = rng.normal(0.0, s_pi, n_cells)
        pixn = rng.normal(0.0, s_pi, n_cells) / tau
        piyy = rng.normal(0.0, s_pi, n_cells)
        piyn = rng.normal(0.0, s_pi, n_cells) / tau
        bulk = np.clip(rng.normal(0.0, s_bulk, n_cells), -0.3 * P, 0.3 * P)
        if not three_d:
            pixn[:] = 0.0
            piyn[:] = 0.0
    else:
        pixx = pixy = pixn = piyy = piyn = bulk = np.zeros(n_cells)
    gev = [E, T, P, pixx, pixy, pixn, piyy, piyn, bulk]
    cols = [tau, x, y, eta, dat, dax, day, dan, ux, uy, un] + [g / HBARC for g in gev]
    return np.stack(cols, axis=1)


def surface_vah(n_cells, seed):
    """Mode-2 (31 column) anisotropic-hydro surface, PL matching: cfg5."""
    rng = np.random.default_rng(seed)
    tau, x, y, eta, dat, dax, day, dan, ux, uy, un = _flow_and_normal(rng, n_cells, True)
    ut = np.sqrt(1.0 + ux * ux + uy * uy + tau * tau * un * un)
    T = 0.150 * (1.0 + rng.uniform(-0.02, 0.02, n_cells))
    E = np.full(n_cells, 0.30)
    P = np.full(n_cells, 0.05)
    PL = P * rng.uniform(0.4, 1.2, n_cells)
    s = 0.002
    pi = [rng.normal(0.0, s, n_cells) for _ in range(10)]   # tt tx ty tn xx xy xn yy yn nn
    for k in (3, 6, 8):
        pi[k] = pi[k] / tau
    pi[9] = pi[9] / (tau * tau)
    Wt = rng.normal(0.0, 0.005, n_cells)
    Wx = rng.normal(0.0, 0.005, n_cells)
    Wy = rng.normal(0.0, 0.005, n_cells)
    Wn = rng.normal(0.0, 0.005, n_cells) / tau
    bulk = np.clip(rng.normal(0.0, 0.002, n_cells), -0.3 * P, 0.3 * P)
    gev = [E, T, P, PL] + pi + [Wt, Wx, Wy, Wn, bulk]
    cols = [tau, x, y, eta, dat, dax, day, dan, ut, ux, uy, un] + [g / HBARC for g in gev]
    return np.stack(cols, axis=1)


def columns_to_cells(columns, mode=1):
    """File columns -> SoA dict in GeV units, one `value * hbarC` per converted entry like the readers."""
    names = MODE1_COLUMNS if mode == 1 else MODE2_COLUMNS
    a = np.asarray(columns, dtype=np.float64)
    if a.shape[1] < len(names):
        raise ValueError("surface has %d columns, mode %d needs %d" % (a.shape[1], mode, len(names)))
    out = {}
    for j, nm in enumerate(names):
        col = np.ascontiguousarray(a[:, j])
        out[nm] = col * HBARC if nm in _GEV_FIELDS else col
    return out


VORTICITY_COLUMNS = ("wtx", "wty", "wtn", "wxy", "wxn", "wyn")


def vorticity(n_cells, seed):
    """Thermal vorticity of a mode-5 surface: the six extra columns (covariant Milne components varpi_{tau x}, varpi_{tau y},
    varpi_{tau eta}, varpi_{xy}, varpi_{x eta}, varpi_{y eta}, dimensionless) as a dict of arrays.  The eta components carry a factor
    tau ~ 5 fm relative to the others, as covariant components do."""
    rng = np.random.default_rng(seed)
    s = np.array([0.02, 0.02, 0.1, 0.02, 0.1, 0.1])
    return {k: rng.normal(0.0, s[j], n_cells) for j, k in enumerate(VORTICITY_COLUMNS)}


THERMAL_SHEAR_COLUMNS = ("xtt", "xtx", "xty", "xtn", "xxx", "xxy", "xxn", "xyy", "xyn", "xnn")


def thermal_shear(n_cells, seed):
    """Thermal shear xi_{mu nu} = (1/2)(d_mu beta_nu + d_nu beta_mu) for input/thermal_shear.dat: the ten covariant Milne components
    xi_{tau tau}, xi_{tau x}, xi_{tau y}, xi_{tau eta}, xi_{xx}, xi_{xy}, xi_{x eta}, xi_{yy}, xi_{y eta}, xi_{eta eta} (dimensionless)
    as a dict of arrays.  Each eta index carries a factor tau ~ 5 fm relative to the others, as covariant components do."""
    rng = np.random.default_rng(seed)
    s = np.array([0.02, 0.02, 0.02, 0.1, 0.02, 0.02, 0.1, 0.02, 0.1, 0.5])
    return {k: rng.normal(0.0, s[j], n_cells) for j, k in enumerate(THERMAL_SHEAR_COLUMNS)}


BARYON_GRADIENT_COLUMNS = ("dt", "dx", "dy", "dn")


def baryon_gradient(n_cells, seed):
    """Gradient of alpha_B = muB/T for input/muB_over_T_gradient.dat: the four covariant Milne components d_tau alpha_B, d_x alpha_B,
    d_y alpha_B (1/fm) and d_eta alpha_B (dimensionless) as a dict of arrays.  The eta component carries a factor tau ~ 5 fm relative to
    the others, as a covariant component does."""
    rng = np.random.default_rng(seed)
    s = np.array([0.1, 0.1, 0.1, 0.5])
    return {k: rng.normal(0.0, s[j], n_cells) for j, k in enumerate(BARYON_GRADIENT_COLUMNS)}
