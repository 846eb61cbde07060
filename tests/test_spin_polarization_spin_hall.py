"""Spin polarization from the spin Hall effect (gradient of alpha_B = muB/T): the oracle against an independent restatement in Milne
coordinates, the algebra of N_she, the anchor to the vorticity oracle's Snorm, cart_gradient against central differences, the side-file
reader, the parameter key, the ABI and (on the GPU) the CUDA path."""
import ctypes as C
import itertools
import os
import subprocess
import tempfile

import numpy as np
import pytest

from common import compare
from is3d_b200 import api, synthetic, tables, workdir
from oracle import cf_polzn, cf_polzn_she

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HBARC = synthetic.HBARC
N_KEYS = ("St", "Sx", "Sy", "Sz")
GB = synthetic.BARYON_GRADIENT_COLUMNS
CHOSEN = [3122, -3122, 2212, -2212, 211, 321]


def _small_grid(fx, dimension):
    """A few points of every table (the eta table thinned in 2+1D) to keep the numpy restatement quick."""
    g = tables.grid(fx)
    g = dict(g, pT=g["pT"][::8].copy(), pT_weight=g["pT_weight"][::8].copy(), phi=g["phi"][::5].copy(), phi_weight=g["phi_weight"][::5].copy(),
             y=g["y"][::4].copy(), y_weight=g["y_weight"][::4].copy())
    if dimension == 2:
        g = dict(g, eta=g["eta"][::12].copy(), eta_weight=g["eta_weight"][::12].copy())
    return g


def _species(fx, chosen=CHOSEN):
    """Baryons, antibaryons and mesons of the list, plus a Theta = -1 species with q_B = 1 (the Lambda's mass and g): the boson
    occupation with a non-zero baryon number."""
    sp = tables.species(fx, 1, chosen)
    i = list(chosen).index(3122) if 3122 in chosen else 0
    return {k: np.append(np.asarray(sp[k], dtype=np.float64), {"sign": -1.0, "baryon": 1.0}.get(k, sp[k][i])) for k in
            ("mass", "sign", "degeneracy", "baryon")}


def _problem(n_cells, seed, dimension, flip=0):
    cells = synthetic.columns_to_cells(synthetic.surface_vh(n_cells, seed, three_d=(dimension == 3)), 1)
    if flip:                                     # cells with u.dsigma <= 0
        for k in ("dat", "dax", "day"):
            cells[k] = cells[k].copy()
        cells["dat"][:flip] = -cells["dat"][:flip]
    return cells, synthetic.baryon_gradient(n_cells, seed + 11)


def _momenta(sp, g, dimension):
    y = np.zeros_like(g["y"]) if dimension == 2 else g["y"]
    yy, ff, pp, mm = np.meshgrid(y, g["phi"], g["pT"], sp["mass"], indexing="ij")     # the flat bin order [y][phi][pT][species]
    mT = np.sqrt(mm * mm + pp * pp)
    return np.stack([(mT * np.cosh(yy)).ravel(), (pp * np.cos(ff)).ravel(), (pp * np.sin(ff)).ravel(), (mT * np.sinh(yy)).ravel()]), mm.ravel()


def numpy_milne(flags, cells, grad, sp, g):
    """N_she^mu and Snorm restated in Milne coordinates: eps^{tau x y eta} = 1/tau, p_mu lowered with g = diag(1, -1, -1, -tau^2),
    d_sigma alpha_B taken from the columns as they are, that_mu = (cosh eta, 0, 0, tau sinh eta), varpi_{rho sigma} replaced by
    -2 q_B that_rho hbar c d_sigma alpha_B / E, the contravariant result converted to Cartesian components (A^t = cosh eta A^tau +
    tau sinh eta A^eta, A^z = sinh eta A^tau + tau cosh eta A^eta).  Evaluated in extended precision (np.longdouble): the Milne
    contraction cancels terms of order cosh^2 eta."""
    L = np.longdouble
    cells = {k: np.asarray(v, dtype=L) for k, v in cells.items()}
    grad = {k: np.asarray(v, dtype=L) for k, v in grad.items()}
    sp = {k: np.asarray(sp[k], dtype=L) for k in ("mass", "sign", "degeneracy", "baryon")}
    g = {k: np.asarray(g[k], dtype=L) for k in ("pT", "phi", "y", "eta", "eta_weight")}
    eps = np.zeros((4, 4, 4, 4), dtype=L)
    for perm in itertools.permutations(range(4)):
        eps[perm] = np.linalg.det(np.eye(4)[list(perm)])
    pref = (2 * np.pi * L(HBARC)) ** -3
    ns, npT, nphi, ny = len(sp["mass"]), len(g["pT"]), len(g["phi"]), len(g["y"])
    d2 = flags["dimension"] == 2
    N = np.zeros((4, ny, nphi, npT, ns), dtype=L); Sn = np.zeros((ny, nphi, npT, ns), dtype=L)
    m = sp["mass"][None, None, :]; sign = sp["sign"][None, None, :]; qB = sp["baryon"][None, None, :]
    pT = g["pT"][None, :, None]; phi = g["phi"][:, None, None]
    mT = np.sqrt(m * m + pT * pT)
    px = pT * np.cos(phi) + 0 * m; py = pT * np.sin(phi) + 0 * m
    for i in range(len(cells["tau"])):
        tau = cells["tau"][i]; ux, uy, un = cells["ux"][i], cells["uy"][i], cells["un"][i]
        ut = np.sqrt(1 + ux * ux + uy * uy + tau * tau * un * un)
        dat, dax, day, dan = (cells[k][i] for k in ("dat", "dax", "day", "dan"))
        if ut * dat + ux * dax + uy * day + un * dan <= 0:
            continue
        z = np.array([grad[k][i] for k in GB], dtype=L) * L(HBARC)
        for iy in range(1 if d2 else ny):
            y = L(0) if d2 else g["y"][iy]
            E = mT * np.cosh(y)
            slots = zip(g["eta"], g["eta_weight"]) if d2 else [(cells["eta"][i], 1.0)]
            for eta, wt in slots:
                pt = mT * np.cosh(y - eta); pn = mT / tau * np.sinh(y - eta)
                pds = wt * (pt * dat + px * dax + py * day + pn * dan)
                pu = pt * ut - px * ux - py * uy - tau * tau * pn * un
                with np.errstate(over="ignore"):
                    f = 1.0 / (np.exp(pu / cells["T"][i]) + sign)
                keep = (pds > 0) if flags["outflow"] else np.ones_like(pds, dtype=bool)
                t = np.where(keep, pds * f, 0.0)
                plow = np.stack(np.broadcast_arrays(pt, -px, -py, -tau * tau * pn))
                that = np.array([np.cosh(eta), 0, 0, tau * np.sinh(eta)], dtype=L)
                W = np.einsum("r,s->rs", that, z)                                     # that_rho zeta_sigma
                A = np.einsum("abcd,bc,d...->a...", eps, W, plow) / tau * (-2.0 * qB / E)
                At = np.cosh(eta) * A[0] + tau * np.sinh(eta) * A[3]
                Az = np.sinh(eta) * A[0] + tau * np.cosh(eta) * A[3]
                Ac = np.stack([At, A[1], A[2], Az])
                Sn[iy] += pref * sp["degeneracy"] * t
                N[:, iy] += pref * sp["degeneracy"] * t * (1 - sign * f) * (-Ac / (8 * m))
    return {k: N[j].ravel().astype(np.float64) for j, k in enumerate(N_KEYS)} | {"Snorm": Sn.ravel().astype(np.float64)}


@pytest.mark.parametrize("dimension,outflow", [(3, 1), (2, 1), (3, 0)])
def test_oracle_matches_milne_restatement(fx, dimension, outflow):
    cells, gb = _problem(20, 5050 + dimension, dimension)
    sp = _species(fx); g = _small_grid(fx, dimension)
    fl = tables.flags(df_mode=1, dimension=dimension, outflow=outflow)
    got, skipped, cond = cf_polzn_she.spin_polarization_spin_hall(fl, cells, gb, sp, g, conditioning=True)
    want = numpy_milne(fl, cells, gb, sp, g)
    assert skipped == 0
    assert np.all(np.abs(got["Snorm"] - want["Snorm"]) <= 1e-13 * np.abs(want["Snorm"]))
    assert np.all(got["St"] == 0)
    assert np.all(np.abs(want["St"]) <= 1e-13 * (cond["Sx"] + cond["Sy"] + cond["Sz"]))      # 0 up to the Milne -> Cartesian rounding
    for k in ("Sx", "Sy", "Sz"):
        assert np.any(got[k] != 0)
        assert np.all(np.abs(got[k] - want[k]) <= 1e-13 * cond[k]), k


def _rest_cell(a):
    cells = {k: np.zeros(1) for k in ("eta", "dax", "day", "dan", "ux", "uy", "un")}
    cells.update(tau=np.ones(1), dat=np.ones(1), T=np.full(1, 0.15), P=np.full(1, 0.05), E=np.full(1, 0.3))
    gb = {k: np.zeros(1) for k in GB}
    gb["dx"] = np.full(1, a)
    return cells, gb


def test_analytic_anchor_cell_at_rest(fx):
    """Only d_x alpha_B = a at rest, eta = 0: N_she = (q_B hbar c a W / (4 m E)) (0, -p^z, p^y), W = p.dsigma f (1 - Theta f)."""
    a = 0.3
    cells, gb = _rest_cell(a)
    sp = _species(fx); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=3)
    r, _ = cf_polzn_she.spin_polarization_spin_hall(fl, cells, gb, sp, g)
    p, m = _momenta(sp, g, 3)
    _, _, _, sg = np.meshgrid(g["y"], g["phi"], g["pT"], sp["sign"], indexing="ij")
    _, _, _, qb = np.meshgrid(g["y"], g["phi"], g["pT"], sp["baryon"], indexing="ij")
    with np.errstate(over="ignore"):
        f = 1.0 / (np.exp(p[0] / 0.15) + sg.ravel())
    fbar = 1 - sg.ravel() * f
    nz = r["Snorm"] > 0
    assert nz.sum() > 0.9 * nz.size
    c = qb.ravel() * HBARC * a * fbar / (4 * m * p[0])           # N / Snorm, Snorm = pref g E f
    want = [np.zeros_like(c), -c * p[3], c * p[2]]
    for k, w in zip(("Sx", "Sy", "Sz"), want):
        got = r[k][nz] / r["Snorm"][nz]
        assert np.allclose(got, w[nz], rtol=1e-12, atol=1e-15 * np.abs(w[nz]).max()), k
    assert np.all(r["St"] == 0) and np.all(r["Sx"] == 0)
    pN = p[1] * r["Sx"] + p[2] * r["Sy"] + p[3] * r["Sz"]
    assert np.all(np.abs(pN) <= 1e-15 * np.abs(p[3] * r["Sz"]) + 1e-300)


def test_algebra_orthogonality_charge_and_linearity(fx):
    cells, gb = _problem(15, 93, 3)
    sp = _species(fx); g = _small_grid(fx, 3)
    fl = tables.flags(df_mode=1, dimension=3)
    r1, _, c1 = cf_polzn_she.spin_polarization_spin_hall(fl, cells, gb, sp, g, conditioning=True)
    assert np.all(r1["St"] == 0)
    p, _ = _momenta(sp, g, 3)
    pN = p[1] * r1["Sx"] + p[2] * r1["Sy"] + p[3] * r1["Sz"]           # p.N_she = E N^t - p.N with N^t = 0
    norm = np.sqrt(sum(r1[k] ** 2 for k in ("Sx", "Sy", "Sz")))
    assert np.all(np.abs(pN) <= 1e-13 * np.sqrt(p[1] ** 2 + p[2] ** 2 + p[3] ** 2) * np.maximum(norm, sum(c1[k] for k in N_KEYS)))
    # mesons: exact zeros; the antibaryon of the list (Lambda-bar: the Lambda's mass, g and Theta) exactly -N(Lambda)
    ns = len(sp["mass"])
    sh = (-1, ns)
    meson = sp["baryon"] == 0
    assert meson.any()
    for k in N_KEYS:
        v = r1[k].reshape(sh)
        assert np.all(v[:, meson] == 0), k
        assert np.array_equal(v[:, CHOSEN.index(-3122)], -v[:, CHOSEN.index(3122)]), k
    assert np.any(r1["Sx"].reshape(sh)[:, CHOSEN.index(3122)] != 0)
    zero = {k: np.zeros_like(v) for k, v in gb.items()}
    r0, _ = cf_polzn_she.spin_polarization_spin_hall(fl, cells, zero, sp, g)
    assert all(np.all(r0[k] == 0) for k in N_KEYS) and np.array_equal(r0["Snorm"], r1["Snorm"])
    gb2 = synthetic.baryon_gradient(15, 94)
    r2, _, c2 = cf_polzn_she.spin_polarization_spin_hall(fl, cells, gb2, sp, g, conditioning=True)
    mix = {k: 2.0 * gb[k] - 0.5 * gb2[k] for k in gb}
    r3, _ = cf_polzn_she.spin_polarization_spin_hall(fl, cells, mix, sp, g)
    for k in ("Sx", "Sy", "Sz"):
        assert np.all(np.abs(r3[k] - (2.0 * r1[k] - 0.5 * r2[k])) <= 1e-13 * (2.0 * c1[k] + 0.5 * c2[k])), k


@pytest.mark.parametrize("dimension", [3, 2])
def test_snorm_is_the_vorticity_oracles(fx, dimension):
    cells, gb = _problem(30, 43 + dimension, dimension, flip=3)
    vort = synthetic.vorticity(30, 5)
    sp = _species(fx); g = _small_grid(fx, dimension)
    fl = tables.flags(df_mode=1, dimension=dimension)
    r, skipped = cf_polzn_she.spin_polarization_spin_hall(fl, cells, gb, sp, g)
    rv, skipped_v = cf_polzn.spin_polarization(fl, cells, vort, sp, g)
    assert skipped == skipped_v == 3
    assert np.array_equal(r["Snorm"], rv["Snorm"])


def test_cart_gradient_matches_central_differences():
    """The oracle's copy of cart_gradient() against d_a alpha of alpha(tau(t, z), x, y, eta(t, z)) = d_tau tau + d_x x + d_y y +
    d_eta eta (linear in the Milne coordinates, so its Milne gradient is the four columns), by central differences in t and z."""
    rng = np.random.default_rng(17)
    for tau, eta in [(0.6, 0.0), (5.0, 1.3), (9.0, -2.4)]:
        d = rng.normal(0.0, 1.0, 4)
        t, z = tau * np.cosh(eta), tau * np.sinh(eta)
        alpha = lambda t, x, y, z: d[0] * np.sqrt(t * t - z * z) + d[1] * x + d[2] * y + d[3] * np.arctanh(z / t)
        h = 1e-6 * tau
        want = np.array([(alpha(t + h, 0, 0, z) - alpha(t - h, 0, 0, z)) / (2 * h), d[1], d[2],
                         (alpha(t, 0, 0, z + h) - alpha(t, 0, 0, z - h)) / (2 * h)])
        got = cf_polzn_she.cart_gradient(d, tau, eta)
        scale = np.abs(d).sum() * max(1.0, 1.0 / tau) * np.cosh(eta)
        assert np.all(np.abs(got - want) <= 1e-8 * scale), (tau, eta, got, want)


def test_boost_invariant_zz_vanishes(fx):
    """2+1D, d_eta alpha_B = 0, a symmetric eta table: the weights are even in eta and zeta_z = -sinh eta d_tau alpha_B is odd, so Z_z
    (and with p^z = 0 at y = 0 every N^x, N^y it feeds) vanishes up to rounding."""
    cells, gb = _problem(25, 71, 2)
    gb["dn"] = np.zeros_like(gb["dn"])
    sp = _species(fx); g = _small_grid(fx, 2)
    assert np.allclose(g["eta"], -g["eta"][::-1]) and np.allclose(g["eta_weight"], g["eta_weight"][::-1])
    assert np.all(cells["un"] == 0) and np.all(cells["dan"] == 0)
    fl = tables.flags(df_mode=1, dimension=2)
    r, _, cond = cf_polzn_she.spin_polarization_spin_hall(fl, cells, gb, sp, g, conditioning=True)
    ssum = cond["Sx"] + cond["Sy"] + cond["Sz"]
    for k in ("Sx", "Sy"):
        assert np.all(np.abs(r[k]) <= 1e-12 * ssum), k
    assert np.any(r["Sz"] != 0)


# ------------------------------------------------------------------------------------------------ host layer, ABI
def _host_dump(wd):
    import struct
    lib = api.lib()
    out = os.path.join(wd, "host_dump.bin")
    lib.is3d_b200_host_error.restype = C.c_char_p
    rc = lib.is3d_b200_host_dump(wd.encode(), out.encode())
    if rc != 0:
        return rc, lib.is3d_b200_host_error().decode()
    rec, data, pos = {}, open(out, "rb").read(), 0
    while pos < len(data):
        (ln,) = struct.unpack_from("<i", data, pos); pos += 4
        name = data[pos:pos + ln].decode(); pos += ln
        (n,) = struct.unpack_from("<q", data, pos); pos += 8
        rec[name] = np.frombuffer(data, dtype="<f8", count=n, offset=pos).copy(); pos += 8 * n
    return rc, rec


def _mode5_columns(n, seed, dimension=3):
    base = synthetic.surface_vh(n, seed, three_d=(dimension == 3))
    vort = synthetic.vorticity(n, seed + 1)
    xi = synthetic.thermal_shear(n, seed + 2)
    gb = synthetic.baryon_gradient(n, seed + 3)
    return np.column_stack([base] + [vort[k] for k in synthetic.VORTICITY_COLUMNS]), base, vort, xi, gb


def _materialize(wd, fx, cols, **kw):
    workdir.materialize(wd, surface_columns=cols, fixture=fx, operation=kw.pop("operation", 1), mode=kw.pop("mode", 5),
                        dimension=kw.pop("dimension", 3), df_mode=1, **kw)
    open(os.path.join(wd, "average_thermodynamic_quantities.dat"), "w").write("0.15\n0.3\n0.05\n0\n0")


def test_reader_keeps_the_gradient_columns(fx):
    cols, _, _, _, gb = _mode5_columns(9, 5)
    with tempfile.TemporaryDirectory() as wd:
        _materialize(wd, fx, cols, baryon_gradient=gb, spin_polarization=1, spin_hall_polarization=1)
        rc, d = _host_dump(wd)
        assert rc == 0, d
        for k, name in zip(GB, ("gbt", "gbx", "gby", "gbn")):
            assert np.array_equal(d[name], gb[k]), k
        _materialize(wd, fx, cols, baryon_gradient=gb, spin_polarization=1)        # without the key: no columns in the dump
        rc, d = _host_dump(wd)
        assert rc == 0 and not any(k in d for k in ("gbt", "gbx", "gby", "gbn"))


def test_reader_rejects_missing_and_short_files(fx):
    cols, _, _, _, gb = _mode5_columns(6, 15)
    a = np.column_stack([gb[k] for k in GB])
    with tempfile.TemporaryDirectory() as wd:
        _materialize(wd, fx, cols, spin_polarization=1, spin_hall_polarization=1)        # no input/muB_over_T_gradient.dat
        rc, msg = _host_dump(wd)
        assert rc == 6 and "muB_over_T_gradient.dat" in msg                             # IS3D_ERR_IO
        _materialize(wd, fx, cols, baryon_gradient=a[:5], spin_polarization=1, spin_hall_polarization=1)
        rc, msg = _host_dump(wd)
        assert rc == 6 and "5 lines" in msg
        _materialize(wd, fx, cols, baryon_gradient=a, spin_polarization=1, spin_hall_polarization=1)
        path = os.path.join(wd, "input", "muB_over_T_gradient.dat")
        lines = open(path).read().split("\n")
        lines[3] = " ".join(lines[3].split()[:3])                                         # a line with three numbers
        open(path, "w").write("\n".join(lines))
        rc, msg = _host_dump(wd)
        assert rc == 6 and "line 4" in msg and "four" in msg
        _materialize(wd, fx, cols, baryon_gradient=a, spin_polarization=1, spin_hall_polarization=1)
        assert _host_dump(wd)[0] == 0


def test_spin_hall_key_rules(fx):
    cols, _, _, _, gb = _mode5_columns(4, 25)
    with tempfile.TemporaryDirectory() as wd:
        for kw in (dict(mode=1, spin_polarization=0), dict(mode=5, spin_polarization=0), dict(mode=5, spin_polarization=1, operation=0)):
            c = cols[:, :-6] if kw["mode"] == 1 else cols
            _materialize(wd, fx, c, baryon_gradient=gb, spin_hall_polarization=1, **kw)
            assert _host_dump(wd)[0] == 2, kw                                             # IS3D_ERR_UNSUPPORTED
        _materialize(wd, fx, cols, baryon_gradient=gb, spin_polarization=1, spin_hall_polarization=0)
        assert _host_dump(wd)[0] == 0


def test_struct_layouts_match_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "is3d_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu %zu\\n", sizeof(is3d_baryon_gradient), offsetof(is3d_baryon_gradient, dt),'
                   ' offsetof(is3d_baryon_gradient, dx), offsetof(is3d_baryon_gradient, dy), offsetof(is3d_baryon_gradient, dn));'
                   ' return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    B = api.BaryonGradient
    assert got == [C.sizeof(B), B.dt.offset, B.dx.offset, B.dy.offset, B.dn.offset]
    assert [f for f, _ in B._fields_] == list(GB) == list(cf_polzn_she.BARYON_GRADIENT_FIELDS) == list(api.BARYON_GRADIENT_FIELDS)


# ------------------------------------------------------------------------------------------------ GPU
def _gpu():
    import torch
    torch.cuda.set_device(0)
    api.init()
    return torch


@pytest.mark.gpu
@pytest.mark.parametrize("dimension,outflow,chosen,memory", [
    (3, 1, "baryons", "host"), (3, 0, "baryons", "device"), (2, 1, "baryons", "host"), (2, 0, "baryons", "device"),
    (3, 1, "chosen_urqmd", "host")])
def test_gpu_parity(fx, dimension, outflow, chosen, memory):
    """Baryons, antibaryons, mesons and a Theta = -1 species with q_B != 0 (the 305-species list too), 3+1D and 2+1D, outflow on and off,
    cells with u.dsigma <= 0, host and device memory: all four arrays against the oracle at 1e-10 per bin, St exactly 0."""
    torch = _gpu()
    n = 40 if chosen == "chosen_urqmd" else 150
    cells, gb = _problem(n, 900 + dimension + 10 * outflow, dimension, flip=5)
    sp = _species(fx) if chosen == "baryons" else tables.species(fx, 1, chosen); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=dimension, outflow=outflow)
    ref, skipped, cond = cf_polzn_she.spin_polarization_spin_hall(fl, cells, gb, sp, g, conditioning=True)
    if memory == "device":
        dc = {k: torch.tensor(v, device="cuda") for k, v in cells.items()}
        dg = {k: torch.tensor(v, device="cuda") for k, v in gb.items()}
        out, st = api.spin_polarization_spin_hall(fl, dc, dg, sp, g, memory="device")
        torch.cuda.synchronize()
        got = {k: v.cpu().numpy() for k, v in out.items()}
    else:
        got, st = api.spin_polarization_spin_hall(fl, cells, gb, sp, g)
    assert skipped == 5 and st["cells_skipped_udsigma"] == 5
    assert np.all(got["St"] == 0)
    assert compare(got["Snorm"], ref["Snorm"])["ok"], compare(got["Snorm"], ref["Snorm"])
    meson = np.tile(np.asarray(sp["baryon"]) == 0, got["Sx"].size // len(sp["mass"]))
    for k in ("Sx", "Sy", "Sz"):
        rep = compare(got[k], ref[k], conditioning=cond[k])
        assert rep["ok"], (k, rep)
        assert np.all(got[k][meson] == 0) and np.any(got[k] != 0), k


def _raw_call(fl, cells, gb, sp, g, fill=7.0):
    """is3d_b200_spin_polarization_spin_hall on host arrays pre-filled with `fill`: (return code, the five arrays)."""
    m = api._Marshal(False)
    no_baryon = sp.get("baryon") is None
    if no_baryon:
        sp = dict(sp, baryon=np.zeros(len(sp["mass"])))
    sf, spc, gr, _, _ = api._marshal_problem(m, cells, sp, g, None, None)
    gd = None
    if gb is not None:
        gd = api.BaryonGradient()
        for k in GB:
            if gb.get(k) is not None:
                setattr(gd, k, m.cells(gb[k]))
    if no_baryon:
        spc.baryon = None
    n = spc.n * gr.n_pT * gr.n_phi * gr.n_y
    out = {k: np.full(n, fill) for k in api.POLARIZATION_FIELDS}
    res = api.PolarizationResult(*[out[k].ctypes.data_as(api._D) for k in api.POLARIZATION_FIELDS])
    f = api.lib().is3d_b200_spin_polarization_spin_hall
    f.restype = C.c_int
    opt = api.Options()
    flags = api.make_flags(fl)
    rc = f(C.byref(flags), C.byref(sf), C.byref(gd) if gd is not None else None, C.byref(spc), C.byref(gr), C.byref(opt), C.byref(res), None)
    return rc, out


@pytest.mark.gpu
def test_gpu_empty_surface_and_errors(fx):
    _gpu()
    sp = _species(fx); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=3)
    cells, gb = _problem(0, 1, 3)
    out, st = api.spin_polarization_spin_hall(fl, cells, gb, sp, g)
    assert all(np.all(v == 0) for v in out.values()) and st["cells_skipped_udsigma"] == 0
    cells, gb = _problem(10, 2, 3)
    massless = dict(sp, mass=np.where(np.arange(len(sp["mass"])) == 0, 0.0, sp["mass"]))
    cases = [(dict(fl, mode=2), gb, sp, 2), (dict(fl, include_baryon=1), gb, sp, 2), (fl, None, sp, 1), (fl, dict(gb, dn=None), sp, 1),
             (fl, dict(gb, dt=None), sp, 1), (fl, gb, massless, 1), (fl, gb, dict(sp, baryon=None), 1)]
    for bad_fl, bad_gb, bad_sp, code in cases:
        rc, arrs = _raw_call(bad_fl, cells, bad_gb, bad_sp, g)
        assert rc == code, (rc, code)
        assert all(np.all(v == 7.0) for v in arrs.values())
    with pytest.raises(api.Is3dError) as e:
        api.spin_polarization_spin_hall(fl, cells, None, sp, g)
    assert e.value.code == 1
    rc, arrs = _raw_call(fl, cells, gb, sp, g)                                     # the same call without a fault adds into the arrays
    assert rc == 0 and np.all(arrs["St"] == 7.0) and np.any(arrs["Sx"] != 7.0)


@pytest.mark.gpu
@pytest.mark.parametrize("dimension", [3, 2])
def test_gpu_snorm_bitwise_reproducible_and_multi(fx, dimension):
    _gpu()
    cells, gb = _problem(300, 677 + dimension, dimension, flip=2)
    vort = synthetic.vorticity(300, 9)
    sp = _species(fx); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=dimension)
    a, _ = api.spin_polarization_spin_hall(fl, cells, gb, sp, g)
    b, _ = api.spin_polarization_spin_hall(fl, cells, gb, sp, g)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    v, _ = api.spin_polarization(fl, cells, vort, sp, g)
    assert np.array_equal(a["Snorm"], v["Snorm"])
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("_multi needs at least two devices")
    api.init_devices(0)
    m, st = api.spin_polarization_spin_hall(fl, cells, gb, sp, g, multi=True)
    assert st["n_gpus"] >= 2
    for k in a:
        scale = np.abs(a[k]).max()
        assert np.abs(m[k] - a[k]).max() <= 1e-13 * scale, k


def _run(wd):
    lib = api.lib()
    lib.is3d_b200_host_error.restype = C.c_char_p
    rc = lib.is3d_b200_run_workdir(wd.encode(), None, C.c_int64(0), None, 0, None)
    assert rc == 0, lib.is3d_b200_host_error().decode()
    res = os.path.join(wd, "results")
    files = sorted(os.path.relpath(os.path.join(d, f), res) for d, _, fs in os.walk(res) for f in fs)
    return files, {f: open(os.path.join(res, f), "rb").read() for f in files if f.startswith("polarization" + os.sep)}


@pytest.mark.gpu
@pytest.mark.parametrize("dimension,shear", [(3, True), (2, False)])
def test_gpu_workdir_spin_hall_files(fx, dimension, shear):
    """With the key: S_she_<mcid>.dat holds the API's spin Hall part and the totals of mean_spin(vort, shear=, spin_hall=), S_ and S_xi_
    are byte-identical, S_fd_ is the feed-down of the summed arrays; without it (absent or 0) the run writes the files it wrote before."""
    _gpu()
    cols, base, vort, xi, gb = _mode5_columns(60, 6421 + dimension, dimension)
    chosen = [211, 3122, -3122, 3212, -3212, 3224, -3224]
    common_kw = dict(spin_polarization=1, polarization_feed_down=1, thermal_shear=xi, baryon_gradient=gb)
    if shear:
        common_kw["thermal_shear_polarization"] = 1
    runs = {}
    for label, extra in (("absent", {}), ("zero", dict(spin_hall_polarization=0)), ("on", dict(spin_hall_polarization=1))):
        with tempfile.TemporaryDirectory() as wd:
            workdir.materialize(wd, surface_columns=cols, chosen=chosen, fixture=fx, operation=1, mode=5, dimension=dimension, df_mode=1,
                                **common_kw, **extra)
            open(os.path.join(wd, "average_thermodynamic_quantities.dat"), "w").write("0.15\n0.3\n0.05\n0\n0")
            runs[label] = _run(wd)
    assert runs["absent"][0] == runs["zero"][0]
    assert not any("S_she_" in f for f in runs["absent"][0])
    for f, text in runs["absent"][1].items():
        assert runs["zero"][1][f] == text, f
    she_files = ["polarization" + os.sep + "S_she_%d.dat" % c for c in chosen]
    assert runs["on"][0] == sorted(runs["absent"][0] + she_files)
    for f, text in runs["absent"][1].items():
        if not os.path.basename(f).startswith("S_fd_"):
            assert runs["on"][1][f] == text, f                        # S_ and S_xi_ byte-identical with the key
    header = runs["on"][1][she_files[0]].decode().split("\n", 1)[0].split()
    assert header == ["y", "phip", "pT", "Snorm", "Sx_she", "Sy_she", "Sz_she", "Sx", "Sy", "Sz", "Sx_rest", "Sy_rest", "Sz_rest"]

    cells = synthetic.columns_to_cells(base, 1)
    sp = tables.species(fx, 1, chosen); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=dimension)
    rv, _ = api.spin_polarization(fl, cells, vort, sp, g)
    rx, _ = api.spin_polarization_shear(fl, cells, xi, sp, g) if shear else (None, None)
    rh, _ = api.spin_polarization_spin_hall(fl, cells, gb, sp, g)
    S, rest = api.mean_spin(rv, sp, g, dimension, shear=rx, spin_hall=rh)
    Sh, _ = api.mean_spin(rh, sp, g, dimension)
    ny = 1 if dimension == 2 else len(g["y"])
    shape = (len(g["y"]), len(g["phi"]), len(g["pT"]), -1)

    def check(text, cols_want, label):
        got = np.loadtxt(text.decode().splitlines(), skiprows=1, ndmin=2)[:, 3:]
        want = np.column_stack([v.reshape(shape)[:ny, :, :, s].ravel() for v in cols_want])
        assert got.shape == want.shape
        scale = np.abs(want).max(axis=0)
        assert np.all(np.abs(got - want) <= 2e-8 * np.abs(want) + 1e-12 * scale), label

    for s, (c, f) in enumerate(zip(chosen, she_files)):
        check(runs["on"][1][f], [rh["Snorm"]] + list(Sh[1:]) + list(S[1:]) + list(rest), c)
    lam = chosen.index(3122)
    assert np.any(rh["Sx"].reshape(shape)[:ny, :, :, lam] != 0)

    total = {k: rv[k] + (rx[k] if shear else 0.0) + rh[k] if k != "Snorm" else rv[k] for k in api.POLARIZATION_FIELDS}
    pdg = tables.pdg_decay_table(fx, 1)
    first = {}
    for n, m in enumerate(pdg["mcid"]):
        first.setdefault(int(m), n)
    fed, _ = api.polarization_decays(pdg, tables.spin_parity(fx, pdg, 1), [first[m] for m in chosen], g, dimension, total)
    Sf, rest_f = api.mean_spin(fed, sp, g, dimension)
    for s, c in enumerate(chosen):
        f = "polarization" + os.sep + "S_fd_%d.dat" % c
        check(runs["on"][1][f], [fed["Snorm"]] + list(Sf) + list(rest_f), ("fd", c))
