"""Spin polarization from thermal shear: the oracle against an independent restatement in Milne coordinates, the algebra of N_xi, the
anchor to the vorticity oracle's Snorm, cart_shear against a numeric Jacobian, the side-file reader, the parameter key, the ABI and (on
the GPU) the CUDA path."""
import ctypes as C
import itertools
import os
import subprocess
import tempfile

import numpy as np
import pytest

from common import compare
from is3d_b200 import api, synthetic, tables, workdir
from oracle import cf_polzn, cf_polzn_xi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HBARC = synthetic.HBARC
N_KEYS = ("St", "Sx", "Sy", "Sz")
XI = synthetic.THERMAL_SHEAR_COLUMNS


def _small_grid(fx, dimension):
    """A few points of every table (the eta table thinned in 2+1D) to keep the numpy restatement quick."""
    g = tables.grid(fx)
    g = dict(g, pT=g["pT"][::8].copy(), pT_weight=g["pT_weight"][::8].copy(), phi=g["phi"][::5].copy(), phi_weight=g["phi_weight"][::5].copy(),
             y=g["y"][::4].copy(), y_weight=g["y_weight"][::4].copy())
    if dimension == 2:
        g = dict(g, eta=g["eta"][::12].copy(), eta_weight=g["eta_weight"][::12].copy())
    return g


def _problem(n_cells, seed, dimension, flip=0):
    cells = synthetic.columns_to_cells(synthetic.surface_vh(n_cells, seed, three_d=(dimension == 3)), 1)
    if flip:                                     # cells with u.dsigma <= 0
        for k in ("dat", "dax", "day"):
            cells[k] = cells[k].copy()
        cells["dat"][:flip] = -cells["dat"][:flip]
    return cells, synthetic.thermal_shear(n_cells, seed + 11)


def _momenta(sp, g, dimension):
    y = np.zeros_like(g["y"]) if dimension == 2 else g["y"]
    yy, ff, pp, mm = np.meshgrid(y, g["phi"], g["pT"], sp["mass"], indexing="ij")     # the flat bin order [y][phi][pT][species]
    mT = np.sqrt(mm * mm + pp * pp)
    return np.stack([(mT * np.cosh(yy)).ravel(), (pp * np.cos(ff)).ravel(), (pp * np.sin(ff)).ravel(), (mT * np.sinh(yy)).ravel()]), mm.ravel()


def numpy_milne(flags, cells, xi, sp, g):
    """N_xi^mu and Snorm restated in Milne coordinates: eps^{tau x y eta} = 1/tau, p_mu lowered with g = diag(1, -1, -1, -tau^2),
    xi_{mu nu} taken from the columns as they are, that_mu = (cosh eta, 0, 0, tau sinh eta) (the lab time direction in covariant Milne
    components at eta), the contravariant result converted to Cartesian components (A^t = cosh eta A^tau + tau sinh eta A^eta,
    A^z = sinh eta A^tau + tau cosh eta A^eta).  Evaluated in extended precision (np.longdouble): the Milne contraction cancels terms
    of order cosh^2 eta, which in double precision would cost ~1e-12 of the per-bin sum of |products| at |eta| = 3."""
    L = np.longdouble
    cells = {k: np.asarray(v, dtype=L) for k, v in cells.items()}
    xi = {k: np.asarray(v, dtype=L) for k, v in xi.items()}
    sp = {k: np.asarray(sp[k], dtype=L) for k in ("mass", "sign", "degeneracy")}
    g = {k: np.asarray(g[k], dtype=L) for k in ("pT", "phi", "y", "eta", "eta_weight")}
    eps = np.zeros((4, 4, 4, 4), dtype=L)
    for perm in itertools.permutations(range(4)):
        eps[perm] = np.linalg.det(np.eye(4)[list(perm)])
    pref = (2 * np.pi * L(HBARC)) ** -3
    ns, npT, nphi, ny = len(sp["mass"]), len(g["pT"]), len(g["phi"]), len(g["y"])
    d2 = flags["dimension"] == 2
    N = np.zeros((4, ny, nphi, npT, ns), dtype=L); Sn = np.zeros((ny, nphi, npT, ns), dtype=L)
    m = np.asarray(sp["mass"])[None, None, :]; sign = np.asarray(sp["sign"])[None, None, :]
    pT = g["pT"][None, :, None]; phi = g["phi"][:, None, None]
    mT = np.sqrt(m * m + pT * pT)
    px = pT * np.cos(phi) + 0 * m; py = pT * np.sin(phi) + 0 * m
    for i in range(len(cells["tau"])):
        tau = cells["tau"][i]; ux, uy, un = cells["ux"][i], cells["uy"][i], cells["un"][i]
        ut = np.sqrt(1 + ux * ux + uy * uy + tau * tau * un * un)
        dat, dax, day, dan = (cells[k][i] for k in ("dat", "dax", "day", "dan"))
        if ut * dat + ux * dax + uy * day + un * dan <= 0:
            continue
        v = [xi[k][i] for k in XI]
        X = np.array([[v[0], v[1], v[2], v[3]], [v[1], v[4], v[5], v[6]], [v[2], v[5], v[7], v[8]], [v[3], v[6], v[8], v[9]]], dtype=L)
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
                pup = np.stack(np.broadcast_arrays(pt, px, py, pn))
                plow = np.stack(np.broadcast_arrays(pt, -px, -py, -tau * tau * pn))
                that = np.array([np.cosh(eta), 0, 0, tau * np.sinh(eta)], dtype=L)
                V = np.einsum("sl,l...->s...", X, pup)
                A = 2.0 * np.einsum("abcd,b,c...,d...->a...", eps, that, V, plow) / tau / E
                At = np.cosh(eta) * A[0] + tau * np.sinh(eta) * A[3]
                Az = np.sinh(eta) * A[0] + tau * np.cosh(eta) * A[3]
                Ac = np.stack([At, A[1], A[2], Az])
                Sn[iy] += pref * sp["degeneracy"] * t
                N[:, iy] += pref * sp["degeneracy"] * t * (1 - sign * f) * (-Ac / (8 * m))
    return {k: N[j].ravel().astype(np.float64) for j, k in enumerate(N_KEYS)} | {"Snorm": Sn.ravel().astype(np.float64)}


@pytest.mark.parametrize("dimension,outflow", [(3, 1), (2, 1), (3, 0)])
def test_oracle_matches_milne_restatement(fx, dimension, outflow):
    cells, xi = _problem(20, 3030 + dimension, dimension)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, dimension)
    fl = tables.flags(df_mode=1, dimension=dimension, outflow=outflow)
    got, skipped, cond = cf_polzn_xi.spin_polarization_shear(fl, cells, xi, sp, g, conditioning=True)
    want = numpy_milne(fl, cells, xi, sp, g)
    assert skipped == 0
    assert np.all(np.abs(got["Snorm"] - want["Snorm"]) <= 1e-13 * np.abs(want["Snorm"]))
    assert np.all(got["St"] == 0)
    assert np.all(np.abs(want["St"]) <= 1e-13 * (cond["Sx"] + cond["Sy"] + cond["Sz"]))      # 0 up to the Milne -> Cartesian rounding
    for k in ("Sx", "Sy", "Sz"):
        assert np.any(got[k] != 0)
        assert np.all(np.abs(got[k] - want[k]) <= 1e-13 * cond[k]), k


def _rest_cell(s):
    cells = {k: np.zeros(1) for k in ("eta", "dax", "day", "dan", "ux", "uy", "un")}
    cells.update(tau=np.ones(1), dat=np.ones(1), T=np.full(1, 0.15), P=np.full(1, 0.05), E=np.full(1, 0.3))
    xi = {k: np.zeros(1) for k in XI}
    xi["xxn"] = np.full(1, s)                    # tau = 1, eta = 0: xi_xz = xi_{x eta} / tau
    return cells, xi


def test_analytic_anchor_cell_at_rest(fx):
    """Only xi_xz = xi_zx = s at rest: N_xi = -(W s / (4 m E)) (-p^x p^y, (p^x)^2 - (p^z)^2, p^y p^z), W = p.dsigma f (1 - Theta f)."""
    s = 0.04
    cells, xi = _rest_cell(s)
    sp = tables.species(fx, 1, "chosen_pikp"); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=3)
    r, _ = cf_polzn_xi.spin_polarization_shear(fl, cells, xi, sp, g)
    p, m = _momenta(sp, g, 3)
    _, _, _, sg = np.meshgrid(g["y"], g["phi"], g["pT"], sp["sign"], indexing="ij")
    with np.errstate(over="ignore"):
        f = 1.0 / (np.exp(p[0] / 0.15) + sg.ravel())
    fbar = 1 - sg.ravel() * f
    nz = r["Snorm"] > 0
    assert nz.sum() > 0.9 * nz.size
    # N / Snorm = -(s (1 - Theta f) / (4 m E)) (...), Snorm = pref g E f
    c = -s * fbar / (4 * m * p[0])
    want = [c * -p[1] * p[2], c * (p[1] ** 2 - p[3] ** 2), c * p[2] * p[3]]
    for k, w in zip(("Sx", "Sy", "Sz"), want):
        got = r[k][nz] / r["Snorm"][nz]
        assert np.allclose(got, w[nz], rtol=1e-12, atol=1e-15 * np.abs(w[nz]).max()), k
    assert np.all(r["St"] == 0)


def test_algebra_orthogonality_zero_and_linearity(fx):
    cells, xi = _problem(15, 91, 3)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, 3)
    fl = tables.flags(df_mode=1, dimension=3)
    r1, _, c1 = cf_polzn_xi.spin_polarization_shear(fl, cells, xi, sp, g, conditioning=True)
    assert np.all(r1["St"] == 0)
    p, _ = _momenta(sp, g, 3)
    pN = p[1] * r1["Sx"] + p[2] * r1["Sy"] + p[3] * r1["Sz"]           # p.N_xi = E N^t - p.N with N^t = 0
    norm = np.sqrt(sum(r1[k] ** 2 for k in ("Sx", "Sy", "Sz")))
    assert np.all(np.abs(pN) <= 1e-13 * np.sqrt(p[1] ** 2 + p[2] ** 2 + p[3] ** 2) * np.maximum(norm, sum(c1[k] for k in N_KEYS)))
    zero = {k: np.zeros_like(v) for k, v in xi.items()}
    r0, _ = cf_polzn_xi.spin_polarization_shear(fl, cells, zero, sp, g)
    assert all(np.all(r0[k] == 0) for k in N_KEYS) and np.array_equal(r0["Snorm"], r1["Snorm"])
    xi2 = synthetic.thermal_shear(15, 92)
    r2, _, c2 = cf_polzn_xi.spin_polarization_shear(fl, cells, xi2, sp, g, conditioning=True)
    mix = {k: 2.0 * xi[k] - 0.5 * xi2[k] for k in xi}
    r3, _ = cf_polzn_xi.spin_polarization_shear(fl, cells, mix, sp, g)
    for k in ("Sx", "Sy", "Sz"):
        assert np.all(np.abs(r3[k] - (2.0 * r1[k] - 0.5 * r2[k])) <= 1e-13 * (2.0 * c1[k] + 0.5 * c2[k])), k


@pytest.mark.parametrize("dimension", [3, 2])
def test_snorm_is_the_vorticity_oracles(fx, dimension):
    cells, xi = _problem(30, 41 + dimension, dimension, flip=3)
    vort = synthetic.vorticity(30, 5)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, dimension)
    fl = tables.flags(df_mode=1, dimension=dimension)
    r, skipped = cf_polzn_xi.spin_polarization_shear(fl, cells, xi, sp, g)
    rv, skipped_v = cf_polzn.spin_polarization(fl, cells, vort, sp, g)
    assert skipped == skipped_v == 3
    assert np.array_equal(r["Snorm"], rv["Snorm"])


def test_cart_shear_matches_numeric_jacobian():
    """The oracle's copy of cart_shear() against xi_ab = J^mu_a J^nu_b xi'_{mu nu} with J = d(tau, x, y, eta)/d(t, x, y, z) taken by
    central differences of tau = sqrt(t^2 - z^2), eta = atanh(z / t)."""
    rng = np.random.default_rng(7)
    order = [(0, 0), (0, 1), (0, 2), (0, 3), (1, 1), (1, 2), (1, 3), (2, 2), (2, 3), (3, 3)]
    for tau, eta in [(0.6, 0.0), (5.0, 1.3), (9.0, -2.4)]:
        x = rng.normal(0.0, 1.0, 10)
        M = np.zeros((4, 4))
        for v, (a, b) in zip(x, order):
            M[a, b] = M[b, a] = v
        t, z = tau * np.cosh(eta), tau * np.sinh(eta)
        milne = lambda t, z: np.array([np.sqrt(t * t - z * z), np.arctanh(z / t)])
        h = 1e-6 * tau
        dt = (milne(t + h, z) - milne(t - h, z)) / (2 * h)
        dz = (milne(t, z + h) - milne(t, z - h)) / (2 * h)
        J = np.eye(4)
        J[0, 0], J[3, 0], J[0, 3], J[3, 3] = dt[0], dt[1], dz[0], dz[1]            # J[mu][a] = d x'^mu / d x^a
        want = J.T @ M @ J
        got = cf_polzn_xi.cart_shear(x, tau, eta)
        scale = np.abs(J.T) @ np.abs(M) @ np.abs(J)
        for v, (a, b) in zip(got, order):
            assert abs(v - want[a, b]) <= 1e-8 * scale[a, b], (tau, eta, a, b)


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
    return np.column_stack([base] + [vort[k] for k in synthetic.VORTICITY_COLUMNS]), base, vort, xi


def _materialize(wd, fx, cols, **kw):
    workdir.materialize(wd, surface_columns=cols, fixture=fx, operation=kw.pop("operation", 1), mode=kw.pop("mode", 5),
                        dimension=kw.pop("dimension", 3), df_mode=1, **kw)
    open(os.path.join(wd, "average_thermodynamic_quantities.dat"), "w").write("0.15\n0.3\n0.05\n0\n0")


def test_reader_keeps_the_thermal_shear_columns(fx):
    cols, _, _, xi = _mode5_columns(9, 5)
    with tempfile.TemporaryDirectory() as wd:
        _materialize(wd, fx, cols, thermal_shear=xi, spin_polarization=1, thermal_shear_polarization=1)
        rc, d = _host_dump(wd)
        assert rc == 0, d
        for k in XI:
            assert np.array_equal(d[k], xi[k]), k
        _materialize(wd, fx, cols, thermal_shear=xi, spin_polarization=1)           # without the key: no columns in the dump
        rc, d = _host_dump(wd)
        assert rc == 0 and not any(k in d for k in XI)


def test_reader_rejects_missing_and_short_files(fx):
    cols, _, _, xi = _mode5_columns(6, 15)
    a = np.column_stack([xi[k] for k in XI])
    with tempfile.TemporaryDirectory() as wd:
        _materialize(wd, fx, cols, spin_polarization=1, thermal_shear_polarization=1)     # no input/thermal_shear.dat
        assert _host_dump(wd)[0] == 6                                                     # IS3D_ERR_IO
        _materialize(wd, fx, cols, thermal_shear=a[:5], spin_polarization=1, thermal_shear_polarization=1)
        rc, msg = _host_dump(wd)
        assert rc == 6 and "5 lines" in msg
        _materialize(wd, fx, cols, thermal_shear=a, spin_polarization=1, thermal_shear_polarization=1)
        path = os.path.join(wd, "input", "thermal_shear.dat")
        lines = open(path).read().split("\n")
        lines[3] = " ".join(lines[3].split()[:9])                                         # a line with nine numbers
        open(path, "w").write("\n".join(lines))
        rc, msg = _host_dump(wd)
        assert rc == 6 and "line 4" in msg
        _materialize(wd, fx, cols, thermal_shear=a, spin_polarization=1, thermal_shear_polarization=1)
        assert _host_dump(wd)[0] == 0


def test_thermal_shear_key_rules(fx):
    cols, _, _, xi = _mode5_columns(4, 25)
    with tempfile.TemporaryDirectory() as wd:
        for kw in (dict(mode=1, spin_polarization=0), dict(mode=5, spin_polarization=0), dict(mode=5, spin_polarization=1, operation=0)):
            c = cols[:, :-6] if kw["mode"] == 1 else cols
            _materialize(wd, fx, c, thermal_shear=xi, thermal_shear_polarization=1, **kw)
            assert _host_dump(wd)[0] == 2, kw                                             # IS3D_ERR_UNSUPPORTED
        _materialize(wd, fx, cols, thermal_shear=xi, spin_polarization=1, thermal_shear_polarization=0)
        assert _host_dump(wd)[0] == 0


def test_struct_layouts_match_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "is3d_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu\\n", sizeof(is3d_thermal_shear), offsetof(is3d_thermal_shear, xtn),'
                   ' offsetof(is3d_thermal_shear, xnn)); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got == [C.sizeof(api.ThermalShear), api.ThermalShear.xtn.offset, api.ThermalShear.xnn.offset]
    assert [f for f, _ in api.ThermalShear._fields_] == list(XI) == list(cf_polzn_xi.THERMAL_SHEAR_FIELDS)


# ------------------------------------------------------------------------------------------------ GPU
def _gpu():
    import torch
    torch.cuda.set_device(0)
    api.init()
    return torch


@pytest.mark.gpu
@pytest.mark.parametrize("dimension,outflow,chosen,memory", [
    (3, 1, "chosen_pikp", "host"), (3, 0, "chosen_pikp", "device"), (2, 1, "chosen_pikp", "host"), (2, 0, "chosen_pikp", "device"),
    (3, 1, "chosen_urqmd", "host")])
def test_gpu_parity(fx, dimension, outflow, chosen, memory):
    """Fermions and bosons (pi/K/p; the 305-species list), 3+1D and 2+1D, outflow on and off, cells with u.dsigma <= 0, host and
    device memory: all four arrays against the oracle at 1e-10 per bin, St exactly 0."""
    torch = _gpu()
    n = 40 if chosen == "chosen_urqmd" else 150
    cells, xi = _problem(n, 700 + dimension + 10 * outflow, dimension, flip=5)
    sp = tables.species(fx, 1, chosen); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=dimension, outflow=outflow)
    ref, skipped, cond = cf_polzn_xi.spin_polarization_shear(fl, cells, xi, sp, g, conditioning=True)
    if memory == "device":
        dc = {k: torch.tensor(v, device="cuda") for k, v in cells.items()}
        dx = {k: torch.tensor(v, device="cuda") for k, v in xi.items()}
        out, st = api.spin_polarization_shear(fl, dc, dx, sp, g, memory="device")
        torch.cuda.synchronize()
        got = {k: v.cpu().numpy() for k, v in out.items()}
    else:
        got, st = api.spin_polarization_shear(fl, cells, xi, sp, g)
    assert skipped == 5 and st["cells_skipped_udsigma"] == 5
    assert np.all(got["St"] == 0)
    assert compare(got["Snorm"], ref["Snorm"])["ok"], compare(got["Snorm"], ref["Snorm"])
    for k in ("Sx", "Sy", "Sz"):
        rep = compare(got[k], ref[k], conditioning=cond[k])
        assert rep["ok"], (k, rep)


@pytest.mark.gpu
def test_gpu_empty_surface_and_errors(fx):
    _gpu()
    sp = tables.species(fx, 1, "chosen_pikp"); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=3)
    cells, xi = _problem(0, 1, 3)
    out, st = api.spin_polarization_shear(fl, cells, xi, sp, g)
    assert all(np.all(v == 0) for v in out.values()) and st["cells_skipped_udsigma"] == 0
    cells, xi = _problem(10, 2, 3)
    for bad, code in [(dict(fl, mode=2), 2), (dict(fl, include_baryon=1), 2)]:
        with pytest.raises(api.Is3dError) as e:
            api.spin_polarization_shear(bad, cells, xi, sp, g)
        assert e.value.code == code
    for shear in (None, dict(xi, xnn=None)):
        with pytest.raises(api.Is3dError) as e:
            api.spin_polarization_shear(fl, cells, shear, sp, g)
        assert e.value.code == 1
    massless = dict(sp, mass=np.where(np.arange(len(sp["mass"])) == 0, 0.0, sp["mass"]))
    with pytest.raises(api.Is3dError) as e:
        api.spin_polarization_shear(fl, cells, xi, massless, g)
    assert e.value.code == 1


@pytest.mark.gpu
@pytest.mark.parametrize("dimension", [3, 2])
def test_gpu_snorm_bitwise_reproducible_and_multi(fx, dimension):
    _gpu()
    cells, xi = _problem(300, 655 + dimension, dimension, flip=2)
    vort = synthetic.vorticity(300, 9)
    sp = tables.species(fx, 1, "chosen_pikp"); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=dimension)
    a, _ = api.spin_polarization_shear(fl, cells, xi, sp, g)
    b, _ = api.spin_polarization_shear(fl, cells, xi, sp, g)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    v, _ = api.spin_polarization(fl, cells, vort, sp, g)
    assert np.array_equal(a["Snorm"], v["Snorm"])
    api.init_devices(0)
    m, st = api.spin_polarization_shear(fl, cells, xi, sp, g, multi=True)
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
@pytest.mark.parametrize("dimension", [3, 2])
def test_gpu_workdir_shear_files(fx, dimension):
    """With the key: S_xi_<mcid>.dat holds the API's shear part and totals, S_<mcid>.dat is byte-identical; without it (absent or 0) the
    run writes the files it wrote before."""
    _gpu()
    cols, base, vort, xi = _mode5_columns(60, 5321 + dimension, dimension)
    chosen = [3122, -3122, 211]
    runs = {}
    for label, extra in (("absent", {}), ("zero", dict(thermal_shear_polarization=0)), ("on", dict(thermal_shear_polarization=1))):
        with tempfile.TemporaryDirectory() as wd:
            workdir.materialize(wd, surface_columns=cols, chosen=chosen, fixture=fx, operation=1, mode=5, dimension=dimension, df_mode=1,
                                spin_polarization=1, thermal_shear=xi, **extra)
            open(os.path.join(wd, "average_thermodynamic_quantities.dat"), "w").write("0.15\n0.3\n0.05\n0\n0")
            runs[label] = _run(wd)
    assert runs["absent"][0] == runs["zero"][0]
    assert not any("S_xi_" in f for f in runs["absent"][0])
    xi_files = ["polarization" + os.sep + "S_xi_%d.dat" % c for c in chosen]
    assert runs["on"][0] == sorted(runs["absent"][0] + xi_files)
    for f, text in runs["absent"][1].items():
        assert runs["on"][1][f] == text == runs["zero"][1][f], f
    header = runs["on"][1][xi_files[0]].decode().split("\n", 1)[0].split()
    assert header == ["y", "phip", "pT", "Snorm", "Sx_xi", "Sy_xi", "Sz_xi", "Sx", "Sy", "Sz", "Sx_rest", "Sy_rest", "Sz_rest"]

    cells = synthetic.columns_to_cells(base, 1)
    sp = tables.species(fx, 1, chosen); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=dimension)
    rv, _ = api.spin_polarization(fl, cells, vort, sp, g)
    rx, _ = api.spin_polarization_shear(fl, cells, xi, sp, g)
    S, rest = api.mean_spin(rv, sp, g, dimension, shear=rx)
    Sxi, _ = api.mean_spin(rx, sp, g, dimension)
    ny = 1 if dimension == 2 else len(g["y"])
    shape = (len(g["y"]), len(g["phi"]), len(g["pT"]), -1)
    for s, c, f in zip(range(len(chosen)), chosen, xi_files):
        got = np.loadtxt(runs["on"][1][f].decode().splitlines(), skiprows=1, ndmin=2)[:, 3:]
        cols_want = [rx["Snorm"]] + list(Sxi[1:]) + list(S[1:]) + list(rest)
        want = np.column_stack([v.reshape(shape)[:ny, :, :, s].ravel() for v in cols_want])
        assert got.shape == want.shape
        scale = np.abs(want).max(axis=0)
        assert np.all(np.abs(got - want) <= 2e-8 * np.abs(want) + 1e-12 * scale), c
