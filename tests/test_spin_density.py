"""Spin density matrix from thermal vorticity: the oracle against an independent matrix-function restatement, the analytic anchor of a
cell at rest, the theta -> 0 limits, the parameter key and struct layout, and (on the GPU) the CUDA path against the oracle, its error
rules and the files of the host layer."""
import ctypes as C
import itertools
import os
import subprocess
import tempfile

import numpy as np
import pytest

from common import compare
from is3d_b200 import api, synthetic, tables, workdir
from oracle import cf_polzn, cf_spin_density

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HBARC = synthetic.HBARC
FIELDS = cf_spin_density.SPIN_DENSITY_FIELDS
VORT = synthetic.VORTICITY_COLUMNS
T_REST = 0.15


def _small_grid(fx, dimension):
    g = tables.grid(fx)
    g = dict(g, pT=g["pT"][::11].copy(), pT_weight=g["pT_weight"][::11].copy(), phi=g["phi"][::8].copy(),
             phi_weight=g["phi_weight"][::8].copy(), y=g["y"][::7].copy(), y_weight=g["y_weight"][::7].copy())
    if dimension == 2:
        g = dict(g, eta=g["eta"][::16].copy(), eta_weight=g["eta_weight"][::16].copy())
    return g


def _problem(n_cells, seed, dimension, scale=1.0, flip=0):
    cells = synthetic.columns_to_cells(synthetic.surface_vh(n_cells, seed, three_d=(dimension == 3)), 1)
    if flip:                                     # cells with u.dsigma <= 0
        for k in ("dat", "dax", "day"):
            cells[k] = cells[k].copy()
        cells["dat"][:flip] = -cells["dat"][:flip]
    vort = {k: scale * v for k, v in synthetic.vorticity(n_cells, seed + 7).items()}
    return cells, vort


def _species(spins, signs, mass=1.0):
    """J = 0, 1/2, ... with the given signs, masses spread around `mass`"""
    sp = [(mass * (1 + 0.1 * i), s, 2 * J + 1) for i, (J, s) in enumerate(itertools.product(spins, signs))]
    return dict(mass=np.array([v[0] for v in sp]), sign=np.array([float(v[1]) for v in sp]), degeneracy=np.array([float(v[2]) for v in sp]),
                baryon=np.zeros(len(sp)))


def spin_matrices(J):
    ms = np.arange(J, -J - 1, -1)
    n = len(ms)
    Sp = np.zeros((n, n), complex)
    for k in range(1, n):
        Sp[k - 1, k] = np.sqrt(J * (J + 1) - ms[k] * (ms[k] + 1))
    return [(Sp + Sp.conj().T) / 2, (Sp - Sp.conj().T) / 2j, np.diag(ms).astype(complex)]


def numpy_matrix(flags, cells, vort, sp, g):
    """The nine sums restated without levels or that: varpi_{mu nu} in Cartesian components as J^T varpi' J with the Jacobian of
    (tau, eta) -> (t, z), theta^mu = -(1/(2m)) eps^{mu rho sigma tau} varpi_{rho sigma} p_tau, theta* by the full boost to the rest frame,
    rho = F(x 1 - theta*.S) with F(z) = 1/(e^z + Theta) as a matrix function (eigendecomposition of the Hermitian argument), and
    <S_i>, <S_i S_j> read off traces."""
    eps = np.zeros((4, 4, 4, 4))
    for perm in itertools.permutations(range(4)):
        eps[perm] = np.linalg.det(np.eye(4)[list(perm)])
    gmet = np.diag([1.0, -1.0, -1.0, -1.0])
    pref = (2 * np.pi * HBARC) ** -3
    d2 = flags["dimension"] == 2
    ns, npT, nphi, ny = len(sp["mass"]), len(g["pT"]), len(g["phi"]), len(g["y"])
    out = np.zeros((9, ny, nphi, npT, ns))
    mats = {J: spin_matrices(J) for J in set(0.5 * (sp["degeneracy"] - 1))}
    pairs = [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2)]
    for i in range(len(cells["tau"])):
        tau = cells["tau"][i]; ux, uy, un = cells["ux"][i], cells["uy"][i], cells["un"][i]
        ut = np.sqrt(1 + ux * ux + uy * uy + tau * tau * un * un)
        dat, dax, day, dan = (cells[k][i] for k in ("dat", "dax", "day", "dan"))
        if ut * dat + ux * dax + uy * day + un * dan <= 0:
            continue
        v = [vort[k][i] for k in VORT]                         # tau x, tau y, tau eta, xy, x eta, y eta
        Wm = np.zeros((4, 4))
        for val, (a, b) in zip(v, [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]):
            Wm[a, b], Wm[b, a] = val, -val
        for iy in range(1 if d2 else ny):
            y = 0.0 if d2 else g["y"][iy]
            for eta, wt in (zip(g["eta"], g["eta_weight"]) if d2 else [(cells["eta"][i], 1.0)]):
                Jac = np.eye(4)                                # Jac[mu'][a] = d(tau, x, y, eta)^mu' / d(t, x, y, z)^a
                Jac[0, 0], Jac[0, 3] = np.cosh(eta), -np.sinh(eta)
                Jac[3, 0], Jac[3, 3] = -np.sinh(eta) / tau, np.cosh(eta) / tau
                Wc = Jac.T @ Wm @ Jac
                for s in range(ns):
                    m, sign, J = sp["mass"][s], sp["sign"][s], 0.5 * (sp["degeneracy"][s] - 1)
                    S = mats[J]
                    for ipT, pT in enumerate(g["pT"]):
                        mT = np.sqrt(m * m + pT * pT)
                        for iphi, phi in enumerate(g["phi"]):
                            pup = np.array([mT * np.cosh(y), pT * np.cos(phi), pT * np.sin(phi), mT * np.sinh(y)])
                            pt, pn = mT * np.cosh(y - eta), mT / tau * np.sinh(y - eta)
                            pds = wt * (pt * dat + pup[1] * dax + pup[2] * day + pn * dan)
                            if flags["outflow"] and pds <= 0:
                                continue
                            x = (pt * ut - pup[1] * ux - pup[2] * uy - tau * tau * pn * un) / cells["T"][i]
                            if x > 709.782712893384:
                                continue
                            theta = -np.einsum("abcd,bc,d->a", eps, Wc, gmet @ pup) / (2 * m)
                            E, p = pup[0], pup[1:]
                            ts = theta[1:] + p / m * (p @ theta[1:] / (E + m) - theta[0])
                            M = x * np.eye(len(S[2])) - sum(ts[k] * S[k] for k in range(3))
                            lam, V = np.linalg.eigh(M)
                            rho = V @ np.diag(1.0 / (np.exp(lam) + sign)) @ V.conj().T
                            Z = np.trace(rho).real
                            row = [Z] + [np.trace(rho @ S[k]).real for k in range(3)]
                            for a, b in pairs:
                                sym = np.trace(rho @ (S[a] @ S[b] + S[b] @ S[a]) / 2).real
                                row.append(sym - (J * (J + 1) / 3 * Z if a == b else 0.0))
                            out[:, iy, iphi, ipT, s] += pref * pds * np.array(row)
    return {k: out[j].ravel() for j, k in enumerate(FIELDS)}


@pytest.mark.parametrize("dimension,scale", [(3, 4.0), (2, 4.0), (3, 40.0)])
def test_oracle_matches_matrix_function_restatement(fx, dimension, scale):
    """J = 0, 1/2, 1, 3/2, 2, 9/2, bosons and fermions, theta up to ~3 (bosons above J theta)."""
    cells, vort = _problem(4, 610 + dimension, dimension, scale=scale)
    sp = _species([0, 0.5, 1, 1.5, 2, 4.5], [-1, 1], mass=1.2)
    g = _small_grid(fx, dimension)
    fl = tables.flags(df_mode=1, dimension=dimension)
    got, skipped, cond = cf_spin_density.spin_density(fl, cells, vort, sp, g, conditioning=True)
    want = numpy_matrix(fl, cells, vort, sp, g)
    assert skipped == 0
    # theta reached: |P| / (J Snorm) is tanh-like in theta, so a large ratio means large theta
    J = np.tile(0.5 * (sp["degeneracy"] - 1), got["Snorm"].size // len(sp["mass"]))
    live = (J > 0) & (got["Snorm"] > 0)
    ratio = np.sqrt(got["Px"] ** 2 + got["Py"] ** 2 + got["Pz"] ** 2)[live] / (J[live] * got["Snorm"][live])
    assert ratio.max() > (0.5 if scale > 10 else 0.01)
    for k in FIELDS:
        assert np.all(np.abs(got[k] - want[k]) <= 1e-12 * cond[k]), (k, np.abs(got[k] - want[k]).max())
        if k != "Snorm":
            assert np.any(got[k] != 0), k


def _rest_cell(w, scale=1.0):
    cells = {k: np.zeros(1) for k in ("eta", "dax", "day", "dan", "ux", "uy", "un")}
    cells.update(tau=np.ones(1), dat=np.ones(1), T=np.full(1, T_REST), P=np.full(1, 0.05), E=np.full(1, 0.3))
    vort = {k: np.zeros(1) for k in VORT}
    vort["wxy"] = np.full(1, w * scale)
    return cells, vort


def _y0_bins(fx, sp):
    g = tables.grid(fx)
    iy = int(np.argmin(np.abs(g["y"])))
    assert g["y"][iy] == 0.0
    ns, npT, nphi = len(sp["mass"]), len(g["pT"]), len(g["phi"])
    idx = np.arange(ns * npT * nphi).reshape(nphi, npT, ns) + iy * ns * npT * nphi
    return g, idx


def test_analytic_anchor_cell_at_rest(fx):
    """Only varpi_xy = w, at rest, y = 0: theta* = (0, 0, w mT/m) and the levels along z are the f_m themselves."""
    w = 0.02
    cells, vort = _rest_cell(w)
    sp = dict(mass=np.array([0.89166, 1.115683, 0.493677]), sign=np.array([-1.0, 1.0, -1.0]), degeneracy=np.array([3.0, 2.0, 1.0]),
              baryon=np.zeros(3))
    g, idx = _y0_bins(fx, sp)
    fl = tables.flags(df_mode=1, dimension=3)
    r, _ = cf_spin_density.spin_density(fl, cells, vort, sp, g)
    S, T = api.spin_moments(r, sp)
    pT = g["pT"][None, :]
    for s in range(3):
        b = idx[:, :, s]
        m, sign, J = sp["mass"][s], sp["sign"][s], 0.5 * (sp["degeneracy"][s] - 1)
        mT = np.sqrt(m * m + pT * pT) + 0 * b
        th = w * mT / m
        f = {mm: 1.0 / (np.exp(mT / T_REST - mm * th) + sign) for mm in np.arange(-J, J + 1)}
        Z = sum(f.values())
        assert np.allclose(r["Snorm"][b], (2 * np.pi * HBARC) ** -3 * mT * Z, rtol=1e-13, atol=0)
        if J == 0:
            assert all(np.all(r[k][b] == 0) for k in FIELDS[1:])
            continue
        assert np.all(S[0][b] == 0) and np.all(S[1][b] == 0)
        assert np.allclose(S[2][b], sum(mm * fm for mm, fm in f.items()) / Z, rtol=1e-13, atol=0)
        if J == 0.5:
            assert np.all(np.abs(T[:, b]) <= 1e-16)
            continue
        rz = api.spin_alignment(r, sp, g, 3, "z")[b]
        rx = api.spin_alignment(r, sp, g, 3, "x")[b]
        ry = api.spin_alignment(r, sp, g, 3, "y")[b]
        rh = api.spin_alignment(r, sp, g, 3, "helicity")[b]
        assert np.allclose(rz, f[0] / Z, rtol=1e-13, atol=0)
        for v in (rx, ry, rh):                                # every axis in the transverse plane sees the same rho00
            assert np.allclose(v, 0.5 * (f[1] + f[-1]) / Z, rtol=1e-13, atol=0)
    assert np.all(np.isnan(api.spin_alignment(r, sp, g, 3, "z")[idx[:, :, 1:]]))      # J != 1


def test_limits_zero_linear_and_second_order(fx):
    cells, vort = _problem(12, 77, 3)
    sp = tables.species(fx, 1, [211, 3122, 313, 3334, -3334])
    g = _small_grid(fx, 3)
    fl = tables.flags(df_mode=1, dimension=3)
    # varpi = 0: P = Q = 0 exactly, Snorm = the vorticity oracle's
    zero = {k: np.zeros_like(v) for k, v in vort.items()}
    r0, _ = cf_spin_density.spin_density(fl, cells, zero, sp, g)
    assert all(np.all(r0[k] == 0) for k in FIELDS[1:])
    rv, _ = cf_polzn.spin_polarization(fl, cells, zero, sp, g)
    assert np.all(np.abs(r0["Snorm"] - rv["Snorm"]) <= 1e-15 * np.abs(rv["Snorm"]))
    # linear order: P / Snorm -> 4J(J+1)/3 S* of the vorticity path, the deviation O(varpi^2)
    J = np.tile(0.5 * (sp["degeneracy"] - 1), r0["Snorm"].size // len(sp["mass"]))
    devs = []
    for lam in (0.5, 0.25):
        v = {k: lam * a for k, a in vort.items()}
        r, _ = cf_spin_density.spin_density(fl, cells, v, sp, g)
        rp, _ = cf_polzn.spin_polarization(fl, cells, v, sp, g)
        _, rest = api.mean_spin(rp, sp, g, 3)
        S, _ = api.spin_moments(r, sp)
        want = 4 * J * (J + 1) / 3 * rest
        devs.append(np.abs(S - want).max() / np.abs(want).max())
    assert 3.5 < devs[0] / devs[1] < 4.5, devs


def test_second_order_at_tiny_theta(fx):
    """lambda = 1e-6: Q / lambda^2 against (theta^2/4)(3 sum m^4 - J(J+1) sum m^2) F''(x) at 1e-8; a naive level sum misses this."""
    w, lam = 0.05, 1e-6
    cells, vort = _rest_cell(w, lam)
    sp = dict(mass=np.array([0.89166, 1.67245, 1.2]), sign=np.array([-1.0, 1.0, -1.0]), degeneracy=np.array([3.0, 4.0, 5.0]),
              baryon=np.zeros(3))
    g, idx = _y0_bins(fx, sp)
    fl = tables.flags(df_mode=1, dimension=3)
    r, _ = cf_spin_density.spin_density(fl, cells, vort, sp, g)
    for s in range(3):
        b = idx[:, :, s].ravel()
        m, sign, J = sp["mass"][s], sp["sign"][s], 0.5 * (sp["degeneracy"][s] - 1)
        ms = np.arange(-J, J + 1)
        mT = np.sqrt(m * m + g["pT"] ** 2)[None, :].repeat(len(g["phi"]), 0).ravel()
        x, th = mT / T_REST, w * mT / m                       # theta / lambda
        e = np.exp(-x)
        F2 = e * (1 - sign * e) / (1 + sign * e) ** 3             # F''(x) of F(z) = 1/(e^z + Theta)
        pref = (2 * np.pi * HBARC) ** -3 * mT
        c2 = th * th / 4 * (3 * np.sum(ms ** 4) - J * (J + 1) * np.sum(ms ** 2)) * F2
        want_zz = pref * c2 * (2.0 / 3.0)                     # Q_zz = K W c2 lam^2 (1 - 1/3), Q_xx = Q_yy = -Q_zz / 2
        got_zz = -(r["Qxx"][b] + r["Qyy"][b]) / lam ** 2
        assert np.all(np.abs(got_zz - want_zz) <= 1e-8 * np.abs(want_zz)), s
        assert np.all(np.abs(r["Qxx"][b] / lam ** 2 + want_zz / 2) <= 1e-8 * np.abs(want_zz))
        naive = sum((3 * mm * mm - J * (J + 1)) / 2 / (np.exp(x - mm * th * lam) + sign) for mm in ms) / lam ** 2
        assert np.abs(naive - c2).max() > 1e-4 * np.abs(c2).max()


# ------------------------------------------------------------------------------------------------ host layer, ABI
def _host_dump(wd):
    lib = api.lib()
    lib.is3d_b200_host_error.restype = C.c_char_p
    rc = lib.is3d_b200_host_dump(wd.encode(), os.path.join(wd, "host_dump.bin").encode())
    return rc, (lib.is3d_b200_host_error().decode() if rc else "")


def _mode5_columns(n, seed, dimension=3):
    base = synthetic.surface_vh(n, seed, three_d=(dimension == 3))
    vort = synthetic.vorticity(n, seed + 1)
    return np.column_stack([base] + [vort[k] for k in VORT]), base, vort


def _materialize(wd, fx, cols, **kw):
    workdir.materialize(wd, surface_columns=cols, fixture=fx, operation=kw.pop("operation", 1), mode=kw.pop("mode", 5),
                        dimension=kw.pop("dimension", 3), df_mode=1, **kw)
    open(os.path.join(wd, "average_thermodynamic_quantities.dat"), "w").write("0.15\n0.3\n0.05\n0\n0")


def test_spin_density_key_rules(fx):
    cols, _, _ = _mode5_columns(4, 25)
    with tempfile.TemporaryDirectory() as wd:
        for kw in (dict(mode=1), dict(mode=5, operation=0)):
            c = cols[:, :-6] if kw["mode"] == 1 else cols
            _materialize(wd, fx, c, spin_density=1, **kw)
            assert _host_dump(wd)[0] == 2, kw                                             # IS3D_ERR_UNSUPPORTED
        _materialize(wd, fx, cols, spin_density=1)                                        # independent of spin_polarization
        assert _host_dump(wd)[0] == 0
        _materialize(wd, fx, cols, spin_density=0)
        assert _host_dump(wd)[0] == 0


def test_struct_layout_matches_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "is3d_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu\\n", sizeof(is3d_spin_density_result), offsetof(is3d_spin_density_result, Px),'
                   ' offsetof(is3d_spin_density_result, Qxx), offsetof(is3d_spin_density_result, Qyz)); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    R = api.SpinDensityResult
    assert got == [C.sizeof(R), R.Px.offset, R.Qxx.offset, R.Qyz.offset]
    assert [f for f, _ in R._fields_] == list(FIELDS)


# ------------------------------------------------------------------------------------------------ GPU
def _gpu():
    import torch
    torch.cuda.set_device(0)
    api.init()
    return torch


CHOSEN = [211, 3122, 313, 333, 3334, -3122]          # pi (J = 0), Lambda, K*0, phi(1020), Omega- (J = 3/2), an antiparticle


@pytest.mark.gpu
@pytest.mark.parametrize("dimension,outflow,memory,cold", [
    (3, 1, "host", False), (3, 0, "device", False), (2, 1, "host", False), (2, 0, "device", False), (3, 1, "host", True)])
def test_gpu_parity(fx, dimension, outflow, memory, cold):
    """All nine arrays against the oracle at 1e-10 per bin (|terms| conditioning), cells with u.dsigma <= 0; cold: T = 2 MeV, where the
    exponential overflows in many bins, which must hold exact zeros."""
    torch = _gpu()
    cells, vort = _problem(150, 900 + dimension + 10 * outflow, dimension, scale=3.0, flip=5)
    if cold:
        cells["T"] = np.full_like(cells["T"], 0.002)
    sp = tables.species(fx, 1, CHOSEN); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=dimension, outflow=outflow)
    ref, skipped, cond = cf_spin_density.spin_density(fl, cells, vort, sp, g, conditioning=True)
    if memory == "device":
        dc = {k: torch.tensor(v, device="cuda") for k, v in cells.items()}
        dv = {k: torch.tensor(v, device="cuda") for k, v in vort.items()}
        out, st = api.spin_density(fl, dc, dv, sp, g, memory="device")
        torch.cuda.synchronize()
        got = {k: v.cpu().numpy() for k, v in out.items()}
    else:
        got, st = api.spin_density(fl, cells, vort, sp, g)
    assert skipped == 5 and st["cells_skipped_udsigma"] == 5
    if cold:
        assert np.mean(ref["Snorm"] == 0) > 0.2 and np.any(ref["Snorm"] != 0)
    for k in FIELDS:
        rep = compare(got[k], ref[k], conditioning=None if k == "Snorm" else cond[k])
        assert rep["ok"], (k, rep)
    n_pi = slice(0, None, len(CHOSEN))                   # pi: J = 0, P = Q = 0 exactly
    assert all(np.all(got[k][n_pi] == 0) for k in FIELDS[1:])


@pytest.mark.gpu
@pytest.mark.parametrize("dimension", [3, 2])
def test_gpu_exact_zero_tiny_theta_and_snorm(fx, dimension):
    _gpu()
    cells, vort = _problem(200, 71 + dimension, dimension)
    sp = tables.species(fx, 1, CHOSEN); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=dimension)
    zero = {k: np.zeros_like(v) for k, v in vort.items()}
    r0, _ = api.spin_density(fl, cells, zero, sp, g)
    assert all(np.all(r0[k] == 0) for k in FIELDS[1:])
    rv, _ = api.spin_polarization(fl, cells, zero, sp, g)
    assert np.all(np.abs(r0["Snorm"] - rv["Snorm"]) <= 1e-15 * np.abs(rv["Snorm"]))
    lam = 1e-6                                           # theta ~ 1e-7: the paired level sums keep Q at its relative accuracy
    tiny = {k: lam * v for k, v in vort.items()}
    got, _ = api.spin_density(fl, cells, tiny, sp, g)
    ref, _ = cf_spin_density.spin_density(fl, cells, tiny, sp, g)
    for k in FIELDS[1:]:
        scale = np.abs(ref[k]).max()
        assert scale > 0, k
        assert np.all(np.abs(got[k] - ref[k]) <= 1e-8 * np.abs(ref[k]) + 1e-12 * scale), k


@pytest.mark.gpu
@pytest.mark.parametrize("dimension", [3, 2])
def test_gpu_bitwise_reproducible(fx, dimension):
    _gpu()
    cells, vort = _problem(300, 655 + dimension, dimension, flip=2)
    sp = tables.species(fx, 1, CHOSEN); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=dimension)
    a, _ = api.spin_density(fl, cells, vort, sp, g)
    b, _ = api.spin_density(fl, cells, vort, sp, g)
    for k in FIELDS:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.gpu
@pytest.mark.skipif("__import__('torch').cuda.device_count() < 2")
def test_gpu_multi_matches_one_device(fx):
    _gpu()
    cells, vort = _problem(400, 8, 3, flip=3)
    sp = tables.species(fx, 1, CHOSEN); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=3)
    a, _ = api.spin_density(fl, cells, vort, sp, g)
    api.init_devices(0)
    m, st = api.spin_density(fl, cells, vort, sp, g, multi=True)
    assert st["n_gpus"] >= 2
    for k in FIELDS:
        assert np.abs(m[k] - a[k]).max() <= 1e-13 * np.abs(a[k]).max(), k


def _call_raw(fl, cells, vort, sp, g, arrays, null=None):
    """is3d_b200_spin_density on caller-owned host arrays (so that an error can be seen to leave them alone); null: a field left NULL"""
    m = api._Marshal(False)
    sf, spc, gr, _, _ = api._marshal_problem(m, cells, sp, g, None, None)
    vo = None
    if vort is not None:
        vo = api.Vorticity()
        for k in api.VORTICITY_FIELDS:
            setattr(vo, k, m.cells(vort[k]))
    res = api.SpinDensityResult()
    for k in FIELDS:
        if k != null:
            setattr(res, k, arrays[k].ctypes.data_as(C.POINTER(C.c_double)))
    opt = api.Options(); opt.memory = 0
    st = api.Stats()
    f = api.lib().is3d_b200_spin_density
    f.restype = C.c_int
    f.argtypes = [C.POINTER(api.Flags), C.POINTER(api.Surface), C.POINTER(api.Vorticity), C.POINTER(api.Species), C.POINTER(api.Grid),
                  C.POINTER(api.Options), C.POINTER(api.SpinDensityResult), C.POINTER(api.Stats)]
    flg = api.make_flags(fl)
    api.lib().is3d_b200_last_error.restype = C.c_char_p
    rc = f(C.byref(flg), C.byref(sf), C.byref(vo) if vo is not None else None, C.byref(spc), C.byref(gr), C.byref(opt), C.byref(res),
           C.byref(st))
    return rc, api.lib().is3d_b200_last_error().decode()


@pytest.mark.gpu
def test_gpu_empty_surface_and_errors(fx):
    _gpu()
    sp = tables.species(fx, 1, CHOSEN); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=3)
    cells, vort = _problem(0, 1, 3)
    out, st = api.spin_density(fl, cells, vort, sp, g)
    assert all(np.all(v == 0) for v in out.values()) and st["cells_skipped_udsigma"] == 0
    cells, vort = _problem(40, 2, 3)
    n = len(sp["mass"]) * len(g["pT"]) * len(g["phi"]) * len(g["y"])
    big = {k: 200.0 * v for k, v in vort.items()}        # K*, phi: u.p/T - theta <= 0 somewhere
    cases = [(dict(fl, mode=2), vort, sp, None, 2), (dict(fl, include_baryon=1), vort, sp, None, 2), (fl, None, sp, None, 1),
             (fl, vort, sp, "Qyz", 1), (fl, vort, sp, "Snorm", 1), (fl, vort, dict(sp, mass=np.where(np.arange(6) == 0, 0.0, sp["mass"])), None, 1),
             (fl, vort, dict(sp, degeneracy=np.where(np.arange(6) == 2, 2.5, sp["degeneracy"])), None, 1),
             (fl, vort, dict(sp, degeneracy=np.where(np.arange(6) == 2, 17.0, sp["degeneracy"])), None, 1),
             (fl, vort, dict(sp, degeneracy=np.where(np.arange(6) == 2, 0.0, sp["degeneracy"])), None, 1),
             (fl, big, sp, None, 1)]
    for fli, v, spi, null, code in cases:
        arrays = {k: np.full(n, 7.0) for k in FIELDS}
        rc, msg = _call_raw(fli, cells, v, spi, g, arrays, null)
        assert rc == code, (rc, msg)
        assert all(np.all(a == 7.0) for a in arrays.values()), msg
    assert "boson evaluations" in msg and int(msg.split()[0]) > 0
    with pytest.raises(RuntimeError, match="-5"):
        cf_spin_density.spin_density(fl, cells, big, sp, g)
    # and a valid call adds into the arrays: the sums are bit-reproducible, so the host add 7 + s is exactly 7 + (the sums of a call
    # into zeros); subtracting 7 again would round away everything below 7 eps
    arrays = {k: np.full(n, 7.0) for k in FIELDS}
    assert _call_raw(fl, cells, vort, sp, g, arrays)[0] == 0
    want, _ = api.spin_density(fl, cells, vort, sp, g)
    for k in FIELDS:
        assert np.array_equal(arrays[k], 7.0 + want[k]), k


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
def test_gpu_workdir_spin_files(fx, dimension):
    """With the key: spin_<mcid>.dat (species with g >= 2) holds spin_moments() of a direct call and S_<mcid>.dat is byte-identical;
    without it (absent or 0) the run writes the files it wrote before."""
    _gpu()
    cols, base, vort = _mode5_columns(60, 4321 + dimension, dimension)
    chosen = [211, 3122, 313, 3334]
    runs = {}
    for label, extra in (("absent", {}), ("zero", dict(spin_density=0)), ("on", dict(spin_density=1))):
        with tempfile.TemporaryDirectory() as wd:
            workdir.materialize(wd, surface_columns=cols, chosen=chosen, fixture=fx, operation=1, mode=5, dimension=dimension, df_mode=1,
                                spin_polarization=1, **extra)
            open(os.path.join(wd, "average_thermodynamic_quantities.dat"), "w").write("0.15\n0.3\n0.05\n0\n0")
            runs[label] = _run(wd)
    assert runs["absent"][0] == runs["zero"][0]
    assert not any("spin_" in f for f in runs["absent"][0])
    spin_files = ["polarization" + os.sep + "spin_%d.dat" % c for c in chosen[1:]]      # the pion (g = 1) gets none
    assert runs["on"][0] == sorted(runs["absent"][0] + spin_files)
    for f, text in runs["absent"][1].items():
        assert runs["on"][1][f] == text == runs["zero"][1][f], f
    header = runs["on"][1][spin_files[0]].decode().split("\n", 1)[0].split()
    assert header == ["y", "phip", "pT", "Snorm", "Sx", "Sy", "Sz", "Txx", "Txy", "Txz", "Tyy", "Tyz", "Tzz"]

    cells = synthetic.columns_to_cells(base, 1)
    sp = tables.species(fx, 1, chosen); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=dimension)
    r, _ = api.spin_density(fl, cells, vort, sp, g)
    S, T = api.spin_moments(r, sp)
    ny = 1 if dimension == 2 else len(g["y"])
    shape = (len(g["y"]), len(g["phi"]), len(g["pT"]), -1)
    for s, f in zip(range(1, len(chosen)), spin_files):
        got = np.loadtxt(runs["on"][1][f].decode().splitlines(), skiprows=1, ndmin=2)[:, 3:]
        want = np.column_stack([v.reshape(shape)[:ny, :, :, s].ravel() for v in [r["Snorm"]] + list(S) + list(T)])
        assert got.shape == want.shape
        scale = np.abs(want).max(axis=0)
        assert np.all(np.abs(got - want) <= 2e-8 * np.abs(want) + 1e-12 * scale), f
