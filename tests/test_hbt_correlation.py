"""HBT correlation functions from the Fourier transform of the emission function: the oracle against an independent restatement with an
explicit lab-frame boost of q and x, its q = 0 sums against the moments and the spectra, analytic anchors, the small-q curvature
against the radii, the host layer and the ABI, and (on the GPU) the CUDA path."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from common import compare
from is3d_b200 import api, synthetic, tables, workdir
from oracle import cf_hbtq
from oracle import cf_oracle as cfo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HBARC = synthetic.HBARC
NORMAL = 1e-140                                  # weights whose squares stay well above the sub-normal range
AXES = np.eye(3)                                 # out, side, long
RAYS = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.0, 0.0, 1.0], [1.0, -1.0, 0.5]])     # the three axes and a diagonal


def _small_grid(fx, dimension):
    """A few points of every table (the eta table thinned in 2+1D, symmetric about 0) to keep the restatements quick."""
    g = tables.grid(fx)
    g = dict(g, pT=g["pT"][::8].copy(), pT_weight=g["pT_weight"][::8].copy(), phi=g["phi"][::5].copy(), phi_weight=g["phi_weight"][::5].copy(),
             y=g["y"][::4].copy(), y_weight=g["y_weight"][::4].copy())
    if dimension == 2:
        g = dict(g, eta=g["eta"][::12].copy(), eta_weight=g["eta_weight"][::12].copy())
    return g


def _cells(n_cells, seed, dimension, flip=0):
    cells = synthetic.columns_to_cells(synthetic.surface_vh(n_cells, seed, three_d=(dimension == 3)), 1)
    if flip:                                     # cells with u.dsigma <= 0
        cells["dat"] = cells["dat"].copy()
        cells["dat"][:flip] = -cells["dat"][:flip]
    return cells


def _one_cell(x=0.0, y=0.0):
    c = synthetic.columns_to_cells(synthetic.surface_vh(1, 8, three_d=True), 1)
    c["x"] = np.full(1, x); c["y"] = np.full(1, y)
    return c


def numpy_lab_boost(flags, cells, sp, g, qrays):
    """Ideal-f weights (the flags must switch delta-f off) at the lab-frame point x = (tau cosh eta, x, y, tau sinh eta); q from the LCMS
    of the bin to the lab with q^0 = beta_perp q_o: a rotation by phi and a longitudinal boost by y; F = sum w exp(-i q.x / hbar c)
    with the Minkowski product q.x = q^0 t - q_x x - q_y y - q_z z.  Returns (Re, Im) shaped (n_dir, n_q, n_bins), sum |w| per bin, and
    sum |w| (1 + |q.x terms| / hbar c) per q point and bin: the lab-frame product cancels where eta ~ y, its rounding is this
    restatement's own floor."""
    assert not flags["include_shear"] and not flags["include_bulk"]
    pref = (2 * np.pi * HBARC) ** -3
    ns, npT, nphi, ny = len(sp["mass"]), len(g["pT"]), len(g["phi"]), len(g["y"])
    d2 = flags["dimension"] == 2
    dirs = np.asarray(qrays["dir"], dtype=float).reshape(-1, 3)
    nd, nq = len(dirs), qrays["n_q"]
    F = np.zeros((nd, nq, ny, nphi, npT, ns), dtype=complex); A = np.zeros((ny, nphi, npT, ns)); B = np.zeros(F.shape)
    m = np.asarray(sp["mass"])[None, None, :]; sign = np.asarray(sp["sign"])[None, None, :]
    pT = g["pT"][None, :, None]; phi = g["phi"][:, None, None]
    mT = np.sqrt(m * m + pT * pT)
    px = pT * np.cos(phi) + 0 * m; py = pT * np.sin(phi) + 0 * m
    beta = pT / mT
    k = np.arange(nq)
    for i in range(len(cells["tau"])):
        tau = cells["tau"][i]; ux, uy, un = cells["ux"][i], cells["uy"][i], cells["un"][i]
        ut = np.sqrt(1 + ux * ux + uy * uy + tau * tau * un * un)
        dat, dax, day, dan = (cells[c][i] for c in ("dat", "dax", "day", "dan"))
        if ut * dat + ux * dax + uy * day + un * dan <= 0:
            continue
        xc, yc = cells["x"][i], cells["y"][i]
        for iy in range(1 if d2 else ny):
            y = 0.0 if d2 else g["y"][iy]
            slots = zip(g["eta"], g["eta_weight"]) if d2 else [(cells["eta"][i], 1.0)]
            for eta, wt in slots:
                pt = mT * np.cosh(y - eta); pn = mT / tau * np.sinh(y - eta)
                pds = wt * (pt * dat + px * dax + py * day + pn * dan)
                pu = pt * ut - px * ux - py * uy - tau * tau * pn * un
                with np.errstate(over="ignore"):
                    f = 1.0 / (np.exp(pu / cells["T"][i]) + sign)
                keep = (pds > 0) if flags["outflow"] else np.ones_like(pds, dtype=bool)
                w = np.where(keep, pds * f, 0.0) * pref * sp["degeneracy"]
                t, z = tau * np.cosh(eta), tau * np.sinh(eta)
                A[iy] += np.abs(w)
                for a, (do, ds, dl) in enumerate(dirs):
                    qo, qs, ql = (k * qrays["dq"] * c for c in (do, ds, dl))
                    qo, qs, ql = (v[:, None, None, None] for v in (qo, qs, ql))
                    q0 = beta * qo                                   # q.K = 0 in the LCMS
                    qt_lab = q0 * np.cosh(y) + ql * np.sinh(y)
                    qz_lab = ql * np.cosh(y) + q0 * np.sinh(y)
                    qx_lab = qo * np.cos(phi) - qs * np.sin(phi)
                    qy_lab = qo * np.sin(phi) + qs * np.cos(phi)
                    qx = qt_lab * t - qx_lab * xc - qy_lab * yc - qz_lab * z
                    F[a, :, iy] += w * np.exp(-1j * qx / HBARC)
                    qxa = ((np.abs(q0) * np.cosh(y) + np.abs(ql * np.sinh(y))) * t + (np.abs(qo) + np.abs(qs)) * (abs(xc) + abs(yc))
                           + (np.abs(ql) * np.cosh(y) + np.abs(q0 * np.sinh(y))) * abs(z))
                    B[a, :, iy] += np.abs(w) * (1.0 + qxa / HBARC)
    F = F.reshape(nd, nq, -1)
    return F.real, F.imag, A.ravel(), B.reshape(nd, nq, -1)


@pytest.mark.parametrize("dimension,outflow", [(3, 1), (2, 1), (3, 0)])
def test_oracle_matches_numpy_lab_boost(fx, dimension, outflow):
    cells = _cells(10, 5050 + dimension, dimension)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, dimension); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=dimension, include_bulk=0, include_shear=0, outflow=outflow)
    qr = dict(dir=RAYS, dq=0.02, n_q=9)
    got, skipped, cond = cf_hbtq.hbt_fourier(fl, cells, sp, g, tab, qr)
    re, im, want_cond, phase_cond = numpy_lab_boost(fl, cells, sp, g, qr)
    assert skipped == 0
    assert np.allclose(cond, want_cond, rtol=1e-12, atol=0)        # ideal f: the |terms| magnitude is sum |w|
    assert np.any(np.abs(got["Im"][:, 1:]) > 1e-3 * cond)             # the phases are not trivial
    assert np.all(np.abs(got["Re"] - re) <= 1e-13 * phase_cond)
    assert np.all(np.abs(got["Im"] - im) <= 1e-13 * phase_cond)


@pytest.mark.parametrize("dimension", [3, 2])
@pytest.mark.parametrize("df_mode,deltaf", [(1, 1), (1, 0), (2, 1), (2, 0)])
def test_oracle_q0_is_the_moments_s0_and_the_spectrum(fx, dimension, df_mode, deltaf):
    cells = _cells(20, 71 + dimension, dimension, flip=3)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, dimension); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=df_mode, dimension=dimension, include_bulk=deltaf, include_shear=deltaf)
    r, skipped, _ = cf_hbtq.hbt_fourier(fl, cells, sp, g, tab, dict(dir=RAYS, dq=0.03, n_q=3))
    m = cf_hbtq.hbt_moments(fl, cells, sp, g, tab)
    dN, skipped_smooth, _ = cfo.smooth(fl, cells, sp, g, tab)
    assert skipped == skipped_smooth == 3
    for d in range(len(RAYS)):
        assert np.array_equal(r["Re"][d, 0], m["S0"])
        assert np.array_equal(r["Re"][d, 0], dN)
        assert np.all(r["Im"][d, 0] == 0)


def test_single_cell_is_fully_coherent(fx):
    """One cell in 3+1D has one space-time point per bin: |F|^2 = S0^2 for every q."""
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, 3); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=3)
    r, _, _ = cf_hbtq.hbt_fourier(fl, _one_cell(3.0, -2.0), sp, g, tab, dict(dir=RAYS, dq=0.05, n_q=11))
    s0 = r["Re"][0, 0]
    nz = s0 > NORMAL
    assert nz.sum() > 0.5 * nz.size
    f2 = r["Re"] ** 2 + r["Im"] ** 2
    assert np.all(np.abs(f2[:, :, nz] - s0[nz] ** 2) <= 1e-13 * s0[nz] ** 2)


def test_two_cells_at_plus_minus_a(fx):
    a = 2.5
    one = _one_cell()
    cells = {k: np.concatenate([v, v]) for k, v in one.items()}
    cells["x"] = np.array([a, -a]); cells["y"] = np.zeros(2)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, 3); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=3)
    dq, n_q = 0.02, 15
    r, _, _ = cf_hbtq.hbt_fourier(fl, cells, sp, g, tab, dict(dir=AXES, dq=dq, n_q=n_q))
    s0 = r["Re"][0, 0]
    nz = s0 > NORMAL
    assert nz.sum() > 0.5 * nz.size
    ratio = (r["Re"] ** 2 + r["Im"] ** 2)[:, :, nz] / s0[nz] ** 2
    phi = np.meshgrid(g["y"], g["phi"], g["pT"], sp["mass"], indexing="ij")[1].ravel()[nz]
    q = (np.arange(n_q) * dq)[:, None]
    assert np.all(np.abs(ratio[0] - np.cos(q * a * np.cos(phi) / HBARC) ** 2) <= 1e-12)
    assert np.all(np.abs(ratio[1] - np.cos(q * a * np.sin(phi) / HBARC) ** 2) <= 1e-12)
    assert np.all(np.abs(ratio[2] - 1.0) <= 1e-12)


@pytest.mark.parametrize("dimension", [3, 2])
def test_transverse_shift_leaves_the_modulus(fx, dimension):
    cells = _cells(15, 313 + dimension, dimension)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, dimension); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=2, dimension=dimension)
    qr = dict(dir=RAYS, dq=0.03, n_q=8)
    r1, _, cond = cf_hbtq.hbt_fourier(fl, cells, sp, g, tab, qr)
    moved = dict(cells, x=cells["x"] + 3.7, y=cells["y"] - 1.9)
    r2, _, _ = cf_hbtq.hbt_fourier(fl, moved, sp, g, tab, qr)
    assert np.array_equal(r1["Re"][:, 0], r2["Re"][:, 0])
    f1, f2 = (r["Re"] ** 2 + r["Im"] ** 2 for r in (r1, r2))
    assert np.all(np.abs(f2 - f1) <= 1e-12 * cond ** 2)


def test_small_q_curvature_is_the_radii(fx):
    """Positive weights (ideal f, outflow = 1): (1 - |F(q)|^2 / S0^2) / (q / hbar c)^2 = d.R^2.d + O(q^2) on every ray d.  These few-cell
    sources have long tails in t* (the O(q^2) term reaches ~1e3 (q / hbar c)^2 d.R^2.d), so the limit is taken from the points q and 2q
    of the ray (Richardson: (4 g(q) - g(2q)) / 3 removes the O(q^2) term), at the q of a geometric ladder with (q / hbar c)^2 d.R^2.d
    nearest 1e-8, where the rounding of 1 - |F|^2 / S0^2 (~3e-16) and the O(q^4) remainder are far below the 1e-5 bar."""
    cells = _cells(20, 4242, 3)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, 3); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=3, include_bulk=0, include_shear=0, outflow=1)
    m = cf_hbtq.hbt_moments(fl, cells, sp, g, tab)
    R = api.hbt_radii(m)
    R2 = np.array([[R["out"], R["outside"], R["outlong"]], [R["outside"], R["side"], R["sidelong"]], [R["outlong"], R["sidelong"], R["long"]]])
    want = np.einsum("ai,ijb,aj->ab", RAYS, R2, RAYS)                    # d.R^2.d per ray and bin
    # the |terms| of <(d.r)^2>: both sides extract a variance from sums dominated by the mean offset (far rapidity bins, where t* and z*
    # reach 1e4 fm, and bins where one cell dominates); a variance below 1e-4 of it loses digits to rounding on both sides
    S2 = np.array([[m["Soo"], m["Sos"], m["Sol"]], [m["Sos"], m["Sss"], m["Ssl"]], [m["Sol"], m["Ssl"], m["Sll"]]])
    raw = np.einsum("ai,ijb,aj->ab", np.abs(RAYS), np.abs(S2), np.abs(RAYS)) / np.where(m["S0"] != 0, m["S0"], 1.0)
    ladder = 10.0 ** np.arange(-7.0, -0.9, 0.25)                         # dq [GeV]
    got = []
    for dq in ladder:
        r, _, _ = cf_hbtq.hbt_fourier(fl, cells, sp, g, tab, dict(dir=RAYS, dq=dq, n_q=3))
        s0 = r["Re"][0, 0]
        ok = s0 > NORMAL
        gk = [np.where(ok, 1.0 - (r["Re"][:, k] ** 2 + r["Im"][:, k] ** 2) / np.where(ok, s0, 1.0) ** 2, np.nan) / (k * dq / HBARC) ** 2
              for k in (1, 2)]
        got.append((4.0 * gk[0] - gk[1]) / 3.0)
    got = np.array(got)
    x2 = (ladder / HBARC)[:, None, None] ** 2 * want[None]
    pick = np.argmin(np.abs(np.log10(np.maximum(x2, 1e-300)) + 8.0), axis=0)
    chosen = np.take_along_axis(got, pick[None], axis=0)[0]
    x2c = np.take_along_axis(x2, pick[None], axis=0)[0]
    ok = np.isfinite(chosen) & (x2c > 5e-9) & (x2c < 2e-8) & (want > 1e-4 * raw)
    assert ok.sum() > 0.5 * ok.size
    assert np.all(np.abs(chosen[ok] - want[ok]) <= 1e-5 * want[ok])


def test_hbt_correlation_formula():
    rng = np.random.default_rng(3)
    sp = dict(sign=np.array([-1.0, 1.0]), degeneracy=np.array([1.0, 2.0]))          # a boson, a spin-1/2 fermion
    re = rng.normal(size=(2, 3, 4)); im = rng.normal(size=(2, 3, 4))
    im[:, 0] = 0.0
    re[:, 0, 3] = 0.0                                                                # bin 3 (species 1): S0 = 0
    C_ = api.hbt_correlation(dict(Re=re, Im=im), sp)
    for b in range(4):
        s, gd = sp["sign"][b % 2], sp["degeneracy"][b % 2]
        for d in range(2):
            for k in range(3):
                want = 1.0 if re[d, 0, b] == 0 else 1.0 - s * (re[d, k, b] ** 2 + im[d, k, b] ** 2) / (gd * re[d, 0, b] ** 2)
                assert np.isclose(C_[d, k, b], want, rtol=1e-14, atol=0)
    assert np.all(C_[:, 0, :3:2] == 2.0)                                             # pions at q = 0: 1 + 1
    assert np.all(C_[:, :, 3] == 1.0)


def test_argument_and_scope_errors(fx):
    """Checked before any device work, so they hold with or without a GPU."""
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, 3); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=3)
    cells = _cells(10, 2, 3)
    qr = dict(dir=AXES, dq=0.01, n_q=5)
    for bad in (dict(fl, df_mode=3), dict(fl, df_mode=4), dict(fl, mode=2), dict(fl, include_baryon=1)):
        with pytest.raises(api.Is3dError) as e:
            api.hbt_fourier(bad, cells, sp, g, tab, qr)
        assert e.value.code == 2, bad                                                  # IS3D_ERR_UNSUPPORTED
    for k in ("x", "y"):
        with pytest.raises(api.Is3dError) as e:
            api.hbt_fourier(fl, {c: v for c, v in cells.items() if c != k}, sp, g, tab, qr)
        assert e.value.code == 1, k
    inf_dir = AXES.copy(); inf_dir[1, 2] = np.inf
    full = tables.grid(fx)
    for bad, grid in ((dict(qr, n_q=0), g), (dict(qr, dir=np.zeros((0, 3))), g), (dict(qr, dq=0.0), g), (dict(qr, dq=-0.01), g),
                      (dict(qr, dq=np.nan), g), (dict(qr, dq=np.inf), g), (dict(qr, dir=inf_dir), g),
                      (dict(qr, dir=RAYS, n_q=2000), full)):                       # 2 x 4 x 2000 x 48384 sums > 4 GiB
        with pytest.raises(api.Is3dError) as e:
            api.hbt_fourier(fl, cells, sp, grid, tab, bad)
        assert e.value.code == 1, bad                                                  # IS3D_ERR_ARGUMENT


def test_correlation_keys_refused_outside_their_scope(fx):
    lib = api.lib()
    chosen = [211, 321, 2212]
    with tempfile.TemporaryDirectory() as wd:
        out = os.path.join(wd, "x.bin").encode()
        for bad in (dict(operation=0, mode=1, df_mode=1), dict(operation=1, mode=2, df_mode=1), dict(operation=1, mode=1, df_mode=3),
                    dict(operation=1, mode=1, df_mode=4), dict(operation=1, mode=1, df_mode=1, include_baryon=1)):
            workdir.materialize(wd, fixture=fx, chosen=chosen, hbt_correlation=211, **bad)
            assert lib.is3d_b200_host_dump(wd.encode(), out) == 2, bad                 # IS3D_ERR_UNSUPPORTED
        for bad in (dict(hbt_correlation=-211), dict(hbt_correlation=211, hbt_dq=0.0), dict(hbt_correlation=211, hbt_q_points=0)):
            workdir.materialize(wd, fixture=fx, chosen=chosen, operation=1, mode=1, df_mode=1, **bad)
            assert lib.is3d_b200_host_dump(wd.encode(), out) == 1, bad                 # IS3D_ERR_ARGUMENT
        for ok in (dict(hbt_correlation=2212), dict(hbt_correlation=211, hbt_dq=0.01, hbt_q_points=5), dict(hbt_correlation=0), {}):
            workdir.materialize(wd, fixture=fx, chosen=chosen, operation=1, mode=1, df_mode=2, **ok)
            assert lib.is3d_b200_host_dump(wd.encode(), out) == 0, ok


def test_struct_layout_matches_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "is3d_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu %zu %zu %zu\\n", sizeof(is3d_hbt_qrays), offsetof(is3d_hbt_qrays, n_q),'
                   ' offsetof(is3d_hbt_qrays, dq), offsetof(is3d_hbt_qrays, dir), sizeof(is3d_hbt_fourier_result),'
                   ' offsetof(is3d_hbt_fourier_result, Re), offsetof(is3d_hbt_fourier_result, Im)); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got == [C.sizeof(api.HbtQrays), api.HbtQrays.n_q.offset, api.HbtQrays.dq.offset, api.HbtQrays.dir.offset,
                   C.sizeof(api.HbtFourierResult), api.HbtFourierResult.Re.offset, api.HbtFourierResult.Im.offset]
    assert [f for f, _ in api.HbtQrays._fields_] == ["n_dir", "n_q", "dq", "dir"]
    assert [f for f, _ in api.HbtFourierResult._fields_] == ["Re", "Im"]


# ------------------------------------------------------------------------------------------------ GPU
def _gpu():
    import torch
    torch.cuda.set_device(0)
    api.init()
    return torch


def _gpu_grid(fx, dimension):
    """Every pT point (several warps of lanes), a third of the phi and y points, every sixth eta point."""
    g = tables.grid(fx)
    g = dict(g, phi=g["phi"][::3].copy(), phi_weight=g["phi_weight"][::3].copy(), y=g["y"][::3].copy(), y_weight=g["y_weight"][::3].copy())
    if dimension == 2:
        g = dict(g, eta=g["eta"][::6].copy(), eta_weight=g["eta_weight"][::6].copy())
    return g


def _check_parity(got, ref, cond):
    """Every Re and Im sum within 1e-10 of the bin's sum of |w| (the phases cancel, so |F| can be far below it); the q = 0 sums, which
    do not cancel, per bin at 1e-10 with the conditioning of tests/common.py."""
    bad = {}
    for k in ("Re", "Im"):
        err = np.abs(got[k] - ref[k])
        if not np.all(err <= 1e-10 * cond):
            bad[k] = float(np.max(err / np.maximum(cond, 1e-300)))
    for d in range(got["Re"].shape[0]):
        rep = compare(got["Re"][d, 0], ref["Re"][d, 0], conditioning=cond)
        if not rep["ok"]:
            bad["Re[%d][0]" % d] = rep
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("dimension,df_mode,deltaf,outflow,memory,n_q,dq", [
    (3, 1, 1, 1, "host", 41, 0.005), (3, 2, 1, 0, "device", 23, 0.01), (3, 1, 0, 0, "host", 22, 0.02), (3, 2, 0, 1, "device", 5, 0.04),
    (2, 1, 1, 1, "device", 41, 0.005), (2, 2, 1, 0, "host", 23, 0.01), (2, 2, 0, 1, "device", 22, 0.02), (2, 1, 0, 0, "host", 5, 0.04),
    (3, 1, 1, 1, "host", 45, 0.3)])
def test_gpu_parity(fx, dimension, df_mode, deltaf, outflow, memory, n_q, dq):
    """pi / K / p (bosons and fermions), 3+1D and 2+1D, both linear delta-f models with delta-f on and off, outflow on and off, cells with
    u.dsigma <= 0, host and device memory, the axes and a diagonal, n_q with a ragged last q tile (23, 45) and an exact one (22), and
    q up to 13 GeV fm^-1 x 10 fm: phases of tens to hundreds of radians, where seed and recurrence drift would show."""
    torch = _gpu()
    cells = _cells(60, 700 + 10 * dimension + df_mode + 3 * deltaf + 7 * outflow, dimension, flip=4)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _gpu_grid(fx, dimension); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=df_mode, dimension=dimension, include_bulk=deltaf, include_shear=deltaf, outflow=outflow)
    qr = dict(dir=RAYS, dq=dq, n_q=n_q)
    ref, skipped, cond = cf_hbtq.hbt_fourier(fl, cells, sp, g, tab, qr)
    if memory == "device":
        dc = {k: torch.tensor(v, device="cuda") for k, v in cells.items()}
        out, st = api.hbt_fourier(fl, dc, sp, g, tab, qr, memory="device")
        torch.cuda.synchronize()
        got = {k: v.cpu().numpy() for k, v in out.items()}
    else:
        got, st = api.hbt_fourier(fl, cells, sp, g, tab, qr)
    assert skipped == 4 and st["cells_skipped_udsigma"] == 4
    assert got["Re"].shape == (len(RAYS), n_q, cfo.n_bins(sp, g))
    _check_parity(got, ref, cond)


@pytest.mark.gpu
@pytest.mark.parametrize("dimension", [3, 2])
def test_gpu_q0_spectra_reproducible_and_multi(fx, dimension):
    _gpu()
    cells = _cells(300, 565 + dimension, dimension, flip=2)
    sp = tables.species(fx, 1, "chosen_pikp"); g = tables.grid(fx); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=dimension)
    qr = dict(dir=RAYS, dq=0.01, n_q=30)
    a, _ = api.hbt_fourier(fl, cells, sp, g, tab, qr)
    b, _ = api.hbt_fourier(fl, cells, sp, g, tab, qr)
    for k in ("Re", "Im"):
        assert np.array_equal(a[k], b[k]), k
    for d in range(1, len(RAYS)):
        assert np.array_equal(a["Re"][d, 0], a["Re"][0, 0])
    assert np.all(a["Im"][:, 0] == 0)
    dN, _ = api.smooth_spectra(fl, cells, sp, g, tab)
    cond = np.zeros_like(dN)
    cfo.smooth(fl, cells, sp, g, tab, conditioning=cond)
    rep = compare(a["Re"][0, 0], dN, conditioning=cond)
    assert rep["ok"], rep
    api.init_devices(0)
    m, _ = api.hbt_fourier(fl, cells, sp, g, tab, qr, multi=True)
    scale = np.maximum(np.abs(a["Re"]).max(axis=(0, 1)), np.abs(a["Im"]).max(axis=(0, 1)))      # per bin, ~ its sum of |w|
    for k in ("Re", "Im"):
        assert np.all(np.abs(m[k] - a[k]) <= 1e-13 * scale), k


@pytest.mark.gpu
def test_gpu_empty_surface_and_table_range(fx):
    _gpu()
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, 3); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=3)
    qr = dict(dir=AXES, dq=0.01, n_q=5)
    out, st = api.hbt_fourier(fl, _cells(0, 1, 3), sp, g, tab, qr)
    assert all(np.all(v == 0) for v in out.values()) and st["cells_skipped_udsigma"] == 0
    hot = _cells(10, 3, 3)
    hot["T"] = hot["T"].copy(); hot["T"][4] = 10.0 * tab["T"].max()
    with pytest.raises(api.Is3dError) as e:
        api.hbt_fourier(fl, hot, sp, g, tab, qr)
    assert e.value.code == 3                                                           # IS3D_ERR_TABLE_RANGE


def _run(wd):
    lib = api.lib()
    lib.is3d_b200_host_error.restype = C.c_char_p
    rc = lib.is3d_b200_run_workdir(wd.encode(), None, C.c_int64(0), None, 0, None)
    assert rc == 0, lib.is3d_b200_host_error().decode()


@pytest.mark.gpu
@pytest.mark.parametrize("dimension,df_mode,mcid", [(3, 1, 211), (2, 2, 2212)])
def test_gpu_workdir_correlation_file(fx, dimension, df_mode, mcid):
    _gpu()
    cols = synthetic.surface_vh(60, 4331 + dimension, three_d=(dimension == 3))
    chosen = [211, 321, 2212]
    dq, n_q = 0.01, 7
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=cols, chosen=chosen, fixture=fx, operation=1, mode=1, dimension=dimension, df_mode=df_mode,
                            hbt_correlation=mcid, hbt_dq=dq, hbt_q_points=n_q)
        _run(wd)
        hbt = sorted(os.listdir(os.path.join(wd, "results", "hbt")))
        path = os.path.join(wd, "results", "hbt", "C_%d.dat" % mcid)
        header = open(path).readline().split()
        got = np.loadtxt(path, skiprows=1, ndmin=2)
    assert hbt == ["C_%d.dat" % mcid]
    assert header == ["y", "phip", "pT", "q", "S0", "C_out", "C_side", "C_long"]
    cells = synthetic.columns_to_cells(cols, 1)
    sp = tables.species(fx, 1, [mcid]); g = tables.grid(fx); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=df_mode, dimension=dimension)
    api.init_devices(0)
    sums, _ = api.hbt_fourier(fl, cells, sp, g, tab, dict(dir=AXES, dq=dq, n_q=n_q), multi=True)
    Cq = api.hbt_correlation(sums, sp)
    ny = 1 if dimension == 2 else len(g["y"])
    shape = (len(g["y"]), len(g["phi"]), len(g["pT"]))
    s0 = sums["Re"][0, 0].reshape(shape)[:ny]
    cq = [np.moveaxis(Cq[d].reshape((n_q,) + shape)[:, :ny], 0, -1) for d in range(3)]          # [y][phi][pT][k]
    yv, phiv, pTv, qv = np.meshgrid(g["y"][:ny] if dimension == 3 else [0.0], g["phi"], g["pT"], np.arange(n_q) * dq, indexing="ij")
    want = np.column_stack([yv.ravel(), phiv.ravel(), pTv.ravel(), qv.ravel(), np.repeat(s0.ravel(), n_q)] + [c.ravel() for c in cq])
    assert got.shape == want.shape
    assert np.all(np.abs(got - want) <= 1e-8 * np.abs(want) + 1e-300), np.max(np.abs(got - want) / np.maximum(np.abs(want), 1e-300))
    q0 = (got[:, 3] == 0) & (got[:, 4] != 0)
    assert np.all(got[q0, 5:] == (2.0 if mcid == 211 else 0.5))                         # C(0) = 1 - sign / g


@pytest.mark.gpu
def test_gpu_workdir_without_the_key_is_unchanged(fx):
    """Without hbt_correlation (or with 0) the run writes the files it always wrote; with it, only C_<mcid>.dat is added."""
    _gpu()
    cols = synthetic.surface_vh(20, 98)
    listing, contents = [], []
    for extra in ({}, dict(hbt_correlation=0, hbt_dq=0.01), dict(hbt_correlation=211)):
        with tempfile.TemporaryDirectory() as wd:
            workdir.materialize(wd, surface_columns=cols, fixture=fx, chosen=[211, 321], operation=1, mode=1, dimension=3, df_mode=1, **extra)
            _run(wd)
            res = os.path.join(wd, "results")
            names = sorted(os.path.relpath(os.path.join(d, f), res) for d, _, fs in os.walk(res) for f in fs)
            listing.append(names)
            contents.append({p: open(os.path.join(res, p), "rb").read() for p in names})
    assert listing[0] == listing[1]
    assert contents[0] == contents[1]
    assert not any(p.startswith("hbt" + os.sep) for p in listing[0])
    assert listing[2] == sorted(listing[0] + [os.path.join("hbt", "C_211.dat")])
    assert all(contents[2][p] == contents[0][p] for p in listing[0])
