"""Spin polarization from thermal vorticity (mode 5 surfaces): the oracle against an independent restatement in Milne coordinates, the
algebra of the mean spin vector, the anchor to the pinned ideal spectra, the reader, the ABI and (on the GPU) the CUDA path."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from common import compare
from is3d_b200 import api, synthetic, tables, workdir
from oracle import cf_oracle as cfo
from oracle import cf_polzn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HBARC = synthetic.HBARC
N_KEYS = ("St", "Sx", "Sy", "Sz")


def _small_grid(fx, dimension):
    """A few points of every table (the eta table thinned in 2+1D) to keep the numpy restatement quick."""
    g = tables.grid(fx)
    g = dict(g, pT=g["pT"][::8].copy(), pT_weight=g["pT_weight"][::8].copy(), phi=g["phi"][::5].copy(), phi_weight=g["phi_weight"][::5].copy(),
             y=g["y"][::4].copy(), y_weight=g["y_weight"][::4].copy())
    if dimension == 2:
        g = dict(g, eta=g["eta"][::12].copy(), eta_weight=g["eta_weight"][::12].copy())
    return g


def _problem(fx, n_cells, seed, dimension, flip=0):
    cells = synthetic.columns_to_cells(synthetic.surface_vh(n_cells, seed, three_d=(dimension == 3)), 1)
    if flip:                                     # cells with u.dsigma <= 0: the spatial normal reversed and enlarged
        for k in ("dat", "dax", "day"):
            cells[k] = cells[k].copy()
        cells["dat"][:flip] = -cells["dat"][:flip]
    return cells, synthetic.vorticity(n_cells, seed + 7)


def numpy_milne(flags, cells, vort, sp, g):
    """N^mu and Snorm restated with the Milne-coordinate contraction: eps^{tau x y eta} = 1/tau, p_mu lowered with
    g = diag(1, -1, -1, -tau^2), varpi_{mu nu} taken from the columns as they are, the contravariant result converted to Cartesian
    components at the slot's eta (A^t = cosh eta A^tau + tau sinh eta A^eta, A^z = sinh eta A^tau + tau cosh eta A^eta)."""
    import itertools
    eps = np.zeros((4, 4, 4, 4))
    for perm in itertools.permutations(range(4)):
        eps[perm] = np.linalg.det(np.eye(4)[list(perm)])
    pref = (2 * np.pi * HBARC) ** -3
    ns, npT, nphi, ny = len(sp["mass"]), len(g["pT"]), len(g["phi"]), len(g["y"])
    d2 = flags["dimension"] == 2
    N = np.zeros((4, ny, nphi, npT, ns)); Sn = np.zeros((ny, nphi, npT, ns))
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
        W = np.zeros((4, 4))
        W[0, 1], W[0, 2], W[0, 3], W[1, 2], W[1, 3], W[2, 3] = (vort[k][i] for k in ("wtx", "wty", "wtn", "wxy", "wxn", "wyn"))
        W = W - W.T
        for iy in range(1 if d2 else ny):              # 2+1D: y = 0 fills the first plane, like the spectra
            y = 0.0 if d2 else g["y"][iy]
            slots = zip(g["eta"], g["eta_weight"]) if d2 else [(cells["eta"][i], 1.0)]
            for eta, wt in slots:
                pt = mT * np.cosh(y - eta); pn = mT / tau * np.sinh(y - eta)
                pds = wt * (pt * dat + px * dax + py * day + pn * dan)
                pu = pt * ut - px * ux - py * uy - tau * tau * pn * un
                with np.errstate(over="ignore"):        # exp overflows to inf far in the tail: f = 0, as in the reference
                    f = 1.0 / (np.exp(pu / cells["T"][i]) + sign)
                keep = (pds > 0) if flags["outflow"] else np.ones_like(pds, dtype=bool)
                t = np.where(keep, pds * f, 0.0)
                plow = np.stack(np.broadcast_arrays(pt, -px, -py, -tau * tau * pn))
                A = np.einsum("abcd,bc,d...->a...", eps, W, plow) / tau
                At = np.cosh(eta) * A[0] + tau * np.sinh(eta) * A[3]
                Az = np.sinh(eta) * A[0] + tau * np.cosh(eta) * A[3]
                Ac = np.stack([At, A[1], A[2], Az])
                Sn[iy] += pref * sp["degeneracy"] * t
                N[:, iy] += pref * sp["degeneracy"] * t * (1 - sign * f) * (-Ac / (8 * m))
    return {k: N[j].ravel() for j, k in enumerate(N_KEYS)} | {"Snorm": Sn.ravel()}


@pytest.mark.parametrize("dimension,outflow", [(3, 1), (2, 1), (3, 0)])
def test_oracle_matches_milne_restatement(fx, dimension, outflow):
    cells, vort = _problem(fx, 20, 2024 + dimension, dimension)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, dimension)
    fl = tables.flags(df_mode=1, dimension=dimension, outflow=outflow)
    got, skipped, cond = cf_polzn.spin_polarization(fl, cells, vort, sp, g, conditioning=True)
    want = numpy_milne(fl, cells, vort, sp, g)
    assert skipped == 0
    assert np.all(np.abs(got["Snorm"] - want["Snorm"]) <= 1e-13 * np.abs(want["Snorm"]))
    for k in N_KEYS:
        assert np.any(got[k] != 0)
        assert np.all(np.abs(got[k] - want[k]) <= 1e-13 * cond[k]), k


def _rest_cell(w):
    cells = {k: np.zeros(1) for k in ("eta", "dax", "day", "dan", "ux", "uy", "un")}
    cells.update(tau=np.ones(1), dat=np.ones(1), T=np.full(1, 0.15), P=np.full(1, 0.05), E=np.full(1, 0.3))
    vort = {k: np.zeros(1) for k in synthetic.VORTICITY_COLUMNS}
    vort["wxy"] = np.full(1, w)
    return cells, vort


def test_sign_anchor_cell_at_rest(fx):
    """Only varpi_xy = w at rest: S^z = w E (1 - Theta f) / (4m) and S^t = w p^z (1 - Theta f) / (4m), i.e. S along the rotation."""
    w = 0.03
    cells, vort = _rest_cell(w)
    sp = tables.species(fx, 1, "chosen_pikp"); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=3)
    r, _ = cf_polzn.spin_polarization(fl, cells, vort, sp, g)
    S, rest = api.mean_spin(r, sp, g, 3)
    yy, ff, pp, mm = np.meshgrid(g["y"], g["phi"], g["pT"], sp["mass"], indexing="ij")
    _, _, _, sg = np.meshgrid(g["y"], g["phi"], g["pT"], sp["sign"], indexing="ij")
    mT = np.sqrt(mm ** 2 + pp ** 2); E = (mT * np.cosh(yy)).ravel(); pz = (mT * np.sinh(yy)).ravel()
    with np.errstate(over="ignore"):
        f = 1.0 / (np.exp(E / 0.15) + sg.ravel())
    fbar = 1 - sg.ravel() * f
    nz = r["Snorm"] > 0
    assert nz.sum() > 0.9 * nz.size
    assert np.allclose(S[3][nz], (w * E * fbar / (4 * mm.ravel()))[nz], rtol=1e-13, atol=0)
    assert np.all(S[3][nz] > 0)
    assert np.allclose(S[0][nz], (w * pz * fbar / (4 * mm.ravel()))[nz], rtol=1e-13, atol=1e-300)
    assert np.all(S[1] == 0) and np.all(S[2] == 0)
    # rest frame: S* = (0, 0, S^z - S^t p^z / (E + m)), along +z
    assert np.all(rest[2][nz] > 0)


def test_algebra_orthogonality_zero_and_linearity(fx):
    cells, vort = _problem(fx, 15, 77, 3)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, 3)
    fl = tables.flags(df_mode=1, dimension=3)
    r1, _, c1 = cf_polzn.spin_polarization(fl, cells, vort, sp, g, conditioning=True)
    yy, ff, pp, mm = np.meshgrid(g["y"], g["phi"], g["pT"], sp["mass"], indexing="ij")
    mT = np.sqrt(mm ** 2 + pp ** 2)
    p = [(mT * np.cosh(yy)).ravel(), (pp * np.cos(ff)).ravel(), (pp * np.sin(ff)).ravel(), (mT * np.sinh(yy)).ravel()]
    N = [r1[k] for k in N_KEYS]
    pN = p[0] * N[0] - p[1] * N[1] - p[2] * N[2] - p[3] * N[3]
    norm = np.sqrt(sum(n * n for n in N))
    assert np.all(np.abs(pN) <= 1e-13 * p[0] * norm)
    zero = {k: np.zeros_like(v) for k, v in vort.items()}
    r0, _ = cf_polzn.spin_polarization(fl, cells, zero, sp, g)
    assert all(np.all(r0[k] == 0) for k in N_KEYS) and np.array_equal(r0["Snorm"], r1["Snorm"])
    vort2 = synthetic.vorticity(15, 78)
    r2, _, c2 = cf_polzn.spin_polarization(fl, cells, vort2, sp, g, conditioning=True)
    mix = {k: 2.0 * vort[k] - 0.5 * vort2[k] for k in vort}
    r3, _ = cf_polzn.spin_polarization(fl, cells, mix, sp, g)
    for k in N_KEYS:
        assert np.all(np.abs(r3[k] - (2.0 * r1[k] - 0.5 * r2[k])) <= 1e-13 * (2.0 * c1[k] + 0.5 * c2[k])), k


@pytest.mark.parametrize("dimension", [3, 2])
def test_snorm_is_the_ideal_spectrum(fx, dimension):
    cells, vort = _problem(fx, 30, 31 + dimension, dimension, flip=3)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, dimension); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=dimension, include_bulk=0, include_shear=0)
    r, skipped = cf_polzn.spin_polarization(fl, cells, vort, sp, g)
    dN, skipped_smooth, _ = cfo.smooth(fl, cells, sp, g, tab)
    assert skipped == skipped_smooth == 3
    assert np.array_equal(r["Snorm"], dN)


def _host_dump(wd):
    import struct
    lib = api.lib()
    out = os.path.join(wd, "host_dump.bin")
    lib.is3d_b200_host_error.restype = C.c_char_p
    assert lib.is3d_b200_host_dump(wd.encode(), out.encode()) == 0, lib.is3d_b200_host_error().decode()
    rec, data, pos = {}, open(out, "rb").read(), 0
    while pos < len(data):
        (ln,) = struct.unpack_from("<i", data, pos); pos += 4
        name = data[pos:pos + ln].decode(); pos += ln
        (n,) = struct.unpack_from("<q", data, pos); pos += 8
        rec[name] = np.frombuffer(data, dtype="<f8", count=n, offset=pos).copy(); pos += 8 * n
    return rec


def _mode5_columns(n, seed, dimension=3):
    base = synthetic.surface_vh(n, seed, three_d=(dimension == 3))
    vort = synthetic.vorticity(n, seed + 1)
    return np.column_stack([base] + [vort[k] for k in synthetic.VORTICITY_COLUMNS]), base, vort


def test_reader_keeps_the_vorticity_columns(fx):
    cols, _, vort = _mode5_columns(9, 5)
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=cols, fixture=fx, operation=1, mode=5, dimension=3, df_mode=1)
        open(os.path.join(wd, "average_thermodynamic_quantities.dat"), "w").write("0.15\n0.3\n0.05\n0\n0")
        d = _host_dump(wd)
    for k in synthetic.VORTICITY_COLUMNS:
        assert np.array_equal(d[k], vort[k]), k


def test_spin_polarization_key_needs_mode5(fx):
    lib = api.lib()
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, fixture=fx, operation=1, mode=1, spin_polarization=1)
        assert lib.is3d_b200_host_dump(wd.encode(), os.path.join(wd, "x.bin").encode()) == 2      # IS3D_ERR_UNSUPPORTED
        workdir.materialize(wd, fixture=fx, operation=1, mode=1, spin_polarization=0)
        assert lib.is3d_b200_host_dump(wd.encode(), os.path.join(wd, "x.bin").encode()) == 0


def test_struct_layouts_match_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "is3d_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu %zu\\n", sizeof(is3d_vorticity), offsetof(is3d_vorticity, wyn),'
                   ' sizeof(is3d_polarization_result), offsetof(is3d_polarization_result, Sz), offsetof(is3d_polarization_result, Snorm));'
                   ' return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got == [C.sizeof(api.Vorticity), api.Vorticity.wyn.offset, C.sizeof(api.PolarizationResult), api.PolarizationResult.Sz.offset,
                   api.PolarizationResult.Snorm.offset]
    assert [f for f, _ in api.Vorticity._fields_] == list(synthetic.VORTICITY_COLUMNS)


# ------------------------------------------------------------------------------------------------ GPU
def _gpu():
    import torch
    torch.cuda.set_device(0)
    api.init()
    return torch


def _check_parity(got, ref, cond):
    assert compare(got["Snorm"], ref["Snorm"])["ok"], compare(got["Snorm"], ref["Snorm"])
    for k in N_KEYS:
        rep = compare(got[k], ref[k], conditioning=cond[k])
        assert rep["ok"], (k, rep)


@pytest.mark.gpu
@pytest.mark.parametrize("dimension,outflow,chosen,memory", [
    (3, 1, "chosen_pikp", "host"), (3, 0, "chosen_pikp", "device"), (2, 1, "chosen_pikp", "host"), (2, 0, "chosen_pikp", "device"),
    (3, 1, "chosen_urqmd", "host")])
def test_gpu_parity(fx, dimension, outflow, chosen, memory):
    """Fermions and bosons (pi/K/p; the 305-species list), 3+1D and 2+1D, outflow on and off, cells with u.dsigma <= 0, host and
    device memory: all five arrays against the oracle at 1e-10 per bin."""
    torch = _gpu()
    n = 40 if chosen == "chosen_urqmd" else 150
    cells, vort = _problem(fx, n, 900 + dimension + 10 * outflow, dimension, flip=5)
    sp = tables.species(fx, 1, chosen); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=dimension, outflow=outflow)
    ref, skipped, cond = cf_polzn.spin_polarization(fl, cells, vort, sp, g, conditioning=True)
    if memory == "device":
        dc = {k: torch.tensor(v, device="cuda") for k, v in cells.items()}
        dv = {k: torch.tensor(v, device="cuda") for k, v in vort.items()}
        out, st = api.spin_polarization(fl, dc, dv, sp, g, memory="device")
        torch.cuda.synchronize()
        got = {k: v.cpu().numpy() for k, v in out.items()}
    else:
        got, st = api.spin_polarization(fl, cells, vort, sp, g)
    assert skipped == 5 and st["cells_skipped_udsigma"] == 5
    _check_parity(got, ref, cond)


@pytest.mark.gpu
def test_gpu_empty_surface_and_errors(fx):
    _gpu()
    sp = tables.species(fx, 1, "chosen_pikp"); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=3)
    cells, vort = _problem(fx, 0, 1, 3)
    out, st = api.spin_polarization(fl, cells, vort, sp, g)
    assert all(np.all(v == 0) for v in out.values()) and st["cells_skipped_udsigma"] == 0
    cells, vort = _problem(fx, 10, 2, 3)
    for bad, code in [(dict(fl, mode=2), 2), (dict(fl, include_baryon=1), 2)]:
        with pytest.raises(api.Is3dError) as e:
            api.spin_polarization(bad, cells, vort, sp, g)
        assert e.value.code == code
    with pytest.raises(api.Is3dError) as e:
        api.spin_polarization(fl, cells, None, sp, g)
    assert e.value.code == 1
    massless = dict(sp, mass=np.where(np.arange(len(sp["mass"])) == 0, 0.0, sp["mass"]))
    with pytest.raises(api.Is3dError) as e:
        api.spin_polarization(fl, cells, vort, massless, g)
    assert e.value.code == 1


@pytest.mark.gpu
@pytest.mark.parametrize("dimension", [3, 2])
def test_gpu_snorm_equals_spectra_and_reproducible(fx, dimension):
    _gpu()
    cells, vort = _problem(fx, 300, 555 + dimension, dimension, flip=2)
    sp = tables.species(fx, 1, "chosen_pikp"); g = tables.grid(fx); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=dimension, include_bulk=0, include_shear=0)
    a, _ = api.spin_polarization(fl, cells, vort, sp, g)
    b, _ = api.spin_polarization(fl, cells, vort, sp, g)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    dN, _ = api.smooth_spectra(fl, cells, sp, g, tab)
    assert compare(a["Snorm"], dN)["ok"], compare(a["Snorm"], dN)
    api.init_devices(0)
    m, st = api.spin_polarization(fl, cells, vort, sp, g, multi=True)
    for k in a:
        scale = np.abs(a[k]).max()
        assert np.abs(m[k] - a[k]).max() <= 1e-13 * scale, k


def _read_polarization(path):
    return np.loadtxt(path, skiprows=1, ndmin=2)


@pytest.mark.gpu
@pytest.mark.parametrize("dimension", [3, 2])
def test_gpu_workdir_polarization_files(fx, dimension):
    _gpu()
    cols, base, vort = _mode5_columns(60, 4321 + dimension, dimension)
    chosen = [3122, -3122, 211]
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=cols, chosen=chosen, fixture=fx, operation=1, mode=5, dimension=dimension, df_mode=1,
                            spin_polarization=1)
        open(os.path.join(wd, "average_thermodynamic_quantities.dat"), "w").write("0.15\n0.3\n0.05\n0\n0")
        lib = api.lib()
        lib.is3d_b200_host_error.restype = C.c_char_p
        rc = lib.is3d_b200_run_workdir(wd.encode(), None, C.c_int64(0), None, 0, None)
        assert rc == 0, lib.is3d_b200_host_error().decode()
        files = {c: _read_polarization(os.path.join(wd, "results", "polarization", "S_%d.dat" % c)) for c in chosen}
        header = open(os.path.join(wd, "results", "polarization", "S_3122.dat")).readline().split()
    assert header == ["y", "phip", "pT", "Snorm", "St", "Sx", "Sy", "Sz", "Sx_rest", "Sy_rest", "Sz_rest"]
    cells = synthetic.columns_to_cells(base, 1)
    sp = tables.species(fx, 1, chosen); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=dimension)
    ref, _ = cf_polzn.spin_polarization(fl, cells, vort, sp, g)
    S, rest = api.mean_spin(ref, sp, g, dimension)
    ny = 1 if dimension == 2 else len(g["y"])
    for s, c in enumerate(chosen):
        want = np.column_stack([ref["Snorm"].reshape(len(g["y"]), len(g["phi"]), len(g["pT"]), -1)[:ny, :, :, s].ravel()] +
                               [v.reshape(len(g["y"]), len(g["phi"]), len(g["pT"]), -1)[:ny, :, :, s].ravel() for v in list(S) + list(rest)])
        got = files[c][:, 3:]
        assert got.shape == want.shape
        scale = np.abs(want).max(axis=0)
        assert np.all(np.abs(got - want) <= 2e-8 * np.abs(want) + 1e-12 * scale), c


@pytest.mark.gpu
def test_gpu_workdir_without_the_key_is_unchanged(fx):
    """Without spin_polarization the mode-5 run writes the files it always wrote, and no polarization file."""
    _gpu()
    cols, _, _ = _mode5_columns(20, 99)
    listing = []
    for extra in ({}, dict(spin_polarization=0)):
        with tempfile.TemporaryDirectory() as wd:
            workdir.materialize(wd, surface_columns=cols, fixture=fx, operation=1, mode=5, dimension=3, df_mode=1, **extra)
            open(os.path.join(wd, "average_thermodynamic_quantities.dat"), "w").write("0.15\n0.3\n0.05\n0\n0")
            assert api.lib().is3d_b200_run_workdir(wd.encode(), None, C.c_int64(0), None, 0, None) == 0
            res = os.path.join(wd, "results")
            listing.append(sorted(os.path.relpath(os.path.join(d, f), res) for d, _, fs in os.walk(res) for f in fs))
    assert listing[0] == listing[1]
    assert not any(p.startswith("polarization" + os.sep) for p in listing[0])
    assert "dN_pTdpTdphidy.dat" in listing[0]
