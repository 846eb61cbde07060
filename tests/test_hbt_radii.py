"""HBT radii from the space-time moments of the emission function: the oracle against an independent restatement with an explicit
lab-frame boost, its S0 against the pinned spectra, analytic anchors, the host layer and the ABI, and (on the GPU) the CUDA path."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from common import compare
from is3d_b200 import api, synthetic, tables, workdir
from oracle import cf_hbt
from oracle import cf_oracle as cfo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HBARC = synthetic.HBARC
FIELDS = cf_hbt.HBT_FIELDS
RADII = api.HBT_RADII
NORMAL = 1e-290                                  # weights well above the sub-normal range


def _small_grid(fx, dimension):
    """A few points of every table (the eta table thinned in 2+1D, symmetric about 0) to keep the numpy restatement quick."""
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


def numpy_lab_boost(flags, cells, sp, g):
    """Ideal-f weights (the flags must switch delta-f off) and coordinates from the lab-frame point (t, x, y, z) = (tau cosh eta, x, y,
    tau sinh eta), boosted to the LCMS of the bin explicitly: t* = t cosh y - z sinh y, z* = z cosh y - t sinh y."""
    assert not flags["include_shear"] and not flags["include_bulk"]
    pref = (2 * np.pi * HBARC) ** -3
    ns, npT, nphi, ny = len(sp["mass"]), len(g["pT"]), len(g["phi"]), len(g["y"])
    d2 = flags["dimension"] == 2
    S = np.zeros((10, ny, nphi, npT, ns)); A = np.zeros_like(S)
    m = np.asarray(sp["mass"])[None, None, :]; sign = np.asarray(sp["sign"])[None, None, :]
    pT = g["pT"][None, :, None]; phi = g["phi"][:, None, None]
    mT = np.sqrt(m * m + pT * pT)
    px = pT * np.cos(phi) + 0 * m; py = pT * np.sin(phi) + 0 * m
    beta = pT / mT
    for i in range(len(cells["tau"])):
        tau = cells["tau"][i]; ux, uy, un = cells["ux"][i], cells["uy"][i], cells["un"][i]
        ut = np.sqrt(1 + ux * ux + uy * uy + tau * tau * un * un)
        dat, dax, day, dan = (cells[k][i] for k in ("dat", "dax", "day", "dan"))
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
                ts, zs = t * np.cosh(y) - z * np.sinh(y), z * np.cosh(y) - t * np.sinh(y)
                o = xc * np.cos(phi) + yc * np.sin(phi) - beta * ts
                s = -xc * np.sin(phi) + yc * np.cos(phi) + 0 * o
                l = zs + 0 * o
                for q, v in enumerate((1, o, s, l, o * o, s * s, l * l, o * s, o * l, s * l)):
                    S[q, iy] += w * v
                # |terms| of this restatement: the boost cancels where eta ~ y
                tsa, zsa = t * np.cosh(y) + abs(z * np.sinh(y)), abs(z) * np.cosh(y) + t * abs(np.sinh(y))
                oa = abs(xc * np.cos(phi)) + abs(yc * np.sin(phi)) + beta * tsa
                sa = abs(xc * np.sin(phi)) + abs(yc * np.cos(phi)) + 0 * oa
                la = zsa + 0 * oa
                for q, v in enumerate((1, oa, sa, la, oa * oa, sa * sa, la * la, oa * sa, oa * la, sa * la)):
                    A[q, iy] += np.abs(w) * v
    return {k: S[q].ravel() for q, k in enumerate(FIELDS)}, {k: A[q].ravel() for q, k in enumerate(FIELDS)}


@pytest.mark.parametrize("dimension,outflow", [(3, 1), (2, 1), (3, 0)])
def test_oracle_matches_numpy_lab_boost(fx, dimension, outflow):
    cells = _cells(12, 4040 + dimension, dimension)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, dimension); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=dimension, include_bulk=0, include_shear=0, outflow=outflow)
    got, skipped, cond = cf_hbt.hbt_moments(fl, cells, sp, g, tab, conditioning=True)
    want, want_cond = numpy_lab_boost(fl, cells, sp, g)
    assert skipped == 0
    for k in FIELDS:
        if not (dimension == 2 and k in ("Sl", "Sol", "Ssl")):          # 2+1D: these vanish (test_2d_long_odd_sums_vanish)
            assert np.any(got[k] != 0), k
        assert np.all(np.abs(got[k] - want[k]) <= 1e-13 * (cond[k] + want_cond[k])), k


@pytest.mark.parametrize("dimension", [3, 2])
@pytest.mark.parametrize("df_mode,deltaf", [(1, 1), (1, 0), (2, 1), (2, 0)])
def test_oracle_s0_is_the_spectrum(fx, dimension, df_mode, deltaf):
    cells = _cells(25, 61 + dimension, dimension, flip=3)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, dimension); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=df_mode, dimension=dimension, include_bulk=deltaf, include_shear=deltaf)
    r, skipped = cf_hbt.hbt_moments(fl, cells, sp, g, tab)
    dN, skipped_smooth, _ = cfo.smooth(fl, cells, sp, g, tab)
    assert skipped == skipped_smooth == 3
    assert np.array_equal(r["S0"], dN)


def _one_cell(x=0.0, y=0.0):
    c = synthetic.columns_to_cells(synthetic.surface_vh(1, 8, three_d=True), 1)
    c["x"] = np.full(1, x); c["y"] = np.full(1, y)
    return c


def test_single_cell_has_zero_radii(fx):
    sp = tables.species(fx, 1, "chosen_pikp"); g = tables.grid(fx); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=3)
    r, _ = cf_hbt.hbt_moments(fl, _one_cell(3.0, -2.0), sp, g, tab)
    R = api.hbt_radii(r)
    nz = r["S0"] > NORMAL                        # the far tails carry sub-normal weights, whose products lose digits
    assert nz.sum() > 0.5 * nz.size
    scale = np.maximum.reduce([np.abs(r[k][nz] / r["S0"][nz]) for k in ("Soo", "Sss", "Sll")])
    for k in RADII:
        assert np.all(np.abs(R[k][nz]) <= 1e-13 * scale), k


def test_two_cells_at_plus_minus_a(fx):
    a = 2.5
    one = _one_cell()
    cells = {k: np.concatenate([v, v]) for k, v in one.items()}
    cells["x"] = np.array([a, -a]); cells["y"] = np.zeros(2)
    sp = tables.species(fx, 1, "chosen_pikp"); g = tables.grid(fx); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=3)
    r, _ = cf_hbt.hbt_moments(fl, cells, sp, g, tab)
    R = api.hbt_radii(r)
    nz = r["S0"] > NORMAL
    assert nz.sum() > 0.5 * nz.size
    phi = np.meshgrid(g["y"], g["phi"], g["pT"], sp["mass"], indexing="ij")[1].ravel()[nz]
    # rounding: R^2_ij is a difference of second moments that include (beta t*)^2 and z*^2 (up to ~1e6 fm^2 in the far rapidity bins)
    tol = 1e-13 * (a * a + np.maximum(r["Soo"][nz], r["Sll"][nz]) / r["S0"][nz])
    assert np.all(np.abs(R["out"][nz] - a * a * np.cos(phi) ** 2) <= tol)
    assert np.all(np.abs(R["side"][nz] - a * a * np.sin(phi) ** 2) <= tol)
    assert np.all(np.abs(R["outside"][nz] + a * a * np.sin(phi) * np.cos(phi)) <= tol)
    for k in ("long", "outlong", "sidelong"):
        assert np.all(np.abs(R[k][nz]) <= tol), k


@pytest.mark.parametrize("dimension", [3, 2])
def test_transverse_shift_leaves_radii(fx, dimension):
    cells = _cells(20, 303 + dimension, dimension)
    sp = tables.species(fx, 1, "chosen_pikp"); g = _small_grid(fx, dimension); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=2, dimension=dimension)
    r1, _ = cf_hbt.hbt_moments(fl, cells, sp, g, tab)
    moved = dict(cells, x=cells["x"] + 3.7, y=cells["y"] - 1.9)
    r2, _ = cf_hbt.hbt_moments(fl, moved, sp, g, tab)
    assert np.array_equal(r1["S0"], r2["S0"])
    R1, R2 = api.hbt_radii(r1), api.hbt_radii(r2)
    for k in RADII:
        assert np.all(np.abs(R2[k] - R1[k]) <= 1e-10 * (1.0 + np.abs(R1[k]))), k


def test_2d_long_odd_sums_vanish(fx):
    """u^eta = dsigma_eta = 0 (and pi^{x eta} = pi^{y eta} = 0) on the symmetric eta table: the weight is even in eta, z* odd."""
    g = _small_grid(fx, 2)
    g["eta"] = 0.5 * (g["eta"] - g["eta"][::-1]); g["eta_weight"] = 0.5 * (g["eta_weight"] + g["eta_weight"][::-1])
    assert np.array_equal(g["eta"], -g["eta"][::-1]) and np.array_equal(g["eta_weight"], g["eta_weight"][::-1])
    cells = _cells(15, 717, 2)
    sp = tables.species(fx, 1, "chosen_pikp"); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=2)
    r, _, cond = cf_hbt.hbt_moments(fl, cells, sp, g, tab, conditioning=True)
    for k in ("Sl", "Sol", "Ssl"):
        assert np.all(np.abs(r[k]) <= 1e-12 * cond[k]), k
    assert np.all(r["Sll"][r["S0"] > NORMAL] > 0)


def test_hbt_radii_formula_and_zero_bins():
    rng = np.random.default_rng(1)
    s = {k: rng.normal(size=5) for k in FIELDS}
    s["S0"][2] = 0.0
    R = api.hbt_radii(s)
    i = 0
    assert np.isclose(R["outlong"][i], s["Sol"][i] / s["S0"][i] - s["So"][i] * s["Sl"][i] / s["S0"][i] ** 2, rtol=1e-14)
    assert all(R[k][2] == 0.0 for k in RADII)


def test_hbt_key_refused_outside_its_scope(fx):
    lib = api.lib()
    with tempfile.TemporaryDirectory() as wd:
        out = os.path.join(wd, "x.bin").encode()
        for bad in (dict(operation=0, mode=1, df_mode=1), dict(operation=1, mode=2, df_mode=1), dict(operation=1, mode=1, df_mode=3),
                    dict(operation=1, mode=1, df_mode=4)):
            workdir.materialize(wd, fixture=fx, hbt_radii=1, **bad)
            assert lib.is3d_b200_host_dump(wd.encode(), out) == 2, bad          # IS3D_ERR_UNSUPPORTED
        for ok in (dict(hbt_radii=1), dict(hbt_radii=0), {}):
            workdir.materialize(wd, fixture=fx, operation=1, mode=1, df_mode=2, **ok)
            assert lib.is3d_b200_host_dump(wd.encode(), out) == 0, ok


def test_struct_layout_matches_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "is3d_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu\\n", sizeof(is3d_hbt_result), offsetof(is3d_hbt_result, Sl),'
                   ' offsetof(is3d_hbt_result, Sos), offsetof(is3d_hbt_result, Ssl)); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got == [C.sizeof(api.HbtResult), api.HbtResult.Sl.offset, api.HbtResult.Sos.offset, api.HbtResult.Ssl.offset]
    assert [f for f, _ in api.HbtResult._fields_] == list(FIELDS)


# ------------------------------------------------------------------------------------------------ GPU
def _gpu():
    import torch
    torch.cuda.set_device(0)
    api.init()
    return torch


@pytest.mark.gpu
@pytest.mark.parametrize("dimension,df_mode,deltaf,outflow,chosen,memory", [
    (3, 1, 1, 1, "chosen_pikp", "host"), (3, 2, 1, 0, "chosen_pikp", "device"), (3, 1, 0, 0, "chosen_pikp", "host"),
    (3, 2, 0, 1, "chosen_pikp", "device"), (2, 1, 1, 1, "chosen_pikp", "host"), (2, 2, 1, 0, "chosen_pikp", "device"),
    (2, 2, 0, 1, "chosen_pikp", "host"), (2, 1, 0, 0, "chosen_pikp", "device"), (3, 1, 1, 1, "chosen_urqmd", "host")])
def test_gpu_parity(fx, dimension, df_mode, deltaf, outflow, chosen, memory):
    """Fermions and bosons (pi/K/p; the 305-species list), 3+1D and 2+1D, both linear delta-f models with delta-f on and off, outflow on
    and off, cells with u.dsigma <= 0, host and device memory: all ten arrays against the oracle at 1e-10 per bin."""
    torch = _gpu()
    n = 30 if chosen == "chosen_urqmd" else 120
    cells = _cells(n, 900 + 10 * dimension + df_mode + 3 * deltaf + 7 * outflow, dimension, flip=5)
    sp = tables.species(fx, 1, chosen); g = tables.grid(fx); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=df_mode, dimension=dimension, include_bulk=deltaf, include_shear=deltaf, outflow=outflow)
    ref, skipped, cond = cf_hbt.hbt_moments(fl, cells, sp, g, tab, conditioning=True)
    if memory == "device":
        dc = {k: torch.tensor(v, device="cuda") for k, v in cells.items()}
        out, st = api.hbt_moments(fl, dc, sp, g, tab, memory="device")
        torch.cuda.synchronize()
        got = {k: v.cpu().numpy() for k, v in out.items()}
    else:
        got, st = api.hbt_moments(fl, cells, sp, g, tab)
    assert skipped == 5 and st["cells_skipped_udsigma"] == 5
    bad = {}
    for k in FIELDS:
        if dimension == 2 and k in ("Sl", "Sol", "Ssl"):
            # odd in eta on the (numerically) symmetric eta table: the exact value is ~0 and both sides are the rounding noise of
            # ~3e4 cancelling terms summed in different orders -- the bar of test_2d_long_odd_sums_vanish
            if not np.all(np.abs(got[k] - ref[k]) <= 1e-12 * cond[k]):
                bad[k] = float(np.max(np.abs(got[k] - ref[k]) / np.maximum(cond[k], 1e-300)))
            continue
        rep = compare(got[k], ref[k], conditioning=cond[k])
        if not rep["ok"]:
            bad[k] = rep
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("dimension", [3, 2])
def test_gpu_s0_equals_spectra_reproducible_and_multi(fx, dimension):
    _gpu()
    cells = _cells(300, 555 + dimension, dimension, flip=2)
    sp = tables.species(fx, 1, "chosen_pikp"); g = tables.grid(fx); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=dimension)
    a, _ = api.hbt_moments(fl, cells, sp, g, tab)
    b, _ = api.hbt_moments(fl, cells, sp, g, tab)
    for k in FIELDS:
        assert np.array_equal(a[k], b[k]), k
    dN, _ = api.smooth_spectra(fl, cells, sp, g, tab)
    cond = np.zeros_like(dN)
    cfo.smooth(fl, cells, sp, g, tab, conditioning=cond)
    rep = compare(a["S0"], dN, conditioning=cond)
    assert rep["ok"], rep
    api.init_devices(0)
    m, _ = api.hbt_moments(fl, cells, sp, g, tab, multi=True)
    for k in FIELDS:
        scale = np.abs(a[k]).max()
        assert np.abs(m[k] - a[k]).max() <= 1e-13 * scale, k


@pytest.mark.gpu
def test_gpu_empty_surface_and_errors(fx):
    _gpu()
    sp = tables.species(fx, 1, "chosen_pikp"); g = tables.grid(fx); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=3)
    out, st = api.hbt_moments(fl, _cells(0, 1, 3), sp, g, tab)
    assert all(np.all(v == 0) for v in out.values()) and st["cells_skipped_udsigma"] == 0
    cells = _cells(10, 2, 3)
    for bad in (dict(fl, df_mode=3), dict(fl, df_mode=4), dict(fl, mode=2), dict(fl, include_baryon=1)):
        with pytest.raises(api.Is3dError) as e:
            api.hbt_moments(bad, cells, sp, g, tab)
        assert e.value.code == 2, bad
    for k in ("x", "y"):
        with pytest.raises(api.Is3dError) as e:
            api.hbt_moments(fl, {c: v for c, v in cells.items() if c != k}, sp, g, tab)
        assert e.value.code == 1, k


def _read_hbt(path):
    return np.loadtxt(path, skiprows=1, ndmin=2)


@pytest.mark.gpu
@pytest.mark.parametrize("dimension,df_mode", [(3, 1), (2, 2)])
def test_gpu_workdir_hbt_files(fx, dimension, df_mode):
    _gpu()
    cols = synthetic.surface_vh(60, 4321 + dimension, three_d=(dimension == 3))
    chosen = [211, 321, 2212]
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=cols, chosen=chosen, fixture=fx, operation=1, mode=1, dimension=dimension, df_mode=df_mode,
                            hbt_radii=1)
        lib = api.lib()
        lib.is3d_b200_host_error.restype = C.c_char_p
        rc = lib.is3d_b200_run_workdir(wd.encode(), None, C.c_int64(0), None, 0, None)
        assert rc == 0, lib.is3d_b200_host_error().decode()
        files = {c: _read_hbt(os.path.join(wd, "results", "hbt", "R2_%d.dat" % c)) for c in chosen}
        header = open(os.path.join(wd, "results", "hbt", "R2_211.dat")).readline().split()
    assert header == ["y", "phip", "pT", "S0", "R2_out", "R2_side", "R2_long", "R2_outside", "R2_outlong", "R2_sidelong"]
    cells = synthetic.columns_to_cells(cols, 1)
    sp = tables.species(fx, 1, chosen); g = tables.grid(fx); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=df_mode, dimension=dimension)
    api.init_devices(0)
    sums, _ = api.hbt_moments(fl, cells, sp, g, tab, multi=True)
    R = api.hbt_radii(sums)
    ny = 1 if dimension == 2 else len(g["y"])
    shape = (len(g["y"]), len(g["phi"]), len(g["pT"]), -1)
    for s, c in enumerate(chosen):
        want = np.column_stack([sums["S0"].reshape(shape)[:ny, :, :, s].ravel()] + [R[k].reshape(shape)[:ny, :, :, s].ravel() for k in RADII])
        got = files[c][:, 3:]
        assert got.shape == want.shape
        scale = np.abs(want).max(axis=0)
        assert np.all(np.abs(got - want) <= 1e-8 * np.abs(want) + 1e-12 * scale), c


@pytest.mark.gpu
def test_gpu_workdir_without_the_key_is_unchanged(fx):
    """Without hbt_radii the run writes the files it always wrote, and no HBT file."""
    _gpu()
    cols = synthetic.surface_vh(20, 99)
    listing, contents = [], []
    for extra in ({}, dict(hbt_radii=0)):
        with tempfile.TemporaryDirectory() as wd:
            workdir.materialize(wd, surface_columns=cols, fixture=fx, operation=1, mode=1, dimension=3, df_mode=1, **extra)
            assert api.lib().is3d_b200_run_workdir(wd.encode(), None, C.c_int64(0), None, 0, None) == 0
            res = os.path.join(wd, "results")
            names = sorted(os.path.relpath(os.path.join(d, f), res) for d, _, fs in os.walk(res) for f in fs)
            listing.append(names)
            contents.append({p: open(os.path.join(res, p), "rb").read() for p in names})
    assert listing[0] == listing[1]
    assert contents[0] == contents[1]
    assert not any(p.startswith("hbt" + os.sep) for p in listing[0])
    assert "dN_pTdpTdphidy.dat" in listing[0]
