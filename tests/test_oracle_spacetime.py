"""operation = 0 oracle (oracle/cf_oracle.c: cfo_spacetime_vh, cfo_spacetime_feqmod) against the reference's output files:
the committed vectors under tests/golden/spacetime_*.npz and, where oracle/_ref exists, a live run."""
import tempfile

import numpy as np
import pytest

from common import jonah_tables, load_spacetime, spacetime_close, spacetime_names, spacetime_problem
from is3d_b200 import synthetic, tables, workdir
from oracle import cf_oracle as cfo


@pytest.mark.parametrize("name", spacetime_names())
def test_oracle_matches_reference_files(name, fx):
    gold = load_spacetime(name)
    fl, cells, sp, g, tab, gla, bins, _ = spacetime_problem(gold["recipe"], fx)
    out, skipped = cfo.spacetime(fl, cells, sp, g, tab, bins, gla)
    assert skipped == 0
    assert list(sp["mcid"]) == list(gold["mcid"])
    spacetime_close(out, gold)
    if "stress_df3" in name:
        assert out["breakdown"] > 0


def test_histograms_are_consistent(fx):
    """size-independent properties: every histogram is a partial sum of the per-cell yields"""
    gold = load_spacetime("dx3_df1")
    fl, cells, sp, g, tab, gla, bins, _ = spacetime_problem(gold["recipe"], fx)
    wide = dict(tau_min=0.0, tau_max=50.0, tau_bins=7, r_min=0.0, r_max=50.0, r_bins=5)      # every cell inside
    out, _ = cfo.spacetime(fl, cells, sp, g, tab, wide, gla)
    np.testing.assert_allclose(out["dN_tau"].sum(axis=1), out["dN_dy"], rtol=1e-13)
    np.testing.assert_allclose(out["dN_r"].sum(axis=1), out["dN_dy"], rtol=1e-13)
    np.testing.assert_allclose(out["dN_taur"].sum(axis=2), out["dN_tau"], rtol=1e-13, atol=1e-300)
    np.testing.assert_allclose(out["dN_taur"].sum(axis=1), out["dN_r"], rtol=1e-13, atol=1e-300)
    np.testing.assert_allclose(out["dN_dydeta"][:, 0], out["dN_dy"], rtol=1e-11)     # one long running sum vs per-cell sums
    # the momentum-integrated yield equals the y-summed, quadrature-weighted spectra of operation = 1
    dN, _, _ = cfo.smooth(fl, cells, sp, g, tab, gla)
    spec = dN.reshape(len(g["y"]), len(g["phi"]), len(g["pT"]), len(sp["mass"]))
    yields = np.einsum("yfps,f,p->s", spec, g["phi_weight"], g["pT_weight"])
    np.testing.assert_allclose(yields, out["dN_dy"], rtol=1e-12)


@pytest.mark.skipif(cfo.ref_binary() is None, reason="oracle/_ref not built (needs IS3D_REFERENCE, see oracle/Makefile)")
@pytest.mark.parametrize("dimension,df_mode,n_cells,stress", [(3, 2, 30, False), (3, 3, 30, True), (2, 4, 8, False)])
def test_reference_binary_agrees(fx, dimension, df_mode, n_cells, stress):
    bins = dict(tau_min=1.0, tau_max=10.0, tau_bins=9, r_min=2.0, r_max=11.0, r_bins=3)      # cells fall outside on both sides
    cols = synthetic.surface_vh(n_cells, 5151 + df_mode, three_d=(dimension == 3), stress=stress)
    sp = tables.species(fx, 1, "chosen_pikp"); g = tables.grid(fx)
    eta_pts = len(g["eta"]) if dimension == 2 else 1
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=cols, chosen="chosen_pikp", fixture=fx, operation=0, mode=1, hrg_eos=1,
                            dimension=dimension, df_mode=df_mode, **bins)
        _, info = cfo.run_reference(wd, what="full")
        per = [cfo.read_spacetime_files(wd, int(m), bins, eta_pts) for m in sp["mcid"]]
        printed = [float(l.split("=")[1]) for l in info["stdout"].splitlines() if l.startswith("dN_dy =")]
    cells = synthetic.columns_to_cells(cols, 1)
    tab = tables.df_tables(fx, 1); gla = tables.laguerre(fx)
    if df_mode == 4:
        tab.update(jonah_tables(cells, fx, 1, gla))
    out, _ = cfo.spacetime(tables.flags(df_mode=df_mode, dimension=dimension), cells, sp, g, tab, bins, gla)
    gold = {k: np.stack([p[k] for p in per]) for k in ("dN_tau", "dN_r", "dN_taur", "dN_dydeta")}
    gold["dN_dy_printed"] = np.array(printed)
    spacetime_close(out, gold)
    if dimension == 3:
        assert abs(per[0]["eta_column"][0] - cells["eta"][-1]) <= 1e-6 * abs(cells["eta"][-1])     # the last cell's eta (:1154)
