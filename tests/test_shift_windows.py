"""The e^{-pT (Bmax - B_k)} table of the shifted-factor kernel (cf_shift.cu) is formed for a window of consecutive cell chunks at
a time, within 4 GiB. With 64 pT points and 240 phi points it takes ~120 KB per cell, so 70 000 cells run as three windows
(the full-size cfg3 surface runs as two): the spectra must match cf_kernel, which has no table, bin by bin with the same zero
pattern. On this grid the 3 x 6 stage does not fit 16-cell tiles at 3 blocks/SM, so the 8-cell tile runs as well."""
import numpy as np
import pytest

from common import compare
from is3d_b200 import api, synthetic, tables

CF_KERNEL = 10            # tile_variant of cf_kernel's 3+1D default shape for the linear-df models


def _grid(fx):
    g = dict(tables.grid(fx))
    n_pT, n_phi = 64, 240
    g["pT"] = np.linspace(0.01, 3.0, n_pT); g["pT_weight"] = np.full(n_pT, 3.0 / n_pT)
    g["phi"] = (np.arange(n_phi) + 0.5) * (2.0 * np.pi / n_phi); g["phi_weight"] = np.full(n_phi, 2.0 * np.pi / n_phi)
    return g


@pytest.mark.gpu
def test_several_table_windows(fx):
    api.init()
    g = _grid(fx)
    sp = tables.species(fx, 1, [211]); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=3)
    _, st_one = api.smooth_spectra(fl, synthetic.columns_to_cells(synthetic.surface_vh(2000, 4245), 1), sp, g, tab, None)
    cells = synthetic.columns_to_cells(synthetic.surface_vh(70_000, 4245), 1)
    got, st = api.smooth_spectra(fl, cells, sp, g, tab, None)
    assert st["tile_variant"] == 22                                  # default: cf_shift_kernel 3 x 6
    # one window at 2000 cells; every further window adds a table kernel and a hot kernel
    assert st["gpu_launches"] >= st_one["gpu_launches"] + 2, (st["gpu_launches"], st_one["gpu_launches"])
    ref, _ = api.smooth_spectra(fl, cells, sp, g, tab, None, tile_variant=CF_KERNEL)
    rep = compare(got, ref)
    assert rep["ok"], rep
    assert np.array_equal(got == 0, ref == 0)
