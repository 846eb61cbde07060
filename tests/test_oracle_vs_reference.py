"""Live check of the oracle against the compiled reference (oracle/_ref), where that binary exists."""
import tempfile

import numpy as np
import pytest

from common import jonah_tables
from is3d_b200 import synthetic, tables, workdir
from oracle import cf_oracle as cfo

pytestmark = pytest.mark.skipif(cfo.ref_binary() is None, reason="oracle/_ref not built (needs IS3D_REFERENCE, see oracle/Makefile)")


@pytest.mark.parametrize("dimension,df_mode,n_cells,stress", [(3, 1, 24, False), (3, 3, 24, True), (3, 4, 24, False), (2, 2, 6, False)])
def test_reference_binary_agrees(fx, dimension, df_mode, n_cells, stress):
    cols = synthetic.surface_vh(n_cells, 4242 + df_mode, three_d=(dimension == 3), stress=stress)
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=cols, chosen="chosen_pikp", fixture=fx, operation=1, mode=1, hrg_eos=1,
                            dimension=dimension, df_mode=df_mode)
        ref, info = cfo.run_reference(wd)
    cells = synthetic.columns_to_cells(cols, 1)
    sp = tables.species(fx, 1, "chosen_pikp"); g = tables.grid(fx); tab = tables.df_tables(fx, 1); gla = tables.laguerre(fx)
    if df_mode == 4:
        tab.update(jonah_tables(cells, fx, 1, gla))
    dN, skipped, bd = cfo.smooth(tables.flags(df_mode=df_mode, dimension=dimension), cells, sp, g, tab, gla)
    assert list(sp["mcid"]) == info["mcid"]
    assert bd == info["breakdown"]
    assert np.array_equal(dN, ref)
