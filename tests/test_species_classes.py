"""The shifted-factor kernel (cf_shift.cu) runs one lane per class of species with bit-equal (mass, sign) and stores the class's
result for every member species, scaled by that species' degeneracy. Species of one class must come out exactly as they would
on lanes of their own, species that differ in any bit of mass or sign must stay apart, and the spectra must match cf_kernel,
which has no classes, bin by bin with the same zero pattern. At 32 pT points a warp holds one class, so a species' spectra do
not depend on which other species share the run (at the same cell chunks: the chunk count follows the number of lane blocks
and the chunk sums are added in that grouping); at 24 and 40 points a warp straddles two classes."""
import numpy as np
import pytest

from common import compare
from is3d_b200 import api, synthetic, tables

CF_KERNEL = 10            # tile_variant of cf_kernel's 3+1D default shape for the linear-df models


def _species_slice(dN, n_species, i):
    return dN.reshape(-1, n_species)[:, i]


def _subset(sp, idx):
    return {k: np.ascontiguousarray(v[idx]) for k, v in sp.items()}


def _cells(n):
    return synthetic.columns_to_cells(synthetic.surface_vh(n, synthetic.SEEDS["cfg3"], three_d=True, viscous=True), 1)


@pytest.mark.gpu
@pytest.mark.parametrize("df_mode", [1, 2])
def test_urqmd_list_species_alone(fx, df_mode):
    api.init()
    sp = tables.species(fx, 1, "chosen_urqmd"); g = tables.grid(fx); tab = tables.df_tables(fx, 1)
    assert len(g["pT"]) == 32
    fl = tables.flags(df_mode=df_mode, dimension=3)
    cells = _cells(20_000)
    got, st = api.smooth_spectra(fl, cells, sp, g, tab, None)
    assert st["tile_variant"] == 22                                  # default: cf_shift_kernel
    ref, _ = api.smooth_spectra(fl, cells, sp, g, tab, None, tile_variant=CF_KERNEL)
    rep = compare(got, ref)
    assert rep["ok"], rep
    assert np.array_equal(got == 0, ref == 0)
    mcid = list(sp["mcid"])
    picks = {"pi+": mcid.index(211), "member of the 14-species class": mcid.index(12214), "antiproton": mcid.index(-2212),
             "eta (a class of its own)": mcid.index(221)}
    n = len(mcid)
    for name, i in picks.items():
        alone, _ = api.smooth_spectra(fl, cells, _subset(sp, [i]), g, tab, None, n_chunks=st["n_chunks"])
        assert np.array_equal(_species_slice(got, n, i), alone), name


def _crafted(sp_pi):
    """pi+, the same mass as a fermion, one ulp heavier, an exact duplicate, and a duplicate with degeneracy 3"""
    m = float(sp_pi["mass"][0])
    mass = np.array([m, m, np.nextafter(m, np.inf), m, m])
    sign = np.array([-1.0, 1.0, -1.0, -1.0, -1.0])
    deg = np.array([1.0, 1.0, 1.0, 1.0, 3.0])
    return dict(mcid=np.array([211, 211, 211, 211, 211]), mass=mass, sign=sign, degeneracy=deg, baryon=np.zeros(5))


@pytest.mark.gpu
def test_crafted_list(fx):
    api.init()
    sp = _crafted(tables.species(fx, 1, [211])); g = tables.grid(fx); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=3)
    cells = _cells(5_000)
    got, st = api.smooth_spectra(fl, cells, sp, g, tab, None)
    ref, _ = api.smooth_spectra(fl, cells, sp, g, tab, None, tile_variant=CF_KERNEL)
    for i in range(5):
        rep = compare(_species_slice(got, 5, i), _species_slice(ref, 5, i))
        assert rep["ok"], (i, rep)
        assert np.array_equal(_species_slice(got, 5, i) == 0, _species_slice(ref, 5, i) == 0), i
    assert np.array_equal(_species_slice(got, 5, 0), _species_slice(got, 5, 3))       # equal (mass, sign, g): bit for bit
    # opposite sign and the heavier mass are classes of their own: each is what it is alone, and differs from pi+
    for i in (1, 2):
        alone, _ = api.smooth_spectra(fl, cells, _subset(sp, [i]), g, tab, None, n_chunks=st["n_chunks"])
        assert np.array_equal(_species_slice(got, 5, i), alone), i
        assert not np.array_equal(_species_slice(got, 5, i), _species_slice(got, 5, 0)), i


@pytest.mark.gpu
@pytest.mark.parametrize("n_pT", [24, 40])
def test_class_boundaries_inside_a_warp(fx, n_pT):
    api.init()
    sp = tables.species(fx, 1, "chosen_urqmd"); tab = tables.df_tables(fx, 1)
    g = dict(tables.grid(fx))
    g["pT"] = np.linspace(0.01, 3.0, n_pT); g["pT_weight"] = np.full(n_pT, 3.0 / n_pT)
    fl = tables.flags(df_mode=1, dimension=3)
    cells = _cells(5_000)
    got, _ = api.smooth_spectra(fl, cells, sp, g, tab, None)
    ref, _ = api.smooth_spectra(fl, cells, sp, g, tab, None, tile_variant=CF_KERNEL)
    rep = compare(got, ref)
    assert rep["ok"], rep
    assert np.array_equal(got == 0, ref == 0)
