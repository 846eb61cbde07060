"""Resonance-decay feed-down (SURVEY 8f, row N3): EmissionFunctionArray::do_resonance_decays, emissionfunction_resonance_decays.cpp.

The reference snapshot disables the routine with an exit(-1) at entry (:126-129); the golden vectors come from the routine's body run
behind oracle/ref_decays_prefix.h (tests/golden/make_decay_vectors.py).  CPU tier: the C oracle is bit-identical to those vectors
(and to the reference binary where it exists) and the host layer's particle list matches the test-side restatement.  GPU tier: the
CUDA path through the C ABI against the oracle / the vectors at 1e-10, and the file interface with do_resonance_decays = 1."""
import ctypes as C
import hashlib
import json
import os
import sys
import tempfile

import numpy as np
import pytest

from common import GOLDEN_DIR
from is3d_b200 import api, synthetic, tables, workdir
from oracle import cf_oracle as cfo

sys.path.insert(0, GOLDEN_DIR)
import make_decay_vectors as mdv      # noqa: E402  (recipes + input builder shared with the generator)

REL_TOL = 1e-10


def _load(name):
    z = np.load(os.path.join(GOLDEN_DIR, "decays_%s.npz" % name))
    return json.loads(str(z["recipe"])), z["dN_in"], z["dN_out"], json.loads(str(z["file_sha256"])), z["mcid"]


def _full(arr, g, ns):
    out = np.zeros(ns * len(g["pT"]) * len(g["phi"]) * len(g["y"]))
    out[:arr.size] = arr
    return out


@pytest.mark.parametrize("name", ["2d", "3d", "3d_full"])
def test_oracle_matches_reference_vectors(fx, name):
    rec, dN_in, dN_out, _, mcid = _load(name)
    g, tabs, cols, dN, pdg, chosen_idx = mdv.case_inputs(fx, rec)
    assert list(mcid) == rec["chosen"]
    plane = dN_in.size
    assert np.array_equal(dN[:plane], dN_in)                              # the thermal input is reproducible from the recipe
    got = cfo.resonance_decays(pdg, chosen_idx, g, rec["dimension"], dN)
    assert np.array_equal(got[:plane], dN_out)                            # bit-identical to the reference routine
    assert np.array_equal(got[plane:], dN[plane:])
    assert (dN_out != dN_in).sum() > 0.3 * plane


def test_oracle_against_live_reference(fx):
    if not os.path.exists(os.path.join(os.path.dirname(cfo.__file__), "_ref", "is3d_ref_decays")):
        pytest.skip("oracle/_ref/is3d_ref_decays not built here")
    rec = dict(dimension=2, n_cells=25, seed=5, strides=dict(pT=2, phi=2, y=1), chosen=[211, -211, 111, 321, 2212, -2212, 113, 223, 2224, -2224, 3122, -3122, 3224, -3224])
    g, tabs, cols, dN, pdg, chosen_idx = mdv.case_inputs(fx, rec)
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=cols, chosen=rec["chosen"], fixture=fx, tables=tabs, operation=1, mode=1, hrg_eos=1, dimension=2,
                            df_mode=1, do_resonance_decays=1)
        ref, info = cfo.run_reference_decays(wd, dN)
    assert np.array_equal(cfo.resonance_decays(pdg, chosen_idx, g, 2, dN), ref)


def test_host_layer_particle_list_has_the_decay_tables(fx):
    """csrc/host_io.cpp read_pdg: stable flags, channels and the anti-baryon daughter rule against tables.pdg_decay_table (which the
    bit-identical oracle-vs-reference runs above pin, anti-baryon parents included)"""
    from test_host_layer import host_dump
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, fixture=fx, operation=1, mode=1, hrg_eos=1, dimension=3, df_mode=1)
        rows = host_dump(wd)
    pdg = tables.pdg_decay_table(fx, 1)
    assert np.array_equal(rows["pdg_mcid"].astype(int), pdg["mcid"])
    assert np.array_equal(rows["pdg_stable"].astype(int), pdg["stable"])
    assert np.array_equal(rows["pdg_decays"].astype(int), pdg["decays"])
    assert np.array_equal(rows["pdg_dec_npart"].astype(int), pdg["dec_npart"])
    assert np.array_equal(rows["pdg_dec_part"].astype(int), np.asarray(pdg["dec_part"]).ravel())
    assert np.array_equal(rows["pdg_dec_br"], pdg["dec_br"])
    assert (pdg["mcid"] < 0).sum() > 100 and (pdg["stable"] == 0).sum() > 200


# ---------------------------------------------------------------------------------------------------------------- GPU tier
def _compare(got, ref):
    nz = ref != 0
    rel = np.abs(got[nz] - ref[nz]) / np.abs(ref[nz])
    return float(rel.max()) if rel.size else 0.0, bool(np.all(got[~nz] == 0)), int(np.isnan(got).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["2d", "3d", "3d_full"])
def test_cuda_decays_match_reference_vectors(fx, name):
    rec, dN_in, dN_out, _, _ = _load(name)
    g, tabs, cols, dN, pdg, chosen_idx = mdv.case_inputs(fx, rec)
    api.init()
    got, st = api.resonance_decays(pdg, chosen_idx, g, rec["dimension"], dN)
    plane = dN_in.size
    max_rel, zeros, nans = _compare(got[:plane], dN_out)
    print(name, "max rel %.3e" % max_rel, "kernel ms %.2f" % st["kernel_ms"], "launches", st["gpu_launches"])
    assert nans == 0 and zeros and max_rel <= REL_TOL, (name, max_rel)
    assert np.array_equal(got[plane:], dN[plane:])
    assert st["gpu_launches"] > 10
    # device-memory path: amended in place, identical numbers
    import torch
    t = torch.tensor(dN, device="cuda")
    api.resonance_decays(pdg, chosen_idx, g, rec["dimension"], t, memory="device")
    torch.cuda.synchronize()
    assert np.array_equal(t.cpu().numpy(), got)


@pytest.mark.gpu
def test_cuda_decays_long_species_lists_against_oracle(fx):
    """the first 150 (2+1D) / 70 (3+1D) species of the 305-species list on reduced momentum grids: ~600 channels incl. anti-baryon
    parents, mass-shifted 2-body channels and 3-body channels.  With these lists the reference's arithmetic makes the nucleon bins NaN
    (a channel whose daughter energy in the parent frame falls below its mass: sqrt of a negative number, :415-416) -- same bins
    here; with the whole list the reference then stops in its large-mT fit ("not enough points"), as does this library (error code)."""
    api.init()
    full = [int(v) for v in fx["chosen_urqmd"]]
    hi_pT = list(range(0, 22, 3)) + list(range(22, 32))            # every parent needs >= 2 points beyond mT = 1.65 M for its tail fit
    for dim, strides, k in ((2, dict(pT=hi_pT, phi=3, y=1), 150), (3, dict(pT=hi_pT, phi=4, y=[7, 9, 10, 11, 13]), 70)):
        rec = dict(dimension=dim, n_cells=30, seed=11, strides=strides, chosen=full[:k])
        g, tabs, cols, dN, pdg, chosen_idx = mdv.case_inputs(fx, rec)
        ref = cfo.resonance_decays(pdg, chosen_idx, g, dim, dN)
        got, st = api.resonance_decays(pdg, chosen_idx, g, dim, dN)
        assert np.array_equal(np.isnan(got), np.isnan(ref))
        fin = ~np.isnan(ref)
        max_rel, zeros, _ = _compare(got[fin], ref[fin])
        print("dim", dim, "species", k, "max rel %.3e" % max_rel, "NaN bins", int((~fin).sum()), "kernel ms %.1f" % st["kernel_ms"])
        assert zeros and max_rel <= REL_TOL, (dim, max_rel)
    # the whole list: the reference exits in estimate_MT_function_of_dNdypTdpTdphi (:2078-2082); here an error code
    rec = dict(dimension=2, n_cells=30, seed=11, strides=dict(pT=hi_pT, phi=3, y=1), chosen=full)
    g, tabs, cols, dN, pdg, chosen_idx = mdv.case_inputs(fx, rec)
    with pytest.raises(api.Is3dError) as e:
        api.resonance_decays(pdg, chosen_idx, g, 2, dN)
    assert e.value.code == 1


@pytest.mark.gpu
def test_run_workdir_with_resonance_decays(fx):
    """file interface: do_resonance_decays = 1 runs spectra + feed-down and writes the two amended-spectra files of the reference"""
    rec, dN_in, dN_out, sha, mcid = _load("3d")
    g, tabs, cols, dN, pdg, chosen_idx = mdv.case_inputs(fx, rec)
    lib = api.lib()
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=cols, chosen=rec["chosen"], fixture=fx, tables=tabs, operation=1, mode=1, hrg_eos=1, dimension=3,
                            df_mode=1, do_resonance_decays=1)
        raw = np.zeros(dN.size); ids = np.zeros(64, dtype=np.int32); st = api.Stats()
        rc = lib.is3d_b200_run_workdir(wd.encode(), raw.ctypes.data_as(C.POINTER(C.c_double)), C.c_int64(raw.size),
                                       ids.ctypes.data_as(C.POINTER(C.c_int32)), 64, C.byref(st))
        assert rc == 0, api.lib().is3d_b200_host_error()
        assert list(ids[:len(rec["chosen"])]) == rec["chosen"]
        # the GPU spectra differ from the oracle's thermal input at the 1e-12 level, the feed-down keeps that
        max_rel, zeros, nans = _compare(raw[:dN_out.size], dN_out)
        assert nans == 0 and max_rel <= REL_TOL, max_rel
        for rel_path in sha:
            text = open(os.path.join(wd, rel_path)).read().split("\n")
            assert len(text) > dN_out.size
        # same layout as the reference's file: header of the dN_dpT file, y phi pT value rows, value = dN * pT
        rows = np.loadtxt(os.path.join(wd, "results", "dN_dpTdphidy_resonance_decays.dat"), skiprows=1)
        rows2 = np.loadtxt(os.path.join(wd, "results", "dN_pTdpTdphidy_resonance_decays.dat"))
        assert rows.shape == rows2.shape == (dN_out.size, 4)
        assert np.allclose(rows[:, 3], rows2[:, 3] * rows2[:, 2], rtol=1e-7, atol=0)
        ns = len(rec["chosen"])
        ref_first = dN_out.reshape(len(g["y"]), len(g["phi"]), len(g["pT"]), ns)[:, :, :, 0].ravel()
        assert np.allclose(rows2[:ref_first.size, 3], ref_first, rtol=2e-8, atol=0)
