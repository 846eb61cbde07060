"""bench.py --dump-outputs: the arrays of the last timed step, written as float64 .npy files so that two builds can be compared."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from common import compare

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, "bench.py", "--steps", "0"], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and "--steps must be >= 1" in r.stderr


def test_dump_outputs_writes_float64_and_refuses_more_than_64_mb(tmp_path):
    import bench
    bench.dump_outputs(str(tmp_path / "d"), {"a": np.arange(6, dtype=np.float32).reshape(2, 3)})
    a = np.load(tmp_path / "d" / "a.npy")
    assert a.dtype == np.float64 and a.shape == (2, 3) and np.array_equal(a, np.arange(6).reshape(2, 3))
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "big"), {"a": np.zeros(bench.DUMP_LIMIT_BYTES // 8 + 1)})
    assert not os.path.exists(tmp_path / "big")


def _bench(out_dir, *extra):
    cmd = [sys.executable, "bench.py", "--steps", "2", "--warmup", "1", "--cells", "3000", "--no-cpu-baseline", "--no-e2e",
           "--dump-outputs", str(out_dir)] + list(extra)
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout)


@pytest.mark.gpu
def test_dumped_spectra_are_what_the_library_computes(fx, tmp_path):
    """default workload (cfg3 model and species list) on a 3000-cell prefix: the dump equals a direct call on the same seeded surface"""
    from is3d_b200 import api, synthetic, tables
    line = _bench(tmp_path / "op1")
    dN = np.load(tmp_path / "op1" / "dN.npy")
    assert sorted(os.listdir(tmp_path / "op1")) == ["dN.npy"] and dN.dtype == np.float64
    assert abs(dN.sum() - line["config"]["spectra_checksum"]) <= 1e-12 * abs(dN.sum())
    api.init()
    sp = tables.species(fx, 1, "chosen_urqmd"); g = tables.grid(fx); tab = tables.df_tables(fx, 1); gla = tables.laguerre(fx)
    cells = synthetic.columns_to_cells(synthetic.surface_vh(3000, synthetic.SEEDS["cfg3"], three_d=True, viscous=True), 1)
    ref, _ = api.smooth_spectra(tables.flags(df_mode=1, dimension=3, include_bulk=1, include_shear=1), cells, sp, g, tab, gla)
    assert dN.shape == ref.shape and compare(dN, ref, tol=1e-12)["ok"]


@pytest.mark.gpu
def test_dumped_spacetime_histograms(fx, tmp_path):
    from is3d_b200 import api, synthetic, tables
    import bench
    line = _bench(tmp_path / "op0", "--operation", "0")
    got = {k: np.load(tmp_path / "op0" / (k + ".npy")) for k in ("dN_tau", "dN_r", "dN_taur", "dN_dydeta", "dN_dy")}
    assert len(os.listdir(tmp_path / "op0")) == 5
    api.init()
    sp = tables.species(fx, 1, "chosen_urqmd"); g = tables.grid(fx); tab = tables.df_tables(fx, 1); gla = tables.laguerre(fx)
    cells = synthetic.columns_to_cells(synthetic.surface_vh(3000, synthetic.SEEDS["cfg3"], three_d=True, viscous=True), 1)
    ref, _ = api.spacetime_distributions(tables.flags(df_mode=1, dimension=3, include_bulk=1, include_shear=1), cells, sp, g, tab, gla,
                                         bench.SPACETIME_BINS)
    for k, v in ref.items():
        assert got[k].shape == v.shape, k
        assert np.abs(got[k] - v).max() <= 1e-12 * np.abs(v).max(), k
    assert abs(got["dN_dy"].sum() - line["config"]["spectra_checksum"]) <= 1e-12 * abs(got["dN_dy"].sum())
