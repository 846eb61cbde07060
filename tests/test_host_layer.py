"""C++ host layer (csrc/host_io.cpp, host_run.cpp) on the CPU: readers against the fixture / the oracle, writers against
the reference's own text output (sha256 recorded in the golden vectors)."""
import ctypes as C
import hashlib
import os
import struct
import tempfile

import numpy as np
import pytest

from common import compare, jonah_tables, load_golden, surface_columns
from is3d_b200 import api, synthetic, tables, workdir
from oracle import cf_oracle as cfo

REF = os.environ.get("IS3D_REFERENCE", "")          # an iS3D checkout, for the checks against its own files


def host_dump(wd):
    lib = api.lib()
    out = os.path.join(wd, "host_dump.bin")
    rc = lib.is3d_b200_host_dump(wd.encode(), out.encode())
    lib.is3d_b200_host_error.restype = C.c_char_p
    assert rc == 0, lib.is3d_b200_host_error().decode()
    rec = {}
    data = open(out, "rb").read()
    pos = 0
    while pos < len(data):
        (ln,) = struct.unpack_from("<i", data, pos); pos += 4
        name = data[pos:pos + ln].decode(); pos += ln
        (n,) = struct.unpack_from("<q", data, pos); pos += 8
        rec[name] = np.frombuffer(data, dtype="<f8", count=n, offset=pos).copy(); pos += 8 * n
    return rec


@pytest.mark.parametrize("eos,chosen", [(1, "chosen_urqmd"), (2, "chosen_smash"), (3, "chosen_box"), (2, "chosen_pikp")])
def test_species_bookkeeping(fx, eos, chosen):
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, chosen=chosen, fixture=fx, hrg_eos=eos, dimension=3, df_mode=1)
        d = host_dump(wd)
    pdg = tables.pdg_table(fx, eos)
    assert np.array_equal(d["pdg_mcid"], pdg["mcid"])                  # incl. synthesised anti-particles, exact order
    assert np.array_equal(d["pdg_mass"], pdg["mass"])
    assert np.array_equal(d["pdg_gspin"], pdg["gspin"])
    assert np.array_equal(d["pdg_sign"], pdg["sign"])
    assert np.array_equal(d["pdg_baryon"], pdg["baryon"])
    sp = tables.species(fx, eos, chosen)
    for k in ("mcid", "mass", "sign", "degeneracy", "baryon"):
        assert np.array_equal(d[k], sp[k]), k
    assert len(d["mcid"]) == len(fx[chosen])


def test_group_particles_sort(fx):
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, chosen="chosen_urqmd", fixture=fx, hrg_eos=1, group_particles=1)
        d = host_dump(wd)
    sp = tables.species(fx, 1, "chosen_urqmd", group_particles=True)
    assert np.array_equal(d["mcid"], sp["mcid"])
    assert np.all(np.diff(d["mass"]) >= 0)


def test_surface_reader_mode1_and_averages(fx):
    cols = synthetic.surface_vh(257, 99)
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=cols, fixture=fx, hrg_eos=1, dimension=3, df_mode=4)
        d = host_dump(wd)
        side = open(os.path.join(wd, "average_thermodynamic_quantities.dat")).read()
    cells = synthetic.columns_to_cells(cols, 1)
    for k in ("tau", "eta", "dat", "dax", "day", "dan", "ux", "uy", "un", "E", "T", "P", "pixx", "pixy", "pixn", "piyy", "piyn", "bulkPi"):
        assert np.array_equal(d[k], cells[k]), k                       # unit conversion = one multiply by hbarC, bit exact
    avg = cfo.surface_averages(cells)
    assert side == "\n".join("%.15g" % v for v in avg)
    assert np.array_equal(d["avg"], [float("%.15g" % v) for v in avg])
    # Jonah lambda/z tables are built at that (text round-tripped) average temperature
    jt = jonah_tables(cells, fx, 1, tables.laguerre(fx))
    assert np.array_equal(d["jonah_x"], jt["jonah_x"])
    assert np.array_equal(d["jonah_lambda2"], jt["jonah_lambda2"])
    assert np.array_equal(d["jonah_z"], jt["jonah_z"])
    assert d["jonah_max"][0] == jt["bulkPi_over_Peq_max"]


def test_surface_reader_mode0(fx):
    """old 26-column format: u^tau and the redundant pi components are skipped / kept, same physics columns"""
    c = synthetic.surface_vh(50, 5)
    z = np.zeros(len(c))
    ut = np.sqrt(1 + c[:, 8] ** 2 + c[:, 9] ** 2 + (c[:, 0] * c[:, 10]) ** 2)
    old = np.column_stack([c[:, :8], ut, c[:, 8:14], z, z, z, z, c[:, 14:19], z, c[:, 19]])
    assert old.shape[1] == 26
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=old, fixture=fx, hrg_eos=1, mode=0)
        d = host_dump(wd)
    cells = synthetic.columns_to_cells(c, 1)
    for k in ("tau", "ux", "un", "E", "T", "pixx", "piyn", "bulkPi"):
        assert np.array_equal(d[k], cells[k]), k


def test_row_count_rule(fx):
    """rows = newline-terminated lines (arsenal.cpp:406-453): an unterminated last line is not a cell"""
    cols = synthetic.surface_vh(10, 3)
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=cols, fixture=fx)
        p = os.path.join(wd, "input", "surface.dat")
        text = open(p).read()
        open(p, "w").write(text.rstrip("\n"))
        d = host_dump(wd)
    assert len(d["tau"]) == 9


def test_missing_parameter_is_an_error(fx):
    lib = api.lib()
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, fixture=fx)
        p = os.path.join(wd, "iS3D_parameters.dat")
        lines = [l for l in open(p) if not l.lower().startswith("r_bins")]
        open(p, "w").writelines(lines)
        assert lib.is3d_b200_host_dump(wd.encode(), os.path.join(wd, "x.bin").encode()) == 6
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, fixture=fx, chosen=[211, 999999])
        assert lib.is3d_b200_host_dump(wd.encode(), os.path.join(wd, "x.bin").encode()) == 6


def test_operation_dispatch_rules(fx):
    """what the host layer accepts: operation 1 (spectra, optionally with the resonance-decay feed-down) and 0 (spacetime
    distributions, viscous hydro only); the sampler, decays outside operation 1 or without decay tables (SMASH box list) and
    mode 2 + operation 0 are refused with IS3D_ERR_UNSUPPORTED"""
    lib = api.lib()
    lib.is3d_b200_host_error.restype = C.c_char_p

    def rc_for(**params):
        with tempfile.TemporaryDirectory() as wd:
            workdir.materialize(wd, fixture=fx, **params)
            rc = lib.is3d_b200_host_dump(wd.encode(), os.path.join(wd, "x.bin").encode())
            return rc, lib.is3d_b200_host_error().decode()

    assert rc_for(operation=1)[0] == 0
    assert rc_for(operation=0)[0] == 0
    rc, msg = rc_for(operation=2)
    assert rc == 2 and "sampler" in msg
    assert rc_for(operation=1, do_resonance_decays=1)[0] == 0
    rc, msg = rc_for(operation=0, do_resonance_decays=1)
    assert rc == 2 and "resonance" in msg
    rc, msg = rc_for(operation=1, do_resonance_decays=1, hrg_eos=3)
    assert rc == 2 and "decay tables" in msg
    rc, msg = rc_for(operation=0, mode=2)
    assert rc == 2 and "anisotropic" in msg


def test_df_tables_and_grids(fx):
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, fixture=fx, hrg_eos=2)
        d = host_dump(wd)
    tab = tables.df_tables(fx, 2); g = tables.grid(fx)
    assert np.array_equal(d["df_T"], tab["T"]) and np.array_equal(d["df_c0"], tab["c0"]) and np.array_equal(d["df_betapi"], tab["betapi"])
    assert np.array_equal(d["pT"], g["pT"]) and np.array_equal(d["phi"], g["phi"]) and np.array_equal(d["y"], g["y"])
    assert np.array_equal(d["eta_tab"], g["eta"]) and np.array_equal(d["eta_weight"], g["eta_weight"])
    gla = tables.laguerre(fx)
    assert np.array_equal(d["gla_root1"], gla["root1"]) and np.array_equal(d["gla_weight2"], gla["weight2"])


def _to_crlf(wd):
    """every parameter, particle-list, quadrature and delta-f file of a work directory rewritten with CRLF line ends"""
    paths = [os.path.join(wd, "iS3D_parameters.dat")]
    for sub in ("PDG", "tables", "deltaf_coefficients"):
        for dirpath, _, files in os.walk(os.path.join(wd, sub)):
            paths += [os.path.join(dirpath, f) for f in files]
    for p in paths:
        with open(p, "rb") as f:
            data = f.read()
        with open(p, "wb") as f:
            f.write(data.replace(b"\n", b"\r\n"))
    return len(paths)


def _check_reference_tables(d, fx):
    sp = tables.species(fx, 1, "chosen_urqmd"); tab = tables.df_tables(fx, 1)
    assert np.array_equal(d["mcid"], sp["mcid"]) and np.array_equal(d["mass"], sp["mass"]) and len(d["mcid"]) == 305
    assert np.array_equal(d["df_c0"], tab["c0"]) and np.array_equal(d["df_F"], tab["F"])
    assert np.array_equal(d["pT"], tables.grid(fx)["pT"])


def test_readers_on_the_reference_files(fx):
    """The reference ships its data files with CRLF line ends: the readers give the same values from CRLF copies of the
    re-materialised files as from the LF ones.  Where IS3D_REFERENCE names an iS3D checkout, also on the reference's own data files
    (real headers)."""
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, chosen="chosen_urqmd", fixture=fx, hrg_eos=1)
        lf = host_dump(wd)
        assert _to_crlf(wd) > 15
        crlf = host_dump(wd)
    assert lf.keys() == crlf.keys()
    for k in lf:
        assert np.array_equal(lf[k], crlf[k], equal_nan=True), k
    _check_reference_tables(crlf, fx)
    if not os.path.isdir(REF):
        return
    import shutil
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, chosen="chosen_urqmd", fixture=fx, hrg_eos=1)
        for sub in ("PDG", "tables", "deltaf_coefficients"):
            shutil.rmtree(os.path.join(wd, sub))
            shutil.copytree(os.path.join(REF, sub), os.path.join(wd, sub))
        shutil.copy(os.path.join(REF, "PDG", "chosen_particles_urqmd_v3.3+.dat"), os.path.join(wd, "PDG", "chosen_particles.dat"))
        shutil.copy(os.path.join(REF, "iS3D_parameters.dat"), os.path.join(wd, "iS3D_parameters.dat"))
        # shipped parameter file: operation 2 / mode 0 / hrg_eos 2 -> edit to the smooth path on the 20-column toy surface
        text = open(os.path.join(wd, "iS3D_parameters.dat")).read()
        import re
        for k, v in (("operation", 1), ("mode", 1), ("hrg_eos", 1), ("dimension", 3), ("df_mode", 1)):
            text = re.sub(r"(?m)^(%s\s*=\s*)\S+" % k, r"\g<1>%s" % v, text)
        open(os.path.join(wd, "iS3D_parameters.dat"), "w").write(text)
        d = host_dump(wd)
    _check_reference_tables(d, fx)


@pytest.mark.parametrize("name", ["toy_df1", "s2_df1"])
def test_writers_byte_identical(fx, name):
    """results/*.dat written from the reference's raw spectra must hash to what the reference itself wrote."""
    gold = load_golden(name)
    lib = api.lib()
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=surface_columns(gold["recipe"], fx), chosen=gold["recipe"]["chosen"], fixture=fx,
                            operation=1, mode=1, **gold["recipe"]["params"])
        dN = np.ascontiguousarray(gold["dN"])
        rc = lib.is3d_b200_write_results(wd.encode(), dN.ctypes.data_as(C.POINTER(C.c_double)), C.c_int64(dN.size))
        assert rc == 0
        for rel, digest in gold["file_sha256"].items():
            got = hashlib.sha256(open(os.path.join(wd, rel), "rb").read()).hexdigest()
            assert got == digest, rel
        # append semantics (ios_base::app): a second run concatenates
        size1 = os.path.getsize(os.path.join(wd, "results", "dN_pTdpTdphidy.dat"))
        assert lib.is3d_b200_write_results(wd.encode(), dN.ctypes.data_as(C.POINTER(C.c_double)), C.c_int64(dN.size)) == 0
        assert os.path.getsize(os.path.join(wd, "results", "dN_pTdpTdphidy.dat")) == 2 * size1


def test_table_builders_match_oracle(fx):
    """is3d_b200_surface_averages / is3d_b200_jonah_tables (C ABI helpers for direct callers) against the oracle"""
    cells = synthetic.columns_to_cells(synthetic.surface_vh(333, 12), 1)
    avg = api.surface_averages(cells)
    assert np.array_equal(avg, [float("%.15g" % v) for v in cfo.surface_averages(cells)])
    pdg = tables.pdg_table(fx, 1); gla = tables.laguerre(fx)
    mine = api.jonah_tables(pdg["mass"], pdg["gspin"].astype(float), pdg["sign"].astype(float), avg[0], gla)
    ref = cfo.jonah_tables(pdg["mass"], pdg["gspin"].astype(float), pdg["sign"].astype(float), avg[0], gla)
    for k in ("jonah_x", "jonah_lambda2", "jonah_z"):
        assert np.array_equal(mine[k], ref[k]), k
    assert mine["bulkPi_over_Peq_max"] == ref["bulkPi_over_Peq_max"]


def test_surface_reader_mode2_and_vah_coefficients(fx):
    """anisotropic-hydro surface (31 columns): alpha_L / Lambda inference and the (Lambda, alpha_L) coefficient lookup"""
    from common import vah_cells
    cols = synthetic.surface_vah(64, 1005)
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=cols, fixture=fx, hrg_eos=1, mode=2, vah=True)
        d = host_dump(wd)
    ref = vah_cells(cols, fx)
    for k in ("tau", "ux", "un", "pitt", "pitn", "pinn", "pixx", "Wx", "Wy", "bulkPi"):
        assert np.array_equal(d[k], ref[k]), k
    for k in ("aL", "Lambda", "c0", "c1", "c2", "c3", "c4"):
        assert np.allclose(d[k], ref[k], rtol=1e-12, atol=0), k


def _alt_format_columns(mode, base):
    """Re-express a mode-1 (20 column) surface in the column layout of another reader (values chosen so that both describe
    the same physical cells where the formats allow it)."""
    hb = synthetic.HBARC
    tau = base[:, 0]
    z = np.zeros(len(base))
    ut = np.sqrt(1 + base[:, 8] ** 2 + base[:, 9] ** 2 + (tau * base[:, 10]) ** 2)
    E, T, P = base[:, 11], base[:, 12], base[:, 13]
    pixx, pixy, pixn, piyy, piyn, bulk = (base[:, k] for k in range(14, 20))
    if mode in (4, 6):
        s = (E + P) / T                                   # entropy density such that p = T s - e
        head = [tau, base[:, 1], base[:, 2], base[:, 3], base[:, 4] / tau, base[:, 5] / tau, base[:, 6] / tau, base[:, 7] / tau,
                ut, base[:, 8], base[:, 9], base[:, 10] * tau, E, T, z + 0.01]
        if mode == 6:
            head += [z, z]
        head += [s, z, z, z, z, pixx, pixy, pixn * tau, piyy, piyn * tau, z, bulk]
        return np.column_stack(head)
    if mode == 7:
        vx, vy = base[:, 8] / ut, base[:, 9] / ut
        return np.column_stack([tau, base[:, 1], base[:, 2], base[:, 3], base[:, 4] / tau, base[:, 5] / tau, base[:, 6] / tau, z,
                                vx, vy, z, z, z, z, z, pixx * hb, pixy * hb, pixn * hb * tau, piyy * hb, piyn * hb * tau, z,
                                bulk * hb, T * hb, E * hb, P * hb, z])
    if mode == 5:
        return np.column_stack([base, z + 0.1, z + 0.2, z + 0.3, z + 0.4, z + 0.5, z + 0.6])
    raise ValueError(mode)


@pytest.mark.parametrize("mode,dimension", [(4, 2), (6, 2), (7, 2), (5, 3), (4, 3)])
def test_other_surface_formats_against_reference(fx, mode, dimension):
    """MUSIC (old/new), hic-eventgen and vorticity surface formats: the C++ reader recovers the mode-1 cells the file was written
    from, up to what the format cannot carry (eta, and dsigma_eta / u^eta where the format drops them), and the oracle kernel gives
    the same spectra from them.  Where oracle/_ref is built, those spectra must also be the reference's from the same file, bit for
    bit."""
    base = synthetic.surface_vh(12, 100 + mode, three_d=(dimension == 3))
    cols = _alt_format_columns(mode, base)
    live = cfo.ref_binary() is not None
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=cols, chosen="chosen_pikp", fixture=fx, operation=1, mode=mode, hrg_eos=1,
                            dimension=dimension, df_mode=1)
        if mode == 5:      # this reader never writes the averages side file; the reference would read a stale one
            open(os.path.join(wd, "average_thermodynamic_quantities.dat"), "w").write("0.15\n0.3\n0.05\n0\n0")
        if live:
            ref, info = cfo.run_reference(wd)
        d = host_dump(wd)
    keys = ("tau", "eta", "dat", "dax", "day", "dan", "ux", "uy", "un", "E", "T", "P", "pixx", "pixy", "pixn", "piyy", "piyn", "bulkPi")
    cells = {k: d[k] for k in keys}
    want = synthetic.columns_to_cells(base, 1)
    if mode in (4, 6, 7):                  # boost-invariant formats: eta := 0, dsigma_eta kept by MUSIC-old 3+1D only
        want["eta"] = np.zeros(12)
        if mode != 4 or dimension == 2:
            want["dan"] = np.zeros(12)
    for k in keys:
        assert np.allclose(cells[k], want[k], rtol=1e-13, atol=0), k        # unit and tau factors: a few ulp
    sp = tables.species(fx, 1, "chosen_pikp"); g = tables.grid(fx); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=dimension)
    dN, skipped, _ = cfo.smooth(fl, cells, sp, g, tab, None)
    assert len(cells["tau"]) == 12 and skipped == 0
    # the per-bin bar of the project: bins deep in the exp(-p.u/T) tail scale a one-ulp cell difference by p.u/T (up to ~700)
    assert compare(dN, cfo.smooth(fl, {k: want[k] for k in keys}, sp, g, tab, None)[0])["ok"]
    if live:
        assert np.array_equal(dN, ref)


def test_vah_in_memory_helpers(fx):
    """is3d_b200_vah_anisotropy / is3d_b200_vah_coefficients give what the file path gives"""
    from common import vah_cells as ref_vah_cells
    cols = synthetic.surface_vah(64, 1005)
    mine = api.vah_cells(cols, fx)
    with tempfile.TemporaryDirectory() as wd:
        workdir.materialize(wd, surface_columns=cols, fixture=fx, hrg_eos=1, mode=2, vah=True)
        d = host_dump(wd)
    for k in ("aL", "Lambda", "c0", "c1", "c2", "c3", "c4"):
        assert np.array_equal(mine[k], d[k]), k
    ref = ref_vah_cells(cols, fx)
    for k in ("aL", "Lambda", "c0", "c4"):
        assert np.allclose(mine[k], ref[k], rtol=1e-12, atol=0), k


# ---------------------------------------------------------------------------------------- anisotropic model: coefficient lookup
def test_vah_coefficients_pinned_to_reference_reader(fx):
    """SURVEY 8a row a3: the (Lambda, alpha_L) -> c0..c4 lookup against the reference's ONLY reader of these tables,
    DeltafReader::load_coefficients (src/cuda/deltafReader.cu:192-277), compiled unmodified into oracle/_ref/vah_ref.
    Vectors: tests/golden/vah_coefficients.npz (make_vah_coeff_vectors.py); where oracle/_ref/vah_ref exists it is re-run live."""
    from is3d_b200 import api
    from oracle import cf_oracle as cfo
    from common import GOLDEN_DIR
    z = np.load(os.path.join(GOLDEN_DIR, "vah_coefficients.npz"))
    aL, Lam, ref = z["aL"], z["Lambda_GeV"], z["c"]
    if os.path.exists(os.path.join(os.path.dirname(cfo.__file__), "_ref", "vah_ref")):
        assert np.array_equal(cfo.run_vah_reference(aL, Lam, fx), ref)                    # the fixture is what the reference computes
    inside = ref[:, 0] != -12345.0                                                           # the reference leaves other cells untouched
    assert 0.9 < inside.mean() < 1.0
    got = api.vah_coefficients(fx, Lam[inside], aL[inside])
    for k in range(5):
        assert np.array_equal(got[k], ref[inside, k]), k                                     # bit-exact: same arithmetic, same order
    # the test-suite's own numpy restatement (tests/common.py vah_cells) agrees as well
    for i in np.flatnonzero(~inside)[:12]:                                                   # outside the table: an error, not garbage
        with pytest.raises(api.Is3dError) as e:
            api.vah_coefficients(fx, Lam[i:i + 1], aL[i:i + 1])
        assert e.value.code == 3
