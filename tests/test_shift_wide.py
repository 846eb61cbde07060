"""The shifted-factor kernel (cf_shift.cu) with wide phi groups: the default 3 slots x 6 phi points of the 14-moment model and
ideal f_eq, 3 x 8 and the other shapes of tile_variant 22..25 (Chapman-Enskog: the staged 7 x 2 .. 7 x 6 shapes), and the
scaled path for groups whose members may be sub-normal.

The CPU test checks the arithmetic of that path in numpy; the GPU tests compare every shape with the oracle on a phi grid
that does not fill the last group (padded phi records take part in Bmax / Bmin), on the stress surface, and on a surface with
fast transverse flow on which six times as many groups as on the plain surface touch the sub-normal range."""
import numpy as np
import pytest

from common import compare
from is3d_b200 import api, synthetic, tables

RARE_X = float(np.frombuffer(np.array([0x40861D9900000000], dtype=np.uint64).tobytes(), dtype=np.float64)[0])     # high word kRareHi
ALIVE_X = 709.782712893384           # ln(DBL_MAX): beyond it the reference's exp(x) overflows and the term is exactly 0
TINY = np.finfo(float).tiny
SHIFT = 64                           # kRareShift
SPECIES = [211, 321, 2212, -3334, 337]


def _underflow_columns(n_cells, seed):
    """cfg3-like surface with transverse flow eight times faster: pT (Bmax - Bmin) reaches thousands, and 2.3 % of the alive
    groups (0.4 % on the plain surface) have members near or beyond the end of the normal range of e^{-x}"""
    s = synthetic.surface_vh(n_cells, seed)
    s[:, 8] *= 8.0; s[:, 9] *= 8.0
    s[:, 4] = np.abs(s[:, 4]) * 5 + 0.5            # keep u.dsigma > 0
    return s


def _arguments(cols, mass, g, npt):
    """x = mT A_j - pT B_k of every (cell, slot, phi group, member, species, pT) and the group minimum, as the kernel forms them"""
    cells = synthetic.columns_to_cells(cols, 1)
    tau, eta, ux, uy, un, T = [np.asarray(cells[k]) for k in ("tau", "eta", "ux", "uy", "un", "T")]
    ut = np.sqrt(1.0 + ux * ux + uy * uy + tau * tau * un * un)
    y = np.asarray(g["y"]); phi = np.asarray(g["phi"]); pT = np.asarray(g["pT"])
    d = y[None, :] - eta[:, None]
    A = (np.cosh(d) * ut[:, None] - tau[:, None] * np.sinh(d) * un[:, None]) / T[:, None]            # [cell, slot]
    B = (np.cos(phi)[None, :] * ux[:, None] + np.sin(phi)[None, :] * uy[:, None]) / T[:, None]        # [cell, phi]
    n_tiles = -(-B.shape[1] // npt)
    Bp = np.zeros((B.shape[0], n_tiles * npt)); Bp[:, :B.shape[1]] = B                                # padded records: B = 0
    Bt = Bp.reshape(B.shape[0], n_tiles, npt)
    mT = np.sqrt(mass[:, None] ** 2 + pT[None, :] ** 2)                                               # [species, pT]
    a = A[:, :, None, None, None] * mT[None, None, None, :, :]                                         # [cell, slot, 1, species, pT]
    q = Bt[:, None, :, :, None, None] * pT                                                             # [cell, 1, tile, k, 1, pT]
    x = a[:, :, :, None] - q                                                                           # [cell, slot, tile, k, species, pT]
    qm = Bt.max(axis=2)[:, None, :, None, None] * pT
    xm = a - qm                                                                                        # [cell, slot, tile, species, pT]
    dB = pT * (Bt.max(axis=2) - Bt.min(axis=2))[:, None, :, None, None]
    d = (Bt.max(axis=2)[:, :, None] - Bt)[:, None, :, :, None, None] * pT                              # [cell, 1, tile, k, 1, pT]
    return x, xm, dB, d


def test_scaled_rare_path_at_npt8(fx):
    """e^{-xm} 2^64 times e^{-pT (Bmax - B_k)} stays a normal number for every member whose exp(x) is finite in the reference,
    scaling back by 2^-64 reproduces e^{-x} (sub-normal results included, to their last place), and the zero pattern is
    exactly that of the reference: zero iff x > ln(DBL_MAX).

    This checks a numpy model of the arithmetic (e^{64 ln2 - xm}, then ldexp by -64), not the kernel's own exp_neg_fast(pe,
    ne + kRareShift) and scale-back constant: a wrong shift sign or constant in the kernel is caught by the GPU tests below
    (test_near_underflow_surface compares every shape with the oracle, zero pattern included)."""
    sp = tables.species(fx, 1, SPECIES); g = tables.grid(fx)
    mass = np.asarray(sp["mass"])
    x, xm, dB, d = _arguments(_underflow_columns(40, 4711), mass, g, 8)
    alive = xm <= ALIVE_X
    rare = alive & (xm + dB >= RARE_X)
    assert rare.sum() > 0.015 * alive.sum(), (rare.sum(), alive.sum())
    with np.errstate(under="ignore"):
        eA = np.where(rare, np.exp(SHIFT * np.log(2.0) - xm), 0.0)               # e^{-xm} 2^64 on the rare groups
        eB = np.where(d <= ALIVE_X, np.exp(-d), 0.0)                                              # the block's table (exp_neg_slow)
        prod = eA[:, :, :, None] * eB
        member = np.broadcast_to(rare[:, :, :, None], x.shape) & (x <= ALIVE_X)
        scaled = np.ldexp(prod, -SHIFT)
        direct = np.exp(-np.where(member, x, 0.0))
    assert member.sum() > 5_000, member.sum()
    assert np.all(eA[rare] <= 2.0 ** SHIFT * 1.0000001) and np.all(eA[rare] >= TINY)
    assert np.all(prod[member] >= TINY)                      # before scaling back every alive member is normal
    sub = member & (direct < TINY)
    assert sub.sum() > 100, sub.sum()                        # the surface reaches sub-normal results
    assert np.all(scaled[member] > 0.0)                      # alive members never flush to zero
    err = np.abs(scaled[member] - direct[member])
    allow = 1e-12 * direct[member] + 2.0 * 2.0 ** -1074      # the product form to 1e-12, sub-normals to their last place
    assert np.all(err <= allow), float(np.max(err / allow))
    dead = np.broadcast_to(rare[:, :, :, None], x.shape) & (x > ALIVE_X)
    assert dead.sum() > 0                                    # members of alive groups beyond ln(DBL_MAX): zeroed per member


def _check(fx, cols, variants, grid=None, df_modes=(1, 2), extras=({}, dict(regulate_deltaf=0, outflow=0))):
    from oracle import cf_oracle as cfo
    api.init()
    cells = synthetic.columns_to_cells(cols, 1)
    sp = tables.species(fx, 1, SPECIES); g = grid or tables.grid(fx); tab = tables.df_tables(fx, 1)
    n_bins = len(SPECIES) * len(g["pT"]) * len(g["phi"]) * len(g["y"])
    for df_mode in df_modes:
        for extra in extras:
            fl = tables.flags(df_mode=df_mode, dimension=3, **extra)
            cond = np.zeros(n_bins)
            ref, _, _ = cfo.smooth(fl, cells, sp, g, tab, None, conditioning=cond)
            for variant in variants:
                got, st = api.smooth_spectra(fl, cells, sp, g, tab, None, tile_variant=variant)
                if variant == 0:
                    assert st["tile_variant"] == 22                          # default: cf_shift_kernel 3 x 6
                rep = compare(got, ref, conditioning=cond)
                assert rep["ok"], (df_mode, extra, variant, rep)
                assert np.array_equal(got == 0, ref == 0), (df_mode, extra, variant)


@pytest.mark.gpu
def test_phi_count_not_a_multiple_of_the_group(fx):
    """21 phi points: the last group has three padded records (B = 0) in the 3 x 6 and 3 x 8 shapes, which enter Bmax / Bmin
    and the group's classification but not the result"""
    g0 = tables.grid(fx)
    g = dict(g0)
    g["phi"] = g0["phi"][:21]; g["phi_weight"] = g0["phi_weight"][:21]
    _check(fx, synthetic.surface_vh(150, 4243), (0, 22, 23, 24, 25), grid=g)


@pytest.mark.gpu
def test_stress_surface_every_shape(fx):
    _check(fx, synthetic.surface_vh(150, 4244, stress=True), (0, 22, 23, 24, 25))


@pytest.mark.gpu
def test_near_underflow_surface(fx):
    """many groups take the scaled path; sub-normal members and dead members inside alive groups are both present
    (test_scaled_rare_path_at_npt8), and the zero pattern of the spectra must be the reference's exactly"""
    _check(fx, _underflow_columns(120, 4711), (0, 22, 23, 24, 25))


@pytest.mark.gpu
def test_ideal_f_eq_on_the_near_underflow_surface(fx):
    """ideal f_eq (no delta-f) through the same slot code, on the near-underflow surface"""
    from oracle import cf_oracle as cfo
    api.init()
    cells = synthetic.columns_to_cells(_underflow_columns(120, 4712), 1)
    sp = tables.species(fx, 1, SPECIES); g = tables.grid(fx); tab = tables.df_tables(fx, 1)
    fl = tables.flags(df_mode=1, dimension=3, include_bulk=0, include_shear=0)
    ref, _, _ = cfo.smooth(fl, cells, sp, g, tab, None)
    for variant in (0, 22, 23, 24, 25):
        got, st = api.smooth_spectra(fl, cells, sp, g, tab, None, tile_variant=variant)
        rep = compare(got, ref)
        assert rep["ok"], (variant, rep)
        assert np.array_equal(got == 0, ref == 0), variant
