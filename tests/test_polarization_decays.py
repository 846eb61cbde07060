"""Feed-down of the hadron spin polarization through 2-body resonance decays (is3d_b200_polarization_decays, DESIGN §17).

CPU tier: the transfer laws against a helicity-amplitude computation with Wigner matrices, the oracle's Lorentz chain against a numpy
restatement, and the oracle's analytic anchors (Snorm bit for bit the decay oracle, linearity, p.N = 0, dilution-only channels, the
slow-parent limit).  GPU tier: the CUDA path through the C ABI against the oracle, bit-identity of Snorm with is3d_b200_resonance_decays,
reproducibility, device memory and the error rules."""
import os
import sys

import numpy as np
import pytest
from scipy.linalg import expm

from common import GOLDEN_DIR, compare
from is3d_b200 import api, tables
from oracle import cf_oracle as cfo
from oracle import cf_polzn_fd as fdo

sys.path.insert(0, GOLDEN_DIR)
import make_decay_vectors as mdv      # noqa: E402  (thermal input builder shared with the decay tests)

FIELDS = ("St", "Sx", "Sy", "Sz", "Snorm")
# Lambda, anti-Lambda, Sigma0 (-> Lambda gamma), Sigma(1385) (-> Lambda pi, Sigma pi), Lambda(1520) (-> Sigma0 pi0 -> Lambda gamma: a
# two-level cascade into Lambda; -> Sigma(1385) pi: spin-3/2 daughter, dilution only)
CHOSEN = [211, -211, 111, 3122, -3122, 3212, -3212, 3224, -3224, 3214, 3114, 3124]
HI_PT = list(range(0, 22, 3)) + list(range(22, 32))        # every parent needs >= 2 points beyond mT = 1.65 M for its tail fit


# ---------------------------------------------------------------------------------------------------- transfer laws (helicity)
def _spin_matrices(J):
    m = np.arange(J, -J - 1, -1)
    Jp = np.zeros((len(m), len(m)), complex)
    for k in range(1, len(m)):
        Jp[k - 1, k] = np.sqrt(J * (J + 1) - m[k] * (m[k] + 1))
    return m, (Jp + Jp.conj().T) / 2, (Jp - Jp.conj().T) / 2j, np.diag(m).astype(complex)


def _rotation(a, b, g):
    Rz = lambda t: np.array([[np.cos(t), -np.sin(t), 0], [np.sin(t), np.cos(t), 0], [0, 0, 1]])
    Ry = lambda t: np.array([[np.cos(t), 0, np.sin(t)], [0, 1, 0], [-np.sin(t), 0, np.cos(t)]])
    return Rz(a) @ Ry(b) @ Rz(g)


def _helicity_daughter_spin(J, S, n, partner, ratio):
    """Mean spin (parent-frame axes) of the spin-1/2 daughter flying along n, for a parent of spin J with <J> = S: linear-order density
    matrix rho = (1 + 3/(J(J+1)) S.J)/(2J+1), amplitudes D^J*_{M, l1 - l2}(phi, theta, -phi) H_{l1 l2}; partner 'meson' (l2 = 0) or
    'photon' (l2 = +-1); ratio = H_{-l1,-l2} / H_{l1,l2} from the Jacob-Wick parity relation."""
    m, Jx, Jy, Jz = _spin_matrices(J)
    rho = (np.eye(len(m)) + 3.0 / (J * (J + 1)) * (S[0] * Jx + S[1] * Jy + S[2] * Jz)) / (2 * J + 1)
    th, ph = np.arccos(n[2]), np.arctan2(n[1], n[0])
    D = expm(-1j * ph * Jz) @ expm(-1j * th * Jy) @ expm(1j * ph * Jz)       # D^J(phi, theta, -phi)_{M' M}
    rhoD = np.zeros((2, 2), complex)
    for l2 in ([0] if partner == "meson" else [1, -1]):
        A = np.zeros((2, len(m)), complex)
        for i, l1 in enumerate((0.5, -0.5)):
            if partner == "photon" and np.sign(l1) != np.sign(l2):
                continue
            lam = l1 - l2
            if abs(lam) <= J:
                A[i] = np.conj(D[:, list(m).index(lam)]) * (1.0 if l1 > 0 else ratio)
        rhoD += A @ rho @ A.conj().T
    sig = (np.array([[0, 1], [1, 0]]), np.array([[0, -1j], [1j, 0]]), np.array([[1, 0], [0, -1]]))
    s_hel = np.array([np.trace(rhoD @ s).real for s in sig]) / 2 / np.trace(rhoD).real
    return _rotation(ph, th, -ph) @ s_hel


def _law(J2, PP, PD, Pm):
    eta = -(-1) ** ((J2 - 1) // 2) * PP * PD * Pm
    a = -eta * (J2 + 1) / 2.0
    return a, 1.0 - a


def test_transfer_law_matches_helicity_amplitudes():
    rng = np.random.default_rng(7)
    for J2 in (1, 3, 5, 7):
        J = J2 / 2.0
        f = 4 * J * (J + 1) / 3                    # true spin of the parent = f x the spin-1/2-normalised array value
        for PP in (1, -1):
            for Pm in (-1, 1):                     # 0- and 0+ partners
                a, b = _law(J2, PP, 1, Pm)
                ratio = PP * 1 * Pm * (-1) ** ((J2 - 1) // 2)      # H_{-1/2,0} = P_P P_D P_m (-1)^(J - 1/2) H_{1/2,0}
                for _ in range(6):
                    S = rng.normal(size=3) * 0.2
                    n = rng.normal(size=3); n /= np.linalg.norm(n)
                    s = _helicity_daughter_spin(J, S * f, n, "meson", ratio)
                    assert np.abs(s - (a * S + b * (S @ n) * n)).max() <= 1e-13 * np.abs(S).max(), (J2, PP, Pm)
    for ratio in (1.0, -1.0):                      # 1/2 -> 1/2 + photon, either parity
        for _ in range(6):
            S = rng.normal(size=3) * 0.2
            n = rng.normal(size=3); n /= np.linalg.norm(n)
            s = _helicity_daughter_spin(0.5, S, n, "photon", ratio)
            assert np.abs(s - (-(S @ n) * n)).max() <= 1e-13 * np.abs(S).max()
    # the averages C = <S*_D> / S*_P of the true spins (Becattini, Cao & Speranza 2019)
    C = lambda J2, PP: (lambda a, b: (a + b / 3.0) / (4 * (J2 / 2) * (J2 / 2 + 1) / 3))(*_law(J2, PP, 1, -1))
    assert np.isclose(C(1, 1), -1 / 3, rtol=0, atol=1e-15) and np.isclose(C(1, -1), 1.0, rtol=0, atol=1e-15)
    assert np.isclose(C(3, 1), 1 / 3, rtol=0, atol=1e-15) and np.isclose(C(3, -1), -1 / 5, rtol=0, atol=1e-15)


# ---------------------------------------------------------------------------------------------------- Lorentz chain
def _np_chain(P, M, Sp, dim2, p, mD, a, b):
    """numpy restatement in rapidity / velocity form: boosts as x' = x + (gamma - 1)(x.u)u - gamma v t with unit velocity u"""
    P = np.asarray(P, float); p = np.asarray(p, float); Sp = np.asarray(Sp, float)

    def boost(x, vel):                             # to the frame moving with velocity vel
        v = np.linalg.norm(vel)
        if v == 0:
            return x.copy()
        u = vel / v; g = 1 / np.sqrt(1 - v * v)
        t, xs = x[0], x[1:]
        return np.concatenate([[g * (t - v * (u @ xs))], xs + (g - 1) * (u @ xs) * u - g * v * t * u])
    if dim2:
        MT = np.sqrt(P[0] ** 2 - P[3] ** 2); Y = np.arctanh(P[3] / P[0])
        S0 = boost(np.concatenate([[0.0], Sp]), -np.array([P[1], P[2], 0.0]) / MT)
        S = boost(S0, np.array([0.0, 0.0, -np.tanh(Y)]))
        Sp = boost(S, P[1:] / P[0])[1:]
    ps = boost(p, P[1:] / P[0])
    n = ps[1:] / np.linalg.norm(ps[1:])
    s = a * Sp + b * (Sp @ n) * n
    q = boost(np.concatenate([[0.0], s]), -ps[1:] / ps[0])
    return boost(q, -P[1:] / P[0])


def test_oracle_chain_matches_numpy_restatement():
    rng = np.random.default_rng(3)
    for dim2 in (0, 1):
        for _ in range(200):
            M, mD = rng.uniform(1.2, 2.0), rng.uniform(0.1, 1.1)
            MT = np.sqrt(M * M + rng.uniform(0, 3) ** 2); Y = rng.uniform(-2, 2); Phi = rng.uniform(0, 2 * np.pi)
            PT = np.sqrt(MT * MT - M * M)
            P = np.array([MT * np.cosh(Y), PT * np.cos(Phi), PT * np.sin(Phi), MT * np.sinh(Y)])
            mt, y, phi = np.sqrt(mD ** 2 + rng.uniform(0, 3) ** 2), rng.uniform(-2, 2), rng.uniform(0, 2 * np.pi)
            pt = np.sqrt(mt * mt - mD * mD)
            p = np.array([mt * np.cosh(y), pt * np.cos(phi), pt * np.sin(phi), mt * np.sinh(y)])
            Sp = rng.normal(size=3) * 0.3; a, b = rng.normal(), rng.normal()
            got = fdo.chain(P, M, Sp, dim2, p, mD, a, b)
            ref = _np_chain(P, M, Sp, dim2, p, mD, a, b)
            scale = np.abs(Sp).max() * (1 + abs(a) + abs(b)) * (P[0] / M) * (p[0] / mD) ** 2
            assert np.abs(got - ref).max() <= 1e-13 * scale
            # the daughter's spin is orthogonal to its momentum
            assert abs(got[0] * p[0] - got[1:] @ p[1:]) <= 1e-13 * scale * p[0]


# ---------------------------------------------------------------------------------------------------- problems
def _spin_inputs(dN, sp_mass, g, dimension, n_species, scale=1.0):
    """The five arrays: Snorm = the thermal spectrum, N^mu = Snorm x the four-vector of a smooth rest-frame spin field S*(p)"""
    y = np.zeros(len(g["y"])) if dimension == 2 else np.asarray(g["y"])
    yy, ff, pp, mm = np.meshgrid(y, g["phi"], g["pT"], np.asarray(sp_mass, float), indexing="ij")
    mT = np.sqrt(pp * pp + mm * mm); E = mT * np.cosh(yy)
    p = np.stack([pp * np.cos(ff), pp * np.sin(ff), mT * np.sinh(yy)])
    Ss = scale * np.stack([0.08 * np.sin(ff) + 0.01 * pp, -0.05 * np.cos(2 * ff) + 0.02, 0.03 * np.sin(ff) * pp - 0.01 * yy])
    pS = (p * Ss).sum(0)
    Nt = pS / mm
    Nv = Ss + p * pS / (mm * (E + mm))
    sn = np.asarray(dN, float)
    return dict(St=(Nt.ravel() * sn), Sx=(Nv[0].ravel() * sn), Sy=(Nv[1].ravel() * sn), Sz=(Nv[2].ravel() * sn), Snorm=sn.copy())


def _problem(fx, dimension, chosen=CHOSEN):
    strides = dict(pT=HI_PT, phi=3, y=1) if dimension == 2 else dict(pT=HI_PT, phi=4, y=[7, 9, 10, 11, 13])
    rec = dict(dimension=dimension, n_cells=30, seed=11, strides=strides, chosen=chosen)
    g, tabs, cols, dN, pdg, chosen_idx = mdv.case_inputs(fx, rec)
    sp_mass = [pdg["mass"][i] for i in chosen_idx]
    sums = _spin_inputs(dN, sp_mass, g, dimension, len(chosen))
    return g, pdg, chosen_idx, sums, tables.spin_parity(fx, pdg, 1)


@pytest.fixture(scope="module")
def problems(fx):
    return {d: _problem(fx, d) for d in (2, 3)}


@pytest.fixture(scope="module")
def oracle_results(problems):
    return {d: fdo.polarization_decays(pdg, spar, idx, g, d, sums, conditioning=True) for d, (g, pdg, idx, sums, spar) in problems.items()}


def test_spin_parity_table(fx):
    pdg = tables.pdg_decay_table(fx, 1)
    sp = tables.spin_parity(fx, pdg, 1)
    mc = list(pdg["mcid"])
    at = lambda m: (int(sp["spin2"][mc.index(m)]), int(sp["parity"][mc.index(m)]))
    assert at(3122) == (1, 1) and at(-3122) == (1, 1) and at(3212) == (1, 1) and at(3224) == (3, 1) and at(-3224) == (3, 1)
    assert at(211) == (0, -1) and at(111) == (0, -1) and at(3124) == (3, -1) and at(22)[1] == 0       # the photon: not in pdg_box
    assert (sp["spin2"] >= 0).all() and set(np.unique(sp["parity"])) <= {-1, 0, 1}


@pytest.mark.parametrize("dimension", [2, 3])
def test_oracle_snorm_is_the_decay_oracle(problems, oracle_results, dimension):
    g, pdg, idx, sums, spar = problems[dimension]
    out, _ = oracle_results[dimension]
    assert np.array_equal(out["Snorm"], cfo.resonance_decays(pdg, idx, g, dimension, sums["Snorm"]))
    ns = len(CHOSEN); L = ns * len(g["pT"]) * len(g["phi"])
    lam = CHOSEN.index(3122)
    for k in ("St", "Sx", "Sy", "Sz"):                         # Lambda is fed, and bins beyond the 2+1D y = 0 plane stay untouched
        assert np.any(out[k][lam:L:ns] != sums[k][lam:L:ns])
        if dimension == 2:
            assert np.array_equal(out[k][L:], sums[k][L:])


@pytest.mark.parametrize("dimension", [2, 3])
def test_oracle_anchors(problems, oracle_results, dimension):
    g, pdg, idx, sums, spar = problems[dimension]
    out, cond = oracle_results[dimension]
    fd = {k: out[k] - sums[k] for k in FIELDS}
    # N = 0 in: exactly zero feed-down into N
    zero = dict(sums, St=np.zeros_like(sums["St"]), Sx=np.zeros_like(sums["St"]), Sy=np.zeros_like(sums["St"]), Sz=np.zeros_like(sums["St"]))
    z = fdo.polarization_decays(pdg, spar, idx, g, dimension, zero)
    for k in ("St", "Sx", "Sy", "Sz"):
        assert np.all(z[k] == 0.0)
    # N x 2 in: feed-down x 2 (the parent's S* doubles; its weights do not change)
    two = dict(sums, **{k: 2.0 * sums[k] for k in ("St", "Sx", "Sy", "Sz")})
    t = fdo.polarization_decays(pdg, spar, idx, g, dimension, two)
    for k in ("St", "Sx", "Sy", "Sz"):
        d2 = t[k] - two[k]
        assert np.all(np.abs(d2 - 2.0 * fd[k]) <= 1e-15 * np.abs(d2) + 4 * np.finfo(float).eps * np.abs(two[k]))
    # p.N_fd = 0 per bin within 1e-12 of the |terms| sum.  N_fd = out - in also carries the rounding of that subtraction, a few ulp of
    # |p.N_in| term by term, which dominates in bins where the feed-down is 1e-6 .. 1e-10 of the primary sums
    y = np.zeros(len(g["y"])) if dimension == 2 else np.asarray(g["y"])
    ms = np.array([pdg["mass"][i] for i in idx])
    yy, ff, pp, mm = np.meshgrid(y, g["phi"], g["pT"], ms, indexing="ij")
    mT = np.sqrt(pp * pp + mm * mm)
    E, px, py, pz = (mT * np.cosh(yy)).ravel(), (pp * np.cos(ff)).ravel(), (pp * np.sin(ff)).ravel(), (mT * np.sinh(yy)).ravel()
    pdot = fd["St"] * E - fd["Sx"] * px - fd["Sy"] * py - fd["Sz"] * pz
    absterm = cond["St"] * E + (cond["Sx"] + cond["Sy"]) * pp.ravel() + cond["Sz"] * np.abs(pz)
    subtraction = 4 * np.finfo(float).eps * (np.abs(out["St"] * E) + np.abs(out["Sx"] * px) + np.abs(out["Sy"] * py) + np.abs(out["Sz"] * pz))
    assert np.all(np.abs(pdot) <= 1e-12 * absterm + subtraction)
    assert np.count_nonzero(absterm) > 0


def test_oracle_dilution_only(problems):
    g, pdg, idx, sums, spar = problems[3]
    # no law anywhere: every parity unknown and no photon channel among the chosen species
    chosen = [211, -211, 111, 3122, -3122, 3224, -3224, 3214, 3114]
    first = {}
    for n, m in enumerate(pdg["mcid"]):
        first.setdefault(int(m), n)
    idx2 = [first[m] for m in chosen]
    s2 = _spin_inputs(np.ones(len(chosen) * len(g["pT"]) * len(g["phi"]) * len(g["y"])), [pdg["mass"][i] for i in idx2], g, 3, len(chosen))
    s2["Snorm"] = np.exp(-np.sqrt(np.add.outer(np.repeat(np.asarray(g["pT"]) ** 2, 1), np.array([pdg["mass"][i] for i in idx2]) ** 2)) / 0.15)
    s2["Snorm"] = np.tile(s2["Snorm"].ravel(), len(g["phi"]) * len(g["y"]))
    unknown = dict(spin2=spar["spin2"], parity=np.zeros_like(spar["parity"]))
    out = fdo.polarization_decays(pdg, unknown, idx2, g, 3, s2)
    for k in ("St", "Sx", "Sy", "Sz"):
        assert np.array_equal(out[k], s2[k])
    assert np.any(out["Snorm"] != s2["Snorm"])
    assert np.array_equal(out["Snorm"], cfo.resonance_decays(pdg, idx2, g, 3, s2["Snorm"]))


# ---------------------------------------------------------------------------------------------------- slow-parent limit
def _mini_list():
    """gamma, pi+, Lambda, Sigma0 -> Lambda gamma, Sigma(1385)+ -> Lambda pi+ (widths 0: no mass shift)"""
    rows = [(22, 0.0, [(1, 1.0, [22])]), (211, 0.13957, [(1, 1.0, [211])]), (3122, 1.115683, [(1, 1.0, [3122])]),
            (3212, 1.192642, [(2, 1.0, [3122, 22])]), (3224, 1.38280, [(2, 1.0, [3122, 211])])]
    out = dict(mcid=[], mass=[], width=[], stable=[], decays=[], dec_first=[], dec_npart=[], dec_br=[], dec_part=[])
    for m, mass, ch in rows:
        out["mcid"].append(m); out["mass"].append(mass); out["width"].append(0.0)
        out["stable"].append(1 if ch[0][0] == 1 else 0); out["decays"].append(len(ch)); out["dec_first"].append(len(out["dec_npart"]))
        for n, br, parts in ch:
            out["dec_npart"].append(n); out["dec_br"].append(br); out["dec_part"].append(parts + [0] * (5 - len(parts)))
    pdg = {k: np.asarray(v) for k, v in out.items()}
    spar = dict(spin2=np.array([2, 0, 1, 1, 3], np.int32), parity=np.array([0, -1, 1, 1, 1], np.int32))
    return pdg, spar


def _slow_parent(parent_row, T=0.02):
    """Lambda fed by one cold parent (Boltzmann spectrum, log-linear in M_T so the interpolation is exact) with uniform rest-frame spin
    S*_P; returns the daughter's momentum-integrated rest-frame spin over S*_P, per axis."""
    pdg, spar = _mini_list()
    n_pT, n_phi = 160, 48
    pT = np.linspace(0.004, 2.2, n_pT); phi = (np.arange(n_phi) + 0.5) * 2 * np.pi / n_phi
    g = dict(pT=pT, phi=phi, phi_weight=np.full(n_phi, 2 * np.pi / n_phi), y=np.array([0.0]), eta=np.array([0.0]), eta_weight=np.array([1.0]))
    chosen = [2, parent_row]                                    # Lambda, parent
    M = pdg["mass"][parent_row]; m = pdg["mass"][2]
    res = []
    for axis in range(3):
        Sp = np.zeros(3); Sp[axis] = 0.1
        sums = {k: np.zeros(2 * n_pT * n_phi) for k in FIELDS}
        ff, pp = np.meshgrid(phi, pT, indexing="ij")
        MT = np.sqrt(pp * pp + M * M)
        sn = np.exp(-(MT - M) / T)
        p = np.stack([pp * np.cos(ff), pp * np.sin(ff), np.zeros_like(pp)])
        pS = (p * Sp[:, None, None]).sum(0)
        sums["Snorm"][1::2] = sn.ravel()
        sums["St"][1::2] = (sn * pS / M).ravel()
        for c, k in enumerate(("Sx", "Sy", "Sz")):
            sums[k][1::2] = (sn * (Sp[c] + p[c] * pS / (M * (MT + M)))).ravel()
        out = fdo.polarization_decays(pdg, spar, chosen, g, 2, sums)
        d = {k: out[k][0::2].reshape(n_phi, n_pT) for k in FIELDS}
        mT = np.sqrt(pp * pp + m * m)
        w = pp * np.gradient(pT)[None, :]                       # pT dpT dphi at y = 0 (boost invariance)
        rest = [d[k] - d["St"] * p[c] / (mT + m) for c, k in enumerate(("Sx", "Sy", "Sz"))]
        res.append((w * rest[axis]).sum() / (w * d["Snorm"]).sum() / Sp[axis])
    return np.array(res)


def test_slow_parent_limit():
    """A cold parent (T = 20 MeV) with uniform S*_P: the daughter's momentum-integrated S* is C S*_P up to O(p*^2 / m_D^2) (Wigner
    rotations and the relativistic part of the daughter's spin four-vector) and O(T / M) (the parent's thermal motion).  Measured
    deviations, per axis: 4e-4 .. 9e-4 for Sigma0 -> Lambda gamma (p* = 74 MeV, (p*/m_Lambda)^2 = 4.5e-3) and 8e-4 .. 1.1e-3 for
    Sigma(1385)+ -> Lambda pi+ (p* = 208 MeV, (p*/m_Lambda)^2 = 3.4e-2).  The bar is (p*/m_Lambda)^2: 5x and 30x the measured deviations,
    and a wrong law (C off by 1/3 or more) is far outside it."""
    pdg, _ = _mini_list()
    mL = pdg["mass"][2]
    for row, ratio, W in ((3, -1.0 / 3.0, 0.0), (4, 5.0 / 3.0, 0.13957)):      # array ratio = C x 4J(J+1)/3: -1/3 x 1, 1/3 x 5
        M = pdg["mass"][row]
        Estar = (M * M + mL * mL - W * W) / (2 * M); pstar = np.sqrt(Estar ** 2 - mL ** 2)
        got = _slow_parent(row)
        dev = np.abs(got / ratio - 1.0)
        print("parent", pdg["mcid"][row], "S*_D / S*_P per axis", got, "expected", ratio, "deviation", dev, "(p*/m)^2", (pstar / mL) ** 2)
        assert np.all(dev <= (pstar / mL) ** 2), (row, got)


# ---------------------------------------------------------------------------------------------------- GPU tier
def _gpu_compare(got, ref, cond):
    """1e-10 per bin; St..Sz with the oracle's conditioning, sum of |term| x (1 + |log dN|) plus |ref| (the feed-down of a bin can cancel
    the primary sums, and a term's weight carries |log dN| ulps from the log / exp of the two math libraries); Snorm plainly"""
    for k in FIELDS:
        r = compare(np.asarray(got[k]), ref[k], conditioning=(cond[k] + np.abs(ref[k])) if k != "Snorm" else None)
        assert r["ok"], (k, r)


@pytest.mark.gpu
@pytest.mark.parametrize("dimension", [2, 3])
def test_cuda_matches_oracle(problems, oracle_results, dimension):
    import torch
    api.init()
    g, pdg, idx, sums, spar = problems[dimension]
    ref, cond = oracle_results[dimension]
    got, st = api.polarization_decays(pdg, spar, idx, g, dimension, sums)
    print("dim", dimension, "kernel ms %.2f" % st["kernel_ms"], "launches", st["gpu_launches"])
    _gpu_compare(got, ref, cond)
    # Snorm bit for bit the spectra feed-down of the same library
    dN, _ = api.resonance_decays(pdg, idx, g, dimension, sums["Snorm"])
    assert np.array_equal(got["Snorm"], dN)
    # bit-reproducible, and the device-memory path gives the same numbers in place
    again, _ = api.polarization_decays(pdg, spar, idx, g, dimension, sums)
    for k in FIELDS:
        assert np.array_equal(again[k], got[k])
    t = {k: torch.tensor(sums[k], device="cuda") for k in FIELDS}
    res, _ = api.polarization_decays(pdg, spar, idx, g, dimension, t, memory="device")
    torch.cuda.synchronize()
    assert res is t
    for k in FIELDS:
        assert np.array_equal(t[k].cpu().numpy(), got[k])
    # the inputs of the host call were not touched
    for k in FIELDS:
        assert np.array_equal(sums[k], problems[dimension][3][k])


@pytest.mark.gpu
def test_cuda_errors_leave_arrays_untouched(problems):
    import torch
    api.init()
    g, pdg, idx, sums, spar = problems[3]
    t = {k: torch.tensor(sums[k], device="cuda") for k in FIELDS}
    # a parent whose tail fit has fewer than 2 points: its spectrum is 0 beyond the first pT points
    bad = {k: v.clone() for k, v in t.items()}
    ns = len(CHOSEN); n_pT = len(g["pT"])
    sn = bad["Snorm"].view(-1, n_pT, ns)
    sn[:, 3:, ns - 1] = 0.0
    before = {k: v.clone() for k, v in bad.items()}
    with pytest.raises(api.Is3dError) as e:
        api.polarization_decays(pdg, spar, idx, g, 3, bad, memory="device")
    assert e.value.code == 1
    torch.cuda.synchronize()
    for k in FIELDS:
        assert torch.equal(bad[k], before[k])
    # argument checks
    for sp_bad in (None, dict(spin2=spar["spin2"] - 2, parity=spar["parity"]), dict(spin2=spar["spin2"], parity=spar["parity"] * 2)):
        with pytest.raises(api.Is3dError) as e:
            api.polarization_decays(pdg, sp_bad, idx, g, 3, sums)
        assert e.value.code == 1
    with pytest.raises(api.Is3dError) as e:
        api.polarization_decays(pdg, spar, idx, g, 4, sums)
    assert e.value.code == 1


# ---------------------------------------------------------------------------------------------------- host layer
def test_host_layer_key_rules_and_parities(fx):
    import tempfile
    from test_spin_polarization_shear import _host_dump, _materialize, _mode5_columns
    cols, _, _, xi = _mode5_columns(4, 31)
    with tempfile.TemporaryDirectory() as wd:
        for kw in (dict(spin_polarization=0), dict(mode=1, spin_polarization=0), dict(spin_polarization=1, operation=0),
                   dict(spin_polarization=1, hrg_eos=3)):
            c = cols[:, :-6] if kw.get("mode") == 1 else cols
            _materialize(wd, fx, c, polarization_feed_down=1, **kw)
            assert _host_dump(wd)[0] == 2, kw                                             # IS3D_ERR_UNSUPPORTED
        _materialize(wd, fx, cols, spin_polarization=1, polarization_feed_down=1)
        rc, d = _host_dump(wd)
        assert rc == 0, d
        pdg = tables.pdg_decay_table(fx, 1)
        sp = tables.spin_parity(fx, pdg, 1)
        assert np.array_equal(d["pdg_mcid"].astype(int), pdg["mcid"])
        assert np.array_equal(d["pdg_spin2"].astype(int), sp["spin2"]) and np.array_equal(d["pdg_parity"].astype(int), sp["parity"])
        os.remove(os.path.join(wd, "PDG", "pdg_box.dat"))
        rc, msg = _host_dump(wd)
        assert rc == 6 and "pdg_box.dat" in msg                                           # IS3D_ERR_IO
        _materialize(wd, fx, cols, spin_polarization=1)                                 # without the key: no box list, no records
        assert not os.path.exists(os.path.join(wd, "PDG", "pdg_box.dat"))
        rc, d = _host_dump(wd)
        assert rc == 0 and "pdg_parity" not in d and "pdg_spin2" not in d


@pytest.mark.gpu
@pytest.mark.parametrize("dimension,shear", [(3, True), (2, False)])
def test_gpu_workdir_feed_down_files(fx, dimension, shear):
    """With the key: S_fd_<mcid>.dat holds api.mean_spin of the fed-down total (vorticity [+ shear]) of direct calls, and S_ / S_xi_ files
    are byte-identical to a run without it; a run without the key (absent or 0) writes the files it wrote before."""
    import tempfile
    from is3d_b200 import synthetic, workdir
    from test_spin_polarization_shear import _mode5_columns, _run
    api.init()
    cols, base, vort, xi = _mode5_columns(60, 7411 + dimension, dimension)
    chosen = [211, -211, 111, 3122, -3122, 3212, -3212, 3224, -3224]
    extra0 = dict(thermal_shear_polarization=1) if shear else {}
    runs = {}
    for label, extra in (("absent", {}), ("zero", dict(polarization_feed_down=0)), ("on", dict(polarization_feed_down=1))):
        with tempfile.TemporaryDirectory() as wd:
            workdir.materialize(wd, surface_columns=cols, chosen=chosen, fixture=fx, operation=1, mode=5, dimension=dimension, df_mode=1,
                                spin_polarization=1, thermal_shear=xi, **extra0, **extra)
            open(os.path.join(wd, "average_thermodynamic_quantities.dat"), "w").write("0.15\n0.3\n0.05\n0\n0")
            runs[label] = _run(wd)
    assert runs["absent"][0] == runs["zero"][0]
    assert not any("S_fd_" in f for f in runs["absent"][0])
    fd_files = ["polarization" + os.sep + "S_fd_%d.dat" % c for c in chosen]
    assert runs["on"][0] == sorted(runs["absent"][0] + fd_files)
    for f, text in runs["absent"][1].items():
        assert runs["on"][1][f] == text == runs["zero"][1][f], f
    header = runs["on"][1][fd_files[0]].decode().split("\n", 1)[0].split()
    assert header == ["y", "phip", "pT", "Snorm", "St", "Sx", "Sy", "Sz", "Sx_rest", "Sy_rest", "Sz_rest"]

    cells = synthetic.columns_to_cells(base, 1)
    sp = tables.species(fx, 1, chosen); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=dimension)
    total, _ = api.spin_polarization(fl, cells, vort, sp, g)
    if shear:
        rx, _ = api.spin_polarization_shear(fl, cells, xi, sp, g)
        total = {k: total[k] + rx[k] if k != "Snorm" else total[k] for k in FIELDS}
    pdg = tables.pdg_decay_table(fx, 1)
    first = {}
    for n, m in enumerate(pdg["mcid"]):
        first.setdefault(int(m), n)
    fed, _ = api.polarization_decays(pdg, tables.spin_parity(fx, pdg, 1), [first[m] for m in chosen], g, dimension, total)
    S, rest = api.mean_spin(fed, sp, g, dimension)
    ny = 1 if dimension == 2 else len(g["y"])
    shape = (len(g["y"]), len(g["phi"]), len(g["pT"]), -1)
    lam = chosen.index(3122)
    assert np.any(fed["Sx"].reshape(shape)[:ny, :, :, lam] != total["Sx"].reshape(shape)[:ny, :, :, lam])
    for s, f in enumerate(fd_files):
        got = np.loadtxt(runs["on"][1][f].decode().splitlines(), skiprows=1, ndmin=2)[:, 3:]
        want = np.column_stack([v.reshape(shape)[:ny, :, :, s].ravel() for v in [fed["Snorm"]] + list(S) + list(rest)])
        assert got.shape == want.shape
        scale = np.abs(want).max(axis=0)
        assert np.all(np.abs(got - want) <= 2e-8 * np.abs(want) + 1e-12 * scale), f
