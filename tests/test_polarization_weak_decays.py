"""Feed-down of the hadron spin polarization through weak decays (is3d_b200_polarization_weak_decays, DESIGN §20): Xi -> Lambda pi with the
Lee-Yang law, Omega- channels that only dilute.

CPU tier: the Lee-Yang law against the spin density of T = s + p sigma.n, the oracle's chain against a numpy restatement, the
parity-conserving limits against the strong feed-down oracle, the slow-parent limit (1 + 2 gamma)/3, the exact structure of the oracle,
the file reader, the key rules, the argument errors and the struct layout.  GPU tier: the CUDA path against the oracle, repeatability,
device memory, error paths, the limits against is3d_b200_polarization_decays, and the work-dir run."""
import ctypes as C
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from common import GOLDEN_DIR, compare
from is3d_b200 import api, tables, workdir
from oracle import cf_polzn_fd as fdo
from oracle import cf_polzn_fdw as fdw

sys.path.insert(0, GOLDEN_DIR)
import make_decay_vectors as mdv      # noqa: E402  (thermal input builder shared with the decay tests)

FIELDS = ("St", "Sx", "Sy", "Sz", "Snorm")
# pi, K, Lambda, Sigma0 (strong -> Lambda gamma), Xi, Xi(1530)0 (strong -> Xi pi), Omega-: the strong pass feeds Lambda and Xi, the weak
# pass then Omega -> Xi0 pi- -> Lambda (a two-level weak cascade), Omega -> Lambda K- (dilution only) and Xi -> Lambda pi (the law)
CHOSEN = [211, -211, 111, 321, -321, 3122, -3122, 3212, -3212, 3312, -3312, 3322, -3322, 3324, 3334]
HI_PT = list(range(0, 22, 3)) + list(range(22, 32))        # every parent needs >= 2 points beyond mT = 1.65 M for its tail fit
# test values of (alpha, phi), not PDG numbers: the tests never depend on a PDG edition
WEAK = dict(parent=[3312, -3312, 3322, -3322, 3334, 3334], daughter=[3122, -3122, 3122, -3122, 3122, 3322],
            partner=[-211, 211, 111, 111, -321, -211], branching=[0.999, 0.999, 0.995, 0.995, 0.68, 0.24],
            alpha=[-0.41, 0.37, -0.33, 0.35, 0.02, 0.05], phi=[0.3, -0.25, 0.12, -0.4, 0.0, 0.0])


# ---------------------------------------------------------------------------------------------------- the law
def test_lee_yang_law_matches_amplitudes():
    rng = np.random.default_rng(5)
    sig = (np.array([[0, 1], [1, 0]]), np.array([[0, -1j], [1j, 0]]), np.array([[1, 0], [0, -1]]))
    for _ in range(200):
        s, p = rng.normal(size=2) + 1j * rng.normal(size=2)
        N = abs(s) ** 2 + abs(p) ** 2
        alpha, beta, gamma = 2 * (np.conj(s) * p).real / N, 2 * (np.conj(s) * p).imag / N, (abs(s) ** 2 - abs(p) ** 2) / N
        assert abs(alpha ** 2 + beta ** 2 + gamma ** 2 - 1) <= 1e-13
        n = rng.normal(size=3); n /= np.linalg.norm(n)
        P = rng.normal(size=3); P *= rng.uniform(0, 1) / np.linalg.norm(P)
        T = s * np.eye(2) + p * sum(n[k] * sig[k] for k in range(3))
        rhoD = T @ ((np.eye(2) + sum(P[k] * sig[k] for k in range(3))) / 2) @ T.conj().T
        rate = np.trace(rhoD).real
        PD = np.array([np.trace(rhoD @ sg).real for sg in sig]) / rate
        assert abs(rate / N - (1 + alpha * P @ n)) <= 1e-13
        want = ((alpha + P @ n) * n + beta * np.cross(P, n) + gamma * np.cross(n, np.cross(P, n))) / (1 + alpha * P @ n)
        assert np.abs(PD - want).max() <= 1e-13
        # the spin-1/2-normalised form of the kernels (S = P/2)
        S = P / 2
        s_num = (alpha / 2 + S @ n) * n + beta * np.cross(S, n) + gamma * (S - (S @ n) * n)
        assert np.abs(s_num / (1 + 2 * alpha * S @ n) - PD / 2).max() <= 1e-13
    # averages over n: yield 1, <s*> = (1 + 2 gamma)/3 S (Lebedev-free check with a symmetric point set)
    g = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]], float)
    S = np.array([0.1, -0.2, 0.05]); alpha, beta, gamma = 0.4, 0.3, np.sqrt(1 - 0.25)
    num = np.array([(alpha / 2 + S @ n) * n + beta * np.cross(S, n) + gamma * (S - (S @ n) * n) for n in g]).mean(0)
    assert np.allclose(num, (1 + 2 * gamma) / 3 * S, rtol=0, atol=1e-15)
    assert np.isclose(np.mean([1 + 2 * alpha * S @ n for n in g]), 1.0, rtol=0, atol=1e-15)


def _np_chain(P, M, Sp, dim2, p, mD, alpha, beta, gamma):
    """numpy restatement in rapidity / velocity form (the _np_chain of the strong feed-down test with the alpha and beta terms)"""
    P = np.asarray(P, float); p = np.asarray(p, float); Sp = np.asarray(Sp, float)

    def boost(x, vel):
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
    s = (alpha / 2 + Sp @ n) * n + beta * np.cross(Sp, n) + gamma * (Sp - (Sp @ n) * n)
    q = boost(np.concatenate([[0.0], s]), -ps[1:] / ps[0])
    return boost(q, -P[1:] / P[0]), 1 + 2 * alpha * (Sp @ n)


def test_oracle_chain_matches_numpy_restatement():
    rng = np.random.default_rng(13)
    for dim2 in (0, 1):
        for _ in range(200):
            M, mD = rng.uniform(1.2, 2.0), rng.uniform(0.1, 1.1)
            MT = np.sqrt(M * M + rng.uniform(0, 3) ** 2); Y = rng.uniform(-2, 2); Phi = rng.uniform(0, 2 * np.pi)
            PT = np.sqrt(MT * MT - M * M)
            P = np.array([MT * np.cosh(Y), PT * np.cos(Phi), PT * np.sin(Phi), MT * np.sinh(Y)])
            mt, y, phi = np.sqrt(mD ** 2 + rng.uniform(0, 3) ** 2), rng.uniform(-2, 2), rng.uniform(0, 2 * np.pi)
            pt = np.sqrt(mt * mt - mD * mD)
            p = np.array([mt * np.cosh(y), pt * np.cos(phi), pt * np.sin(phi), mt * np.sinh(y)])
            Sp = rng.normal(size=3) * 0.3
            alpha = rng.uniform(-1, 1); ph = rng.uniform(-np.pi, np.pi)
            beta, gamma = np.sqrt(1 - alpha ** 2) * np.sin(ph), np.sqrt(1 - alpha ** 2) * np.cos(ph)
            got, yg = fdw.chain(P, M, Sp, dim2, p, mD, alpha, beta, gamma)
            ref, yr = _np_chain(P, M, Sp, dim2, p, mD, alpha, beta, gamma)
            scale = (np.abs(Sp).max() + 1) * (P[0] / M) * (p[0] / mD) ** 2
            assert np.abs(got - ref).max() <= 1e-13 * scale
            assert abs(yg - yr) <= 1e-13 * scale
            assert abs(got[0] * p[0] - got[1:] @ p[1:]) <= 1e-13 * scale * p[0]


# ---------------------------------------------------------------------------------------------------- mini lists
def _mini_list(weak_parent, partner_parity=-1):
    """pi-, Lambda, Xi- (mass 1.32171): with weak_parent Xi is stable (the weak table feeds Lambda), otherwise it has the strong channel
    Xi -> Lambda pi-; widths 0 (no mass shift).  Parities: Xi, Lambda +, pi- partner_parity."""
    xi = [(1, 1.0, [3312])] if weak_parent else [(2, 1.0, [3122, -211])]
    rows = [(-211, 0.13957, [(1, 1.0, [-211])]), (3122, 1.115683, [(1, 1.0, [3122])]), (3312, 1.32171, xi)]
    out = dict(mcid=[], mass=[], width=[], stable=[], decays=[], dec_first=[], dec_npart=[], dec_br=[], dec_part=[])
    for m, mass, ch in rows:
        out["mcid"].append(m); out["mass"].append(mass); out["width"].append(0.0)
        out["stable"].append(1 if ch[0][0] == 1 else 0); out["decays"].append(len(ch)); out["dec_first"].append(len(out["dec_npart"]))
        for n, br, parts in ch:
            out["dec_npart"].append(n); out["dec_br"].append(br); out["dec_part"].append(parts + [0] * (5 - len(parts)))
    pdg = {k: np.asarray(v) for k, v in out.items()}
    spar = dict(spin2=np.array([0, 1, 1], np.int32), parity=np.array([partner_parity, 1, 1], np.int32))
    return pdg, spar


def _row(alpha, phi):
    return dict(parent=[3312], daughter=[3122], partner=[-211], branching=[1.0], alpha=[alpha], phi=[phi])


def _mini_grid(n_pT=24, n_phi=12, T=None):
    pT = np.linspace(0.02, 2.6, n_pT); phi = (np.arange(n_phi) + 0.5) * 2 * np.pi / n_phi
    return dict(pT=pT, phi=phi, phi_weight=np.full(n_phi, 2 * np.pi / n_phi), y=np.array([0.0]), eta=np.array([0.0]), eta_weight=np.array([1.0]))


def _mini_sums(g, masses, T=0.15, spin=True):
    """chosen = [Lambda, Xi]: thermal Snorm, and N = Snorm x the four-vector of a smooth rest-frame spin field (Lambda: a different one)"""
    ff, pp = np.meshgrid(g["phi"], g["pT"], indexing="ij")
    sums = {k: np.zeros(2 * pp.size) for k in FIELDS}
    for s, m in enumerate(masses):
        MT = np.sqrt(pp * pp + m * m)
        sn = np.exp(-(MT - m) / T) * (1 + 0.2 * np.cos(2 * ff))
        p = np.stack([pp * np.cos(ff), pp * np.sin(ff), np.zeros_like(pp)])
        Ss = np.stack([0.08 * np.sin(ff) + 0.01 * pp, -0.05 * np.cos(2 * ff) + 0.02, 0.03 * np.sin(ff) * pp]) * (1.0 if s else -0.5)
        if not spin:
            Ss = Ss * 0.0
        pS = (p * Ss).sum(0)
        sums["Snorm"][s::2] = sn.ravel()
        sums["St"][s::2] = (sn * pS / m).ravel()
        for c, k in enumerate(("Sx", "Sy", "Sz")):
            sums[k][s::2] = (sn * (Ss[c] + p[c] * pS / (m * (MT + m)))).ravel()
    return sums


@pytest.mark.parametrize("phi,partner_parity", [(np.pi, -1), (0.0, 1)])
def test_parity_conserving_limit_is_the_strong_law(phi, partner_parity):
    """(alpha, phi) = (0, pi) is the 1/2+ -> 1/2+ 0- law of the strong feed-down, (0, 0) its S-wave law (a 0+ partner): all five arrays
    agree with cfo_polarization_decays at 1e-13 of the conditioning."""
    g = _mini_grid()
    pw, sp = _mini_list(True); ps, sps = _mini_list(False, partner_parity)
    sums = _mini_sums(g, [pw["mass"][1], pw["mass"][2]])
    got, cond = fdw.polarization_weak_decays(pw, sp, _row(0.0, phi), [1, 2], g, 2, sums, conditioning=True)
    ref = fdo.polarization_decays(ps, sps, [1, 2], g, 2, sums)
    for k in FIELDS:
        assert np.all(np.abs(got[k] - ref[k]) <= 1e-13 * (cond[k] + np.abs(ref[k]))), k
    assert np.any(got["Sx"] != sums["Sx"]) and np.any(got["Snorm"] != sums["Snorm"])


def _slow_parent(alpha, phi, T=0.02):
    """Lambda fed by one cold Xi (Boltzmann spectrum, log-linear in M_T) with uniform rest-frame spin S*_P; returns the daughter's
    momentum-integrated rest-frame spin over S*_P, per axis (the construction of the strong feed-down test)."""
    pdg, spar = _mini_list(True)
    n_pT, n_phi = 160, 48
    pT = np.linspace(0.004, 2.2, n_pT); phi_t = (np.arange(n_phi) + 0.5) * 2 * np.pi / n_phi
    g = dict(pT=pT, phi=phi_t, phi_weight=np.full(n_phi, 2 * np.pi / n_phi), y=np.array([0.0]), eta=np.array([0.0]), eta_weight=np.array([1.0]))
    M = pdg["mass"][2]; m = pdg["mass"][1]
    res = []
    for axis in range(3):
        Sp = np.zeros(3); Sp[axis] = 0.1
        sums = {k: np.zeros(2 * n_pT * n_phi) for k in FIELDS}
        ff, pp = np.meshgrid(phi_t, pT, indexing="ij")
        MT = np.sqrt(pp * pp + M * M)
        sn = np.exp(-(MT - M) / T)
        p = np.stack([pp * np.cos(ff), pp * np.sin(ff), np.zeros_like(pp)])
        pS = (p * Sp[:, None, None]).sum(0)
        sums["Snorm"][1::2] = sn.ravel()
        sums["St"][1::2] = (sn * pS / M).ravel()
        for c, k in enumerate(("Sx", "Sy", "Sz")):
            sums[k][1::2] = (sn * (Sp[c] + p[c] * pS / (M * (MT + M)))).ravel()
        out = fdw.polarization_weak_decays(pdg, spar, _row(alpha, phi), [1, 2], g, 2, sums)
        d = {k: out[k][0::2].reshape(n_phi, n_pT) for k in FIELDS}
        mT = np.sqrt(pp * pp + m * m)
        w = pp * np.gradient(pT)[None, :]
        rest = [d[k] - d["St"] * p[c] / (mT + m) for c, k in enumerate(("Sx", "Sy", "Sz"))]
        res.append((w * rest[axis]).sum() / (w * d["Snorm"]).sum() / Sp[axis])
    return np.array(res)


def test_slow_parent_limit():
    """A cold Xi (T = 20 MeV) with uniform S*_P: the Lambda's momentum-integrated S* / S*_P is C = (1 + 2 gamma)/3 up to O((p*/m_Lambda)^2)
    = 1.6e-2 (Wigner rotations, the relativistic part of the spin four-vector) and O(T/M); the alpha/2 n and beta S x n parts average out."""
    pdg, _ = _mini_list(True)
    M, m, W = pdg["mass"][2], pdg["mass"][1], pdg["mass"][0]
    Estar = (M * M + m * m - W * W) / (2 * M); bar = (np.sqrt(Estar ** 2 - m * m) / m) ** 2
    for alpha, phi in ((-0.4, 0.6), (0.7, -2.0), (0.0, np.pi)):
        gamma = np.sqrt(1 - alpha ** 2) * np.cos(phi)
        got = _slow_parent(alpha, phi)
        C_want = (1 + 2 * gamma) / 3
        print("alpha", alpha, "phi", phi, "S*_D / S*_P per axis", got, "expected", C_want, "bar", bar)
        assert np.all(np.abs(got - C_want) <= bar), (alpha, phi, got, C_want)


# ---------------------------------------------------------------------------------------------------- problems
def _spin_inputs(dN, sp_mass, g, dimension, scale=1.0):
    y = np.zeros(len(g["y"])) if dimension == 2 else np.asarray(g["y"])
    yy, ff, pp, mm = np.meshgrid(y, g["phi"], g["pT"], np.asarray(sp_mass, float), indexing="ij")
    mT = np.sqrt(pp * pp + mm * mm); E = mT * np.cosh(yy)
    p = np.stack([pp * np.cos(ff), pp * np.sin(ff), mT * np.sinh(yy)])
    Ss = scale * np.stack([0.08 * np.sin(ff) + 0.01 * pp, -0.05 * np.cos(2 * ff) + 0.02, 0.03 * np.sin(ff) * pp - 0.01 * yy])
    pS = (p * Ss).sum(0)
    sn = np.asarray(dN, float)
    return dict(St=(pS / mm).ravel() * sn, Sx=(Ss[0] + p[0] * pS / (mm * (E + mm))).ravel() * sn,
                Sy=(Ss[1] + p[1] * pS / (mm * (E + mm))).ravel() * sn, Sz=(Ss[2] + p[2] * pS / (mm * (E + mm))).ravel() * sn, Snorm=sn.copy())


def _problem(fx, dimension):
    """the list of CHOSEN with thermal spectra, spin sums, and the strong feed-down (oracle) already applied"""
    strides = dict(pT=HI_PT, phi=3, y=1) if dimension == 2 else dict(pT=HI_PT, phi=4, y=[7, 9, 10, 11, 13])
    rec = dict(dimension=dimension, n_cells=30, seed=17, strides=strides, chosen=CHOSEN)
    g, tabs, cols, dN, pdg, idx = mdv.case_inputs(fx, rec)
    spar = tables.spin_parity(fx, pdg, 1)
    sums = fdo.polarization_decays(pdg, spar, idx, g, dimension, _spin_inputs(dN, [pdg["mass"][i] for i in idx], g, dimension))
    return g, pdg, idx, sums, spar


@pytest.fixture(scope="module")
def problems(fx):
    return {d: _problem(fx, d) for d in (2, 3)}


@pytest.fixture(scope="module")
def oracle_results(problems):
    return {d: fdw.polarization_weak_decays(pdg, spar, WEAK, idx, g, d, sums, conditioning=True) for d, (g, pdg, idx, sums, spar) in problems.items()}


@pytest.mark.parametrize("dimension", [2, 3])
def test_oracle_feeds_lambda_and_cascade(problems, oracle_results, dimension):
    g, pdg, idx, sums, spar = problems[dimension]
    out, _ = oracle_results[dimension]
    ns = len(CHOSEN); L = ns * len(g["pT"]) * len(g["phi"])
    for m in (3122, -3122):
        s = CHOSEN.index(m)
        for k in FIELDS:
            assert np.any(out[k][s:L:ns] != sums[k][s:L:ns]), (m, k)
    x0 = CHOSEN.index(3322)                                        # Omega -> Xi0 pi- (J = 3/2, no law) only dilutes
    assert np.any(out["Snorm"][x0:L:ns] != sums["Snorm"][x0:L:ns])
    for k in FIELDS[:4]:
        assert np.array_equal(out[k][x0::ns], sums[k][x0::ns])
    for m in (211, 321, -321, 3212, 3312, 3324, 3334):           # partners, strong parents and weak parents are not fed
        s = CHOSEN.index(m)
        for k in FIELDS:
            assert np.array_equal(out[k][s::ns], sums[k][s::ns]), (m, k)
    # the two-level cascade: without the Omega rows, Xi0 is not fed and Lambda gains less
    no_omega = {k: v[:4] for k, v in WEAK.items()}
    o2 = fdw.polarization_weak_decays(pdg, spar, no_omega, idx, g, dimension, sums)
    x0 = CHOSEN.index(3322)
    assert np.array_equal(o2["Snorm"][x0::ns], sums["Snorm"][x0::ns])
    lam = CHOSEN.index(3122)
    assert out["Snorm"][lam:L:ns].sum() > o2["Snorm"][lam:L:ns].sum()       # not bin by bin: the yield 1 + 2 alpha S.n depends on Xi0's S*


def test_oracle_exact_structure(problems):
    g, pdg, idx, sums, spar = problems[3]
    zeroN = dict(sums, **{k: np.zeros_like(sums["St"]) for k in ("St", "Sx", "Sy", "Sz")})
    # S*_P = 0: bit-identical for any phi at fixed alpha, N_D linear in alpha
    base = fdw.polarization_weak_decays(pdg, spar, WEAK, idx, g, 3, zeroN)
    other = fdw.polarization_weak_decays(pdg, spar, dict(WEAK, phi=[2.0, -1.0, 0.7, 3.0, 1.0, -2.0]), idx, g, 3, zeroN)
    for k in FIELDS:
        assert np.array_equal(base[k], other[k]), k
    half = fdw.polarization_weak_decays(pdg, spar, dict(WEAK, alpha=[0.5 * a for a in WEAK["alpha"]]), idx, g, 3, zeroN)
    for k in ("St", "Sx", "Sy", "Sz"):
        assert np.all(np.abs(2 * half[k] - base[k]) <= 1e-15 * np.abs(base[k]).max()), k
    assert np.any(base["Sx"] != 0.0)                                                   # the helicity of unpolarised parents
    # alpha = 0: Snorm bit-identical for any parent polarization
    a0 = dict(WEAK, alpha=[0.0] * 6)
    s1 = fdw.polarization_weak_decays(pdg, spar, a0, idx, g, 3, sums)
    s2 = fdw.polarization_weak_decays(pdg, spar, a0, idx, g, 3, zeroN)
    assert np.array_equal(s1["Snorm"], s2["Snorm"])
    # doubling the parents' N doubles N_D - N_D|N=0
    # to 1e-15 of the conditioning (every point's term carries the alpha/2 n part, which the subtraction of N_D|N=0 cancels) plus the
    # rounding of the subtractions of the arrays themselves
    full, cond = fdw.polarization_weak_decays(pdg, spar, WEAK, idx, g, 3, sums, conditioning=True)
    two = dict(sums, **{k: 2.0 * sums[k] for k in ("St", "Sx", "Sy", "Sz")})
    t, cond2 = fdw.polarization_weak_decays(pdg, spar, WEAK, idx, g, 3, two, conditioning=True)
    for k in ("St", "Sx", "Sy", "Sz"):
        d1 = (full[k] - sums[k]) - base[k]; d2 = (t[k] - two[k]) - base[k]
        sub = 8 * np.finfo(float).eps * (np.abs(two[k]) + np.abs(t[k]) + np.abs(full[k]) + np.abs(sums[k]) + np.abs(base[k]))
        assert np.all(np.abs(d2 - 2.0 * d1) <= 1e-15 * cond2[k] + sub), k
    # an empty table changes nothing
    empty = {k: [] for k in WEAK}
    e = fdw.polarization_weak_decays(pdg, spar, empty, idx, g, 3, sums)
    for k in FIELDS:
        assert np.array_equal(e[k], sums[k])
    # p.N_D = 0 within 1e-12 of the conditioning
    fd = {k: full[k] - sums[k] for k in FIELDS}
    ms = np.array([pdg["mass"][i] for i in idx])
    yy, ff, pp, mm = np.meshgrid(np.asarray(g["y"]), g["phi"], g["pT"], ms, indexing="ij")
    mT = np.sqrt(pp * pp + mm * mm)
    E, px, py, pz = (mT * np.cosh(yy)).ravel(), (pp * np.cos(ff)).ravel(), (pp * np.sin(ff)).ravel(), (mT * np.sinh(yy)).ravel()
    pdot = fd["St"] * E - fd["Sx"] * px - fd["Sy"] * py - fd["Sz"] * pz
    absterm = cond["St"] * E + (cond["Sx"] + cond["Sy"]) * pp.ravel() + cond["Sz"] * np.abs(pz)
    subtraction = 4 * np.finfo(float).eps * (np.abs(full["St"] * E) + np.abs(full["Sx"] * px) + np.abs(full["Sy"] * py) + np.abs(full["Sz"] * pz))
    assert np.all(np.abs(pdot) <= 1e-12 * absterm + subtraction)
    assert np.count_nonzero(absterm) > 0


# ---------------------------------------------------------------------------------------------------- reader, key, errors, layout
def test_weak_table_reader(tmp_path):
    f = tmp_path / "weak_decays.dat"
    f.write_text("# parent daughter partner br alpha phi\n\n3312 3122 -211 0.9989 -0.376 0.011   # Xi-\n  -3312 -3122 211 0.9989 0.376 -0.011\n")
    w = tables.weak_decays(str(f))
    assert list(w["parent"]) == [3312, -3312] and list(w["partner"]) == [-211, 211]
    assert np.array_equal(w["alpha"], [-0.376, 0.376]) and np.array_equal(w["phi"], [0.011, -0.011])
    f.write_text("3312 3122 -211 0.9989 -0.376\n")
    with pytest.raises(ValueError):
        tables.weak_decays(str(f))


def _mode5(fx, wd, **kw):
    from test_spin_polarization_shear import _materialize, _mode5_columns
    cols, _, _, _ = _mode5_columns(4, 31)
    _materialize(wd, fx, cols, **kw)


def test_host_layer_key_rules_reader_and_dump(fx):
    from test_spin_polarization_shear import _host_dump
    weak = {k: v[:2] for k, v in WEAK.items()}
    with tempfile.TemporaryDirectory() as wd:
        _mode5(fx, wd, spin_polarization=1, polarization_weak_decays=1, weak_decays=weak)
        rc, msg = _host_dump(wd)
        assert rc == 2 and "polarization_feed_down" in msg                               # IS3D_ERR_UNSUPPORTED
        _mode5(fx, wd, spin_polarization=1, polarization_feed_down=1, polarization_weak_decays=1, weak_decays=weak)
        rc, d = _host_dump(wd)
        assert rc == 0, d
        for k in ("parent", "daughter", "partner", "branching", "alpha", "phi"):
            assert np.array_equal(d["weak_" + k], np.asarray(weak[k], float)), k
        path = os.path.join(wd, "PDG", "weak_decays.dat")
        text = open(path).read()
        open(path, "w").write(text + "# a comment line\n\n3322 3122 111 0.99 -0.375 0.005 # trailing comment\n")
        rc, d = _host_dump(wd)
        assert rc == 0 and list(d["weak_parent"]) == [3312, -3312, 3322]
        for bad in ("3322 3122 111 0.99 -0.375\n", "3322 3122 111 0.99 -0.375 0.005 7\n", "3322 3122 pi0 0.99 -0.375 0.005\n"):
            open(path, "w").write(text + bad)
            rc, msg = _host_dump(wd)
            assert rc == 6 and "weak_decays.dat" in msg, bad                             # IS3D_ERR_IO
        os.remove(path)
        rc, msg = _host_dump(wd)
        assert rc == 6 and "weak_decays.dat" in msg
        _mode5(fx, wd, spin_polarization=1, polarization_feed_down=1, polarization_weak_decays=0)
        rc, d = _host_dump(wd)
        assert rc == 0 and not any(k.startswith("weak_") for k in d)


def test_struct_layout_matches_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "is3d_b200.h"\nint main(void) { printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", '
                   "sizeof(is3d_weak_decays), offsetof(is3d_weak_decays, parent), offsetof(is3d_weak_decays, daughter), "
                   "offsetof(is3d_weak_decays, partner), offsetof(is3d_weak_decays, branching), offsetof(is3d_weak_decays, alpha), "
                   "offsetof(is3d_weak_decays, phi), offsetof(is3d_weak_decays, n)); return 0; }\n")
    inc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include")
    exe = tmp_path / "layout"
    subprocess.check_call([fdo._compiler(), "-I", inc, "-o", str(exe), str(src)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    W = api.WeakDecays
    assert got == [C.sizeof(W), W.parent.offset, W.daughter.offset, W.partner.offset, W.branching.offset, W.alpha.offset, W.phi.offset, W.n.offset]


def _argument_errors(pdg, spar, idx, g, sums):
    """(label, weak table) pairs that is3d_b200_polarization_weak_decays rejects with IS3D_ERR_ARGUMENT"""
    def w(**kw):
        return dict(WEAK, **{k: list(v) for k, v in kw.items()})
    return [("unknown id", w(daughter=[3122, -3122, 3122, -3122, 3122, 99999])),
            ("mc id 0", w(partner=[-211, 211, 111, 111, -321, 0])),
            ("unstable parent", w(parent=[3312, -3312, 3322, -3322, 3334, 3212], daughter=[3122, -3122, 3122, -3122, 3122, 3122],
                                  partner=[-211, 211, 111, 111, -321, 22])),
            ("unstable daughter", w(daughter=[3122, -3122, 3122, -3122, 3122, 3212], partner=[-211, 211, 111, 111, -321, 111])),
            ("branching < 0", w(branching=[0.999, 0.999, 0.995, 0.995, 0.68, -0.1])),
            ("branching > 1", w(branching=[0.999, 1.5, 0.995, 0.995, 0.68, 0.24])),
            ("branching sum > 1", w(branching=[0.999, 0.999, 0.995, 0.995, 0.68, 0.4])),
            ("|alpha| > 1", w(alpha=[-0.41, 0.37, -0.33, 1.01, 0.02, 0.05])),
            ("alpha nan", w(alpha=[-0.41, 0.37, float("nan"), 0.35, 0.02, 0.05])),
            ("phi inf", w(phi=[0.3, -0.25, 0.12, float("inf"), 0.0, 0.0])),
            ("closed channel", w(parent=[3312, -3312, 3322, -3322, 3334, 3322], daughter=[3122, -3122, 3122, -3122, 3122, 3122],
                                 partner=[-211, 211, 111, 111, -321, 321]))]


def test_argument_errors_without_device(problems):
    """the table checks run on the host before any device work, so they hold on a machine without a GPU too"""
    g, pdg, idx, sums, spar = problems[2]
    for label, bad in _argument_errors(pdg, spar, idx, g, sums):
        with pytest.raises(api.Is3dError) as e:
            api.polarization_weak_decays(pdg, spar, bad, idx, g, 2, sums)
        assert e.value.code == 1, label
    for label, args in (("NULL table", dict(weak=None)), ("NULL spin table", dict(spin_parity=None))):
        kw = dict(spin_parity=spar, weak=WEAK); kw.update(args)
        with pytest.raises(api.Is3dError) as e:
            api.polarization_weak_decays(pdg, kw["spin_parity"], kw["weak"], idx, g, 2, sums)
        assert e.value.code == 1, label
    neg = api.WeakDecays(); neg.n = -1
    f = api.lib().is3d_b200_polarization_weak_decays
    keep = []
    p, gg, ia = api._decay_problem(pdg, g, keep)
    sp = api.SpinParity(); sp.spin2 = ia(spar["spin2"]); sp.parity = ia(spar["parity"])
    arrs = {k: np.array(sums[k], copy=True) for k in FIELDS}
    res = api.PolarizationResult(**{k: arrs[k].ctypes.data_as(C.POINTER(C.c_double)) for k in FIELDS})
    rc = f(C.byref(p), C.byref(sp), C.byref(neg), len(idx), ia(idx), C.byref(gg), 2, None, C.byref(res), None)
    assert rc == 1


# ---------------------------------------------------------------------------------------------------- GPU tier
def _gpu_compare(got, ref, cond):
    """1e-10 per bin of the oracle's conditioning (sum of |term| x (1 + |log dN|), St..Sz with the largest component of each point's
    four-vector) plus |ref|"""
    for k in FIELDS:
        r = compare(np.asarray(got[k]), ref[k], conditioning=cond[k] + np.abs(ref[k]))
        print(k, "max deviation / conditioning %.3g" % r["max_rel"])
        assert r["ok"], (k, r)


@pytest.mark.gpu
@pytest.mark.parametrize("dimension", [2, 3])
def test_cuda_matches_oracle(problems, oracle_results, dimension):
    import torch
    api.init()
    g, pdg, idx, sums, spar = problems[dimension]
    ref, cond = oracle_results[dimension]
    got, st = api.polarization_weak_decays(pdg, spar, WEAK, idx, g, dimension, sums)
    print("dim", dimension, "kernel ms %.2f" % st["kernel_ms"], "launches", st["gpu_launches"])
    _gpu_compare(got, ref, cond)
    again, _ = api.polarization_weak_decays(pdg, spar, WEAK, idx, g, dimension, sums)
    for k in FIELDS:
        assert np.array_equal(again[k], got[k])
    t = {k: torch.tensor(sums[k], device="cuda") for k in FIELDS}
    res, _ = api.polarization_weak_decays(pdg, spar, WEAK, idx, g, dimension, t, memory="device")
    torch.cuda.synchronize()
    assert res is t
    for k in FIELDS:
        assert np.array_equal(t[k].cpu().numpy(), got[k])
    e, _ = api.polarization_weak_decays(pdg, spar, {k: [] for k in WEAK}, idx, g, dimension, sums)
    for k in FIELDS:
        assert np.array_equal(e[k], sums[k])


@pytest.mark.gpu
def test_cuda_strong_then_weak_on_device(fx):
    """the two passes in order on the GPU (strong pass of the library, then the weak pass) against the oracle's two passes"""
    api.init()
    strides = dict(pT=HI_PT, phi=3, y=1)
    rec = dict(dimension=2, n_cells=30, seed=17, strides=strides, chosen=CHOSEN)
    g, tabs, cols, dN, pdg, idx = mdv.case_inputs(fx, rec)
    spar = tables.spin_parity(fx, pdg, 1)
    primary = _spin_inputs(dN, [pdg["mass"][i] for i in idx], g, 2)
    strong, _ = api.polarization_decays(pdg, spar, idx, g, 2, primary)
    got, _ = api.polarization_weak_decays(pdg, spar, WEAK, idx, g, 2, strong)
    # the oracle's weak pass on the library's strong output: the strong pass itself is checked by test_polarization_decays
    ref, cond = fdw.polarization_weak_decays(pdg, spar, WEAK, idx, g, 2, strong, conditioning=True)
    _gpu_compare(got, ref, cond)


@pytest.mark.gpu
def test_cuda_errors_leave_arrays_untouched(problems):
    import torch
    api.init()
    g, pdg, idx, sums, spar = problems[3]
    t = {k: torch.tensor(sums[k], device="cuda") for k in FIELDS}
    before = {k: v.clone() for k, v in t.items()}
    for label, bad in _argument_errors(pdg, spar, idx, g, sums):
        with pytest.raises(api.Is3dError) as e:
            api.polarization_weak_decays(pdg, spar, bad, idx, g, 3, t, memory="device")
        assert e.value.code == 1, label
    # a weak parent whose tail fit has fewer than 2 points: Omega's spectrum is 0 beyond the first pT points
    ns = len(CHOSEN); n_pT = len(g["pT"])
    t["Snorm"].view(-1, n_pT, ns)[:, 3:, CHOSEN.index(3334)] = 0.0
    before = {k: v.clone() for k, v in t.items()}
    with pytest.raises(api.Is3dError) as e:
        api.polarization_weak_decays(pdg, spar, WEAK, idx, g, 3, t, memory="device")
    assert e.value.code == 1
    torch.cuda.synchronize()
    for k in FIELDS:
        assert torch.equal(t[k], before[k])


@pytest.mark.gpu
@pytest.mark.parametrize("phi,partner_parity", [(np.pi, -1), (0.0, 1)])
def test_cuda_parity_conserving_limit(phi, partner_parity):
    """(alpha, phi) = (0, pi) and (0, 0) on the GPU against is3d_b200_polarization_decays with the strong channel: the two paths sum in
    different orders, so within 1e-13 of the conditioning rather than bit for bit"""
    api.init()
    g = _mini_grid()
    pw, sp = _mini_list(True); ps, sps = _mini_list(False, partner_parity)
    sums = _mini_sums(g, [pw["mass"][1], pw["mass"][2]])
    got, _ = api.polarization_weak_decays(pw, sp, _row(0.0, phi), [1, 2], g, 2, sums)
    ref, _ = api.polarization_decays(ps, sps, [1, 2], g, 2, sums)
    _, cond = fdw.polarization_weak_decays(pw, sp, _row(0.0, phi), [1, 2], g, 2, sums, conditioning=True)
    for k in FIELDS:
        assert np.all(np.abs(got[k] - ref[k]) <= 1e-13 * (cond[k] + np.abs(ref[k]))), k


@pytest.mark.gpu
@pytest.mark.parametrize("dimension", [3, 2])
def test_gpu_workdir_weak_decay_files(fx, dimension):
    """With the key: S_fdw_<mcid>.dat holds api.mean_spin of direct calls (strong pass, then weak pass); S_, S_fd_ are byte-identical with
    and without the key; a run without the key (absent or 0) writes exactly the files it wrote before."""
    from is3d_b200 import synthetic
    from test_spin_polarization_shear import _mode5_columns, _run
    api.init()
    cols, base, vort, xi = _mode5_columns(60, 9311 + dimension, dimension)
    chosen = [211, -211, 111, 3122, -3122, 3212, 3312, -3312, 3322, 3334]
    weak = {k: [v for v, p, d in zip(WEAK[k], WEAK["parent"], WEAK["daughter"]) if p in chosen and d in chosen] for k in WEAK}
    runs = {}
    for label, extra in (("absent", {}), ("zero", dict(polarization_weak_decays=0)), ("on", dict(polarization_weak_decays=1))):
        with tempfile.TemporaryDirectory() as wd:
            workdir.materialize(wd, surface_columns=cols, chosen=chosen, fixture=fx, operation=1, mode=5, dimension=dimension, df_mode=1,
                                spin_polarization=1, polarization_feed_down=1, weak_decays=weak, **extra)
            open(os.path.join(wd, "average_thermodynamic_quantities.dat"), "w").write("0.15\n0.3\n0.05\n0\n0")
            runs[label] = _run(wd)
    assert runs["absent"][0] == runs["zero"][0]
    assert not any("S_fdw_" in f for f in runs["absent"][0])
    fdw_files = ["polarization" + os.sep + "S_fdw_%d.dat" % c for c in chosen]
    assert runs["on"][0] == sorted(runs["absent"][0] + fdw_files)
    for f, text in runs["absent"][1].items():
        assert runs["on"][1][f] == text == runs["zero"][1][f], f
    header = runs["on"][1][fdw_files[0]].decode().split("\n", 1)[0].split()
    assert header == ["y", "phip", "pT", "Snorm", "St", "Sx", "Sy", "Sz", "Sx_rest", "Sy_rest", "Sz_rest"]

    cells = synthetic.columns_to_cells(base, 1)
    sp = tables.species(fx, 1, chosen); g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=dimension)
    total, _ = api.spin_polarization(fl, cells, vort, sp, g)
    pdg = tables.pdg_decay_table(fx, 1)
    first = {}
    for n, m in enumerate(pdg["mcid"]):
        first.setdefault(int(m), n)
    idx = [first[m] for m in chosen]
    spar = tables.spin_parity(fx, pdg, 1)
    fed, _ = api.polarization_decays(pdg, spar, idx, g, dimension, total)
    fedw, _ = api.polarization_weak_decays(pdg, spar, weak, idx, g, dimension, fed)
    S, rest = api.mean_spin(fedw, sp, g, dimension)
    ny = 1 if dimension == 2 else len(g["y"])
    shape = (len(g["y"]), len(g["phi"]), len(g["pT"]), -1)
    lam = chosen.index(3122)
    assert np.any(fedw["Sx"].reshape(shape)[:ny, :, :, lam] != fed["Sx"].reshape(shape)[:ny, :, :, lam])
    for s, f in enumerate(fdw_files):
        got = np.loadtxt(runs["on"][1][f].decode().splitlines(), skiprows=1, ndmin=2)[:, 3:]
        want = np.column_stack([v.reshape(shape)[:ny, :, :, s].ravel() for v in [fedw["Snorm"]] + list(S) + list(rest)])
        assert got.shape == want.shape
        scale = np.abs(want).max(axis=0)
        assert np.all(np.abs(got - want) <= 2e-8 * np.abs(want) + 1e-12 * scale), f
