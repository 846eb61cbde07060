"""In-memory versions of the small input tables (species list, momentum grid, delta-f coefficient rows, Laguerre
nodes) built from the numeric fixture, for callers that drive the C ABI directly (bench.py, tests) instead of going
through an iS3D working directory.  The C++ host layer (csrc/host_io.cpp) produces the same tables from the text
files; tests/test_host_layer.py checks the two against each other.

Species bookkeeping mirrors the reference: anti-baryons are synthesised right after each baryon
(readindata.cpp:1491-1536), sign = -1 for even baryon number (:1541-1546), chosen species keep the order of the
chosen-particles file (emissionfunction.cpp:336-351), optional mass bubble sort (:354-369).
"""
import numpy as np

from . import workdir

_PDG_KEY = {1: "pdg_urqmd", 2: "pdg_smash", 3: "pdg_box"}


def pdg_table(fx, hrg_eos):
    """Full particle list incl. synthesised anti-particles: dict of arrays mcid, mass, gspin, baryon, sign."""
    key = _PDG_KEY[hrg_eos]
    mcid, mass, gspin, baryon, sign = [], [], [], [], []
    if hrg_eos in (1, 2):
        for i in range(len(fx[key + "/mcid"])):
            b = int(fx[key + "/baryon"][i])
            rows = [(int(fx[key + "/mcid"][i]), b)]
            if b > 0:
                rows.append((-rows[0][0], -b))
            for m, bb in rows:
                mcid.append(m); mass.append(float(fx[key + "/mass"][i])); gspin.append(int(fx[key + "/gspin"][i]))
                baryon.append(bb); sign.append(-1 if bb % 2 == 0 else 1)
    else:
        # SMASH box list: quantum numbers decoded from the MC id digits (readindata.cpp:1201-1424)
        for i in range(len(fx[key + "/name"])):
            for m in fx[key + "/mcid"][i]:
                m = int(m)
                if m == 0:
                    continue
                d = [(abs(m) // 10 ** k) % 10 for k in range(10)]
                nJ, nq3, nq2, nq1 = d[0] + d[7], d[1], d[2], d[3]
                is_baryon = nq1 != 0
                b = 1 if is_baryon else 0
                g = nJ
                s = 1 if is_baryon else -1
                has_anti = (b != 0) or (nq2 != nq3)
                for mm, bb in ([(m, b), (-m, -b)] if has_anti else [(m, b)]):
                    mcid.append(mm); mass.append(float(fx[key + "/mass"][i])); gspin.append(g); baryon.append(bb); sign.append(s)
    return dict(mcid=np.array(mcid, dtype=np.int64), mass=np.array(mass), gspin=np.array(gspin, dtype=np.int64),
                baryon=np.array(baryon, dtype=np.int64), sign=np.array(sign, dtype=np.int64))


def pdg_decay_table(fx, hrg_eos):
    """The reference's particle_info array incl. decay channels (readindata.cpp:1440-1568, hrg_eos 1 / 2): anti-baryons right behind
    their baryon with the daughters' ids negated unless the daughter is a neutral non-strange meson (:1512-1530); `stable` when the
    first channel has one product (:1487-1488).  Channels are flattened: rows dec_first[i] .. dec_first[i] + decays[i]."""
    key = _PDG_KEY[hrg_eos]
    g = lambda k: fx["%s/%s" % (key, k)]
    owner = g("dec_owner"); dn = g("dec_n"); br = g("dec_br"); parts = g("dec_parts")
    first = np.searchsorted(owner, np.arange(len(g("mcid"))))
    out = dict(mcid=[], mass=[], width=[], baryon=[], charge=[], strange=[], stable=[], decays=[], dec_first=[], dec_npart=[], dec_br=[], dec_part=[])

    def push(mcid, i, b, q, s, chans):
        out["mcid"].append(int(mcid)); out["mass"].append(float(g("mass")[i])); out["width"].append(float(g("width")[i]))
        out["baryon"].append(b); out["charge"].append(q); out["strange"].append(s)
        out["stable"].append(1 if (chans and chans[0][0] == 1) else 0)
        out["decays"].append(len(chans)); out["dec_first"].append(len(out["dec_npart"]))
        for n_, b_, p_ in chans:
            out["dec_npart"].append(int(n_)); out["dec_br"].append(float(b_)); out["dec_part"].append([int(v) for v in p_])

    for i in range(len(g("mcid"))):
        chans = [(int(dn[j]), float(br[j]), [int(v) for v in parts[j]]) for j in range(first[i], first[i] + int(g("decays")[i]))]
        b, q, s = int(g("baryon")[i]), int(g("charge")[i]), int(g("strange")[i])
        push(g("mcid")[i], i, b, q, s, chans)
        if b > 0:
            anti = []
            for n_, b_, p_ in chans:
                pp = []
                for v in p_:
                    if v == 0:
                        pp.append(0); continue
                    try:
                        idx = out["mcid"].index(v)                       # first match among the particles read so far
                        neutral = out["baryon"][idx] == 0 and out["charge"][idx] == 0 and out["strange"][idx] == 0
                    except ValueError:
                        neutral = False                                  # the reference reads one past the list here
                    pp.append(v if neutral else -v)
                anti.append((n_, b_, pp))
            push(-int(g("mcid")[i]), i, -b, -q, -s, anti)
    return {k: np.asarray(v) for k, v in out.items()}


def box_parities(fx):
    """Intrinsic parity by |MC id| from the SMASH box list (PDG/pdg_box.dat, the column read_pdg_smash_box parses): {|mcid|: +1 / -1}."""
    out = {}
    for i in range(len(fx["pdg_box/name"])):
        p = str(fx["pdg_box/parity"][i])
        for m in fx["pdg_box/mcid"][i]:
            if int(m) != 0 and p in "+-":
                out.setdefault(abs(int(m)), 1 if p == "+" else -1)
    return out


def spin_parity(fx, pdg, hrg_eos=1):
    """The is3d_spin_parity table of a particle list pdg (tables.pdg_decay_table order): spin2 = 2J = gspin - 1 of the list, parity
    from PDG/pdg_box.dat by |MC id| (charge conjugation keeps the product of parities of a decay), 0 for an id the box list lacks."""
    key = _PDG_KEY[hrg_eos]
    gspin = {abs(int(m)): int(g) for m, g in zip(fx[key + "/mcid"], fx[key + "/gspin"])}
    par = box_parities(fx)
    spin2 = np.array([gspin[abs(int(m))] - 1 for m in pdg["mcid"]], dtype=np.int32)
    parity = np.array([par.get(abs(int(m)), 0) for m in pdg["mcid"]], dtype=np.int32)
    return dict(spin2=spin2, parity=parity)


def weak_decays(path):
    """Read a weak-decay table (PDG/weak_decays.dat, this project's own format): one channel per line, `parent_mcid daughter_mcid
    partner_mcid branching alpha phi` (phi in radians), `#` starts a comment.  Returns the dict of the six columns that
    api.polarization_weak_decays takes; a malformed line raises ValueError (the host layer's IS3D_ERR_IO)."""
    cols = {k: [] for k in ("parent", "daughter", "partner", "branching", "alpha", "phi")}
    with open(path) as f:
        for n, line in enumerate(f, 1):
            tok = line.split("#", 1)[0].split()
            if not tok:
                continue
            if len(tok) != 6:
                raise ValueError("%s:%d: expected 6 columns, found %d" % (path, n, len(tok)))
            ids = [int(t) for t in tok[:3]]
            vals = [float(t) for t in tok[3:]]
            for k, v in zip(cols, ids + vals):
                cols[k].append(v)
    return dict(parent=np.array(cols["parent"], np.int32), daughter=np.array(cols["daughter"], np.int32),
                partner=np.array(cols["partner"], np.int32), branching=np.array(cols["branching"]), alpha=np.array(cols["alpha"]),
                phi=np.array(cols["phi"]))


def species(fx, hrg_eos=1, chosen="chosen_urqmd", group_particles=False):
    pdg = pdg_table(fx, hrg_eos)
    ids = fx[chosen] if isinstance(chosen, str) else np.asarray(chosen, dtype=np.int64)
    first = {}
    for n, m in enumerate(pdg["mcid"]):
        first.setdefault(int(m), n)
    idx = [first[int(m)] for m in ids]          # KeyError if a chosen id is absent (the reference leaves garbage there)
    if group_particles:
        idx = list(idx)
        for m in range(len(idx)):
            for n in range(len(idx) - m - 1):
                if pdg["mass"][idx[n]] > pdg["mass"][idx[n + 1]]:
                    idx[n], idx[n + 1] = idx[n + 1], idx[n]
    idx = np.array(idx, dtype=np.int64)
    return dict(mcid=pdg["mcid"][idx].copy(), mass=pdg["mass"][idx].copy(),
                sign=pdg["sign"][idx].astype(np.float64), degeneracy=pdg["gspin"][idx].astype(np.float64),
                baryon=pdg["baryon"][idx].astype(np.float64))


def grid(fx, tables=None):
    t = tables or {}
    pT = np.asarray(t.get("pT", fx["pT_tab"])); phi = np.asarray(t.get("phi", fx["phi_tab"]))
    y = np.asarray(t.get("y", fx["y_tab"])); eta = np.asarray(t.get("eta", fx["eta_tab"]))
    return dict(pT=pT[:, 0].copy(), pT_weight=pT[:, 1].copy(), phi=phi[:, 0].copy(), phi_weight=phi[:, 1].copy(),
                y=y[:, 0].copy(), y_weight=y[:, 1].copy(), eta=eta[:, 0].copy(), eta_weight=eta[:, 1].copy())


def df_tables(fx, hrg_eos=1):
    eos = {1: "urqmd", 2: "smash", 3: "smash_box"}[hrg_eos]
    out = {k: fx["df_%s/%s" % (eos, k)].copy() for k in ("T", "c0", "c1", "c2", "c3", "c4", "F", "G", "betabulk", "betaV", "betapi")}
    out["jonah_x"] = None
    return out


def laguerre(fx):
    return dict(root1=fx["gla_root"][1].copy(), weight1=fx["gla_weight"][1].copy(),
                root2=fx["gla_root"][2].copy(), weight2=fx["gla_weight"][2].copy())


def flags(df_mode=1, dimension=3, include_baryon=0, include_bulk=1, include_shear=1, include_diff=0,
          regulate_deltaf=1, outflow=1, deta_min=1.0e-5, mass_pion0=0.138):
    return dict(df_mode=df_mode, dimension=dimension, include_baryon=include_baryon, include_bulk=include_bulk,
                include_shear=include_shear, include_diff=include_diff, regulate_deltaf=regulate_deltaf, outflow=outflow,
                deta_min=deta_min, mass_pion0=mass_pion0)


load_fixture = workdir.load_fixture
