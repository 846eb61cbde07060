"""Time of the polarization feed-down (is3d_b200_polarization_decays) next to the spectra feed-down (is3d_b200_resonance_decays) on the same
particle list and grid.

The 150-species prefix of the urqmd chosen list (the list of DESIGN §12), the full 32 pT x 24 phi x 21 y grid, thermal spectra from the
GPU spectra path on a seeded 3+1D surface; the four spin sums are Snorm times the four-vector of a smooth rest-frame spin field.  Both
calls work on device arrays (memory = device).  Times are the CUDA events of the library (kernel = the feed-down between the copies in
and out, call = the whole entry point).  2+1D uses the y = 0 plane only, as the reference does; 3+1D is reported when every parent of
the list has the two tail-fit points the feed-down needs, and as an error string otherwise.  Prints one JSON line with the GPU's name
and power limit, read in the same process.

    python tools/bench_polarization_decays.py [--species N] [--steps K] [--warmup W]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from bench_polarization_shear import gpu_identity  # noqa: E402

FIELDS = ("St", "Sx", "Sy", "Sz", "Snorm")


def spin_sums(dN, mass, g, dimension):
    y = np.zeros(len(g["y"])) if dimension == 2 else np.asarray(g["y"])
    yy, ff, pp, mm = np.meshgrid(y, g["phi"], g["pT"], np.asarray(mass, float), indexing="ij")
    mT = np.sqrt(pp * pp + mm * mm); E = mT * np.cosh(yy)
    p = np.stack([pp * np.cos(ff), pp * np.sin(ff), mT * np.sinh(yy)])
    Ss = np.stack([0.08 * np.sin(ff) + 0.01 * pp, -0.05 * np.cos(2 * ff) + 0.02, 0.03 * np.sin(ff) * pp - 0.01 * yy])
    pS = (p * Ss).sum(0)
    N = [pS / mm] + [Ss[c] + p[c] * pS / (mm * (E + mm)) for c in range(3)]
    return {k: N[i].ravel() * dN for i, k in enumerate(FIELDS[:4])} | dict(Snorm=np.array(dN, copy=True))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--species", type=int, default=150)
    ap.add_argument("--cells", type=int, default=20000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    import torch
    from is3d_b200 import api, synthetic, tables
    if not torch.cuda.is_available():
        raise SystemExit("bench_polarization_decays needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(0)
    api.init()
    fx = tables.load_fixture()
    chosen = [int(v) for v in fx["chosen_urqmd"]][:args.species]
    pdg = tables.pdg_decay_table(fx, 1)
    spar = tables.spin_parity(fx, pdg, 1)
    first = {}
    for n, m in enumerate(pdg["mcid"]):
        first.setdefault(int(m), n)
    idx = [first[m] for m in chosen]
    sp = tables.species(fx, 1, chosen)
    g = tables.grid(fx)
    out = dict(workload="%d-species urqmd prefix, %d pT x %d phi x %d y" % (len(chosen), len(g["pT"]), len(g["phi"]), len(g["y"])),
               steps=args.steps, gpu=gpu_identity(torch), dimensions={})
    for dim in (2, 3):
        cells = synthetic.columns_to_cells(synthetic.surface_vh(args.cells, synthetic.SEEDS["cfg3"], three_d=(dim == 3)), 1)
        dN, _ = api.smooth_spectra(tables.flags(df_mode=1, dimension=dim), cells, sp, g, tables.df_tables(fx, 1), tables.laguerre(fx))
        sums = spin_sums(dN, sp["mass"], g, dim)
        dev = {k: torch.tensor(v, device="cuda") for k, v in sums.items()}

        def run_pol():
            work = {k: v.clone() for k, v in dev.items()}
            return api.polarization_decays(pdg, spar, idx, g, dim, work, memory="device")[1]

        def run_dec():
            work = dev["Snorm"].clone()
            return api.resonance_decays(pdg, idx, g, dim, work, memory="device")[1]
        try:
            res = {}
            for label, fn in (("polarization_decays", run_pol), ("resonance_decays", run_dec)):
                for _ in range(args.warmup):
                    fn()
                st = [fn() for _ in range(args.steps)]
                res[label] = dict(kernel_ms=float(np.median([s["kernel_ms"] for s in st])), call_ms=float(np.median([s["total_ms"] for s in st])),
                                  launches=int(st[-1]["gpu_launches"]))
            res["polarization_over_spectra_kernel_time"] = res["polarization_decays"]["kernel_ms"] / res["resonance_decays"]["kernel_ms"]
            out["dimensions"][str(dim)] = res
        except api.Is3dError as e:
            out["dimensions"][str(dim)] = dict(error=str(e))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
