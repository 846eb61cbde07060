"""Time of the weak-decay polarization feed-down (is3d_b200_polarization_weak_decays) next to the strong one (is3d_b200_polarization_decays)
on the same particle list and grid.

The 150-species prefix of the urqmd chosen list (DESIGN §17; it contains Lambda, Xi-, Xi0 and Omega-), the full 32 pT x 24 phi x 21 y
grid, thermal spectra from the GPU spectra path on a seeded surface, spin sums from tools/bench_polarization_decays.py, and a weak table
with test values of (alpha, phi) for the Xi and Omega channels of DESIGN §20.  The weak pass runs on the output of the strong pass.  Both
calls work on device arrays; times are the CUDA events of the library, one warm-up and the median of 3 calls.  Prints one JSON line with
the GPU's name, power limit and maximum SM clock, read in the same process.

    python tools/bench_polarization_weak_decays.py [--species N] [--steps K] [--warmup W]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from bench_polarization_decays import spin_sums  # noqa: E402
from bench_polarization_shear import gpu_identity  # noqa: E402

WEAK = dict(parent=[3312, -3312, 3322, -3322, 3334, 3334, 3334, -3334, -3334, -3334],
            daughter=[3122, -3122, 3122, -3122, 3122, 3322, 3312, -3122, -3322, -3312],
            partner=[-211, 211, 111, 111, -321, -211, 111, 321, 211, 111],
            branching=[0.999, 0.999, 0.995, 0.995, 0.678, 0.236, 0.086, 0.678, 0.236, 0.086],
            alpha=[-0.38, 0.38, -0.37, 0.37, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0], phi=[0.01, -0.01, 0.005, -0.005, 0, 0, 0, 0, 0, 0])


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
        raise SystemExit("bench_polarization_weak_decays needs a CUDA device (there is no CPU fallback)")
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
    keep = [r for r in range(len(WEAK["parent"])) if WEAK["parent"][r] in chosen and WEAK["daughter"][r] in chosen]
    weak = {k: [v[r] for r in keep] for k, v in WEAK.items()}
    out = dict(workload="%d-species urqmd prefix, %d pT x %d phi x %d y, %d weak rows with a chosen parent and daughter"
               % (len(chosen), len(g["pT"]), len(g["phi"]), len(g["y"]), len(keep)), steps=args.steps, gpu=gpu_identity(torch), dimensions={})
    for dim in (2, 3):
        cells = synthetic.columns_to_cells(synthetic.surface_vh(args.cells, synthetic.SEEDS["cfg3"], three_d=(dim == 3)), 1)
        dN, _ = api.smooth_spectra(tables.flags(df_mode=1, dimension=dim), cells, sp, g, tables.df_tables(fx, 1), tables.laguerre(fx))
        dev = {k: torch.tensor(v, device="cuda") for k, v in spin_sums(dN, sp["mass"], g, dim).items()}
        try:
            api.polarization_decays(pdg, spar, idx, g, dim, dev, memory="device")          # the weak pass runs on the strong pass's output

            def run_weak():
                work = {k: v.clone() for k, v in dev.items()}
                return api.polarization_weak_decays(pdg, spar, weak, idx, g, dim, work, memory="device")[1]

            def run_strong():
                work = {k: v.clone() for k, v in dev.items()}
                return api.polarization_decays(pdg, spar, idx, g, dim, work, memory="device")[1]
            res = {}
            for label, fn in (("polarization_weak_decays", run_weak), ("polarization_decays", run_strong)):
                for _ in range(args.warmup):
                    fn()
                st = [fn() for _ in range(args.steps)]
                res[label] = dict(kernel_ms=float(np.median([s["kernel_ms"] for s in st])), call_ms=float(np.median([s["total_ms"] for s in st])),
                                  launches=int(st[-1]["gpu_launches"]))
            res["weak_over_strong_kernel_time"] = res["polarization_weak_decays"]["kernel_ms"] / res["polarization_decays"]["kernel_ms"]
            out["dimensions"][str(dim)] = res
        except api.Is3dError as e:
            out["dimensions"][str(dim)] = dict(error=str(e))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
