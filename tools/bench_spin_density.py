"""Throughput of the spin-density path (is3d_b200_spin_density, cf_spin_density_kernel) next to the vorticity polarization path
(cf_polzn_kernel) on the same surface and species, in the same process.

Seeded 1M-cell 3+1D surface (the cfg3 generator) with synthetic thermal vorticity, the full 32 pT x 24 phi x 21 y grid, surface arrays
resident on the GPU (memory = device), two species lists: the vector mesons and hyperons that spin-alignment and polarization users
run (K*0, anti-K*0, phi(1020), Lambda, anti-Lambda, Omega-, anti-Omega+) and the 305-species list of the headline benchmark.  One
warm-up call, then the median of --steps timed calls.  Prints one JSON line with kernel and call times and evaluations/s of both paths
(CUDA events of the library; the call time also by host clock around synchronised calls) and the GPU's name, power limit and maximum SM
clock, read in the same process.

    python tools/bench_spin_density.py [--cells N] [--steps K] [--warmup W]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_polarization_shear import gpu_identity, timed  # noqa: E402

VECTOR_AND_HYPERONS = [313, -313, 333, 3122, -3122, 3334, -3334]


def rates(r):
    return dict(kernel_ms=r["kernel_ms"], call_ms=r["call_ms"], wall_ms=r["wall_s"] * 1e3,
                kernel_evals_per_s=r["evaluations"] / (r["kernel_ms"] * 1e-3), call_evals_per_s=r["evaluations"] / r["wall_s"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    if args.steps < 2:
        raise SystemExit("--steps must be >= 2")
    import torch
    from is3d_b200 import api, synthetic, tables
    if not torch.cuda.is_available():
        raise SystemExit("bench_spin_density needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(0)
    api.init()
    fx = tables.load_fixture()
    cells = synthetic.columns_to_cells(synthetic.surface_vh(args.cells, synthetic.SEEDS["cfg3"], three_d=True), 1)
    vort = synthetic.vorticity(args.cells, synthetic.SEEDS["cfg3"] + 1)
    dc = {k: torch.tensor(v, device="cuda") for k, v in cells.items()}
    dv = {k: torch.tensor(v, device="cuda") for k, v in vort.items()}
    g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=3)
    out = dict(workload="%d-cell 3+1D mode-5 surface, %d pT x %d phi x %d y, surface on the device" % (args.cells, len(g["pT"]), len(g["phi"]), len(g["y"])),
               steps=args.steps, warmup=args.warmup, gpu=gpu_identity(torch), lists={})
    for label, chosen in (("vector_mesons_hyperons", VECTOR_AND_HYPERONS), ("pdg305", "chosen_urqmd")):
        sp = tables.species(fx, 1, chosen)
        sd = timed(lambda: api.spin_density(fl, dc, dv, sp, g, memory="device")[1], args.steps, args.warmup, torch)
        vor = timed(lambda: api.spin_polarization(fl, dc, dv, sp, g, memory="device")[1], args.steps, args.warmup, torch)
        out["lists"][label] = dict(species=len(sp["mass"]), evaluations_per_call=sd["evaluations"],
                                   cf_spin_density_kernel=rates(sd), cf_polzn_kernel=rates(vor),
                                   spin_density_over_polzn_kernel_time=sd["kernel_ms"] / vor["kernel_ms"])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
