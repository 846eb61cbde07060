"""Throughput of the HBT-moment path (is3d_b200_hbt_moments) next to the spectra (is3d_b200_smooth_spectra) on the same surface.

Seeded 1M-cell 3+1D viscous surface (the cfg3 generator), df_mode 1 with shear and bulk delta-f, the full 32 pT x 24 phi x 21 y grid,
surface arrays resident on the GPU (memory = device), two species lists: pi / K / p (what HBT analyses run) and the 305-species list
of the headline benchmark (comparable with bench.py).  Prints one JSON line with the kernel time and evaluations/s of both paths (CUDA
events of the library, kernel and whole call), their ratio, and the GPU's name and power limit, read in the same process.

    python tools/bench_hbt.py [--cells N] [--steps K] [--warmup W]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_polarization import gpu_identity, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    import torch
    from is3d_b200 import api, synthetic, tables
    if not torch.cuda.is_available():
        raise SystemExit("bench_hbt needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(0)
    api.init()
    fx = tables.load_fixture()
    cells = synthetic.columns_to_cells(synthetic.surface_vh(args.cells, synthetic.SEEDS["cfg3"], three_d=True), 1)
    dc = {k: torch.tensor(v, device="cuda") for k, v in cells.items()}
    g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=3)
    tab = tables.df_tables(fx, 1)
    out = dict(workload="%d-cell 3+1D surface, df_mode 1, %d pT x %d phi x %d y" % (args.cells, len(g["pT"]), len(g["phi"]), len(g["y"])),
               steps=args.steps, gpu=gpu_identity(torch), lists={})
    for label, chosen in (("pi_K_p", [211, 321, 2212]), ("pdg305", "chosen_urqmd")):
        sp = tables.species(fx, 1, chosen)
        hbt = timed(lambda: api.hbt_moments(fl, dc, sp, g, tab, memory="device")[1], args.steps, args.warmup, torch)
        spec = timed(lambda: api.smooth_spectra(fl, dc, sp, g, tab, memory="device")[1], args.steps, args.warmup, torch)
        out["lists"][label] = dict(
            species=len(sp["mass"]),
            evaluations_per_call=hbt["evaluations"],
            hbt=dict(kernel_evals_per_s=hbt["evaluations"] / (hbt["kernel_ms"] * 1e-3), call_evals_per_s=hbt["evaluations"] / hbt["wall_s"],
                     kernel_ms=hbt["kernel_ms"], call_ms=hbt["call_ms"]),
            spectra=dict(kernel_evals_per_s=spec["evaluations"] / (spec["kernel_ms"] * 1e-3), call_evals_per_s=spec["evaluations"] / spec["wall_s"],
                         kernel_ms=spec["kernel_ms"], call_ms=spec["call_ms"]),
            hbt_over_spectra_kernel_time=hbt["kernel_ms"] / spec["kernel_ms"])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
