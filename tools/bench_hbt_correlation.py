"""Throughput of the HBT Fourier path (is3d_b200_hbt_fourier) next to the HBT moments (is3d_b200_hbt_moments) on the same surface.

Seeded 1M-cell 3+1D viscous surface (the cfg3 generator), df_mode 1 with shear and bulk delta-f, the full 32 pT x 24 phi x 21 y grid,
pi+ only (HBT is an identical-particle measurement), surface arrays resident on the GPU (memory = device), the out, side and long rays
with 41 q points each (what results/hbt/C_<mcid>.dat holds by default).  Prints one JSON line with the kernel and call time,
evaluations/s and phase terms/s (evaluations x rays x q points) of the Fourier path, its kernel-time ratio to the moments, and the GPU's
name and power limit, read in the same process.

    python tools/bench_hbt_correlation.py [--cells N] [--steps K] [--warmup W] [--q-points N] [--dq GEV]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_polarization import gpu_identity, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--q-points", type=int, default=41)
    ap.add_argument("--dq", type=float, default=0.005)
    args = ap.parse_args()
    import torch
    from is3d_b200 import api, synthetic, tables
    if not torch.cuda.is_available():
        raise SystemExit("bench_hbt_correlation needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(0)
    api.init()
    fx = tables.load_fixture()
    cells = synthetic.columns_to_cells(synthetic.surface_vh(args.cells, synthetic.SEEDS["cfg3"], three_d=True), 1)
    dc = {k: torch.tensor(v, device="cuda") for k, v in cells.items()}
    g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=3)
    tab = tables.df_tables(fx, 1)
    sp = tables.species(fx, 1, [211])
    qr = dict(dir=np.eye(3), dq=args.dq, n_q=args.q_points)
    fourier = timed(lambda: api.hbt_fourier(fl, dc, sp, g, tab, qr, memory="device")[1], args.steps, args.warmup, torch)
    moments = timed(lambda: api.hbt_moments(fl, dc, sp, g, tab, memory="device")[1], args.steps, args.warmup, torch)
    ev = fourier["evaluations"]
    terms = ev * 3 * args.q_points
    out = dict(workload="%d-cell 3+1D surface, df_mode 1, pi+ only, %d pT x %d phi x %d y, 3 rays x %d q (dq %g GeV)"
               % (args.cells, len(g["pT"]), len(g["phi"]), len(g["y"]), args.q_points, args.dq),
               steps=args.steps, gpu=gpu_identity(torch),
               evaluations_per_call=ev, phase_terms_per_call=terms,
               fourier=dict(kernel_ms=fourier["kernel_ms"], call_ms=fourier["call_ms"],
                            kernel_evals_per_s=ev / (fourier["kernel_ms"] * 1e-3), kernel_phase_terms_per_s=terms / (fourier["kernel_ms"] * 1e-3),
                            call_evals_per_s=ev / fourier["wall_s"], call_phase_terms_per_s=terms / fourier["wall_s"]),
               moments=dict(kernel_ms=moments["kernel_ms"], call_ms=moments["call_ms"],
                            kernel_evals_per_s=moments["evaluations"] / (moments["kernel_ms"] * 1e-3)),
               fourier_over_moments_kernel_time=fourier["kernel_ms"] / moments["kernel_ms"])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
