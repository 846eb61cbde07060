"""Throughput of the thermal-shear polarization path (is3d_b200_spin_polarization_shear) next to the vorticity path on the same surface.

Seeded 1M-cell 3+1D surface (the cfg3 generator) with synthetic thermal vorticity and thermal shear, the full 32 pT x 24 phi x 21 y
grid, surface arrays resident on the GPU (memory = device), two species lists: Lambda / anti-Lambda (what polarization users run) and
the 305-species list of the headline benchmark.  Prints one JSON line with evaluations/s of both paths (CUDA events of the library,
kernel and whole call) and the GPU's name and power limit, read in the same process.

    python tools/bench_polarization_shear.py [--cells N] [--steps K] [--warmup W]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def gpu_identity(torch):
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power, clock = (float(v) for v in out.split(","))
    except (OSError, ValueError, subprocess.TimeoutExpired):
        power, clock = None, None
    return dict(name=name, power_limit_w=power, max_sm_clock_mhz=clock)


def timed(fn, steps, warmup, torch):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    kernel, total = [], []
    t0 = time.perf_counter()
    for _ in range(steps):
        st = fn()
        kernel.append(st["kernel_ms"]); total.append(st["total_ms"])
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / steps
    return dict(kernel_ms=float(np.median(kernel)), call_ms=float(np.median(total)), wall_s=wall, evaluations=int(st["evaluations"]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    import torch
    from is3d_b200 import api, synthetic, tables
    if not torch.cuda.is_available():
        raise SystemExit("bench_polarization_shear needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(0)
    api.init()
    fx = tables.load_fixture()
    cells = synthetic.columns_to_cells(synthetic.surface_vh(args.cells, synthetic.SEEDS["cfg3"], three_d=True), 1)
    vort = synthetic.vorticity(args.cells, synthetic.SEEDS["cfg3"] + 1)
    xi = synthetic.thermal_shear(args.cells, synthetic.SEEDS["cfg3"] + 2)
    dc = {k: torch.tensor(v, device="cuda") for k, v in cells.items()}
    dv = {k: torch.tensor(v, device="cuda") for k, v in vort.items()}
    dx = {k: torch.tensor(v, device="cuda") for k, v in xi.items()}
    g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=3)
    out = dict(workload="%d-cell 3+1D surface with thermal vorticity and shear, %d pT x %d phi x %d y" % (args.cells, len(g["pT"]), len(g["phi"]), len(g["y"])),
               steps=args.steps, gpu=gpu_identity(torch), lists={})
    for label, chosen in (("lambda_antilambda", [3122, -3122]), ("pdg305", "chosen_urqmd")):
        sp = tables.species(fx, 1, chosen)
        xis = timed(lambda: api.spin_polarization_shear(fl, dc, dx, sp, g, memory="device")[1], args.steps, args.warmup, torch)
        vor = timed(lambda: api.spin_polarization(fl, dc, dv, sp, g, memory="device")[1], args.steps, args.warmup, torch)
        out["lists"][label] = dict(
            species=len(sp["mass"]),
            evaluations_per_call=xis["evaluations"],
            shear=dict(kernel_evals_per_s=xis["evaluations"] / (xis["kernel_ms"] * 1e-3), call_evals_per_s=xis["evaluations"] / xis["wall_s"],
                       kernel_ms=xis["kernel_ms"], call_ms=xis["call_ms"]),
            vorticity=dict(kernel_evals_per_s=vor["evaluations"] / (vor["kernel_ms"] * 1e-3), call_evals_per_s=vor["evaluations"] / vor["wall_s"],
                           kernel_ms=vor["kernel_ms"], call_ms=vor["call_ms"]),
            shear_over_vorticity_kernel_time=xis["kernel_ms"] / vor["kernel_ms"])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
