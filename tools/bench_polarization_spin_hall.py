"""Throughput of the spin Hall polarization path (is3d_b200_spin_polarization_spin_hall) next to the vorticity path on the same surface.

Seeded 1M-cell 3+1D surface (the cfg3 generator) with synthetic thermal vorticity and gradient of muB/T, the full 32 pT x 24 phi x 21 y
grid, surface arrays resident on the GPU (memory = device), two species lists: Lambda / anti-Lambda (what polarization users run) and
the 305-species list of the headline benchmark.  One warm-up call, then the median of --steps calls of each path, alternated so that
both see the same clocks.  Prints one JSON line with evaluations/s of both paths (CUDA events of the library, kernel and whole call)
and the GPU's name, power limit and maximum SM clock, read in the same process.

    python tools/bench_polarization_spin_hall.py [--cells N] [--steps K] [--warmup W]
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


def timed_pair(fns, steps, warmup, torch):
    """Warm-up calls of every path, then `steps` rounds that call each path once: per path the median kernel and call time."""
    for fn in fns:
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    res = [dict(kernel=[], total=[], wall=[]) for _ in fns]
    for _ in range(steps):
        for fn, r in zip(fns, res):
            t0 = time.perf_counter()
            st = fn()
            torch.cuda.synchronize()
            r["wall"].append(time.perf_counter() - t0)
            r["kernel"].append(st["kernel_ms"]); r["total"].append(st["total_ms"]); r["evaluations"] = int(st["evaluations"])
    return [dict(kernel_ms=float(np.median(r["kernel"])), call_ms=float(np.median(r["total"])), wall_s=float(np.median(r["wall"])),
                 evaluations=r["evaluations"]) for r in res]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    import torch
    from is3d_b200 import api, synthetic, tables
    if not torch.cuda.is_available():
        raise SystemExit("bench_polarization_spin_hall needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(0)
    api.init()
    fx = tables.load_fixture()
    cells = synthetic.columns_to_cells(synthetic.surface_vh(args.cells, synthetic.SEEDS["cfg3"], three_d=True), 1)
    vort = synthetic.vorticity(args.cells, synthetic.SEEDS["cfg3"] + 1)
    gb = synthetic.baryon_gradient(args.cells, synthetic.SEEDS["cfg3"] + 3)
    dc = {k: torch.tensor(v, device="cuda") for k, v in cells.items()}
    dv = {k: torch.tensor(v, device="cuda") for k, v in vort.items()}
    dg = {k: torch.tensor(v, device="cuda") for k, v in gb.items()}
    g = tables.grid(fx)
    fl = tables.flags(df_mode=1, dimension=3)
    out = dict(workload="%d-cell 3+1D surface with thermal vorticity and grad(muB/T), %d pT x %d phi x %d y" % (args.cells, len(g["pT"]), len(g["phi"]), len(g["y"])),
               steps=args.steps, gpu=gpu_identity(torch), lists={})
    for label, chosen in (("lambda_antilambda", [3122, -3122]), ("pdg305", "chosen_urqmd")):
        sp = tables.species(fx, 1, chosen)
        she, vor = timed_pair([lambda: api.spin_polarization_spin_hall(fl, dc, dg, sp, g, memory="device")[1],
                               lambda: api.spin_polarization(fl, dc, dv, sp, g, memory="device")[1]], args.steps, args.warmup, torch)
        out["lists"][label] = dict(
            species=len(sp["mass"]),
            evaluations_per_call=she["evaluations"],
            spin_hall=dict(kernel_evals_per_s=she["evaluations"] / (she["kernel_ms"] * 1e-3), call_evals_per_s=she["evaluations"] / she["wall_s"],
                           kernel_ms=she["kernel_ms"], call_ms=she["call_ms"]),
            vorticity=dict(kernel_evals_per_s=vor["evaluations"] / (vor["kernel_ms"] * 1e-3), call_evals_per_s=vor["evaluations"] / vor["wall_s"],
                           kernel_ms=vor["kernel_ms"], call_ms=vor["call_ms"]),
            spin_hall_over_vorticity_kernel_time=she["kernel_ms"] / vor["kernel_ms"])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
